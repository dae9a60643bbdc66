"""ctypes binding of libsblk.so (C ABI declared in include/sblk.h).

There is deliberately NO fallback: if the shared library is missing or a call fails, a RuntimeError
is raised.  PyTorch is used by callers only for device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsblk.so")

_lock = threading.Lock()
_lib = None

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_ll = ctypes.c_longlong



class EncoderStackArgs(ctypes.Structure):
    """Mirror of `sblk_encoder_stack_args` (include/sblk.h)."""
    _fields_ = ([(n, _vp) for n in (
        "x_in", "w_in", "b_in", "ln_in_gamma", "ln_in_beta", "pe", "w_heads", "b_heads", "w_fc", "b_fc", "ln1_gamma",
        "ln1_beta", "w_1", "b_1", "w_2", "b_2", "ln2_gamma", "ln2_beta", "lengths", "out", "workspace")] +
        [(n, _i) for n in ("N", "T", "n_layers", "n_head", "d_k", "d_model", "d_in", "d_inner")] +
        [("scale", _f), ("eps", _f), ("cluster_size", _i), ("debug_stamps", _vp), ("resident_counter", _vp),
         ("no_multicast", _i), ("groups_per_cluster", _i)])


# name -> (restype, argtypes); must list EVERY symbol include/sblk.h declares (tests check this).
SIGNATURES = {
    "sblk_version": (_i, []),
    "sblk_last_error": (ctypes.c_char_p, []),
    "sblk_init": (_i, []),
    "sblk_watchdog_code": (ctypes.c_uint, []),
    "sblk_set_pdl": (_i, [_i]),
    "sblk_set_sm_limit": (_i, [_i]),
    "sblk_set_stem_variant": (_i, [_i]),
    "sblk_launch_count": (_ll, []),
    "sblk_pack_conv3d": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp]),
    "sblk_pack_conv2d": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_cast_f32_bf16": (_i, [_vp, _vp, _ll, _vp]),
    "sblk_enc16_format": (_i, []),
    "sblk_cast_f32_enc16": (_i, [_vp, _vp, _ll, _vp]),
    "sblk_l2_prefetch": (_i, [ctypes.POINTER(_vp), ctypes.POINTER(_ll), _i, _vp]),
    "sblk_gate_wait": (_i, [_vp, _i, _i, _vp]),
    "sblk_prep_clip_elems": (_ll, [_i, _i]),
    "sblk_prep_clip": (_i, [_vp, _vp, _i, _i, _vp]),
    "sblk_prep_clip_u8": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "sblk_conv3d_bn_relu_pool_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "sblk_stem_fused_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_flat_rows": (_ll, [_i, _i, _i]),
    "sblk_flatconv3x3_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "sblk_flatconv3x3_dir_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_conv2d_igemm_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_conv2d_igemm_ext_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i,
                                       _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_conv_block_flag_words": (_i, [_i, _i, _i, _i]),
    "sblk_conv_block_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_conv2d_dual_igemm_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i,
                                        _vp]),
    "sblk_avgpool_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "sblk_avgpool_scale_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_gemm_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_add_layernorm_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "sblk_attention_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "sblk_gemm_splitk_plan": (_i, [_i, _i, _i]),
    "sblk_gemm_splitk_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_sum_layernorm_fwd": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "sblk_gemm_ln_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "sblk_qkv_group_clips": (_i, [_i]),
    "sblk_qkv_attention_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "sblk_p2p_alloc": (_i, [_ll, ctypes.POINTER(_vp), _vp]),
    "sblk_p2p_open": (_i, [_vp, ctypes.POINTER(_vp)]),
    "sblk_p2p_close": (_i, [_vp, _i]),
    "sblk_p2p_gather_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _ll, ctypes.c_uint, _vp]),
    "sblk_set_p2p_timeout_ms": (ctypes.c_uint, [ctypes.c_uint]),
    "sblk_gemm_fmt_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_transpose16": (_i, [_vp, _vp, _ll, _i, _ll, _ll, _i, _vp]),
    "sblk_im2col_t": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _ll, _vp]),
    "sblk_stem_im2col": (_i, [_vp, _vp, _i, _i, _i, _ll, _vp]),
    "sblk_stem_im2col_u8": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _ll, _vp]),
    "sblk_colreduce_workspace_floats": (_ll, [_i]),
    "sblk_colreduce": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp]),
    "sblk_bn_finalize": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _f, _f, _f, _vp]),
    "sblk_bn_apply_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp]),
    "sblk_bn_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _vp]),
    "sblk_maxpool3x3s2_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_maxpool3x3s2_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "sblk_avgpool_bwd": (_i, [_vp, _vp, _ll, _i, _i, _vp]),
    "sblk_zero_stuff2": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "sblk_relu_bwd": (_i, [_vp, _vp, _ll, _vp]),
    "sblk_ln_bwd_workspace_floats": (_ll, []),
    "sblk_ln_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "sblk_attention_train_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "sblk_attention_train_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "sblk_xattention_train_fwd": (_i, [_vp] * 7 + [_i] * 9 + [_f, _vp]),
    "sblk_xattention_train_bwd": (_i, [_vp] * 10 + [_i] * 12 + [_f, _vp]),
    "sblk_xattention_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "sblk_embed_pe_fwd": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "sblk_bidir_mix_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "sblk_bidir_mix_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "sblk_embed_bwd": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "sblk_encoder_stack_workspace_bytes": (_ll, [_i, _i, _i]),
    "sblk_encoder_stack_fwd": (_i, [ctypes.POINTER(EncoderStackArgs), _vp]),
}


def load():
    """Load libsblk.so once; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback for the visual-encoder path.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().sblk_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        lib = load()
        wd = lib.sblk_watchdog_code()
        extra = f" [pipeline watchdog 0x{wd:08x}]" if wd else ""
        raise RuntimeError(f"{what} failed (rc={rc}): {last_error()}{extra}")
