"""Thin tensor-level wrappers over the libsblk C ABI.

Each function validates dtype / device / contiguity, allocates the output with torch (device memory is
torch's job, arithmetic is not) and enqueues the kernel on torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

BF16 = torch.bfloat16
F32 = torch.float32
_ENC16 = None


def enc16_dtype():
    """torch dtype of the transformer encoder's 16-bit GEMM / attention operands ("enc16", include/sblk.h): float16 in
    the default build (LayerNorm-bounded values: 3 more mantissa bits than bf16 at the same tcgen05 kind::f16 rate),
    bfloat16 when libsblk was built with -DSBLK_ENC_FP16=0.  The convolutional trunk is always bf16."""
    global _ENC16
    if _ENC16 is None:
        _ENC16 = torch.float16 if int(_lib.load().sblk_enc16_format()) == 1 else torch.bfloat16
    return _ENC16


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (no CPU fallback exists), got {t.device}")
    if t.dtype != dtype:
        raise RuntimeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous tensor")


# Optional per-launch trace (bench.py / profiling): when a list is installed with `trace(list)`, every wrapper
# brackets its launch with CUDA events on the launching stream and appends
# {"name", "tag", "flops", "bytes", "start", "end"}; algorithmic flops/bytes are the figures DESIGN.md states.
_TRACE = None


class trace:
    def __init__(self, sink):
        self.sink = sink

    def __enter__(self):
        global _TRACE
        self._prev, _TRACE = _TRACE, self.sink
        return self.sink

    def __exit__(self, *exc):
        global _TRACE
        _TRACE = self._prev
        return False


def _call(name, tag, flops, nbytes, *args):
    fn = getattr(_lib.load(), name)
    tr = _TRACE
    if tr is None:
        _lib.check(fn(*args), name)
        return
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    _lib.check(fn(*args), name)
    e1.record(s)
    tr.append(dict(name=name, tag=tag, flops=flops, bytes=nbytes, start=e0, end=e1))


def init() -> int:
    """Per-device setup; returns the SM count."""
    n = _lib.load().sblk_init()
    if n <= 0:
        raise RuntimeError(f"sblk_init failed (rc={n}): {_lib.last_error()}")
    return n


def set_pdl(enable: bool) -> bool:
    return bool(_lib.load().sblk_set_pdl(1 if enable else 0))


def set_sm_limit(max_sms: int) -> int:
    """Size persistent grids of this thread's next launches for at most `max_sms` SMs (0 = all); returns the old limit."""
    return int(_lib.load().sblk_set_sm_limit(int(max_sms)))


def set_stem_variant(variant: int) -> int:
    """Stem kernel of this thread's next launches: 0 = transposed, filter in tensor memory (default); 1 = the
    pixel-major round-1 kernel (A/B measurements).  Returns the previous value."""
    return int(_lib.load().sblk_set_stem_variant(int(variant)))


def launch_count() -> int:
    return int(_lib.load().sblk_launch_count())


# ------------------------------------------------------------------------------------ packers
def pack_conv3d(w, gamma, beta, mean, var, eps=1e-5):
    for t, n in ((w, "w"), (gamma, "gamma"), (beta, "beta"), (mean, "mean"), (var, "var")):
        _req(t, F32, n)
    if tuple(w.shape) != (64, 1, 5, 7, 7):
        raise RuntimeError(f"pack_conv3d: weight shape {tuple(w.shape)} != (64,1,5,7,7)")
    wp = torch.empty((64, 320), dtype=BF16, device=w.device)
    bias = torch.empty((64,), dtype=F32, device=w.device)
    _call("sblk_pack_conv3d", "pack", 0, 0, _p(w), _p(gamma), _p(beta), _p(mean), _p(var), eps, _p(wp), _p(bias),
          _stream())
    return wp, bias


def pack_conv2d(w, gamma=None, beta=None, mean=None, var=None, eps=1e-5):
    _req(w, F32, "w")
    for t, n in ((gamma, "gamma"), (beta, "beta"), (mean, "mean"), (var, "var")):
        _req(t, F32, n)
    co, ci, r, s = w.shape
    wp = torch.empty((co, r, s, ci), dtype=BF16, device=w.device)
    bias = torch.empty((co,), dtype=F32, device=w.device)
    _call("sblk_pack_conv2d", "pack", 0, 0, _p(w), _p(gamma), _p(beta), _p(mean), _p(var), eps, _p(wp), _p(bias),
          co, ci, r, s, _stream())
    return wp, bias


def cast_bf16(x, out=None):
    _req(x, F32, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=BF16, device=x.device)
    _req(out, BF16, "out")
    _call("sblk_cast_f32_bf16", f"cast n={x.numel()}", 0, 6 * x.numel(), _p(x), _p(out), x.numel(), _stream())
    return out


def cast_enc16(x, out=None):
    """fp32 -> the encoder's 16-bit operand format (weights [out,in] are already K-major; fp16 saturates at 65504)."""
    _req(x, F32, "x")
    e16 = enc16_dtype()
    if out is None:
        out = torch.empty(x.shape, dtype=e16, device=x.device)
    _req(out, e16, "out")
    _call("sblk_cast_f32_enc16", f"cast n={x.numel()}", 0, 6 * x.numel(), _p(x), _p(out), x.numel(), _stream())
    return out


def l2_prefetch(tensors):
    """Hint: pull the storage of every (CUDA, contiguous) tensor in `tensors` into L2 on the current stream (one launch
    per 24 tensors)."""
    ts = [t for t in tensors if t is not None and t.numel() > 0]
    if not ts:
        return
    for t in ts:
        if not t.is_cuda or not t.is_contiguous():
            raise RuntimeError("l2_prefetch: expected contiguous CUDA tensors")
    ptrs = (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    nbytes = (ctypes.c_longlong * len(ts))(*[t.numel() * t.element_size() for t in ts])
    _lib.check(_lib.load().sblk_l2_prefetch(ptrs, nbytes, len(ts), _stream()), "sblk_l2_prefetch")


def gate_wait(gate, count, timeout_us=300):
    """Co-scheduling hint: hold the current stream until `count` more CTAs of a kernel launched with
    `resident_counter=gate` (encoder_stack) have started running, or `timeout_us` passed.  gate: int32 [2] CUDA tensor,
    zero-initialised once and then owned by the pair of launches."""
    _req(gate, torch.int32, "gate")
    if gate.numel() < 2:
        raise RuntimeError("gate_wait: gate must hold two int32 words")
    _lib.check(_lib.load().sblk_gate_wait(_p(gate), int(count), int(timeout_us), _stream()), "sblk_gate_wait")


# ------------------------------------------------------------------------------------ frontend
def prep_clip(x, out=None):
    """x fp32 [N,1,T,88,88] (or [N,T,88,88]) -> (flat bf16 row-Toeplitz clip, N, T) for conv3d_bn_relu_pool."""
    _req(x, F32, "x")
    if x.dim() == 5:
        n, c, t, h, w = x.shape
        if c != 1:
            raise RuntimeError("prep_clip: expected one (gray) channel")
    else:
        n, t, h, w = x.shape
    if (h, w) != (88, 88):
        raise RuntimeError(f"prep_clip: frames must be 88x88, got {h}x{w}")
    elems = int(_lib.load().sblk_prep_clip_elems(n, t))
    if out is None:
        out = torch.empty((elems,), dtype=BF16, device=x.device)
    _req(out, BF16, "out")
    if out.numel() < elems:
        raise RuntimeError(f"prep_clip: output needs {elems} bf16 elements, got {out.numel()}")
    _call("sblk_prep_clip", f"prep N={n} T={t}", 0, 4 * x.numel() + 2 * elems, _p(x), _p(out), n, t, _stream())
    return out, n, t


class FlatActs:
    """Activations in the zero-haloed flat layout of csrc/sblk_flatconv2.cuh: `data` is bf16 [rows, C] with pixel
    (f, y, x) at row (f*(H+1) + 1 + y)*(W+2) + 1 + x and zeros everywhere else."""
    __slots__ = ("data", "f", "h", "w")

    def __init__(self, data, f, h, w):
        self.data, self.f, self.h, self.w = data, f, h, w

    @property
    def c(self):
        return self.data.shape[1]

    def dense(self):
        """-> bf16 NHWC [F,H,W,C] copy (tests / debugging; torch indexing only)."""
        f, h, w, c = self.f, self.h, self.w, self.c
        v = self.data[(w + 2):(w + 2) + f * (h + 1) * (w + 2)].view(f, h + 1, w + 2, c)
        return v[:, :h, 1:w + 1, :].contiguous()


def flat_rows(f, h, w):
    return int(_lib.load().sblk_flat_rows(f, h, w))


def flat_frames(x, f0, f1):
    """Frames [f0, f1) of FlatActs `x` as FlatActs over a row slice of the same storage.  The layout is linear in the
    frame index and consecutive frames share one zero halo row, so the slice is itself a valid zero-haloed flat buffer
    (its first / last rows are the halo rows in front of frames f0 / f1)."""
    if not 0 <= f0 < f1 <= x.f:
        raise RuntimeError(f"flat_frames: bad frame range [{f0}, {f1}) of {x.f}")
    r0 = f0 * (x.h + 1) * (x.w + 2)
    return FlatActs(x.data[r0:r0 + ((f1 - f0) * (x.h + 1) + 1) * (x.w + 2)], f1 - f0, x.h, x.w)


def prep_clip_u8(x_u8, lut, t_out=None, crop=(4, 4), out=None):
    """Raw uint8 gray frames [N,T_in,H0,W0] -> (prepped bf16 clip, N, T_out) for conv3d_bn_relu_pool, fusing the reference
    loader's /255, ColorNormalize, 88x88 crop and frame zero-padding (data_gen.py:122-125,276-296).  `lut`: bf16 [256]
    (synth.normalize_lut()).  `crop`: (y1, x1) for every frame (CenterCrop of 96x96 = (4, 4)) or an int32 CUDA tensor
    [N*T_in, 2] of per-frame offsets (RandomCrop)."""
    if not x_u8.is_cuda or x_u8.dtype != torch.uint8 or not x_u8.is_contiguous() or x_u8.dim() != 4:
        raise RuntimeError("prep_clip_u8: expected a contiguous CUDA uint8 tensor [N,T,H0,W0] (no CPU fallback exists)")
    _req(lut, BF16, "lut")
    if lut.numel() != 256:
        raise RuntimeError("prep_clip_u8: lut must hold 256 bf16 values")
    n, t_in, h0, w0 = x_u8.shape
    t_out = t_in if t_out is None else int(t_out)
    crop_t, cy, cx = None, 0, 0
    if torch.is_tensor(crop):
        _req(crop, torch.int32, "crop")
        if tuple(crop.shape) != (n * t_in, 2):
            raise RuntimeError(f"prep_clip_u8: per-frame crop must be int32 [{n * t_in}, 2]")
        crop_t = crop
    else:
        cy, cx = int(crop[0]), int(crop[1])
    elems = int(_lib.load().sblk_prep_clip_elems(n, t_out))
    if elems <= 0:
        raise RuntimeError(f"prep_clip_u8: bad clip shape N={n} T={t_out}")
    if out is None:
        out = torch.empty((elems,), dtype=BF16, device=x_u8.device)
    _req(out, BF16, "out")
    if out.numel() < elems:
        raise RuntimeError(f"prep_clip_u8: output needs {elems} bf16 elements, got {out.numel()}")
    _call("sblk_prep_clip_u8", f"prep_u8 N={n} T={t_out}", 0, x_u8.numel() + 2 * elems, _p(x_u8), _p(lut), _p(crop_t), cy,
          cx, _p(out), n, t_in, t_out, h0, w0, _stream())
    return out, n, t_out


class RawClip:
    """An un-prepped stem input for the FUSED stem (sblk_stem_fused_fwd): the kernel's producer warps build the
    row-Toeplitz entries themselves, so no prepped copy of the clip is written.  kind "f32": x fp32 [N,1,T,88,88] /
    [N,T,88,88]; kind "u8": raw uint8 frames [N,T_in,H0,W0] + normalisation table + crop + frame padding."""
    __slots__ = ("kind", "x", "lut", "crop", "n", "t_in", "t")

    def __init__(self, kind, x, n, t_in, t, lut=None, crop=None):
        self.kind, self.x, self.n, self.t_in, self.t, self.lut, self.crop = kind, x, n, t_in, t, lut, crop


def raw_clip(x):
    """fp32 clips for the fused stem (same checks as prep_clip; nothing is launched)."""
    _req(x, F32, "x")
    if x.dim() == 5:
        n, c, t, h, w = x.shape
        if c != 1:
            raise RuntimeError("raw_clip: expected one (gray) channel")
    else:
        n, t, h, w = x.shape
    if (h, w) != (88, 88):
        raise RuntimeError(f"raw_clip: frames must be 88x88, got {h}x{w}")
    return RawClip("f32", x, n, t, t)


def raw_clip_u8(x_u8, lut, t_out=None, crop=(4, 4)):
    """Raw uint8 frames for the fused stem (same checks as prep_clip_u8; nothing is launched)."""
    if not x_u8.is_cuda or x_u8.dtype != torch.uint8 or not x_u8.is_contiguous() or x_u8.dim() != 4:
        raise RuntimeError("raw_clip_u8: expected a contiguous CUDA uint8 tensor [N,T,H0,W0] (no CPU fallback exists)")
    _req(lut, BF16, "lut")
    if lut.numel() != 256:
        raise RuntimeError("raw_clip_u8: lut must hold 256 bf16 values")
    n, t_in, h0, w0 = x_u8.shape
    t_out = t_in if t_out is None else int(t_out)
    if torch.is_tensor(crop):
        _req(crop, torch.int32, "crop")
        if tuple(crop.shape) != (n * t_in, 2):
            raise RuntimeError(f"raw_clip_u8: per-frame crop must be int32 [{n * t_in}, 2]")
    else:
        crop = (int(crop[0]), int(crop[1]))
    return RawClip("u8", x_u8, n, t_in, t_out, lut=lut, crop=crop)


def conv3d_bn_relu_pool(xp, wp, bias, out=None, flat=False):
    """Stem: prepped clip (out, N, T) of prep_clip[_u8] — or a RawClip (fused: no prepped copy) — -> bf16 NHWC
    [N*T,22,22,64], or FlatActs when flat=True."""
    raw = xp if isinstance(xp, RawClip) else None
    if raw is not None:
        n, t, dev_ = raw.n, raw.t, raw.x.device
    else:
        xp, n, t = xp
        _req(xp, BF16, "xp")
        dev_ = xp.device
    _req(wp, BF16, "wp"); _req(bias, F32, "bias")
    if out is None:
        shape = (flat_rows(n * t, 22, 22), 64) if flat else (n * t, 22, 22, 64)
        out = torch.empty(shape, dtype=BF16, device=dev_)
    _req(out, BF16, "out")
    flops = 2 * 64 * 44 * 44 * 245 * n * t
    if raw is None:
        _call("sblk_conv3d_bn_relu_pool_fwd", f"conv3d N={n} T={t}", flops,
              2 * xp.numel() + 2 * out.numel(), _p(xp), _p(wp), _p(bias), _p(out), n, t, 1 if flat else 0, _stream())
    elif raw.kind == "f32":
        _call("sblk_stem_fused_fwd", f"conv3d N={n} T={t}", flops, 4 * raw.x.numel() + 2 * out.numel(),
              _p(raw.x), None, None, None, 0, 0, _p(wp), _p(bias), _p(out), n, t, t, 88, 88, 1 if flat else 0, _stream())
    else:
        crop_t, cy, cx = (raw.crop, 0, 0) if torch.is_tensor(raw.crop) else (None, raw.crop[0], raw.crop[1])
        h0, w0 = raw.x.shape[2], raw.x.shape[3]
        _call("sblk_stem_fused_fwd", f"conv3d N={n} T={t}", flops, raw.x.numel() + 2 * out.numel(),
              None, _p(raw.x), _p(raw.lut), _p(crop_t), cy, cx, _p(wp), _p(bias), _p(out), n, raw.t_in, t, h0, w0,
              1 if flat else 0, _stream())
    return FlatActs(out, n * t, 22, 22) if flat else out


def pack_flat_weight(wp):
    """pack_conv2d's bf16 [C,3,3,C] -> [C, 10*C]: the 9 taps followed by a CxC identity (residual via the tensor core)."""
    _req(wp, BF16, "wp")
    c = wp.shape[0]
    if tuple(wp.shape) != (c, 3, 3, c):
        raise RuntimeError(f"pack_flat_weight: weight shape {tuple(wp.shape)} != {(c, 3, 3, c)}")
    return torch.cat([wp.view(c, 9 * c), torch.eye(c, dtype=BF16, device=wp.device)], dim=1).contiguous()


def conv3x3_flat(x, wp, bias, relu=True, residual=None, out=None, reverse=False):
    """Stride-1 3x3 conv over FlatActs (C -> C, C = 64 or 128) -> FlatActs.  wp bf16 [C, 10*C] (pack_flat_weight).
    reverse: every CTA pair walks its tile range backwards (sblk_flatconv3x3_dir_fwd) — alternate it between the
    consecutive convs of a stage so each conv starts on the rows the previous one touched last (L2 reuse); same bits."""
    _req(x.data, BF16, "x"); _req(wp, BF16, "wp"); _req(bias, F32, "bias")
    c = x.c
    if tuple(wp.shape) != (c, 10 * c):
        raise RuntimeError(f"conv3x3_flat: weight shape {tuple(wp.shape)} != {(c, 10 * c)} (use pack_flat_weight)")
    if residual is not None:
        _req(residual.data, BF16, "residual")
        if residual.data.shape != x.data.shape:
            raise RuntimeError("conv3x3_flat: residual shape mismatch")
    if out is None:
        out = torch.empty_like(x.data)
    _req(out, BF16, "out")
    _call("sblk_flatconv3x3_dir_fwd", f"flatconv3x3 H={x.h} {c}->{c}", 2 * x.f * x.h * x.w * c * 9 * c,
          2 * (x.data.numel() + wp.numel() + out.numel() + (0 if residual is None else residual.data.numel())),
          _p(x.data), _p(wp), _p(bias), None if residual is None else _p(residual.data), _p(out), x.f, x.h, x.w, c,
          1 if relu else 0, 1 if reverse else 0, _stream())
    return FlatActs(out, x.f, x.h, x.w)


def _conv_input(x):
    if isinstance(x, FlatActs):
        _req(x.data, BF16, "x")
        f, h, w, cin = x.f, x.h, x.w, x.c
        return (x.data.data_ptr() + (w + 3) * cin * 2, f, h, w, cin, w + 2, (h + 1) * (w + 2), x.data.numel())
    _req(x, BF16, "x")
    f, h, w, cin = x.shape
    return (x.data_ptr(), f, h, w, cin, 0, 0, x.numel())


def conv2d_dual(x, wp, bias, wp_ds, bias_ds, stride=2, relu=True, flat_ws=None):
    """BasicBlock head with a downsample branch in one launch:
    (relu(conv3x3_s(x) + bias), conv1x1_s(x) + bias_ds), both bf16 NHWC [F,P,Q,Cout].
    flat_ws = (buf, buf_ds): two bf16 [flat_rows(F,P,Q), Cout] workspaces whose halo rows are zero -> both outputs are
    written into them in the flat layout and returned as FlatActs (input of conv3x3_flat)."""
    _req(wp, BF16, "wp"); _req(bias, F32, "bias"); _req(wp_ds, BF16, "wp_ds"); _req(bias_ds, F32, "bias_ds")
    xptr, f, h, w, cin, row_pitch, frame_pitch, x_elems = _conv_input(x)
    cout = wp.shape[0]
    if tuple(wp.shape) != (cout, 3, 3, cin) or tuple(wp_ds.shape) != (cout, 1, 1, cin):
        raise RuntimeError(f"conv2d_dual: weight shapes {tuple(wp.shape)} / {tuple(wp_ds.shape)} do not match Cin={cin}")
    p = (h + 2 - 3) // stride + 1
    q = (w + 2 - 3) // stride + 1
    if flat_ws is not None:
        out, out_ds = flat_ws
        _req(out, BF16, "flat_ws[0]"); _req(out_ds, BF16, "flat_ws[1]")
        if tuple(out.shape) != (flat_rows(f, p, q), cout) or tuple(out_ds.shape) != tuple(out.shape):
            raise RuntimeError(f"conv2d_dual: flat workspaces must be [{flat_rows(f, p, q)}, {cout}]")
    else:
        out = torch.empty((f, p, q, cout), dtype=BF16, device=wp.device)
        out_ds = torch.empty((f, p, q, cout), dtype=BF16, device=wp.device)
    _call("sblk_conv2d_dual_igemm_fwd", f"conv3x3+ds H={h} {cin}->{cout} s{stride}", 2 * f * p * q * cout * 10 * cin,
          2 * (x_elems + wp.numel() + wp_ds.numel() + 2 * f * p * q * cout),
          xptr, _p(wp), _p(bias), _p(wp_ds), _p(bias_ds), _p(out), _p(out_ds), f, h, w, cin, cout, stride,
          1 if relu else 0, row_pitch, frame_pitch, 0 if flat_ws is None else 1, _stream())
    if flat_ws is not None:
        return FlatActs(out, f, p, q), FlatActs(out_ds, f, p, q)
    return out, out_ds


def conv2d(x, wp, bias, stride=1, relu=True, residual=None, out=None, ext=None):
    """x bf16 NHWC [F,H,W,Cin] (or FlatActs), wp bf16 [Cout,R,S,Cin] -> bf16 NHWC [F,P,Q,Cout].
    ext = (x2, w2, stride2): K-extension (sblk_conv2d_igemm_ext_fwd) — the 1x1 / stride2 conv of x2 (NHWC or FlatActs)
    with w2 [Cout,1,1,Cin2] is accumulated into the same fp32 tile before bias / residual / ReLU: a BasicBlock's
    downsample branch folded into its conv2 (pass bias = folded bn2 shift + folded downsample shift)."""
    _req(wp, BF16, "wp"); _req(bias, F32, "bias"); _req(residual, BF16, "residual")
    xptr, f, h, w, cin, row_pitch, frame_pitch, x_elems = _conv_input(x)
    cout, r, s, cin2 = wp.shape
    if cin2 != cin:
        raise RuntimeError(f"conv2d: Cin mismatch {cin} vs {cin2}")
    pad = 1 if r == 3 else 0
    p = (h + 2 * pad - r) // stride + 1
    q = (w + 2 * pad - s) // stride + 1
    if out is None:
        out = torch.empty((f, p, q, cout), dtype=BF16, device=wp.device)
    _req(out, BF16, "out")
    if residual is not None and residual.numel() != out.numel():
        raise RuntimeError("conv2d: residual shape mismatch")
    if ext is not None:
        x2, w2, stride2 = ext
        _req(w2, BF16, "ext w2")
        x2ptr, f2, h2, w2_, c2, rp2, fp2, x2_elems = _conv_input(x2)
        if f2 != f or tuple(w2.shape) != (cout, 1, 1, c2):
            raise RuntimeError(f"conv2d: extension shapes F={f2} w2={tuple(w2.shape)} do not match F={f} Cout={cout} Cin2={c2}")
        if ((h2 - 1) // stride2 + 1, (w2_ - 1) // stride2 + 1) != (p, q):
            raise RuntimeError("conv2d: the extension's output grid does not match the conv's")
        _call("sblk_conv2d_igemm_ext_fwd", f"conv{r}x{s}+ds H={h} {cin}->{cout} s{stride}",
              2 * f * p * q * cout * (r * s * cin + c2),
              2 * (x_elems + x2_elems + wp.numel() + w2.numel() + out.numel() + (0 if residual is None else residual.numel())),
              xptr, _p(wp), _p(bias), _p(residual), _p(out), f, h, w, cin, cout, r, s, stride, pad, 1 if relu else 0,
              row_pitch, frame_pitch, x2ptr, _p(w2), h2, w2_, c2, stride2, rp2, fp2, _stream())
        return out
    _call("sblk_conv2d_igemm_fwd", f"conv{r}x{s} H={h} {cin}->{cout} s{stride}", 2 * f * p * q * cout * r * s * cin,
          2 * (x_elems + wp.numel() + out.numel() + (0 if residual is None else residual.numel())),
          xptr, _p(wp), _p(bias), _p(residual), _p(out), f, h, w, cin, cout, r, s, stride, pad, 1 if relu else 0,
          row_pitch, frame_pitch, _stream())
    return out


_BLOCK_FLAGS = {}   # (device index, stream) -> zeroed uint32 counters of conv_block (self-resetting: zeroed once)


def _block_flags(dev, words):
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), int(_stream()))
    t = _BLOCK_FLAGS.get(key)
    if t is None or t.numel() < words:
        t = torch.zeros(max(1024, words), dtype=torch.int32, device=dev)
        _BLOCK_FLAGS[key] = t
    return t


def conv_block(x, w1, b1, w2, b2, w_ds=None, stride=1, out=None, y1=None, flags=None):
    """A whole BasicBlock of ResNet layer 3 / layer 4 in one launch (sblk_conv_block_fwd): x bf16 NHWC [F,H,W,Cin] or
    FlatActs; w1 [Cout,3,3,Cin], w2 [Cout,3,3,Cout] with Cout 256 or 512, w_ds [Cout,1,1,Cin] or None (identity residual);
    b2 must already include the folded downsample shift.  `flags`: zeroed int32 counters for Cout = 512 (default: one
    cached tensor per device and stream).  Returns out bf16 [F,P,Q,Cout], or None when the problem has more work units per
    CTA pair than the kernel takes (the caller then launches the two convs one by one)."""
    _req(w1, BF16, "w1"); _req(b1, F32, "b1"); _req(w2, BF16, "w2"); _req(b2, F32, "b2"); _req(w_ds, BF16, "w_ds")
    xptr, f, h, w, cin, row_pitch, frame_pitch, x_elems = _conv_input(x)
    cout = w1.shape[0]
    if tuple(w1.shape) != (cout, 3, 3, cin) or tuple(w2.shape) != (cout, 3, 3, cout):
        raise RuntimeError(f"conv_block: filter shapes {tuple(w1.shape)} / {tuple(w2.shape)} do not match Cin={cin}, Cout={cout}")
    if w_ds is not None and tuple(w_ds.shape) != (cout, 1, 1, cin):
        raise RuntimeError(f"conv_block: downsample filter shape {tuple(w_ds.shape)} != {(cout, 1, 1, cin)}")
    p = (h + 2 - 3) // stride + 1
    q = (w + 2 - 3) // stride + 1
    if out is None:
        out = torch.empty((f, p, q, cout), dtype=BF16, device=w1.device)
    if y1 is None:
        y1 = torch.empty((f, p, q, cout), dtype=BF16, device=w1.device)
    _req(out, BF16, "out"); _req(y1, BF16, "y1")
    if out.numel() != f * p * q * cout or y1.numel() != out.numel():
        raise RuntimeError("conv_block: out / y1 must hold F*P*Q*Cout elements")
    lib = _lib.load()
    if cout > 256 and flags is None:
        words = int(lib.sblk_conv_block_flag_words(f, h, w, stride))
        if words <= 0:
            raise RuntimeError("conv_block: bad shape")
        flags = _block_flags(w1.device, words)
    _req(flags, torch.int32, "flags")
    flops = 2 * f * p * q * cout * (9 * cin + 9 * cout + (cin if w_ds is not None else 0))
    nbytes = 2 * (x_elems + w1.numel() + w2.numel() + 3 * out.numel())
    try:
        _call("sblk_conv_block_fwd", f"block H={h} {cin}->{cout} s{stride}", flops, nbytes,
              xptr, _p(w1), _p(b1), _p(w2), _p(b2), _p(w_ds), _p(y1), _p(flags), _p(out), f, h, w, cin, cout, stride,
              row_pitch, frame_pitch, _stream())
    except RuntimeError as e:
        if "tiles per pair" in str(e):
            return None
        raise
    return out


def avgpool(x, want_f32=True, want_bf16=False, out_f32=None, out_bf16=None, scale=None, enc16=False):
    """bf16 NHWC [F, ..., C] -> (fp32 [F, C] | None, 16-bit [F, C] | None) mean over the pixels, optionally times the
    fp32 factor `scale` [F, C] (dropout mask / (1 - p) drawn ahead of time).  enc16=True writes the 16-bit copy in the
    encoder's operand format (enc16_dtype(): it is the encoder stack's x_in) instead of bf16."""
    o16_dt = enc16_dtype() if enc16 else BF16
    _req(x, BF16, "x"); _req(out_f32, F32, "out_f32"); _req(out_bf16, o16_dt, "out_bf16"); _req(scale, F32, "scale")
    f, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (f * c)
    for name, t_ in (("out_f32", out_f32), ("out_bf16", out_bf16), ("scale", scale)):
        if t_ is not None and t_.numel() != f * c:
            raise RuntimeError(f"avgpool: {name} has {t_.numel()} elements, expected {f * c}")
    o32 = out_f32 if out_f32 is not None else (torch.empty((f, c), dtype=F32, device=x.device) if want_f32 else None)
    o16 = out_bf16 if out_bf16 is not None else (torch.empty((f, c), dtype=o16_dt, device=x.device) if want_bf16 else None)
    _call("sblk_avgpool_scale_fwd", f"avgpool HW={hw} C={c}", 0, 2 * x.numel() + (4 if o32 is not None else 0) * f * c +
          (2 if o16 is not None else 0) * f * c + (4 if scale is not None else 0) * f * c,
          _p(x), _p(scale), _p(o32), _p(o16), f, hw, c, 1 if enc16 else 0, _stream())
    return o32, o16


# ------------------------------------------------------------------------------------ encoder
# (16-bit operands of everything below are in the encoder operand format, enc16_dtype())
def gemm(a, w, bias=None, residual=None, relu=False, out_bf16=False, out_f32=False):
    """a bf16 [M,K], w bf16 [N,K] -> (bf16 [M,N] | None, fp32 [M,N] | None)."""
    _req(a, enc16_dtype(), "a"); _req(w, enc16_dtype(), "w"); _req(bias, F32, "bias"); _req(residual, enc16_dtype(), "residual")
    m, k = a.shape
    n, k2 = w.shape
    if k2 != k:
        raise RuntimeError(f"gemm: K mismatch {k} vs {k2}")
    o16 = torch.empty((m, n), dtype=enc16_dtype(), device=a.device) if out_bf16 else None
    o32 = torch.empty((m, n), dtype=F32, device=a.device) if out_f32 else None
    _call("sblk_gemm_fwd", f"gemm N={n} K={k}", 2 * m * n * k,
          2 * (m * k + n * k) + m * n * ((2 if out_bf16 else 0) + (4 if out_f32 else 0)),
          _p(a), _p(w), _p(bias), _p(residual), _p(o16), _p(o32), m, n, k, 1 if relu else 0, _stream())
    return o16, o32


def add_layernorm(x, gamma, beta, residual=None, pe=None, lengths=None, T=1, eps=1e-5, want_f32=True,
                  want_bf16=True, out_f32=None):
    _req(x, F32, "x"); _req(gamma, F32, "gamma"); _req(beta, F32, "beta"); _req(residual, F32, "residual")
    _req(pe, F32, "pe"); _req(lengths, torch.int32, "lengths"); _req(out_f32, F32, "out_f32")
    m, d = x.shape
    if out_f32 is not None and tuple(out_f32.shape) != (m, d):
        raise RuntimeError(f"add_layernorm: out_f32 shape {tuple(out_f32.shape)} != {(m, d)}")
    o32 = out_f32 if out_f32 is not None else (torch.empty((m, d), dtype=F32, device=x.device) if want_f32 else None)
    o16 = torch.empty((m, d), dtype=enc16_dtype(), device=x.device) if want_bf16 else None
    _call("sblk_add_layernorm_fwd", "add_layernorm", 0,
          m * d * (4 + (4 if residual is not None else 0) + (4 if want_f32 else 0) + (2 if want_bf16 else 0)),
          _p(x), _p(residual), _p(gamma), _p(beta), _p(pe), _p(lengths), _p(o32), _p(o16), m, T, d, eps, _stream())
    return o32, o16


def gemm_ln(a, w, gamma, beta, bias=None, residual=None, pe=None, lengths=None, T=1, eps=1e-5, want_f32=True,
            want_bf16=True, out_f32=None):
    """LayerNorm(a @ w.T + bias + residual) * gamma + beta (+ pe[m % T]) (* pad mask) in one launch.
    a bf16 [M,K], w bf16 [512,K], residual fp32 [M,512] -> (fp32 [M,512] | None, bf16 [M,512] | None)."""
    _req(a, enc16_dtype(), "a"); _req(w, enc16_dtype(), "w"); _req(bias, F32, "bias"); _req(residual, F32, "residual")
    _req(gamma, F32, "gamma"); _req(beta, F32, "beta"); _req(pe, F32, "pe"); _req(lengths, torch.int32, "lengths")
    _req(out_f32, F32, "out_f32")
    m, k = a.shape
    n, k2 = w.shape
    if k2 != k:
        raise RuntimeError(f"gemm_ln: K mismatch {k} vs {k2}")
    if residual is not None and tuple(residual.shape) != (m, n):
        raise RuntimeError(f"gemm_ln: residual shape {tuple(residual.shape)} != {(m, n)}")
    if out_f32 is not None and tuple(out_f32.shape) != (m, n):
        raise RuntimeError(f"gemm_ln: out_f32 shape {tuple(out_f32.shape)} != {(m, n)}")
    o32 = out_f32 if out_f32 is not None else (torch.empty((m, n), dtype=F32, device=a.device) if want_f32 else None)
    o16 = torch.empty((m, n), dtype=enc16_dtype(), device=a.device) if want_bf16 else None
    _call("sblk_gemm_ln_fwd", f"gemm+ln K={k}", 2 * m * n * k,
          2 * (m * k + n * k) + m * n * ((4 if residual is not None else 0) + (4 if o32 is not None else 0) +
                                         (2 if want_bf16 else 0)),
          _p(a), _p(w), _p(bias), _p(residual), _p(gamma), _p(beta), _p(pe), _p(lengths), _p(o32), _p(o16), m, n, k, T,
          eps, _stream())
    return o32, o16


def linear_ln(a, w, gamma, beta, bias=None, residual=None, pe=None, lengths=None, T=1, eps=1e-5, want_bf16=True,
              out_f32=None, fused=None):
    """LayerNorm(a @ w.T + bias + residual) * gamma + beta (+ pe) (* pad mask) -> (fp32 [M,512], bf16 [M,512] | None).

    Strategy by token count: when a 128-row tiling already fills the machine the cluster-fused kernel (gemm_ln) does
    it in one launch; at small M (the BASELINE 928 tokens) the GEMM is operand-delivery bound per SM, so it runs
    split-K over all SMs into fp32 partials that the LayerNorm kernel sums (deterministic, no atomics)."""
    _req(a, enc16_dtype(), "a"); _req(w, enc16_dtype(), "w")
    m, k = a.shape
    n = w.shape[0]
    splits = int(_lib.load().sblk_gemm_splitk_plan(m, n, k))
    if splits < 1:
        raise RuntimeError(f"linear_ln: {_lib.last_error()}")
    # fused: None = by token count (below); True / False force the one-launch cluster kernel / the split-K pair
    if fused is True or (fused is None and splits == 1 and (m + 127) // 128 * 4 >= 64):
        return gemm_ln(a, w, gamma, beta, bias=bias, residual=residual, pe=pe, lengths=lengths, T=T, eps=eps,
                       want_bf16=want_bf16, out_f32=out_f32)
    _req(bias, F32, "bias"); _req(residual, F32, "residual"); _req(gamma, F32, "gamma"); _req(beta, F32, "beta")
    _req(pe, F32, "pe"); _req(lengths, torch.int32, "lengths"); _req(out_f32, F32, "out_f32")
    if w.shape[1] != k or n != 512:
        raise RuntimeError(f"linear_ln: weight shape {tuple(w.shape)} does not match K={k}, d_model=512")
    parts = torch.empty((splits, m, n), dtype=F32, device=a.device)
    _call("sblk_gemm_splitk_fwd", f"gemm splitK={splits} N={n} K={k}", 2 * m * n * k,
          2 * (m * k + n * k) + 4 * splits * m * n, _p(a), _p(w), None, _p(parts), m, n, k, splits, _stream())
    o32 = out_f32 if out_f32 is not None else torch.empty((m, n), dtype=F32, device=a.device)
    o16 = torch.empty((m, n), dtype=enc16_dtype(), device=a.device) if want_bf16 else None
    _call("sblk_sum_layernorm_fwd", f"sum{splits}+layernorm", 0,
          m * n * (4 * splits + (4 if residual is not None else 0) + 4 + (2 if want_bf16 else 0)),
          _p(parts), splits, _p(bias), _p(residual), _p(gamma), _p(beta), _p(pe), _p(lengths), _p(o32), _p(o16), m, T, n,
          eps, _stream())
    return o32, o16


def pack_qkv_heads(wq, wk, wv, bq, bk, bv, h, d_k=64):
    """bf16 [h*d_k, K] x3 + fp32 [h*d_k] x3 -> head-major (bf16 [h*3*d_k, K], fp32 [h*3*d_k]) for qkv_attention
    (pure re-indexing of already packed weights; no arithmetic)."""
    for t_, n_ in ((wq, "wq"), (wk, "wk"), (wv, "wv")):
        _req(t_, enc16_dtype(), n_)
    for t_, n_ in ((bq, "bq"), (bk, "bk"), (bv, "bv")):
        _req(t_, F32, n_)
    k = wq.shape[1]
    w = torch.stack([wq.view(h, d_k, k), wk.view(h, d_k, k), wv.view(h, d_k, k)], dim=1).reshape(h * 3 * d_k, k)
    b = torch.stack([bq.view(h, d_k), bk.view(h, d_k), bv.view(h, d_k)], dim=1).reshape(h * 3 * d_k)
    return w.contiguous(), b.contiguous()


def qkv_attention(x, w_heads, b_heads, n, t, h, d_k=64, lengths=None, scale=None):
    """x bf16 [n*t, K] -> heads-concatenated self-attention output bf16 [n*t, h*d_k] (projection + attention fused)."""
    _req(x, enc16_dtype(), "x"); _req(w_heads, enc16_dtype(), "w_heads"); _req(b_heads, F32, "b_heads")
    _req(lengths, torch.int32, "lengths")
    k = x.shape[1]
    if tuple(x.shape) != (n * t, k) or tuple(w_heads.shape) != (h * 3 * d_k, k) or b_heads.numel() != h * 3 * d_k:
        raise RuntimeError(f"qkv_attention: shapes x{tuple(x.shape)} w{tuple(w_heads.shape)} do not match "
                           f"n={n} t={t} h={h} d_k={d_k}")
    out = torch.empty((n * t, h * d_k), dtype=enc16_dtype(), device=x.device)
    if scale is None:
        scale = 1.0 / (d_k ** 0.5)
    _call("sblk_qkv_attention_fwd", f"qkv+attention T={t}", 2 * n * t * 3 * h * d_k * k + 4 * n * h * t * t * d_k,
          2 * (x.numel() + w_heads.numel() + out.numel()),
          _p(x), _p(w_heads), _p(b_heads), _p(lengths), _p(out), n, t, h, d_k, k, scale, _stream())
    return out


def attention(qkv, n, t, h, d_k=64, lengths=None, want_probs=False, scale=None):
    _req(qkv, enc16_dtype(), "qkv"); _req(lengths, torch.int32, "lengths")
    if tuple(qkv.shape) != (n * t, 3 * h * d_k):
        raise RuntimeError(f"attention: qkv shape {tuple(qkv.shape)} != {(n * t, 3 * h * d_k)}")
    out = torch.empty((n * t, h * d_k), dtype=enc16_dtype(), device=qkv.device)
    probs = torch.empty((h * n, t, t), dtype=F32, device=qkv.device) if want_probs else None
    if scale is None:
        scale = 1.0 / (d_k ** 0.5)
    _call("sblk_attention_fwd", f"attention T={t}", 4 * n * h * t * t * d_k, 2 * qkv.numel() + 2 * out.numel(),
          _p(qkv), _p(out), _p(probs), _p(lengths), n, t, h, d_k, scale, _stream())
    return out, probs


def encoder_stack_supported(n_head, d_k, d_v, d_model, d_in, d_inner, t, n_layers):
    """Shapes the one-launch encoder stack (csrc/sblk_encoder_stack.cuh) implements."""
    return (n_head == 8 and d_k == 64 and d_v == 64 and d_model == 512 and 0 < t <= 128 and n_layers >= 1 and
            d_in % 128 == 0 and d_inner % 1024 == 0 and d_inner <= 2048)


def encoder_stack(x16, stk, n, t, lengths=None, scale=0.125, eps=1e-5, out=None, workspace=None, debug_stamps=None,
                  cluster_size=0, resident_counter=None, multicast=True, groups_per_cluster=1):
    """The whole encoder stack in one launch.  x16 bf16 [n*t, d_in]; `stk` = dict of STACKED packed tensors
    (w_in, b_in, g_in, be_in, pe, w_heads, b_heads, w_fc, b_fc, g1, be1, w_1, b_1, w_2, b_2, g2, be2, n_layers, d_inner)
    -> fp32 [n*t, 512]."""
    _req(x16, enc16_dtype(), "x16"); _req(lengths, torch.int32, "lengths"); _req(out, F32, "out")
    for k_ in ("w_in", "w_heads", "w_fc", "w_1", "w_2"):
        _req(stk[k_], enc16_dtype(), k_)
    for k_ in ("b_in", "g_in", "be_in", "pe", "b_heads", "b_fc", "g1", "be1", "b_1", "b_2", "g2", "be2"):
        _req(stk[k_], F32, k_)
    m, d_in = x16.shape
    nl, d_inner = stk["n_layers"], stk["d_inner"]
    if m != n * t:
        raise RuntimeError(f"encoder_stack: {m} rows != n*t = {n * t}")
    if (tuple(stk["w_in"].shape) != (512, d_in) or tuple(stk["w_heads"].shape) != (nl * 1536, 512) or
            tuple(stk["w_fc"].shape) != (nl * 512, 512) or tuple(stk["w_1"].shape) != (nl * d_inner, 512) or
            tuple(stk["w_2"].shape) != (nl * 512, d_inner) or stk["pe"].shape[-1] != 512 or stk["pe"].shape[0] < t):
        raise RuntimeError("encoder_stack: stacked weight shapes do not match the layer configuration")
    if out is None:
        out = torch.empty((m, 512), dtype=F32, device=x16.device)
    elif tuple(out.shape) != (m, 512):
        raise RuntimeError(f"encoder_stack: out shape {tuple(out.shape)} != {(m, 512)}")
    lib = _lib.load()
    need = int(lib.sblk_encoder_stack_workspace_bytes(n, t, d_inner))
    if workspace is None:
        workspace = torch.empty((need,), dtype=torch.uint8, device=x16.device)
    elif workspace.numel() * workspace.element_size() < need or not workspace.is_cuda:
        raise RuntimeError(f"encoder_stack: workspace needs {need} bytes of device memory")
    a = _lib.EncoderStackArgs()
    a.x_in, a.w_in, a.b_in = _p(x16), _p(stk["w_in"]), _p(stk["b_in"])
    a.ln_in_gamma, a.ln_in_beta, a.pe = _p(stk["g_in"]), _p(stk["be_in"]), _p(stk["pe"])
    a.w_heads, a.b_heads, a.w_fc, a.b_fc = _p(stk["w_heads"]), _p(stk["b_heads"]), _p(stk["w_fc"]), _p(stk["b_fc"])
    a.ln1_gamma, a.ln1_beta = _p(stk["g1"]), _p(stk["be1"])
    a.w_1, a.b_1, a.w_2, a.b_2 = _p(stk["w_1"]), _p(stk["b_1"]), _p(stk["w_2"]), _p(stk["b_2"])
    a.ln2_gamma, a.ln2_beta = _p(stk["g2"]), _p(stk["be2"])
    a.lengths, a.out, a.workspace = _p(lengths), _p(out), _p(workspace)
    a.N, a.T, a.n_layers, a.n_head, a.d_k, a.d_model, a.d_in, a.d_inner = n, t, nl, 8, 64, 512, d_in, d_inner
    a.scale, a.eps = scale, eps
    a.cluster_size = int(cluster_size)   # 0 = automatic
    a.debug_stamps = _p(debug_stamps)   # optional int64 [1 + 4*n_layers, 8] device tensor (profiling aid)
    a.resident_counter = _p(resident_counter)   # optional int32 [2] device tensor (co-scheduling gate, see gate_wait)
    a.no_multicast = 0 if multicast else 1
    a.groups_per_cluster = int(groups_per_cluster)   # 2: two clip groups interleaved per cluster (bit-identical)
    flops = 2 * m * 512 * d_in + nl * (2 * m * 512 * (4 * 512 + 2 * d_inner) + 4 * n * 8 * t * t * 64)
    wbytes = 2 * (512 * d_in + nl * (4 * 512 * 512 + 2 * 512 * d_inner))
    _call("sblk_encoder_stack_fwd", f"encoder stack L={nl} T={t} N={n}", flops, wbytes + m * (2 * d_in + 4 * 512),
          ctypes.byref(a), _stream())
    return out
