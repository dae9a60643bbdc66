"""Tensor-level wrappers over the TRAINING entry points of the libsblk C ABI (include/sblk.h, "training path").

Same conventions as ops.py: validate, allocate with torch, enqueue on torch's current stream; no fallback.
Gradients and convolutional activations are bf16, saved encoder activations are enc16 (ops.enc16_dtype()),
parameter gradients / statistics / the encoder's residual-stream gradient are fp32.
"""
from __future__ import annotations

import torch

from . import _lib
from .ops import BF16, F32, _call, _p, _req, _stream, enc16_dtype

_WS = {}


def _workspace(dev, floats):
    """Reusable fp32 scratch for the two-stage reductions (per device; grown on demand; stream-ordered reuse)."""
    key = str(dev)
    ws = _WS.get(key)
    if ws is None or ws.numel() < floats:
        ws = _WS[key] = torch.empty((int(floats),), dtype=F32, device=dev)
    return ws


def _is16(t, name):
    if t is None:
        return
    if not t.is_cuda or t.dtype not in (BF16, torch.float16) or not t.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous CUDA 16-bit float tensor")


def gemm_fmt(a, w, bias=None, residual=None, relu=False, out16=False, out_f32=False, splits=1, fp16=False):
    """a [M,K] x w [N,K]^T with explicit operand format (fp16=False: bf16).  splits > 1 -> fp32 partials [splits,M,N]."""
    dt = torch.float16 if fp16 else BF16
    _req(a, dt, "a"); _req(w, dt, "w"); _req(bias, F32, "bias"); _req(residual, dt, "residual")
    m, k = a.shape
    n, k2 = w.shape
    if k2 != k:
        raise RuntimeError(f"gemm_fmt: K mismatch {k} vs {k2}")
    o16 = torch.empty((m, n), dtype=dt, device=a.device) if out16 else None
    if splits > 1:
        o32 = torch.empty((splits, m, n), dtype=F32, device=a.device)
    else:
        o32 = torch.empty((m, n), dtype=F32, device=a.device) if out_f32 else None
    _call("sblk_gemm_fmt_fwd", f"gemm_fmt N={n} K={k} splits={splits}", 2 * m * n * k, 2 * (m * k + n * k),
          _p(a), _p(w), _p(bias), _p(residual), _p(o16), _p(o32), m, n, k, 1 if relu else 0, int(splits),
          1 if fp16 else 0, _stream())
    return o16, o32


def transpose16(x, ld_out=None, to_bf16=False):
    """16-bit [R, C] -> [C, ld_out] (zero-filled past R).  to_bf16: re-round IEEE fp16 input to bf16."""
    _is16(x, "x")
    r, c = x.shape
    ld_out = r if ld_out is None else int(ld_out)
    convert = 1 if (to_bf16 and x.dtype == torch.float16) else 0
    out = torch.empty((c, ld_out), dtype=BF16 if (convert or x.dtype == BF16) else x.dtype, device=x.device)
    _call("sblk_transpose16", f"transpose16 C={c}", 0, 2 * (r * c + c * ld_out), _p(x), _p(out), r, c, c, ld_out, convert,
          _stream())
    return out


def im2col_t(x, r, s, stride, pad, ld_out):
    """NHWC bf16 [F,H,W,C] -> [r*s*C, ld_out] (K-major B operand of the wgrad GEMM)."""
    _req(x, BF16, "x")
    f, h, w, c = x.shape
    out = torch.empty((r * s * c, int(ld_out)), dtype=BF16, device=x.device)
    _call("sblk_im2col_t", f"im2col_t {r}x{s} C={c}", 0, 2 * (x.numel() + out.numel()), _p(x), _p(out), f, h, w, c, r, s,
          stride, pad, int(ld_out), _stream())
    return out


def stem_im2col(x, transposed=False, ld_out=None):
    """x fp32 [N,T,88,88] (or [N,1,T,88,88]) -> bf16 [M,256] or (transposed) [256, ld_out]."""
    _req(x, F32, "x")
    if x.dim() == 5:
        x = x[:, 0]
    n, t, h, w = x.shape
    if (h, w) != (88, 88):
        raise RuntimeError("stem_im2col: frames must be 88x88")
    m = n * t * 44 * 44
    if transposed:
        ld_out = int(ld_out)
        out = torch.empty((256, ld_out), dtype=BF16, device=x.device)
    else:
        ld_out = 256
        out = torch.empty((m, 256), dtype=BF16, device=x.device)
    _call("sblk_stem_im2col", "stem_im2col", 0, 4 * x.numel() + 2 * out.numel(), _p(x), _p(out), n, t,
          1 if transposed else 0, ld_out, _stream())
    return out


def stem_im2col_u8(x_u8, lut, t_out, crop, flip=None, transposed=False, ld_out=None):
    """Raw uint8 gray frames [N,T_in,H0,W0] -> the stem_im2col of the clip the training loader builds from them (/255,
    ColorNormalize, 88x88 crop, optional horizontal mirror of the crop, zero-padding to `t_out` frames), bit for bit.
    `lut`: bf16 [256] (synth.normalize_lut()).  `crop`: (y1, x1) for every frame, or int32 [N*T_in, 2] per-frame (y1, x1)
    offsets (RandomCrop; a CPU tensor is range-checked here and uploaded, offsets already on the GPU are clamped into the
    frame by the kernel).  `flip`: None or a bool / integer tensor [N], nonzero = mirror that clip."""
    if not torch.is_tensor(x_u8) or not x_u8.is_cuda or x_u8.dtype != torch.uint8 or x_u8.dim() != 4:
        raise RuntimeError("stem_im2col_u8: expected a CUDA uint8 tensor [N,T,H0,W0] (no CPU fallback exists)")
    if not x_u8.is_contiguous():
        raise RuntimeError("stem_im2col_u8: expected a contiguous tensor")
    _req(lut, BF16, "lut")
    if lut.numel() != 256:
        raise RuntimeError("stem_im2col_u8: lut must hold 256 bf16 values")
    n, t_in, h0, w0 = x_u8.shape
    t_out = int(t_out)
    crop_t, cy, cx = None, 0, 0
    if torch.is_tensor(crop):
        crop_t = crop_offsets_to(crop, n * t_in, h0, w0, x_u8.device)
    else:
        cy, cx = int(crop[0]), int(crop[1])
    flip_t = None if flip is None else flip_flags_to(flip, n, x_u8.device)
    m = n * t_out * 44 * 44
    if transposed:
        ld_out = m if ld_out is None else int(ld_out)
        out = torch.empty((256, ld_out), dtype=BF16, device=x_u8.device)
    else:
        ld_out = 256
        out = torch.empty((m, 256), dtype=BF16, device=x_u8.device)
    _call("sblk_stem_im2col_u8", "stem_im2col_u8", 0, x_u8.numel() + 2 * out.numel(), _p(x_u8), _p(lut), _p(crop_t), cy,
          cx, _p(flip_t), _p(out), n, t_in, t_out, h0, w0, 1 if transposed else 0, ld_out, _stream())
    return out


def crop_offsets_to(crop, frames, h0, w0, device):
    """Per-frame crop offsets as the int32 [frames, 2] (y1, x1) CUDA tensor the uint8 stem reads.  Offsets that arrive on
    the CPU must keep the 88x88 crop inside the h0 x w0 frame (RuntimeError otherwise); on the GPU they cannot be read
    without a synchronisation, and the kernel clamps them."""
    if crop.dtype != torch.int32 or tuple(crop.shape) != (frames, 2):
        raise RuntimeError(f"crop: per-frame offsets must be int32 [{frames}, 2], got {crop.dtype} {tuple(crop.shape)}")
    if not crop.is_cuda:
        y, x = crop[:, 0], crop[:, 1]
        bad = (y < 0) | (y > h0 - 88) | (x < 0) | (x > w0 - 88)
        if bool(bad.any()):
            i = int(bad.nonzero()[0, 0])
            raise RuntimeError(f"crop: offset ({int(y[i])}, {int(x[i])}) of frame {i} leaves the {h0}x{w0} frame")
    return crop.to(device=device).contiguous()


def flip_flags_to(flip, n, device):
    """Per-clip mirror flags (bool / integer [n], nonzero = mirror) as the int32 CUDA tensor the uint8 stem reads."""
    if not torch.is_tensor(flip) or flip.dtype.is_floating_point or flip.dtype.is_complex or tuple(flip.shape) != (n,):
        raise RuntimeError(f"flip: expected a bool or integer tensor [{n}], got "
                           f"{flip.dtype if torch.is_tensor(flip) else type(flip).__name__} "
                           f"{tuple(flip.shape) if torch.is_tensor(flip) else ''}")
    return flip.to(device=device, dtype=torch.int32).contiguous()


def colreduce(mode, a, b=None, c=None, mean=None, rstd=None):
    """Deterministic per-channel reductions (see include/sblk.h: sblk_colreduce) -> fp32 [2, C]."""
    if mode == 2:
        _req(a, F32, "a")
    else:
        _is16(a, "a")
    _is16(b, "b"); _is16(c, "c"); _req(mean, F32, "mean"); _req(rstd, F32, "rstd")
    ch = a.shape[-1]
    m = a.numel() // ch
    lib = _lib.load()
    ws = _workspace(a.device, lib.sblk_colreduce_workspace_floats(ch))
    out = torch.empty((2, ch), dtype=F32, device=a.device)
    _call("sblk_colreduce", f"colreduce mode={mode} C={ch}", 0, a.numel() * a.element_size(), int(mode), _p(a), _p(b),
          _p(c), _p(mean), _p(rstd), m, ch, 1 if a.dtype == torch.float16 else 0, _p(ws), _p(out), _stream())
    return out


def bn_finalize(sums, count, eps, momentum, running_mean=None, running_var=None):
    _req(sums, F32, "sums"); _req(running_mean, F32, "running_mean"); _req(running_var, F32, "running_var")
    ch = sums.shape[1]
    mean = torch.empty((ch,), dtype=F32, device=sums.device)
    rstd = torch.empty((ch,), dtype=F32, device=sums.device)
    _call("sblk_bn_finalize", "bn_finalize", 0, 0, _p(sums), _p(mean), _p(rstd), _p(running_mean), _p(running_var), ch,
          float(count), float(eps), float(momentum), _stream())
    return mean, rstd


def bn_apply(x, mean, rstd, gamma, beta, residual=None, relu=True):
    _req(x, BF16, "x"); _req(residual, BF16, "residual")
    for t_, n_ in ((mean, "mean"), (rstd, "rstd"), (gamma, "gamma"), (beta, "beta")):
        _req(t_, F32, n_)
    ch = x.shape[-1]
    m = x.numel() // ch
    out = torch.empty_like(x)
    _call("sblk_bn_apply_fwd", f"bn_apply C={ch}", 0, 2 * x.numel() * (2 + (residual is not None)), _p(x), _p(residual),
          _p(mean), _p(rstd), _p(gamma), _p(beta), _p(out), m, ch, 1 if relu else 0, _stream())
    return out


def bn_bwd(dy, out_act, x, mean, rstd, gamma, sums, want_dres=False):
    _req(dy, BF16, "dy"); _req(out_act, BF16, "out_act"); _req(x, BF16, "x"); _req(sums, F32, "sums")
    ch = x.shape[-1]
    m = x.numel() // ch
    dx = torch.empty_like(x)
    dres = torch.empty_like(x) if want_dres else None
    _call("sblk_bn_bwd", f"bn_bwd C={ch}", 0, 2 * x.numel() * 4, _p(dy), _p(out_act), _p(x), _p(mean), _p(rstd),
          _p(gamma), _p(sums), _p(dx), _p(dres), m, ch, _stream())
    return dx, dres


def maxpool_fwd(x):
    _req(x, BF16, "x")
    f, h, w, c = x.shape
    out = torch.empty((f, (h - 1) // 2 + 1, (w - 1) // 2 + 1, c), dtype=BF16, device=x.device)
    _call("sblk_maxpool3x3s2_fwd", "maxpool fwd", 0, 2 * (x.numel() + out.numel()), _p(x), _p(out), f, h, w, c, _stream())
    return out


def maxpool_bwd(x, pooled, dy):
    """x: the pooled layer's input (a ReLU output), pooled: maxpool_fwd(x), dy: gradient of pooled."""
    _req(x, BF16, "x"); _req(pooled, BF16, "pooled"); _req(dy, BF16, "dy")
    f, h, w, c = x.shape
    if pooled.shape != dy.shape:
        raise RuntimeError("maxpool_bwd: pooled / dy shape mismatch")
    dx = torch.empty_like(x)
    _call("sblk_maxpool3x3s2_bwd", "maxpool bwd", 0, 2 * (2 * x.numel() + 2 * dy.numel()), _p(x), _p(pooled), _p(dy),
          _p(dx), f, h, w, c, _stream())
    return dx


def avgpool_bwd(dfeat, hw):
    _req(dfeat, F32, "dfeat")
    f, c = dfeat.shape
    dx = torch.empty((f, hw, c), dtype=BF16, device=dfeat.device)
    _call("sblk_avgpool_bwd", "avgpool bwd", 0, 4 * dfeat.numel() + 2 * dx.numel(), _p(dfeat), _p(dx), f, hw, c, _stream())
    return dx


def zero_stuff2(dy, h, w):
    _req(dy, BF16, "dy")
    f, p, q, c = dy.shape
    out = torch.empty((f, h, w, c), dtype=BF16, device=dy.device)
    _call("sblk_zero_stuff2", "zero_stuff2", 0, 2 * (dy.numel() + out.numel()), _p(dy), _p(out), f, h, w, c, p, q, _stream())
    return out


def relu_bwd_(dh, h):
    _req(dh, BF16, "dh"); _req(h, enc16_dtype(), "h")
    _call("sblk_relu_bwd", "relu_bwd", 0, 6 * dh.numel(), _p(dh), _p(h), dh.numel(), _stream())
    return dh


def ln_bwd(dy, z, gamma, lengths=None, T=1, eps=1e-5, want_f32=True, want_bf16=True):
    """-> (dz fp32 | None, dz bf16 | None, dgamma [512], dbeta [512])."""
    _req(dy, F32, "dy"); _req(z, F32, "z"); _req(gamma, F32, "gamma"); _req(lengths, torch.int32, "lengths")
    m, d = z.shape
    if d != 512 or tuple(dy.shape) != (m, d):
        raise RuntimeError(f"ln_bwd: expected [M,512] tensors, got {tuple(dy.shape)} / {tuple(z.shape)}")
    lib = _lib.load()
    ws = _workspace(z.device, lib.sblk_ln_bwd_workspace_floats())
    dz32 = torch.empty_like(z) if want_f32 else None
    dz16 = torch.empty((m, d), dtype=BF16, device=z.device) if want_bf16 else None
    dgb = torch.empty((2, 512), dtype=F32, device=z.device)
    _call("sblk_ln_bwd", "ln_bwd", 0, 4 * 3 * m * d, _p(dy), _p(z), _p(gamma), _p(lengths), _p(dz32), _p(dz16), _p(dgb),
          _p(ws), m, T, float(eps), _stream())
    return dz32, dz16, dgb[0], dgb[1]


def _rows(t, name, rows, cols):
    """t: a 2-D CUDA tensor view with unit column stride, >= rows rows and >= cols columns -> its row pitch."""
    if t.dim() != 2 or t.stride(1) != 1 or t.shape[0] < rows or t.shape[1] < cols:
        raise RuntimeError(f"{name}: expected a [>= {rows}, >= {cols}] row-major view, got {tuple(t.shape)} "
                           f"strides {t.stride()}")
    return t.stride(0)


def xattention_train_fwd(q, k, v, n, lq, lk, h, causal=False, drop=None, klens=None, scale=0.125):
    """Training attention with separate sources (include/sblk.h: sblk_xattention_train_fwd).  q [n*lq, >= h*64], k / v
    [n*lk, >= h*64]: enc16 row-major views (column slices of one buffer allowed); drop fp32 [h*n, lq, lk] or None;
    klens int32 [n] or None -> (out enc16 [n*lq, h*64], probs fp32 [h*n, lq, lk])."""
    e16 = enc16_dtype()
    for t_, nm in ((q, "q"), (k, "k"), (v, "v")):
        if not t_.is_cuda or t_.dtype != e16:
            raise RuntimeError(f"{nm}: expected a CUDA {e16} tensor (no CPU fallback exists)")
    _req(drop, F32, "drop"); _req(klens, torch.int32, "klens")
    ldq = _rows(q, "q", n * lq, h * 64)
    ldk, ldv = _rows(k, "k", n * lk, h * 64), _rows(v, "v", n * lk, h * 64)
    if drop is not None and tuple(drop.shape) != (h * n, lq, lk):
        raise RuntimeError(f"xattention_train_fwd: drop shape {tuple(drop.shape)} != {(h * n, lq, lk)}")
    probs = torch.empty((h * n, lq, lk), dtype=F32, device=q.device)
    out = torch.empty((n * lq, h * 64), dtype=e16, device=q.device)
    _call("sblk_xattention_train_fwd", f"xattention train fwd Lq={lq} Lk={lk}", 4 * n * h * lq * lk * 64,
          2 * (n * lq + 2 * n * lk + n * lq) * h * 64 + 4 * probs.numel(), _p(q), _p(k), _p(v), _p(drop), _p(probs),
          _p(out), _p(klens), ldq, ldk, ldv, h * 64, n, lq, lk, h, 1 if causal else 0, float(scale), _stream())
    return out, probs


def xattention_train_bwd(q, k, v, probs, dout, n, lq, lk, h, causal=False, drop=None, klens=None, scale=0.125,
                         dq=None, dk=None, dv=None):
    """Backward of xattention_train_fwd: dout bf16 [n*lq, h*64] -> (dq bf16, dk bf16, dv bf16).  The outputs are
    allocated [n*lq | n*lk, h*64] unless row-major views to write into are given (e.g. the thirds of one dqkv buffer)."""
    e16 = enc16_dtype()
    for t_, nm in ((q, "q"), (k, "k"), (v, "v")):
        if not t_.is_cuda or t_.dtype != e16:
            raise RuntimeError(f"{nm}: expected a CUDA {e16} tensor (no CPU fallback exists)")
    _req(probs, F32, "probs"); _req(dout, BF16, "dout"); _req(drop, F32, "drop"); _req(klens, torch.int32, "klens")
    if tuple(probs.shape) != (h * n, lq, lk) or (drop is not None and tuple(drop.shape) != (h * n, lq, lk)):
        raise RuntimeError(f"xattention_train_bwd: probs / drop must be [{h * n}, {lq}, {lk}]")
    ldq = _rows(q, "q", n * lq, h * 64)
    ldk, ldv = _rows(k, "k", n * lk, h * 64), _rows(v, "v", n * lk, h * 64)
    lddo = _rows(dout, "dout", n * lq, h * 64)
    grads = []
    for g_, rows, nm in ((dq, n * lq, "dq"), (dk, n * lk, "dk"), (dv, n * lk, "dv")):
        if g_ is None:
            g_ = torch.empty((rows, h * 64), dtype=BF16, device=q.device)
        elif not g_.is_cuda or g_.dtype != BF16:
            raise RuntimeError(f"{nm}: expected a CUDA bfloat16 tensor")
        grads.append((g_, _rows(g_, nm, rows, h * 64)))
    (dq, lddq), (dk, lddk), (dv, lddv) = grads
    _call("sblk_xattention_train_bwd", f"xattention train bwd Lq={lq} Lk={lk}", 8 * n * h * lq * lk * 64,
          2 * (2 * n * lq + 2 * n * lk) * h * 64 + 4 * probs.numel(), _p(q), _p(k), _p(v), _p(drop), _p(probs),
          _p(dout), _p(dq), _p(dk), _p(dv), _p(klens), ldq, ldk, ldv, lddo, lddq, lddk, lddv, n, lq, lk, h,
          1 if causal else 0, float(scale), _stream())
    return dq, dk, dv


def attention_train_fwd(qkv, n, t, h, drop=None, lengths=None, scale=0.125):
    e16 = enc16_dtype()
    _req(qkv, e16, "qkv"); _req(drop, F32, "drop"); _req(lengths, torch.int32, "lengths")
    if tuple(qkv.shape) != (n * t, 3 * h * 64):
        raise RuntimeError(f"attention_train_fwd: qkv shape {tuple(qkv.shape)}")
    probs = torch.empty((h * n, t, t), dtype=F32, device=qkv.device)
    out = torch.empty((n * t, h * 64), dtype=e16, device=qkv.device)
    _call("sblk_attention_train_fwd", "attention train fwd", 4 * n * h * t * t * 64, 2 * qkv.numel(), _p(qkv), _p(drop),
          _p(probs), _p(out), _p(lengths), n, t, h, float(scale), _stream())
    return out, probs


def attention_train_bwd(qkv, probs, dout, n, t, h, drop=None, lengths=None, scale=0.125):
    _req(qkv, enc16_dtype(), "qkv"); _req(probs, F32, "probs"); _req(dout, BF16, "dout"); _req(drop, F32, "drop")
    dqkv = torch.empty((n * t, 3 * h * 64), dtype=BF16, device=qkv.device)
    _call("sblk_attention_train_bwd", "attention train bwd", 8 * n * h * t * t * 64, 2 * qkv.numel(), _p(qkv), _p(drop),
          _p(probs), _p(dout), _p(dqkv), _p(lengths), n, t, h, float(scale), _stream())
    return dqkv


def bidir_mix_bwd(g_l2r, g_r2l, n, L):
    """Backward of the bidirectional mixing (include/sblk.h: sblk_bidir_mix_bwd): fp32 [n*L, D] x2 -> (d_l2r, d_r2l)."""
    _req(g_l2r, F32, "g_l2r"); _req(g_r2l, F32, "g_r2l")
    if g_l2r.shape != g_r2l.shape or g_l2r.dim() != 2 or g_l2r.shape[0] != n * L:
        raise RuntimeError(f"bidir_mix_bwd: gradients must both be [{n * L}, D], got {tuple(g_l2r.shape)} / "
                           f"{tuple(g_r2l.shape)}")
    d = g_l2r.shape[1]
    d_l2r, d_r2l = torch.empty_like(g_l2r), torch.empty_like(g_r2l)
    _call("sblk_bidir_mix_bwd", "bidir_mix bwd", 3 * g_l2r.numel(), 16 * g_l2r.numel(), _p(g_l2r), _p(g_r2l), _p(d_l2r),
          _p(d_r2l), n, L, d, _stream())
    return d_l2r, d_r2l


def embed_bwd(tokens, L, dx, vocab, scale=1.0):
    """Embedding gradient (include/sblk.h: sblk_embed_bwd): tokens int64 [n, >= L] (any row pitch, unit column stride),
    dx fp32 [n*L, D] -> fp32 [vocab, D]."""
    if not tokens.is_cuda or tokens.dtype != torch.int64 or tokens.dim() != 2 or tokens.stride(1) != 1:
        raise RuntimeError("embed_bwd: tokens must be a CUDA int64 [n, >= L] tensor with unit column stride")
    _req(dx, F32, "dx")
    n = tokens.shape[0]
    if tokens.shape[1] < L or dx.dim() != 2 or dx.shape[0] != n * L:
        raise RuntimeError(f"embed_bwd: tokens {tuple(tokens.shape)} / dx {tuple(dx.shape)} do not match L={L}")
    d = dx.shape[1]
    demb = torch.empty((int(vocab), d), dtype=F32, device=dx.device)
    _call("sblk_embed_bwd", "embed bwd", dx.numel(), 4 * (dx.numel() + demb.numel()), _p(tokens), tokens.stride(0),
          _p(dx), _p(demb), n * L, L, d, int(vocab), float(scale), _stream())
    return demb
