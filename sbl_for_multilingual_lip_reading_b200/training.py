"""Training mode of the drop-in modules: forward with batch statistics + backward through libsblk.

What the reference does under `model.train()` + `loss.backward()` on the hot path (stage-1 pre-training,
VSR_visual_frontend_pretraining_on_LRW_LRW1000_classify/train.py:107-146; SBL train.py:177-210) is autograd over the
stock nn modules.  Here every block of the path is a `torch.autograd.Function` whose forward AND backward are libsblk
launches (ops / ops_train); autograd only chains the blocks, so parameter gradients become available block by block
(DistributedDataParallel's bucketed NCCL all-reduce overlaps the rest of the backward: the "encoder gradient allreduce"
of BASELINE configs[3]).

  frontend: Conv3d stem as im2col + tcgen05 GEMM -> BatchNorm3d with BATCH statistics (running stats updated like
            nn.BatchNorm: momentum 0.1, unbiased variance) -> ReLU -> 3x3/s2 max-pool -> 8 BasicBlocks (raw tcgen05 convs
            + batch-stat BN + ReLU + residual) -> average pool -> the reference's always-on F.dropout(0.5)
  backward: dgrad of a stride-1 conv = the forward conv kernel with the flipped, transposed filter (stride 2: over the
            zero-stuffed gradient); wgrad = split-K tcgen05 GEMM dY^T x im2col^T; BN / ReLU / pool derivative kernels
  encoder : per layer  QKV GEMM -> training attention (dropout on the probabilities) -> fc GEMM -> dropout -> +residual
            -> LayerNorm -> w_1 GEMM + ReLU -> w_2 GEMM -> dropout -> +residual -> LayerNorm, and the mirror-image backward
  decoder : 16 steps x 2 directions x n_layers of the same blocks plus the decoder-encoder attention over K | V projected
            once per call, embedding, bidirectional mixing and output projection Functions (decoder_forward_train)

Precision: bf16 conv operands / activations / gradients, enc16 encoder activations, fp32 accumulation, statistics,
LayerNorm / softmax math, residual-stream gradients and parameter gradients.  Dropout masks are drawn with
`torch.nn.functional.dropout(ones)` — the same generator, call order and shapes as the reference's nn.Dropout /
F.dropout calls, so a seeded reference run draws the same masks; the mask multiply itself is the only torch arithmetic
on the path (plus fp32 gradient additions where two branches meet).
"""
from __future__ import annotations

import random

import torch
import torch.nn.functional as F

from . import ops
from . import ops_train as ot

BF16 = torch.bfloat16
F32 = torch.float32


# ------------------------------------------------------------------------------------------------------------------
# building blocks (no autograd): raw convs, their dgrad / wgrad, batch-stat BatchNorm
# ------------------------------------------------------------------------------------------------------------------
def _zeros_bias(c, dev):
    return torch.zeros((c,), dtype=F32, device=dev)


def pack_conv_weight(w):
    """fp32 [Co,Ci,R,S] -> bf16 [Co,R,S,Ci] (no BatchNorm fold: training BN runs on batch statistics)."""
    wp, _ = ops.pack_conv2d(w.detach().contiguous())
    return wp


def pack_conv_weight_dgrad(w):
    """fp32 [Co,Ci,R,S] -> bf16 [Ci,R,S,Co] with the taps flipped: the filter of the dgrad conv."""
    wt = w.detach().flip(2, 3).permute(1, 0, 2, 3).contiguous()      # [Ci,Co,R,S] flipped (layout only)
    wp, _ = ops.pack_conv2d(wt)
    return wp


def conv_raw(x, wp, stride):
    """bf16 NHWC conv without bias / activation: the pre-BatchNorm tensor the batch statistics are taken from."""
    return ops.conv2d(x, wp, _zeros_bias(wp.shape[0], x.device), stride=stride, relu=False)


def conv_dgrad(dy, wp_d, stride, in_hw):
    """Gradient w.r.t. the conv input.  dy bf16 [F,P,Q,Co]; wp_d from pack_conv_weight_dgrad; in_hw = (H, W)."""
    if stride == 2:
        dy = ot.zero_stuff2(dy, in_hw[0], in_hw[1])
    return ops.conv2d(dy, wp_d, _zeros_bias(wp_d.shape[0], dy.device), stride=1, relu=False)


def _wgrad_gemm(dy2d, col_t_fn, n_out):
    """dW [Co, K] = dY^T [Co, M] x colT [K, M]^T as a split-K tcgen05 GEMM; col_t_fn(ld) builds colT with row pitch ld."""
    m, co = dy2d.shape
    tiles = -(-co // 128) * max(1, n_out // 128)
    splits = max(1, min(32, 148 // tiles))
    kb = -(-m // 64)
    splits = max(1, min(splits, kb // 4)) if kb >= 8 else 1
    ld = -(-m // (64 * splits)) * 64 * splits
    dy_t = ot.transpose16(dy2d, ld_out=ld)
    col_t = col_t_fn(ld)
    _, parts = ot.gemm_fmt(dy_t, col_t, out_f32=True, splits=splits)
    return parts.sum(0) if splits > 1 else parts


def conv_wgrad(x, dy, r, stride):
    """fp32 [Co,Ci,r,r] weight gradient of conv(x, w, stride) given dy (pad = r // 2)."""
    f, h, w_, ci = x.shape
    co = dy.shape[-1]
    pad = r // 2
    dw = _wgrad_gemm(dy.reshape(-1, co), lambda ld: ot.im2col_t(x, r, r, stride, pad, ld), r * r * ci)
    # ([Co,Ci*r*r] round trip: canonical strides even for 1x1 filters, as DDP's gradient buckets expect)
    return dw.view(co, r, r, ci).permute(0, 3, 1, 2).reshape(co, ci * r * r).contiguous().view(co, ci, r, r)


class _BNState:
    __slots__ = ("mean", "rstd")


def bn_forward_train(raw, bn, residual=None, relu=True):
    """Batch-statistics BatchNorm (+ residual) (+ ReLU) of raw bf16 [.., C]; updates bn's running stats like nn.BatchNorm."""
    c = raw.shape[-1]
    count = raw.numel() // c
    sums = ot.colreduce(0, raw)
    momentum = 0.1 if bn.momentum is None else bn.momentum
    track = bn.track_running_stats and bn.running_mean is not None
    mean, rstd = ot.bn_finalize(sums, count, bn.eps, momentum, bn.running_mean if track else None,
                                bn.running_var if track else None)
    if track and bn.num_batches_tracked is not None:
        bn.num_batches_tracked += 1
    out = ot.bn_apply(raw, mean, rstd, bn.weight.detach(), bn.bias.detach(), residual=residual, relu=relu)
    st = _BNState()
    st.mean, st.rstd = mean, rstd
    return out, st


def bn_backward_train(dy, out_act, raw, st, gamma, want_dres=False):
    """-> (d_raw bf16, dgamma fp32, dbeta fp32, d_residual bf16 | None); out_act = the block output (ReLU mask) or None."""
    sums = ot.colreduce(1, dy, out_act, raw, st.mean, st.rstd)
    dx, dres = ot.bn_bwd(dy, out_act, raw, st.mean, st.rstd, gamma.detach(), sums, want_dres=want_dres)
    return dx, sums[1].clone(), sums[0].clone(), dres


def _add16(a, b):
    return (a.float() + b.float()).to(BF16)


# ------------------------------------------------------------------------------------------------------------------
# frontend Functions
# ------------------------------------------------------------------------------------------------------------------
class StemSource:
    """What StemFn reads its clip from: the fp32 clip `x` [N,T,88,88] (lut None), or the loader's raw uint8 frames `x`
    [N,T_in,H0,W0] with the normalisation table, the crop ((y1, x1) or int32 CUDA [N*T_in, 2]), the per-clip flip
    (int32 CUDA [N] or None) and the padded frame count `t` (ops_train.stem_im2col_u8).  The forward and the wgrad of
    the backward both build their im2col from it, so a uint8 source keeps no fp32 clip alive between them."""
    __slots__ = ("x", "lut", "crop", "flip", "t")

    def __init__(self, x, lut=None, crop=None, flip=None, t=None):
        self.x, self.lut, self.crop, self.flip = x, lut, crop, flip
        self.t = x.shape[1] if t is None else int(t)

    @classmethod
    def clip(cls, x):
        x = x.detach()
        return cls((x[:, 0] if x.dim() == 5 else x).contiguous().float())

    def im2col(self, transposed=False, ld_out=None):
        if self.lut is None:
            return ot.stem_im2col(self.x, transposed=transposed, ld_out=ld_out)
        return ot.stem_im2col_u8(self.x, self.lut, self.t, self.crop, self.flip, transposed=transposed, ld_out=ld_out)


class StemFn(torch.autograd.Function):
    """frontend3D in training mode (video_frontend.py:99-104): Conv3d -> BatchNorm3d(batch stats) -> ReLU -> MaxPool3d,
    output bf16 NHWC [N*T, 22, 22, 64] (the reference's transpose(1,2).contiguous().view, :113-115, is the layout).
    `src`: a StemSource, or the fp32 clip itself."""

    @staticmethod
    def forward(ctx, src, w, gamma, beta, bn):
        if not isinstance(src, StemSource):
            src = StemSource.clip(src)
        n, t = src.x.shape[0], src.t
        col = src.im2col()
        w2d = torch.zeros((64, 256), dtype=F32, device=w.device)
        w2d[:, :245] = w.detach().reshape(64, 245)
        wp = ops.cast_bf16(w2d)
        raw, _ = ot.gemm_fmt(col, wp, out16=True)
        del col
        act, st = bn_forward_train(raw, bn, relu=True)                    # [M, 64] = [F,44,44,64]
        act4 = act.view(n * t, 44, 44, 64)
        out = ot.maxpool_fwd(act4)
        crop = src.crop if torch.is_tensor(src.crop) else None
        ctx.save_for_backward(src.x, src.lut, crop, src.flip, raw, act4, gamma, out)
        ctx.st = st
        ctx.t, ctx.crop = src.t, (src.crop if crop is None else None)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, lut, crop, flip, raw, act4, gamma, pooled = ctx.saved_tensors
        src = StemSource(x, lut, ctx.crop if crop is None else crop, flip, ctx.t)
        dact = ot.maxpool_bwd(act4, pooled, dout.contiguous())
        draw, dgamma, dbeta, _ = bn_backward_train(dact.view(-1, 64), act4.view(-1, 64), raw, ctx.st, gamma)
        dw = _wgrad_gemm(draw, lambda ld: src.im2col(transposed=True, ld_out=ld), 256)
        dw = dw[:, :245].reshape(64, 1, 5, 7, 7).contiguous()
        return None, dw, dgamma, dbeta, None


class BasicBlockFn(torch.autograd.Function):
    """BasicBlock.forward in training mode (video_frontend.py:28-41, downsample :68-72) on bf16 NHWC activations."""

    @staticmethod
    def forward(ctx, x, w1, g1, b1, w2, g2, b2, wd, gd, bd, blk):
        x = x.detach().contiguous()
        stride = blk.stride
        raw1 = conv_raw(x, pack_conv_weight(w1), stride)
        a1, st1 = bn_forward_train(raw1, blk.bn1, relu=True)
        raw2 = conv_raw(a1, pack_conv_weight(w2), 1)
        if wd is not None:
            rawd = conv_raw(x, pack_conv_weight(wd), stride)
            res, std = bn_forward_train(rawd, blk.downsample[1], relu=False)
        else:
            rawd, std, res = None, None, x
        out, st2 = bn_forward_train(raw2, blk.bn2, residual=res, relu=True)
        ctx.save_for_backward(x, raw1, a1, raw2, out, rawd, w1, w2, wd, g1, g2, gd)
        ctx.st = (st1, st2, std)
        ctx.stride = stride
        return out

    @staticmethod
    def backward(ctx, dout):
        x, raw1, a1, raw2, out, rawd, w1, w2, wd, g1, g2, gd = ctx.saved_tensors
        st1, st2, std = ctx.st
        stride = ctx.stride
        dout = dout.contiguous()
        # out = relu(bn2(conv2(a1)) + res)
        draw2, dg2, db2, dres = bn_backward_train(dout, out, raw2, st2, g2, want_dres=True)
        dw2 = conv_wgrad(a1, draw2, 3, 1)
        da1 = conv_dgrad(draw2, pack_conv_weight_dgrad(w2), 1, a1.shape[1:3])
        # a1 = relu(bn1(conv1(x)))
        draw1, dg1, db1, _ = bn_backward_train(da1, a1, raw1, st1, g1)
        dw1 = conv_wgrad(x, draw1, 3, stride)
        dx = conv_dgrad(draw1, pack_conv_weight_dgrad(w1), stride, x.shape[1:3])
        if wd is not None:
            drawd, dgd, dbd, _ = bn_backward_train(dres, None, rawd, std, gd)
            dwd = conv_wgrad(x, drawd, 1, stride)
            dx = _add16(dx, conv_dgrad(drawd, pack_conv_weight_dgrad(wd), stride, x.shape[1:3]))
        else:
            dwd = dgd = dbd = None
            dx = _add16(dx, dres)
        return dx, dw1, dg1, db1, dw2, dg2, db2, dwd, dgd, dbd, None


class AvgPoolFn(torch.autograd.Function):
    """AdaptiveAvgPool2d(1) + view (video_frontend.py:87-88): bf16 NHWC [F,H,W,C] -> fp32 [F,C]."""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = tuple(x.shape)
        feat, _ = ops.avgpool(x.detach().contiguous())
        return feat

    @staticmethod
    def backward(ctx, dfeat):
        f, h, w, c = ctx.shape
        return ot.avgpool_bwd(dfeat.contiguous().float(), h * w).view(f, h, w, c)


def frontend_forward_train(fe, x):
    """Lipreading._frontend_forward in training mode -> fp32 features [N*T, 512] (autograd-connected).  `x`: the fp32
    clip [N,1,T,88,88] or a StemSource (the loader's raw uint8 frames)."""
    conv, bn = fe.frontend3D[0], fe.frontend3D[1]
    a = StemFn.apply(x, conv.weight, bn.weight, bn.bias, bn)
    for layer in (fe.resnet18.layer1, fe.resnet18.layer2, fe.resnet18.layer3, fe.resnet18.layer4):
        for blk in layer:
            if blk.downsample is not None:
                ds = (blk.downsample[0].weight, blk.downsample[1].weight, blk.downsample[1].bias)
            else:
                ds = (None, None, None)
            a = BasicBlockFn.apply(a, blk.conv1.weight, blk.bn1.weight, blk.bn1.bias, blk.conv2.weight, blk.bn2.weight,
                                   blk.bn2.bias, ds[0], ds[1], ds[2], blk)
    return AvgPoolFn.apply(a)


# ------------------------------------------------------------------------------------------------------------------
# encoder Functions
# ------------------------------------------------------------------------------------------------------------------
def _lin_bwd(dy16, dy32, x16, w, bias=True):
    """Linear backward: dy16 bf16 [M,out] (GEMM operand), dy32 fp32 or None (bias gradient source), x16 saved enc16
    input [M,in], w fp32 [out,in]  ->  (dW fp32 [out,in], db fp32 [out] | None when bias=False)."""
    m, n_out = dy16.shape
    kb = -(-m // 64)
    splits = 1
    for s_ in (8, 4, 2):
        if kb >= 4 * s_:
            splits = s_
            break
    ld = -(-m // (64 * splits)) * 64 * splits
    dy_t = ot.transpose16(dy16, ld_out=ld)
    x_t = ot.transpose16(x16, ld_out=ld, to_bf16=True)
    _, parts = ot.gemm_fmt(dy_t, x_t, out_f32=True, splits=splits)
    dw = parts.sum(0) if splits > 1 else parts
    if not bias:
        return dw, None
    db = ot.colreduce(2, dy32)[0].clone() if dy32 is not None else ot.colreduce(4, dy16)[0].clone()
    return dw, db


def _lin_dgrad(dy16, w, out_f32=True):
    """dx = dy W: dy16 bf16 [M,out], w fp32 [out,in] -> fp32 (or bf16) [M,in]."""
    wt = ops.cast_bf16(w.detach().t().contiguous())                   # [in, out] = the K-major B operand
    o16, o32 = ot.gemm_fmt(dy16, wt, out16=not out_f32, out_f32=out_f32)
    return o32 if out_f32 else o16


def _e16(w):
    return ops.cast_enc16(w.detach().contiguous())


# Blocks shared by the encoder and decoder layers: every block ends in  out = LayerNorm(dropout(y) + x)  with the fp32
# pre-normalisation sum z saved for the backward.
def _drop_res_ln(y, d, x, g, be, lengths, t, eps, want16=True):
    """-> (out fp32, out enc16 | None, z fp32) of LayerNorm(y * d + x) (d None: no dropout)."""
    if d is not None:
        y = y * d
    z = y + x
    out, out16 = ops.add_layernorm(z, g.detach(), be.detach(), lengths=lengths, T=t, eps=eps, want_bf16=want16)
    return out, out16, z


def _ln_drop_bwd(dout, z, g, d, lengths, t, eps):
    """Backward of _drop_res_ln -> (dz fp32 = the residual's gradient, dy fp32, dy bf16, dgamma, dbeta)."""
    dz32, dz16, dg, dbe = ot.ln_bwd(dout, z, g.detach(), lengths=lengths, T=t, eps=eps)
    if d is None:
        return dz32, dz32, dz16, dg, dbe
    dy32 = dz32 * d
    return dz32, dy32, ops.cast_bf16(dy32), dg, dbe


def _ffn_fwd(x, x16, w1, b1, w2, b2, g, be, d, lengths, t, eps, want16):
    """PositionwiseFeedForward (module.py:47-52) -> (out fp32, out enc16 | None, saved (h16, z))."""
    h16, _ = ops.gemm(x16, _e16(w1), bias=b1.detach(), relu=True, out_bf16=True)
    _, y = ops.gemm(h16, _e16(w2), bias=b2.detach(), out_f32=True)
    out, out16, z = _drop_res_ln(y, d, x, g, be, lengths, t, eps, want16)
    return out, out16, (h16, z)


def _ffn_bwd(dout, x16, saved, w1, w2, g, d, lengths, t, eps):
    """-> (dx fp32, dw1, db1, dw2, db2, dgamma, dbeta)."""
    h16, z = saved
    dz32, dy32, dy16, dg, dbe = _ln_drop_bwd(dout, z, g, d, lengths, t, eps)
    dw2, db2 = _lin_bwd(dy16, dy32, h16, w2)
    dh = _lin_dgrad(dy16, w2, out_f32=False)
    ot.relu_bwd_(dh, h16)
    dw1, db1 = _lin_bwd(dh, None, x16, w1)
    return dz32 + _lin_dgrad(dh, w1), dw1, db1, dw2, db2, dg, dbe


def _self_attn_fwd(x, x16, wq, bq, wk, bk, wv, bv, wfc, bfc, g, be, d_attn, d_fc, lengths, n, t, h, scale, eps,
                   causal=None):
    """MultiHeadAttention as self-attention (attention.py:32-60) on [n*t, 512] rows -> (out fp32, out enc16,
    saved (qkv16, probs, att16, z)).  causal None: the encoder's packed kernel pair (sblk_attention_train_*);
    True / False: the separate-source pair (sblk_xattention_train_*) with / without the subsequent mask."""
    hd = wq.shape[0]
    wqkv = ops.cast_enc16(torch.cat([wq.detach(), wk.detach(), wv.detach()], 0).contiguous())
    bqkv = torch.cat([bq.detach(), bk.detach(), bv.detach()]).contiguous()
    qkv16, _ = ops.gemm(x16, wqkv, bias=bqkv, out_bf16=True)
    if causal is None:
        att16, probs = ot.attention_train_fwd(qkv16, n, t, h, drop=d_attn, lengths=lengths, scale=scale)
    else:
        att16, probs = ot.xattention_train_fwd(qkv16[:, :hd], qkv16[:, hd:2 * hd], qkv16[:, 2 * hd:], n, t, t, h,
                                               causal=causal, drop=d_attn, klens=lengths, scale=scale)
    _, y = ops.gemm(att16, _e16(wfc), bias=bfc.detach(), out_f32=True)
    out, out16, z = _drop_res_ln(y, d_fc, x, g, be, lengths, t, eps)
    return out, out16, (qkv16, probs, att16, z)


def _self_attn_bwd(dout, x16, saved, wq, wk, wv, wfc, g, d_attn, d_fc, lengths, n, t, h, scale, eps, causal=None):
    """-> (dx fp32, dwq, dbq, dwk, dbk, dwv, dbv, dwfc, dbfc, dgamma, dbeta)."""
    qkv16, probs, att16, z = saved
    hd = wq.shape[0]
    dz32, dy32, dy16, dg, dbe = _ln_drop_bwd(dout, z, g, d_fc, lengths, t, eps)
    dwfc, dbfc = _lin_bwd(dy16, dy32, att16, wfc)
    datt = _lin_dgrad(dy16, wfc, out_f32=False)
    if causal is None:
        dqkv = ot.attention_train_bwd(qkv16, probs, datt, n, t, h, drop=d_attn, lengths=lengths, scale=scale)
    else:
        dqkv = torch.empty((n * t, 3 * hd), dtype=BF16, device=x16.device)
        ot.xattention_train_bwd(qkv16[:, :hd], qkv16[:, hd:2 * hd], qkv16[:, 2 * hd:], probs, datt, n, t, t, h,
                                causal=causal, drop=d_attn, klens=lengths, scale=scale, dq=dqkv[:, :hd],
                                dk=dqkv[:, hd:2 * hd], dv=dqkv[:, 2 * hd:])
    wqkv = torch.cat([wq.detach(), wk.detach(), wv.detach()], 0)
    dwqkv, dbqkv = _lin_bwd(dqkv, None, x16, wqkv)
    dx = dz32 + _lin_dgrad(dqkv, wqkv)
    return (dx, dwqkv[:hd].contiguous(), dbqkv[:hd].contiguous(), dwqkv[hd:2 * hd].contiguous(),
            dbqkv[hd:2 * hd].contiguous(), dwqkv[2 * hd:].contiguous(), dbqkv[2 * hd:].contiguous(), dwfc, dbfc, dg, dbe)


class EncoderInFn(torch.autograd.Function):
    """LayerNorm(linear_in(x)) + positional encoding (encoder.py:53-55, before the dropout)."""

    @staticmethod
    def forward(ctx, x, w, b, g, be, pe, t, eps):
        x = x.detach().contiguous().float()
        x16 = ops.cast_enc16(x)
        _, z = ops.gemm(x16, ops.cast_enc16(w.detach().contiguous()), bias=b.detach(), out_f32=True)
        out, _ = ops.add_layernorm(z, g.detach(), be.detach(), pe=pe, T=t, eps=eps, want_bf16=False)
        ctx.save_for_backward(x16, z, w, g)
        ctx.t, ctx.eps = t, eps
        return out

    @staticmethod
    def backward(ctx, dout):
        x16, z, w, g = ctx.saved_tensors
        dz32, dz16, dg, dbe = ot.ln_bwd(dout.contiguous().float(), z, g.detach(), T=ctx.t, eps=ctx.eps)
        dw, db = _lin_bwd(dz16, dz32, x16, w)
        dx = _lin_dgrad(dz16, w) if ctx.needs_input_grad[0] else None
        return dx, dw, db, dg, dbe, None, None, None


class EncoderLayerFn(torch.autograd.Function):
    """EncoderLayer.forward in training mode (encoder.py:83-91; attention.py:32-60,72-83; module.py:47-52).
    drops = (attention-probability, fc-output, ffn-output) dropout factors mask / (1 - p), or None each."""

    @staticmethod
    def forward(ctx, x, wq, bq, wk, bk, wv, bv, wfc, bfc, g1, be1, w1, b1, w2, b2, g2, be2, drops, lengths, n, t, h, scale,
                eps):
        x = x.detach().contiguous()
        d_attn, d_fc, d_ffn = drops
        x16 = ops.cast_enc16(x)
        x1, x1_16, sa = _self_attn_fwd(x, x16, wq, bq, wk, bk, wv, bv, wfc, bfc, g1, be1, d_attn, d_fc, lengths, n, t, h,
                                       scale, eps)
        out, _, ff = _ffn_fwd(x1, x1_16, w1, b1, w2, b2, g2, be2, d_ffn, lengths, t, eps, want16=False)
        ctx.save_for_backward(x16, *sa, x1_16, *ff, wq, wk, wv, wfc, w1, w2, g1, g2)
        ctx.misc = (drops, lengths, n, t, h, scale, eps)
        return out

    @staticmethod
    def backward(ctx, dout):
        x16, qkv16, probs, att16, z1, x1_16, h16, z2, wq, wk, wv, wfc, w1, w2, g1, g2 = ctx.saved_tensors
        (d_attn, d_fc, d_ffn), lengths, n, t, h, scale, eps = ctx.misc
        dx1, dw1, db1, dw2, db2, dg2, dbe2 = _ffn_bwd(dout.contiguous().float(), x1_16, (h16, z2), w1, w2, g2, d_ffn,
                                                      lengths, t, eps)
        dx, dwq, dbq, dwk, dbk, dwv, dbv, dwfc, dbfc, dg1, dbe1 = _self_attn_bwd(
            dx1, x16, (qkv16, probs, att16, z1), wq, wk, wv, wfc, g1, d_attn, d_fc, lengths, n, t, h, scale, eps)
        return (dx, dwq, dbq, dwk, dbk, dwv, dbv, dwfc, dbfc, dg1, dbe1, dw1, db1, dw2, db2, dg2, dbe2, None, None, None,
                None, None, None, None)


def _drop_factor(shape, p, dev, training):
    """mask / (1 - p) as nn.Dropout would apply it (same generator and shape as the reference's call), or None."""
    if not training or p <= 0.0:
        return None
    return F.dropout(torch.ones(shape, dtype=F32, device=dev), p=p, training=True)


def encoder_forward_train(enc, padded_input, lens):
    """Encoder.forward in training mode (encoder.py:36-67) -> (enc_output fp32 [N,T,512],), autograd-connected."""
    n, t, d_in = padded_input.shape
    m = n * t
    dev = padded_input.device
    p = float(enc.dropout_rate)
    lengths = None
    if any(v < t for v in lens):
        lengths = torch.tensor(lens, dtype=torch.int32, device=dev)
    x = padded_input.reshape(m, d_in)
    pe = enc.positional_encoding.pe[0]
    y = EncoderInFn.apply(x, enc.linear_in.weight, enc.linear_in.bias, enc.layer_norm_in.weight, enc.layer_norm_in.bias, pe,
                          t, enc.layer_norm_in.eps)
    y = enc.dropout(y.view(n, t, -1)).reshape(m, -1)           # nn.Dropout: torch autograd, reference mask order
    h = enc.n_head
    for lyr in enc.layer_stack:
        a, f = lyr.slf_attn, lyr.pos_ffn
        # the reference draws: attention-probability dropout (attention.py:79), fc dropout (:57), ffn dropout (module.py:50)
        drops = (_drop_factor((h * n, t, t), p, dev, enc.training), _drop_factor((n, t, enc.d_model), p, dev, enc.training),
                 _drop_factor((n, t, enc.d_model), p, dev, enc.training))
        drops = tuple(None if d is None else d.reshape(-1, d.shape[-1]) if d.dim() == 3 and d.shape[-1] == enc.d_model
                      else d for d in drops)
        y = EncoderLayerFn.apply(y, a.w_qs.weight, a.w_qs.bias, a.w_ks.weight, a.w_ks.bias, a.w_vs.weight, a.w_vs.bias,
                                 a.fc.weight, a.fc.bias, a.layer_norm.weight, a.layer_norm.bias, f.w_1.weight, f.w_1.bias,
                                 f.w_2.weight, f.w_2.bias, f.layer_norm.weight, f.layer_norm.bias, drops, lengths, n, t, h,
                                 1.0 / a.temperature, a.layer_norm.eps)
    return (y.view(n, t, enc.d_model),)


# ------------------------------------------------------------------------------------------------------------------
# decoder Functions (the SBL bidirectional decoder, decoder.py; DESIGN.md §9 "training")
# ------------------------------------------------------------------------------------------------------------------
class EncoderKVFn(torch.autograd.Function):
    """K | V projections of the encoder outputs for one decoder layer's enc_attn, computed once per call and read by all
    16 steps.  Returns (kv fp32 [n*t, 2*hd], kv enc16): the fp32 tensor carries the gradient (autograd sums the 16
    steps' contributions in fp32), the enc16 copy is the attention kernel's operand."""

    @staticmethod
    def forward(ctx, enc, enc16, wk, bk, wv, bv):
        wkv = torch.cat([wk.detach(), wv.detach()], 0)
        kv16, kv32 = ops.gemm(enc16, ops.cast_enc16(wkv.contiguous()), bias=torch.cat([bk.detach(), bv.detach()]),
                              out_bf16=True, out_f32=True)
        ctx.mark_non_differentiable(kv16)
        ctx.save_for_backward(enc16, wk, wv)
        return kv32, kv16

    @staticmethod
    def backward(ctx, dkv, _):
        enc16, wk, wv = ctx.saved_tensors
        hd = wk.shape[0]
        wkv = torch.cat([wk.detach(), wv.detach()], 0)
        dkv = dkv.contiguous()
        dkv16 = ops.cast_bf16(dkv)
        dw, db = _lin_bwd(dkv16, dkv, enc16, wkv)
        denc = _lin_dgrad(dkv16, wkv) if ctx.needs_input_grad[0] else None
        return denc, None, dw[:hd].contiguous(), db[:hd].contiguous(), dw[hd:].contiguous(), db[hd:].contiguous()


class DecoderEmbedFn(torch.autograd.Function):
    """tgt_word_emb(ys[:, :L]) * scale + positional encoding (decoder.py:323-327) -> (x fp32 [n*L, 512], x enc16)."""

    @staticmethod
    def forward(ctx, emb, ys, L, pe, scale):
        n = ys.shape[0]
        e = emb.detach().float().contiguous()
        x32 = torch.empty((n * L, e.shape[1]), dtype=F32, device=e.device)
        x16 = torch.empty((n * L, e.shape[1]), dtype=ops.enc16_dtype(), device=e.device)
        ops._call("sblk_embed_pe_fwd", "embed_pe", 0, 6 * x32.numel(), ys.data_ptr(), ys.stride(0), e.data_ptr(),
                  pe.data_ptr(), x32.data_ptr(), x16.data_ptr(), n * L, L, e.shape[1], e.shape[0], float(scale),
                  ops._stream())
        ctx.mark_non_differentiable(x16)
        # the token buffer itself, not a copy: the decode loop only writes columns >= L after this step
        ctx.ys, ctx.L, ctx.vocab, ctx.scale = ys, L, e.shape[0], scale
        return x32, x16

    @staticmethod
    def backward(ctx, dx, _):
        return ot.embed_bwd(ctx.ys, ctx.L, dx.contiguous(), ctx.vocab, ctx.scale), None, None, None, None


class BidirMixFn(torch.autograd.Function):
    """The synchronous bidirectional mixing (decoder.py:336-346,358-362) -> (l2r' fp32, r2l' fp32, l2r' enc16,
    r2l' enc16)."""

    @staticmethod
    def forward(ctx, l2r, r2l, n, L):
        a32, b32 = torch.empty_like(l2r), torch.empty_like(r2l)
        a16 = torch.empty(l2r.shape, dtype=ops.enc16_dtype(), device=l2r.device)
        b16 = torch.empty_like(a16)
        ops._call("sblk_bidir_mix_fwd", "bidir_mix", 3 * l2r.numel(), 20 * l2r.numel(), l2r.data_ptr(), r2l.data_ptr(),
                  a32.data_ptr(), b32.data_ptr(), a16.data_ptr(), b16.data_ptr(), n, L, l2r.shape[1], ops._stream())
        ctx.mark_non_differentiable(a16, b16)
        ctx.n, ctx.L = n, L
        return a32, b32, a16, b16

    @staticmethod
    def backward(ctx, ga, gb, _a, _b):
        d_l2r, d_r2l = ot.bidir_mix_bwd(ga.contiguous(), gb.contiguous(), ctx.n, ctx.L)
        return d_l2r, d_r2l, None, None


class DecoderLayerFn(torch.autograd.Function):
    """DecoderLayer.forward in training mode (decoder.py:396-408): self-attention over the prefix (subsequent mask when
    `causal`), attention over the encoder's K | V (kv fp32 / kv16 from EncoderKVFn, no mask), FFN.  x fp32 [n*L, 512],
    x16 its enc16 copy or None.  drops = (self-attention probabilities, self fc output, enc-attention probabilities,
    enc fc output, ffn output) factors mask / (1 - p), or None each.  -> (out fp32, out enc16)."""

    @staticmethod
    def forward(ctx, x, x16, kv, kv16, wq, bq, wk, bk, wv, bv, wfc, bfc, g1, be1, wq2, bq2, wfc2, bfc2, g2, be2, w1, b1,
                w2, b2, g3, be3, drops, n, L, t_enc, h, causal, scale1, scale2, eps):
        x = x.detach().contiguous()
        x16 = ops.cast_enc16(x) if x16 is None else x16
        hd = wq2.shape[0]
        d_a1, d_f1, d_a2, d_f2, d_ffn = drops
        x1, x1_16, sa = _self_attn_fwd(x, x16, wq, bq, wk, bk, wv, bv, wfc, bfc, g1, be1, d_a1, d_f1, None, n, L, h,
                                       scale1, eps[0], causal=bool(causal))
        q16, _ = ops.gemm(x1_16, _e16(wq2), bias=bq2.detach(), out_bf16=True)
        att2, probs2 = ot.xattention_train_fwd(q16, kv16[:, :hd], kv16[:, hd:], n, L, t_enc, h, drop=d_a2,
                                               scale=scale2)
        _, y2 = ops.gemm(att2, _e16(wfc2), bias=bfc2.detach(), out_f32=True)
        x2, x2_16, z2 = _drop_res_ln(y2, d_f2, x1, g2, be2, None, L, eps[1])
        out, out16, ff = _ffn_fwd(x2, x2_16, w1, b1, w2, b2, g3, be3, d_ffn, None, L, eps[2], want16=True)
        ctx.mark_non_differentiable(out16)
        ctx.save_for_backward(x16, *sa, x1_16, q16, kv16, probs2, att2, z2, x2_16, *ff, wq, wk, wv, wfc, wq2, wfc2, w1,
                              w2, g1, g2, g3)
        ctx.misc = (drops, n, L, t_enc, h, causal, scale1, scale2, eps)
        return out, out16

    @staticmethod
    def backward(ctx, dout, _):
        (x16, qkv16, probs1, att1, z1, x1_16, q16, kv16, probs2, att2, z2, x2_16, h16, z3, wq, wk, wv, wfc, wq2, wfc2, w1,
         w2, g1, g2, g3) = ctx.saved_tensors
        (d_a1, d_f1, d_a2, d_f2, d_ffn), n, L, t_enc, h, causal, scale1, scale2, eps = ctx.misc
        hd = wq2.shape[0]
        dx2, dw1, db1, dw2, db2, dg3, dbe3 = _ffn_bwd(dout.contiguous().float(), x2_16, (h16, z3), w1, w2, g3, d_ffn,
                                                      None, L, eps[2])
        # x2 = LN(dropout(fc2(attention(q(x1), K, V))) + x1)
        dz2, dy32, dy16, dg2, dbe2 = _ln_drop_bwd(dx2, z2, g2, d_f2, None, L, eps[1])
        dwfc2, dbfc2 = _lin_bwd(dy16, dy32, att2, wfc2)
        datt2 = _lin_dgrad(dy16, wfc2, out_f32=False)
        dkv = torch.empty((n * t_enc, 2 * hd), dtype=BF16, device=x16.device)
        dq2, _, _ = ot.xattention_train_bwd(q16, kv16[:, :hd], kv16[:, hd:], probs2, datt2, n, L, t_enc, h, drop=d_a2,
                                            scale=scale2, dk=dkv[:, :hd], dv=dkv[:, hd:])
        dwq2, dbq2 = _lin_bwd(dq2, None, x1_16, wq2)
        dx1 = dz2 + _lin_dgrad(dq2, wq2)
        dx, dwq, dbq, dwk, dbk, dwv, dbv, dwfc, dbfc, dg1, dbe1 = _self_attn_bwd(
            dx1, x16, (qkv16, probs1, att1, z1), wq, wk, wv, wfc, g1, d_a1, d_f1, None, n, L, h, scale1, eps[0],
            causal=bool(causal))
        return (dx, None, dkv.float(), None, dwq, dbq, dwk, dbk, dwv, dbv, dwfc, dbfc, dg1, dbe1, dwq2, dbq2, dwfc2, dbfc2,
                dg2, dbe2, dw1, db1, dw2, db2, dg3, dbe3) + (None,) * 9


class DecoderProjFn(torch.autograd.Function):
    """tgt_word_prj(dec_output[:, -1]) (decoder.py:364-365): the last position's enc16 row of every clip times the
    [vocab, 512] weight, zero-padded to 64 rows like Decoder._get_packed -> logits fp32 [n, vocab]."""

    @staticmethod
    def forward(ctx, x, x16, w, n, L):
        vocab, d = w.shape
        last16 = x16.view(n, L, d)[:, -1].contiguous()
        wp = torch.zeros((64, d), dtype=F32, device=w.device)
        wp[:vocab] = w.detach()
        _, logits = ops.gemm(last16, ops.cast_enc16(wp), out_f32=True)
        ctx.save_for_backward(last16, wp)
        ctx.n, ctx.L, ctx.vocab = n, L, vocab
        return logits[:, :vocab].contiguous()

    @staticmethod
    def backward(ctx, dlogits):
        last16, wp = ctx.saved_tensors
        n, L, vocab = ctx.n, ctx.L, ctx.vocab
        dl = torch.zeros((n, 64), dtype=F32, device=wp.device)
        dl[:, :vocab] = dlogits
        dl16 = ops.cast_bf16(dl)
        dw, _ = _lin_bwd(dl16, None, last16, wp, bias=False)
        dx = torch.zeros((n, L, wp.shape[1]), dtype=F32, device=wp.device)
        dx[:, -1] = _lin_dgrad(dl16, wp)
        return dx.view(n * L, -1), None, dw[:vocab].contiguous(), None, None


def decoder_forward_train(dec, padded_input_l2r, padded_input_r2l, encoder_outputs):
    """Decoder.forward in training mode (reference decoder.py:79-191) -> (logits_l2r [N,16,vocab], gold_l2r,
    logits_r2l, gold_r2l), the logits autograd-connected to every decoder parameter and to `encoder_outputs`.

    16 steps; step i recomputes the whole prefix of length L = i + 1 in both directions (subsequent mask in the first
    layer only, the mixing after every layer) and feeds, per the reference's coin `random.random() > 0.5`, the step's
    own argmax (a constant for autograd) or the gold token.  Dropout factors are drawn with _drop_factor in this order
    (DESIGN.md §9): per step, the embedding's of l2r then r2l; then per layer, l2r then r2l, each as (self-attention
    probabilities [H*N, L, L], self fc output [N*L, 512], enc-attention probabilities [H*N, L, t_enc], enc fc output,
    ffn output); the embedding's are [N*L, 512]."""
    ys_out = {}
    _, ys_out["l2r"] = dec.preprocess(padded_input_l2r)
    _, ys_out["r2l"] = dec.preprocess(padded_input_r2l)
    n, t_enc, dm = encoder_outputs.shape
    dev = encoder_outputs.device
    h = dec.n_head
    p = float(dec.dropout.p)
    enc = encoder_outputs.float().contiguous().view(n * t_enc, dm)
    enc16 = ops.cast_enc16(enc.detach())
    layers = {"l2r": [dec.layer_first_l2r] + list(dec.layer_stack_l2r),
              "r2l": [dec.layer_first_r2l] + list(dec.layer_stack_r2l)}
    kv = {d: [EncoderKVFn.apply(enc, enc16, l_.enc_attn.w_ks.weight, l_.enc_attn.w_ks.bias, l_.enc_attn.w_vs.weight,
                                l_.enc_attn.w_vs.bias) for l_ in layers[d]] for d in ("l2r", "r2l")}
    prj = {"l2r": dec.tgt_word_prj_l2r.weight, "r2l": dec.tgt_word_prj_r2l.weight}
    pe = dec.positional_encoding.pe[0]
    ys = {d: torch.full((n, dec.maxlen + 1), dec.sos_id, dtype=torch.long, device=dev) for d in ("l2r", "r2l")}
    logits = {"l2r": [], "r2l": []}
    for i in range(dec.maxlen):
        L = i + 1
        x = {}
        for d in ("l2r", "r2l"):
            x32, x16 = DecoderEmbedFn.apply(dec.tgt_word_emb.weight, ys[d], L, pe, float(dec.x_logit_scale))
            f = _drop_factor((n * L, dm), p, dev, True)
            x[d] = (x32, x16) if f is None else (x32 * f, None)
        for li in range(dec.n_layers):
            for d in ("l2r", "r2l"):
                lyr = layers[d][li]
                a, c, ff = lyr.slf_attn, lyr.enc_attn, lyr.pos_ffn
                drops = tuple(_drop_factor(s_, p, dev, True) for s_ in ((h * n, L, L), (n * L, dm), (h * n, L, t_enc),
                                                                         (n * L, dm), (n * L, dm)))
                x[d] = DecoderLayerFn.apply(
                    x[d][0], x[d][1], kv[d][li][0], kv[d][li][1], a.w_qs.weight, a.w_qs.bias, a.w_ks.weight,
                    a.w_ks.bias, a.w_vs.weight, a.w_vs.bias, a.fc.weight, a.fc.bias, a.layer_norm.weight,
                    a.layer_norm.bias, c.w_qs.weight, c.w_qs.bias, c.fc.weight, c.fc.bias, c.layer_norm.weight,
                    c.layer_norm.bias, ff.w_1.weight, ff.w_1.bias, ff.w_2.weight, ff.w_2.bias, ff.layer_norm.weight,
                    ff.layer_norm.bias, drops, n, L, t_enc, h, li == 0, 1.0 / a.temperature, 1.0 / c.temperature,
                    (a.layer_norm.eps, c.layer_norm.eps, ff.layer_norm.eps))
            a32, b32, a16, b16 = BidirMixFn.apply(x["l2r"][0], x["r2l"][0], n, L)
            x = {"l2r": (a32, a16), "r2l": (b32, b16)}
        step = {d: DecoderProjFn.apply(x[d][0], x[d][1], prj[d], n, L) for d in ("l2r", "r2l")}
        is_teacher = random.random() > 0.5          # decoder.py:176 (the flag's name is the reference's)
        for d in ("l2r", "r2l"):
            logits[d].append(step[d])
            ys[d][:, i + 1] = step[d].detach().argmax(-1) if is_teacher else ys_out[d][:, i].to(dev)
    return torch.stack(logits["l2r"], 1), ys_out["l2r"], torch.stack(logits["r2l"], 1), ys_out["r2l"]
