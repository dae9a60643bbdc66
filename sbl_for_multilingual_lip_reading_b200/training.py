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

Precision: bf16 conv operands / activations / gradients, enc16 encoder activations, fp32 accumulation, statistics,
LayerNorm / softmax math, residual-stream gradients and parameter gradients.  Dropout masks are drawn with
`torch.nn.functional.dropout(ones)` — the same generator, call order and shapes as the reference's nn.Dropout /
F.dropout calls, so a seeded reference run draws the same masks; the mask multiply itself is the only torch arithmetic
on the path (plus fp32 gradient additions where two branches meet).
"""
from __future__ import annotations

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
def _lin_bwd(dy16, dy32, x16, w):
    """Linear backward: dy16 bf16 [M,out] (GEMM operand), dy32 fp32 or None (bias gradient source), x16 saved enc16
    input [M,in], w fp32 [out,in]  ->  (dW fp32 [out,in], db fp32 [out])."""
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
    db = ot.colreduce(2, dy32)[0].clone() if dy32 is not None else ot.colreduce(4, dy16)[0].clone()
    return dw, db


def _lin_dgrad(dy16, w, out_f32=True):
    """dx = dy W: dy16 bf16 [M,out], w fp32 [out,in] -> fp32 (or bf16) [M,in]."""
    wt = ops.cast_bf16(w.detach().t().contiguous())                   # [in, out] = the K-major B operand
    o16, o32 = ot.gemm_fmt(dy16, wt, out16=not out_f32, out_f32=out_f32)
    return o32 if out_f32 else o16


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
        m = n * t
        d_attn, d_fc, d_ffn = drops
        x16 = ops.cast_enc16(x)
        wqkv = ops.cast_enc16(torch.cat([wq.detach(), wk.detach(), wv.detach()], 0).contiguous())
        bqkv = torch.cat([bq.detach(), bk.detach(), bv.detach()]).contiguous()
        qkv16, _ = ops.gemm(x16, wqkv, bias=bqkv, out_bf16=True)
        att16, probs = ot.attention_train_fwd(qkv16, n, t, h, drop=d_attn, lengths=lengths, scale=scale)
        _, y1 = ops.gemm(att16, ops.cast_enc16(wfc.detach().contiguous()), bias=bfc.detach(), out_f32=True)
        if d_fc is not None:
            y1 = y1 * d_fc
        z1 = y1 + x
        x1, x1_16 = ops.add_layernorm(z1, g1.detach(), be1.detach(), lengths=lengths, T=t, eps=eps)
        h16, _ = ops.gemm(x1_16, ops.cast_enc16(w1.detach().contiguous()), bias=b1.detach(), relu=True, out_bf16=True)
        _, y2 = ops.gemm(h16, ops.cast_enc16(w2.detach().contiguous()), bias=b2.detach(), out_f32=True)
        if d_ffn is not None:
            y2 = y2 * d_ffn
        z2 = y2 + x1
        out, _ = ops.add_layernorm(z2, g2.detach(), be2.detach(), lengths=lengths, T=t, eps=eps, want_bf16=False)
        ctx.save_for_backward(x16, qkv16, probs, att16, z1, x1_16, h16, z2, wq, wk, wv, wfc, w1, w2, g1, g2)
        ctx.misc = (drops, lengths, n, t, h, scale, eps)
        return out

    @staticmethod
    def backward(ctx, dout):
        x16, qkv16, probs, att16, z1, x1_16, h16, z2, wq, wk, wv, wfc, w1, w2, g1, g2 = ctx.saved_tensors
        (d_attn, d_fc, d_ffn), lengths, n, t, h, scale, eps = ctx.misc
        # x2 = LN(z2) * keep ; z2 = dropout(w_2 relu(w_1 x1)) + x1
        dz2_32, dz2_16, dg2, dbe2 = ot.ln_bwd(dout.contiguous().float(), z2, g2.detach(), lengths=lengths, T=t, eps=eps)
        if d_ffn is not None:
            dy2_32 = dz2_32 * d_ffn
            dy2_16 = ops.cast_bf16(dy2_32)
        else:
            dy2_32, dy2_16 = dz2_32, dz2_16
        dw2, db2 = _lin_bwd(dy2_16, dy2_32, h16, w2)
        dh = _lin_dgrad(dy2_16, w2, out_f32=False)
        ot.relu_bwd_(dh, h16)
        dw1, db1 = _lin_bwd(dh, None, x1_16, w1)
        dx1 = dz2_32 + _lin_dgrad(dh, w1)
        # x1 = LN(z1) * keep ; z1 = dropout(fc(attention)) + x
        dz1_32, dz1_16, dg1, dbe1 = ot.ln_bwd(dx1, z1, g1.detach(), lengths=lengths, T=t, eps=eps)
        if d_fc is not None:
            dy1_32 = dz1_32 * d_fc
            dy1_16 = ops.cast_bf16(dy1_32)
        else:
            dy1_32, dy1_16 = dz1_32, dz1_16
        dwfc, dbfc = _lin_bwd(dy1_16, dy1_32, att16, wfc)
        datt = _lin_dgrad(dy1_16, wfc, out_f32=False)
        dqkv = ot.attention_train_bwd(qkv16, probs, datt, n, t, h, drop=d_attn, lengths=lengths, scale=scale)
        wqkv = torch.cat([wq.detach(), wk.detach(), wv.detach()], 0)
        dwqkv, dbqkv = _lin_bwd(dqkv, None, x16, wqkv)
        dx = dz1_32 + _lin_dgrad(dqkv, wqkv)
        hk = wq.shape[0]
        return (dx, dwqkv[:hk].contiguous(), dbqkv[:hk].contiguous(), dwqkv[hk:2 * hk].contiguous(),
                dbqkv[hk:2 * hk].contiguous(), dwqkv[2 * hk:].contiguous(), dbqkv[2 * hk:].contiguous(), dwfc, dbfc, dg1,
                dbe1, dw1, db1, dw2, db2, dg2, dbe2, None, None, None, None, None, None, None)


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
