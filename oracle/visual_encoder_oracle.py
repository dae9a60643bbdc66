"""CPU oracle for the visual-encoder hot path — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A functional, fp32, CPU restatement of the reference's algorithm for the path
Conv3d frontend -> per-frame ResNet-18 trunk -> transformer Encoder.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may import this file;
the product package (sbl_for_multilingual_lip_reading_b200/) never does.

Every function cites the reference lines it restates (paths relative to
/root/reference/SBL_Multilingual_Lip_reading/).  The arithmetic itself lives in PyTorch (un-vendored
third-party dependency of the reference, "Pytorch: 1.3+" README.md:11; torch 2.11.0 here), so the
restatement calls the same torch.nn.functional primitives the reference's nn.Modules dispatch to, on a
plain {reference state-dict key -> tensor} dict.

Pinning: the reference ships NO tests, fixtures or golden vectors for this path (SURVEY.md §8c,
"parity unpinned" upstream).  The oracle is therefore pinned against outputs of the reference modules
themselves, imported from /root/reference in the build container by tests/golden/make_golden.py and
committed as tests/golden/*.npz; tests/test_oracle_golden.py checks every one of them.

The reference's always-on `F.dropout(x, p=0.5)` (transformer/video_frontend.py:122, training=True by
default, so active under model.eval()) is exposed as an explicit `dropout_mask` argument: parity runs pass
None (identity) on both sides, exactly as the goldens were produced from `_frontend_forward`.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

BN_EPS = 1e-5  # nn.BatchNorm2d/3d default, never overridden (video_frontend.py:21,24,71,101)
LN_EPS = 1e-5  # nn.LayerNorm default (attention.py:25, module.py:45, encoder.py:28)


# ----------------------------------------------------------------------------------------------
# visual frontend  (transformer/video_frontend.py)
# ----------------------------------------------------------------------------------------------
def _bn(x, sd, prefix):
    """Eval-mode BatchNorm with running statistics (video_frontend.py:21,24,71,101)."""
    return F.batch_norm(x, sd[prefix + ".running_mean"], sd[prefix + ".running_var"], sd[prefix + ".weight"],
                        sd[prefix + ".bias"], training=False, momentum=0.1, eps=BN_EPS)


def frontend3d(x, sd, prefix="frontend3D"):
    """Conv3d(1,64,(5,7,7),(1,2,2),(2,3,3),bias=False) + BatchNorm3d + ReLU + MaxPool3d((1,3,3),(1,2,2),(0,1,1)).
    video_frontend.py:99-104.  x: [N,1,T,88,88] -> [N,64,T,22,22]."""
    y = F.conv3d(x, sd[prefix + ".0.weight"], None, stride=(1, 2, 2), padding=(2, 3, 3))
    y = _bn(y, sd, prefix + ".1")
    y = F.relu(y)
    return F.max_pool3d(y, kernel_size=(1, 3, 3), stride=(1, 2, 2), padding=(0, 1, 1))


def basic_block(x, sd, prefix, stride, has_downsample):
    """BasicBlock.forward, video_frontend.py:28-41 (conv3x3: :10-12; downsample: :68-72)."""
    residual = x
    out = F.conv2d(x, sd[prefix + ".conv1.weight"], None, stride=stride, padding=1)
    out = F.relu(_bn(out, sd, prefix + ".bn1"))
    out = F.conv2d(out, sd[prefix + ".conv2.weight"], None, stride=1, padding=1)
    out = _bn(out, sd, prefix + ".bn2")
    if has_downsample:
        residual = F.conv2d(x, sd[prefix + ".downsample.0.weight"], None, stride=stride, padding=0)
        residual = _bn(residual, sd, prefix + ".downsample.1")
    return F.relu(out + residual)


def resnet18_trunk(x, sd, prefix="resnet18"):
    """ResNet.forward with layers [2,2,2,2], planes 64/128/256/512, strides 1/2/2/2, AdaptiveAvgPool2d(1).
    video_frontend.py:46-53,65-80,82-89.  x: [F,64,22,22] -> [F,512]."""
    for li, stride in ((1, 1), (2, 2), (3, 2), (4, 2)):
        x = basic_block(x, sd, f"{prefix}.layer{li}.0", stride, has_downsample=(li != 1))
        x = basic_block(x, sd, f"{prefix}.layer{li}.1", 1, has_downsample=False)
    x = F.adaptive_avg_pool2d(x, 1)
    return x.view(x.size(0), -1)


def frontend_forward(x, sd, prefix=""):
    """Lipreading._frontend_forward, video_frontend.py:111-117.  x: [N,1,T,88,88] -> [N*T,512]."""
    y = frontend3d(x, sd, prefix + "frontend3D")
    y = y.transpose(1, 2).contiguous()
    y = y.view(-1, 64, y.size(3), y.size(4))
    return resnet18_trunk(y, sd, prefix + "resnet18")


def lipreading_forward(x, sd, prefix="", dropout_mask=None):
    """Lipreading.forward, video_frontend.py:119-125.  dropout_mask: None (parity mode, identity) or a
    {0,1} float tensor [N*T,512]; the reference draws it with F.dropout(p=0.5) -> kept values are scaled x2."""
    frame_len = x.size(2)
    y = frontend_forward(x, sd, prefix)
    if dropout_mask is not None:
        y = y * dropout_mask * 2.0
    return y.view(-1, frame_len, 512)


# ----------------------------------------------------------------------------------------------
# transformer encoder  (transformer/encoder.py, attention.py, module.py, utils.py)
# ----------------------------------------------------------------------------------------------
def positional_encoding_table(max_len=5000, d_model=512):
    """PositionalEncoding.__init__, module.py:14-25 -> pe [1,max_len,d_model]."""
    pe = torch.zeros(max_len, d_model)
    position = torch.arange(0, max_len).unsqueeze(1).float()
    div_term = torch.exp(torch.arange(0, d_model, 2).float() * -(math.log(10000.0) / d_model))
    pe[:, 0::2] = torch.sin(position * div_term)
    pe[:, 1::2] = torch.cos(position * div_term)
    return pe.unsqueeze(0)


def non_pad_mask(n, t, input_lengths, dtype=torch.float32):
    """get_non_pad_mask, utils.py:98-113: [N,T,1], 1 where t < length."""
    lengths = torch.as_tensor(list(input_lengths), dtype=torch.long)
    return (torch.arange(t)[None, :] < lengths[:, None]).to(dtype).unsqueeze(-1)


def attn_pad_mask(n, t, input_lengths, expand_length):
    """get_attn_pad_mask, utils.py:140-147: bool [N,expand_length,T], True where KEY t >= length."""
    pad = non_pad_mask(n, t, input_lengths).squeeze(-1).lt(1)
    return pad.unsqueeze(1).expand(-1, expand_length, -1)


def multi_head_attention(x, sd, prefix, n_head, d_k, d_v, mask, kv=None):
    """MultiHeadAttention.forward, attention.py:32-60, with ScaledDotProductAttention.forward, attention.py:72-83
    (temperature = d_k ** 0.5, attention.py:23).  Queries and the residual come from x; keys and values from kv
    (default x: self-attention; the decoder's enc_attn passes the encoder outputs).  mask: bool [N, len_q, len_k],
    True = masked, or None."""
    kv = x if kv is None else kv
    sz_b, len_q, _ = x.shape
    len_k = kv.shape[1]
    residual = x
    q = F.linear(x, sd[prefix + ".w_qs.weight"], sd[prefix + ".w_qs.bias"]).view(sz_b, len_q, n_head, d_k)
    k = F.linear(kv, sd[prefix + ".w_ks.weight"], sd[prefix + ".w_ks.bias"]).view(sz_b, len_k, n_head, d_k)
    v = F.linear(kv, sd[prefix + ".w_vs.weight"], sd[prefix + ".w_vs.bias"]).view(sz_b, len_k, n_head, d_v)
    q = q.permute(2, 0, 1, 3).contiguous().view(-1, len_q, d_k)  # (n_head*b) x T x d_k, index h*b + i
    k = k.permute(2, 0, 1, 3).contiguous().view(-1, len_k, d_k)
    v = v.permute(2, 0, 1, 3).contiguous().view(-1, len_k, d_v)
    attn = torch.bmm(q, k.transpose(1, 2)) / float(d_k ** 0.5)
    if mask is not None:
        attn = attn.masked_fill(mask.repeat(n_head, 1, 1).bool(), float("-inf"))
    attn = torch.softmax(attn, dim=2)
    out = torch.bmm(attn, v)
    out = out.view(n_head, sz_b, len_q, d_v).permute(1, 2, 0, 3).contiguous().view(sz_b, len_q, -1)
    out = F.linear(out, sd[prefix + ".fc.weight"], sd[prefix + ".fc.bias"])
    out = F.layer_norm(out + residual, (out.size(-1),), sd[prefix + ".layer_norm.weight"],
                       sd[prefix + ".layer_norm.bias"], LN_EPS)
    return out, attn


def positionwise_ffn(x, sd, prefix):
    """PositionwiseFeedForward.forward, module.py:47-52."""
    h = F.linear(F.relu(F.linear(x, sd[prefix + ".w_1.weight"], sd[prefix + ".w_1.bias"])),
                 sd[prefix + ".w_2.weight"], sd[prefix + ".w_2.bias"])
    return F.layer_norm(h + x, (x.size(-1),), sd[prefix + ".layer_norm.weight"], sd[prefix + ".layer_norm.bias"],
                        LN_EPS)


def encoder_forward(padded_input, input_lengths, sd, prefix="", n_layers=6, n_head=8, d_k=64, d_v=64,
                    return_attns=False):
    """Encoder.forward (eval: dropout = identity), encoder.py:36-67 and EncoderLayer.forward, encoder.py:83-91.
    Returns (enc_output,) or (enc_output, [attn per layer]) exactly like the reference."""
    n, t, _ = padded_input.shape
    npm = non_pad_mask(n, t, input_lengths)                       # encoder.py:47
    mask = attn_pad_mask(n, t, input_lengths, t)                  # encoder.py:48-49
    x = F.linear(padded_input, sd[prefix + "linear_in.weight"], sd[prefix + "linear_in.bias"])
    x = F.layer_norm(x, (x.size(-1),), sd[prefix + "layer_norm_in.weight"], sd[prefix + "layer_norm_in.bias"], LN_EPS)
    x = x + sd[prefix + "positional_encoding.pe"][:, :t]          # encoder.py:53-55, module.py:26-32
    attns = []
    for i in range(n_layers):
        lp = f"{prefix}layer_stack.{i}"
        x, attn = multi_head_attention(x, sd, lp + ".slf_attn", n_head, d_k, d_v, mask)
        x = x * npm                                               # encoder.py:86
        x = positionwise_ffn(x, sd, lp + ".pos_ffn")
        x = x * npm                                               # encoder.py:89
        if return_attns:
            attns.append(attn)
    if return_attns:
        return x, attns
    return (x,)


def visual_encoder_forward(x, sd, n_layers=6, frontend_prefix="visual_frontend.", encoder_prefix="encoder.",
                           dropout_mask=None):
    """The hot path as Transformer.forward / recognize drive it, transformer.py:31-38,55-67:
    x [N,1,T,88,88] -> frontend -> [N,T,512] -> encoder with input_lengths = [T]*N -> [N,T,512]."""
    feat = lipreading_forward(x, sd, frontend_prefix, dropout_mask)
    n, t, _ = feat.shape
    return encoder_forward(feat, [t] * n, sd, encoder_prefix, n_layers=n_layers)[0]


# ----------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md §8d / BASELINE.md §3)
# ----------------------------------------------------------------------------------------------
def flops_per_clip(t, n_layers=6):
    """2*MACs of every contraction on the path for one T-frame clip."""
    return t * (60712960 + 571604992 + 524288 + n_layers * 6291456) + n_layers * 2048 * t * t
