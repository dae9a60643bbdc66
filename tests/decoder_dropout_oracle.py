"""Training-mode dropout for the float64 decoder oracle — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

oracle/decoder_oracle.step_logits restates the decoder in evaluation mode.  This module restates one decode step with
the training-mode dropout made explicit, from the same pieces (embedding, masks, layer prefixes, the aliased mixing):
every factor is mask / (1 - p) as the decoder drew it, or None where no dropout applies.  With every factor None it
computes what step_logits computes (tests/test_decoder_train_cpu.py pins that).

drops for one step: {direction: {"emb": [N*L, d_model] | None, "layers": [per layer (self-attention probabilities
[N_HEAD*N, L, L], self fc output [N*L, d_model], enc-attention probabilities [N_HEAD*N, L, t_enc], enc fc output,
ffn output)]}} — the order and shapes of training.decoder_forward_train (DESIGN.md §9).
Imported by tests/ and by tools/decoder_train_probe.py only.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import decoder_oracle as O
from oracle.visual_encoder_oracle import LN_EPS


def _mul(x, f):
    return x if f is None else x * f.to(x.dtype).view(x.shape)


def attention(x, sd, prefix, mask, kv, d_attn, d_fc):
    """MultiHeadAttention (attention.py:32-60, 72-83) with dropout factors on the probabilities (index h*N + b) and on
    the fc output."""
    kv = x if kv is None else kv
    n, len_q, _ = x.shape
    len_k = kv.shape[1]
    h, dk, dv = O.N_HEAD, O.D_K, O.D_V
    q = F.linear(x, sd[prefix + ".w_qs.weight"], sd[prefix + ".w_qs.bias"]).view(n, len_q, h, dk)
    k = F.linear(kv, sd[prefix + ".w_ks.weight"], sd[prefix + ".w_ks.bias"]).view(n, len_k, h, dk)
    v = F.linear(kv, sd[prefix + ".w_vs.weight"], sd[prefix + ".w_vs.bias"]).view(n, len_k, h, dv)
    q = q.permute(2, 0, 1, 3).reshape(-1, len_q, dk)
    k = k.permute(2, 0, 1, 3).reshape(-1, len_k, dk)
    v = v.permute(2, 0, 1, 3).reshape(-1, len_k, dv)
    attn = torch.bmm(q, k.transpose(1, 2)) / float(dk ** 0.5)
    if mask is not None:
        attn = attn.masked_fill(mask.repeat(h, 1, 1).bool(), float("-inf"))
    attn = _mul(torch.softmax(attn, dim=2), d_attn)
    out = torch.bmm(attn, v).view(h, n, len_q, dv).permute(1, 2, 0, 3).reshape(n, len_q, -1)
    out = _mul(F.linear(out, sd[prefix + ".fc.weight"], sd[prefix + ".fc.bias"]), d_fc)
    return F.layer_norm(out + x, (out.size(-1),), sd[prefix + ".layer_norm.weight"], sd[prefix + ".layer_norm.bias"],
                        LN_EPS)


def decoder_layer(x, enc, sd, prefix, slf_mask, drops):
    """DecoderLayer with the five dropout factors of one layer and direction."""
    d_a1, d_f1, d_a2, d_f2, d_ffn = drops
    x = attention(x, sd, prefix + ".slf_attn", slf_mask, None, d_a1, d_f1)
    x = attention(x, sd, prefix + ".enc_attn", None, enc, d_a2, d_f2)
    p = prefix + ".pos_ffn"
    y = F.linear(F.relu(F.linear(x, sd[p + ".w_1.weight"], sd[p + ".w_1.bias"])), sd[p + ".w_2.weight"],
                 sd[p + ".w_2.bias"])
    return F.layer_norm(_mul(y, d_ffn) + x, (x.size(-1),), sd[p + ".layer_norm.weight"], sd[p + ".layer_norm.bias"],
                        LN_EPS)


def step_logits(sd, ys_l2r, ys_r2l, enc, L, drops, x_logit_scale=1.0):
    """decoder_oracle.step_logits in training mode: one step for the prefixes ys[:, :L] with the step's dropout factors
    -> (logits_l2r, logits_r2l) [N, vocab] of the last position."""
    n = ys_l2r.shape[0]
    x = {d: _mul(O.embed(sd, ys, L, x_logit_scale), drops[d]["emb"]) for d, ys in (("l2r", ys_l2r), ("r2l", ys_r2l))}
    m = O.subsequent_mask(n, L, enc.device)
    for li in range(O.n_layers(sd)):
        for d in ("l2r", "r2l"):
            x[d] = decoder_layer(x[d], enc, sd, O.layer_prefix(d, li), m if li == 0 else None, drops[d]["layers"][li])
        x["l2r"], x["r2l"] = O.bidir_mix(x["l2r"], x["r2l"])
    return (F.linear(x["l2r"][:, -1], sd["tgt_word_prj_l2r.weight"]),
            F.linear(x["r2l"][:, -1], sd["tgt_word_prj_r2l.weight"]))
