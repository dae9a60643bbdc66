"""Oracle for the SBL bidirectional decoder — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A functional restatement, in the style of `visual_encoder_oracle.py`, of what the drop-in decoder
(sbl_for_multilingual_lip_reading_b200/decoder.py, DESIGN.md §9, include/sblk.h) computes: functions on a plain
{state-dict key -> tensor} dict with the drop-in's keys (`tgt_word_emb.weight`, `positional_encoding.pe`,
`layer_first_{l2r,r2l}.*`, `layer_stack_{l2r,r2l}.{i}.*`, `tgt_word_prj_{l2r,r2l}.weight`).  Every function is
dtype- and device-agnostic: the tests run it in float64 on CUDA (kernel parity) or in fp32 on the CPU.

Pinning: the reference sources (SBL transformer/decoder.py) are not part of this repository, so this file restates the
semantics the drop-in documents, which round 2 validated against the reference decoder on a B200.  Where oracle/_ref
is staged, tests/test_decoder_oracle_cpu.py pins `step_logits` to the reference `Decoder` itself; elsewhere that test
skips and the oracle is pinned only to the documentation.

Per decode step, with prefix length L (the whole prefix is recomputed at every step):
  x = emb[y[:, :L]] * x_logit_scale + pe[:L]                                   (both directions, one embedding table)
  per layer: self-attention (subsequent mask, key j > query i masked, in the FIRST layer only), attention over all
             encoder frames (no mask), position-wise FFN; then the bidirectional mixing (`bidir_mix`)
  logits = tgt_word_prj_{l2r,r2l}(x[:, L-1])
Only `tests/` import this file.
"""
from __future__ import annotations

import torch

from .visual_encoder_oracle import multi_head_attention, positionwise_ffn

IGNORE_ID = -1
MAXLEN = 16          # decode steps, and pad_list's hard-coded max_len
N_HEAD, D_K, D_V = 8, 64, 64


def subsequent_mask(n, L, device):
    """get_subsequent_mask: bool [n, L, L], True where key j > query i."""
    return torch.triu(torch.ones(L, L, dtype=torch.bool, device=device), diagonal=1).unsqueeze(0).expand(n, -1, -1)


def n_layers(sd):
    """Layers per direction: layer_first + layer_stack.{0..n-2}."""
    stack = {k.split(".")[1] for k in sd if k.startswith("layer_stack_l2r.")}
    return 1 + len(stack)


def layer_prefix(direction, li):
    return f"layer_first_{direction}" if li == 0 else f"layer_stack_{direction}.{li - 1}"


def embed(sd, ys, L, x_logit_scale=1.0):
    """tgt_word_emb(ys[:, :L]) * x_logit_scale + positional_encoding -> [N, L, d_model]."""
    return sd["tgt_word_emb.weight"][ys[:, :L]] * x_logit_scale + sd["positional_encoding.pe"][:, :L]


def decoder_layer(x, enc, sd, prefix, slf_mask):
    """DecoderLayer: self-attention (slf_mask or None), decoder-encoder attention over every frame, FFN."""
    x, _ = multi_head_attention(x, sd, prefix + ".slf_attn", N_HEAD, D_K, D_V, slf_mask)
    x, _ = multi_head_attention(x, sd, prefix + ".enc_attn", N_HEAD, D_K, D_V, None, kv=enc)
    return positionwise_ffn(x, sd, prefix + ".pos_ffn")


def bidir_mix(l2r, r2l):
    """The synchronous bidirectional mixing as the reference writes it: two in-place loops over aliases of the hidden
    states, the second of which reads the already updated left-to-right stream.  Returns new tensors."""
    l2r, r2l = l2r.clone(), r2l.clone()
    L = l2r.size(1)
    for i in range(L):
        l2r[:, i] = l2r[:, i] + r2l[:, L - 1 - i]
    for i in range(L):
        r2l[:, i] = r2l[:, i] + l2r[:, L - 1 - i]
    return l2r, r2l


def step_logits(sd, ys_l2r, ys_r2l, enc, L, x_logit_scale=1.0, mask=subsequent_mask, mask_every_layer=False,
                mix=bidir_mix):
    """One decode step for the prefixes ys[:, :L] -> (logits_l2r, logits_r2l) [N, vocab] of the last position.
    `mask`, `mask_every_layer` and `mix` exist so that tests can build deliberately wrong variants."""
    n = ys_l2r.shape[0]
    x = {"l2r": embed(sd, ys_l2r, L, x_logit_scale), "r2l": embed(sd, ys_r2l, L, x_logit_scale)}
    m = mask(n, L, enc.device)
    for li in range(n_layers(sd)):
        slf = m if (li == 0 or mask_every_layer) else None
        for d in ("l2r", "r2l"):
            x[d] = decoder_layer(x[d], enc, sd, layer_prefix(d, li), slf)
        x["l2r"], x["r2l"] = mix(x["l2r"], x["r2l"])
    return (torch.nn.functional.linear(x["l2r"][:, -1], sd["tgt_word_prj_l2r.weight"]),
            torch.nn.functional.linear(x["r2l"][:, -1], sd["tgt_word_prj_r2l.weight"]))


def greedy(sd, enc, sos_id=0, x_logit_scale=1.0):
    """Greedy bidirectional decoding, 16 steps without early stop, both directions from <sos> ->
    (ys_l2r, ys_r2l) int64 [N, 17] and (logits_l2r, logits_r2l) [N, 16, vocab], like Decoder._greedy(want_logits=True)."""
    n = enc.shape[0]
    ys = {d: torch.full((n, MAXLEN + 1), sos_id, dtype=torch.long, device=enc.device) for d in ("l2r", "r2l")}
    logits = {"l2r": [], "r2l": []}
    for i in range(MAXLEN):
        lg = step_logits(sd, ys["l2r"], ys["r2l"], enc, i + 1, x_logit_scale)
        for d, v in zip(("l2r", "r2l"), lg):
            logits[d].append(v)
            ys[d][:, i + 1] = v.argmax(-1)
    return ys["l2r"], ys["r2l"], torch.stack(logits["l2r"], 1), torch.stack(logits["r2l"], 1)


def pad_list(xs, pad_value, max_len=MAXLEN):
    """utils.pad_list: [len(xs), max_len] filled with pad_value, row i starting with xs[i] (longer rows raise)."""
    pad = xs[0].new_full((len(xs), max_len) + tuple(xs[0].shape[1:]), pad_value)
    for i, x in enumerate(xs):
        pad[i, :x.size(0)] = x
    return pad


def preprocess(padded, sos, eos):
    """Decoder.preprocess as per-utterance loops: drop IGNORE_ID entries, <sos> + y and y + <eos>, both padded to 16
    columns with eos -> (ys_in_pad, ys_out_pad)."""
    ys = [y[y != IGNORE_ID] for y in padded]
    ys_in = [torch.cat([y.new_full((1,), sos), y]) for y in ys]
    ys_out = [torch.cat([y, y.new_full((1,), eos)]) for y in ys]
    return pad_list(ys_in, eos), pad_list(ys_out, eos)
