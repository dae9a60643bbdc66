"""Drop-in replacement for the reference transformer encoder (transformer/encoder.py + the parts of
attention.py / module.py / utils.py it uses).

`Encoder` has the reference constructor signature, attributes, state-dict keys and return convention
((enc_output,) 1-tuple, or (enc_output, [attn]*n_layers) with return_attns=True — callers unpack with
`enc_out, *_ = self.encoder(...)`, transformer/transformer.py:38).  Submodules are parameter holders with the
reference's names and initialisation; the forward pass runs libsblk kernels only:

    cast -> linear_in GEMM -> LayerNorm + PE  -> n_layers x {
        [per-head QKV projection + softmax attention] (one launch) -> fc GEMM -> residual + LayerNorm (+pad mask)
        w_1 GEMM + ReLU -> w_2 GEMM -> residual + LayerNorm (+pad mask) }
    (GEMM -> LayerNorm pairs: split-K partials summed by the LayerNorm kernel at small token counts, one
    cluster-fused launch at large ones; see ops.linear_ln)

The residual stream stays fp32; GEMM operands are 16-bit (`ops.enc16_dtype()`: fp16 by default — the encoder's
values are LayerNorm-bounded, so the 3 extra mantissa bits over bf16 cost nothing) with fp32 accumulation.
Masks are never materialised: `input_lengths` goes to the kernels as an int32 vector
(reference builds them with a Python loop twice per call, transformer/utils.py:98-113,140-147).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from . import ops


class PositionalEncoding(nn.Module):
    """Holder of the reference sin/cos table buffer `pe` [1,max_len,d_model] (transformer/module.py:8-32)."""

    def __init__(self, d_model, max_len=5000):
        super().__init__()
        pe = torch.zeros(max_len, d_model, requires_grad=False)
        position = torch.arange(0, max_len).unsqueeze(1).float()
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * -(math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer('pe', pe.unsqueeze(0))

    def forward(self, input):
        return self.pe[:, :input.size(1)]


class _SelfAttentionParams(nn.Module):
    """Parameter holder mirroring reference MultiHeadAttention.__init__ (transformer/attention.py:9-30)."""

    def __init__(self, n_head, d_model, d_k, d_v, dropout=0.1):
        super().__init__()
        self.n_head, self.d_k, self.d_v = n_head, d_k, d_v
        self.w_qs = nn.Linear(d_model, n_head * d_k)
        self.w_ks = nn.Linear(d_model, n_head * d_k)
        self.w_vs = nn.Linear(d_model, n_head * d_v)
        nn.init.normal_(self.w_qs.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_ks.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_vs.weight, mean=0, std=np.sqrt(2.0 / (d_model + d_v)))
        self.temperature = float(np.power(d_k, 0.5))
        self.layer_norm = nn.LayerNorm(d_model)
        self.fc = nn.Linear(n_head * d_v, d_model)
        nn.init.xavier_normal_(self.fc.weight)
        self.dropout = nn.Dropout(dropout)


class _FeedForwardParams(nn.Module):
    """Parameter holder mirroring reference PositionwiseFeedForward.__init__ (transformer/module.py:40-45)."""

    def __init__(self, d_model, d_ff, dropout=0.1):
        super().__init__()
        self.w_1 = nn.Linear(d_model, d_ff)
        self.w_2 = nn.Linear(d_ff, d_model)
        self.dropout = nn.Dropout(dropout)
        self.layer_norm = nn.LayerNorm(d_model)


class EncoderLayer(nn.Module):
    """Holder with the reference EncoderLayer attribute names (transformer/encoder.py:70-81)."""

    def __init__(self, d_model, d_inner, n_head, d_k, d_v, dropout=0.1):
        super().__init__()
        self.slf_attn = _SelfAttentionParams(n_head, d_model, d_k, d_v, dropout=dropout)
        self.pos_ffn = _FeedForwardParams(d_model, d_inner, dropout=dropout)


class _PackedEncoder:
    __slots__ = ("key", "w_in", "layers", "stacked")


class Encoder(nn.Module):
    """Drop-in for reference Encoder (transformer/encoder.py:8-67)."""

    def __init__(self, d_input, n_layers, n_head, d_k, d_v, d_model, d_inner, dropout=0.1, pe_maxlen=5000):
        super().__init__()
        self.d_input = d_input
        self.n_layers = n_layers
        self.n_head = n_head
        self.d_k = d_k
        self.d_v = d_v
        self.d_model = d_model
        self.d_inner = d_inner
        self.dropout_rate = dropout
        self.pe_maxlen = pe_maxlen

        self.linear_in = nn.Linear(d_input, d_model)
        self.layer_norm_in = nn.LayerNorm(d_model)
        self.positional_encoding = PositionalEncoding(d_model, max_len=pe_maxlen)
        self.dropout = nn.Dropout(dropout)
        self.layer_stack = nn.ModuleList([
            EncoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout) for _ in range(n_layers)])
        self._packed = None
        self._len_cache = {}
        self._streams = {}
        self.parallel_chains = 4   # clip groups run as concurrent kernel chains (1 = single chain)
        self.fused_stack = True    # one-launch cluster kernel for the whole stack when the shape allows it
        self.fused_stack_max_groups = 12
        # batches with more clip groups than one launch holds are cut into sub-batches of `chunk_groups` groups that go
        # through the SAME one-launch stack (alternating over two streams), so a clip's output bits never depend on the
        # batch it arrives in; False = use the per-step kernels for such batches (different rounding points, ~1e-3 apart)
        self.chunk_large_batches = True
        self.chunk_groups = 8
        self.split_clusters = True   # 8-11 clip groups: 7 as 16-CTA clusters + the rest as 8-CTA clusters, concurrently
        self.stack_cluster_size = 0  # 0 = automatic; 8 / 16 force the cluster size of the one-launch stack (disables the split)
        # clip groups per cluster of the one-launch stack when stack_cluster_size is forced: 2 = two groups interleaved
        # (half the SMs for ~1.5x the time: the pipelined plan's co-running encoder); bit-identical to 1
        self.stack_groups_per_cluster = 1

    def __getstate__(self):
        st = self.__dict__.copy()
        st["_packed"] = None
        st["_len_cache"] = {}
        st["_streams"] = {}
        return st

    # attributes of modules pickled by earlier versions that nothing reads any more (the plans' former hooks)
    _RETIRED = ("_resident_counter", "_x16_override")

    def __setstate__(self, st):
        self.__dict__.update({k: v for k, v in st.items() if k not in self._RETIRED})
        self.__dict__.setdefault("_streams", {})
        self.__dict__.setdefault("_len_cache", {})
        self.__dict__.setdefault("parallel_chains", 4)
        self.__dict__.setdefault("fused_stack", True)
        self.__dict__.setdefault("fused_stack_max_groups", 12)
        self.__dict__.setdefault("chunk_large_batches", True)
        self.__dict__.setdefault("chunk_groups", 8)
        self.__dict__.setdefault("split_clusters", True)
        self.__dict__.setdefault("stack_cluster_size", 0)
        self.__dict__.setdefault("stack_groups_per_cluster", 1)

    # ------------------------------------------------------------------------------------------
    def _check_config(self):
        if self.d_model != 512 or self.d_k != 64 or self.d_v != 64:
            raise RuntimeError(f"Encoder (libsblk): only d_model=512, d_k=d_v=64 are implemented "
                               f"(got d_model={self.d_model}, d_k={self.d_k}, d_v={self.d_v}); no fallback path")
        if self.d_input % 64 or self.d_inner % 64 or (self.n_head * self.d_k) % 64:
            raise RuntimeError("Encoder (libsblk): d_input, d_inner and n_head*d_k must be multiples of 64")

    def _cache_key(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def _check_train_config(self, t, return_attns):
        if return_attns:
            raise RuntimeError("Encoder (libsblk): return_attns is an evaluation feature (training path returns no maps)")
        if t > 64:
            raise RuntimeError(f"Encoder (libsblk): training attention is implemented for T <= 64 frames (got {t})")
        if self.n_head * self.d_k != 512 or self.d_input % 64 or self.d_inner % 64:
            raise RuntimeError("Encoder (libsblk): training path needs n_head*d_k == 512 and 64-aligned widths")

    def invalidate_packed(self):
        """Drop the packed (bf16 / enc16, BN-folded) weight cache.  The cache key is (data_ptr, tensor._version) of every
        parameter and buffer, which `load_state_dict`, optimizer steps and `.to()` all change; edits THROUGH `.data`
        (`p.data.copy_()`, `m.weight.data.normal_()`) do not bump the version counter, so call this after them."""
        self._packed = None

    def _apply(self, fn, *args, **kwargs):
        self._packed = None
        return super()._apply(fn, *args, **kwargs)

    def _get_packed(self):
        key = self._cache_key()
        pk = self._packed
        if pk is not None and pk.key == key:
            return pk
        pk = _PackedEncoder()
        pk.key = key
        pk.w_in = ops.cast_enc16(self.linear_in.weight.detach().contiguous())
        pk.layers = []
        nl, hk, dm, di = len(self.layer_stack), self.n_head * self.d_k, self.d_model, self.d_inner
        dev = self.linear_in.weight.device
        # per-layer tensors are STACKED along dim 0 (one TMA descriptor per weight kind for the one-launch stack,
        # include/sblk.h: sblk_encoder_stack_fwd); the per-step kernels use per-layer views of the same storage
        stk = dict(n_layers=nl, d_inner=di,
                   w_in=pk.w_in, b_in=self.linear_in.bias.detach().float().contiguous(),
                   g_in=self.layer_norm_in.weight.detach().float().contiguous(),
                   be_in=self.layer_norm_in.bias.detach().float().contiguous(),
                   pe=self.positional_encoding.pe[0],
                   w_heads=torch.empty((nl * 3 * hk, dm), dtype=ops.enc16_dtype(), device=dev),
                   b_heads=torch.empty((nl * 3 * hk,), dtype=torch.float32, device=dev),
                   w_fc=torch.empty((nl * dm, hk), dtype=ops.enc16_dtype(), device=dev),
                   w_1=torch.empty((nl * di, dm), dtype=ops.enc16_dtype(), device=dev),
                   w_2=torch.empty((nl * dm, di), dtype=ops.enc16_dtype(), device=dev))

        def cat(ts):
            return (torch.cat([t_.detach().float().reshape(-1) for t_ in ts]).contiguous() if ts
                    else torch.empty((0,), dtype=torch.float32, device=dev))

        stk["b_fc"] = cat([l_.slf_attn.fc.bias for l_ in self.layer_stack])
        stk["g1"] = cat([l_.slf_attn.layer_norm.weight for l_ in self.layer_stack])
        stk["be1"] = cat([l_.slf_attn.layer_norm.bias for l_ in self.layer_stack])
        stk["b_1"] = cat([l_.pos_ffn.w_1.bias for l_ in self.layer_stack])
        stk["b_2"] = cat([l_.pos_ffn.w_2.bias for l_ in self.layer_stack])
        stk["g2"] = cat([l_.pos_ffn.layer_norm.weight for l_ in self.layer_stack])
        stk["be2"] = cat([l_.pos_ffn.layer_norm.bias for l_ in self.layer_stack])
        for li, lyr in enumerate(self.layer_stack):
            a, f = lyr.slf_attn, lyr.pos_ffn
            wqkv = torch.empty((3 * hk, self.d_model), dtype=ops.enc16_dtype(), device=a.w_qs.weight.device)
            ops.cast_enc16(a.w_qs.weight.detach().contiguous(), out=wqkv[0:hk])
            ops.cast_enc16(a.w_ks.weight.detach().contiguous(), out=wqkv[hk:2 * hk])
            ops.cast_enc16(a.w_vs.weight.detach().contiguous(), out=wqkv[2 * hk:3 * hk])
            bqkv = torch.cat([a.w_qs.bias.detach(), a.w_ks.bias.detach(), a.w_vs.bias.detach()]).contiguous()
            # head-major copy (q_h | k_h | v_h per head) for the fused projection + attention kernel
            wheads, bheads = ops.pack_qkv_heads(wqkv[0:hk], wqkv[hk:2 * hk], wqkv[2 * hk:3 * hk],
                                                a.w_qs.bias.detach(), a.w_ks.bias.detach(), a.w_vs.bias.detach(),
                                                self.n_head, self.d_k)
            stk["w_heads"][li * 3 * hk:(li + 1) * 3 * hk].copy_(wheads)
            stk["b_heads"][li * 3 * hk:(li + 1) * 3 * hk].copy_(bheads)
            pk.layers.append(dict(
                wqkv=wqkv, bqkv=bqkv,
                wheads=stk["w_heads"][li * 3 * hk:(li + 1) * 3 * hk], bheads=stk["b_heads"][li * 3 * hk:(li + 1) * 3 * hk],
                wfc=ops.cast_enc16(a.fc.weight.detach().contiguous(), out=stk["w_fc"][li * dm:(li + 1) * dm]),
                w1=ops.cast_enc16(f.w_1.weight.detach().contiguous(), out=stk["w_1"][li * di:(li + 1) * di]),
                w2=ops.cast_enc16(f.w_2.weight.detach().contiguous(), out=stk["w_2"][li * dm:(li + 1) * dm])))
        pk.stacked = stk
        self._packed = pk
        return pk

    def _use_fused_stack(self, n, t, return_attns):
        """The one-launch stack wins while its clusters (one per clip group of <= 128 token rows) run as a single wave:
        measured on B200 at T=29, 6 layers: 176 vs 205 us (8 clips), 176 vs 217 (16), 219 vs 278 (32), 434 vs 410 (64).
        Larger batches fill the machine with the per-step kernels instead."""
        if return_attns or not self.fused_stack or len(self.layer_stack) == 0:
            return False
        if t > 128 or (not self.chunk_large_batches and -(-n // max(1, 128 // t)) > self.fused_stack_max_groups):
            return False
        if not ops.encoder_stack_supported(self.n_head, self.d_k, self.d_v, self.d_model, self.d_input, self.d_inner,
                                           t, len(self.layer_stack)):
            return False
        eps = self.layer_norm_in.eps
        temp = self.layer_stack[0].slf_attn.temperature
        return all(l_.slf_attn.layer_norm.eps == eps and l_.pos_ffn.layer_norm.eps == eps and
                   l_.slf_attn.temperature == temp for l_ in self.layer_stack)

    def _side_streams(self, device, k):
        key = str(device)
        pool = self._streams.setdefault(key, [])
        while len(pool) < k:
            pool.append(torch.cuda.Stream(device=device))
        return pool[:k]

    def _run_chain(self, x, out, pk, n0, n1, t, lengths, return_attns, attns):
        """The whole encoder stack for clips [n0, n1) on the current stream; writes rows of `out` (fp32 [N*T, d])."""
        nc = n1 - n0
        xs = x[n0 * t:n1 * t]
        lens_c = None if lengths is None else lengths[n0:n1]
        pe = self.positional_encoding.pe[0]
        last = len(self.layer_stack) - 1
        x16 = ops.cast_enc16(xs)
        # encoder.py:53-55 — LN(linear_in(x)) + PE in one launch ; no pad mask at this point
        x32, x16 = ops.linear_ln(x16, pk.w_in, self.layer_norm_in.weight.detach(), self.layer_norm_in.bias.detach(),
                               bias=self.linear_in.bias.detach(), pe=pe, T=t, eps=self.layer_norm_in.eps,
                               out_f32=out[n0 * t:n1 * t] if last < 0 else None)
        for li, (lyr, w) in enumerate(zip(self.layer_stack, pk.layers)):
            a, f = lyr.slf_attn, lyr.pos_ffn
            if return_attns:  # attention maps requested: unfused projection + attention kernel that writes them
                qkv16, _ = ops.gemm(x16, w["wqkv"], bias=w["bqkv"], out_bf16=True)
                att16, probs = ops.attention(qkv16, nc, t, self.n_head, self.d_k, lengths=lens_c,
                                             want_probs=True, scale=1.0 / a.temperature)
                attns.append(probs)
            else:
                att16 = ops.qkv_attention(x16, w["wheads"], w["bheads"], nc, t, self.n_head, self.d_k,
                                          lengths=lens_c, scale=1.0 / a.temperature)
            # attention.py:57-58 — fc + LayerNorm(out + residual), then `*= non_pad_mask` (encoder.py:86)
            x32, x16 = ops.linear_ln(att16, w["wfc"], a.layer_norm.weight.detach(), a.layer_norm.bias.detach(),
                                   bias=a.fc.bias.detach(), residual=x32, lengths=lens_c, T=t, eps=a.layer_norm.eps)
            # module.py:49-51 — w_2(relu(w_1(x))) + LayerNorm(out + x), then `*= non_pad_mask` (encoder.py:89)
            h16, _ = ops.gemm(x16, w["w1"], bias=f.w_1.bias.detach(), relu=True, out_bf16=True)
            x32, x16 = ops.linear_ln(h16, w["w2"], f.layer_norm.weight.detach(), f.layer_norm.bias.detach(),
                                   bias=f.w_2.bias.detach(), residual=x32, lengths=lens_c, T=t, eps=f.layer_norm.eps,
                                   want_bf16=li != last, out_f32=out[n0 * t:n1 * t] if li == last else None)

    def forward(self, padded_input, input_lengths, return_attns=False):
        """padded_input: N x T x d_input (fp32, CUDA); input_lengths: N ints -> (enc_output N x T x d_model,)"""
        self._check_config()
        if not padded_input.is_cuda:
            raise RuntimeError("Encoder (libsblk) runs on a B200 CUDA device only; no CPU fallback exists")
        n, t, d_in = padded_input.shape
        if d_in != self.d_input:
            raise RuntimeError(f"Encoder: last dim {d_in} != d_input {self.d_input}")
        if t > self.pe_maxlen:
            raise RuntimeError(f"Encoder: T={t} exceeds pe_maxlen={self.pe_maxlen}")
        if t > 128:
            raise RuntimeError(f"Encoder (libsblk): T={t} > 128 frames per clip is not implemented (attention tiles hold "
                               f"one clip; the reference allows up to pe_maxlen={self.pe_maxlen}); no fallback path")
        lens = [int(v) for v in input_lengths]
        if len(lens) != n:
            raise RuntimeError(f"Encoder: {len(lens)} input_lengths for batch {n}")
        if n == 0:   # empty batch: nothing to launch (the reference returns empty tensors as well)
            out = padded_input.new_zeros((0, t, self.d_model), dtype=torch.float32)
            return (out, [padded_input.new_zeros((0, t, t)) for _ in self.layer_stack]) if return_attns else (out,)
        if self.training:
            # model.train(): dropout active, every block a torch.autograd.Function backed by libsblk (training.py)
            self._check_train_config(t, return_attns)
            from . import training
            return training.encoder_forward_train(self, padded_input.float(), lens)
        return self._forward_eval(padded_input, lens, return_attns)

    def _forward_eval(self, padded_input, lens, return_attns=False, *, x16=None, cluster_size=None,
                      groups_per_cluster=None, resident_counter=None):
        """The evaluation forward of checked arguments.  The CUDA-graph plans (runner.py) pass the 16-bit copy of the
        input they already hold (`x16` [N*T, d_input]: no cast launch, `padded_input` only gives the shape; one-launch
        stack only), the cluster size and clip groups per cluster of the one-launch stack (default: stack_cluster_size /
        stack_groups_per_cluster) and the `resident_counter` of ops.gate_wait."""
        cl = self.stack_cluster_size if cluster_size is None else cluster_size
        gpc = self.stack_groups_per_cluster if groups_per_cluster is None else groups_per_cluster
        n, t, d_in = padded_input.shape
        m = n * t
        x = padded_input.detach()
        if x.dtype != torch.float32:
            x = x.float()
        x = x.contiguous().view(m, d_in)
        with torch.cuda.device(x.device):
            pk = self._get_packed()
            lengths = None
            if any(v < t for v in lens):  # all-keep masks (every reference call site) cost nothing
                ck = (x.device, tuple(lens))  # staged once per distinct lengths vector (CUDA-graph capturable)
                lengths = self._len_cache.get(ck)
                if lengths is None:
                    if len(self._len_cache) > 64:
                        self._len_cache.clear()
                    lengths = torch.tensor(lens, dtype=torch.int32, device=x.device)
                    self._len_cache[ck] = lengths
            out = torch.empty((m, self.d_model), dtype=torch.float32, device=x.device)
            attns = []
            # Clips are independent through the whole stack (attention is per clip, LayerNorm per token), and at
            # BASELINE batch sizes every kernel of the stack is latency-bound (~3 us fixed cost x 43 launches), so
            # the batch is split into a few clip groups whose kernel chains run concurrently on side streams
            # (fork / join with events: capturable into a CUDA graph as parallel branches).
            if self._use_fused_stack(n, t, return_attns):
                # the whole stack as ONE launch: a cluster per clip group, no inter-group synchronisation
                stk = pk.stacked
                scale = 1.0 / self.layer_stack[0].slf_attn.temperature
                x16 = ops.cast_enc16(x) if x16 is None else x16
                g_clips = max(1, 128 // t)
                groups = -(-n // g_clips)
                if groups > self.fused_stack_max_groups:
                    # large batch: sub-batches of whole clip groups through the same kernel, two launches in flight
                    # (2 x 8 clusters of 8 CTAs = 128 SMs); cluster sizes 8 / 16 are bit-identical, so is any chunking
                    step = max(1, int(self.chunk_groups)) * g_clips
                    main = torch.cuda.current_stream()
                    side = self._side_streams(x.device, 1)[0]
                    fork = torch.cuda.Event()
                    fork.record(main)
                    side.wait_event(fork)
                    for ci, n0 in enumerate(range(0, n, step)):
                        n1 = min(n, n0 + step)
                        with torch.cuda.stream(side if ci & 1 else main):
                            ops.encoder_stack(x16[n0 * t:n1 * t], stk, n1 - n0, t,
                                              lengths=None if lengths is None else lengths[n0:n1], scale=scale,
                                              eps=self.layer_norm_in.eps, out=out[n0 * t:n1 * t],
                                              cluster_size=cl or 8)
                    join = torch.cuda.Event()
                    join.record(side)
                    main.wait_event(join)
                    return (out.view(n, t, self.d_model),)
                if self.split_clusters and cl == 0 and 7 < groups <= 11:
                    # Only 7 clusters of 16 CTAs are co-resident on a B200, and 16-CTA clusters are the faster ones (each
                    # CTA streams half the weights).  The first 7 clip groups run as 16-CTA clusters; the remaining 1-4
                    # groups run at the same time, on a side stream, as 8-CTA clusters in the SMs the big clusters leave
                    # free.  Both cluster sizes are bit-identical (tests), so nothing depends on the split.
                    n0 = 7 * g_clips
                    main = torch.cuda.current_stream()
                    side = self._side_streams(x.device, 1)[0]
                    ev = torch.cuda.Event()
                    ev.record(main)
                    side.wait_event(ev)
                    with torch.cuda.stream(side):
                        ops.encoder_stack(x16[n0 * t:], stk, n - n0, t, lengths=None if lengths is None else lengths[n0:],
                                          scale=scale, eps=self.layer_norm_in.eps, out=out[n0 * t:], cluster_size=8)
                        ev2 = torch.cuda.Event()
                        ev2.record(side)
                    ops.encoder_stack(x16[:n0 * t], stk, n0, t, lengths=None if lengths is None else lengths[:n0],
                                      scale=scale, eps=self.layer_norm_in.eps, out=out[:n0 * t], cluster_size=16)
                    main.wait_event(ev2)
                else:
                    ops.encoder_stack(x16, stk, n, t, lengths=lengths, scale=scale, eps=self.layer_norm_in.eps, out=out,
                                      cluster_size=cl, resident_counter=resident_counter,
                                      groups_per_cluster=gpc if cl else 1)
                return (out.view(n, t, self.d_model),)
            if x16 is not None:
                raise RuntimeError("Encoder: a 16-bit input copy is only read by the one-launch stack")
            groups = 1 if return_attns else max(1, min(self.parallel_chains, n // 4))
            if groups == 1:
                self._run_chain(x, out, pk, 0, n, t, lengths, return_attns, attns)
            else:
                main = torch.cuda.current_stream()
                side = self._side_streams(x.device, groups - 1)
                fork = torch.cuda.Event()
                fork.record(main)
                bounds = [(g * n) // groups for g in range(groups + 1)]
                for g in range(groups):
                    st = main if g == 0 else side[g - 1]
                    if g > 0:
                        st.wait_event(fork)
                    with torch.cuda.stream(st):
                        self._run_chain(x, out, pk, bounds[g], bounds[g + 1], t, lengths, False, attns)
                for g in range(1, groups):
                    ev = torch.cuda.Event()
                    ev.record(side[g - 1])
                    main.wait_event(ev)
            x32 = out
        enc_output = x32.view(n, t, self.d_model)
        if return_attns:
            return enc_output, attns
        return enc_output,
