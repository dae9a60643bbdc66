"""Drop-in replacement for the reference SBL bidirectional decoder (SURVEY.md §8f.1): greedy decoding and the
teacher-forced forward of `transformer/decoder.py` on libsblk kernels.

`Decoder` has the reference constructor signature, attributes and state-dict keys (`tgt_word_emb`, `positional_encoding`,
`layer_first_{l2r,r2l}`, `layer_stack_{l2r,r2l}.{i}.{slf_attn,enc_attn,pos_ffn}.*`, `tgt_word_prj_{l2r,r2l}`), so a
reference checkpoint loads unchanged and `Transformer.forward` / `recognize` (transformer/transformer.py:22-69) call it
as they call the reference class.  Submodules are parameter holders; the arithmetic is:

  per decode step (prefix length L = step + 1, both directions; the reference recomputes the whole prefix each step and
  so does this — the synchronous bidirectional mixing changes every earlier position's hidden state when L grows):
    embedding + positional encoding                                   sblk_embed_pe_fwd
    6 x { QKV GEMM -> self-attention (subsequent mask in the FIRST layer only, decoder.py:329-331 vs :349-357)
          -> fc GEMM + residual + LayerNorm -> Q GEMM -> attention over the CACHED encoder keys / values
          -> fc GEMM + residual + LayerNorm -> w_1 GEMM + ReLU -> w_2 GEMM + residual + LayerNorm }   (tcgen05 GEMMs)
    after the first layer and after every later layer: l2r' = l2r + flip(r2l); r2l' = r2l + flip(l2r')   sblk_bidir_mix_fwd
    logits = tgt_word_prj(last position); argmax / teacher token appended (host glue, as in the reference)

  The encoder-side K / V projections of all 12 decoder layers are computed ONCE per call (the reference recomputes them
  at each of the 16 steps).  Operands are enc16 (fp16) with fp32 accumulation, LayerNorm, softmax and residual streams.

Training: in `model.train()`, `forward` runs the same 16 steps as autograd Functions over libsblk forward and backward
kernels (training.decoder_forward_train, DESIGN.md §9): the logits reach every decoder parameter and the encoder
outputs.  It reads the live parameters (no packed cache), so an optimizer step is seen by the next call.  Greedy
decoding (`recognize_beam`) stays an evaluation feature.
"""
from __future__ import annotations

import random

import torch
import torch.nn as nn

from . import _lib, ops
from .encoder import PositionalEncoding, _FeedForwardParams, _SelfAttentionParams

IGNORE_ID = -1        # reference config.py:28


def pad_list(xs, pad_value):
    """reference transformer/utils.py:1-9 — note the hard-coded max_len = 16."""
    n_batch = len(xs)
    max_len = 16
    pad = xs[0].new(n_batch, max_len, *xs[0].size()[1:]).fill_(pad_value)
    for i in range(n_batch):
        pad[i, :xs[i].size(0)] = xs[i]
    return pad


class DecoderLayer(nn.Module):
    """Holder with the reference DecoderLayer attribute names (decoder.py:388-394)."""

    def __init__(self, d_model, d_inner, n_head, d_k, d_v, dropout=0.1):
        super().__init__()
        self.slf_attn = _SelfAttentionParams(n_head, d_model, d_k, d_v, dropout=dropout)
        self.enc_attn = _SelfAttentionParams(n_head, d_model, d_k, d_v, dropout=dropout)
        self.pos_ffn = _FeedForwardParams(d_model, d_inner, dropout=dropout)


class Decoder(nn.Module):
    """Drop-in for reference Decoder (transformer/decoder.py:15-386)."""

    def __init__(self, sos_id, eos_id, n_tgt_vocab, d_word_vec, n_layers, n_head, d_k, d_v, d_model, d_inner, dropout=0.1,
                 tgt_emb_prj_weight_sharing=True, pe_maxlen=5000):
        super().__init__()
        self.sos_id = sos_id
        self.eos_id = eos_id
        self.n_tgt_vocab = n_tgt_vocab
        self.d_word_vec = d_word_vec
        self.n_layers = n_layers
        self.n_head = n_head
        self.d_k = d_k
        self.d_v = d_v
        self.d_model = d_model
        self.d_inner = d_inner
        self.dropout = dropout
        self.tgt_emb_prj_weight_sharing = tgt_emb_prj_weight_sharing
        self.pe_maxlen = pe_maxlen

        self.tgt_word_emb = nn.Embedding(n_tgt_vocab, d_word_vec)
        self.positional_encoding = PositionalEncoding(d_model, max_len=pe_maxlen)
        self.dropout = nn.Dropout(dropout)
        self.layer_first_l2r = DecoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout)
        self.layer_stack_l2r = nn.ModuleList([DecoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout)
                                              for _ in range(self.n_layers - 1)])
        self.layer_first_r2l = DecoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout)
        self.layer_stack_r2l = nn.ModuleList([DecoderLayer(d_model, d_inner, n_head, d_k, d_v, dropout=dropout)
                                              for _ in range(self.n_layers - 1)])
        self.x_logit_scale = 1.
        self.tgt_word_prj_l2r = nn.Linear(512, 58, bias=False)     # 58 = 56 + <sos> + <eos>, hard-coded like the reference
        self.tgt_word_prj_r2l = nn.Linear(512, 58, bias=False)
        self.maxlen = 16
        self._packed = None
        self._plans = {}
        self.use_cuda_graphs = True     # decode steps replayed as CUDA graphs per (batch, encoder length); False = eager
        self.fused_ln = None            # ops.linear_ln strategy: None = by token count, True = always the cluster kernel
        self.two_streams = True         # the two directions of a layer run concurrently (they only meet in the mixing)
        self._side = {}

    def __getstate__(self):
        st = self.__dict__.copy()
        st["_packed"] = None
        st["_plans"] = {}
        st["_side"] = {}
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self.__dict__.setdefault("_plans", {})
        self.__dict__.setdefault("use_cuda_graphs", True)
        self.__dict__.setdefault("fused_ln", None)
        self.__dict__.setdefault("two_streams", True)
        self.__dict__.setdefault("_side", {})

    # ------------------------------------------------------------------------------------------
    def preprocess(self, padded_input):
        """reference decoder.py:62-77 + utils.pad_list: drop IGNORE_ID entries, <sos> + y / y + <eos>, both padded to 16
        columns with eos.  Same result as the reference's per-utterance Python loops, as a handful of tensor ops (the
        loops cost ~0.1 ms per utterance on the GPU: 60 ms at batch 512)."""
        y = padded_input
        n, w = y.shape
        keep = y != IGNORE_ID
        lens = keep.sum(1)
        if int(lens.max()) + 1 > 16:       # the reference's pad_list cannot hold it either (max_len = 16)
            raise RuntimeError("Decoder.preprocess: target longer than 15 tokens does not fit pad_list's max_len = 16")
        order = torch.argsort((~keep).to(torch.int8), dim=1, stable=True)      # kept tokens first, original order
        ys = torch.gather(y, 1, order)
        if w < 16:
            ys = torch.cat([ys, ys.new_full((n, 16 - w), self.eos_id)], 1)
        ys = ys[:, :16]
        cols = torch.arange(16, device=y.device)[None, :]
        ys_out_pad = torch.where(cols < lens[:, None], ys, ys.new_full((), self.eos_id))
        shifted = torch.cat([ys.new_full((n, 1), self.sos_id), ys[:, :15]], 1)
        ys_in_pad = torch.where(cols <= lens[:, None], shifted, ys.new_full((), self.eos_id))
        return ys_in_pad, ys_out_pad

    # ------------------------------------------------------------------------------------------
    def _cache_key(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def invalidate_packed(self):
        self._packed = None
        self._plans = {}

    def _check(self, enc, train_forward=False):
        if self.training and not train_forward:
            raise RuntimeError("Decoder (libsblk): greedy decoding (recognize_beam) is an evaluation feature; call "
                               "model.eval() first (in training mode only forward is available)")
        if self.d_model != 512 or self.d_k != 64 or self.d_v != 64 or self.n_head != 8 or self.d_word_vec != 512:
            raise RuntimeError("Decoder (libsblk): only d_model = d_word_vec = 512, 8 heads of 64 are implemented")
        if not enc.is_cuda:
            raise RuntimeError("Decoder (libsblk) runs on a B200 CUDA device only; no CPU fallback exists")
        t_max = 64 if train_forward else 128      # the training attention kernel holds <= 64 keys
        if enc.dim() != 3 or enc.size(2) != 512 or enc.size(1) > t_max:
            raise RuntimeError(f"Decoder (libsblk): encoder outputs must be [N, T <= {t_max}, 512]"
                               f"{' in training' if train_forward else ''}, got {tuple(enc.shape)}")

    def _pack_layer(self, lyr):
        a, c, f = lyr.slf_attn, lyr.enc_attn, lyr.pos_ffn
        cat = lambda ts: torch.cat([t.detach() for t in ts], 0).contiguous()      # noqa: E731
        e16 = ops.cast_enc16
        return dict(
            wqkv=e16(cat([a.w_qs.weight, a.w_ks.weight, a.w_vs.weight])), bqkv=cat([a.w_qs.bias, a.w_ks.bias, a.w_vs.bias]),
            wfc=e16(a.fc.weight.detach().contiguous()), bfc=a.fc.bias.detach(), g1=a.layer_norm.weight.detach(),
            be1=a.layer_norm.bias.detach(), eps1=a.layer_norm.eps, scale1=1.0 / a.temperature,
            wq=e16(c.w_qs.weight.detach().contiguous()), bq=c.w_qs.bias.detach(),
            wkv=e16(cat([c.w_ks.weight, c.w_vs.weight])), bkv=cat([c.w_ks.bias, c.w_vs.bias]),
            wfc2=e16(c.fc.weight.detach().contiguous()), bfc2=c.fc.bias.detach(), g2=c.layer_norm.weight.detach(),
            be2=c.layer_norm.bias.detach(), eps2=c.layer_norm.eps, scale2=1.0 / c.temperature,
            w1=e16(f.w_1.weight.detach().contiguous()), b1=f.w_1.bias.detach(),
            w2=e16(f.w_2.weight.detach().contiguous()), b2=f.w_2.bias.detach(), g3=f.layer_norm.weight.detach(),
            be3=f.layer_norm.bias.detach(), eps3=f.layer_norm.eps)

    def _get_packed(self):
        key = self._cache_key()
        pk = self._packed
        if pk is not None and pk["key"] == key:
            return pk
        dev = self.tgt_word_emb.weight.device
        pk = {"key": key}
        pk["l2r"] = [self._pack_layer(self.layer_first_l2r)] + [self._pack_layer(l_) for l_ in self.layer_stack_l2r]
        pk["r2l"] = [self._pack_layer(self.layer_first_r2l)] + [self._pack_layer(l_) for l_ in self.layer_stack_r2l]
        for d, prj in (("l2r", self.tgt_word_prj_l2r), ("r2l", self.tgt_word_prj_r2l)):
            w = torch.zeros((64, 512), dtype=torch.float32, device=dev)      # 58 -> 64 rows (tcgen05 N granularity)
            w[:prj.weight.shape[0]] = prj.weight.detach()
            pk["prj_" + d] = ops.cast_enc16(w)
        pk["emb"] = self.tgt_word_emb.weight.detach().float().contiguous()
        pk["pe"] = self.positional_encoding.pe[0]
        self._packed = pk
        return pk

    # ------------------------------------------------------------------------------------------
    def _layer(self, w, x32, x16, n, L, kv16, t_enc, causal):
        """One DecoderLayer.forward (decoder.py:396-408) on [n*L, 512] rows; kv16 = cached encoder K | V [n*t_enc, 1024]."""
        lib = _lib.load()
        e16 = ops.enc16_dtype()
        dev = x32.device
        st = torch.cuda.current_stream().cuda_stream
        # self-attention over the decoded prefix
        qkv16, _ = ops.gemm(x16, w["wqkv"], bias=w["bqkv"], out_bf16=True)
        att16 = torch.empty((n * L, 512), dtype=e16, device=dev)
        _lib.check(lib.sblk_xattention_fwd(qkv16.data_ptr(), qkv16.data_ptr() + 512 * 2, qkv16.data_ptr() + 1024 * 2,
                                           att16.data_ptr(), None, 1536, 1536, 1536, 512, n, L, L, 8, 1 if causal else 0,
                                           w["scale1"], st), "sblk_xattention_fwd")
        x32, x16 = ops.linear_ln(att16, w["wfc"], w["g1"], w["be1"], bias=w["bfc"], residual=x32, T=L, eps=w["eps1"],
                                 fused=self.fused_ln)
        # decoder-encoder attention (dec_enc_attn_mask=None at every reference call site of the greedy / sampled loops)
        q16, _ = ops.gemm(x16, w["wq"], bias=w["bq"], out_bf16=True)
        att16 = torch.empty((n * L, 512), dtype=e16, device=dev)
        _lib.check(lib.sblk_xattention_fwd(q16.data_ptr(), kv16.data_ptr(), kv16.data_ptr() + 512 * 2, att16.data_ptr(),
                                           None, 512, 1024, 1024, 512, n, L, t_enc, 8, 0, w["scale2"], st),
                   "sblk_xattention_fwd")
        x32, x16 = ops.linear_ln(att16, w["wfc2"], w["g2"], w["be2"], bias=w["bfc2"], residual=x32, T=L, eps=w["eps2"],
                                 fused=self.fused_ln)
        # position-wise feed-forward
        h16, _ = ops.gemm(x16, w["w1"], bias=w["b1"], relu=True, out_bf16=True)
        return ops.linear_ln(h16, w["w2"], w["g3"], w["be3"], bias=w["b2"], residual=x32, T=L, eps=w["eps3"],
                             fused=self.fused_ln)

    def _encoder_kv(self, pk, enc):
        """K | V projections of the encoder outputs for every decoder layer of both directions (once per call)."""
        n, t, _ = enc.shape
        enc16 = ops.cast_enc16(enc.detach().float().contiguous().view(n * t, 512))
        return {d: [ops.gemm(enc16, w["wkv"], bias=w["bkv"], out_bf16=True)[0] for w in pk[d]] for d in ("l2r", "r2l")}

    def _step(self, pk, kv, ys_l2r, ys_r2l, L, t_enc):
        """All layers for the prefixes ys[:, :L] (ys: int64 [N, >= L] token buffers, any row pitch) ->
        (logits_l2r, logits_r2l) fp32 [N, 58] of the LAST position."""
        lib = _lib.load()
        n = ys_l2r.shape[0]
        dev = ys_l2r.device
        e16 = ops.enc16_dtype()
        st = torch.cuda.current_stream().cuda_stream
        x = {}
        for d, ys in (("l2r", ys_l2r), ("r2l", ys_r2l)):
            x32 = torch.empty((n * L, 512), dtype=torch.float32, device=dev)
            x16 = torch.empty((n * L, 512), dtype=e16, device=dev)
            _lib.check(lib.sblk_embed_pe_fwd(ys.data_ptr(), ys.stride(0), pk["emb"].data_ptr(), pk["pe"].data_ptr(),
                                             x32.data_ptr(), x16.data_ptr(), n * L, L, 512, pk["emb"].shape[0],
                                             float(self.x_logit_scale), st), "sblk_embed_pe_fwd")
            x[d] = (x32, x16)
        main = torch.cuda.current_stream(dev)
        side = None
        if self.two_streams:
            side = self._side.get(str(dev))
            if side is None:
                side = self._side[str(dev)] = torch.cuda.Stream(device=dev)
        for li in range(self.n_layers):
            if side is None:
                for d in ("l2r", "r2l"):
                    x[d] = self._layer(pk[d][li], x[d][0], x[d][1], n, L, kv[d][li], t_enc, causal=(li == 0))
            else:   # fork: r2l on the side stream next to l2r; join before the mixing (capturable as graph branches)
                fork = torch.cuda.Event()
                fork.record(main)
                side.wait_event(fork)
                old = x["r2l"]      # allocated on `main`, read on `side`: kept alive until main has joined, so that its
                #                     memory cannot be handed to a main-stream allocation while the side branch reads it
                with torch.cuda.stream(side):
                    new_r2l = self._layer(pk["r2l"][li], old[0], old[1], n, L, kv["r2l"][li], t_enc, causal=(li == 0))
                    join = torch.cuda.Event()
                    join.record(side)
                x["l2r"] = self._layer(pk["l2r"][li], x["l2r"][0], x["l2r"][1], n, L, kv["l2r"][li], t_enc,
                                       causal=(li == 0))
                main.wait_event(join)
                x["r2l"] = new_r2l
                del old
            a32, b32 = torch.empty_like(x["l2r"][0]), torch.empty_like(x["r2l"][0])
            a16, b16 = torch.empty_like(x["l2r"][1]), torch.empty_like(x["r2l"][1])
            _lib.check(lib.sblk_bidir_mix_fwd(x["l2r"][0].data_ptr(), x["r2l"][0].data_ptr(), a32.data_ptr(), b32.data_ptr(),
                                              a16.data_ptr(), b16.data_ptr(), n, L, 512, st), "sblk_bidir_mix_fwd")
            x["l2r"], x["r2l"] = (a32, a16), (b32, b16)
        out = []
        for d in ("l2r", "r2l"):
            last = x[d][1].view(n, L, 512)[:, -1].contiguous()              # dec_output[:, -1] (decoder.py:364-365)
            _, logits = ops.gemm(last, pk["prj_" + d], out_f32=True)
            out.append(logits[:, :self.tgt_word_prj_l2r.weight.shape[0]])
        return out

    # ------------------------------------------------------------------------------------------
    # ------------------------------------------------------------------------------------------
    def _plan(self, pk, n, t_enc, dev):
        """CUDA graphs of the 16 decode steps for one (batch, encoder length): a step is ~150 short launches, so eager
        decoding is host-bound (38 ms per 16-clip call against ~8 ms of GPU work).  Static buffers: encoder outputs,
        the 12 cached K|V projections, both token buffers [N, 17] and the per-step logits; graph L recomputes the prefix
        of length L.  All graphs share one memory pool (they never run concurrently).  The settings the captured steps
        depend on (fused_ln, two_streams) are part of the key, so changing one takes effect at the next call."""
        key = (n, t_enc, str(dev), pk["key"], self.fused_ln, self.two_streams)
        plan = self._plans.get(key)
        if plan is not None:
            return plan
        if len(self._plans) >= 4:
            self._plans.clear()
        plan = {"enc": torch.zeros((n, t_enc, 512), dtype=torch.float32, device=dev),
                "ys_l2r": torch.full((n, self.maxlen + 1), self.sos_id, dtype=torch.long, device=dev),
                "ys_r2l": torch.full((n, self.maxlen + 1), self.sos_id, dtype=torch.long, device=dev),
                "logits": [], "graphs": [], "stream": torch.cuda.Stream(device=dev)}
        stream = plan["stream"]
        stream.wait_stream(torch.cuda.current_stream(dev))
        prev_pdl = ops.set_pdl(True)        # consecutive tcgen05 launches overlap prologue / tail inside the graphs
        try:
            self._capture(plan, pk, n, t_enc, stream)
        finally:
            ops.set_pdl(prev_pdl)
        torch.cuda.current_stream(dev).wait_stream(stream)
        self._plans[key] = plan
        return plan

    def _capture(self, plan, pk, n, t_enc, stream):
        with torch.cuda.stream(stream):
            kv = self._encoder_kv(pk, plan["enc"])                       # warm-up (sizes kernels), then captured
            self._step(pk, kv, plan["ys_l2r"], plan["ys_r2l"], 2, t_enc)
            stream.synchronize()
            pool = torch.cuda.graph_pool_handle()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool, stream=stream):
                plan["kv"] = self._encoder_kv(pk, plan["enc"])
            plan["kv_graph"] = g
            for L in range(1, self.maxlen + 1):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool, stream=stream):
                    lg = self._step(pk, plan["kv"], plan["ys_l2r"], plan["ys_r2l"], L, t_enc)
                    lg = (lg[0].clone(), lg[1].clone())
                plan["graphs"].append(g)
                plan["logits"].append(lg)

    def _decode(self, encoder_outputs, next_tokens, want_logits):
        """Shared loop of recognize_beam / forward: next_tokens(i, logits_l2r, logits_r2l) -> ([N] int64, [N] int64)."""
        self._check(encoder_outputs)
        dev = encoder_outputs.device
        keep = ([], [])
        with torch.no_grad(), torch.cuda.device(dev):
            pk = self._get_packed()
            n, t_enc = encoder_outputs.size(0), encoder_outputs.size(1)
            if self.use_cuda_graphs:
                plan = self._plan(pk, n, t_enc, dev)
                plan["enc"].copy_(encoder_outputs.detach().float())
                plan["ys_l2r"].fill_(self.sos_id)
                plan["ys_r2l"].fill_(self.sos_id)
                plan["kv_graph"].replay()
                ys_l2r, ys_r2l = plan["ys_l2r"], plan["ys_r2l"]
            else:
                kv = self._encoder_kv(pk, encoder_outputs)
                ys_l2r = torch.full((n, self.maxlen + 1), self.sos_id, dtype=torch.long, device=dev)
                ys_r2l = torch.full((n, self.maxlen + 1), self.sos_id, dtype=torch.long, device=dev)
            for i in range(self.maxlen):
                if self.use_cuda_graphs:
                    plan["graphs"][i].replay()
                    pred_l2r, pred_r2l = plan["logits"][i]
                else:
                    pred_l2r, pred_r2l = self._step(pk, kv, ys_l2r, ys_r2l, i + 1, t_enc)
                if want_logits:
                    keep[0].append(pred_l2r.clone())
                    keep[1].append(pred_r2l.clone())
                nxt_l2r, nxt_r2l = next_tokens(i, pred_l2r, pred_r2l)
                ys_l2r[:, i + 1] = nxt_l2r
                ys_r2l[:, i + 1] = nxt_r2l
            ys_l2r, ys_r2l = ys_l2r.clone(), ys_r2l.clone()
        if want_logits:
            return ys_l2r, ys_r2l, torch.stack(keep[0], 1), torch.stack(keep[1], 1)
        return ys_l2r, ys_r2l, None, None

    def recognize_beam(self, encoder_outputs):
        """Greedy bidirectional decoding, reference decoder.py:301-385 -> (ys_l2r, ys_r2l) int64 [N, 1 + 16]."""
        ys_l2r, ys_r2l, _, _ = self._greedy(encoder_outputs, want_logits=False)
        return ys_l2r, ys_r2l

    def _greedy(self, encoder_outputs, want_logits):
        """-> (ys_l2r, ys_r2l, logits_l2r | None, logits_r2l | None), logits fp32 [N, 16, 58] (tests: margin analysis)."""
        return self._decode(encoder_outputs, lambda i, a, b: (a.argmax(-1), b.argmax(-1)), want_logits)

    def forward(self, padded_input_l2r, padded_input_r2l, encoder_outputs, encoder_input_lengths, return_attns=False):
        """Sampled teacher forcing, reference decoder.py:79-191: 16 steps, each feeding either the model's own argmax or
        the gold token (`random.random() > 0.5`, the reference's coin) -> (logits_l2r [N,16,58], gold_l2r, logits_r2l,
        gold_r2l).  In training mode the logits are autograd-connected (training.decoder_forward_train)."""
        if self.training:
            if return_attns:
                raise RuntimeError("Decoder (libsblk): return_attns is not implemented in training mode")
            self._check(encoder_outputs, train_forward=True)
            from .training import decoder_forward_train
            return decoder_forward_train(self, padded_input_l2r, padded_input_r2l, encoder_outputs)
        ys_in_pad_l2r, ys_out_pad_l2r = self.preprocess(padded_input_l2r)
        ys_in_pad_r2l, ys_out_pad_r2l = self.preprocess(padded_input_r2l)
        dev = encoder_outputs.device

        def next_tokens(i, pred_l2r, pred_r2l):
            is_teacher = random.random() > 0.5          # decoder.py:176 (the flag's name is the reference's)
            if is_teacher:
                return pred_l2r.argmax(-1), pred_r2l.argmax(-1)
            return ys_out_pad_l2r[:, i].to(dev), ys_out_pad_r2l[:, i].to(dev)

        _, _, out_l2r, out_r2l = self._decode(encoder_outputs, next_tokens, want_logits=True)
        return out_l2r, ys_out_pad_l2r, out_r2l, ys_out_pad_r2l
