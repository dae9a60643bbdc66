"""`-m gpu` parity against the UNMODIFIED reference running on the same B200 (oracle/_ref, staged by
oracle/fetch_ref.py): the reference's own `Transformer.recognize` / `Transformer.forward` and SBL bidirectional decoder
run ON TOP of the drop-in visual frontend + encoder (dropin.patch_reference), next to the all-reference fp32 model
(cuDNN / cuBLAS fp32, TF32 off) on identical synthetic inputs and weights.

  * greedy-decode token parity on 1,000 structured clips (BASELINE.json north_star; transformer/transformer.py:45-69,
    transformer/decoder.py:301-385), margin-aware, with the bf16-rounding control measured in the same run
  * teacher-forced `Transformer.forward` logits (transformer/transformer.py:22-43, decoder.py:79-191)
  * stage-by-stage error budget (stem, every ResNet layer, features, every encoder layer)

The tests that need only the reference's frontend and encoder (the error budget, the always-on dropout mask, the
decoder's CUDA-graph steps) run them as oracle/reference_modules.py restates them, with the forward pinned to the
reference's own outputs by tests/test_oracle_golden.py, so they need no staged files; the others skip where
oracle/_ref is not staged.

Results are also written to gpurun_out/r02_*.json (copied to profiles/ by the builder).
"""
import json
import os
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT_DIR = os.path.join(ROOT, "gpurun_out")
T = 29


def rel_fro(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _dump(name, obj):
    os.makedirs(OUT_DIR, exist_ok=True)
    with open(os.path.join(OUT_DIR, name), "w") as f:
        json.dump(obj, f, indent=1)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    assert ops.init() > 0
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def models(dev):
    """(reference namespace, all-reference fp32 model on cuda, reference Transformer + decoder on the drop-ins)."""
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import dropin, synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder as B200Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading as B200Lipreading
    if not ref_runtime.available():
        pytest.skip("oracle/_ref not staged (python oracle/fetch_ref.py needs /root/reference)")
    ref_runtime.fp32_exact()
    R = ref_runtime.load_reference("sbl")
    sd = dict(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, 6, prefix="encoder."))
    ref = ref_runtime.build_sbl_reference(R, sd).to(dev).eval()
    assert type(ref.visual_frontend).__module__ == "transformer.video_frontend"
    with dropin.patched_reference(R.dir):
        # exactly what train.py:58-69 / test.py:86-97 do, with the patched names in place
        import transformer.encoder as tenc
        import transformer.transformer as ttr
        torch.manual_seed(7)
        enc = tenc.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        dec = R.Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                        pe_maxlen=5000)
        ours = ttr.Transformer(enc, dec, None)
    assert isinstance(ours.visual_frontend, B200Lipreading) and isinstance(ours.encoder, B200Encoder)
    assert type(ours.decoder).__module__ == "transformer.decoder"
    ours.load_state_dict(ref.state_dict())       # the 537-key reference state dict loads unchanged
    ours = ours.to(dev).eval()
    ours.visual_frontend.always_on_dropout = False
    return R, ref, ours


@pytest.fixture(scope="module")
def fe_enc(dev):
    """The reference frontend + 6-layer encoder in fp32 (oracle/reference_modules.py) next to the drop-in frontend +
    encoder, on cuda, with the synthetic weights of `models`; eval mode, the drop-in's always-on dropout off."""
    import types
    from oracle import ref_runtime, reference_modules as RM
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder as B200Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading as B200Lipreading
    ref_runtime.fp32_exact()
    fe_sd, enc_sd = synth.frontend_state_dict(1), synth.encoder_state_dict(2, 6)
    m = types.SimpleNamespace(fe_ref=RM.Lipreading(), enc_ref=RM.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1),
                              fe=B200Lipreading(), enc=B200Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1))
    for mod, sd in ((m.fe_ref, fe_sd), (m.enc_ref, enc_sd), (m.fe, fe_sd), (m.enc, enc_sd)):
        mod.load_state_dict(sd)
        mod.to(dev).eval()
    m.fe.always_on_dropout = False
    return m


class _Tap:
    """Records the outputs of a module (forward hook)."""

    def __init__(self, module, pick=lambda o: o):
        self.outs = []
        self._h = module.register_forward_hook(lambda m, i, o: self.outs.append(pick(o).detach()))

    def close(self):
        self._h.remove()


def _recognize(model, x, enc_override=None):
    """model.recognize(x) (or the decoder's greedy search on `enc_override`) -> (l2r, r2l, enc_out, logits_l2r, logits_r2l),
    logits = [16 x [N,58]] as the reference's output projections produced them (decoder.py:368-369)."""
    taps = (_Tap(model.decoder.tgt_word_prj_l2r), _Tap(model.decoder.tgt_word_prj_r2l),
            _Tap(model.encoder, pick=lambda o: o[0]))
    try:
        if enc_override is None:
            l2r, r2l = model.recognize(x)
            enc_out = taps[2].outs[0]
        else:
            l2r, r2l = model.decoder.recognize_beam(enc_override)
            enc_out = enc_override
        return l2r, r2l, enc_out, torch.stack(taps[0].outs, 1), torch.stack(taps[1].outs, 1)
    finally:
        for t_ in taps:
            t_.close()


def _first_divergence(a, b):
    """per clip: index of the first decode step whose emitted token differs (16 = never).  a, b: [N, 17] with <sos>."""
    ne = (a[:, 1:] != b[:, 1:])
    first = torch.where(ne.any(1), ne.float().argmax(1), torch.full((a.shape[0],), ne.shape[1], device=a.device))
    return first.long()


def test_greedy_tokens_reference_decoder_on_dropins_1000_clips(models, dev):
    """north_star: identical greedy decode tokens on 1,000 synthetic clips — `Transformer.recognize` of the reference on
    the drop-ins vs the all-reference fp32 model.  Random decoder weights put many clips on argmax near-ties, so the
    assertion is margin-aware: the control (the reference's own encoder output rounded ONCE to bf16, i.e. the
    irreducible perturbation of any 16-bit hand-off) is decoded in the same run; every clip whose smallest top-1/top-2
    logit margin is clear of the largest logit movement the control shows MUST decode identically, near-ties are
    counted, and >= 990 / 1000 sequences must be identical in each direction."""
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    R, ref, ours = models
    chunk, chunks = 40, 25
    stats = {d: dict(same=0, ctl_same=0, clear=0, clear_same=0, ctl_clear_same=0) for d in ("l2r", "r2l")}
    worst_err, ctl_err, thr = 0.0, 0.0, {"l2r": 0.0, "r2l": 0.0}
    distinct = {"l2r": set(), "r2l": set()}
    per_chunk = []
    with torch.no_grad(), ref_runtime.dropout_neutralised(R):
        for c in range(chunks):
            x = synth.structured_clips(chunk, T, seed=5000 + c)[:, 0].to(dev)          # [N,T,88,88], as test.py feeds it
            a = _recognize(ref, x)
            b = _recognize(ours, x)
            ctl_in = a[2].to(torch.bfloat16).float()
            k = _recognize(ref, None, enc_override=ctl_in)
            worst_err = max(worst_err, rel_fro(b[2], a[2]))
            ctl_err = max(ctl_err, rel_fro(ctl_in, a[2]))
            rec = {"chunk": c, "enc_rel_err": rel_fro(b[2], a[2])}
            for di, d in enumerate(("l2r", "r2l")):
                ta, tb, tk = a[di], b[di], k[di]
                la, lk = a[3 + di], k[3 + di]                                       # [N,16,58]
                top2 = la.topk(2, dim=-1).values
                margin = (top2[..., 0] - top2[..., 1]).min(dim=1).values               # smallest margin of the sequence
                # logit movement of the control on the steps whose prefix is still identical to the reference's
                fd = _first_divergence(ta, tk)
                steps = torch.arange(la.shape[1], device=dev)[None, :]
                valid = steps <= fd[:, None]
                move = ((lk - la).abs().max(dim=-1).values * valid).max()
                thr[d] = max(thr[d], 2.0 * float(move))
                same = (ta == tb).all(1)
                ctl_same = (ta == tk).all(1)
                rec[d] = {"same": int(same.sum()), "ctl_same": int(ctl_same.sum()), "margins": margin.tolist(),
                          "same_mask": same.tolist(), "ctl_same_mask": ctl_same.tolist()}
                stats[d]["same"] += int(same.sum())
                stats[d]["ctl_same"] += int(ctl_same.sum())
                for row in ta.tolist():
                    distinct[d].add(tuple(row))
            per_chunk.append(rec)
    # margin-aware pass over all clips with the run-wide threshold
    for d in ("l2r", "r2l"):
        for rec in per_chunk:
            for mg, s_, cs in zip(rec[d]["margins"], rec[d]["same_mask"], rec[d]["ctl_same_mask"]):
                if mg > thr[d]:
                    stats[d]["clear"] += 1
                    stats[d]["clear_same"] += int(s_)
                    stats[d]["ctl_clear_same"] += int(cs)
    total = chunk * chunks
    res = {"clips": total, "frames": T,
           "encoder_output_rel_fro_err_max_chunk": worst_err, "control_bf16_rounding_rel_err": ctl_err,
           "margin_threshold_logits": thr,
           "l2r": stats["l2r"], "r2l": stats["r2l"],
           "distinct_reference_sequences": {d: len(v) for d, v in distinct.items()},
           "how": "reference Transformer.recognize (transformer.py:45-69) + Decoder.recognize_beam (decoder.py:301-385) "
                  "from oracle/_ref on cuda: all-reference fp32 model vs the same classes on the drop-in frontend + "
                  "encoder (dropin.patch_reference); control = reference encoder output rounded once to bf16",
           "enc16": str(ops.enc16_dtype())}
    _dump("r02_greedy_token_parity.json", res)
    print(json.dumps(res))
    assert worst_err < 4e-3, f"encoder output error {worst_err:.2e} (bar 4e-3, north_star tolerance 1e-2)"
    for d in ("l2r", "r2l"):
        s_ = stats[d]
        assert s_["clear_same"] == s_["clear"], f"{d}: a clip with a clear margin decoded differently: {s_}"
        assert s_["same"] >= 990, f"{d}: only {s_['same']}/1000 identical sequences (control {s_['ctl_same']})"
        flips, ctl_flips = total - s_["same"], total - s_["ctl_same"]
        assert flips <= max(2 * ctl_flips, 10), f"{d}: {flips} flips vs {ctl_flips} for the bf16 control"


def test_recognize_with_always_on_dropout_draws_the_reference_mask(fe_enc, dev):
    """What `recognize` runs before the decoder (transformer.py:55-67), untouched on both sides: frontend with the
    always-on dropout(0.5) of video_frontend.py:122 active, then the encoder.  Under the same CUDA seed the drop-in draws
    the very same Philox mask (same torch call on the same shape), so encoder outputs stay within tolerance of the
    reference's fp32 modules."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    m = fe_enc
    n = 8
    x = synth.structured_clips(n, T, seed=77).to(dev)                     # [N,1,T,88,88], as recognize views it
    m.fe.always_on_dropout = True
    try:
        with torch.no_grad():
            torch.manual_seed(11)
            a, = m.enc_ref(m.fe_ref(x), [T] * n)
            torch.manual_seed(11)
            b, = m.enc(m.fe(x), [T] * n)
            torch.manual_seed(12)
            c, = m.enc(m.fe(x), [T] * n)
    finally:
        m.fe.always_on_dropout = False
    assert rel_fro(b, a) < 4e-3
    assert rel_fro(c, a) > 0.05          # a different seed really is a different mask


def test_teacher_forced_forward_reference_decoder_on_dropins(models, dev):
    """BASELINE configs[4] shape: `Transformer.forward` (transformer.py:22-43) — new encoder + reference bidirectional
    decoder, teacher-forced with the reference's own coin flips (decoder.py:176, `random.random()` seeded alike)."""
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import synth
    R, ref, ours = models
    n, t = 16, 30
    g = torch.Generator().manual_seed(3)
    x = synth.structured_clips(n, t, seed=123)[:, 0].to(dev)
    tgt = torch.full((n, 14), -1, dtype=torch.long)
    for i in range(n):   # data_gen.py:297-302: ids in [2,58), padded with IGNORE_ID; r2l = reversed
        ln = int(torch.randint(3, 12, (1,), generator=g))
        tgt[i, :ln] = torch.randint(2, 58, (ln,), generator=g)
    tgt_r = tgt.clone()
    for i in range(n):
        ln = int((tgt[i] >= 0).sum())
        tgt_r[i, :ln] = tgt[i, :ln].flip(0)
    tgt, tgt_r = tgt.to(dev), tgt_r.to(dev)
    with torch.no_grad(), ref_runtime.dropout_neutralised(R):
        random.seed(7)
        pa = ref(x, tgt, tgt_r)
        random.seed(7)
        pb = ours(x, tgt, tgt_r)
    assert torch.equal(pa[1], pb[1]) and torch.equal(pa[3], pb[3])      # gold labels
    e_l2r, e_r2l = rel_fro(pb[0], pa[0]), rel_fro(pb[2], pa[2])
    _dump("r02_teacher_forced_forward.json", {"batch": n, "frames": t, "pred_l2r_rel_err": e_l2r,
                                               "pred_r2l_rel_err": e_r2l})
    assert e_l2r < 1e-2 and e_r2l < 1e-2, (e_l2r, e_r2l)


def test_stage_error_budget(fe_enc, dev):
    """Where the error comes from: relative Frobenius error of every stage boundary of the CUDA path against the
    all-reference fp32 model on the same 8 structured clips (each stage fed by the path's own previous stage, i.e.
    accumulated error).  bf16 trunk, enc16 encoder: features <= 4e-3, encoder output <= 4e-3 (north_star: 1e-2)."""
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    n = 8
    x = synth.structured_clips(n, T, seed=4242).to(dev)                   # [N,1,T,88,88]
    fe_ref, fe, enc_ref = fe_enc.fe_ref, fe_enc.fe, fe_enc.enc_ref
    taps = {"stem": _Tap(fe_ref.frontend3D)}
    for li in range(1, 5):
        taps[f"layer{li}"] = _Tap(getattr(fe_ref.resnet18, f"layer{li}"))
    for i, lyr in enumerate(enc_ref.layer_stack):
        taps[f"enc_layer{i}"] = _Tap(lyr, pick=lambda o: o[0])
    with torch.no_grad():
        feat_ref = fe_ref._frontend_forward(x).view(n, T, 512)            # the frontend without its always-on dropout
        enc_ref(feat_ref, [T] * n)
    want = {k: v.outs[0] for k, v in taps.items()}
    for v in taps.values():
        v.close()
    table = {}
    with torch.no_grad():
        pk = fe._get_packed()
        a = ops.conv3d_bn_relu_pool(ops.prep_clip(x), pk.c3w, pk.c3b, flat=True)
        stem_ref = want["stem"].transpose(1, 2).contiguous().view(-1, 64, 22, 22)
        table["stem"] = rel_fro(a.dense().permute(0, 3, 1, 2), stem_ref)
        bi = 0
        for li in range(1, 5):
            for b in range(2):
                (st, w1, b1, w2, b2, ds) = pk.blocks[bi]
                if isinstance(a, ops.FlatActs) and st == 1 and ds is None:
                    h = ops.conv3x3_flat(a, w1, b1, relu=True)
                    a = ops.conv3x3_flat(h, w2, b2, relu=True, residual=a)
                elif ds is not None and w2.dim() == 2:
                    h, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=st, relu=True,
                                             flat_ws=fe._flat_workspace(a, w1.shape[0], st))
                    a = ops.conv3x3_flat(h, w2, b2, relu=True, residual=res)
                elif ds is not None:
                    h, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=st, relu=True)
                    a = ops.conv2d(h, w2, b2, stride=1, relu=True, residual=res)
                else:
                    h = ops.conv2d(a, w1, b1, stride=st, relu=True)
                    a = ops.conv2d(h, w2, b2, stride=1, relu=True, residual=a)
                bi += 1
            got = a.dense() if isinstance(a, ops.FlatActs) else a
            table[f"layer{li}"] = rel_fro(got.permute(0, 3, 1, 2), want[f"layer{li}"])
        feat = fe(x)
        table["features"] = rel_fro(feat, feat_ref)
        esd = synth.encoder_state_dict(2, 6)
        for k in range(1, 7):
            enc_k = Encoder(512, k, 8, 64, 64, 512, 2048).to(dev).eval()
            enc_k.load_state_dict({kk: v for kk, v in esd.items()
                                   if not kk.startswith("layer_stack.") or int(kk.split(".")[1]) < k})
            out_k, = enc_k(feat, [T] * n)
            table[f"enc_layer{k - 1}"] = rel_fro(out_k, want[f"enc_layer{k - 1}"])
            # the encoder alone, fed the REFERENCE features (its own contribution)
            if k == 6:
                own, = enc_k(feat_ref, [T] * n)
                table["encoder_alone_on_reference_features"] = rel_fro(own, want["enc_layer5"])
    _dump("r02_stage_error_table.json", {"clips": n, "frames": T, "rel_fro_err_vs_reference_fp32": table,
                                         "enc16": str(ops.enc16_dtype())})
    print(json.dumps(table))
    assert table["features"] < 4e-3, table
    assert table["enc_layer5"] < 4e-3, table
    assert max(table.values()) < 1e-2, table


# ------------------------------------------------------------------ row f.1: the SBL decoder on libsblk
@pytest.fixture(scope="module")
def native_decoder(models, dev):
    """The libsblk Decoder loaded from the reference decoder's state dict (same keys)."""
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    R, ref, ours = models
    dec = Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1, pe_maxlen=5000)
    sd = ref.decoder.state_dict()
    assert sorted(sd) == sorted(dec.state_dict())
    dec.load_state_dict(sd)
    return dec.to(dev).eval()


def test_native_decoder_init_matches_reference_under_same_seed(models):
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    R, ref, ours = models
    torch.manual_seed(123)
    a = R.Decoder(0, 1, 58, 512, 2, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1, pe_maxlen=100)
    torch.manual_seed(123)
    b = Decoder(0, 1, 58, 512, 2, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1, pe_maxlen=100)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)


def test_native_decoder_teacher_forced_logits(models, native_decoder, dev):
    """Decoder.forward (decoder.py:79-191) on the SAME encoder outputs and the same coin flips: logits of all 16 steps
    within 5e-3 of the reference decoder (fp16 operands, fp32 accumulation / LayerNorm / softmax / mixing)."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    R, ref, ours = models
    n, t = 16, 30
    g = torch.Generator().manual_seed(5)
    x = synth.structured_clips(n, t, seed=321)[:, 0].to(dev)
    tgt = torch.full((n, 14), -1, dtype=torch.long)
    for i in range(n):
        ln = int(torch.randint(3, 12, (1,), generator=g))
        tgt[i, :ln] = torch.randint(2, 58, (ln,), generator=g)
    tgt_r = tgt.clone()
    for i in range(n):
        ln = int((tgt[i] >= 0).sum())
        tgt_r[i, :ln] = tgt[i, :ln].flip(0)
    tgt, tgt_r = tgt.to(dev), tgt_r.to(dev)
    from oracle import ref_runtime
    with torch.no_grad(), ref_runtime.dropout_neutralised(R):
        feat = ref.visual_frontend(x.unsqueeze(4).permute(0, 4, 1, 2, 3))
        enc, *_ = ref.encoder(feat, [t] * n)
        random.seed(11)
        pa = ref.decoder(tgt, tgt_r, enc, [t] * n)
        random.seed(11)
        pb = native_decoder(tgt, tgt_r, enc, [t] * n)
    assert torch.equal(pa[1], pb[1]) and torch.equal(pa[3], pb[3])
    e1, e2 = rel_fro(pb[0], pa[0]), rel_fro(pb[2], pa[2])
    _dump("r02_native_decoder_teacher_forced.json", {"pred_l2r_rel_err": e1, "pred_r2l_rel_err": e2})
    assert e1 < 5e-3 and e2 < 5e-3, (e1, e2)


def test_native_decoder_greedy_tokens_1000_clips(models, native_decoder, dev):
    """recognize_beam (decoder.py:301-385) of the libsblk decoder vs the reference decoder on the reference's own fp32
    encoder outputs for the 1,000 structured clips, margin-aware like the encoder test: every sequence whose smallest
    top-1/top-2 margin is clear of 2 x the largest logit difference between the two decoders (measured on the steps whose
    prefixes are still identical) must be identical; near-ties are counted."""
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import synth
    R, ref, ours = models
    chunk, chunks = 40, 25
    res = {d: dict(same=0, clear=0, clear_same=0) for d in ("l2r", "r2l")}
    thr = {"l2r": 0.0, "r2l": 0.0}
    recs = []
    with torch.no_grad(), ref_runtime.dropout_neutralised(R):
        for c in range(chunks):
            x = synth.structured_clips(chunk, T, seed=5000 + c)[:, 0].to(dev)
            a = _recognize(ref, x)
            b = native_decoder._greedy(a[2], want_logits=True)
            for di, d in enumerate(("l2r", "r2l")):
                la, lb = a[3 + di], b[2 + di]
                top2 = la.topk(2, dim=-1).values
                margin = (top2[..., 0] - top2[..., 1]).min(dim=1).values
                # BOTH directions feed every step (bidirectional mixing): a prefix is "still identical" while both are
                fd = torch.minimum(_first_divergence(a[0], b[0]), _first_divergence(a[1], b[1]))
                valid = torch.arange(la.shape[1], device=dev)[None, :] <= fd[:, None]
                thr[d] = max(thr[d], 2.0 * float(((lb - la).abs().max(dim=-1).values * valid).max()))
                same = (a[di] == b[di]).all(1)
                recs.append((d, margin.tolist(), same.tolist()))
                res[d]["same"] += int(same.sum())
    for d, margins, sames in recs:
        for mg, s_ in zip(margins, sames):
            if mg > thr[d]:
                res[d]["clear"] += 1
                res[d]["clear_same"] += int(s_)
    out = {"clips": chunk * chunks, "margin_threshold_logits": thr, **res}
    _dump("r02_native_decoder_greedy_parity.json", out)
    print(json.dumps(out))
    for d in ("l2r", "r2l"):
        assert res[d]["clear_same"] == res[d]["clear"], (d, res[d])
        assert res[d]["same"] >= 970, (d, res[d])


def test_reference_transformer_on_all_dropins_recognize(models, dev):
    """`Transformer.recognize` with frontend, encoder AND decoder replaced (dropin.patch_reference(..., decoder=True)):
    the whole SBL model on libsblk, assembled by the reference's own Transformer class."""
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import dropin, synth
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder as B200Decoder
    R, ref, ours = models
    with dropin.patched_reference(R.dir, decoder=True):
        import transformer.decoder as tdec
        import transformer.encoder as tenc
        import transformer.transformer as ttr
        enc = tenc.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        dec = tdec.Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                           pe_maxlen=5000)
        full = ttr.Transformer(enc, dec, None)
    assert isinstance(full.decoder, B200Decoder)
    full.load_state_dict(ref.state_dict())
    full = full.to(dev).eval()
    full.visual_frontend.always_on_dropout = False
    x = synth.structured_clips(40, T, seed=5003)[:, 0].to(dev)
    with torch.no_grad(), ref_runtime.dropout_neutralised(R):
        a_l2r, a_r2l = ref.recognize(x)
        b_l2r, b_r2l = full.recognize(x)
    assert b_l2r.shape == a_l2r.shape == (40, 17) and b_l2r.dtype == torch.long
    assert int((a_l2r == b_l2r).all(1).sum()) >= 38 and int((a_r2l == b_r2l).all(1).sum()) >= 36


def test_native_decoder_cuda_graph_steps_equal_eager(fe_enc, dev):
    """The captured decode steps (one CUDA graph per prefix length, PDL on) return the bits of the eager launches, for
    two different batch shapes in a row (plans are cached per shape) and after a weight change.  Decoder weights: the
    reference initialisation under a fixed seed; encoder outputs: the reference's fp32 frontend + encoder."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    torch.manual_seed(7)
    native_decoder = Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                             pe_maxlen=5000).to(dev).eval()
    with torch.no_grad():
        for n, t, seed in ((5, 29, 1), (12, 40, 2), (5, 29, 3)):
            x = synth.structured_clips(n, t, seed=600 + seed).to(dev)
            feat = fe_enc.fe_ref._frontend_forward(x).view(n, t, 512)
            enc, *_ = fe_enc.enc_ref(feat, [t] * n)
            native_decoder.use_cuda_graphs = True
            a = native_decoder._greedy(enc, want_logits=True)
            native_decoder.use_cuda_graphs = False
            b = native_decoder._greedy(enc, want_logits=True)
            native_decoder.use_cuda_graphs = True
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
            assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
        # in-place weight update -> packed weights and plans are rebuilt
        w = native_decoder.tgt_word_prj_l2r.weight
        before = native_decoder._greedy(enc, want_logits=True)[2]
        with torch.no_grad():
            w.mul_(0.5)
        after = native_decoder._greedy(enc, want_logits=True)[2]
        with torch.no_grad():
            w.mul_(2.0)
        assert torch.allclose(after, before * 0.5, rtol=2e-2, atol=1e-3) and not torch.equal(after, before)
