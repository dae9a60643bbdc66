"""`-m gpu`: the SBL decoder's training path on libsblk (training.decoder_forward_train, DESIGN.md §9 "training").

Kernels are checked against float64 autograd on the same enc16 / bf16 operands, element-wise with
err = max |got - want| / (|want| + rms(want)) (as in test_decoder_gpu.py; 16-bit results in units U of their format's
unit roundoff).  The whole decoder is checked against float64 autograd through oracle/decoder_oracle.step_logits
(with dropout: tests/decoder_dropout_oracle.step_logits): logits element-wise, gradients as relative Frobenius errors |got - want| / |want| per parameter.  Bars are about twice
the maxima measured on a B200 (DESIGN.md §9 lists both); the gradient bar is no looser than the encoder's 3e-2.
With SBLK_TEST_OUT_DIR set, the measured maxima are written to decoder_train_gpu_errors.json there.
"""
import json
import os
import random

import pytest
import torch

import decoder_dropout_oracle as DO
from oracle import decoder_oracle as O

pytestmark = pytest.mark.gpu

SOS, EOS, VOCAB = 0, 1, 58
SCALE = 0.125
MEASURED = {}

ATT_OUT_BAR_U = 1.2          # attention output, enc16 U
ATT_PROBS_BAR = 1e-5         # saved fp32 probabilities
ATT_GRAD_BAR_U = 1.2         # dQ / dK / dV, bf16 U
EMB_BAR = 3e-6               # embedding gradient (fp32 sums)
LOGITS_BAR_U = 10.0          # logits of all 16 steps, enc16 U
GRAD_BAR = 3e-2              # relative Frobenius error of every parameter gradient and of the encoder-output gradient


def _u(dtype=None):
    from sbl_for_multilingual_lip_reading_b200 import ops
    return torch.finfo(dtype or ops.enc16_dtype()).eps / 2


def _record(name, value, bar):
    m = MEASURED.setdefault(name, {"max": 0.0, "bar": bar})
    m["max"] = max(m["max"], float(value))


@pytest.fixture(scope="module", autouse=True)
def _dump_measured():
    yield
    out_dir = os.environ.get("SBLK_TEST_OUT_DIR")
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "decoder_train_gpu_errors.json"), "w") as f:
            json.dump(MEASURED, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    assert ops.init() > 0
    return torch.device("cuda:0")


def _err(got, want):
    got, want = got.double(), want.double()
    assert torch.equal(got.isnan(), want.isnan()), "NaN pattern differs from the float64 reference"
    ok = ~want.isnan()
    g, w = got[ok], want[ok]
    if w.numel() == 0:
        return 0.0
    s = w.pow(2).mean().sqrt()
    if s == 0:                    # a gradient that is zero in exact arithmetic (one key: softmax is constant)
        return float((g - w).abs().max())
    return float(((g - w).abs() / (w.abs() + s)).max())


def _fro(got, want):
    return float((got.double() - want.double()).norm() / want.double().norm())


# ------------------------------------------------------------------------------------------ training attention
ATT_CASES = ([("self", L, L, c) for L in (1, 7, 16) for c in (1, 0)] +
             [("cross", lq, lk, 0) for lq in (1, 7, 16) for lk in (1, 29, 64)])


@pytest.mark.parametrize("case", ATT_CASES, ids=lambda c: "{}-Lq{}-Lk{}-causal{}".format(*c))
def test_xattention_train_against_float64_autograd(case, dev):
    """sblk_xattention_train_fwd / _bwd in the decoder's two layouts (self-attention: Q | K | V thirds of one
    [rows, 1536] buffer, gradients into the thirds of one dqkv buffer; cross: Q [rows, 512], K | V [rows, 1024],
    dK | dV into the halves of one buffer), with and without dropout factors: output, probabilities, dQ, dK, dV.
    A second backward is bit-identical."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    layout, lq, lk, causal = case
    e16 = ops.enc16_dtype()
    n, h = 5, 8
    g = torch.Generator(device=dev).manual_seed(100 * lq + lk + causal)
    if layout == "self":
        buf = (torch.randn(n * lq, 1536, generator=g, device=dev) * 1.5).to(e16)
        q, k, v = buf[:, :512], buf[:, 512:1024], buf[:, 1024:]
    else:
        q = (torch.randn(n * lq, 512, generator=g, device=dev) * 1.5).to(e16)
        kv = (torch.randn(n * lk, 1024, generator=g, device=dev) * 1.5).to(e16)
        k, v = kv[:, :512], kv[:, 512:]
    dout = torch.randn(n * lq, 512, generator=g, device=dev).to(torch.bfloat16)
    for use_drop in (False, True):
        drop = None
        if use_drop:
            drop = (torch.rand(h * n, lq, lk, generator=g, device=dev) > 0.1).float() / 0.9
        out, probs = ot.xattention_train_fwd(q, k, v, n, lq, lk, h, causal=bool(causal), drop=drop, scale=SCALE)
        if layout == "self":
            dqkv = torch.empty((n * lq, 1536), dtype=torch.bfloat16, device=dev)
            grads = ot.xattention_train_bwd(q, k, v, probs, dout, n, lq, lk, h, causal=bool(causal), drop=drop,
                                            scale=SCALE, dq=dqkv[:, :512], dk=dqkv[:, 512:1024], dv=dqkv[:, 1024:])
            again = ot.attention_train_bwd(buf, probs, dout, n, lq, h, drop=drop, scale=SCALE) if not causal else None
        else:
            dkv = torch.empty((n * lk, 1024), dtype=torch.bfloat16, device=dev)
            grads = ot.xattention_train_bwd(q, k, v, probs, dout, n, lq, lk, h, drop=drop, scale=SCALE,
                                            dk=dkv[:, :512], dv=dkv[:, 512:])
            again = None
        grads2 = ot.xattention_train_bwd(q, k, v, probs, dout, n, lq, lk, h, causal=bool(causal), drop=drop, scale=SCALE)
        for a, b in zip(grads, grads2):
            assert torch.equal(a, b), "backward is not deterministic"
        if again is not None:                  # the encoder's packed kernel pair computes the same bits
            assert torch.equal(again, dqkv)
        # float64 autograd on the same operands
        Q = q.double().reshape(n, lq, h, 64).permute(0, 2, 1, 3).requires_grad_()
        K = k.double().reshape(n, lk, h, 64).permute(0, 2, 1, 3).requires_grad_()
        V = v.double().reshape(n, lk, h, 64).permute(0, 2, 1, 3).requires_grad_()
        s = (Q @ K.transpose(-1, -2)) * SCALE
        if causal:
            s = s.masked_fill(torch.ones(lq, lk, dtype=torch.bool, device=dev).triu(1), float("-inf"))
        p = torch.softmax(s, -1)                                             # [n, h, lq, lk]
        pd = p if drop is None else p * drop.double().view(h, n, lq, lk).transpose(0, 1)
        o = (pd @ V).permute(0, 2, 1, 3).reshape(n * lq, h * 64)
        o.backward(dout.double())
        want = {"dq": Q.grad.permute(0, 2, 1, 3).reshape(n * lq, 512),
                "dk": K.grad.permute(0, 2, 1, 3).reshape(n * lk, 512),
                "dv": V.grad.permute(0, 2, 1, 3).reshape(n * lk, 512)}
        e_out = _err(out, o.detach()) / _u()
        e_p = _err(probs, p.detach().transpose(0, 1).reshape(h * n, lq, lk))
        e_g = max(_err(got, want[nm]) for got, nm in zip(grads, ("dq", "dk", "dv"))) / _u(torch.bfloat16)
        _record("xattn_train_out_U", e_out, ATT_OUT_BAR_U)
        _record("xattn_train_probs", e_p, ATT_PROBS_BAR)
        _record("xattn_train_grads_bf16_U", e_g, ATT_GRAD_BAR_U)
        assert e_out <= ATT_OUT_BAR_U and e_p <= ATT_PROBS_BAR and e_g <= ATT_GRAD_BAR_U, (case, use_drop, e_out, e_p, e_g)


def test_xattention_train_rejects_bad_arguments(dev):
    """Shapes beyond Lq, Lk <= 64, empty shapes, short row pitches and null pointers return an error before launching."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops
    lib = _lib.load()
    e16 = ops.enc16_dtype()
    st = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros((65 * 2, 1536), dtype=e16, device=dev)
    probs = torch.zeros((8 * 2 * 65 * 65,), dtype=torch.float32, device=dev)
    out = torch.zeros((65 * 2, 512), dtype=e16, device=dev)
    g = torch.zeros((65 * 2, 1536), dtype=torch.bfloat16, device=dev)
    b = buf.data_ptr()

    def fwd(lq, lk, ld=1536, n=2, qp=b):
        return lib.sblk_xattention_train_fwd(qp, b + 1024, b + 2048, None, probs.data_ptr(), out.data_ptr(), None, ld, ld,
                                             ld, 512, n, lq, lk, 8, 0, SCALE, st)

    def bwd(lq, lk, ldg=1536, dk=g.data_ptr() + 1024):
        return lib.sblk_xattention_train_bwd(b, b + 1024, b + 2048, None, probs.data_ptr(), out.data_ptr(), g.data_ptr(),
                                             dk, g.data_ptr() + 2048, None, 1536, 1536, 1536, 512, ldg, ldg, ldg, 2, lq,
                                             lk, 8, 0, SCALE, st)
    before = ops.launch_count()
    assert fwd(65, 16) < 0 and "Lq <= 64" in _lib.last_error()
    assert fwd(16, 65) < 0 and "Lk <= 64" in _lib.last_error()
    assert fwd(0, 16) < 0 and fwd(16, 0) < 0 and fwd(4, 4, n=0) < 0
    assert fwd(4, 4, ld=500) < 0 and "pitches" in _lib.last_error()
    assert fwd(4, 4, qp=None) < 0 and "null" in _lib.last_error()
    assert bwd(65, 4) < 0 and bwd(4, 65) < 0
    assert bwd(4, 4, ldg=256) < 0 and "pitches" in _lib.last_error()
    assert bwd(4, 4, dk=None) < 0 and "null" in _lib.last_error()
    assert ops.launch_count() == before
    assert fwd(64, 64) == 0 and bwd(64, 64) == 0
    torch.cuda.synchronize()
    # the tensor wrappers refuse mismatched factors and short views
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    with pytest.raises(RuntimeError):
        ot.xattention_train_fwd(buf[:8, :512], buf[:8, 512:1024], buf[:8, 1024:], 2, 4, 4, 8,
                                drop=torch.ones((8, 4, 4), device=dev))
    with pytest.raises(RuntimeError):
        ot.xattention_train_fwd(buf[:7, :512], buf[:8, 512:1024], buf[:8, 1024:], 2, 4, 4, 8)


# ------------------------------------------------------------------------------------------ mixing / embedding backward
def test_bidir_mix_bwd_is_autograd_bit_for_bit(dev):
    """sblk_bidir_mix_bwd against autograd through the oracle's aliased loops in fp32, bit for bit (odd L included)."""
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator(device=dev).manual_seed(9)
    for n in (1, 5):
        for L in (1, 2, 3, 7, 16):
            a = torch.randn(n, L, 512, generator=g, device=dev, requires_grad=True)
            b = torch.randn(n, L, 512, generator=g, device=dev, requires_grad=True)
            ga = torch.randn(n, L, 512, generator=g, device=dev) * 3
            gb = torch.randn(n, L, 512, generator=g, device=dev) * 3
            x, y = O.bidir_mix(a, b)
            torch.autograd.backward([x, y], [ga, gb])
            d_l2r, d_r2l = ot.bidir_mix_bwd(ga.view(n * L, 512), gb.view(n * L, 512), n, L)
            assert torch.equal(d_l2r.view(n, L, 512), a.grad) and torch.equal(d_r2l.view(n, L, 512), b.grad), (n, L)


def test_embed_bwd_against_index_add(dev):
    """sblk_embed_bwd against index_add in float64, tokens in the decoder's [N, 17] buffers; ids that repeat in every
    row (a whole batch of one id, and one id at every position of a row) and out-of-range ids (clamped as in the
    forward); two runs bit-identical."""
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator(device=dev).manual_seed(10)
    worst = 0.0
    for n, L in ((1, 1), (7, 16), (240, 16), (300, 5)):
        for scale in (1.0, 0.5):
            tok = torch.randint(0, VOCAB, (n, 17), generator=g, device=dev)
            tok[:, 0] = SOS                                   # <sos> in every row
            tok[0, :L] = 5                                    # one id at every position of a row
            if n > 2:
                tok[1, L - 1] = -3
                tok[2, 0] = VOCAB + 4
            dx = torch.randn(n * L, 512, generator=g, device=dev)
            got = ot.embed_bwd(tok, L, dx, VOCAB, scale)
            assert torch.equal(got, ot.embed_bwd(tok, L, dx, VOCAB, scale))
            ids = tok[:, :L].clamp(0, VOCAB - 1).reshape(-1)
            want = torch.zeros(VOCAB, 512, dtype=torch.float64, device=dev).index_add_(0, ids, dx.double()) * scale
            worst = max(worst, _err(got, want))
    _record("embed_bwd", worst, EMB_BAR)
    assert worst <= EMB_BAR, worst


# ------------------------------------------------------------------------------------------ the whole decoder
def _decoder(n_layers, dev, p=0.0):
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    torch.manual_seed(7)
    return Decoder(SOS, EOS, VOCAB, 512, n_layers, 8, 64, 64, 512, 2048, dropout=p, tgt_emb_prj_weight_sharing=1,
                   pe_maxlen=5000).to(dev).train()


def _targets(n, seed):
    g = torch.Generator().manual_seed(seed)
    tgt = torch.full((n, 14), O.IGNORE_ID, dtype=torch.long)
    tgt_r = tgt.clone()
    for i in range(n):
        ln = 0 if i == 0 else int(torch.randint(1, 13, (1,), generator=g))
        slots = torch.randperm(14, generator=g)[:ln].sort().values
        toks = torch.randint(2, VOCAB, (ln,), generator=g)
        tgt[i, slots] = toks
        tgt_r[i, slots] = toks.flip(0)
    return tgt, tgt_r


@pytest.fixture(scope="module")
def enc_pool(dev):
    """Encoder outputs of the drop-in frontend + encoder (synthetic weights, evaluation mode) on 64 structured clips of
    64 frames; get(n, t, seed) -> [n, t, 512].  (With iid Gaussian encoder outputs these untrained decoders are far
    more sensitive to operand rounding: the evaluation path itself is ~170 U from the float64 oracle at 6 layers.)"""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    enc = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1)
    enc.load_state_dict(synth.encoder_state_dict(2, 6))
    fe, enc = fe.to(dev).eval(), enc.to(dev).eval()
    fe.always_on_dropout = False
    with torch.no_grad():
        pool = torch.cat([enc(fe(synth.structured_clips(16, 64, seed=900 + c).to(dev)), [64] * 16)[0].float()
                          for c in range(4)]).contiguous()

    def get(n, t, seed):
        # frame j of clip b from a random one of the 64 clips: a structured clip's encoder outputs barely change from
        # frame to frame, which would leave the keys of the decoder-encoder attention all alike (their gradients ~0)
        idx = torch.randint(0, 64, (n, t), generator=torch.Generator().manual_seed(seed)).to(dev)
        return pool[idx, torch.arange(t, device=dev)[None, :]].contiguous()
    return get


def _run(dec, n, t, seed, dev, enc_pool):
    """One training forward + backward of sum(logits * G) -> (logits (l2r, r2l), {name: grad}, enc grad, G, enc)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    enc = enc_pool(n, t, seed).requires_grad_()
    tgt, tgt_r = _targets(n, seed)
    G = (torch.randn(n, 16, VOCAB, generator=g, device=dev), torch.randn(n, 16, VOCAB, generator=g, device=dev))
    dec.zero_grad(set_to_none=True)
    la, gold_a, lb, gold_b = dec(tgt.to(dev), tgt_r.to(dev), enc, [t] * n)
    assert la.shape == (n, 16, VOCAB) and lb.shape == (n, 16, VOCAB) and la.requires_grad
    ((la * G[0]).sum() + (lb * G[1]).sum()).backward()
    grads = {k: p_.grad for k, p_ in dec.named_parameters()}
    return (la.detach(), lb.detach()), grads, enc.grad, G, enc.detach(), (tgt, tgt_r)


def _oracle(dec, enc, ys, G, drops=None, **variant):
    """float64 autograd through step_logits on the fed tokens ys = (ys_l2r, ys_r2l) [N, 17]."""
    sd = {k: v.detach().double().clone().requires_grad_(k != "positional_encoding.pe")
          for k, v in dec.state_dict().items()}
    e = enc.double().clone().requires_grad_()
    if drops is None:
        steps = [O.step_logits(sd, ys[0], ys[1], e, L, **variant) for L in range(1, 17)]
    else:
        steps = [DO.step_logits(sd, ys[0], ys[1], e, L, drops[L - 1]) for L in range(1, 17)]
    la, lb = torch.stack([s[0] for s in steps], 1), torch.stack([s[1] for s in steps], 1)
    ((la * G[0].double()).sum() + (lb * G[1].double()).sum()).backward()
    return (la.detach(), lb.detach()), {k: v.grad for k, v in sd.items() if k != "positional_encoding.pe"}, e.grad


def _grad_errs(grads, egrad, want_grads, want_egrad, plain_keys=None):
    """Relative Frobenius error per parameter, and of the encoder-output gradient.
    Key projections are measured on the scale of the same block's fc-weight gradient: softmax is invariant to a score
    offset per query, so the key gradients of a clip sum to zero (dK^T 1 = 0).  The key-bias gradient is zero in exact
    arithmetic and the key-weight gradient dK^T X keeps only what is left after the per-clip mean of X cancels (in the
    last layer only the last position's query gets a gradient, so almost nothing is left); the rounding of the enc16
    forward operands and of the bf16 dK does not cancel with it.  Their plain relative errors go to `plain_keys`."""
    errs = {}
    for k, w in want_grads.items():
        e = (grads[k].double() - w).norm()
        if ".w_ks." in k:
            if plain_keys is not None and k.endswith("weight"):
                plain_keys[k] = float(e / w.norm())
            errs[k] = float(e / want_grads[k.split(".w_ks.")[0] + ".fc.weight"].norm())
        else:
            errs[k] = float(e / w.norm())
    errs["encoder_outputs"] = _fro(egrad, want_egrad)
    return errs


def _gold_tokens(tgt, tgt_r, dev):
    return O.preprocess(tgt, SOS, EOS)[0].to(dev), O.preprocess(tgt_r, SOS, EOS)[0].to(dev)


def _ys17(ys16, dev):
    return torch.cat([ys16, torch.full((ys16.shape[0], 1), EOS, dtype=torch.long, device=dev)], 1)


DEC_CASES = [(1, 1, 29), (2, 7, 30), (6, 5, 29), (6, 64, 64), (2, 64, 30)]


@pytest.mark.parametrize("case", DEC_CASES, ids=lambda c: "L{}-N{}-T{}".format(*c))
def test_decoder_training_against_float64_autograd(case, dev, enc_pool, monkeypatch):
    """Dropout 0, coin forced to the gold token: the logits of all 16 steps, every parameter gradient and the gradient
    of the encoder outputs against float64 autograd through the oracle; for (6, 5, 29) also at least 10x the bar away
    from two wrong oracles (unaliased mixing, the subsequent mask in every layer)."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    n_layers, n, t = case
    dec = _decoder(n_layers, dev)
    monkeypatch.setattr(random, "random", lambda: 0.0)
    before = ops.launch_count()
    logits, grads, egrad, G, enc, (tgt, tgt_r) = _run(dec, n, t, 1000 * n_layers + n + t, dev, enc_pool)
    MEASURED.setdefault("launches_per_forward_backward", {})["L{}-N{}-T{}".format(*case)] = ops.launch_count() - before
    assert set(grads) == {k for k, _ in dec.named_parameters()}
    ys = tuple(_ys17(y, dev) for y in _gold_tokens(tgt, tgt_r, dev))
    want_l, want_g, want_e = _oracle(dec, enc, ys, G)
    e_l = max(_err(logits[0], want_l[0]), _err(logits[1], want_l[1])) / _u()
    plain = {}
    errs = _grad_errs(grads, egrad, want_g, want_e, plain)
    MEASURED.setdefault("key_weight_grad_plain_rel_fro", {})["L{}-N{}-T{}".format(*case)] = max(plain.values())
    worst = max(errs.values())
    _record("logits_U", e_l, LOGITS_BAR_U)
    _record("grad_rel_fro", worst, GRAD_BAR)
    MEASURED.setdefault("grad_rel_fro_worst_param", {})["L{}-N{}-T{}".format(*case)] = [max(errs, key=errs.get), worst]
    assert e_l <= LOGITS_BAR_U, (case, e_l)
    assert worst <= GRAD_BAR, (case, max(errs, key=errs.get), worst)
    if case == (6, 5, 29):
        def _unaliased_mix(l2r, r2l):
            return l2r + r2l.flip(1), r2l + l2r.flip(1)
        for name, kw in (("unaliased_mixing", dict(mix=_unaliased_mix)), ("mask_in_every_layer", dict(mask_every_layer=True))):
            _, bad_g, bad_e = _oracle(dec, enc, ys, G, **kw)
            dist = max(_grad_errs(grads, egrad, bad_g, bad_e).values())
            _record("grad_dist_" + name, dist, 10 * GRAD_BAR)
            assert dist >= 10 * GRAD_BAR, (name, dist)


def _record_draws(monkeypatch):
    from sbl_for_multilingual_lip_reading_b200 import training
    drawn = []
    orig = training._drop_factor

    def rec(shape, p, dev, train):
        f = orig(shape, p, dev, train)
        drawn.append(f)
        return f
    monkeypatch.setattr(training, "_drop_factor", rec)
    return drawn


def _drops_by_step(drawn, n_layers):
    """The documented draw order: per step, embedding l2r, r2l; per layer l2r then r2l, 5 factors each."""
    it = iter(drawn)
    steps = []
    for _ in range(16):
        st = {"l2r": {"emb": next(it), "layers": []}, "r2l": {"emb": None, "layers": []}}
        st["r2l"]["emb"] = next(it)
        for _li in range(n_layers):
            for d in ("l2r", "r2l"):
                st[d]["layers"].append(tuple(next(it) for _ in range(5)))
        steps.append(st)
    assert next(it, None) is None, "more factors drawn than the documented order accounts for"
    return steps


def test_decoder_training_with_dropout(dev, enc_pool, monkeypatch):
    """p = 0.1: the factors the decoder drew, fed to the float64 oracle in the documented order, give the same logits
    and gradients within the same bars."""
    n_layers, n, t = 2, 6, 30
    dec = _decoder(n_layers, dev, p=0.1)
    monkeypatch.setattr(random, "random", lambda: 0.0)
    drawn = _record_draws(monkeypatch)
    logits, grads, egrad, G, enc, (tgt, tgt_r) = _run(dec, n, t, 77, dev, enc_pool)
    assert len(drawn) == 16 * (2 + 10 * n_layers) and all(f is not None for f in drawn)
    drops = _drops_by_step(drawn, n_layers)
    ys = tuple(_ys17(y, dev) for y in _gold_tokens(tgt, tgt_r, dev))
    want_l, want_g, want_e = _oracle(dec, enc, ys, G, drops=drops)
    e_l = max(_err(logits[0], want_l[0]), _err(logits[1], want_l[1])) / _u()
    worst = max(_grad_errs(grads, egrad, want_g, want_e).values())
    _record("dropout_logits_U", e_l, LOGITS_BAR_U)
    _record("dropout_grad_rel_fro", worst, GRAD_BAR)
    assert e_l <= LOGITS_BAR_U and worst <= GRAD_BAR, (e_l, worst)
    # the factors matter: without them the oracle is far away
    no_l, _, _ = _oracle(dec, enc, ys, G)
    assert max(_err(logits[0], no_l[0]), _err(logits[1], no_l[1])) / _u() > 10 * LOGITS_BAR_U


def test_decoder_training_model_branch_of_the_coin(dev, enc_pool, monkeypatch):
    """Coin always on the model's own argmax: the tokens fed at step i + 1 are rebuilt from the returned step-i logits;
    the oracle on those tokens gives the same logits and gradients."""
    n_layers, n, t = 2, 8, 29
    dec = _decoder(n_layers, dev)
    monkeypatch.setattr(random, "random", lambda: 1.0)
    logits, grads, egrad, G, enc, _ = _run(dec, n, t, 55, dev, enc_pool)
    ys = []
    for lg in logits:
        y = torch.full((n, 17), SOS, dtype=torch.long, device=dev)
        y[:, 1:] = lg.argmax(-1)
        ys.append(y)
    want_l, want_g, want_e = _oracle(dec, enc, tuple(ys), G)
    e_l = max(_err(logits[0], want_l[0]), _err(logits[1], want_l[1])) / _u()
    worst = max(_grad_errs(grads, egrad, want_g, want_e).values())
    _record("model_branch_logits_U", e_l, LOGITS_BAR_U)
    _record("model_branch_grad_rel_fro", worst, GRAD_BAR)
    assert e_l <= LOGITS_BAR_U and worst <= GRAD_BAR, (e_l, worst)


def test_decoder_training_sees_optimizer_steps(dev, enc_pool, monkeypatch):
    """forward + backward, Adam step, forward again: the second call matches the oracle on the updated weights; after
    model.eval(), recognize_beam equals a fresh Decoder loaded with the updated state dict, bit for bit."""
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    n_layers, n, t = 2, 4, 30
    dec = _decoder(n_layers, dev)
    monkeypatch.setattr(random, "random", lambda: 0.0)
    with torch.no_grad():                                    # the eval plan is built (and cached) before the update
        dec.eval()
        dec.recognize_beam(torch.randn(n, t, 512, device=dev))
        dec.train()
    opt = torch.optim.Adam(dec.parameters(), lr=1e-3)
    _run(dec, n, t, 5, dev, enc_pool)
    opt.step()
    logits, _, _, G, enc, (tgt, tgt_r) = _run(dec, n, t, 6, dev, enc_pool)
    ys = tuple(_ys17(y, dev) for y in _gold_tokens(tgt, tgt_r, dev))
    want_l, _, _ = _oracle(dec, enc, ys, G)
    e_l = max(_err(logits[0], want_l[0]), _err(logits[1], want_l[1])) / _u()
    assert e_l <= LOGITS_BAR_U, e_l
    dec.eval()
    fresh = Decoder(SOS, EOS, VOCAB, 512, n_layers, 8, 64, 64, 512, 2048, dropout=0.0).to(dev).eval()
    fresh.load_state_dict(dec.state_dict())
    x = torch.randn(16, t, 512, generator=torch.Generator(device=dev).manual_seed(3), device=dev)
    with torch.no_grad():
        a, b = dec.recognize_beam(x), fresh.recognize_beam(x)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_assembled_sbl_training_step(dev):
    """Drop-in Lipreading + Encoder + Decoder in model.train() on 8 synthetic 30-frame clips, loss 0.5 (CE_l2r + CE_r2l)
    with ignore_index = -1, backward: every parameter of the three modules gets a finite gradient and every decoder
    weight and bias a non-zero one."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    n, t = 8, 30
    fe = Lipreading().to(dev).train()
    fe.load_state_dict(synth.frontend_state_dict(1))
    enc = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).to(dev).train()
    enc.load_state_dict(synth.encoder_state_dict(2, 6))
    dec = _decoder(6, dev, p=0.1)
    x = synth.structured_clips(n, t, seed=21).to(dev)
    tgt, tgt_r = _targets(n, 21)
    torch.manual_seed(1)
    random.seed(1)
    out, = enc(fe(x), [t] * n)
    la, gold_a, lb, gold_b = dec(tgt.to(dev), tgt_r.to(dev), out, [t] * n)
    ce = torch.nn.functional.cross_entropy
    loss = 0.5 * (ce(la.reshape(-1, VOCAB), gold_a.reshape(-1), ignore_index=-1) +
                  ce(lb.reshape(-1, VOCAB), gold_b.reshape(-1), ignore_index=-1))
    loss.backward()
    assert torch.isfinite(loss)
    for mod in (fe, enc, dec):
        for name, p_ in mod.named_parameters():
            assert p_.grad is not None and torch.isfinite(p_.grad).all(), name
    for name, p_ in dec.named_parameters():
        assert p_.grad.abs().max() > 0, name
