"""`-m gpu`: the SBL decoder on libsblk against the float64 oracle (oracle/decoder_oracle.py), with no reference sources.

Kernel tests feed the kernels enc16 operands and feed the same values, upcast to float64, to the reference, so what is
left is the kernel's own error (fp32 accumulation, __expf, the final rounding).  Every element is checked:
err = max |got - want| / (|want| + rms(want)) over the output, against a bar set at about twice the maximum measured on
a B200 (DESIGN.md §9 lists both).  Bars of 16-bit results are in units of U, the unit roundoff of the enc16 format.

The sensitivity asserts compute deliberately wrong oracles (causal mask off by one, mixing without the reference's
aliasing, the subsequent mask in every layer) and require the kernels to sit at least 10x the bar away from each.
With SBLK_TEST_OUT_DIR set, the measured maxima are also written to decoder_gpu_errors.json in that directory.
"""
import json
import os

import pytest
import torch

from oracle import decoder_oracle as O

pytestmark = pytest.mark.gpu

SOS, EOS, VOCAB = 0, 1, 58
MEASURED = {}

# bars (U = enc16 unit roundoff: 2^-11 for fp16, 2^-8 for bf16); measured maxima in DESIGN.md §9
XATTN_BAR_U = 1.7            # attention output, rounded once to enc16              (measured 0.85 U)
GEMM16_BAR_U = 1.6           # ops.gemm 16-bit output                               (measured 0.80 U)
GEMM32_BAR = 2.5e-5          # ops.gemm fp32 output: fp32 accumulation only         (measured 1.21e-5)
LN32_BAR = 2e-5              # ops.linear_ln fp32 output                            (measured 1.00e-5)
LN16_BAR_U = 1.6             # ops.linear_ln 16-bit output                          (measured 0.79 U)
LOGITS_BAR_U = 10.0          # teacher-forced logits of the whole decoder           (measured 4.99 U)
GREEDY_MIN_SAME = 180        # of 200 sequences per direction: 2x the measured flips (r2l 190 / 200, all near-ties)


def _u():
    from sbl_for_multilingual_lip_reading_b200 import ops
    return torch.finfo(ops.enc16_dtype()).eps / 2


def _record(name, value, bar):
    m = MEASURED.setdefault(name, {"max": 0.0, "bar": bar})
    m["max"] = max(m["max"], float(value))


@pytest.fixture(scope="module", autouse=True)
def _dump_measured():
    yield
    out_dir = os.environ.get("SBLK_TEST_OUT_DIR")
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "decoder_gpu_errors.json"), "w") as f:
        json.dump(MEASURED, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    assert ops.init() > 0
    return torch.device("cuda:0")


def _err(got, want):
    """max |got - want| / (|want| + rms(want)); NaN must sit exactly where the reference has NaN."""
    got, want = got.double(), want.double()
    assert torch.equal(got.isnan(), want.isnan()), "NaN pattern differs from the float64 reference"
    ok = ~want.isnan()
    g, w = got[ok], want[ok]
    if w.numel() == 0:
        return 0.0
    s = w.pow(2).mean().sqrt()
    return float(((g - w).abs() / (w.abs() + s)).max())


def _dist(got, variant):
    """Distance of the kernel from a deliberately wrong oracle, in the units of _err (NaN in the variant: infinite)."""
    got, variant = got.double(), variant.double()
    fin = variant[~variant.isnan()]
    s = fin.pow(2).mean().sqrt() if fin.numel() else torch.ones((), dtype=torch.float64, device=got.device)
    d = (got - variant).abs() / (variant.abs() + s)
    return float(d.nan_to_num(nan=float("inf")).max())


# ------------------------------------------------------------------------------------------ sblk_xattention_fwd
LQ = (1, 2, 16, 17, 31, 32)
LK = (1, 16, 31, 32, 33, 64, 65, 127, 128)        # the kernel's 32-key lanes change at 32, 64, 96
HN = ((1, 1), (3, 5), (8, 64))
KLENS = ("none", "ragged", "one", "over", "zero")
SCALE = 0.125


def _klens(mode, n, lk, g, dev):
    if mode == "none":
        return None
    if mode == "ragged":
        v = torch.randint(1, lk + 1, (n,), generator=g, device=dev)
    elif mode == "one":
        v = torch.ones(n, dtype=torch.long, device=dev)
    elif mode == "over":                                   # clamped to Lk
        v = lk + 1 + torch.randint(0, 100, (n,), generator=g, device=dev)
    else:                                                  # every other clip has no valid key: NaN rows
        v = torch.where(torch.arange(n, device=dev) % 2 == 0, 0, lk)
    return v.to(torch.int32).contiguous()


def _xattn_ref(scores, v, lq, lk, causal, klens, causal_mask=lambda i, j: j > i):
    """scores float64 [n, h, lq, lk] (already scaled), v [n, h, lk, 64] -> [n*lq, h*64]."""
    n, h = scores.shape[:2]
    dev = scores.device
    i = torch.arange(lq, device=dev)[:, None]
    j = torch.arange(lk, device=dev)[None, :]
    mask = torch.zeros((n, 1, lq, lk), dtype=torch.bool, device=dev)
    if causal:
        mask = mask | causal_mask(i, j)
    if klens is not None:
        mask = mask | (j[None, None] >= klens.long()[:, None, None, None])
    p = torch.softmax(scores.masked_fill(mask, float("-inf")), dim=-1)
    return (p @ v).permute(0, 2, 1, 3).reshape(n * lq, h * 64)


@pytest.mark.parametrize("layout", ["self", "cross"])
def test_xattention_against_float64(layout, dev):
    """Both of the decoder's layouts: self-attention reads Q, K, V at columns 0, 512, 1024 of one [rows, 1536] buffer;
    decoder-encoder attention reads Q [rows, 512] and K | V [rows, 1024].  Every other case writes through ldo = H*64 +
    64 with a sentinel in the guard columns and in a guard row after the output, which must survive."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops
    lib = _lib.load()
    e16 = ops.enc16_dtype()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(31 if layout == "self" else 32)
    worst, off_by_one, cases = 0.0, float("inf"), 0
    sentinel = torch.tensor(-1234.0, dtype=e16, device=dev)
    for h, n in HN:
        for lq in LQ:
            for lk in LK:
                if layout == "self":
                    buf = (torch.randn(n * max(lq, lk), 1536, generator=g, device=dev) * 1.5).to(e16)
                    q, k, v = buf[:, :512], buf[:, 512:1024], buf[:, 1024:]
                    ptrs = (buf.data_ptr(), buf.data_ptr() + 512 * 2, buf.data_ptr() + 1024 * 2)
                    lds = (1536, 1536, 1536)
                else:
                    q = (torch.randn(n * lq, 512, generator=g, device=dev) * 1.5).to(e16)
                    kv = (torch.randn(n * lk, 1024, generator=g, device=dev) * 1.5).to(e16)
                    k, v = kv[:, :512], kv[:, 512:]
                    ptrs = (q.data_ptr(), kv.data_ptr(), kv.data_ptr() + 512 * 2)
                    lds = (512, 1024, 1024)
                Q = q[:n * lq, :h * 64].double().reshape(n, lq, h, 64).permute(0, 2, 1, 3)
                K = k[:n * lk, :h * 64].double().reshape(n, lk, h, 64).permute(0, 2, 1, 3)
                V = v[:n * lk, :h * 64].double().reshape(n, lk, h, 64).permute(0, 2, 1, 3)
                scores = (Q @ K.transpose(-1, -2)) * SCALE
                for causal in (0, 1):
                    for mode in KLENS:
                        kl = _klens(mode, n, lk, g, dev)
                        extra = 64 if (cases % 2) else 0
                        ldo = h * 64 + extra
                        out = torch.full((n * lq + 1, ldo), float(sentinel), dtype=e16, device=dev)
                        _lib.check(lib.sblk_xattention_fwd(*ptrs, out.data_ptr(), None if kl is None else kl.data_ptr(),
                                                           *lds, ldo, n, lq, lk, h, causal, SCALE, st),
                                   "sblk_xattention_fwd")
                        want = _xattn_ref(scores, V, lq, lk, causal, kl)
                        got = out[:n * lq, :h * 64]
                        worst = max(worst, _err(got, want) / _u())
                        assert (out[n * lq] == sentinel).all(), "write past the last output row"
                        if extra:
                            assert (out[:, h * 64:] == sentinel).all(), "write into the guard columns"
                        if mode == "zero":
                            assert got.reshape(n, lq, -1)[0::2].isnan().all() and not got.reshape(n, lq, -1)[1::2].isnan().any()
                        if causal and mode == "none" and lq == lk and lq >= 16:
                            # the subsequent mask off by one (key j >= query i also masked): row 0 is all-masked
                            # there, so measure rows 1.. of every clip
                            bad = _xattn_ref(scores, V, lq, lk, causal, None, causal_mask=lambda i, j: j >= i)
                            sl = (slice(None), slice(1, None))
                            off_by_one = min(off_by_one, _dist(got.reshape(n, lq, -1)[sl], bad.reshape(n, lq, -1)[sl]) / _u())
                        cases += 1
    _record(f"xattention_{layout}_U", worst, XATTN_BAR_U)
    assert cases == len(HN) * len(LQ) * len(LK) * 2 * len(KLENS)
    assert worst <= XATTN_BAR_U, f"xattention {layout}: {worst:.3f} U (bar {XATTN_BAR_U} U)"
    if layout == "self":
        _record("xattention_self_dist_causal_off_by_one_U", off_by_one, 10 * XATTN_BAR_U)
        assert off_by_one >= 10 * XATTN_BAR_U, off_by_one


# ------------------------------------------------------------------------------------------ sblk_embed_pe_fwd
@pytest.mark.parametrize("scale", [1.0, 0.5])
def test_embed_pe_against_float64(scale, dev):
    """tokens in the decoder's [N, 17] int64 buffers (row pitch 17 > L), ids 0 and vocab-1 included: the fp32 output is
    within one fp32 ulp of float64 and the enc16 output is the fp32 output rounded."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops
    from sbl_for_multilingual_lip_reading_b200.encoder import PositionalEncoding
    lib = _lib.load()
    e16 = ops.enc16_dtype()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(5)
    emb = torch.randn(VOCAB, 512, generator=g, device=dev).contiguous()
    pe = PositionalEncoding(512, max_len=5000).pe[0].to(dev).contiguous()
    n = 7
    worst = 0.0
    for L in (1, 2, 16):
        tok = torch.randint(0, VOCAB, (n, 17), generator=g, device=dev)
        tok[0, :L] = 0
        tok[1, :L] = VOCAB - 1
        tok[2, L - 1] = VOCAB - 1
        out32 = torch.empty((n * L, 512), dtype=torch.float32, device=dev)
        out16 = torch.empty((n * L, 512), dtype=e16, device=dev)
        _lib.check(lib.sblk_embed_pe_fwd(tok.data_ptr(), tok.stride(0), emb.data_ptr(), pe.data_ptr(), out32.data_ptr(),
                                         out16.data_ptr(), n * L, L, 512, VOCAB, scale, st), "sblk_embed_pe_fwd")
        want = (emb.double()[tok[:, :L]] * scale + pe.double()[:L]).reshape(n * L, 512)
        ulp = (torch.nextafter(out32.abs(), torch.tensor(float("inf"), device=dev)) - out32.abs()).double()
        worst = max(worst, float(((out32.double() - want).abs() / ulp).max()))
        assert torch.equal(out16, out32.to(e16))
        # the pad token rows read vocab row 0 / vocab-1
        assert torch.equal(out32.view(n, L, 512)[0], (emb[0] * scale + pe[:L]))
        assert torch.equal(out32.view(n, L, 512)[1], (emb[VOCAB - 1] * scale + pe[:L]))
    _record(f"embed_pe_fp32_ulps_scale{scale}", worst, 1.0)
    assert worst <= 1.0, f"{worst} ulp"


def test_embed_pe_clamps_out_of_range_ids(dev):
    """Ids below 0 read row 0 and ids >= vocab read row vocab-1 (include/sblk.h), with no error."""
    from sbl_for_multilingual_lip_reading_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(6)
    emb = torch.randn(VOCAB, 512, generator=g, device=dev)
    pe = torch.randn(16, 512, generator=g, device=dev)
    L = 4
    bad = torch.tensor([[-1, -(1 << 40), VOCAB, 1 << 40] + [0] * 13], dtype=torch.long, device=dev)
    clamped = torch.tensor([[0, 0, VOCAB - 1, VOCAB - 1] + [0] * 13], dtype=torch.long, device=dev)
    outs = []
    for tok in (bad, clamped):
        o = torch.empty((L, 512), dtype=torch.float32, device=dev)
        _lib.check(lib.sblk_embed_pe_fwd(tok.data_ptr(), 17, emb.data_ptr(), pe.data_ptr(), o.data_ptr(), None, L, L, 512,
                                         VOCAB, 1.0, st), "sblk_embed_pe_fwd")
        outs.append(o)
    assert torch.equal(outs[0], outs[1])


# ------------------------------------------------------------------------------------------ sblk_bidir_mix_fwd
def test_bidir_mix_is_the_aliased_loops_bit_for_bit(dev):
    """fp32 outputs bit-equal to the reference's in-place loops run in fp32 (the kernel claims their summation order),
    enc16 outputs bit-equal to the rounded fp32 outputs; odd L covers the middle element."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops
    lib = _lib.load()
    e16 = ops.enc16_dtype()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(8)
    for n in (1, 5):
        for L in (1, 2, 3, 16):
            l2r = torch.randn(n * L, 512, generator=g, device=dev) * 3
            r2l = torch.randn(n * L, 512, generator=g, device=dev) * 3
            a32, b32 = torch.empty_like(l2r), torch.empty_like(r2l)
            a16 = torch.empty((n * L, 512), dtype=e16, device=dev)
            b16 = torch.empty_like(a16)
            _lib.check(lib.sblk_bidir_mix_fwd(l2r.data_ptr(), r2l.data_ptr(), a32.data_ptr(), b32.data_ptr(),
                                              a16.data_ptr(), b16.data_ptr(), n, L, 512, st), "sblk_bidir_mix_fwd")
            wa, wb = O.bidir_mix(l2r.view(n, L, 512), r2l.view(n, L, 512))
            assert torch.equal(a32.view(n, L, 512), wa) and torch.equal(b32.view(n, L, 512), wb), (n, L)
            assert torch.equal(a16, a32.to(e16)) and torch.equal(b16, b32.to(e16))
            # the unaliased form (r2l + flip(l2r)) is a different function
            assert not torch.equal(b32.view(n, L, 512), r2l.view(n, L, 512) + l2r.view(n, L, 512).flip(1))


def test_decoder_entries_reject_bad_arguments_on_the_host(dev):
    """Argument checks that return an error before anything is launched."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops
    lib = _lib.load()
    e16 = ops.enc16_dtype()
    st = torch.cuda.current_stream().cuda_stream
    x = torch.zeros(4 * 512, dtype=torch.float32, device=dev)
    y = torch.zeros_like(x)
    o1, o2 = torch.empty_like(x), torch.empty_like(x)
    h1 = torch.empty(4 * 512 + 8, dtype=e16, device=dev)
    h2 = torch.empty_like(h1)
    mix = lambda *p: lib.sblk_bidir_mix_fwd(*p, 1, 4, 512, st)                        # noqa: E731
    for p in ((x, y, o1, o2, h1.data_ptr() + 2, h2.data_ptr()), (x, y, o1, o2, h1.data_ptr(), h2.data_ptr() + 4)):
        assert mix(p[0].data_ptr(), p[1].data_ptr(), p[2].data_ptr(), p[3].data_ptr(), p[4], p[5]) != 0
        assert "8-byte" in _lib.last_error()
    assert mix(x.data_ptr(), y.data_ptr(), x.data_ptr(), o2.data_ptr(), h1.data_ptr(), h2.data_ptr()) != 0
    assert "alias" in _lib.last_error()
    assert mix(x.data_ptr(), y.data_ptr(), o1.data_ptr(), y.data_ptr(), h1.data_ptr(), h2.data_ptr()) != 0
    assert mix(x.data_ptr(), y.data_ptr(), o1.data_ptr(), o2.data_ptr(), h1.data_ptr() + 8, h2.data_ptr()) == 0
    torch.cuda.synchronize()
    q = torch.zeros((64 * 129, 1536), dtype=e16, device=dev)
    out = torch.zeros((64 * 33, 512), dtype=e16, device=dev)
    att = lambda lq, lk: lib.sblk_xattention_fwd(q.data_ptr(), q.data_ptr(), q.data_ptr(), out.data_ptr(), None,  # noqa
                                                 1536, 1536, 1536, 512, 1, lq, lk, 8, 1, SCALE, st)
    assert att(33, 16) != 0 and "Lq <= 32" in _lib.last_error()
    assert att(16, 129) != 0 and "Lk <= 128" in _lib.last_error()
    assert att(32, 128) == 0
    tok = torch.zeros((1, 17), dtype=torch.long, device=dev)
    emb = torch.zeros((VOCAB, 512), device=dev)
    o = torch.empty((1, 512), device=dev)
    assert lib.sblk_embed_pe_fwd(tok.data_ptr(), 17, emb.data_ptr(), emb.data_ptr(), o.data_ptr(), h1.data_ptr() + 2,
                                 1, 1, 512, VOCAB, 1.0, st) != 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ GEMM / LayerNorm entries
GEMM_M = (1, 5, 16, 17, 127, 129, 2304, 2305, 8192)


def _operands(m, n, k, g, dev, e16):
    a = torch.randn(m, k, generator=g, device=dev).to(e16)
    w = (torch.randn(n, k, generator=g, device=dev) / k ** 0.5).to(e16)
    bias = torch.randn(n, generator=g, device=dev) * 0.1
    return a, w, bias


@pytest.mark.parametrize("m", GEMM_M)
def test_gemm_against_float64(m, dev):
    """ops.gemm at the decoder's row counts (M = N*L from a single row up): bias + residual + ReLU with 16-bit and fp32
    outputs, and the plain product into fp32."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    e16 = ops.enc16_dtype()
    g = torch.Generator(device=dev).manual_seed(1000 + m)
    w16, w32 = 0.0, 0.0
    for k in (512, 2048):
        for n in (64, 512, 1024, 1536, 2048):
            a, w, bias = _operands(m, n, k, g, dev, e16)
            res = torch.randn(m, n, generator=g, device=dev).to(e16)
            prod = a.double() @ w.double().t()
            o16, o32 = ops.gemm(a, w, bias=bias, residual=res, relu=True, out_bf16=True, out_f32=True)
            want = torch.relu(prod + bias.double() + res.double())
            w16 = max(w16, _err(o16, want) / _u())
            w32 = max(w32, _err(o32, want))
            _, p32 = ops.gemm(a, w, out_f32=True)
            w32 = max(w32, _err(p32, prod))
    _record("gemm_16bit_out_U", w16, GEMM16_BAR_U)
    _record("gemm_fp32_out", w32, GEMM32_BAR)
    assert w16 <= GEMM16_BAR_U, (m, w16)
    assert w32 <= GEMM32_BAR, (m, w32)


@pytest.mark.parametrize("m", GEMM_M)
def test_linear_ln_against_float64(m, dev):
    """ops.linear_ln (Linear + bias + fp32 residual + LayerNorm(512)) with fused = None / True / False: the split-K pair
    and the one-launch cluster kernel, each at every decoder row count; fused=None picks the cluster kernel on a
    148-SM B200 only from M = 2305 on."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    e16 = ops.enc16_dtype()
    g = torch.Generator(device=dev).manual_seed(2000 + m)
    T = max(L for L in range(1, 17) if m % L == 0)          # T = L, the prefix length of the rows
    w32, w16 = 0.0, 0.0
    for k in (512, 2048):
        a, w, bias = _operands(m, 512, k, g, dev, e16)
        res = torch.randn(m, 512, generator=g, device=dev)
        gamma = torch.rand(512, generator=g, device=dev) + 0.5
        beta = torch.randn(512, generator=g, device=dev) * 0.1
        z = a.double() @ w.double().t() + bias.double() + res.double()
        want = torch.nn.functional.layer_norm(z, (512,), gamma.double(), beta.double(), 1e-5)
        for fused in (None, True, False):
            tr = []
            with ops.trace(tr):
                o32, o16 = ops.linear_ln(a, w, gamma, beta, bias=bias, residual=res, T=T, eps=1e-5, fused=fused)
            names = [t_["name"] for t_ in tr]
            one_launch = names == ["sblk_gemm_ln_fwd"]
            assert one_launch or names == ["sblk_gemm_splitk_fwd", "sblk_sum_layernorm_fwd"], names
            if fused is not None:
                assert one_launch == fused
            elif torch.cuda.get_device_properties(dev).multi_processor_count == 148:
                assert one_launch == (m >= 2305), (m, names)
            w32 = max(w32, _err(o32, want))
            w16 = max(w16, _err(o16, want) / _u())
    _record("linear_ln_fp32_out", w32, LN32_BAR)
    _record("linear_ln_16bit_out_U", w16, LN16_BAR_U)
    assert w32 <= LN32_BAR, (m, w32)
    assert w16 <= LN16_BAR_U, (m, w16)


# ------------------------------------------------------------------------------------------ the whole decoder
@pytest.fixture(scope="module")
def enc_pool(dev):
    """Encoder outputs of the drop-in frontend + encoder (synthetic weights) on structured clips: 200 clips of 29
    frames (t_enc = 1 uses their first frame) and 32 clips of 128 frames; get(n, t) tiles them to n clips."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    enc = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1)
    enc.load_state_dict(synth.encoder_state_dict(2, 6))
    fe, enc = fe.to(dev).eval(), enc.to(dev).eval()
    fe.always_on_dropout = False
    pool = {}
    with torch.no_grad():
        for clips, t in ((200, 29), (32, 128)):
            outs = []
            for c0 in range(0, clips, 40):
                c = min(40, clips - c0)
                x = synth.structured_clips(c, t, seed=700 + t + c0).to(dev)
                outs.append(enc(fe(x), [t] * c)[0].float())
            pool[t] = torch.cat(outs).contiguous()

    def get(n, t):
        base = pool[128] if t == 128 else pool[29][:, :t]
        return base[torch.arange(n, device=dev) % base.shape[0]].contiguous()
    return get


def _decoder(n_layers, dev):
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    torch.manual_seed(7)                                   # the reference initialisation under a fixed seed
    return Decoder(SOS, EOS, VOCAB, 512, n_layers, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                   pe_maxlen=5000).to(dev).eval()


def _sd64(dec, dev):
    return {k: v.detach().to(dev, torch.float64) for k, v in dec.state_dict().items()}


def _targets(n, seed):
    """[n, 14] l2r targets (ids in [2, 58)) with ragged lengths, IGNORE_ID inside and after the tokens, and a
    zero-length target in row 0; r2l = the kept tokens reversed, in the same slots."""
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


def _oracle_steps(sd, ys_l2r, ys_r2l, enc, **variant):
    steps = [O.step_logits(sd, ys_l2r, ys_r2l, enc, L, **variant) for L in range(1, O.MAXLEN + 1)]
    return torch.stack([s[0] for s in steps], 1), torch.stack([s[1] for s in steps], 1)


def _unaliased_mix(l2r, r2l):
    return l2r + r2l.flip(1), r2l + l2r.flip(1)


# (n_layers, N, t_enc, fused_ln): every value of every factor at least once; N = 512 reaches the cluster LayerNorm
# kernel through fused_ln=None from prefix length 5 on (M = 512 * L >= 2305)
TF_CASES = [(1, 1, 1, None), (2, 5, 29, None), (6, 5, 29, True), (6, 5, 128, False), (2, 512, 29, None),
            (6, 512, 128, None), (1, 512, 1, False), (2, 1, 128, True), (6, 1, 29, None)]


@pytest.mark.parametrize("case", TF_CASES, ids=lambda c: "L{}-N{}-T{}-fused{}".format(*c))
def test_teacher_forced_logits_against_float64(case, dev, enc_pool, monkeypatch):
    """Decoder.forward with the coin forced to the gold token on ragged targets (interior IGNORE_ID, one empty target):
    every step's logits against the oracle's step_logits on the oracle's ys_in_pad, with the two directions on two
    streams and on one (bit-identical)."""
    from sbl_for_multilingual_lip_reading_b200 import decoder as decoder_mod
    n_layers, n, t, fused = case
    dec = _decoder(n_layers, dev)
    dec.fused_ln = fused
    enc = enc_pool(n, t)
    tgt, tgt_r = _targets(n, seed=n * 1000 + t + n_layers)
    monkeypatch.setattr(decoder_mod.random, "random", lambda: 0.0)           # `random.random() > 0.5` never: gold
    outs = {}
    with torch.no_grad():
        for two in (True, False):
            dec.two_streams = two
            outs[two] = dec(tgt.to(dev), tgt_r.to(dev), enc, [t] * n)
    assert len(dec._plans) == 2                                               # one captured plan per setting
    a, b = outs[True], outs[False]
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])
    in_l2r, out_l2r = O.preprocess(tgt, SOS, EOS)
    in_r2l, out_r2l = O.preprocess(tgt_r, SOS, EOS)
    assert torch.equal(a[1].cpu(), out_l2r) and torch.equal(a[3].cpu(), out_r2l)
    sd = _sd64(dec, dev)
    enc64 = enc.double()
    ys_l2r, ys_r2l = in_l2r.to(dev), in_r2l.to(dev)
    with torch.no_grad():
        want = _oracle_steps(sd, ys_l2r, ys_r2l, enc64)
        err = max(_err(a[0], want[0]), _err(a[2], want[1])) / _u()
        _record("teacher_forced_logits_U", err, LOGITS_BAR_U)
        MEASURED.setdefault("teacher_forced_logits_U_per_case", {})["L{}-N{}-T{}-fused{}".format(*case)] = err
        assert err <= LOGITS_BAR_U, (case, err)
        if case == (6, 5, 29, True):
            variants = {"causal_mask_j_ge_i": dict(mask=lambda n_, L, d: torch.triu(
                            torch.ones(L, L, dtype=torch.bool, device=d), 0).expand(n_, -1, -1)),
                        "causal_mask_leaks_next_key": dict(mask=lambda n_, L, d: torch.triu(
                            torch.ones(L, L, dtype=torch.bool, device=d), 2).expand(n_, -1, -1)),
                        "mask_in_every_layer": dict(mask_every_layer=True),
                        "unaliased_mixing": dict(mix=_unaliased_mix)}
            for name, kw in variants.items():
                bad = _oracle_steps(sd, ys_l2r, ys_r2l, enc64, **kw)
                dist = max(_dist(a[0], bad[0]), _dist(a[2], bad[1])) / _u()
                _record("teacher_forced_dist_" + name + "_U", dist, 10 * LOGITS_BAR_U)
                assert dist >= 10 * LOGITS_BAR_U, (name, dist)


def _first_divergence(a, b):
    """per clip: index of the first decode step whose emitted token differs (16 = never).  a, b: [N, 17] with <sos>."""
    ne = a[:, 1:] != b[:, 1:]
    return torch.where(ne.any(1), ne.float().argmax(1), torch.full((a.shape[0],), ne.shape[1], device=a.device)).long()


def test_greedy_decode_against_float64_200_clips(dev, enc_pool):
    """recognize_beam on 200 clips against the oracle's greedy decode, margin-aware: every sequence whose smallest oracle
    top-1/top-2 margin is clear of 2x the largest logit difference (on the steps whose prefixes are still identical in
    both directions) decodes identically; near-ties are counted.  With these weights many r2l sequences pass through
    near-ties (76 of 200 on a B200, 10 of them decoded differently), so the share of identical sequences is held at
    GREEDY_MIN_SAME: twice the measured number of differing sequences."""
    dec = _decoder(6, dev)
    n = 200
    enc = enc_pool(n, 29)
    with torch.no_grad():
        toks = dec.recognize_beam(enc)
        got = dec._greedy(enc, want_logits=True)
        want = O.greedy(_sd64(dec, dev), enc.double())
    assert torch.equal(toks[0], got[0]) and torch.equal(toks[1], got[1])
    fd = torch.minimum(_first_divergence(want[0], got[0]), _first_divergence(want[1], got[1]))
    valid = torch.arange(O.MAXLEN, device=dev)[None, :] <= fd[:, None]
    res = {}
    for di, d in enumerate(("l2r", "r2l")):
        la, lb = want[2 + di], got[2 + di]
        top2 = la.topk(2, dim=-1).values
        margin = (top2[..., 0] - top2[..., 1]).min(dim=1).values
        thr = 2.0 * float(((lb.double() - la).abs().max(dim=-1).values * valid).max())
        same = (want[di] == got[di]).all(1)
        clear = margin > thr
        res[d] = {"same": int(same.sum()), "clear": int(clear.sum()), "clear_same": int((same & clear).sum()),
                  "near_ties": int((~clear).sum()), "margin_threshold_logits": thr,
                  "distinct_sequences": len({tuple(r) for r in want[di].tolist()})}
    MEASURED["greedy_200_clips"] = res
    print(json.dumps(res))
    for d in ("l2r", "r2l"):
        assert res[d]["clear_same"] == res[d]["clear"], (d, res[d])
        assert res[d]["same"] >= GREEDY_MIN_SAME, (d, res[d])
