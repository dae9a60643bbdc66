"""GPU parity tests (run with -m gpu on a B200): the libsblk path, called through the drop-in modules and
the C ABI, against (1) the golden outputs of the reference itself, (2) the CPU oracle on seeded inputs at
small sizes, and (3) size-independent properties at the BASELINE config sizes.

Tolerance (BASELINE.json north_star): encoder outputs within 1e-2 relative error (bf16 operands, fp32
accumulation) — measured as relative Frobenius error; features of the frontend get the same bar.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REL_TOL = 1e-2


def rel_fro(a, b):
    a = torch.as_tensor(a).float().cpu()
    b = torch.as_tensor(b).float().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    assert torch.isfinite(a).all()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    assert ops.init() > 0
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def frontend(dev):
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    m = Lipreading()
    m.load_state_dict(synth.frontend_state_dict(1))
    m.always_on_dropout = False
    return m.to(dev).eval()


@pytest.fixture(scope="module")
def encoder6(dev):
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    m = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
    m.load_state_dict(synth.encoder_state_dict(2, 6))
    return m.to(dev).eval()


# ------------------------------------------------------------------ golden vectors (reference outputs)
def test_golden_frontend_config1(frontend, dev, golden):
    """BASELINE config 1: one 29x88x88 clip, Conv3d frontend + ResNet-18 trunk."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(1, 29, seed=7).to(dev)
    with torch.no_grad():
        feat = frontend._frontend_forward(x)
        out = frontend(x)
    assert out.shape == (1, 29, 512) and out.dtype == torch.float32
    assert rel_fro(feat, golden["frontend_c1"]) < REL_TOL


def test_golden_frontend_zero_padded_frames(frontend, dev, golden):
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(2, 6, seed=8, pad_frames=1).to(dev)
    with torch.no_grad():
        assert rel_fro(frontend._frontend_forward(x), golden["frontend_N2_T6_pad1"]) < REL_TOL


def test_golden_stem(frontend, dev, golden):
    """Conv3d + BN + ReLU + MaxPool3d kernel alone vs the reference's frontend3D output."""
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    x = synth.synthetic_clips(1, 2, seed=11).to(dev)
    pk = frontend._get_packed()
    out = ops.conv3d_bn_relu_pool(ops.prep_clip(x), pk.c3w, pk.c3b)            # [F,22,22,64] NHWC
    ref = torch.from_numpy(golden["frontend3d_T2"])[0].permute(1, 2, 3, 0)     # [64,T,22,22] -> [T,22,22,64]
    assert rel_fro(out, ref) < REL_TOL


def test_golden_encoder(encoder6, dev, golden, golden_inputs):
    with torch.no_grad():
        out = encoder6(torch.from_numpy(golden_inputs["xin"]).to(dev), [29])
        assert isinstance(out, tuple) and len(out) == 1
        assert rel_fro(out[0], golden["encoder6_N1_T29"]) < REL_TOL
        out40, = encoder6(torch.from_numpy(golden_inputs["xin40"]).to(dev), [40])
        assert rel_fro(out40, golden["encoder6_N1_T40"]) < REL_TOL


def test_golden_encoder_three_layers(dev, golden, golden_inputs):
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    enc3 = Encoder(512, 3, 8, 64, 64, 512, 2048)
    enc3.load_state_dict(synth.encoder_state_dict(3, 3))
    enc3 = enc3.to(dev).eval()
    with torch.no_grad():
        out, = enc3(torch.from_numpy(golden_inputs["xin3"]).to(dev), [31, 31])
    assert rel_fro(out, golden["encoder3_N2_T31"]) < REL_TOL


def test_golden_encoder_ragged_lengths_and_attns(encoder6, dev, golden, golden_inputs):
    with torch.no_grad():
        out, attns = encoder6(torch.from_numpy(golden_inputs["xin_r"]).to(dev), [12, 7, 1], return_attns=True)
    assert rel_fro(out, golden["encoder6_ragged_out"]) < REL_TOL
    assert len(attns) == 6 and attns[0].shape == (24, 12, 12)
    assert rel_fro(attns[0], golden["encoder6_ragged_attn0"]) < REL_TOL
    assert rel_fro(attns[5], golden["encoder6_ragged_attn5"]) < REL_TOL
    assert float(out[1, 7:].abs().max()) == 0.0 and float(out[2, 1:].abs().max()) == 0.0


def test_golden_whole_hot_path(frontend, encoder6, dev, golden):
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(2, 6, seed=8, pad_frames=1).to(dev)
    with torch.no_grad():
        feat = frontend(x)
        out, = encoder6(feat, [6, 6])
    assert rel_fro(out, golden["visual_encoder_N2_T6"]) < REL_TOL


# ------------------------------------------------------------------ oracle on seeded inputs
@pytest.mark.parametrize("n,t", [(1, 1), (1, 5), (3, 7), (2, 29), (1, 40)])
def test_oracle_whole_path(frontend, encoder6, dev, n, t):
    from oracle import visual_encoder_oracle as O
    from sbl_for_multilingual_lip_reading_b200 import synth
    sd = {}
    sd.update(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, 6, prefix="encoder."))
    x = synth.synthetic_clips(n, t, seed=100 + n * 50 + t)
    with torch.no_grad():
        ref_feat = O.lipreading_forward(x, sd, "visual_frontend.")
        ref = O.visual_encoder_forward(x, sd)
        feat = frontend(x.to(dev))
        out, = encoder6(feat, [t] * n)
    assert rel_fro(feat, ref_feat) < REL_TOL
    assert rel_fro(out, ref) < REL_TOL


def test_oracle_basic_block_chain(frontend, dev):
    """Every ResNet stage boundary against the oracle (catches a wrong layer that later layers would blur)."""
    from oracle import visual_encoder_oracle as O
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(1, 3, seed=5)
    with torch.no_grad():
        y = O.frontend3d(x, sd).transpose(1, 2).contiguous().view(-1, 64, 22, 22)
        pk = frontend._get_packed()
        a = ops.conv3d_bn_relu_pool(ops.prep_clip(x.to(dev)), pk.c3w, pk.c3b, flat=True)   # zero-haloed flat layout
        assert rel_fro(a.dense().permute(0, 3, 1, 2), y) < REL_TOL
        bi = 0
        for li, stride in ((1, 1), (2, 2), (3, 2), (4, 2)):
            for b in range(2):
                y = O.basic_block(y, sd, f"resnet18.layer{li}.{b}", stride if b == 0 else 1, b == 0 and li != 1)
                (st, w1, b1, w2, b2, ds) = pk.blocks[bi]
                if isinstance(a, ops.FlatActs) and st == 1 and ds is None:   # layer1, layer2.1: flat shifted-window kernel
                    h = ops.conv3x3_flat(a, w1, b1, relu=True)
                    a = ops.conv3x3_flat(h, w2, b2, relu=True, residual=a)
                elif ds is not None and w2.dim() == 2:   # layer2.0: fused conv1 + downsample writes the flat layout
                    h, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=st, relu=True,
                                             flat_ws=frontend._flat_workspace(a, w1.shape[0], st))
                    a = ops.conv3x3_flat(h, w2, b2, relu=True, residual=res)
                else:         # layers 3-4: TMA-im2col kernels on dense NHWC (unfused conv1 / downsample here)
                    h = ops.conv2d(a, w1, b1, stride=st, relu=True)
                    res = a if ds is None else ops.conv2d(a, ds[0], ds[1], stride=st, relu=False)
                    a = ops.conv2d(h, w2, b2, stride=1, relu=True, residual=res)
                got = a.dense() if isinstance(a, ops.FlatActs) else a
                assert rel_fro(got.permute(0, 3, 1, 2), y) < REL_TOL, f"layer{li}.{b}"
                bi += 1


@pytest.mark.parametrize("f,h,cin,cout,flat_in", [(5, 11, 128, 256, True), (29, 11, 128, 256, False),
                                                  (7, 6, 256, 512, False), (3, 22, 64, 128, True)])
def test_conv2d_k_extension_folds_the_downsample_branch(dev, f, h, cin, cout, flat_in):
    """sblk_conv2d_igemm_ext_fwd: relu(conv3x3(y) + conv1x1_s2(x) + bias) in one accumulator (BasicBlock conv2 + the
    downsample branch, video_frontend.py:35-41,68-72) against a torch fp32 reference of the same bf16 operands, and
    against the unfused launches (which round the branch to bf16 first).  Ragged M (last pair tile partly empty),
    dense and flat (pitched) block inputs, 128- and 256-wide tiles."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(f * 1000 + h)
    bf = torch.bfloat16
    p = (h - 1) // 2 + 1
    x = torch.randn(f, h, h, cin, generator=g).to(bf)
    y = torch.randn(f, p, p, cout, generator=g).to(bf)
    w2 = (torch.randn(cout, 3, 3, cout, generator=g) / (3 * cout ** 0.5)).to(bf)
    wd = (torch.randn(cout, 1, 1, cin, generator=g) / cin ** 0.5).to(bf)
    bias = torch.randn(cout, generator=g)
    ref = torch.nn.functional.conv2d(y.float().permute(0, 3, 1, 2), w2.float().permute(0, 3, 1, 2), padding=1)
    ref = ref + torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), wd.float().permute(0, 3, 1, 2), stride=2)
    ref = torch.relu(ref + bias.view(1, -1, 1, 1)).permute(0, 2, 3, 1)
    xd = x.to(dev)
    if flat_in:
        xin = ops.FlatActs(torch.zeros(ops.flat_rows(f, h, h), cin, dtype=bf, device=dev), f, h, h)
        xin.data.view(-1)[:] = 0
        rows = ((torch.arange(f).view(-1, 1, 1) * (h + 1) + 1 + torch.arange(h).view(1, -1, 1)) * (h + 2) + 1 +
                torch.arange(h).view(1, 1, -1)).reshape(-1).to(dev)
        xin.data[rows] = xd.reshape(-1, cin)
    else:
        xin = xd
    yd, w2d, wdd, bd = y.to(dev), w2.to(dev), wd.to(dev), bias.to(dev)
    got = ops.conv2d(yd, w2d, bd, stride=1, relu=True, ext=(xin, wdd, 2))
    torch.cuda.synchronize()
    assert tuple(got.shape) == (f, p, p, cout)
    assert rel_fro(got, ref) < 4e-3          # one bf16 rounding of the output
    zero = torch.zeros(cout, device=dev)
    res = ops.conv2d(xin, wdd, zero, stride=2, relu=False)
    unfused = ops.conv2d(yd, w2d, bd, stride=1, relu=True, residual=res)
    assert rel_fro(got, unfused) < 6e-3      # the unfused form rounds the branch to bf16 before adding it
    # the extension must not disturb the plain conv: zero extension filter == no extension, bit for bit
    plain = ops.conv2d(yd, w2d, bd, stride=1, relu=True)
    got0 = ops.conv2d(yd, w2d, bd, stride=1, relu=True, ext=(xin, torch.zeros_like(wdd), 2))
    assert torch.equal(plain, got0)


def test_fold_downsample_matches_dual_heads(frontend, dev):
    """Lipreading.fold_downsample (layers 3-4: conv1 on 256-wide tiles, branch folded into conv2) against the dual-head
    path of round 1 and the oracle."""
    from oracle import visual_encoder_oracle as O
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(2, 7, seed=21)
    sd = synth.frontend_state_dict(1, prefix="visual_frontend.")
    old = frontend.fold_downsample
    try:
        with torch.no_grad():
            frontend.fold_downsample = True
            a = frontend._frontend_forward(x.to(dev))
            frontend.fold_downsample = False
            b = frontend._frontend_forward(x.to(dev))
            ref = O.lipreading_forward(x, sd, "visual_frontend.")
    finally:
        frontend.fold_downsample = old
    assert rel_fro(a, b) < 4e-3
    assert rel_fro(a.view(-1, 512), ref.view(-1, 512)) < REL_TOL
    assert rel_fro(a.view(-1, 512), ref.view(-1, 512)) <= rel_fro(b.view(-1, 512), ref.view(-1, 512)) * 1.1


@pytest.mark.parametrize("f,h,cin,cout,stride,flat_in", [
    (29, 11, 128, 256, 2, True), (928, 11, 128, 256, 2, True), (5, 6, 256, 256, 1, False), (928, 6, 256, 256, 1, False),
    (1, 6, 256, 256, 1, False), (9, 12, 64, 256, 2, False),
    (928, 6, 256, 512, 2, False), (928, 3, 512, 512, 1, False), (30, 6, 256, 512, 2, False), (3, 3, 512, 512, 1, False)])
def test_conv_block_is_bit_identical_to_the_two_launches(dev, f, h, cin, cout, stride, flat_in):
    """sblk_conv_block_fwd (a whole layer-3 / layer-4 BasicBlock in one launch: pair tiles of whole frames run conv1 and
    then conv2, video_frontend.py:28-41,68-72) against the conv-by-conv launches: same bits, for head blocks (stride 2 +
    folded downsample branch, flat or dense input) and identity blocks, Cout = 256 (pair-wide mbarrier) and 512 (two
    column tiles on neighbouring pairs, self-resetting global counters — launched three times to check the reset), one
    tile / partial last tile / several units per CTA pair, and a limited grid."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(f * 10 + h + cout)
    bf = torch.bfloat16
    x = torch.randn(f, h, h, cin, generator=g).to(bf).to(dev)
    w1 = (torch.randn(cout, 3, 3, cin, generator=g) / (9 * cin) ** 0.5).to(bf).to(dev)
    w2 = (torch.randn(cout, 3, 3, cout, generator=g) / (9 * cout) ** 0.5).to(bf).to(dev)
    b1, b2 = torch.randn(cout, generator=g).to(dev), torch.randn(cout, generator=g).to(dev)
    head = stride == 2 or cin != cout
    wd = (torch.randn(cout, 1, 1, cin, generator=g) / cin ** 0.5).to(bf).to(dev) if head else None
    if flat_in:
        xin = ops.FlatActs(torch.zeros(ops.flat_rows(f, h, h), cin, dtype=bf, device=dev), f, h, h)
        rows = ((torch.arange(f).view(-1, 1, 1) * (h + 1) + 1 + torch.arange(h).view(1, -1, 1)) * (h + 2) + 1 +
                torch.arange(h).view(1, 1, -1)).reshape(-1).to(dev)
        xin.data[rows] = x.reshape(-1, cin)
    else:
        xin = x
    y = ops.conv2d(xin, w1, b1, stride=stride, relu=True)
    if head:
        want = ops.conv2d(y, w2, b2, stride=1, relu=True, ext=(xin, wd, stride))
    else:
        want = ops.conv2d(y, w2, b2, stride=1, relu=True, residual=x)
    for limit in (0, 0, 0, 24, 4):
        prev = ops.set_sm_limit(limit) if limit else None
        try:
            got = ops.conv_block(xin, w1, b1, w2, b2, w_ds=wd, stride=stride)
        finally:
            if prev is not None:
                ops.set_sm_limit(prev)
        torch.cuda.synchronize(dev)
        if got is None:      # more than 32 units per CTA pair on the limited grid: the caller launches conv by conv
            assert limit == 4 and f > 100
            continue
        assert torch.equal(got, want), (limit,)


def test_fuse_blocks_leaves_the_frontend_bit_identical(frontend, dev):
    """Lipreading.fuse_blocks (layers 3-4 as one launch per block) returns exactly the features of the conv-by-conv path."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(3, 9, seed=33).to(dev)
    old = frontend.fuse_blocks
    try:
        with torch.no_grad():
            frontend.fuse_blocks = True
            a = frontend._frontend_forward(x)
            frontend.fuse_blocks = False
            b = frontend._frontend_forward(x)
    finally:
        frontend.fuse_blocks = old
    assert torch.equal(a, b)


# ------------------------------------------------------------------ edge cases and error behaviour
def test_dropout_always_on_like_reference(dev):
    """Reference quirk (video_frontend.py:122): dropout(0.5) is active in eval mode; same torch RNG call."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    m = Lipreading()
    m.load_state_dict(synth.frontend_state_dict(1))
    m = m.to(dev).eval()
    x = synth.synthetic_clips(1, 4, seed=9).to(dev)
    with torch.no_grad():
        torch.manual_seed(3)
        a = m(x)
        torch.manual_seed(3)
        b = m(x)
        c = m(x)
        feat = m._frontend_forward(x)
        torch.manual_seed(3)
        expect = torch.nn.functional.dropout(feat, p=0.5).view(1, 4, 512)
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert torch.equal(a, expect)
    zeros = (a == 0).float().mean().item()
    assert 0.4 < zeros < 0.7


def test_state_dict_reload_invalidates_packed_weights(dev):
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    enc = Encoder(512, 1, 8, 64, 64, 512, 2048)
    enc.load_state_dict(synth.encoder_state_dict(5, 1))
    enc = enc.to(dev).eval()
    x = torch.randn(2, 9, 512, device=dev)
    with torch.no_grad():
        a, = enc(x, [9, 9])
        enc.load_state_dict(synth.encoder_state_dict(6, 1))
        b, = enc(x, [9, 9])
        enc.load_state_dict(synth.encoder_state_dict(5, 1))
        c, = enc(x, [9, 9])
    assert not torch.allclose(a, b) and torch.equal(a, c)


def test_c_abi_rejects_bad_arguments(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops
    with pytest.raises(RuntimeError, match="multiples of 64"):
        ops.gemm(torch.zeros(8, 48, dtype=ops.enc16_dtype(), device=dev),
                 torch.zeros(64, 48, dtype=ops.enc16_dtype(), device=dev), out_f32=True)
    with pytest.raises(RuntimeError, match="only 512"):
        ops.add_layernorm(torch.zeros(4, 256, device=dev), torch.ones(256, device=dev), torch.zeros(256, device=dev))
    with pytest.raises(RuntimeError, match="T=200"):
        ops.attention(torch.zeros(200, 1536, dtype=ops.enc16_dtype(), device=dev), 1, 200, 8)
    with pytest.raises(RuntimeError, match="expected dtype"):
        ops.conv2d(torch.zeros(1, 22, 22, 64, device=dev), torch.zeros(64, 3, 3, 64, dtype=torch.bfloat16, device=dev),
                   torch.zeros(64, device=dev))
    # K-extension (sblk_conv2d_igemm_ext_fwd): the branch's output grid must be the conv's; Cout must allow the CTA-pair kernel
    bf = torch.bfloat16
    y = torch.zeros(2, 6, 6, 128, dtype=bf, device=dev)
    w = torch.zeros(128, 3, 3, 128, dtype=bf, device=dev)
    with pytest.raises(RuntimeError, match="output grid"):
        ops.conv2d(y, w, torch.zeros(128, device=dev), ext=(torch.zeros(2, 9, 9, 64, dtype=bf, device=dev),
                                                           torch.zeros(128, 1, 1, 64, dtype=bf, device=dev), 2))
    with pytest.raises(RuntimeError, match="do not match"):
        ops.conv2d(y, w, torch.zeros(128, device=dev), ext=(torch.zeros(2, 11, 11, 64, dtype=bf, device=dev),
                                                           torch.zeros(64, 1, 1, 64, dtype=bf, device=dev), 2))
    lib_err = None
    try:   # Cout = 64: no CTA-pair kernel -> the C ABI refuses (no silent fallback)
        ops.conv2d(torch.zeros(2, 6, 6, 64, dtype=bf, device=dev), torch.zeros(64, 3, 3, 64, dtype=bf, device=dev),
                   torch.zeros(64, device=dev), ext=(torch.zeros(2, 11, 11, 64, dtype=bf, device=dev),
                                                     torch.zeros(64, 1, 1, 64, dtype=bf, device=dev), 2))
    except RuntimeError as e:
        lib_err = str(e)
    assert lib_err is not None and "CTA-pair" in lib_err


# ------------------------------------------------------------------ one-launch encoder stack (cluster kernel)
@pytest.mark.parametrize("n,t,lens", [(1, 1, None), (4, 29, None), (5, 29, [29, 3, 17, 29, 1]), (3, 40, [40, 17, 1]),
                                      (9, 31, None), (2, 100, [100, 64]), (32, 29, None), (40, 30, None)])
def test_encoder_stack_matches_oracle_and_per_step_kernels(encoder6, dev, n, t, lens):
    """sblk_encoder_stack_fwd (one launch, a thread-block cluster per clip group) against the CPU oracle and against
    the per-step kernels, for single / multiple / partial groups, ragged lengths and both cluster sizes
    (<= 7 groups run clusters of 16 CTAs, more run clusters of 8)."""
    from oracle import visual_encoder_oracle as O
    from sbl_for_multilingual_lip_reading_b200 import synth
    g = torch.Generator().manual_seed(1000 + 31 * n + t)
    x = torch.randn(n, t, 512, generator=g)
    ln = lens if lens is not None else [t] * n
    assert encoder6._use_fused_stack(n, t, False)
    with torch.no_grad():
        fused, = encoder6(x.to(dev), ln)
        encoder6.fused_stack = False
        try:
            steps, = encoder6(x.to(dev), ln)
        finally:
            encoder6.fused_stack = True
        ref = O.encoder_forward(x, ln, synth.encoder_state_dict(2, 6), n_layers=6)[0]
    assert rel_fro(fused, ref) < REL_TOL
    assert rel_fro(fused, steps) < REL_TOL
    if lens is not None:   # `*= non_pad_mask` (encoder.py:86,89): padded positions are exactly zero
        for b, l_ in enumerate(lens):
            assert float(fused[b, l_:].abs().max() if l_ < t else 0.0) == 0.0


def test_encoder_stack_cluster_sizes_agree(encoder6, dev):
    """Clusters of 8 and of 16 CTAs, with and without TMA multicast of the activation tiles, are bit-identical
    (LayerNorm statistics are merged from the same sixteen 32-column partials in the same order), so a clip's
    output does not depend on how many clips share its batch."""
    g = torch.Generator().manual_seed(77)
    x = torch.randn(6, 29, 512, generator=g).to(dev)
    from sbl_for_multilingual_lip_reading_b200 import ops
    outs = []
    lens = torch.tensor([29, 29, 5, 29, 12, 29], dtype=torch.int32, device=dev)
    with torch.no_grad():
        stk = encoder6._get_packed().stacked
        x16 = ops.cast_enc16(x.view(-1, 512).contiguous())
        for cl, mc in ((16, True), (16, False), (8, True), (8, False)):
            outs.append(ops.encoder_stack(x16, stk, 6, 29, lengths=lens, cluster_size=cl, multicast=mc).clone())
        outs.append(encoder6(x, [29, 29, 5, 29, 12, 29])[0].reshape(-1, 512).clone())
    assert all(torch.equal(outs[0], o) for o in outs[1:])


@pytest.mark.parametrize("n,t,ragged", [(32, 29, False), (7, 29, True), (9, 40, True), (1, 5, False), (7, 100, False)])
def test_encoder_stack_two_groups_per_cluster_is_bit_identical(encoder6, dev, n, t, ragged):
    """groups_per_cluster=2: a cluster runs two clip groups through the stack alternately (second TMEM accumulator,
    loads / MMAs of one group behind the epilogues / barriers of the other).  All arithmetic is per group, so the
    output equals the one-group-per-cluster launch bit for bit — odd group counts (a cluster with a single group),
    partial groups, ragged lengths, both cluster sizes."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(5000 + 17 * n + t)
    x16 = ops.cast_enc16(torch.randn(n * t, 512, generator=g).to(dev))
    lens = torch.randint(1, t + 1, (n,), generator=g).to(torch.int32).to(dev) if ragged else None
    with torch.no_grad():
        stk = encoder6._get_packed().stacked
        ref = ops.encoder_stack(x16, stk, n, t, lengths=lens, cluster_size=8, groups_per_cluster=1).clone()
        groups = -(-n // max(1, 128 // t))
        for cl in (8, 16):
            if cl == 16 and -(-groups // 2) > 7:
                continue
            out = ops.encoder_stack(x16, stk, n, t, lengths=lens, cluster_size=cl, groups_per_cluster=2)
            assert torch.equal(out, ref), f"cluster size {cl}"


@pytest.mark.parametrize("n,t", [(1, 1), (1, 2), (2, 5), (3, 7), (2, 29), (1, 40)])
def test_stem_variants_agree_bit_for_bit(frontend, dev, n, t):
    """The transposed stem (filter in tensor memory, two output frames per pixel operand, max-pool in registers:
    csrc/sblk_stem_t.cuh, the default) against the pixel-major stem of round 1 (csrc/sblk_conv3d.cuh): both layouts,
    odd and even frame counts (a half-empty last frame pair), clip edges, zero halos of the flat layout — and a
    limited grid (sblk_set_sm_limit), which only moves the work partition."""
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    pk = frontend._get_packed()
    x = synth.synthetic_clips(n, t, seed=900 + 10 * n + t).to(dev)
    xp = ops.prep_clip(x)
    outs = {}
    try:
        for var in (0, 1):
            ops.set_stem_variant(var)
            outs[var] = ops.conv3d_bn_relu_pool(xp, pk.c3w, pk.c3b).clone()
            dirty = torch.full((ops.flat_rows(n * t, 22, 22), 64), 3.0, dtype=torch.bfloat16, device=dev)
            fl = ops.conv3d_bn_relu_pool(xp, pk.c3w, pk.c3b, out=dirty, flat=True)
            assert torch.equal(fl.dense(), outs[var])
            grid = fl.data.view(-1, 24, 64)
            frames = grid[1:].view(n * t, 23, 24, 64)
            assert float(grid[0].abs().sum() + frames[:, 22].abs().sum() + frames[:, :, 0].abs().sum()
                         + frames[:, :, 23].abs().sum()) == 0.0
        ops.set_stem_variant(0)
        old = ops.set_sm_limit(6)
        try:
            few = ops.conv3d_bn_relu_pool(xp, pk.c3w, pk.c3b)
        finally:
            ops.set_sm_limit(old)
    finally:
        ops.set_stem_variant(0)
    assert torch.equal(outs[0], outs[1])
    assert torch.equal(few, outs[0])


@pytest.mark.parametrize("n,t", [(1, 1), (1, 2), (2, 5), (3, 7), (2, 29), (1, 40)])
def test_fused_stem_is_bit_identical_to_prep_plus_stem(frontend, dev, n, t):
    """sblk_stem_fused_fwd (the stem's producer warps build the row-Toeplitz entries straight from the fp32 clip or the
    raw uint8 frames; no prepped copy of the clip) against sblk_prep_clip[_u8] + sblk_conv3d_bn_relu_pool_fwd: both
    output layouts, odd / even frame counts, clip edges, a limited grid, uniform and per-frame crops, frame padding."""
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    pk = frontend._get_packed()
    x = synth.synthetic_clips(n, t, seed=1300 + 10 * n + t).to(dev)
    ref = ops.conv3d_bn_relu_pool(ops.prep_clip(x), pk.c3w, pk.c3b)
    assert torch.equal(ops.conv3d_bn_relu_pool(ops.raw_clip(x), pk.c3w, pk.c3b), ref)
    ref_flat = ops.conv3d_bn_relu_pool(ops.prep_clip(x), pk.c3w, pk.c3b, flat=True)
    dirty = torch.full((ops.flat_rows(n * t, 22, 22), 64), 3.0, dtype=torch.bfloat16, device=dev)
    got_flat = ops.conv3d_bn_relu_pool(ops.raw_clip(x), pk.c3w, pk.c3b, out=dirty, flat=True)
    assert torch.equal(got_flat.data, ref_flat.data)
    old = ops.set_sm_limit(6)
    try:
        assert torch.equal(ops.conv3d_bn_relu_pool(ops.raw_clip(x), pk.c3w, pk.c3b), ref)
    finally:
        ops.set_sm_limit(old)
    # raw uint8 frames: uniform crop, frame padding, per-frame crops
    lut = synth.normalize_lut().to(dev)
    u8 = synth.synthetic_u8_clips(n, t, h0=100, w0=92, seed=n + t).to(dev)
    g = torch.Generator().manual_seed(n * 7 + t)
    offs = torch.stack([torch.randint(0, 13, (n * t,), generator=g), torch.randint(0, 5, (n * t,), generator=g)], 1)
    for crop, t_out in (((6, 2), t), ((12, 4), t + 3), (offs.int().to(dev), t + 1)):
        r = ops.conv3d_bn_relu_pool(ops.prep_clip_u8(u8, lut, t_out, crop), pk.c3w, pk.c3b, flat=True)
        f = ops.conv3d_bn_relu_pool(ops.raw_clip_u8(u8, lut, t_out, crop), pk.c3w, pk.c3b, flat=True)
        assert torch.equal(f.data, r.data)


def test_fused_stem_through_the_modules_and_its_error_behaviour(frontend, dev):
    """Lipreading.forward / forward_u8 with and without the fused stem return the same bits; the C ABI rejects calls
    that name no input, both inputs, or an fp32 clip with frame padding."""
    import ctypes
    from sbl_for_multilingual_lip_reading_b200 import _lib, ops, synth
    x = synth.synthetic_clips(3, 7, seed=77).to(dev)
    u8 = synth.synthetic_u8_clips(2, 6, seed=78).to(dev)
    saved = (frontend.fuse_prep, frontend.fuse_prep_u8)
    with torch.no_grad():   # one-time work (weight packing, normalisation table) outside the launch counts
        frontend(x[:1]), frontend.forward_u8(u8[:1], frames=6)
    try:
        outs = []
        for fuse in (False, True):
            frontend.fuse_prep = frontend.fuse_prep_u8 = fuse
            before = ops.launch_count()
            with torch.no_grad():
                outs.append((frontend(x), frontend.forward_u8(u8, frames=8)))
            outs.append(ops.launch_count() - before)
    finally:
        frontend.fuse_prep, frontend.fuse_prep_u8 = saved
    assert torch.equal(outs[0][0], outs[2][0]) and torch.equal(outs[0][1], outs[2][1])
    assert outs[3] == outs[1] - 2          # one launch less per forward
    lib = _lib.load()
    pk = frontend._get_packed()
    out = torch.empty((7, 22, 22, 64), dtype=torch.bfloat16, device=dev)
    xa = x[:1].contiguous()
    p = lambda t_: ctypes.c_void_p(t_.data_ptr())
    none = ctypes.c_void_p(0)
    assert lib.sblk_stem_fused_fwd(none, none, none, none, 0, 0, p(pk.c3w), p(pk.c3b), p(out), 1, 7, 7, 88, 88, 0, none) != 0
    assert "exactly one" in _lib.last_error()
    assert lib.sblk_stem_fused_fwd(p(xa), p(u8), none, none, 0, 0, p(pk.c3w), p(pk.c3b), p(out), 1, 7, 7, 88, 88, 0, none) != 0
    assert lib.sblk_stem_fused_fwd(p(xa), none, none, none, 0, 0, p(pk.c3w), p(pk.c3b), p(out), 1, 7, 8, 88, 88, 0, none) != 0
    assert "T_out == T_in" in _lib.last_error()
    lut = synth.normalize_lut().to(dev)
    assert lib.sblk_stem_fused_fwd(none, p(u8), p(lut), none, 9, 4, p(pk.c3w), p(pk.c3b), p(out), 1, 6, 7, 96, 96, 0, none) != 0
    assert "crop offset" in _lib.last_error()


def test_frontend_accepts_a_misaligned_input_view(frontend, dev):
    """A contiguous clip tensor that starts at an odd storage offset (not 16-byte aligned) gives the same features."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(2, 5, seed=9).to(dev)
    flat = torch.empty(x.numel() + 1, device=dev)
    flat[1:].copy_(x.view(-1))
    xv = flat[1:].view_as(x)
    assert xv.is_contiguous() and xv.data_ptr() % 16 != 0
    with torch.no_grad():
        assert torch.equal(frontend(xv), frontend(x))


def test_empty_batch(frontend, encoder6, dev):
    """N = 0 (e.g. the tail of a sharded loader): empty outputs of the reference's shapes, no launch."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    before = ops.launch_count()
    with torch.no_grad():
        f = frontend(torch.empty((0, 1, 29, 88, 88), device=dev))
        out, = encoder6(f, [])
        out2, attns = encoder6(f, [], return_attns=True)
    assert f.shape == (0, 29, 512) and out.shape == (0, 29, 512) and out2.shape == (0, 29, 512)
    assert len(attns) == 6 and ops.launch_count() == before


def test_encoder_stack_rejects_unsupported_shapes(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    enc = Encoder(512, 1, 8, 64, 64, 512, 2048)
    enc.load_state_dict(synth.encoder_state_dict(4, 1))
    enc = enc.to(dev).eval()
    stk = enc._get_packed().stacked
    x16 = torch.zeros(4 * 130, 512, dtype=ops.enc16_dtype(), device=dev)
    with pytest.raises(RuntimeError, match="T <= 128"):
        ops.encoder_stack(x16, stk, 4, 130)
    with pytest.raises(RuntimeError, match="workspace"):
        ops.encoder_stack(x16[:40], stk, 4, 10, workspace=torch.empty(16, dtype=torch.uint8, device=dev))
    # configurations outside the fused kernel's envelope take the per-step kernels (still libsblk, never torch)
    wide = Encoder(512, 1, 8, 64, 64, 512, 1024 + 64).to(dev).eval()
    assert not wide._use_fused_stack(2, 10, False)
    assert not enc._use_fused_stack(2, 10, True) and enc._use_fused_stack(2, 10, False)


# ------------------------------------------------------------------ 1,000 synthetic clips: identical top-1 class
def test_top1_class_identical_on_1000_synthetic_clips(frontend, encoder6, dev):
    """BASELINE.json north_star: identical top-1 class on 1,000 synthetic clips.  The labels in
    tests/golden/top1_1000.npz come from the unmodified reference modules (tests/golden/make_golden_top1.py);
    the stage-1 heads (fc_1500 / fc_2, ...classify/transformer/transformer.py:13-14) run in fp32 on both sides.
    (1) plain heads: every one of the 1,000 clips must get the reference's word and language class;
    (2) centred word head (pooled output minus the reference mean `mu`, which removes the clip-independent part that
        dominates with random weights and spreads the clips over hundreds of classes): every clip whose reference
        top-1 / top-2 margin is clear of the bf16 error must agree, near-ties are counted and bounded."""
    import os
    from sbl_for_multilingual_lip_reading_b200 import synth
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "top1_1000.npz")
    g = np.load(path)
    chunk, chunks, t = int(g["chunk"]), int(g["chunks"]), int(g["frames"])
    heads = synth.classifier_heads(9)
    mu = torch.from_numpy(g["mu"]).to(dev)
    w1 = heads["fc_1500.weight"].to(dev)
    top1, lang, top1c, err = [], [], [], []
    with torch.no_grad():
        for c in range(chunks):
            x = synth.structured_clips(chunk, t, seed=5000 + c).to(dev)
            out, = encoder6(frontend(x), [t] * chunk)
            logits, ll = synth.classify(out, heads)
            top1.append(logits.argmax(dim=1).cpu())
            lang.append(ll.argmax(dim=1).cpu())
            top1c.append(((out.mean(dim=1) - mu) @ w1.t()).argmax(dim=1).cpu())
    top1, lang, top1c = torch.cat(top1).numpy(), torch.cat(lang).numpy(), torch.cat(top1c).numpy()
    assert top1.shape == (chunk * chunks,) and chunk * chunks >= 1000
    assert (top1 == g["top1"]).all(), f"{(top1 != g['top1']).sum()} of 1000 word classes differ"
    assert (lang == g["lang"]).all()
    same = top1c == g["top1_centred"]
    clear = g["margin_centred"] > 0.015
    print(f"centred head: {len(set(g['top1_centred'].tolist()))} reference classes, agreement {same.mean():.4f}, "
          f"{int(clear.sum())} clips with a clear margin")
    assert same[clear].all(), f"{(~same[clear]).sum()} clips with a clear reference margin disagree"
    assert same.mean() >= 0.6


# ------------------------------------------------------------------ fused uint8 input pipeline (SURVEY.md 8f.3)
def test_fused_u8_input_pipeline_is_bit_identical(frontend, dev, golden):
    """sblk_prep_clip_u8 (raw uint8 frames -> /255 -> ColorNormalize -> 88x88 crop -> frame zero-padding -> prepped
    layout) against sblk_prep_clip of the clip the reference loader builds on the CPU (golden from the reference's own
    cvtransforms, tests/golden/input_pipeline.npz): the prepped buffers and the frontend features must be
    bit-identical, for the eval path (centre crop) and for per-frame RandomCrop offsets."""
    import os
    import random
    from sbl_for_multilingual_lip_reading_b200 import ops, synth
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "input_pipeline.npz"))
    u8 = synth.synthetic_u8_clips(1, 29, seed=21).to(dev)
    lut = synth.normalize_lut().to(dev)
    ref30 = torch.from_numpy(g["eval_T30"]).view(1, 1, 30, 88, 88).to(dev)
    def written(buf, n_, t_):   # the buffer ends with over-read slack that neither kernel writes
        return buf[:n_ * (t_ + 4) * 2 * 2072 * 8]

    a, _, _ = ops.prep_clip(ref30)
    b, n, t = ops.prep_clip_u8(u8, lut, 30, (4, 4))
    assert (n, t) == (1, 30) and torch.equal(written(a, 1, 30), written(b, 1, 30))
    random.seed(5)
    offs = []
    for _ in range(29):
        x1 = random.randint(0, 8)
        y1 = random.randint(0, 8)
        offs.append((y1, x1))
    ref31 = torch.from_numpy(g["train_crop_T31"]).view(1, 1, 31, 88, 88).to(dev)
    a, _, _ = ops.prep_clip(ref31)
    b, _, _ = ops.prep_clip_u8(u8, lut, 31, torch.tensor(offs, dtype=torch.int32, device=dev))
    assert torch.equal(written(a, 1, 31), written(b, 1, 31))
    with torch.no_grad():
        f_ref = frontend(ref30)
        f_u8 = frontend.forward_u8(u8, frames=30)
    assert f_u8.shape == (1, 30, 512) and torch.equal(f_ref, f_u8)
    # a multi-clip batch, other raw sizes, error behaviour
    u8b = synth.synthetic_u8_clips(3, 7, h0=100, w0=92, seed=3).to(dev)
    from oracle import input_pipeline_oracle as P
    refb = torch.from_numpy(np.stack([P.eval_clip(c, 9) for c in u8b.cpu().numpy()])).unsqueeze(1).to(dev)
    with torch.no_grad():
        assert torch.equal(frontend(refb), frontend.forward_u8(u8b, frames=9, crop=(6, 2)))
    with pytest.raises(RuntimeError, match="crop offset"):
        ops.prep_clip_u8(u8, lut, 30, (9, 4))
    with pytest.raises(RuntimeError, match="frames="):
        frontend.forward_u8(u8, frames=5)


# ------------------------------------------------------------------ BASELINE-size properties
def test_config2_batch_independence_and_determinism(frontend, encoder6, dev):
    """Config 2 (32 x 29 x 88 x 88): clips are independent in eval mode (SURVEY.md §8e), so clip i of the
    batch-32 run must equal the same clip run alone; and two runs must be bit-identical."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.synthetic_clips(32, 29, seed=7).to(dev)
    with torch.no_grad():
        out, = encoder6(frontend(x), [29] * 32)
        out2, = encoder6(frontend(x), [29] * 32)
        single, = encoder6(frontend(x[5:6].contiguous()), [29])
        part, = encoder6(frontend(x[16:].contiguous()), [29] * 16)
    assert out.shape == (32, 29, 512)
    assert torch.equal(out, out2)
    assert rel_fro(out[5:6], single) < 1e-6
    assert rel_fro(out[16:], part) < 1e-6


_CACHES = ("_packed", "_flat_ws", "_streams", "_lut", "_len_cache")


def _settings(*mods):
    """Every attribute of the modules but their caches (the dicts of parameters, submodules, hooks copied one level)."""
    return [{k: dict(v) if isinstance(v, dict) else v for k, v in m.__dict__.items() if k not in _CACHES} for m in mods]


def _eager_launches(fe, enc, x, lens):
    """libsblk launches of one eager enc(fe(x))."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    before = ops.launch_count()
    with torch.no_grad():
        enc(fe(x), lens)
    torch.cuda.synchronize()
    return ops.launch_count() - before


@pytest.mark.parametrize("n,t,lens", [(32, 29, None), (8, 40, None), (6, 29, [29, 11, 29, 3, 20, 29])])
def test_pipelined_plan_is_bit_identical_and_leaves_modules_unchanged(frontend, encoder6, dev, n, t, lens):
    """runner.PipelinedVisualEncoderPlan (the encoder stack of batch i-1 co-running with the clip prep + stem of batch i
    on the SMs it leaves free, ordered by the sblk_gate_wait kernel) must return, one step late, exactly what the
    drop-in modules return for each batch: same kernels, only grid sizes and scheduling differ.  Shapes: BASELINE
    configs[1], the configs[2] per-GPU shard (8 clips x 40 frames), a ragged-length batch.  Also through submit_host
    (pinned host in / out) and drain(); building, replaying and draining the plan leaves the modules as they were."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.runner import PipelinedVisualEncoderPlan
    lens = [t] * n if lens is None else lens
    xs = [synth.synthetic_clips(n, t, seed=50 + i) for i in range(4)]
    with torch.no_grad():
        want = [encoder6(frontend(x.to(dev)), lens)[0].cpu() for x in xs]
    settings, launches = _settings(frontend, encoder6), _eager_launches(frontend, encoder6, xs[0].to(dev), lens)
    plan = PipelinedVisualEncoderPlan(frontend, encoder6, n, t, device=dev, lengths=lens)
    try:
        # device-resident inputs
        got = []
        for i, x in enumerate(xs):
            with torch.cuda.stream(plan.compute):
                plan.x[i % 2].copy_(x.to(dev))
                prev = plan.forward_device(i % 2)
                if i > 0:
                    got.append(prev.clone())
            plan.compute.synchronize()
        plan._i = len(xs)
        last = plan.drain()
        plan.compute.synchronize()
        got.append(last.clone())
        torch.cuda.synchronize(dev)
        for i in range(len(xs)):
            assert torch.equal(got[i].cpu(), want[i]), f"device path, batch {i}"
        assert int(plan.gate[0]) == int(plan.gate[1]) > 0   # every encoder CTA reported in, every gate accounted for
        # host path: k inputs in, the k outputs of those inputs out (shifted by one call, the last one by drain)
        plan._i = 0
        hin = [x.pin_memory() for x in xs]
        hout = [torch.empty((n, t, 512), dtype=torch.float32).pin_memory() for _ in range(len(xs) + 1)]
        for i in range(len(xs)):
            plan.submit_host(hin[i], hout[i])
        plan.drain(hout[len(xs)])
        plan.synchronize()
        for i in range(len(xs)):
            assert torch.equal(hout[i + 1], want[i]), f"host path, batch {i}"
    finally:
        plan.close()
    assert _settings(frontend, encoder6) == settings
    assert _eager_launches(frontend, encoder6, xs[0].to(dev), lens) == launches


@pytest.mark.parametrize("n,t,lens", [(32, 29, None), (8, 40, None), (5, 29, [29, 11, 29, 3, 20])])
def test_plain_plan_with_fused_tail_is_bit_identical_and_leaves_modules_unchanged(frontend, encoder6, dev, n, t, lens):
    """runner.VisualEncoderPlan (one batch per replay) with its fused tail — dropout factor drawn on a side stream, the
    pooling launch writes the encoder's 16-bit operand — returns exactly what the drop-in modules return, through
    forward_device and through submit_host, and leaves the modules as they were: the same settings, the same eager
    launches (no hint for the encoder's weights added to the frontend's forward)."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.runner import VisualEncoderPlan
    lens = [t] * n if lens is None else lens
    xs = [synth.synthetic_clips(n, t, seed=70 + i) for i in range(3)]
    with torch.no_grad():
        want = [encoder6(frontend(x.to(dev)), lens)[0].cpu() for x in xs]
    settings, launches = _settings(frontend, encoder6), _eager_launches(frontend, encoder6, xs[0].to(dev), lens)
    plan = VisualEncoderPlan(frontend, encoder6, n, t, device=dev, lengths=lens)
    try:
        assert hasattr(plan, "feat16")          # the fused tail is in use for these shapes
        for i, x in enumerate(xs):
            with torch.cuda.stream(plan.compute):
                plan.x[i % 2].copy_(x.to(dev))
                out = plan.forward_device(i % 2)
            plan.compute.synchronize()
            assert torch.equal(out.cpu(), want[i]), f"device path, batch {i}"
        hin = [x.pin_memory() for x in xs]
        hout = [torch.empty((n, t, 512), dtype=torch.float32).pin_memory() for _ in xs]
        for i in range(len(xs)):
            plan.submit_host(hin[i], hout[i])
        plan.synchronize()
        for i in range(len(xs)):
            assert torch.equal(hout[i], want[i]), f"host path, batch {i}"
    finally:
        plan.close()
    assert _settings(frontend, encoder6) == settings
    assert _eager_launches(frontend, encoder6, xs[0].to(dev), lens) == launches


def test_modules_pickled_by_an_earlier_version_run(frontend, encoder6, dev):
    """Modules pickled before the plans passed their schedule as arguments carry the retired attributes (the plans'
    hooks, the multi-chain frontend's settings): they load without them and compute what the current modules compute."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe, enc = Lipreading.__new__(Lipreading), Encoder.__new__(Encoder)
    fe.__setstate__(dict(frontend.__getstate__(), parallel_chains=2, chain_sm_limit=74, l2_prefetch_extra=None,
                         _overlap=None, _tail=None, _block_hook=None))
    enc.__setstate__(dict(encoder6.__getstate__(), _x16_override=None, _resident_counter=None))
    x = synth.synthetic_clips(16, 29, seed=11).to(dev)
    with torch.no_grad():
        want, = encoder6(frontend(x), [29] * 16)
        got, = enc(fe(x), [29] * 16)
    assert torch.equal(got, want)


def test_plain_plan_draws_a_fresh_dropout_mask_every_replay(encoder6, dev):
    """The reference's always-on dropout (video_frontend.py:122) inside the plain plan's fused tail: a new mask per
    replay, about half of the features zeroed."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.runner import VisualEncoderPlan
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe = fe.to(dev).eval()
    assert fe.always_on_dropout
    x = synth.synthetic_clips(4, 29, seed=9).to(dev)
    plan = VisualEncoderPlan(fe, encoder6, 4, 29, device=dev)
    outs = []
    try:
        with torch.cuda.stream(plan.compute):
            for i in range(3):
                plan.x[i % 2].copy_(x)
                outs.append(plan.forward_device(i % 2).clone())
            zero_frac = (plan.feat16[0] == 0).float().mean().item()
        plan.compute.synchronize()
    finally:
        plan.close()
    fe.always_on_dropout = False
    with torch.no_grad():
        clean, = encoder6(fe(x), [29] * 4)
    assert 0.45 < zero_frac < 0.55
    for o in outs:
        assert torch.isfinite(o).all() and not torch.equal(o, clean)
    assert not torch.equal(outs[0], outs[1]) and not torch.equal(outs[1], outs[2])


def test_avgpool_with_dropout_factor_matches_pool_then_dropout(dev):
    """sblk_avgpool_scale_fwd: pooling times the pre-drawn dropout factor (F.dropout(ones) under the same seed draws the
    same Philox mask as F.dropout(features)) is bit-identical to pooling followed by the reference's always-on
    F.dropout(x, p=0.5) (video_frontend.py:122), in fp32 and in the bf16 copy the encoder reads."""
    import torch.nn.functional as F
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn(928, 3, 3, 512, generator=g).to(torch.bfloat16).to(dev)
    pooled, _ = ops.avgpool(x)
    torch.manual_seed(5)
    want = F.dropout(pooled, p=0.5)
    torch.manual_seed(5)
    scale = F.dropout(torch.ones_like(pooled), p=0.5)
    got32, got16 = ops.avgpool(x, want_f32=True, want_bf16=True, scale=scale)
    _, gote16 = ops.avgpool(x, want_f32=False, want_bf16=True, scale=scale, enc16=True)
    torch.cuda.synchronize(dev)
    assert 0.4 < (want == 0).float().mean().item() < 0.6
    assert torch.equal(got32, want)
    assert torch.equal(got16, ops.cast_bf16(want))
    assert gote16.dtype == ops.enc16_dtype() and torch.equal(gote16, ops.cast_enc16(want))
    with pytest.raises(RuntimeError):
        ops.avgpool(x, scale=scale[:10])


def test_pipelined_plan_draws_a_fresh_dropout_mask_every_replay(encoder6, dev):
    """With the reference's always-on dropout enabled the pipelined plan must still apply it (a new mask per replay,
    about half of the features zeroed): same clip batch three times -> three different finite outputs, all different
    from the dropout-free output."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.runner import PipelinedVisualEncoderPlan
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe = fe.to(dev).eval()
    assert fe.always_on_dropout
    x = synth.synthetic_clips(4, 29, seed=9).to(dev)
    plan = PipelinedVisualEncoderPlan(fe, encoder6, 4, 29, device=dev)
    outs = []
    try:
        with torch.cuda.stream(plan.compute):
            for i in range(4):
                plan.x[i % 2].copy_(x)
                prev = plan.forward_device(i % 2)
                if i > 0:
                    outs.append(prev.clone())
            zero_frac = (plan.feat16[0] == 0).float().mean().item()
        plan.compute.synchronize()
    finally:
        plan.close()
    fe.always_on_dropout = False
    with torch.no_grad():
        clean, = encoder6(fe(x), [29] * 4)
    assert 0.45 < zero_frac < 0.55
    for o in outs:
        assert torch.isfinite(o).all() and not torch.equal(o, clean)
    assert not torch.equal(outs[0], outs[1]) and not torch.equal(outs[1], outs[2])


@pytest.mark.parametrize("c,h", [(64, 22), (128, 11)])
def test_flat_conv_over_frame_ranges_is_bit_identical(dev, c, h):
    """A flat 3x3 conv issued over frame ranges (ops.flat_frames; the pipelined plan runs half of layer1.0.conv1's frames
    inside its head) writes exactly the bits of the whole-buffer launch, halo rows included, with and without residual."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(11)
    f = 61
    rows = ops.flat_rows(f, h, h)
    data = torch.zeros(rows, c, dtype=torch.bfloat16, device=dev)
    v = data[(h + 2):(h + 2) + f * (h + 1) * (h + 2)].view(f, h + 1, h + 2, c)
    v[:, :h, 1:h + 1, :] = torch.randn(f, h, h, c, generator=g).to(torch.bfloat16).to(dev)
    x = ops.FlatActs(data, f, h, h)
    w = ops.pack_flat_weight((torch.randn(c, 3, 3, c, generator=g) / (9 * c) ** 0.5).to(torch.bfloat16).to(dev))
    bias = torch.randn(c, generator=g).to(dev)
    for res in (None, x):
        whole = ops.conv3x3_flat(x, w, bias, relu=True, residual=res)
        parts = torch.full_like(data, float("nan"))
        for f0, f1 in ((0, 17), (17, 18), (18, f)):
            ops.conv3x3_flat(ops.flat_frames(x, f0, f1), w, bias, relu=True,
                             residual=None if res is None else ops.flat_frames(res, f0, f1),
                             out=ops.flat_frames(ops.FlatActs(parts, f, h, h), f0, f1).data)
        torch.cuda.synchronize(dev)
        assert torch.equal(parts, whole.data)


@pytest.mark.parametrize("c,h,f", [(64, 22, 61), (128, 11, 61), (64, 22, 1), (128, 11, 300)])
def test_flat_conv_reverse_tile_order_is_bit_identical(dev, c, h, f):
    """sblk_flatconv3x3_dir_fwd: walking every CTA pair's tile range backwards (the frontend alternates the direction
    between consecutive convs for L2 reuse) changes nothing in the output, with / without residual, full / limited grid."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(13 + f)
    rows = ops.flat_rows(f, h, h)
    data = torch.zeros(rows, c, dtype=torch.bfloat16, device=dev)
    v = data[(h + 2):(h + 2) + f * (h + 1) * (h + 2)].view(f, h + 1, h + 2, c)
    v[:, :h, 1:h + 1, :] = torch.randn(f, h, h, c, generator=g).to(torch.bfloat16).to(dev)
    x = ops.FlatActs(data, f, h, h)
    w = ops.pack_flat_weight((torch.randn(c, 3, 3, c, generator=g) / (9 * c) ** 0.5).to(torch.bfloat16).to(dev))
    bias = torch.randn(c, generator=g).to(dev)
    for res, limit in ((None, 0), (x, 0), (x, 20)):
        prev = ops.set_sm_limit(limit) if limit else None
        try:
            fwd = ops.conv3x3_flat(x, w, bias, relu=True, residual=res)
            bwd = ops.conv3x3_flat(x, w, bias, relu=True, residual=res, reverse=True)
        finally:
            if prev is not None:
                ops.set_sm_limit(prev)
        torch.cuda.synchronize(dev)
        assert torch.equal(fwd.data, bwd.data)


def test_gate_wait_times_out_and_rejects_bad_arguments(dev):
    """sblk_gate_wait is a scheduling hint: with nobody bumping the counter it must give up after its timeout (not
    hang) and still advance its target word; bad arguments fail loudly."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    gate = torch.zeros(2, dtype=torch.int32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ops.gate_wait(gate, 64, timeout_us=200)
    e1.record()
    torch.cuda.synchronize(dev)
    assert gate.tolist() == [0, 64]
    assert 0.15 < e0.elapsed_time(e1) < 50.0
    gate[0] = 128   # already satisfied: returns at once
    ops.gate_wait(gate, 64, timeout_us=10_000_000)
    torch.cuda.synchronize(dev)
    assert gate.tolist() == [128, 128]
    with pytest.raises(RuntimeError):
        ops.gate_wait(gate, 0)
    with pytest.raises(RuntimeError):
        ops.gate_wait(torch.zeros(2, dtype=torch.float32, device=dev), 8)


def test_config2_linearity_of_conv_stage(frontend, dev):
    """conv(a*x) = a*conv(x) for a power-of-two a (exact in bf16/fp32 without bias/ReLU clipping):
    checks the implicit GEMM at the full layer-1 size M = 928*22*22."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(0)
    x = torch.randn(928, 22, 22, 64, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(64, 3, 3, 64, generator=g) / 24).to(torch.bfloat16).to(dev)
    zero = torch.zeros(64, device=dev)
    a = ops.conv2d(x, w, zero, relu=False)
    b = ops.conv2d(x * 4, w, zero, relu=False)
    assert torch.equal(a.float() * 4, b.float())
    # spot-check 4096 random outputs against an fp64 dot product
    idx = torch.randint(0, 928 * 22 * 22, (4096,), generator=g)
    f, yy, xx = idx // 484, (idx % 484) // 22, idx % 22
    xp = torch.nn.functional.pad(x.float().cpu(), (0, 0, 1, 1, 1, 1))
    patches = torch.stack([xp[f, yy + r, xx + s] for r in range(3) for s in range(3)], dim=1)  # [4096,9,64]
    ref = torch.einsum("ptc,otc->po", patches.double(), w.float().cpu().reshape(64, 9, 64).double())
    got = a.reshape(-1, 64)[idx.to(dev)].float().cpu().double()
    assert ((got - ref).norm() / ref.norm()).item() < 5e-3


def _to_flat(x):
    from sbl_for_multilingual_lip_reading_b200 import ops
    f, h, w, c = x.shape
    data = torch.zeros(ops.flat_rows(f, h, w), c, dtype=torch.bfloat16, device=x.device)
    v = data[(w + 2):(w + 2) + f * (h + 1) * (w + 2)].view(f, h + 1, w + 2, c)
    v[:, :h, 1:w + 1, :] = x
    return ops.FlatActs(data, f, h, w)


def test_config2_flat_conv_properties(dev):
    """Flat shifted-window conv at the full layer-1 size (928 frames): linearity (exact for power-of-two scaling),
    zero halos, residual exactness (R*I on the tensor core), agreement with the im2col kernel and an fp64 spot check."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn(928, 22, 22, 64, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(64, 3, 3, 64, generator=g) / 24).to(torch.bfloat16).to(dev)
    wf = ops.pack_flat_weight(w)
    zero = torch.zeros(64, device=dev)
    xf, xf4 = _to_flat(x), _to_flat(x * 4)
    a = ops.conv3x3_flat(xf, wf, zero, relu=False)
    b = ops.conv3x3_flat(xf4, wf, zero, relu=False)
    assert torch.equal(a.dense().float() * 4, b.dense().float())
    # halo rows / columns are exactly zero
    d = a.data.float().clone()
    d[24:24 + 928 * 23 * 24].view(928, 23, 24, 64)[:, :22, 1:23, :] = 0
    assert bool((d == 0).all())
    # same numbers as the TMA-im2col kernel on the dense layout (both accumulate in fp32, different order)
    ref = ops.conv2d(x, w, zero, relu=False)
    assert rel_fro(a.dense(), ref) < 1e-3
    # residual through the identity MMA == adding it afterwards in fp32 and rounding once
    r = ops.conv3x3_flat(xf, wf, zero, relu=True, residual=xf)
    idx = torch.randint(0, 928 * 484, (4096,), generator=g)
    f, yy, xx = idx // 484, (idx % 484) // 22, idx % 22
    xp = torch.nn.functional.pad(x.float().cpu(), (0, 0, 1, 1, 1, 1))
    patches = torch.stack([xp[f, yy + rr, xx + ss] for rr in range(3) for ss in range(3)], dim=1)
    conv = torch.einsum("ptc,otc->po", patches.double(), w.float().cpu().reshape(64, 9, 64).double())
    want = torch.relu(conv + x.float().cpu().reshape(-1, 64)[idx].double())
    got = r.dense().reshape(-1, 64)[idx.to(dev)].float().cpu().double()
    assert ((got - want).norm() / want.norm()).item() < 5e-3


# ------------------------------------------------------------------ nn.DataParallel (reference train.py:114-115)
def test_data_parallel_two_gpus_matches_single_gpu():
    """The reference wraps the model in nn.DataParallel (train.py:114-115): replicas run in worker THREADS on
    different devices at the same time.  The drop-ins must give the single-GPU result (per-device library state,
    caller's device and stream, per-replica packed-weight caches)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading

    class Path(torch.nn.Module):   # what Transformer.forward runs before the decoder (transformer.py:31-38)
        def __init__(self):
            super().__init__()
            self.visual_frontend = Lipreading()
            self.visual_frontend.load_state_dict(synth.frontend_state_dict(1))
            self.visual_frontend.always_on_dropout = False
            self.encoder = Encoder(512, 2, 8, 64, 64, 512, 2048)
            self.encoder.load_state_dict(synth.encoder_state_dict(2, 2))

        def forward(self, x):
            feat = self.visual_frontend(x)
            out, *_ = self.encoder(feat, [feat.size(1)] * feat.size(0))
            return out

    model = Path().to("cuda:0").eval()
    x = synth.synthetic_clips(6, 5, seed=77).to("cuda:0")
    with torch.no_grad():
        single = model(x)
        dp = torch.nn.DataParallel(model, device_ids=[0, 1])
        for _ in range(2):
            multi = dp(x)
    assert multi.device == single.device and multi.shape == (6, 5, 512)
    assert torch.equal(multi, single)


def test_p2p_gather_two_gpus():
    """sblk_p2p_gather_fwd (one-shot all-gather over NVLink peer memory, CUDA IPC between the per-GPU processes)
    against ncclAllGather on 2 GPUs, six steps with alternating buffers (tests/p2p_gather_worker.py under torchrun)."""
    import os
    import subprocess
    import sys
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.join(here, "p2p_gather_worker.py")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("p2p gather OK") == 2


def test_integration_md_ctypes_snippet_runs(dev):
    """INTEGRATION.md §3 shows the ctypes stub a maintainer would write against include/sblk.h: execute exactly that
    snippet and check what it computed against torch's conv2d on the same bf16 operands."""
    import os
    import torch.nn.functional as F
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "INTEGRATION.md")) as f:
        md = f.read()
    block = md.split("## 3.")[1].split("```python")[1].split("```")[0]
    ns = {}
    cwd = os.getcwd()
    os.chdir(root)          # the snippet loads the library by its repo-relative path
    try:
        torch.manual_seed(0)
        exec(compile(block, "INTEGRATION.md#3", "exec"), ns)
    finally:
        os.chdir(cwd)
    torch.cuda.synchronize(dev)
    x, wp, out = ns["x"], ns["wp"], ns["out"]
    want = F.relu(F.conv2d(x.float().permute(0, 3, 1, 2), wp.float().permute(0, 3, 1, 2), padding=1)).permute(0, 2, 3, 1)
    assert rel_fro(out, want) < REL_TOL
