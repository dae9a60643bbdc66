"""`-m gpu` tests of the training path (BASELINE configs[3]; SURVEY.md 8f.2): every new kernel against the torch op it
replaces, then the drop-in modules in `model.train()` — forward with batch statistics, backward, running-stat updates —
against autograd through the reference's modules in fp32 on the same B200 (oracle/reference_modules.py: the reference
classes restated in torch.nn, pinned to the reference's own outputs by tests/test_oracle_golden.py).

Tolerance: relative Frobenius error; 2e-2 for gradients (bf16 operands and bf16 gradient tensors, fp32 accumulation),
stated per assertion where a deep chain needs more.
"""
import json
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT_DIR = os.path.join(ROOT, "gpurun_out")
BF = torch.bfloat16


def rel(a, b):
    a, b = a.float(), b.float()
    assert a.shape == b.shape, (a.shape, b.shape)
    assert torch.isfinite(a).all(), "non-finite values"
    return ((a - b).norm() / (b.norm() + 1e-20)).item()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    from oracle import ref_runtime
    assert ops.init() > 0
    ref_runtime.fp32_exact()
    return torch.device("cuda:0")


# ----------------------------------------------------------------------------------------------- kernels vs torch ops
def test_transpose16_and_format_conversion(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1000, 192, generator=g).to(BF).to(dev)
    y = ot.transpose16(x, ld_out=1024)
    assert y.shape == (192, 1024) and torch.equal(y[:, :1000], x.t()) and float(y[:, 1000:].abs().max()) == 0.0
    h = torch.randn(333, 64, generator=g).to(torch.float16).to(dev)
    z = ot.transpose16(h, ld_out=384, to_bf16=True)
    assert z.dtype == BF and torch.equal(z[:, :333], h.float().to(BF).t())


@pytest.mark.parametrize("c,r,stride", [(64, 3, 1), (64, 3, 2), (128, 1, 2)])
def test_im2col_t_matches_unfold(dev, c, r, stride):
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator().manual_seed(2)
    f, h = 5, 11
    x = torch.randn(f, h, h, c, generator=g).to(BF).to(dev)
    pad = r // 2
    p = (h + 2 * pad - r) // stride + 1
    m = f * p * p
    ld = -(-m // 64) * 64
    got = ot.im2col_t(x, r, r, stride, pad, ld)
    u = F.unfold(x.float().permute(0, 3, 1, 2), (r, r), padding=pad, stride=stride)      # [F, C*r*r, L], index c*(r*r)+tap
    want = u.view(f, c, r * r, p * p).permute(2, 1, 0, 3).reshape(r * r * c, m)
    assert torch.equal(got[:, :m].float(), want) and float(got[:, m:].abs().max() if ld > m else 0.0) == 0.0


def test_stem_im2col_gemm_is_the_conv3d(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops, ops_train as ot
    g = torch.Generator().manual_seed(3)
    n, t = 2, 4
    x = torch.randn(n, t, 88, 88, generator=g).to(dev)
    w = (torch.randn(64, 1, 5, 7, 7, generator=g) / 16).to(dev)
    col = ot.stem_im2col(x)
    m = n * t * 44 * 44
    ld = -(-m // 128) * 128 + 128
    col_t = ot.stem_im2col(x, transposed=True, ld_out=ld)
    assert torch.equal(col_t[:, :m], col.t()) and float(col_t[:, m:].abs().max()) == 0.0
    w2d = torch.zeros(64, 256, device=dev)
    w2d[:, :245] = w.reshape(64, 245)
    raw, _ = ot.gemm_fmt(col, ops.cast_bf16(w2d), out16=True)
    want = F.conv3d(x.to(BF).float().unsqueeze(1), w.to(BF).float(), stride=(1, 2, 2), padding=(2, 3, 3))
    want = want.permute(0, 2, 3, 4, 1).reshape(m, 64)
    assert rel(raw, want) < 5e-3


def test_gemm_fmt_bf16_split_k_small_m(dev):
    """the wgrad shape: few output rows (M = 64 < one 128-row tile), very long K, split-K partials."""
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator().manual_seed(4)
    a = torch.randn(64, 4096, generator=g).to(BF).to(dev)
    w = torch.randn(192, 4096, generator=g).to(BF).to(dev)
    _, parts = ot.gemm_fmt(a, w, out_f32=True, splits=8)
    assert parts.shape == (8, 64, 192)
    assert rel(parts.sum(0), a.float() @ w.float().t()) < 1e-4
    o16, _ = ot.gemm_fmt(a, w, out16=True)
    assert rel(o16, a.float() @ w.float().t()) < 5e-3


@pytest.mark.parametrize("c", [64, 512])
def test_batchnorm_training_forward_backward(dev, c):
    from sbl_for_multilingual_lip_reading_b200 import training as tr
    g = torch.Generator().manual_seed(5)
    m = 5000
    raw = (torch.randn(m, c, generator=g) * 1.5 + 0.3).to(BF).to(dev)
    res = torch.randn(m, c, generator=g).to(BF).to(dev)
    dy = torch.randn(m, c, generator=g).to(BF).to(dev)
    bn = torch.nn.BatchNorm2d(c).to(dev)
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5); bn.bias.normal_(0, 0.1)
    ref_bn = torch.nn.BatchNorm2d(c).to(dev)
    ref_bn.load_state_dict(bn.state_dict())
    out, st = tr.bn_forward_train(raw, bn, residual=res, relu=True)
    x32 = raw.float().requires_grad_(True)
    r32 = res.float().requires_grad_(True)
    want = F.relu(ref_bn(x32.t().reshape(1, c, m, 1)).reshape(c, m).t() + r32)
    want.backward(dy.float())
    assert rel(out, want) < 5e-3
    assert rel(bn.running_mean, ref_bn.running_mean) < 1e-4 and rel(bn.running_var, ref_bn.running_var) < 1e-4
    assert int(bn.num_batches_tracked) == 1
    # the backward masks with the module's own (bf16) output, as the fused pipeline does
    dx, dgamma, dbeta, dres = tr.bn_backward_train(dy, out, raw, st, bn.weight, want_dres=True)
    assert rel(dx, x32.grad) < 2e-2
    assert rel(dgamma, ref_bn.weight.grad) < 2e-2 and rel(dbeta, ref_bn.bias.grad) < 2e-2
    assert rel(dres, r32.grad) < 1e-2


def test_maxpool_forward_backward(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator().manual_seed(6)
    x = torch.relu(torch.randn(3, 44, 44, 64, generator=g)).to(BF).to(dev)
    dy = torch.randn(3, 22, 22, 64, generator=g).to(BF).to(dev)
    x32 = x.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    want = F.max_pool2d(x32, 3, 2, 1)
    want.backward(dy.float().permute(0, 3, 1, 2))
    out = ot.maxpool_fwd(x)
    assert torch.equal(out.float(), want.detach().permute(0, 2, 3, 1))
    dx = ot.maxpool_bwd(x, out, dy)
    wg = x32.grad.permute(0, 2, 3, 1)
    # ties (exact zeros after ReLU, equal bf16 values) go to the first maximum in both implementations
    mism = ((dx.float() - wg).abs() > 1e-2 * wg.abs().max()).float().mean().item()
    assert mism < 2e-3, mism


def test_layernorm_backward(dev):
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot
    g = torch.Generator().manual_seed(7)
    n, t = 5, 29
    z = (torch.randn(n * t, 512, generator=g) * 2 + 0.5).to(dev)
    dy = torch.randn(n * t, 512, generator=g).to(dev)
    gamma = (torch.rand(512, generator=g) + 0.5).to(dev)
    beta = torch.randn(512, generator=g).to(dev)
    lens = [29, 3, 17, 29, 1]
    keep = (torch.arange(t)[None, :] < torch.tensor(lens)[:, None]).float().reshape(-1, 1).to(dev)
    z32 = z.clone().requires_grad_(True)
    g32, b32 = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    (F.layer_norm(z32, (512,), g32, b32, 1e-5) * keep).backward(dy)
    dz32, dz16, dg, db = ot.ln_bwd(dy, z, gamma, lengths=torch.tensor(lens, dtype=torch.int32, device=dev), T=t)
    assert rel(dz32, z32.grad) < 1e-4 and rel(dz16, z32.grad) < 5e-3
    assert rel(dg, g32.grad) < 1e-4 and rel(db, b32.grad) < 1e-4


@pytest.mark.parametrize("t,use_drop", [(29, False), (40, True), (7, True)])
def test_attention_training_forward_backward(dev, t, use_drop):
    from sbl_for_multilingual_lip_reading_b200 import ops, ops_train as ot
    g = torch.Generator().manual_seed(8)
    n, h = 3, 8
    e16 = ops.enc16_dtype()
    qkv = torch.randn(n * t, 3 * h * 64, generator=g).to(e16).to(dev)
    dout = torch.randn(n * t, h * 64, generator=g).to(BF).to(dev)
    lens = [t, max(1, t // 2), t]
    lengths = torch.tensor(lens, dtype=torch.int32, device=dev)
    drop = None
    if use_drop:
        drop = F.dropout(torch.ones(h * n, t, t, device=dev), p=0.1)
    out, probs = ot.attention_train_fwd(qkv, n, t, h, drop=drop, lengths=lengths)
    dqkv = ot.attention_train_bwd(qkv, probs, dout, n, t, h, drop=drop, lengths=lengths)
    # torch reference in the reference's own layout (attention.py:41-55,72-83)
    x = qkv.float().requires_grad_(True)
    q, k, v = (x[:, i * 512:(i + 1) * 512].view(n, t, h, 64).permute(2, 0, 1, 3).reshape(h * n, t, 64) for i in range(3))
    att = torch.bmm(q, k.transpose(1, 2)) / 8.0
    mask = (torch.arange(t, device=dev)[None, :] >= lengths[:, None]).unsqueeze(1).expand(-1, t, -1).repeat(h, 1, 1)
    att = torch.softmax(att.masked_fill(mask, float("-inf")), dim=2)
    pd = att if drop is None else att * drop
    o = torch.bmm(pd, v).view(h, n, t, 64).permute(1, 2, 0, 3).reshape(n * t, 512)
    o.backward(dout.float())
    assert rel(probs, att.detach()) < 1e-5
    assert rel(out, o.detach()) < 2e-3
    assert rel(dqkv, x.grad) < 5e-3


@pytest.mark.parametrize("cin,cout,r,stride,h", [(64, 64, 3, 1, 22), (64, 128, 3, 2, 22), (128, 256, 3, 2, 11),
                                                 (256, 512, 1, 2, 6), (512, 512, 3, 1, 3)])
def test_conv_dgrad_wgrad_match_autograd(dev, cin, cout, r, stride, h):
    from sbl_for_multilingual_lip_reading_b200 import training as tr
    g = torch.Generator().manual_seed(9)
    f = 37
    x = torch.randn(f, h, h, cin, generator=g).to(BF).to(dev)
    w = (torch.randn(cout, cin, r, r, generator=g) / (r * r * cin) ** 0.5).to(dev)
    x32 = x.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    w32 = w.to(BF).float().requires_grad_(True)
    y = F.conv2d(x32, w32, stride=stride, padding=r // 2)
    dy = torch.randn(y.shape, generator=g).to(dev).to(BF)
    y.backward(dy.float())
    raw = tr.conv_raw(x, tr.pack_conv_weight(w), stride)
    assert rel(raw.permute(0, 3, 1, 2), y.detach()) < 5e-3
    dyn = dy.permute(0, 2, 3, 1).contiguous()
    dx = tr.conv_dgrad(dyn, tr.pack_conv_weight_dgrad(w), stride, (h, h))
    assert rel(dx.permute(0, 3, 1, 2), x32.grad) < 5e-3
    dw = tr.conv_wgrad(x, dyn, r, stride)
    assert rel(dw, w32.grad) < 1e-3


# ------------------------------------------------------------------------- modules vs the reference's autograd
class _RoundSTE(torch.autograd.Function):
    """bf16 rounding with a straight-through gradient: gives the reference the drop-in's STORAGE precision."""

    @staticmethod
    def forward(ctx, x):
        return x.to(BF).float()

    @staticmethod
    def backward(ctx, g):
        return g


def _match_storage_precision(ref_frontend):
    """Forward hooks that round the reference frontend's activations to bf16 exactly where the libsblk training path
    stores them (raw conv outputs, BN(+ReLU) outputs of conv1 / downsample / stem, block outputs).  In a ReLU network
    with batch-statistics BatchNorm a 1e-2 forward perturbation flips ~1 % of the ReLU masks per layer, which alone moves
    the fp32 gradients by 5 % (last block) to 35 % (first layers) in relative Frobenius norm — measured with fp32
    backward formulas in tools/exp/quant_emulate_train.py; against this precision-matched reference what remains is
    the error of the backward kernels themselves."""
    hooks = []
    rnd = lambda m, i, o: _RoundSTE.apply(o)   # noqa: E731
    for name, mod in ref_frontend.named_modules():
        if isinstance(mod, (torch.nn.Conv2d, torch.nn.Conv3d)):
            hooks.append(mod.register_forward_hook(rnd))
        elif isinstance(mod, torch.nn.BatchNorm3d) or name.endswith(".bn1") or name.endswith("downsample.1"):
            hooks.append(mod.register_forward_hook(rnd))
        elif type(mod).__name__ == "BasicBlock":
            hooks.append(mod.register_forward_hook(rnd))
    return hooks


def _bf16_values(sd):
    return {k: (v.to(BF).float() if v.dtype == torch.float32 and v.dim() >= 2 else v) for k, v in sd.items()}


def _grad_table(ours, ref, names=None):
    rows = {}
    rp = dict(ref.named_parameters())
    for k, p in ours.named_parameters():
        if names is not None and k not in names:
            continue
        assert p.grad is not None, f"no gradient for {k}"
        rows[k] = rel(p.grad, rp[k].grad)
    return rows


def _cosine(a, b):
    a, b = a.float().flatten(), b.float().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def _is_key_bias(k):
    # d loss / d (key bias) is identically zero: a constant added to every key shifts each query's logits uniformly and
    # softmax ignores it; both implementations return rounding noise there, so it is checked on an absolute scale
    return k.endswith("slf_attn.w_ks.bias")


def test_encoder_training_matches_reference_autograd(dev):
    """Encoder in model.train() with dropout = 0: output, input gradient and every parameter gradient against autograd
    through the reference Encoder (encoder.py / attention.py / module.py, restated in oracle/reference_modules.py), ragged
    lengths included.
    Tolerance 3e-2: gradient tensors and GEMM operands of the backward are bf16 (measured 1e-2 .. 2.2e-2)."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    n, t, L = 6, 29, 3
    sd = synth.encoder_state_dict(2, L)
    ref = R.Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.0, pe_maxlen=5000).to(dev).train()
    ours = Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.0, pe_maxlen=5000).to(dev).train()
    ref.load_state_dict(sd); ours.load_state_dict(sd)
    g = torch.Generator().manual_seed(10)
    x = torch.randn(n, t, 512, generator=g).to(dev)
    dy = torch.randn(n, t, 512, generator=g).to(dev)
    lens = [29, 29, 5, 29, 12, 29]
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    oa, = ref(xa, lens)
    oa.backward(dy)
    ob, = ours(xb, lens)
    assert ob.requires_grad
    ob.backward(dy)
    table = _grad_table(ours, ref)
    table["__output__"] = rel(ob, oa)
    table["__input_grad__"] = rel(xb.grad, xa.grad)
    os.makedirs(OUT_DIR, exist_ok=True)
    with open(os.path.join(OUT_DIR, "r02_train_encoder_grad_errors.json"), "w") as f:
        json.dump(table, f, indent=1)
    rp, op = dict(ref.named_parameters()), dict(ours.named_parameters())
    for k in [k for k in table if _is_key_bias(k)]:
        scale = rp[k.replace("w_ks", "w_qs")].grad.norm()
        assert op[k].grad.norm() < 1e-2 * scale and rp[k].grad.norm() < 1e-2 * scale
        del table[k]
    worst = max(table, key=table.get)
    print("encoder training: worst", worst, table[worst])
    assert table["__output__"] < 4e-3
    assert table[worst] < 3e-2, (worst, table[worst])


def test_encoder_training_dropout_draws_reference_masks(dev):
    """With dropout 0.1 and the same CUDA seed the training path draws its masks with the same torch calls, shapes and
    order as the reference's nn.Dropout modules, so outputs stay within tolerance of the seeded reference run."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    n, t, L = 4, 29, 2
    sd = synth.encoder_state_dict(2, L)
    ref = R.Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).to(dev).train()
    ours = Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).to(dev).train()
    ref.load_state_dict(sd); ours.load_state_dict(sd)
    x = torch.randn(n, t, 512, generator=torch.Generator().manual_seed(11)).to(dev)
    with torch.no_grad():
        torch.manual_seed(21)
        oa, = ref(x, [t] * n)
        torch.manual_seed(21)
        ob, = ours(x, [t] * n)
        torch.manual_seed(22)
        oc, = ours(x, [t] * n)
    assert rel(ob, oa) < 1e-2, rel(ob, oa)
    assert rel(oc, oa) > 0.05


def _frontend_pair(dev, matched):
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    sd = synth.frontend_state_dict(1)
    if matched:
        sd = _bf16_values(sd)
    ref = R.Lipreading().to(dev).train()
    ours = Lipreading().to(dev).train()
    ref.load_state_dict(sd); ours.load_state_dict(sd)
    hooks = _match_storage_precision(ref) if matched else []
    return ref, ours, hooks


def _frontend_step(ref, ours, dev, n, t, matched):
    from sbl_for_multilingual_lip_reading_b200 import synth
    x = synth.structured_clips(n, t, seed=31).to(dev)
    if matched:
        x = x.to(BF).float()
    dy = torch.randn(n, t, 512, generator=torch.Generator().manual_seed(12)).to(dev)
    torch.manual_seed(5)
    oa = ref(x)
    oa.backward(dy)
    torch.manual_seed(5)
    ob = ours(x)
    ob.backward(dy)
    return oa, ob


def test_frontend_training_against_fp32_reference(dev):
    """Lipreading in model.train() against autograd through the reference frontend in fp32 (cuDNN): forward within 2.5e-2
    (two bf16 roundings per conv under batch statistics), BatchNorm running statistics updated like nn.BatchNorm, every
    parameter gradient pointing the same way (cosine > 0.9: the Frobenius distance itself is dominated by ReLU masks
    flipped by the forward perturbation, see _match_storage_precision)."""
    ref, ours, _ = _frontend_pair(dev, matched=False)
    oa, ob = _frontend_step(ref, ours, dev, 4, 7, matched=False)
    assert rel(ob, oa) < 2.5e-2
    rb = dict(ref.named_buffers())
    for k, b in ours.named_buffers():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert rel(b, rb[k]) < 5e-3, k
        elif k.endswith("num_batches_tracked"):
            assert int(b) == int(rb[k]) == 1
    rp = dict(ref.named_parameters())
    cos = {k: _cosine(p.grad, rp[k].grad) for k, p in ours.named_parameters()}
    worst = min(cos, key=cos.get)
    print("frontend training vs fp32: lowest gradient cosine", worst, cos[worst])
    assert cos[worst] > 0.9, (worst, cos[worst])


@pytest.mark.parametrize("layer,idx,h", [(1, 0, 22), (2, 0, 22), (3, 0, 11), (4, 1, 3)])
def test_basic_block_training_backward_against_precision_matched_reference(dev, layer, idx, h):
    """The backward kernels of one BasicBlock (stride-1 / strided head with downsample): the reference block with its
    activations rounded to bf16 at the drop-in's storage points (straight-through) and bf16-representable weights and
    input differentiates the same function up to accumulation order; what is left is the bf16 rounding of the gradient
    tensors (and the few ReLU masks a 1-ulp forward difference still flips)."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import synth, training as tr
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    sd = _bf16_values(synth.frontend_state_dict(1))
    ref_fe, our_fe = R.Lipreading().to(dev).train(), Lipreading().to(dev).train()
    ref_fe.load_state_dict(sd); our_fe.load_state_dict(sd)
    rblk = getattr(ref_fe.resnet18, f"layer{layer}")[idx]
    oblk = getattr(our_fe.resnet18, f"layer{layer}")[idx]
    hooks = _match_storage_precision(rblk)
    hooks.append(rblk.register_forward_hook(lambda m, i, o: _RoundSTE.apply(o)))
    g = torch.Generator().manual_seed(40 + layer)
    f = 24
    cin = oblk.conv1.weight.shape[1]
    x = torch.relu(torch.randn(f, h, h, cin, generator=g)).to(BF).to(dev)
    xa = x.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    try:
        ya = rblk(xa)
    finally:
        for hk in hooks:
            hk.remove()
    dy = torch.randn(ya.shape, generator=g).to(dev).to(BF)
    ya.backward(dy.float())
    xb = x.clone().requires_grad_(True)
    ds = oblk.downsample
    yb = tr.BasicBlockFn.apply(xb, oblk.conv1.weight, oblk.bn1.weight, oblk.bn1.bias, oblk.conv2.weight, oblk.bn2.weight,
                               oblk.bn2.bias, ds[0].weight if ds is not None else None,
                               ds[1].weight if ds is not None else None, ds[1].bias if ds is not None else None, oblk)
    yb.backward(dy.permute(0, 2, 3, 1).contiguous())
    table = _grad_table(oblk, rblk)
    table["__output__"] = rel(yb.permute(0, 3, 1, 2), ya)
    table["__input_grad__"] = rel(xb.grad.permute(0, 3, 1, 2), xa.grad)
    worst = max(table, key=table.get)
    print(f"layer{layer}.{idx}: output {table['__output__']:.2e}, worst {worst} {table[worst]:.3e}")
    assert table["__output__"] < 3e-3
    assert table[worst] < 4e-2, (worst, table[worst], table)


def test_stem_training_backward_against_precision_matched_reference(dev):
    """Conv3d + BatchNorm3d(batch stats) + ReLU + MaxPool3d in training mode: output and parameter gradients against the
    reference frontend3D with bf16 storage points (see above)."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import synth, training as tr
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    sd = _bf16_values(synth.frontend_state_dict(1))
    ref_fe, our_fe = R.Lipreading().to(dev).train(), Lipreading().to(dev).train()
    ref_fe.load_state_dict(sd); our_fe.load_state_dict(sd)
    hooks = _match_storage_precision(ref_fe.frontend3D)
    n, t = 2, 6
    x = synth.structured_clips(n, t, seed=55).to(dev).to(BF).float()
    try:
        ya = ref_fe.frontend3D(x)                                             # [N,64,T,22,22]
    finally:
        for hk in hooks:
            hk.remove()
    dy = torch.randn(ya.shape, generator=torch.Generator().manual_seed(3)).to(dev).to(BF)
    ya.backward(dy.float())
    conv, bn = our_fe.frontend3D[0], our_fe.frontend3D[1]
    yb = tr.StemFn.apply(x, conv.weight, bn.weight, bn.bias, bn)              # [N*T,22,22,64]
    yb.backward(dy.permute(0, 2, 3, 4, 1).reshape(n * t, 22, 22, 64).contiguous())
    table = _grad_table(our_fe.frontend3D, ref_fe.frontend3D)
    table["__output__"] = rel(yb.view(n, t, 22, 22, 64).permute(0, 4, 1, 2, 3), ya)
    worst = max(table, key=table.get)
    print("stem:", table)
    assert table["__output__"] < 3e-3
    assert table[worst] < 4e-2, (worst, table[worst])
    assert rel(bn.running_var, ref_fe.frontend3D[1].running_var) < 1e-3


def test_stage1_training_step_with_reference_heads(dev):
    """One optimisation step of the stage-1 classification model the way ...classify/train.py:107-146 runs it (frontend +
    3-layer encoder + fc_1500 / fc_2 heads, CrossEntropy losses, Adam): the project's stage1.Stage1Classifier (drop-in
    frontend + encoder, the reference's attribute names and keys) against the all-reference fp32 model as
    oracle/reference_modules.py restates it; dropout 0 so that both see the same function.  The reference side's loss
    must equal the loss the original classes computed in the same step (tests/golden/reference_training.json).
    Assembling the reference's own Transformer class on the drop-ins (dropin.patched_reference) needs the reference
    sources and is not what this test runs.  The reference forward's pooling line (transformer.py:31,
    `torch.mean(..., dim=2, keepdim=True)` -> fc_1500 on a width-1 tensor) cannot run as written; the heads are applied
    as SURVEY.md states their evident intent: word logits from the time average, language logits from frame 30."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import stage1, synth
    n, t = 8, 31
    sd = dict(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(3, 3, prefix="encoder_v."))
    ref = R.build_stage1(sd).to(dev).train()
    for m_ in ref.modules():
        if isinstance(m_, torch.nn.Dropout):
            m_.p = 0.0
    ours = stage1.Stage1Classifier(n_layers_enc=3, dropout=0.0)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(dev).train()
    assert type(ours.visual_frontend).__module__.startswith("sbl_for_multilingual_lip_reading_b200")

    def step(model, seed):
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
        x = synth.structured_clips(n, t, seed=77).to(dev)                        # [N,1,T,88,88]
        y = torch.randint(0, 1500, (n,), generator=torch.Generator().manual_seed(1)).to(dev)
        lang = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(2)).to(dev)
        torch.manual_seed(seed)
        feat = model.visual_frontend(x)
        out, *_ = model.encoder_v(feat, [t] * n)
        v_t = model.fc_1500(out.mean(dim=1))
        v_l = model.fc_2(out[:, 30, :])
        loss = F.cross_entropy(v_t, y) + 0.1 * F.cross_entropy(v_l, lang)
        opt.zero_grad()
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        opt.step()
        return float(loss.detach()), grads

    la, ga = step(ref, 3)
    lb, gb = step(ours, 3)
    with open(os.path.join(ROOT, "tests", "golden", "reference_training.json")) as f:
        want = json.load(f)["stage1_step_loss"]
    assert abs(la - want) < 1e-5 * abs(want), (la, want)
    cos = {k: _cosine(gb[k], ga[k]) for k in ga if not _is_key_bias(k)}
    with open(os.path.join(OUT_DIR, "r02_train_stage1_step.json"), "w") as f:
        json.dump({"loss_reference": la, "loss_b200": lb, "grad_cosine": cos}, f, indent=1)
    worst = min(cos, key=cos.get)
    print("stage-1 step: loss", la, lb, "lowest gradient cosine", worst, cos[worst])
    assert abs(la - lb) < 2e-3 * abs(la)
    assert cos[worst] > 0.9, (worst, cos[worst])
    head = {k: rel(gb[k], ga[k]) for k in ga if k.startswith("fc_")}
    assert max(head.values()) < 2e-2, head
    # a second step runs on the updated weights (packed caches follow the optimizer's in-place updates)
    lb2, _ = step(ours, 4)
    la2, _ = step(ref, 4)
    assert abs(la2 - lb2) < 5e-3 * abs(la2)


def test_ddp_gradient_allreduce_two_gpus():
    """BASELINE configs[3]: the stage-1 model under DistributedDataParallel on 2 GPUs — every rank ends the backward with
    the NCCL-averaged gradient of the libsblk backward (tests/ddp_train_worker.py under torchrun)."""
    import subprocess
    import sys
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(here, "ddp_train_worker.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ddp gradient all-reduce OK") == 2


def test_stage1_module_has_the_reference_state_dict(dev):
    """stage1.Stage1Classifier mirrors ...classify/transformer/transformer.py key for key."""
    from oracle import reference_modules as R
    from sbl_for_multilingual_lip_reading_b200 import stage1
    ref = R.build_stage1()
    ours = stage1.Stage1Classifier(n_layers_enc=3)
    a, b = ref.state_dict(), ours.state_dict()
    assert sorted(a) == sorted(b)
    assert all(a[k].shape == b[k].shape and a[k].dtype == b[k].dtype for k in a)
    ours.load_state_dict(a)
