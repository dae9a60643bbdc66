"""`-m gpu` tests of the training path fed from the loader's raw uint8 frames (ops_train.stem_im2col_u8,
Lipreading.forward_u8 and Stage1Classifier.forward(u8=...) in model.train()).

The reference for every check is the fp32 clip the reference loader builds on the host, as
oracle/input_pipeline_oracle.py restates it (float64 normalise -> crop -> mirror -> float32 frame padding), fed through
the existing fp32 training path.  The uint8 path must reproduce it bit for bit: the stem's im2col, and from there the
logits, the loss, the BatchNorm running statistics and every parameter gradient.
"""
import os
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sbl_for_multilingual_lip_reading_b200 import ops
    assert ops.init() > 0
    return torch.device("cuda:0")


def oracle_clips(u8, offsets, flips, t_out):
    """The loader's fp32 clips [N, t_out, 88, 88] of raw frames u8 [N, T_in, H0, W0] (numpy) with per-frame (y1, x1)
    offsets [N*T_in, 2], mirrored where flips[n]."""
    from oracle import input_pipeline_oracle as P
    n, t_in = u8.shape[:2]
    clips = []
    for i in range(n):
        v = P.crop_at(P.load_and_normalize(u8[i]), [tuple(o) for o in offsets[i * t_in:(i + 1) * t_in]])
        if flips[i]:
            v = v[:, :, ::-1]
        clips.append(P.pad_frames(v, t_out))
    return torch.from_numpy(np.stack(clips))


def u8_frames(n, t_in, h0=96, w0=96, seed=21):
    from sbl_for_multilingual_lip_reading_b200 import synth
    return synth.synthetic_u8_clips(n, t_in, h0=h0, w0=w0, seed=seed)


def check_im2col(dev, u8, crop, flips, t_out, offsets):
    """stem_im2col_u8 against stem_im2col of the oracle clip, both orientations, every element."""
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot, synth
    lut = synth.normalize_lut().to(dev)
    ref = oracle_clips(u8.numpy(), offsets, flips or [False] * u8.shape[0], t_out).to(dev)
    x = u8.to(dev)
    flip = None if flips is None else torch.tensor(flips, dtype=torch.bool)
    got = ot.stem_im2col_u8(x, lut, t_out, crop, flip=flip)
    assert torch.equal(got, ot.stem_im2col(ref))
    m = u8.shape[0] * t_out * 44 * 44
    for ld in (m, m + 2, m + 1936 + 130):             # ld_out > M: zero columns past M, a partial frame slot
        got_t = ot.stem_im2col_u8(x, lut, t_out, crop, flip=flip, transposed=True, ld_out=ld)
        assert torch.equal(got_t, ot.stem_im2col(ref, transposed=True, ld_out=ld)), ld
    return ref


# ----------------------------------------------------------------------------------------------------- the kernel
def test_im2col_u8_golden_random_crop(dev):
    """The reference's own RandomCrop golden (random.seed(5), 29 frames padded to 31): the oracle clip equals the golden
    and the uint8 im2col equals the fp32 im2col of it."""
    from sbl_for_multilingual_lip_reading_b200.video_frontend import random_crop_offsets
    g = np.load(os.path.join(HERE, "golden", "input_pipeline.npz"))
    u8 = u8_frames(1, 29, seed=21)
    random.seed(5)
    offs = random_crop_offsets(1, 29)
    ref = check_im2col(dev, u8, offs, [False], 31, offs.numpy())
    assert np.array_equal(ref[0].cpu().numpy(), g["train_crop_T31"])
    check_im2col(dev, u8, offs.to(dev), [False], 31, offs.numpy())          # offsets already on the GPU


@pytest.mark.parametrize("n,t_in,t_out,h0,w0,case", [
    (3, 7, 9, 96, 96, "centre"),
    (32, 5, 5, 96, 96, "corners"),
    (3, 6, 8, 100, 92, "random"),
    (1, 4, 4, 88, 88, "zero"),
    (1, 3, 6, 96, 96, "corners"),
])
def test_im2col_u8_crops_flips_and_shapes(dev, n, t_in, t_out, h0, w0, case):
    u8 = u8_frames(n, t_in, h0, w0, seed=100 + n + h0)
    frames = n * t_in
    if case == "centre":
        crop = ((h0 - 88) // 2, (w0 - 88) // 2)
        offs = np.tile(np.array(crop, dtype=np.int32), (frames, 1))
    elif case == "corners":
        corners = [(0, 0), (0, 8), (8, 0), (8, 8)]
        offs = np.array([corners[i % 4] for i in range(frames)], dtype=np.int32)
        crop = torch.from_numpy(offs)
    elif case == "random":
        from sbl_for_multilingual_lip_reading_b200.video_frontend import random_crop_offsets
        crop = random_crop_offsets(n, t_in, h0, w0, rng=random.Random(3))
        offs = crop.numpy()
        assert offs[:, 0].max() <= h0 - 88 and offs[:, 1].max() <= w0 - 88
    else:
        crop = (0, 0)
        offs = np.zeros((frames, 2), dtype=np.int32)
    flips = [i % 3 == 1 for i in range(n)] if n > 1 else [True]
    check_im2col(dev, u8, crop, flips, t_out, offs)
    check_im2col(dev, u8, crop, None, t_out, offs)                           # flip=None: no clip mirrored


def test_im2col_u8_clamps_device_offsets(dev):
    """Per-frame offsets in device memory cannot be checked by the C ABI; the kernel clamps them into the frame."""
    u8 = u8_frames(2, 3, seed=9)
    bad = torch.tensor([(-5, 20), (12, -3), (100, 100), (8, 8), (-1, -1), (3, 9)], dtype=torch.int32)
    clamped = bad.clamp(0, 8).numpy()
    check_im2col(dev, u8, bad.to(dev), [True, False], 4, clamped)


def _abi(dev, **over):
    """sblk_stem_im2col_u8 with valid arguments except `over`; -> (rc, sblk_last_error())."""
    from sbl_for_multilingual_lip_reading_b200 import _lib, synth
    lib = _lib.load()
    x = torch.zeros((1, 4, 96, 96), dtype=torch.uint8, device=dev)
    lut = synth.normalize_lut().to(dev)
    out = torch.empty((256 * 4 * 1936 + 64,), dtype=torch.bfloat16, device=dev)
    a = dict(x=x.data_ptr(), lut=lut.data_ptr(), crop=None, cy=4, cx=4, flip=None, out=out.data_ptr(), N=1, T_in=4,
             T_out=4, H0=96, W0=96, transposed=0, ld_out=256, stream=torch.cuda.current_stream().cuda_stream)
    a.update(over)
    rc = lib.sblk_stem_im2col_u8(*a.values())
    torch.cuda.synchronize()
    return rc, _lib.last_error()


def test_im2col_u8_rejections(dev):
    """Each argument check returns a negative code and a message without launching; the Python wrapper validates what
    it can see on the host."""
    from sbl_for_multilingual_lip_reading_b200 import ops_train as ot, synth
    rc, msg = _abi(dev)
    assert rc == 0, msg
    m = 4 * 1936
    cases = [
        (dict(x=None), "null pointer"),
        (dict(lut=None), "null pointer"),
        (dict(out=None), "null pointer"),
        (dict(T_out=3), "bad shape"),
        (dict(H0=87), "bad shape"),
        (dict(W0=80), "bad shape"),
        (dict(N=0), "bad shape"),
        (dict(cy=9), "crop offset"),
        (dict(cx=-1), "crop offset"),
        (dict(transposed=1, ld_out=m - 2), "ld_out must be even and >= M"),
        (dict(transposed=1, ld_out=m + 1), "ld_out must be even and >= M"),
        (dict(transposed=1, ld_out=65536 * 1936), "too many frames"),
        (dict(N=1 << 22, T_in=4, T_out=31), "too many frames"),
    ]
    for over, want in cases:
        rc, msg = _abi(dev, **over)
        assert rc < 0 and want in msg, (over, rc, msg)
    out = torch.empty((256 * 4 * 1936 + 64,), dtype=torch.bfloat16, device=dev)
    rc, msg = _abi(dev, out=out.data_ptr() + 2)
    assert rc < 0 and "16-byte aligned" in msg, msg
    # the wrapper
    x = torch.zeros((2, 4, 96, 96), dtype=torch.uint8, device=dev)
    lut = synth.normalize_lut().to(dev)
    with pytest.raises(RuntimeError, match="leaves the 96x96 frame"):
        ot.stem_im2col_u8(x, lut, 4, torch.tensor([[0, 0]] * 7 + [[0, 9]], dtype=torch.int32))
    with pytest.raises(RuntimeError, match="int32"):
        ot.stem_im2col_u8(x, lut, 4, torch.zeros((8, 2), dtype=torch.int64))
    with pytest.raises(RuntimeError, match="crop offset"):
        ot.stem_im2col_u8(x, lut, 4, (4, 9))
    with pytest.raises(RuntimeError, match="flip"):
        ot.stem_im2col_u8(x, lut, 4, (4, 4), flip=torch.ones(2))
    with pytest.raises(RuntimeError, match="flip"):
        ot.stem_im2col_u8(x, lut, 4, (4, 4), flip=torch.ones(3, dtype=torch.bool))
    with pytest.raises(RuntimeError, match="bad shape"):
        ot.stem_im2col_u8(x, lut, 3, (4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ot.stem_im2col_u8(x.cpu(), lut, 4, (4, 4))


# ------------------------------------------------------------------------------------------------ module parity
def _batch(dev, n, t_in, seed):
    from sbl_for_multilingual_lip_reading_b200.video_frontend import random_crop_offsets
    u8 = u8_frames(n, t_in, seed=seed)
    offs = random_crop_offsets(n, t_in, rng=random.Random(seed))
    flips = [i % 2 == 0 for i in range(n)]
    ref = oracle_clips(u8.numpy(), offs.numpy(), flips, 31).to(dev)
    return u8.to(dev), offs, torch.tensor(flips), ref


def _assert_same_state(a, b):
    for (k, p), (k2, q) in zip(a.named_parameters(), b.named_parameters()):
        assert k == k2
        assert torch.equal(p.grad, q.grad), k
    for (k, p), (k2, q) in zip(a.named_buffers(), b.named_buffers()):
        assert torch.equal(p, q), k


def test_stage1_step_u8_equals_fp32(dev):
    """One stage-1 step (and a second after an Adam update) of Stage1Classifier in train(): forward(u8=...) against
    forward(oracle fp32 clip), same torch seed -> same dropout masks.  Logits, loss, every BN running statistic and
    every parameter gradient are identical."""
    from sbl_for_multilingual_lip_reading_b200 import stage1
    n = 4
    torch.manual_seed(0)
    a = stage1.Stage1Classifier(n_layers_enc=3).load_synthetic(1, 3).to(dev).train()
    b = stage1.Stage1Classifier(n_layers_enc=3)
    b.load_state_dict(a.state_dict())
    b = b.to(dev).train()
    opt_a = torch.optim.Adam(a.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
    opt_b = torch.optim.Adam(b.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
    y = torch.randint(0, 1500, (n,), generator=torch.Generator().manual_seed(1)).to(dev)
    lang = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(2)).to(dev)
    for step, seed in enumerate((31, 32)):
        u8, offs, flips, ref = _batch(dev, n, 29, 40 + step)

        def run(model, opt, **inp):
            torch.manual_seed(seed)
            v_t, v_l = model(**inp)
            loss = F.cross_entropy(v_t, y) + 0.1 * F.cross_entropy(v_l, lang)
            opt.zero_grad()
            loss.backward()
            return v_t.detach(), v_l.detach(), loss.detach()

        ra = run(a, opt_a, padded_input_visual=ref)
        rb = run(b, opt_b, u8=u8, frames=31, crop=offs, flip=flips)
        for p, q in zip(ra, rb):
            assert torch.equal(p, q), step
        _assert_same_state(a, b)
        assert int(b.visual_frontend.frontend3D[1].num_batches_tracked) == step + 1
        opt_a.step()
        opt_b.step()


def test_lipreading_forward_u8_train_equals_fp32(dev):
    """Lipreading.forward_u8 alone in train(): features (after the always-on dropout), running statistics and
    gradients equal forward(oracle fp32 clip), for two steps with an Adam update between them."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    a, b = Lipreading(), Lipreading()
    a.load_state_dict(synth.frontend_state_dict(1))
    b.load_state_dict(synth.frontend_state_dict(1))
    a, b = a.to(dev).train(), b.to(dev).train()
    opt_a, opt_b = torch.optim.Adam(a.parameters(), lr=1e-3), torch.optim.Adam(b.parameters(), lr=1e-3)
    for step in range(2):
        u8, offs, flips, ref = _batch(dev, 3, 29, 60 + step)
        dy = torch.randn((3, 31, 512), generator=torch.Generator().manual_seed(step)).to(dev)
        torch.manual_seed(5 + step)
        fa = a(ref.unsqueeze(1))
        torch.manual_seed(5 + step)
        fb = b.forward_u8(u8, frames=31, crop=offs.to(dev), flip=flips.to(dev))
        assert fb.shape == (3, 31, 512) and fb.requires_grad
        assert torch.equal(fa, fb)
        opt_a.zero_grad()
        opt_b.zero_grad()
        fa.backward(dy)
        fb.backward(dy)
        _assert_same_state(a, b)
        opt_a.step()
        opt_b.step()


def test_forward_u8_eval_rejects_flip(dev):
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe = fe.to(dev).eval()
    u8 = u8_frames(2, 5).to(dev)
    with pytest.raises(RuntimeError, match="flip"):
        fe.forward_u8(u8, frames=6, flip=torch.tensor([True, False]))
    with torch.no_grad():
        assert fe.forward_u8(u8, frames=6).shape == (2, 6, 512)


def test_u8_stem_saves_no_fp32_clip(dev):
    """The training forward through the uint8 path keeps the uint8 frames and the offsets for the backward, never a
    float32 clip (checked on every tensor autograd saves; the fp32 path is the positive control of the check)."""
    from sbl_for_multilingual_lip_reading_b200 import synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe = fe.to(dev).train()
    n, t_in, t = 2, 29, 31
    u8, offs, flips, ref = _batch(dev, n, t_in, 70)

    def saved(fn):
        seen = []

        def pack(x):
            seen.append((x.dtype, tuple(x.shape)))
            return x
        with torch.autograd.graph.saved_tensors_hooks(pack, lambda x: x):
            out = fn()
        out.sum().backward()
        return seen

    def clip_like(s):
        return [d for d in s if d[0] == torch.float32 and len(d[1]) >= 2 and d[1][-2:] == (88, 88)]

    s_fp32 = saved(lambda: fe(ref.unsqueeze(1)))
    assert clip_like(s_fp32), s_fp32
    s_u8 = saved(lambda: fe.forward_u8(u8, frames=t, crop=offs, flip=flips))
    assert not clip_like(s_u8), s_u8
    assert (torch.uint8, (n, t_in, 96, 96)) in s_u8
    assert (torch.int32, (n * t_in, 2)) in s_u8 and (torch.int32, (n,)) in s_u8


def test_ddp_u8_gradient_allreduce_two_gpus():
    """Stage1Classifier under DistributedDataParallel fed with forward(u8=...) on 2 GPUs: gradients identical on both
    ranks and equal to the NCCL average of each shard's single-rank gradients (tests/ddp_train_u8_worker.py)."""
    import subprocess
    import sys
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29537", os.path.join(HERE, "ddp_train_u8_worker.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ddp u8 gradient all-reduce OK") == 2
