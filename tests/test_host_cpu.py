"""CPU-only checks of the host side: C-ABI surface, state-dict contract, init parity, pickling,
loud failure without a GPU."""
import io
import json
import ctypes
import os
import pickle
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/SBL_Multilingual_Lip_reading"

from sbl_for_multilingual_lip_reading_b200 import _lib, synth  # noqa: E402
from sbl_for_multilingual_lip_reading_b200.encoder import Encoder  # noqa: E402
from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading, visual_frontend  # noqa: E402


def _contract():
    with open(os.path.join(ROOT, "tests", "golden", "state_dict_contract.json")) as f:
        return json.load(f)


def _header_functions():
    src = open(os.path.join(ROOT, "include", "sblk.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sblk_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/sblk.h but not exported by libsblk.so"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert sorted(_lib.SIGNATURES) == names
    assert lib.sblk_version() == 200


def test_library_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    rc = lib.sblk_init()
    assert rc < 0
    assert "cuda" in _lib.last_error().lower()


def _integration_snippet():
    with open(os.path.join(ROOT, "INTEGRATION.md")) as f:
        md = f.read()
    block = md.split("## 3.")[1].split("```python")[1].split("```")[0]
    return block


def test_integration_snippet_matches_the_header():
    """The ctypes stub INTEGRATION.md shows must bind the function the header declares (argument count and order)."""
    block = _integration_snippet()
    m = re.search(r"sblk_conv2d_igemm_fwd\.argtypes = \[(.*?)\]", block)
    assert m, "no argtypes line in the INTEGRATION.md snippet"
    shown = [t.strip() for t in m.group(1).split(",")]
    sig = _lib.SIGNATURES["sblk_conv2d_igemm_fwd"][1]
    assert len(shown) == len(sig) == 18
    assert [t == "vp" for t in shown] == [a is ctypes.c_void_p for a in sig]
    call = re.search(r"lib\.sblk_conv2d_igemm_fwd\((.*?)\)\n", block, re.S).group(1)
    call = re.sub(r"#.*", "", call)
    # x.data_ptr() style arguments contain parentheses: count top-level commas
    depth, nargs = 0, 1
    for ch in call:
        depth += ch == "("
        depth -= ch == ")"
        nargs += (ch == "," and depth == 0)
    assert nargs == 18, f"the example call passes {nargs} arguments"


def test_sass_is_blackwell_native():
    """tcgen05 / TMA / TMEM instructions must be in the shipped binary (B200_PROFILING.md evidence table)."""
    try:
        sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=120).stdout
    except FileNotFoundError:
        pytest.skip("cuobjdump not available")
    assert "UTCHMMA" in sass, "no tcgen05.mma in libsblk.so"
    assert "UTMALDG" in sass and "IM2COL" in sass, "no TMA (im2col) loads in libsblk.so"
    assert "LDTM" in sass, "no tcgen05.ld in libsblk.so"
    assert "UBLKCP" in sass, "no bulk-copy (cp.async.bulk) loads in libsblk.so"
    # the warp-level mma.sync path is allowed ONLY in the tiny per-head attention kernel (0.05 % of the FLOPs,
    # SURVEY.md K9); every dense contraction (convs, linears) must be tcgen05
    func = None
    for line in sass.splitlines():
        if "Function :" in line:
            func = line.split("Function :")[1].strip()
        elif " HMMA" in line:
            # (the one-launch encoder stack embeds the same per-head attention routine next to its tcgen05 GEMMs)
            assert func is not None and ("attention_kernel" in func or "encoder_stack_kernel" in func), \
                f"legacy mma.sync in {func}"
    for name in ("igemm_kernel", "igemm2_kernel", "conv3d_bn_relu_pool_kernel", "flatconv2_kernel", "gemm_ln512_kernel",
                 "qkv_attention_kernel", "encoder_stack_kernel"):
        body = [seg for seg in sass.split("Function :") if name in seg.splitlines()[0]]
        assert body and all("UTCHMMA" in seg for seg in body), f"{name} does not use tcgen05.mma"


def test_state_dict_contract_frontend():
    c = _contract()["Lipreading"]
    sd = Lipreading().state_dict()
    assert list(sd.keys()) == list(c.keys()) or sorted(sd.keys()) == sorted(c.keys())
    for k, (shape, dtype) in c.items():
        assert list(sd[k].shape) == shape and str(sd[k].dtype) == dtype, k


def test_state_dict_contract_encoder():
    c = _contract()["Encoder6"]
    sd = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).state_dict()
    assert sorted(sd.keys()) == sorted(c.keys())
    for k, (shape, dtype) in c.items():
        assert list(sd[k].shape) == shape and str(sd[k].dtype) == dtype, k


def test_synth_state_dicts_load():
    fe = Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    enc = Encoder(512, 3, 8, 64, 64, 512, 2048)
    enc.load_state_dict(synth.encoder_state_dict(3, 3))


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference tree not present (GPU box)")
def test_init_parity_with_reference_under_same_seed():
    """Same torch seed -> bit-identical initial weights as the reference constructors, and the reference
    Transformer assembles with the drop-in classes patched in (transformer/transformer.py:9-20)."""
    sys.path.insert(0, REF)
    try:
        from transformer.encoder import Encoder as RefEncoder
        from transformer.video_frontend import Lipreading as RefLipreading
        torch.manual_seed(7)
        a = RefLipreading().state_dict()
        torch.manual_seed(7)
        b = Lipreading().state_dict()
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert torch.equal(a[k], b[k]), k
        torch.manual_seed(7)
        a = RefEncoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).state_dict()
        torch.manual_seed(7)
        b = Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).state_dict()
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert torch.equal(a[k], b[k]), k
    finally:
        sys.path.remove(REF)


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference tree not present (GPU box)")
def test_reference_transformer_assembles_on_dropins():
    from sbl_for_multilingual_lip_reading_b200 import dropin
    with dropin.patched_reference(REF) as mods:
        from transformer.decoder import Decoder
        from transformer.transformer import Transformer
        enc = mods["transformer.encoder"].Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        dec = Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                      pe_maxlen=5000)
        model = Transformer(enc, dec, None)
        assert type(model.visual_frontend).__module__.startswith("sbl_for_multilingual_lip_reading_b200")
        assert type(model.encoder).__module__.startswith("sbl_for_multilingual_lip_reading_b200")
        c = _contract()
        assert len(model.state_dict()) == c["Transformer_num_keys"]
        hot = sorted(k for k in model.state_dict() if k.startswith(("visual_frontend.", "encoder.")))
        assert hot == c["Transformer_hot_path_keys"]


def test_modules_pickle_roundtrip_drops_retired_attributes():
    """Checkpoints are whole pickled modules in the reference (utils.py:22-33)."""
    fe = visual_frontend(None)
    enc = Encoder(512, 2, 8, 64, 64, 512, 2048)
    buf = io.BytesIO()
    torch.save({"fe": fe, "enc": enc}, buf)
    buf.seek(0)
    back = torch.load(buf, weights_only=False)
    for k, v in fe.state_dict().items():
        assert torch.equal(v, back["fe"].state_dict()[k])
    assert pickle.loads(pickle.dumps(enc)).n_layers == 2
    # module settings travel with a checkpoint
    enc.stack_cluster_size = 8
    assert pickle.loads(pickle.dumps(enc)).stack_cluster_size == 8
    enc.stack_cluster_size = 0
    # modules pickled by an earlier version: the attributes its plans and its multi-chain frontend used are dropped,
    # attributes added since come back with their defaults, and nothing else differs from a module built today
    old_fe = dict(fe.__getstate__(), parallel_chains=2, chain_sm_limit=74, l2_prefetch_extra=[torch.zeros(4)],
                  _overlap=(84, 0, None), _tail=(None, None), _block_hook=None)
    old_enc = dict(enc.__getstate__(), _x16_override=None, _resident_counter=None)
    for k in ("stack_cluster_size", "split_clusters"):
        old_enc.pop(k)
    fe3, enc3 = Lipreading.__new__(Lipreading), Encoder.__new__(Encoder)
    fe3.__setstate__(old_fe); enc3.__setstate__(old_enc)
    assert set(fe3.__dict__) == set(fe.__dict__) and set(enc3.__dict__) == set(enc.__dict__)
    assert enc3.stack_cluster_size == 0 and enc3.split_clusters is True
    for k, v in fe.state_dict().items():
        assert torch.equal(v, fe3.state_dict()[k])


def test_cpu_input_is_rejected_loudly():
    fe = Lipreading().eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        fe(torch.zeros(1, 1, 2, 88, 88))
    enc = Encoder(512, 1, 8, 64, 64, 512, 2048).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(torch.zeros(1, 4, 512), [4])


def test_unsupported_encoder_config_is_rejected():
    enc = Encoder(512, 1, 4, 32, 32, 256, 1024).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="only d_model=512"):
        enc(torch.zeros(1, 4, 512), [4])


def test_training_mode_has_no_cpu_fallback_either():
    """model.train() runs the libsblk training path (training.py): on a CPU tensor it must fail loudly, never fall back."""
    fe = Lipreading().train()
    with pytest.raises(RuntimeError, match="CUDA"):
        fe(torch.zeros(1, 1, 2, 88, 88))
    enc = Encoder(512, 1, 8, 64, 64, 512, 2048).train()
    with pytest.raises(RuntimeError, match="CUDA"):
        enc(torch.zeros(1, 2, 512), [2, 2][:1])
    # switching modes re-packs the BN-folded evaluation weights (training updates running stats from a kernel)
    fe._packed = object()
    fe.eval()
    assert fe._packed is None


def test_flat_frames_is_a_valid_flat_sub_buffer():
    """ops.flat_frames (used to run a frame range of a flat conv inside the pipelined plan's head): frames [f0, f1) of the
    zero-haloed flat layout are a row slice of the same storage that is itself a valid flat buffer — same pixels, halo
    rows zero, size sblk_flat_rows(f1 - f0, H, W) — and the slices of a partition cover every row."""
    from sbl_for_multilingual_lip_reading_b200 import ops
    f, h, w, c = 7, 5, 6, 8
    rows = ops.flat_rows(f, h, w)
    assert rows == (f * (h + 1) + 1) * (w + 2)
    data = torch.zeros(rows, c)
    dense = torch.randn(f, h, w, c)
    v = data[(w + 2):(w + 2) + f * (h + 1) * (w + 2)].view(f, h + 1, w + 2, c)
    v[:, :h, 1:w + 1, :] = dense
    x = ops.FlatActs(data, f, h, w)
    assert torch.equal(x.dense(), dense)
    covered = torch.zeros(rows, dtype=torch.bool)
    for f0, f1 in ((0, 3), (3, 4), (4, 7)):
        sub = ops.flat_frames(x, f0, f1)
        assert sub.data.shape[0] == ops.flat_rows(f1 - f0, h, w) and sub.data.is_contiguous()
        assert sub.data.data_ptr() == data.data_ptr() + f0 * (h + 1) * (w + 2) * c * 4
        assert torch.equal(sub.dense(), dense[f0:f1])
        assert not sub.data[:w + 2].any() and not sub.data[-(w + 2):].any()   # halo rows in front of frames f0 / f1
        r0 = f0 * (h + 1) * (w + 2)
        covered[r0:r0 + sub.data.shape[0]] = True
    assert covered.all()
    with pytest.raises(RuntimeError):
        ops.flat_frames(x, 3, 3)
    with pytest.raises(RuntimeError):
        ops.flat_frames(x, 0, 8)
