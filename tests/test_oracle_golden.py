"""The CPU oracle must reproduce every golden vector produced by the reference itself
(tests/golden/make_golden.py, run against /root/reference in the build container)."""
import numpy as np
import torch

from oracle import visual_encoder_oracle as O
from sbl_for_multilingual_lip_reading_b200 import synth

TOL = 2e-5  # same torch primitives on the same CPU: differences are op-fusion level only


def close(a, b, tol=TOL):
    a = torch.as_tensor(a).float()
    b = torch.as_tensor(b).float()
    assert a.shape == b.shape, (a.shape, b.shape)
    err = (a - b).abs().max().item() / (b.abs().max().item() + 1e-12)
    assert err < tol, err


def test_frontend3d(golden):
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(1, 2, seed=11)
    close(O.frontend3d(x, sd), golden["frontend3d_T2"])


def test_basic_blocks(golden):
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(1, 2, seed=11)
    y = O.frontend3d(x, sd).transpose(1, 2).contiguous().view(-1, 64, 22, 22)
    l10 = O.basic_block(y, sd, "resnet18.layer1.0", 1, False)
    close(l10, golden["layer1_0_T2"])
    l11 = O.basic_block(l10, sd, "resnet18.layer1.1", 1, False)
    close(O.basic_block(l11, sd, "resnet18.layer2.0", 2, True), golden["layer2_0_T2"])


def test_frontend_config1(golden):
    """BASELINE config 1: one 29x88x88 clip through Conv3d frontend + ResNet-18 trunk."""
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(1, 29, seed=7)
    close(O.frontend_forward(x, sd), golden["frontend_c1"])
    close(O.lipreading_forward(x, sd), golden["frontend_c1"].reshape(1, 29, 512))


def test_frontend_zero_padded_frame(golden):
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(2, 6, seed=8, pad_frames=1)
    close(O.frontend_forward(x, sd), golden["frontend_N2_T6_pad1"])


def test_encoder_full_lengths(golden, golden_inputs):
    sd6 = synth.encoder_state_dict(2, 6)
    close(O.encoder_forward(torch.from_numpy(golden_inputs["xin"]), [29], sd6)[0], golden["encoder6_N1_T29"])
    close(O.encoder_forward(torch.from_numpy(golden_inputs["xin40"]), [40], sd6)[0], golden["encoder6_N1_T40"])
    sd3 = synth.encoder_state_dict(3, 3)
    close(O.encoder_forward(torch.from_numpy(golden_inputs["xin3"]), [31, 31], sd3, n_layers=3)[0],
          golden["encoder3_N2_T31"])


def test_encoder_ragged_and_attns(golden, golden_inputs):
    sd6 = synth.encoder_state_dict(2, 6)
    out, attns = O.encoder_forward(torch.from_numpy(golden_inputs["xin_r"]), [12, 7, 1], sd6, return_attns=True)
    close(out, golden["encoder6_ragged_out"])
    close(attns[0], golden["encoder6_ragged_attn0"])
    close(attns[5], golden["encoder6_ragged_attn5"])
    assert len(attns) == 6 and attns[0].shape == (8 * 3, 12, 12)
    # padded query rows are zeroed by the non_pad_mask multiplies (encoder.py:86,89)
    assert float(out[1, 7:].abs().max()) == 0.0 and float(out[2, 1:].abs().max()) == 0.0


def test_whole_hot_path(golden):
    sd = {}
    sd.update(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, 6, prefix="encoder."))
    x = synth.synthetic_clips(2, 6, seed=8, pad_frames=1)
    close(O.visual_encoder_forward(x, sd), golden["visual_encoder_N2_T6"])


def test_dropout_mask_semantics():
    """F.dropout(p=0.5) keeps with prob 0.5 and scales by 2 (video_frontend.py:122)."""
    sd = synth.frontend_state_dict(1)
    x = synth.synthetic_clips(1, 1, seed=3)
    base = O.lipreading_forward(x, sd)
    mask = (torch.arange(512) % 2).float().view(1, 512)
    dropped = O.lipreading_forward(x, sd, dropout_mask=mask)
    assert torch.equal(dropped.view(-1)[0::2], torch.zeros(256))
    close(dropped.view(-1)[1::2], 2.0 * base.view(-1)[1::2])


def test_positional_encoding_table():
    sd6 = synth.encoder_state_dict(2, 1)
    assert torch.equal(O.positional_encoding_table(5000, 512), sd6["positional_encoding.pe"])


def test_flops_formula():
    # SURVEY.md §8d exact integers
    assert O.flops_per_clip(29, 6) == 19457472512
    assert O.flops_per_clip(30, 6) == 20128788480
    assert O.flops_per_clip(31, 6) == 20800129024
    assert O.flops_per_clip(40, 6) == 26843299840
    assert O.flops_per_clip(31, 3) == 20209119232


def test_top1_labels_first_chunk():
    """The oracle reproduces the reference's top-1 labels (plain and centred heads) on the first 8 of the 1,000
    clips of tests/golden/top1_1000.npz (the GPU suite checks all 1,000 against the CUDA path)."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "top1_1000.npz"))
    sd = {}
    sd.update(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, 6, prefix="encoder."))
    heads = synth.classifier_heads(9)
    x = synth.structured_clips(int(g["chunk"]), int(g["frames"]), seed=5000)[:8]
    with torch.no_grad():
        out = O.visual_encoder_forward(x, sd)
        logits, ll = synth.classify(out, heads)
        lc = (out.mean(dim=1) - torch.from_numpy(g["mu"])) @ heads["fc_1500.weight"].t()
    assert (logits.argmax(dim=1).numpy() == g["top1"][:8]).all()
    assert (ll.argmax(dim=1).numpy() == g["lang"][:8]).all()
    v, i = lc.topk(2, dim=1)
    close(v[:, 0] - v[:, 1], g["margin_centred"][:8], tol=1e-3)
    assert (i[:, 0].numpy() == g["top1_centred"][:8]).all()


def test_input_pipeline_oracle_matches_reference_transforms():
    """oracle/input_pipeline_oracle.py against tests/golden/input_pipeline.npz (the reference's cvtransforms functions):
    eval path (centre crop, pad 29 -> 30) and train-style per-frame crops (offsets drawn like RandomCrop, pad -> 31)."""
    import os
    import random
    from oracle import input_pipeline_oracle as P
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "input_pipeline.npz"))
    u8 = synth.synthetic_u8_clips(1, 29, seed=21)[0].numpy()
    assert np.array_equal(P.eval_clip(u8, 30), g["eval_T30"])
    random.seed(5)
    offs = []
    for _ in range(29):            # cvtransforms.RandomCrop draws x1 then y1 for every frame
        x1 = random.randint(0, 8)
        y1 = random.randint(0, 8)
        offs.append((y1, x1))
    got = P.pad_frames(P.crop_at(P.load_and_normalize(u8), offs), 31)
    assert np.array_equal(got, g["train_crop_T31"])
    # the 256-entry table the CUDA path uses is the same arithmetic, rounded to bf16 once
    lut = synth.normalize_lut().float().numpy()
    ref = P.load_and_normalize(np.arange(256, dtype=np.uint8)).astype(np.float32)
    assert np.array_equal(lut, torch.from_numpy(ref).to(torch.bfloat16).float().numpy())


# ------------------------------------------------------------- the module-form restatement (oracle/reference_modules.py)
def test_reference_modules_state_dicts_match_the_reference_contract():
    """Same keys, shapes and dtypes as the reference's Lipreading and 6-layer Encoder (tests/golden/state_dict_contract.json),
    and the stage-1 model is those two plus its word and language heads."""
    import json
    import os
    from oracle import reference_modules as RM
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "state_dict_contract.json")) as f:
        contract = json.load(f)

    def table(m):
        return {k: [list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()}
    assert table(RM.Lipreading()) == contract["Lipreading"]
    assert table(RM.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)) == contract["Encoder6"]
    s1 = table(RM.build_stage1())
    want = {"visual_frontend." + k: v for k, v in contract["Lipreading"].items()}
    want.update({"encoder_v." + k: v for k, v in contract["Encoder6"].items() if not k.startswith("layer_stack.")
                 or int(k.split(".")[1]) < 3})
    want.update({"fc_1500.weight": [[1500, 512], "torch.float32"], "fc_1500.bias": [[1500], "torch.float32"],
                 "fc_2.weight": [[2, 512], "torch.float32"], "fc_2.bias": [[2], "torch.float32"]})
    assert s1 == want


def test_reference_modules_reproduce_the_reference_outputs(golden, golden_inputs):
    """In eval mode, with the always-on frontend dropout left out (`_frontend_forward`, as the goldens were produced) and
    encoder dropout inactive, the modules reproduce every golden vector of the reference modules."""
    from oracle import reference_modules as RM
    fe = RM.Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe.eval()
    enc6 = RM.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
    enc6.load_state_dict(synth.encoder_state_dict(2, 6))
    enc6.eval()
    enc3 = RM.Encoder(512, 3, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
    enc3.load_state_dict(synth.encoder_state_dict(3, 3))
    enc3.eval()
    with torch.no_grad():
        x = synth.synthetic_clips(1, 2, seed=11)
        close(fe.frontend3D(x), golden["frontend3d_T2"])
        y = fe.frontend3D(x).transpose(1, 2).contiguous().view(-1, 64, 22, 22)
        close(fe.resnet18.layer1[0](y.clone()), golden["layer1_0_T2"])
        close(fe.resnet18.layer2[0](fe.resnet18.layer1(y.clone())), golden["layer2_0_T2"])
        close(fe._frontend_forward(synth.synthetic_clips(1, 29, seed=7)), golden["frontend_c1"])
        feat = fe._frontend_forward(synth.synthetic_clips(2, 6, seed=8, pad_frames=1))
        close(feat, golden["frontend_N2_T6_pad1"])
        close(enc6(torch.from_numpy(golden_inputs["xin"]), [29])[0], golden["encoder6_N1_T29"])
        close(enc6(torch.from_numpy(golden_inputs["xin40"]), [40])[0], golden["encoder6_N1_T40"])
        close(enc3(torch.from_numpy(golden_inputs["xin3"]), [31, 31])[0], golden["encoder3_N2_T31"])
        out, attns = enc6(torch.from_numpy(golden_inputs["xin_r"]), [12, 7, 1], return_attns=True)
        close(out, golden["encoder6_ragged_out"])
        close(attns[0], golden["encoder6_ragged_attn0"])
        close(attns[5], golden["encoder6_ragged_attn5"])
        close(enc6(feat.view(2, 6, 512), [6, 6])[0], golden["visual_encoder_N2_T6"])


def test_reference_modules_dropout_sites():
    """Training-mode dropout: the frontend's always-on F.dropout(p=0.5) on the pooled features, and the encoder's four
    draws in the reference's order and shapes — input [N,T,512], then per layer attention probabilities [H*N,T,T], the
    fc output and the feed-forward output (both [N,T,512])."""
    from oracle import reference_modules as RM
    n, t, L = 2, 5, 2
    enc = RM.Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000).train()
    seen = []
    for name, m in enc.named_modules():
        if isinstance(m, torch.nn.Dropout):
            m.register_forward_hook(lambda mod, i, o, name=name: seen.append((name, tuple(i[0].shape))))
    enc(torch.randn(n, t, 512), [t] * n)
    want = [("dropout", (n, t, 512))]
    for i in range(L):
        want += [(f"layer_stack.{i}.slf_attn.attention.dropout", (8 * n, t, t)),
                 (f"layer_stack.{i}.slf_attn.dropout", (n, t, 512)), (f"layer_stack.{i}.pos_ffn.dropout", (n, t, 512))]
    assert seen == want
    fe = RM.Lipreading()
    fe.load_state_dict(synth.frontend_state_dict(1))
    fe.eval()
    x = synth.synthetic_clips(1, 3, seed=3)
    with torch.no_grad():
        base = fe._frontend_forward(x).view(1, 3, 512)
        torch.manual_seed(0)
        dropped = fe(x)
    kept = dropped != 0
    assert 0.3 < float(kept.float().mean()) < 0.7
    close(dropped[kept], 2.0 * base[kept])
