"""CPU checks of the SBL decoder's host side and of its oracle (oracle/decoder_oracle.py): `Decoder.preprocess` against
the reference's per-utterance loops, the state-dict keys the oracle reads, the decoder's share of the 537-key model
state dict, and (where oracle/_ref is staged) the oracle against the reference `Decoder` itself."""
import json
import os

import pytest
import torch

from oracle import decoder_oracle as O
from sbl_for_multilingual_lip_reading_b200.decoder import IGNORE_ID, Decoder

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOS, EOS = 0, 1


def _decoder(n_layers=6, seed=7):
    torch.manual_seed(seed)
    return Decoder(SOS, EOS, 58, 512, n_layers, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                   pe_maxlen=5000).eval()


def _targets(width, seed):
    """Seeded [rows, width] targets: ids in [2, 58) with IGNORE_ID in the interior and at the end of rows, one all-IGNORE
    row and, where the width allows, a row with the longest target that fits (15 kept tokens)."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for r in range(24):
        y = torch.randint(2, 58, (width,), generator=g)
        kept = int(torch.randint(0, min(15, width) + 1, (1,), generator=g))
        if r == 0:
            kept = 0
        elif r == 1:
            kept = min(15, width)
        keep = torch.zeros(width, dtype=torch.bool)
        keep[torch.randperm(width, generator=g)[:kept]] = True
        if r == 2 and width > 2:                      # a contiguous target followed by trailing IGNORE_IDs only
            keep = torch.arange(width) < min(kept, width - 1)
        rows.append(torch.where(keep, y, torch.full_like(y, IGNORE_ID)))
    return torch.stack(rows)


@pytest.mark.parametrize("width", [1, 5, 15, 16, 17, 31])
def test_preprocess_matches_the_per_utterance_loops(width):
    dec = _decoder(n_layers=1)
    y = _targets(width, seed=100 + width)
    assert (y == IGNORE_ID).all(1).any()
    if width > 2:
        assert ((y[:, 1:] == IGNORE_ID) & (y[:, :-1] != IGNORE_ID)).any()     # an IGNORE_ID right after a token
        assert ((y[:, :-1] == IGNORE_ID) & (y[:, 1:] != IGNORE_ID)).any()     # a token right after an IGNORE_ID
    got_in, got_out = dec.preprocess(y)
    want_in, want_out = O.preprocess(y, SOS, EOS)
    assert got_in.shape == got_out.shape == (y.shape[0], 16)
    assert torch.equal(got_in, want_in) and torch.equal(got_out, want_out)


def test_preprocess_rejects_more_than_15_tokens():
    dec = _decoder(n_layers=1)
    y = torch.full((3, 20), IGNORE_ID, dtype=torch.long)
    y[0, :15] = 7                        # fits: <sos> + 15 tokens = 16 columns
    dec.preprocess(y)
    O.preprocess(y, SOS, EOS)
    y[1, 2:18] = 9                       # 16 kept tokens, with leading and trailing IGNORE_IDs
    with pytest.raises(RuntimeError, match="15 tokens"):
        dec.preprocess(y)
    with pytest.raises(RuntimeError):
        O.preprocess(y, SOS, EOS)


class _Recording(dict):
    def __init__(self, *a):
        super().__init__(*a)
        self.read = set()

    def __getitem__(self, k):
        self.read.add(k)
        return super().__getitem__(k)


def test_oracle_reads_every_decoder_key_and_no_other():
    dec = _decoder(n_layers=6)
    sd = _Recording(dec.state_dict())
    assert len(sd) == 316
    g = torch.Generator().manual_seed(1)
    enc = torch.randn(2, 3, 512, generator=g)
    ys = torch.randint(2, 58, (2, 17), generator=g)
    with torch.no_grad():
        a, b = O.step_logits(sd, ys, ys.flip(1), enc, 2)
    assert a.shape == b.shape == (2, 58) and torch.isfinite(a).all() and torch.isfinite(b).all()
    assert sd.read == set(sd.keys())
    assert O.n_layers(sd) == 6


def test_decoder_and_hot_path_keys_make_the_model_state_dict():
    with open(os.path.join(ROOT, "tests", "golden", "state_dict_contract.json")) as f:
        c = json.load(f)
    keys = set(_decoder(n_layers=6).state_dict())
    hot = set(c["Transformer_hot_path_keys"])
    assert len(keys) == 316 and not keys & hot
    assert len(keys) + len(hot) == c["Transformer_num_keys"] == 537


def test_oracle_mixing_is_the_documented_closed_form():
    """The aliased loops give l2r' = l2r + flip(r2l), r2l' = 2 r2l + flip(l2r) (include/sblk.h), which differs from
    the unaliased r2l + flip(l2r) by exactly r2l."""
    g = torch.Generator().manual_seed(3)
    for L in (1, 2, 3, 16):
        l2r, r2l = torch.randn(2, L, 8, generator=g, dtype=torch.float64), torch.randn(2, L, 8, generator=g,
                                                                                        dtype=torch.float64)
        a, b = O.bidir_mix(l2r, r2l)
        torch.testing.assert_close(a, l2r + r2l.flip(1), rtol=1e-15, atol=1e-15)
        torch.testing.assert_close(b, 2 * r2l + l2r.flip(1), rtol=1e-14, atol=1e-14)


def _ref_staged():
    from oracle import ref_runtime
    return ref_runtime.available()


@pytest.mark.skipif(not _ref_staged(), reason="oracle/_ref not staged (python oracle/fetch_ref.py needs the reference)")
def test_step_logits_equal_the_reference_decoder():
    """fp32 on the CPU: the reference Decoder's greedy decode (its per-step output projections, tapped) against
    `step_logits` on the reference's own tokens and the same weights."""
    from oracle import ref_runtime
    R = ref_runtime.load_reference("sbl")
    torch.manual_seed(7)
    ref = R.Decoder(SOS, EOS, 58, 512, 2, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                    pe_maxlen=5000).eval()
    g = torch.Generator().manual_seed(4)
    enc = torch.randn(3, 7, 512, generator=g)
    taps = {"l2r": [], "r2l": []}
    hooks = [getattr(ref, "tgt_word_prj_" + d).register_forward_hook(lambda m, i, o, d=d: taps[d].append(o.detach()))
             for d in ("l2r", "r2l")]
    try:
        with torch.no_grad():
            ys_l2r, ys_r2l = ref.recognize_beam(enc)
    finally:
        for h in hooks:
            h.remove()
    sd = ref.state_dict()
    assert len(taps["l2r"]) == len(taps["r2l"]) == 16
    with torch.no_grad():
        for i in range(16):
            a, b = O.step_logits(sd, ys_l2r, ys_r2l, enc, i + 1)
            torch.testing.assert_close(a, taps["l2r"][i].reshape(a.shape), rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(b, taps["r2l"][i].reshape(b.shape), rtol=1e-4, atol=1e-4)
