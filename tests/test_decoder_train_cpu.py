"""Host-side checks of the SBL decoder's training mode that need no GPU: what it refuses, and the float64 restatement
of its dropout (tests/decoder_dropout_oracle.py) against the evaluation oracle (oracle/decoder_oracle.py)."""
import pytest
import torch

import decoder_dropout_oracle as DO
from oracle import decoder_oracle as O

SOS, EOS, VOCAB = 0, 1, 58


def _decoder(n_layers=1):
    from sbl_for_multilingual_lip_reading_b200.decoder import Decoder
    torch.manual_seed(7)
    return Decoder(SOS, EOS, VOCAB, 512, n_layers, 8, 64, 64, 512, 2048, dropout=0.1).train()


def _tgt(n):
    return torch.randint(2, VOCAB, (n, 5)), torch.randint(2, VOCAB, (n, 5))


def test_training_forward_refuses_cpu_tensors():
    dec = _decoder()
    a, b = _tgt(2)
    with pytest.raises(RuntimeError, match="CUDA"):
        dec(a, b, torch.randn(2, 29, 512), [29, 29])


class _FakeCuda:
    """Stands in for a CUDA tensor in the shape / mode checks, which run before anything touches a device."""

    def __init__(self, shape):
        self.shape = torch.Size(shape)
        self.is_cuda = True

    def dim(self):
        return len(self.shape)

    def size(self, i):
        return self.shape[i]


def test_training_forward_refuses_long_encoder_outputs_and_return_attns():
    dec = _decoder()
    a, b = _tgt(2)
    with pytest.raises(RuntimeError, match="T <= 64"):
        dec(a, b, _FakeCuda((2, 65, 512)), [65, 65])
    with pytest.raises(RuntimeError, match="return_attns"):
        dec(a, b, _FakeCuda((2, 29, 512)), [29, 29], return_attns=True)
    dec.eval()                                      # evaluation keeps its own limit (<= 128 frames)
    with pytest.raises(RuntimeError, match="T <= 128"):
        dec._check(_FakeCuda((2, 129, 512)))
    dec._check(_FakeCuda((2, 65, 512)))


def test_recognize_beam_refuses_training_mode():
    dec = _decoder()
    with pytest.raises(RuntimeError, match=r"model\.eval\(\)"):
        dec.recognize_beam(_FakeCuda((2, 29, 512)))


def test_dropout_oracle_without_factors_is_the_evaluation_oracle():
    """The dropout restatement with every factor None, and with every factor 1, is decoder_oracle.step_logits (float64,
    CPU); a zeroed factor changes the result."""
    dec = _decoder(2)
    sd = {k: v.detach().double() for k, v in dec.state_dict().items()}
    n, L, t = 3, 4, 6
    g = torch.Generator().manual_seed(0)
    enc = torch.randn(n, t, 512, generator=g, dtype=torch.float64)
    ys = torch.randint(0, VOCAB, (n, 17), generator=g), torch.randint(0, VOCAB, (n, 17), generator=g)

    def ones(k):
        return (torch.ones(8 * n, L, L, dtype=torch.float64), torch.ones(n * L, 512, dtype=torch.float64),
                torch.ones(8 * n, L, t, dtype=torch.float64), torch.ones(n * L, 512, dtype=torch.float64) * k,
                torch.ones(n * L, 512, dtype=torch.float64))
    want = O.step_logits(sd, ys[0], ys[1], enc, L)
    none = {d: {"emb": None, "layers": [(None,) * 5, (None,) * 5]} for d in ("l2r", "r2l")}
    for a, b in zip(DO.step_logits(sd, ys[0], ys[1], enc, L, none), want):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12)
    drops = {d: {"emb": torch.ones(n * L, 512, dtype=torch.float64), "layers": [ones(1.0), ones(1.0)]}
             for d in ("l2r", "r2l")}
    for a, b in zip(DO.step_logits(sd, ys[0], ys[1], enc, L, drops), want):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12)
    drops["r2l"]["layers"][1] = ones(0.0)
    bad = DO.step_logits(sd, ys[0], ys[1], enc, L, drops)
    assert not torch.allclose(bad[1], want[1], rtol=1e-6, atol=1e-6)
