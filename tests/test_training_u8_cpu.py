"""Host-side parts of the uint8 training input (no GPU): the RandomCrop offset helper against the reference's golden,
and the argument checks of Lipreading.forward_u8 / Stage1Classifier.forward, which raise instead of falling back."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import input_pipeline_oracle as P
from sbl_for_multilingual_lip_reading_b200 import ops_train as ot, synth
from sbl_for_multilingual_lip_reading_b200.video_frontend import Lipreading, random_crop_offsets

HERE = os.path.dirname(os.path.abspath(__file__))


def test_random_crop_offsets_reproduce_the_reference_random_crop():
    """random.seed(5) + the helper + crop_at + pad_frames == train_crop_T31, which the reference's own
    cvtransforms.RandomCrop produced (tests/golden/input_pipeline.npz)."""
    g = np.load(os.path.join(HERE, "golden", "input_pipeline.npz"))
    u8 = synth.synthetic_u8_clips(1, 29, seed=21)[0].numpy()
    random.seed(5)
    offs = random_crop_offsets(1, 29)
    assert offs.dtype == torch.int32 and offs.shape == (29, 2)
    got = P.pad_frames(P.crop_at(P.load_and_normalize(u8), [tuple(o) for o in offs.tolist()]), 31)
    assert np.array_equal(got, g["train_crop_T31"])
    assert torch.equal(random_crop_offsets(1, 29, rng=random.Random(5)), offs)


def test_random_crop_offsets_ranges():
    offs = random_crop_offsets(5, 7, h0=100, w0=92, rng=random.Random(1))
    assert offs.shape == (35, 2)
    assert int(offs[:, 0].min()) >= 0 and int(offs[:, 0].max()) <= 12
    assert int(offs[:, 1].min()) >= 0 and int(offs[:, 1].max()) <= 4
    assert int(offs[:, 0].max()) > 4                  # y really spans the taller frame
    assert torch.equal(random_crop_offsets(2, 3, 88, 88), torch.zeros((6, 2), dtype=torch.int32))
    with pytest.raises(ValueError):
        random_crop_offsets(1, 1, h0=80)


def test_forward_u8_rejects_cpu_and_wrong_dtypes():
    from sbl_for_multilingual_lip_reading_b200.stage1 import Stage1Classifier
    fe = Lipreading().train()
    u8 = synth.synthetic_u8_clips(2, 5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fe.forward_u8(u8, frames=6)
    with pytest.raises(RuntimeError, match="uint8"):
        fe.forward_u8(u8.float(), frames=6)
    with pytest.raises(RuntimeError, match="uint8"):
        fe.forward_u8(u8[0], frames=6)
    fe.eval()
    with pytest.raises(RuntimeError, match="flip"):
        fe.forward_u8(u8, flip=torch.tensor([True, False]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fe.forward_u8(u8, frames=6)
    model = Stage1Classifier(n_layers_enc=1).train()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(u8=u8, frames=6)
    with pytest.raises(RuntimeError, match="uint8"):
        model(u8=u8.to(torch.int16), frames=6)


def test_stage1_forward_takes_exactly_one_input():
    from sbl_for_multilingual_lip_reading_b200.stage1 import Stage1Classifier
    model = Stage1Classifier(n_layers_enc=1).train()
    u8 = synth.synthetic_u8_clips(1, 3)
    x = torch.zeros((1, 3, 88, 88))
    with pytest.raises(RuntimeError, match="exactly one"):
        model(x, u8=u8)
    with pytest.raises(RuntimeError, match="exactly one"):
        model()
    with pytest.raises(RuntimeError, match="u8 input only"):
        model(x, frames=3)
    with pytest.raises(RuntimeError, match="u8 input only"):
        model(x, flip=torch.tensor([True]))


def test_host_offsets_and_flags_are_checked_before_upload():
    with pytest.raises(RuntimeError, match="leaves the 96x96 frame"):
        ot.crop_offsets_to(torch.tensor([[0, 0], [9, 0]], dtype=torch.int32), 2, 96, 96, "cpu")
    with pytest.raises(RuntimeError, match="leaves the 100x92 frame"):
        ot.crop_offsets_to(torch.tensor([[12, 5]], dtype=torch.int32), 1, 100, 92, "cpu")
    with pytest.raises(RuntimeError, match="int32"):
        ot.crop_offsets_to(torch.zeros((2, 2), dtype=torch.int64), 2, 96, 96, "cpu")
    with pytest.raises(RuntimeError, match=r"int32 \[3, 2\]"):
        ot.crop_offsets_to(torch.zeros((2, 2), dtype=torch.int32), 3, 96, 96, "cpu")
    ok = ot.crop_offsets_to(torch.tensor([[12, 4]], dtype=torch.int32), 1, 100, 92, "cpu")
    assert ok.tolist() == [[12, 4]]
    with pytest.raises(RuntimeError, match="flip"):
        ot.flip_flags_to(torch.ones(2), 2, "cpu")
    with pytest.raises(RuntimeError, match="flip"):
        ot.flip_flags_to([True, False], 2, "cpu")
    with pytest.raises(RuntimeError, match="flip"):
        ot.flip_flags_to(torch.ones(3, dtype=torch.bool), 2, "cpu")
    assert ot.flip_flags_to(torch.tensor([True, False]), 2, "cpu").tolist() == [1, 0]
