"""Stage-1 pre-training model (BASELINE configs[3]): visual frontend + transformer encoder + word / language heads.

Mirror of `VSR_visual_frontend_pretraining_on_LRW_LRW1000_classify/transformer/transformer.py:6-38` with the reference's
attribute names (`visual_frontend`, `encoder_v`, `fc_1500`, `fc_2`), so its state dict is key-for-key the reference's.
The reference forward cannot run as written — `torch.mean(out, dim=2, keepdim=True)` (:31) hands `fc_1500` a width-1
tensor — so the heads are applied as the file's evident intent (and its commented-out line :30) state: word logits from
the time-pooled encoder output, language logits from frame 30 (SURVEY.md §0, §8f.2).  The two heads are plain
`nn.Linear` on [N,512] vectors (outside the hot path, as in the reference); everything below them runs libsblk, in
`model.train()` through `training.py` (batch-statistics BatchNorm, dropout, backward).

Data-parallel training is one process per GPU under `torch.nn.parallel.DistributedDataParallel`: the backward is a chain
of per-block autograd Functions, so DDP's bucketed NCCL all-reduce of finished gradients overlaps the rest of the
backward; BatchNorm statistics stay per replica like the reference's `nn.DataParallel` (train.py:82).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import synth
from .encoder import Encoder
from .video_frontend import visual_frontend


class Stage1Classifier(nn.Module):
    def __init__(self, n_layers_enc=3, n_head=8, d_k=64, d_v=64, d_model=512, d_inner=2048, dropout=0.1, pe_maxlen=5000,
                 pt=None):
        super().__init__()
        self.visual_frontend = visual_frontend(pt)
        self.encoder_v = Encoder(512, n_layers_enc, n_head, d_k, d_v, d_model, d_inner, dropout=dropout,
                                 pe_maxlen=pe_maxlen)
        self.fc_1500 = nn.Linear(512, 1500)
        self.fc_2 = nn.Linear(512, 2)

    def load_synthetic(self, frontend_seed=1, encoder_seed=3):
        self.visual_frontend.load_state_dict(synth.frontend_state_dict(frontend_seed))
        self.encoder_v.load_state_dict(synth.encoder_state_dict(encoder_seed, len(self.encoder_v.layer_stack)))
        return self

    def forward(self, padded_input_visual=None, *, u8=None, frames=None, crop=None, flip=None):
        """padded_input_visual: [N,T,88,88] (as train.py:112-116 feeds it) or [N,1,T,88,88] -> (word logits [N,1500],
        language logits [N,2]).  Or, instead of it, `u8`: the loader's raw uint8 gray frames [N,T_in,H0,W0], cropped at
        `crop` (default the centre of 96x96 frames; per-frame offsets from video_frontend.random_crop_offsets),
        mirrored where `flip` [N] is set (model.train() only) and zero-padded to `frames` frames, all on the GPU
        (Lipreading.forward_u8).  The uint8 input goes through forward so that DistributedDataParallel, which prepares
        its gradient all-reduce inside forward, sees the step."""
        if (padded_input_visual is None) == (u8 is None):
            raise RuntimeError("Stage1Classifier.forward: pass exactly one of padded_input_visual and u8")
        if u8 is not None:
            feat = self.visual_frontend.forward_u8(u8, frames=frames, crop=(4, 4) if crop is None else crop, flip=flip)
        else:
            if frames is not None or crop is not None or flip is not None:
                raise RuntimeError("Stage1Classifier.forward: frames / crop / flip apply to the u8 input only")
            x = padded_input_visual
            if x.dim() == 4:
                x = x.view(x.size(0), -1, x.size(1), x.size(2), x.size(3))          # transformer.py:23
            feat = self.visual_frontend(x)
        n, t = feat.size(0), feat.size(1)
        out, *_ = self.encoder_v(feat, [t] * n)
        pooled = torch.mean(out, dim=1)
        lang = out[:, min(30, t - 1), :]
        return self.fc_1500(pooled), self.fc_2(lang)
