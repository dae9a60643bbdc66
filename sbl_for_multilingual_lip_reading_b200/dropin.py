"""Make the reference's own scripts run on the B200-native encoder without editing them.

The reference has no plugin ABI: `train.py` / `test.py` import `transformer.encoder.Encoder` and
`transformer.transformer.Transformer`, and `Transformer.__init__` calls `visual_frontend(pt)`
(SBL_Multilingual_Lip_reading/train.py:58-69, transformer/transformer.py:3,11).  `patch_reference` puts the
reference directory on sys.path, imports those modules and rebinds the class / factory names to the drop-ins,
so everything constructed afterwards (by the unmodified scripts) uses libsblk for the visual-encoder path
while the SBL bidirectional decoder, loss, optimizer and data code stay the reference's.

    python -m sbl_for_multilingual_lip_reading_b200.dropin /path/to/SBL_Multilingual_Lip_reading/test.py [args]
"""
from __future__ import annotations

import contextlib
import importlib
import runpy
import sys

from . import decoder as _dec
from . import encoder as _enc
from . import video_frontend as _vf

_PATCHED = {
    "transformer.video_frontend": {
        "Lipreading": _vf.Lipreading, "ResNet": _vf.ResNet, "BasicBlock": _vf.BasicBlock,
        "conv3x3": _vf.conv3x3, "visual_frontend": _vf.visual_frontend,
    },
    "transformer.encoder": {"Encoder": _enc.Encoder, "EncoderLayer": _enc.EncoderLayer},
    # transformer.py does `from .video_frontend import visual_frontend` -> rebind its own global too
    "transformer.transformer": {"visual_frontend": _vf.visual_frontend},
}


# opt-in: the SBL bidirectional decoder on libsblk (decoder.py): greedy decode and teacher-forced forward, and in
# model.train() the training forward + backward, so train.py runs on it too
_PATCHED_DECODER = {"transformer.decoder": {"Decoder": _dec.Decoder, "DecoderLayer": _dec.DecoderLayer}}


def patch_reference(ref_dir, decoder=False):
    """Rebind the hot-path names inside the reference package found at `ref_dir` (decoder=True: the SBL decoder too,
    for evaluation and for `train.py`'s training steps).
    Returns ({module name: module}, {(<module>, <attr>): original}) so the patch can be undone."""
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    mods, saved = {}, {}
    table = dict(_PATCHED)
    if decoder:
        table.update(_PATCHED_DECODER)
    for mod_name, names in table.items():
        mod = importlib.import_module(mod_name)
        mods[mod_name] = mod
        for attr, repl in names.items():
            saved[(mod_name, attr)] = getattr(mod, attr, None)
            setattr(mod, attr, repl)
    return mods, saved


def unpatch_reference(ref_dir, saved):
    for (mod_name, attr), orig in saved.items():
        mod = sys.modules.get(mod_name)
        if mod is not None and orig is not None:
            setattr(mod, attr, orig)
    if ref_dir in sys.path:
        sys.path.remove(ref_dir)


@contextlib.contextmanager
def patched_reference(ref_dir, decoder=False):
    mods, saved = patch_reference(ref_dir, decoder=decoder)
    try:
        yield mods
    finally:
        unpatch_reference(ref_dir, saved)


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        raise SystemExit("usage: python -m sbl_for_multilingual_lip_reading_b200.dropin <reference script.py> [args...]")
    script = argv[0]
    import os
    ref_dir = os.path.dirname(os.path.abspath(script))
    patch_reference(ref_dir)
    sys.argv = argv
    runpy.run_path(script, run_name="__main__")


if __name__ == "__main__":
    main()
