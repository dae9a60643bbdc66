#!/usr/bin/env python
"""Graph-replay timing of the two halves of the hot path (frontend / encoder) at BASELINE configs[1] shape."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sbl_for_multilingual_lip_reading_b200 import ops, synth
from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
from sbl_for_multilingual_lip_reading_b200.video_frontend import visual_frontend

dev = torch.device("cuda")
ops.init()
ops.set_pdl(os.environ.get("NO_PDL") is None)
N, T = int(os.environ.get("N", 32)), int(os.environ.get("T", 29))
fe = visual_frontend(None); fe.load_state_dict(synth.frontend_state_dict(1))
enc = Encoder(512, 6, 8, 64, 64, 512, 2048); enc.load_state_dict(synth.encoder_state_dict(2, 6))
fe, enc = fe.to(dev).eval(), enc.to(dev).eval()
x = synth.synthetic_clips(N, T, seed=7).to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def graph_time(fn, reps=30):
    s = torch.cuda.Stream()
    with torch.no_grad(), torch.cuda.stream(s):
        for _ in range(3):
            fn()
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g, stream=s):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2] * 1e3


with torch.no_grad():
    feat = fe(x)
fe.l2_prefetch = False
print(f"frontend (prep+stem+trunk+pool+dropout): {graph_time(lambda: fe(x)):.1f} us")
for cl, mc in (("16", "1"), ("8", "1")):
    os.environ["SBLK_ENC_STACK_CL"], os.environ["SBLK_ENC_STACK_MC"] = cl, mc
    enc.fused_stack = True
    print(f"encoder  (6 layers), one launch, cluster {cl} multicast {mc}: {graph_time(lambda: enc(feat, [T] * N)):.1f} us")
os.environ.pop("SBLK_ENC_STACK_CL"); os.environ.pop("SBLK_ENC_STACK_MC")
for sc in (False, True, False, True):
    enc.split_clusters = sc
    print(f"encoder  (6 layers), one launch, split clusters {sc}: {graph_time(lambda: enc(feat, [T] * N)):.1f} us")
for pf in (False, True, False, True, False, True):
    fe.l2_prefetch = pf
    print(f"whole path (one-launch encoder), L2 weight prefetch {pf}: {graph_time(lambda: enc(fe(x), [T] * N)):.1f} us")
enc.fused_stack = False
for pc in [int(v) for v in os.environ.get("CHAINS", "4").split(",")]:
    enc.parallel_chains = pc
    print(f"encoder  (6 layers), {pc} chains:           {graph_time(lambda: enc(feat, [T] * N)):.1f} us")
print(f"whole path:                              {graph_time(lambda: enc(fe(x), [T] * N)):.1f} us")
