#!/usr/bin/env python
"""Where does the one-batch-per-replay frontend spend its time?  Graph replays (PDL on, cold L2) of the frontend cut
after the stem / after k residual blocks, with and without the L2 weight prefetch; differences = in-graph cost per block."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from sbl_for_multilingual_lip_reading_b200 import ops, synth
from sbl_for_multilingual_lip_reading_b200.video_frontend import visual_frontend
dev = torch.device("cuda"); ops.init()
N, T = 32, 29
fe = visual_frontend(None); fe.load_state_dict(synth.frontend_state_dict(1)); fe = fe.to(dev).eval()
fe.always_on_dropout = False
x = synth.synthetic_clips(N, T, seed=7).to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

def graph_time(fn, reps=16):
    s = torch.cuda.Stream()
    with torch.no_grad(), torch.cuda.stream(s):
        fn(); fn()
        s.synchronize()
        gr = torch.cuda.CUDAGraph()
        old = ops.set_pdl(True)
        with torch.cuda.graph(gr, stream=s):
            fn()
        ops.set_pdl(old)
        ts = []
        for i in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s); gr.replay(); e1.record(s)
            s.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
    ts = sorted(ts[2:])
    return ts[len(ts) // 2]

pk = fe._get_packed()
full = list(pk.blocks)
feat = torch.empty(N * T, 512, device=dev)
names = ["stem only", "+layer1.0", "+layer1.1", "+layer2.0", "+layer2.1", "+layer3.0", "+layer3.1", "+layer4.0", "+layer4.1"]
for pf in (True, False):
    fe.l2_prefetch = pf
    prev = 0.0
    for k in range(0, 9):
        pk.blocks = full[:k]
        def run():
            xp = ops.raw_clip(x)
            a = ops.conv3d_bn_relu_pool(xp, pk.c3w, pk.c3b, flat=True)
            for bi, (stride, w1, b1, w2, b2, ds) in enumerate(pk.blocks):
                if isinstance(a, ops.FlatActs) and stride == 1 and ds is None:
                    y = ops.conv3x3_flat(a, w1, b1, relu=True)
                    a = ops.conv3x3_flat(y, w2, b2, relu=True, residual=a)
                elif ds is not None and w2.dim() == 2:
                    y, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=stride, relu=True,
                                             flat_ws=fe._flat_workspace(a, w1.shape[0], stride))
                    a = ops.conv3x3_flat(y, w2, b2, relu=True, residual=res)
                elif ds is not None:
                    y = ops.conv2d(a, w1, b1, stride=stride, relu=True)
                    a = ops.conv2d(y, w2, ds[2], stride=1, relu=True, ext=(a, ds[0], stride))
                else:
                    y = ops.conv2d(a, w1, b1, stride=stride, relu=True)
                    a = ops.conv2d(y, w2, b2, stride=1, relu=True, residual=a)
            return a
        t = graph_time(run)
        print(f"l2_prefetch={pf} (not used in this hand-rolled chain) {names[k]:12s}: {t:7.1f} us  (+{t - prev:.1f})", flush=True)
        prev = t
    pk.blocks = full
    t = graph_time(lambda: fe._frontend_forward(x))
    print(f"l2_prefetch={pf}: whole frontend through the module (stem .. avgpool): {t:.1f} us", flush=True)
    if not pf:
        break
