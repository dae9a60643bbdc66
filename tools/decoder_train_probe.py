"""Time the SBL decoder's training forward + backward on libsblk against the same computation in fp32 torch autograd.

    python tools/decoder_train_probe.py [--batches 16,64,240] [--t 30] [--layers 6] [--p 0.1] [--rounds 3] [--iters 3]
                                        [--out FILE]

libsblk arm: Decoder in model.train() (training.decoder_forward_train), loss = sum(logits * G), backward.  fp32 arm: the
float64 restatement of the training step (tests/decoder_dropout_oracle.step_logits) run in fp32 with TF32 off under torch
autograd, with dropout factors drawn in the same order and shapes: it stands in for the reference decoder, whose sources
this repository does not carry.  Both arms feed the gold tokens (coin forced), use the same weights and encoder outputs.  Each round times
`iters` calls of each arm with CUDA events (after one warm-up call per arm and batch), the arms alternating; the probe
prints the median and the min-max over rounds of the per-call time, the libsblk launches per call, the peak
allocated memory of one call of each arm, and the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import decoder_dropout_oracle as DO  # noqa: E402
from sbl_for_multilingual_lip_reading_b200 import ops  # noqa: E402
from sbl_for_multilingual_lip_reading_b200.decoder import Decoder  # noqa: E402

VOCAB = 58


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def _oracle_drops(n, t, n_layers, p, dev):
    def f(shape):
        return F.dropout(torch.ones(shape, device=dev), p=p, training=True) if p > 0 else None
    steps = []
    for i in range(16):
        L = i + 1
        st = {d: {"emb": f((n * L, 512)), "layers": []} for d in ("l2r", "r2l")}
        for _ in range(n_layers):
            for d in ("l2r", "r2l"):
                st[d]["layers"].append((f((8 * n, L, L)), f((n * L, 512)), f((8 * n, L, t)), f((n * L, 512)),
                                        f((n * L, 512))))
        steps.append(st)
    return steps


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="16,64,240")
    ap.add_argument("--t", type=int, default=30)
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--p", type=float, default=0.1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("decoder_train_probe: no CUDA device (the probe measures on the GPU only)")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    ops.init()
    name, power = _card()
    random.random = lambda: 0.0                                       # the coin always feeds the gold token
    torch.manual_seed(7)
    dec = Decoder(0, 1, VOCAB, 512, a.layers, 8, 64, 64, 512, 2048, dropout=a.p).to(dev).train()
    sd = {k: v.detach().clone().requires_grad_(k != "positional_encoding.pe") for k, v in dec.state_dict().items()}
    lines = [f"card: {name}, power limit {power}; decoder {a.layers} layers, t_enc = {a.t}, dropout p = {a.p}; "
             f"forward + backward per call, {a.iters} calls per round, {a.rounds} alternating rounds"]
    results = []
    for n in [int(b) for b in a.batches.split(",")]:
        g = torch.Generator(device=dev).manual_seed(n)
        enc = torch.randn(n, a.t, 512, generator=g, device=dev)
        tgt = torch.randint(2, VOCAB, (n, 12), device=dev)
        tgt_r = tgt.flip(1)
        G = (torch.randn(n, 16, VOCAB, generator=g, device=dev), torch.randn(n, 16, VOCAB, generator=g, device=dev))
        ys = [torch.cat([y, torch.ones((n, 1), dtype=torch.long, device=dev)], 1)
              for y in (dec.preprocess(tgt)[0], dec.preprocess(tgt_r)[0])]

        def ours():
            e = enc.clone().requires_grad_()
            la, _, lb, _ = dec(tgt, tgt_r, e, [a.t] * n)
            ((la * G[0]).sum() + (lb * G[1]).sum()).backward()

        def fp32():
            e = enc.clone().requires_grad_()
            drops = _oracle_drops(n, a.t, a.layers, a.p, dev)
            steps = [DO.step_logits(sd, ys[0], ys[1], e, L, drops[L - 1]) for L in range(1, 17)]
            la, lb = torch.stack([s[0] for s in steps], 1), torch.stack([s[1] for s in steps], 1)
            ((la * G[0]).sum() + (lb * G[1]).sum()).backward()

        arms = {"libsblk": ours, "fp32_torch": fp32}
        peak, times = {}, {k: [] for k in arms}
        for k, fn in arms.items():                                    # warm-up + peak memory of one call
            fn()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            before = ops.launch_count()
            fn()
            torch.cuda.synchronize()
            peak[k] = torch.cuda.max_memory_allocated() - base
            if k == "libsblk":
                launches = ops.launch_count() - before
        for _ in range(a.rounds):
            for k, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _i in range(a.iters):
                    fn()
                e1.record()
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.iters)
        dec.zero_grad(set_to_none=True)
        for v in sd.values():
            v.grad = None
        r = {"batch": n, "launches_per_call": launches,
             **{f"{k}_ms": {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in times.items()},
             **{f"{k}_peak_alloc_GB": peak[k] / 1e9 for k in arms}}
        r["speedup"] = r["fp32_torch_ms"]["median"] / r["libsblk_ms"]["median"]
        results.append(r)
        lines.append(f"batch {n:4d}: libsblk {r['libsblk_ms']['median']:9.2f} ms ({r['libsblk_ms']['min']:.2f}-"
                     f"{r['libsblk_ms']['max']:.2f})  fp32 torch {r['fp32_torch_ms']['median']:9.2f} ms "
                     f"({r['fp32_torch_ms']['min']:.2f}-{r['fp32_torch_ms']['max']:.2f})  x{r['speedup']:.2f}  "
                     f"launches/call {launches}  peak alloc libsblk {r['libsblk_peak_alloc_GB']:.2f} GB, fp32 torch "
                     f"{r['fp32_torch_peak_alloc_GB']:.2f} GB")
        print(lines[-1], flush=True)
    lines.append(json.dumps({"card": name, "power_limit": power, "results": results}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    print(lines[0])


if __name__ == "__main__":
    main()
