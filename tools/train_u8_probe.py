"""Measures the uint8 training input (ops_train.stem_im2col_u8, Stage1Classifier.forward(u8=...)) against the fp32 clip
input at the BASELINE configs[3] shape (256 clips x 29 loader frames padded to 31, one GPU).  One command:

    python tools/train_u8_probe.py [--out DIR]

1. kernel time of stem_im2col_u8 against stem_im2col, both orientations: CUDA events over many launches after a
   warm-up, alternated in rounds; bytes from shapes (input read once + the bf16 im2col written once);
2. device-timed stage-1 step (the bench.py config3 model, Adam, loss) fed from device-resident fp32 clips against
   device-resident uint8 frames with per-frame crops and flips, alternated in rounds;
3. end to end from pinned host memory, alternated three times each: (a) the loader's host work (float64 normalise, crop,
   mirror, float32 frame padding, as oracle/input_pipeline_oracle.py) + the fp32 copy + the step, against (b) the
   uint8 copy + the step.  Copies are cudaMemcpyAsync from pinned memory on a copy stream, one batch ahead of the step.
   The host work runs in this process's main thread while the GPU runs the previous step.
Prints the GPU name and power limit first; writes the log to DIR/train_u8_probe.log when --out is given.
"""
import argparse
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

LINES = []


def say(*a):
    s = " ".join(str(x) for x in a)
    print(s, flush=True)
    LINES.append(s)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"


def spread(v):
    return f"median {statistics.median(v):.3f} (min {min(v):.3f}, max {max(v):.3f}, n={len(v)})"


def host_clips(u8, offs, flips, t_out, out):
    """The reference loader's fp32 clips, written into `out` [N, t_out, 88, 88] (numpy view of pinned memory)."""
    from oracle import input_pipeline_oracle as P
    n, t_in = u8.shape[:2]
    for i in range(n):
        v = P.crop_at(P.load_and_normalize(u8[i]), offs[i * t_in:(i + 1) * t_in])
        if flips[i]:
            v = v[:, :, ::-1]
        out[i] = P.pad_frames(v, t_out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--kernel-iters", type=int, default=30)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_u8_probe: needs a CUDA device (no CPU timing is reported)")
    from sbl_for_multilingual_lip_reading_b200 import ops, ops_train as ot, stage1, synth
    from sbl_for_multilingual_lip_reading_b200.video_frontend import random_crop_offsets
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    say("card (name, power limit, max SM clock):", card())
    ops.init()
    n, t_in, t = args.clips, 29, 31
    u8_host = synth.synthetic_u8_clips(n, t_in, seed=40)
    offs = random_crop_offsets(n, t_in, rng=random.Random(40))
    flips = torch.tensor([i % 2 == 0 for i in range(n)])
    clip_host = np.empty((n, t, 88, 88), dtype=np.float32)
    t0 = time.perf_counter()
    host_clips(u8_host.numpy(), offs.tolist(), flips.tolist(), t, clip_host)
    say(f"host loader work for one batch of {n} clips (numpy, one thread): {1e3 * (time.perf_counter() - t0):.1f} ms")
    u8 = u8_host.to(dev)
    clip = torch.from_numpy(clip_host).to(dev)
    crop_d, flip_d = offs.to(dev), flips.to(dev)
    lut = synth.normalize_lut().to(dev)

    # ---- 1. kernels
    m = n * t * 44 * 44
    out_bytes = 2 * m * 256
    kern = {
        ("fp32", 0): lambda: ot.stem_im2col(clip),
        ("u8", 0): lambda: ot.stem_im2col_u8(u8, lut, t, crop_d, flip_d),
        ("fp32", 1): lambda: ot.stem_im2col(clip, transposed=True, ld_out=m),
        ("u8", 1): lambda: ot.stem_im2col_u8(u8, lut, t, crop_d, flip_d, transposed=True, ld_out=m),
    }
    in_bytes = {"fp32": clip.numel() * 4, "u8": u8.numel() + crop_d.numel() * 4 + flip_d.numel() * 4}
    for tr in (0, 1):
        a = kern[("fp32", tr)]()
        b = kern[("u8", tr)]()
        assert torch.equal(a, b), "uint8 and fp32 im2col differ"
        del a, b
    say(f"\n1. stem im2col, N={n} T_in={t_in} T_out={t} (M={m}); output {out_bytes / 1e9:.3f} GB, input fp32 "
        f"{in_bytes['fp32'] / 1e6:.1f} MB / uint8 {in_bytes['u8'] / 1e6:.1f} MB")
    times = {k: [] for k in kern}
    out = None
    for k, fn in kern.items():                       # warm-up
        for _ in range(3):
            out = fn()
    del out
    for _ in range(3):                               # rounds, alternating
        for k, fn in kern.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.kernel_iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / args.kernel_iters)
    for tr in (0, 1):
        for src in ("fp32", "u8"):
            v = times[(src, tr)]
            gbs = [(in_bytes[src] + out_bytes) / (ms * 1e-3) / 1e9 for ms in v]
            say(f"  {'transposed' if tr else 'row-major '} {src:4s}: ms/launch {spread(v)}; GB/s {spread(gbs)}")
    # (each timed launch also allocates its output with torch's caching allocator, identically for both kernels)

    # ---- 2. device-timed step
    torch.manual_seed(7)
    model = stage1.Stage1Classifier(n_layers_enc=3, dropout=0.1).load_synthetic(1, 3).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
    y = torch.randint(0, 1500, (n,), generator=torch.Generator().manual_seed(0)).to(dev)
    lang = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(100)).to(dev)

    def step(inp):
        v_t, v_l = model(**inp)
        loss = F.cross_entropy(v_t, y) + 0.1 * F.cross_entropy(v_l, lang)
        opt.zero_grad()
        loss.backward()
        opt.step()

    feeds = {"fp32": lambda c=None: dict(padded_input_visual=clip if c is None else c),
             "u8": lambda c=None: dict(u8=u8 if c is None else c, frames=t, crop=crop_d, flip=flip_d)}
    for name in feeds:
        for _ in range(2):
            step(feeds[name]())
    torch.cuda.synchronize()
    say(f"\n2. stage-1 step (config3 model, Adam), device-resident input, {args.steps} steps per round")
    st = {k: [] for k in feeds}
    for _ in range(3):
        for name in feeds:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(feeds[name]())
            e1.record()
            torch.cuda.synchronize()
            st[name].append(e0.elapsed_time(e1) / args.steps)
    for name in feeds:
        say(f"  {name:4s}: ms/step {spread(st[name])}; clips/s {spread([n / (v * 1e-3) for v in st[name]])}")

    # ---- 3. end to end from pinned host memory
    copy = torch.cuda.Stream()
    comp = torch.cuda.current_stream()
    pin = {"fp32": [torch.empty((n, t, 88, 88), dtype=torch.float32).pin_memory() for _ in range(2)],
           "u8": [u8_host.clone().pin_memory() for _ in range(2)]}
    devbuf = {"fp32": [torch.empty((n, t, 88, 88), dtype=torch.float32, device=dev) for _ in range(2)],
              "u8": [torch.empty_like(u8) for _ in range(2)]}
    u8_np = u8_host.numpy()

    def run_e2e(name, steps):
        """Batch i+1 is prepared on the host and copied on `copy` while step i runs on `comp`."""
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [None, None]

        def stage(i):
            s = i % 2
            if consumed[s] is not None:
                consumed[s].synchronize()              # the step that read this slot has finished with it
            if name == "fp32":
                host_clips(u8_np, offs.tolist(), flips.tolist(), t, pin["fp32"][s].numpy())
            with torch.cuda.stream(copy):
                devbuf[name][s].copy_(pin[name][s], non_blocking=True)
                copied[s].record(copy)

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stage(0)
        for i in range(steps):
            comp.wait_event(copied[i % 2])
            step(feeds[name](devbuf[name][i % 2]))
            ev = torch.cuda.Event()
            ev.record(comp)
            consumed[i % 2] = ev
            if i + 1 < steps:
                stage(i + 1)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps

    for name in feeds:
        run_e2e(name, 2)
    say(f"\n3. end to end from pinned host memory, {args.e2e_steps} steps per run, (a) fp32 = host loader work + "
        f"{4 * n * t * 88 * 88 / 1e6:.1f} MB copy, (b) u8 = {n * t_in * 96 * 96 / 1e6:.1f} MB copy")
    e2e = {k: [] for k in feeds}
    for _ in range(3):
        for name in feeds:
            e2e[name].append(run_e2e(name, args.e2e_steps))
    for name in feeds:
        say(f"  {name:4s}: ms/step {spread(e2e[name])}; clips/s {spread([n / (v * 1e-3) for v in e2e[name]])}")
    say("card (name, power limit, max SM clock):", card())
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "train_u8_probe.log"), "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
