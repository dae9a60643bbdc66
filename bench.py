#!/usr/bin/env python
"""bench.py — visual-encoder clips/sec on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's sm_100a path (libsblk)
  python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference modules (oracle/_ref) on the host CPU
  torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU, clip batch sharded (weak scaling)

A step = one forward of the hot path (Conv3d frontend -> ResNet-18 trunk -> 6-layer transformer Encoder,
always-on dropout included, exactly what `Transformer.forward` runs before the decoder,
SBL_Multilingual_Lip_reading/transformer/transformer.py:34-38) over one synthetic LRW-shaped batch
(BASELINE.json configs[1]: 32 clips x 29 frames x 88 x 88 per GPU).

  value   device-timed (CUDA events on the launching stream), inputs resident in HBM, L2 flushed between steps
  e2e     same metric through the host-facing call: pinned host fp32 clips in, H2D + forward + D2H of the encoder
          output every step (double-buffered), wall clock bracketed by synchronize
  roofline        dominant kernel: algorithmic FLOPs per launch / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline    the reference's own modules (oracle/_ref, staged by oracle/fetch_ref.py) on the host cores, same batch
  sustained / config2 / gather_verified / h2d_ceiling_gbs   see DESIGN.md §5 (also nested under roofline / config / e2e,
                  the keys the driver keeps whole)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "visual_encoder_clips_per_sec"
UNIT = "clips/s"
FALLBACK_PEAKS = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}


def flops_per_clip(t, layers):
    """SURVEY.md §8d / BASELINE.md §3: 2*MACs of Conv3d + 20 ResNet convs + linear_in + per-layer linears + bmm."""
    return t * (60712960 + 571604992 + 524288 + layers * 6291456) + layers * 2048 * t * t


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            if "bf16_tflops" in d and "hbm_gbs" in d:
                d["_source"] = "measured"
                return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    """Samples SM clock + throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference algorithm) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_setup(layers):
    """The reference's own visual frontend + Encoder (oracle/_ref: unmodified files of /root/reference staged by
    oracle/fetch_ref.py), fp32, eval mode, all host cores.  Falls back to the functional oracle port only if the staged
    files are missing (kind says which)."""
    import torch
    from sbl_for_multilingual_lip_reading_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    from oracle import ref_runtime
    if ref_runtime.available():
        R = ref_runtime.load_reference("sbl")
        torch.manual_seed(7)
        fe = R.Lipreading()
        fe.load_state_dict(synth.frontend_state_dict(1))
        enc = R.Encoder(512, layers, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        enc.load_state_dict(synth.encoder_state_dict(2, layers))
        fe, enc = fe.eval(), enc.eval()

        def step(x):
            # transformer/transformer.py:31-38 — frontend (always-on dropout included), input_lengths = [T]*N, encoder
            with torch.no_grad():
                feat = fe(x)
                out, *_ = enc(feat, [feat.size(1)] * feat.size(0))
            return out
        return step, cores, "reference"
    from oracle import visual_encoder_oracle as O
    sd = {}
    sd.update(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, layers, prefix="encoder."))

    def step(x):
        with torch.no_grad():
            gen = torch.Generator().manual_seed(0)
            n, t = x.shape[0], x.shape[2]
            mask = (torch.rand((n * t, 512), generator=gen) >= 0.5).float()  # always-on dropout(0.5)
            return O.visual_encoder_forward(x, sd, dropout_mask=mask)
    return step, cores, "port"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from sbl_for_multilingual_lip_reading_b200 import synth
    step, cores, kind = cpu_reference_setup(args.layers)
    sample = args.ref_clips if args.ref_clips > 0 else args.batch
    x = synth.synthetic_clips(sample, args.frames, seed=7)
    t0 = time.perf_counter()
    step(x)                                         # first warm-up step doubles as the cost probe
    probe = time.perf_counter() - t0
    if args.ref_clips <= 0 and probe * (args.steps + args.warmup) > 240.0:
        # keep the whole run within a few minutes on slow hosts: a bounded sample of the batch, stated in `sample`
        sample = max(1, int(sample * 240.0 / (probe * (args.steps + args.warmup))))
        x = x[:sample].contiguous()
    for _ in range(max(args.warmup - 1, 0)):
        step(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(x)
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    desc = (f"{sample} clips x {args.frames} frames per step" +
            ("" if sample == args.batch else f" (bounded sample of the {args.batch}-clip batch)") +
            (": unmodified reference Lipreading + Encoder modules from oracle/_ref" if kind == "reference"
             else ": oracle port (oracle/_ref not staged)") + ", fp32, eval mode")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(args, world):
    if (args.batch, args.frames) == (32, 29):
        name, shape = "BASELINE configs[1]", "LRW-shaped"
    elif (args.batch, args.frames) == (8, 40):
        name, shape = "BASELINE configs[2] (batch 64 sharded across 8 B200: 8 clips per GPU)", "LRW-1000-shaped"
    else:
        name, shape = "custom shape", "LRW-style"
    return {
        "workload": (f"{name}: full visual encoder forward (Conv3d frontend + ResNet-18 trunk + "
                     f"{args.layers}-layer transformer Encoder), {shape} {args.frames}x88x88 gray clips, "
                     f"batch {args.batch} per B200"),
        "clips_per_gpu": args.batch, "frames": args.frames, "encoder_layers": args.layers,
        "global_batch": args.batch * world, "parallelism": f"dp{world}",
        "l2": "L2 flushed (256 MiB write) between timed steps; e2e inputs stream from pinned host memory",
    }


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: run on (and first-touch the pinned host buffers from) the CPUs of the NUMA node the GPU hangs
    off, so the per-step host->device copy does not cross the socket interconnect.  Returns the node or None."""
    try:
        import torch
        props = torch.cuda.get_device_properties(local_rank)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


class Shape:
    """One (clips per GPU, frames) workload on this rank: plans, input pools, output gathering, device-timed loop."""

    def __init__(self, ctx, B, T, want_latency_plan=True):
        import torch
        from sbl_for_multilingual_lip_reading_b200 import sharding, synth
        from sbl_for_multilingual_lip_reading_b200.runner import PipelinedVisualEncoderPlan, VisualEncoderPlan
        self.ctx, self.B, self.T = ctx, B, T
        args, dev, fe, enc = ctx.args, ctx.dev, ctx.fe, ctx.enc
        self.pipelined, self.pipeline_note = False, "off (--no-pipeline)"
        self.plan = None
        if not args.no_pipeline:
            try:
                self.plan = PipelinedVisualEncoderPlan(fe, enc, B, T, device=dev, pdl=not args.no_pdl)
                self.pipelined = True
                self.pipeline_note = (
                    f"2-stage software pipeline: step i = encoder stack of batch i-1 (8-CTA clusters) next to clip prep + "
                    f"Conv3d stem of batch i on {self.plan.head_sm_limit} SMs, then the trunk of batch i at full width; "
                    f"value/e2e are steady-state throughput, `latency` is the unpipelined plan")
            except Exception as e:  # noqa: BLE001  (shape outside the plan's envelope: the one-batch plan is timed)
                self.pipeline_note = f"off ({e})"
        self.plan_lat = (VisualEncoderPlan(fe, enc, B, T, device=dev, slots=2, pdl=not args.no_pdl)
                         if (want_latency_plan or self.plan is None) else None)
        if self.plan is None:
            self.plan = self.plan_lat
        self.pool_n = 4
        self.host_pool = [synth.synthetic_clips(B, T, seed=100 + 17 * ctx.rank + i + 1000 * T).pin_memory()
                          for i in range(self.pool_n)]
        self.dev_pool = [h.to(dev) for h in self.host_pool]
        self.out_host = [torch.empty((B, T, 512), dtype=torch.float32).pin_memory() for _ in range(2)]
        self.gathered = (torch.empty((ctx.world * B, T, 512), dtype=torch.float32, device=dev)
                         if ctx.world > 1 else None)
        # output gathering: one-shot peer-memory kernel over NVLink (sharding.P2PGather) or, with --gather nccl, NCCL
        self.p2p, self.gather_mode = None, (args.gather if ctx.world > 1 else None)
        if ctx.world > 1 and args.gather == "p2p":
            import torch.distributed as dist
            err = None
            try:
                self.p2p = sharding.P2PGather(B * T * 512, dev)
            except Exception as e:  # noqa: BLE001  (e.g. CUDA IPC not permitted in this container)
                err = e
            ok = torch.tensor([0 if err else 1], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # the choice must be the same on every rank
            if int(ok.item()) == 0:
                self.p2p, self.gather_mode = None, f"nccl (peer-memory gather unavailable: {err})"
        self.gather_stream = torch.cuda.Stream(device=dev) if ctx.world > 1 else None
        self.pending = None
        self.defer = self.pipelined and ctx.world > 1 and not args.inline_gather
        self.last_out = None   # this rank's [B,T,512] output of the latest device_step

    def make_plan(self, **kw):
        from sbl_for_multilingual_lip_reading_b200.runner import PipelinedVisualEncoderPlan, VisualEncoderPlan
        a = self.ctx.args
        if self.pipelined:
            return PipelinedVisualEncoderPlan(self.ctx.fe, self.ctx.enc, self.B, self.T, device=self.ctx.dev,
                                              pdl=not a.no_pdl, **kw)
        return VisualEncoderPlan(self.ctx.fe, self.ctx.enc, self.B, self.T, device=self.ctx.dev, slots=2,
                                 pdl=not a.no_pdl, **kw)

    def gather_outputs(self, out):
        """output gathering (the DataParallel `gather` of the reference, train.py:115): one kernel that stores this
        rank's block into every peer's buffer over NVLink and waits for all peers' blocks; or NCCL.  Returns the
        gathered [world*B*T*512] fp32 view."""
        import torch.distributed as dist
        if os.environ.get("SBLK_BENCH_NO_GATHER"):   # diagnosis only (what the gather + its lock-step cost): the line says so
            return out.view(-1)
        if self.p2p is not None:
            return self.p2p(out.view(-1))
        if self.gathered is not None:
            dist.all_gather_into_tensor(self.gathered, out)
            return self.gathered.view(-1)
        return out.view(-1)

    def device_step(self, i, plan=None, defer=None, flush=True):
        """inputs already in HBM; L2 flushed before the timed part; returns (start, end) events.  With the pipelined plan
        the step's output is the previous batch's: one frontend pass + one encoder pass per step.  Multi-GPU: every step
        contains exactly one output gather inside its event pair — in stream after the replay, or (pipelined plan) the
        gather of the PREVIOUS step's output on a side stream next to this step's replay, so that a rank waiting for
        its peers' blocks keeps computing (the output buffer it reads is not written by this replay)."""
        import torch
        plan = self.plan if plan is None else plan
        defer = self.defer if defer is None else defer
        s = i % plan.slots
        with torch.cuda.stream(plan.compute):
            plan.x[s].copy_(self.dev_pool[i % self.pool_n])
            if flush:
                self.ctx.flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(plan.compute)
            gather_first = bool(os.environ.get("SBLK_BENCH_GATHER_FIRST"))   # diagnosis: the round-2 issue order
            if defer and self.pending is not None and gather_first:
                self.gather_stream.wait_event(e0)
                with torch.cuda.stream(self.gather_stream):
                    self.gather_outputs(self.pending)
            out = plan.forward_device(s)
            self.last_out = out
            if defer and self.pending is not None and not gather_first:
                # issued BEHIND the replay: the step's first kernels (encoder clusters, gated stem) get their SMs before
                # the gather's small CTAs look for room beside them
                self.gather_stream.wait_event(e0)
                with torch.cuda.stream(self.gather_stream):
                    self.gather_outputs(self.pending)
            if defer:
                plan.compute.wait_stream(self.gather_stream)
                self.pending = out
            else:
                self.gather_outputs(out)
            e1.record(plan.compute)
        return e0, e1

    def flush_pending_gather(self):
        """the last deferred gather (every rank issues the same number of gathers)"""
        import torch
        if self.pending is not None:
            with torch.cuda.stream(self.plan.compute):
                self.gather_outputs(self.pending)
            self.pending = None

    def time_device(self, steps, warmup, plan=None, defer=None, sampler=None):
        """-> ms per step (sum of the per-step event pairs, max over ranks)."""
        from sbl_for_multilingual_lip_reading_b200 import sharding
        for i in range(warmup):
            self.device_step(i, plan, defer)
        self.ctx.barrier()
        if sampler is not None:
            sampler.start()
        evs = [self.device_step(warmup + i, plan, defer) for i in range(steps)]
        self.ctx.barrier()
        if sampler is not None:
            sampler.stop()
        self.flush_pending_gather()
        self.ctx.barrier()
        return sharding.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), self.ctx.dev) / steps

    def verify_gather(self):
        if os.environ.get("SBLK_BENCH_NO_GATHER"):
            return "skipped: SBLK_BENCH_NO_GATHER diagnostic run (no output gathering in the timed region)"
        return self._verify_gather()

    def _verify_gather(self):
        """One untimed check that the gather the timed region uses delivers what NCCL's all-gather delivers."""
        import torch
        import torch.distributed as dist
        if self.ctx.world == 1:
            return None
        with torch.cuda.stream(self.plan.compute):
            out = self.plan.forward_device(0).clone()
            got = self.gather_outputs(out).clone()
            want = torch.empty((self.ctx.world * out.numel(),), dtype=torch.float32, device=self.ctx.dev)
            dist.all_gather_into_tensor(want, out.view(-1))
        self.plan.compute.synchronize()
        ok = torch.tensor([1 if torch.equal(got, want) else 0], dtype=torch.int32, device=self.ctx.dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(int(ok.item()))


class Ctx:
    pass


DUMP_BUDGET_BYTES = 64 << 20


def dump_output(out_dir, name, t, seed=0):
    """--dump-outputs: write `t` as <out_dir>/<name>.npy in float32.  Above the 64 MiB budget it is cut to a fixed, seeded
    sample of its rows along dim 0 (sorted indices, the same for the same shape)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    t = t.detach().float()
    row_bytes = t[0].numel() * 4
    if t.numel() * 4 > DUMP_BUDGET_BYTES:
        keep = max(1, DUMP_BUDGET_BYTES // row_bytes)
        idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(seed))[:keep].sort().values
        t = t[idx.to(t.device)]
    np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner ignores
    # NCCL_DEBUG_FILE) is sent to stderr by pointing fd 1 at fd 2 for the whole run; the line goes to the saved fd
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout; stdout carries exactly ONE JSON line, so NCCL's log goes to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/sblk_bench_nccl_%h_%p.log")
        dist.init_process_group("nccl", device_id=dev)

    from sbl_for_multilingual_lip_reading_b200 import ops, sharding, synth
    from sbl_for_multilingual_lip_reading_b200.encoder import Encoder
    from sbl_for_multilingual_lip_reading_b200.video_frontend import visual_frontend

    ops.init()
    B, T, L = args.batch, args.frames, args.layers
    fe = visual_frontend(None)
    fe.load_state_dict(synth.frontend_state_dict(1))
    enc = Encoder(512, L, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
    enc.load_state_dict(synth.encoder_state_dict(2, L))
    fe, enc = fe.to(dev).eval(), enc.to(dev).eval()
    torch.manual_seed(1234 + rank)

    ctx = Ctx()
    ctx.args, ctx.dev, ctx.fe, ctx.enc, ctx.world, ctx.rank = args, dev, fe, enc, world, rank
    ctx.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    ctx.barrier = barrier

    peaks = load_peaks()
    fpc = flops_per_clip(T, L)
    main = Shape(ctx, B, T)
    plan, pipelined = main.plan, main.pipelined
    sampler = ClockSampler(local_rank)

    # ---- device-timed run (the metric) -----------------------------------------------------
    dev_ms = main.time_device(args.steps, args.warmup, sampler=sampler)
    value = world * B / (dev_ms * 1e-3)
    if args.dump_outputs:
        out = main.last_out
        if world > 1:   # what the caller receives: every rank's block, gathered in rank order
            full = torch.empty((world * B, T, 512), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(full, out.contiguous())
            out = full
        if rank == 0:
            dump_output(args.dump_outputs, "encoder_output", out)

    # ---- end-to-end run (host buffers, H2D + D2H inside the timed region).  Measured right after the device-timed run:
    # both are K-step bursts on a GPU that has not yet been driven into its power cap by the seconds-long `sustained`
    # run below (tools/exp/e2e_probe.py: the same loop takes 0.657 ms/step on a cool GPU and 0.72 after ~100 ms of
    # back-to-back load — the graph replays themselves slow down, the 0.54 ms input copy stays hidden) ---------------
    def e2e_run(pl, pool, k):
        for i in range(k):
            pl.submit_host(pool[i % main.pool_n], main.out_host[i % 2])
        if pipelined:   # k inputs in, the k outputs OF THOSE inputs out: the last batch's encoder runs here
            pl.drain(main.out_host[k % 2])
        pl.synchronize()

    def e2e_time(pl, pool, smp=None):
        e2e_run(pl, pool, max(args.warmup, 3))
        barrier()
        if smp is not None:
            smp.start()
        t0 = time.perf_counter()
        e2e_run(pl, pool, args.steps)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if smp is not None:
            smp.stop()
        return sharding.max_over_ranks(dt, dev)

    def cool_down():
        # every burst leg (device-timed, e2e, e2e_u8, latency) starts from an idle GPU: ~100 ms of back-to-back load is
        # enough to pull this box into its power cap (the regime the `sustained` key reports), and a leg that merely
        # runs later in the script would otherwise be measured in a different clock regime than the one before it
        barrier()
        time.sleep(args.cool_down_seconds)
        barrier()

    cool_down()
    e2e_s = e2e_time(plan, main.host_pool, sampler)
    e2e_value = world * B * args.steps / e2e_s
    checksum = float(main.out_host[(args.steps - 1) % 2].double().abs().mean())  # the D2H result is really read

    # ---- end-to-end through the fused uint8 input pipeline (SURVEY.md 8f.3, an ADDITIONAL key: `e2e` above keeps the
    # reference's fp32 model boundary): the host ships the loader's raw uint8 frames [B, T, 96, 96] (9.2 KB/frame
    # instead of 31 KB) and /255, ColorNormalize, centre crop are done by the clip-prep kernel ----------------------
    e2e_u8 = None
    if not args.no_u8:
        plan8 = main.make_plan(u8_input=(T, 96, 96))
        host_u8 = [synth.synthetic_u8_clips(B, T, seed=300 + 17 * rank + i).pin_memory() for i in range(main.pool_n)]
        cool_down()
        u8_s = e2e_time(plan8, host_u8)
        e2e_u8 = {"value": world * B * args.steps / u8_s, "unit": UNIT, "h2d_bytes_per_step": B * T * 96 * 96,
                  "d2h_bytes_per_step": B * T * 512 * 4, "ms_per_step": 1e3 * u8_s / args.steps,
                  "input": "raw uint8 gray frames [B,T,96,96] from pinned host memory; /255, ColorNormalize, 88x88 "
                           "centre crop fused into the clip-prep kernel (bit-identical to the fp32 path)",
                  "result_checksum": float(main.out_host[(args.steps - 1) % 2].double().abs().mean())}
        del plan8

    # ---- one-batch latency of the unpipelined plan (same timing rules; extra key, not the metric) ----------
    latency = None
    if pipelined:
        lat_n = min(args.steps, 20)
        cool_down()
        lat_ms = main.time_device(lat_n, 3, plan=main.plan_lat, defer=False)
        latency = {"ms_per_step": lat_ms, "clips_per_s": world * B / (lat_ms * 1e-3), "steps": lat_n,
                   "frac_of_bf16_peak": B / (lat_ms * 1e-3) * fpc / 1e12 / float(peaks["bf16_tflops"]),
                   "plan": "VisualEncoderPlan (one batch per replay, nothing overlapped across batches)"}

    gather_verified = main.verify_gather()

    # ---- sustained regime: >= sustained_seconds of back-to-back steps, NO flush, NO gaps (a dataset-length run sits in
    # the power-capped clock regime MEASURED_PEAKS.json documents; each step's ~0.6 GB of activation traffic evicts L2 by
    # itself).  One event pair around the whole region; clocks sampled during it. ------------------------------------
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(50, int(args.sustained_seconds / (dev_ms * 1e-3)))
        for i in range(5):
            main.device_step(i, flush=False)
        barrier()
        sus_sampler = ClockSampler(local_rank)
        sus_sampler.start()
        with torch.cuda.stream(plan.compute):
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(plan.compute)
        for i in range(n_sus):
            main.device_step(i, flush=False)
        with torch.cuda.stream(plan.compute):
            s1.record(plan.compute)
        barrier()
        sus_sampler.stop()
        main.flush_pending_gather()
        barrier()
        sus_ms = sharding.max_over_ranks(s0.elapsed_time(s1), dev) / n_sus
        sus_tf = B / (sus_ms * 1e-3) * fpc / 1e12
        sustained = {"seconds": sus_ms * n_sus * 1e-3, "steps": n_sus, "ms_per_step": sus_ms,
                     "clips_per_s": world * B / (sus_ms * 1e-3), "tflops_per_gpu": sus_tf,
                     "frac_of_bf16_sustained": sus_tf / float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])),
                     "frac_of_bf16_burst": sus_tf / float(peaks["bf16_tflops"]),
                     "clocks": sus_sampler.summary(),
                     "how": "back-to-back pipelined steps (input copy + graph replay + gather), no L2 flush, no host "
                            "gaps, one CUDA event pair around the whole region, max over ranks"}

    # ---- host->device ceiling: the same pinned clip batches copied back to back by every rank at once, nothing else ----
    h2d_bytes = B * T * 88 * 88 * 4
    cp_stream = torch.cuda.Stream(device=dev)
    reps = max(20, args.steps)
    with torch.cuda.stream(cp_stream):
        for i in range(3):
            plan.x[0].copy_(main.host_pool[i % main.pool_n], non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    with torch.cuda.stream(cp_stream):
        for i in range(reps):
            plan.x[i % 2].copy_(main.host_pool[i % main.pool_n], non_blocking=True)
    cp_stream.synchronize()
    cp_s = sharding.max_over_ranks(time.perf_counter() - t0, dev)
    barrier()
    h2d_ceiling_gbs = world * reps * h2d_bytes / cp_s / 1e9
    h2d_ceiling_clips = world * reps * B / cp_s

    # ---- BASELINE configs[2]: LRW-1000-shaped 40-frame clips, batch 64 sharded across 8 GPUs = 8 clips per GPU --------
    config2 = None
    if not args.no_config2 and (B, T) != (8, 40):
        c2 = Shape(ctx, 8, 40)
        cool_down()      # (this leg follows the sustained run)
        c2_ms = c2.time_device(args.steps, args.warmup)
        c2_lat = c2.time_device(min(args.steps, 20), 3, plan=c2.plan_lat, defer=False) if c2.pipelined else None
        f2 = flops_per_clip(40, L)
        config2 = {"workload": f"BASELINE configs[2]: 40-frame clips, encoder forward, 8 clips per GPU x {world} GPU(s) = "
                               f"global batch {8 * world}" + (" (the configuration itself)" if world == 8 else
                                                             " (1/8 .. shard of it; --gpus 8 runs the configuration)"),
                   "value": world * 8 / (c2_ms * 1e-3), "unit": UNIT, "ms_per_step": c2_ms, "n_gpus": world,
                   "latency_ms_unpipelined": c2_lat, "pipelined": c2.pipelined,
                   "frac_of_bf16_peak": 8 / (c2_ms * 1e-3) * f2 / 1e12 / float(peaks["bf16_tflops"]),
                   "gather_verified": c2.verify_gather()}
        del c2

    # ---- per-kernel roofline (rank 0): eager traced passes, PDL off so every launch is timed alone --------
    line_extra = {}
    breakdown = []
    if rank == 0:
        ctx_sms = int(ops.init())
        prev_pdl = ops.set_pdl(False)
        prev_cl = enc.stack_cluster_size
        if pipelined:
            enc.stack_cluster_size = plan.enc_cluster   # the launch the timed region uses (one launch, one cluster size)
        agg = {}
        passes = 5
        with torch.no_grad():
            for rep in range(passes + 1):
                sink = []
                ctx.flush.zero_()
                with ops.trace(sink):
                    out, = enc(fe(main.dev_pool[rep % main.pool_n]), [T] * B)
                torch.cuda.synchronize(dev)
                if rep == 0:
                    continue  # warm-up pass
                for r in sink:
                    key = (r["name"], r["tag"])
                    a = agg.setdefault(key, {"ms": 0.0, "launches": 0, "flops": r["flops"], "bytes": r["bytes"]})
                    a["ms"] += r["start"].elapsed_time(r["end"])
                    a["launches"] += 1
        ops.set_pdl(bool(prev_pdl))
        enc.stack_cluster_size = prev_cl
        total_ms = sum(a["ms"] for a in agg.values()) / passes
        rows = sorted(agg.items(), key=lambda kv: -kv[1]["ms"])
        for (name, tag), a in rows[:8]:
            per = a["ms"] / a["launches"]
            breakdown.append({"kernel": name.replace("sblk_", ""), "case": tag, "n": a["launches"] // passes,
                              "us": round(per * 1e3, 1), "share": round(a["ms"] / passes / total_ms, 3),
                              "tflops": round(a["flops"] / (per * 1e-3) / 1e12) if a["flops"] else None})
        traffic_table = {}
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            try:
                with open(tp) as f:
                    traffic_table = json.load(f)
            except Exception:
                traffic_table = {}

        def roofline_of(row):
            (name, tag), a = row
            per_s = a["ms"] / a["launches"] * 1e-3
            if a["flops"]:
                ach, peak = a["flops"] / per_s / 1e12, float(peaks["bf16_tflops"])
                roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak}
            else:
                ach, peak = a["bytes"] / per_s / 1e9, float(peaks["hbm_gbs"])
                roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}
            roof.update({"traffic": traffic_table.get(f"{name}|{tag}"), "kernel": name, "case": tag,
                         "avg_launch_us": per_s * 1e6, "launches_per_step": a["launches"] // passes,
                         "share_of_step": a["ms"] / passes / total_ms,
                         "peak_source": peaks["_source"] + " (MEASURED_PEAKS.json burst figure: kernel timed alone)"})
            return roof

        roof = roofline_of(rows[0])
        if pipelined and rows[0][0][0] == "sblk_encoder_stack_fwd":
            # in the pipelined plan the stack runs on the side stream next to the next batch's prep + stem: the largest
            # kernel group of the step's critical path is reported as well
            roof["note"] = ("latency-bound dependent chain (25 GEMM stages) holding `sms_held` of the GPU's SMs; overlapped "
                            "with the next batch's frontend head by the pipelined plan in the `as_pipelined` form, see "
                            "critical_path and path")
            nxt = [r for r in rows if r[0][0] != "sblk_encoder_stack_fwd"]
            if nxt:
                roof["critical_path"] = roofline_of(nxt[0])
            # the figures above time the stack in its one-group-per-cluster form (clusters of `enc_cluster` CTAs, one per
            # clip group); the pipelined plan launches it with `enc_gpc` groups interleaved per cluster on fewer SMs.
            # Time that form alone as well and say how many SMs each form holds: `frac` divides by the WHOLE GPU's peak.
            try:
                gpc, cl = int(plan.enc_gpc), int(plan.enc_cluster)
                groups = -(-B // max(1, 128 // T))
                roof["sms_held"] = cl * groups
                roof["frac_of_held_sms_peak"] = roof["frac"] * ctx_sms / max(1, cl * groups)
                if gpc > 1:
                    saved = (enc.stack_cluster_size, enc.stack_groups_per_cluster)
                    enc.stack_cluster_size, enc.stack_groups_per_cluster = cl, gpc
                    feat_probe = torch.randn(B, T, 512, device=dev)
                    ts = []
                    with torch.no_grad():
                        for rep in range(6):
                            ctx.flush.zero_()
                            sink2 = []
                            with ops.trace(sink2):
                                enc(feat_probe, [T] * B)
                            torch.cuda.synchronize(dev)
                            ts += [r_["start"].elapsed_time(r_["end"]) for r_ in sink2
                                   if r_["name"] == "sblk_encoder_stack_fwd"]
                    enc.stack_cluster_size, enc.stack_groups_per_cluster = saved
                    us = sorted(ts[1:])[len(ts[1:]) // 2] * 1e3
                    held = cl * -(-groups // gpc)
                    ach = roof["achieved"] * roof["avg_launch_us"] / us
                    roof["as_pipelined"] = {"groups_per_cluster": gpc, "sms_held": held, "avg_launch_us": us,
                                            "achieved": ach, "frac": ach / roof["peak"],
                                            "frac_of_held_sms_peak": ach / roof["peak"] * ctx_sms / max(1, held),
                                            "what": "the stack launch of the pipelined plan (same kernel, clip groups "
                                                    "interleaved per cluster) timed alone like the figures above"}
            except Exception as e:  # noqa: BLE001  (a diagnostic key must not cost the line)
                roof["as_pipelined"] = {"error": str(e)}
        path_tf = value / world * fpc / 1e12
        roof["path"] = {"flops_per_clip": fpc, "achieved_tflops_per_gpu": path_tf,
                        "frac_of_bf16_peak": path_tf / float(peaks["bf16_tflops"]),
                        "frac_of_bf16_sustained": path_tf / float(peaks.get("bf16_tflops_sustained",
                                                                            peaks["bf16_tflops"])),
                        "eager_traced_ms_per_step": total_ms}
        if latency is not None:
            roof["unpipelined"] = {"ms_per_step": latency["ms_per_step"], "frac_of_bf16_peak": latency["frac_of_bf16_peak"]}
        if sustained is not None:
            roof["sustained"] = {k: sustained[k] for k in ("seconds", "ms_per_step", "clips_per_s", "tflops_per_gpu",
                                                           "frac_of_bf16_sustained", "frac_of_bf16_burst", "clocks")}
        line_extra["roofline"] = roof

        # ---- CPU baseline beside it (rank 0, N == 1 only): the reference's own modules on the same batch --------------
        if world == 1 and not args.no_cpu_baseline:
            step, cores, kind = cpu_reference_setup(L)
            xs = main.host_pool[0].clone()
            t0 = time.perf_counter()
            step(xs)
            probe = time.perf_counter() - t0
            sample = B
            if probe > args.cpu_seconds / 2:        # slow host: bounded sample of the batch
                sample = max(1, int(B * args.cpu_seconds / 2 / probe))
                xs = xs[:sample].contiguous()
            reps, t0 = 0, time.perf_counter()
            while True:
                step(xs)
                reps += 1
                if time.perf_counter() - t0 > args.cpu_seconds or reps >= 200:
                    break
            dt = time.perf_counter() - t0
            line_extra["cpu_baseline"] = {
                "value": sample * reps / dt, "unit": UNIT, "cores": cores, "kind": kind,
                "sample": f"{reps} forwards of {sample} clips x {T} frames" +
                          ("" if sample == B else f" (first {sample} clips of the {B}-clip batch)") +
                          (", unmodified reference Lipreading + Encoder from oracle/_ref" if kind == "reference" else
                           ", oracle/visual_encoder_oracle.py port") +
                          f", fp32, torch {torch.__version__} CPU, {dt:.1f} s"}

    if rank == 0:
        clocks = sampler.summary()
        cfg = dict(workload_config(args, world), host_numa_node_rank0=numa_node,
                   gather=main.gather_mode if world == 1 or not main.defer else
                   f"{main.gather_mode}, one gather per step inside its event pair: the previous step's output, on a "
                   f"side stream next to this step's replay",
                   gather_verified=gather_verified, pipeline=main.pipeline_note,
                   operands="bf16 conv trunk, " + str(ops.enc16_dtype()).replace("torch.", "") +
                            " transformer-encoder operands (same tcgen05 kind::f16 rate), fp32 accumulate / LN / softmax")
        if config2 is not None:
            cfg["config2"] = config2
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": B * T * 512 * 4, "ms_per_step": 1e3 * e2e_s / args.steps,
               "regime": "burst: K steps from an idle GPU (--cool-down-seconds pause after the device-timed leg), before the sustained run (see `sustained` for the power-capped regime)",
               "timing": "wall clock, synchronize on both sides, double-buffered H2D/compute/D2H",
               "result_checksum": checksum,
               "h2d_ceiling_gbs": h2d_ceiling_gbs, "h2d_ceiling_clips_per_s": h2d_ceiling_clips,
               "h2d_ceiling_how": f"copy-only: every rank copies its pinned {h2d_bytes / 1e6:.1f} MB fp32 clip batches "
                                  f"back to back ({reps} copies), all {world} rank(s) at once, aggregate bytes / max time"}
        if e2e_u8 is not None:
            e2e["u8"] = e2e_u8
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": cfg,
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": plan.launches_per_forward * args.steps,
            "gpu_launches_per_step": plan.launches_per_forward,
        }
        line.update(line_extra)
        # extra keys, shortest / most important LAST (the driver keeps the tail of the line next to the parsed contract keys)
        line["breakdown"] = breakdown
        line["latency"] = latency
        line["e2e_u8"] = e2e_u8
        line["h2d_ceiling_gbs"] = h2d_ceiling_gbs
        line["config2"] = config2
        line["sustained"] = sustained
        line["gather_verified"] = gather_verified
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_config4_sweep(args):
    """BASELINE configs[4]: the full SBL multilingual model, teacher-forced forward (`Transformer.forward`,
    transformer/transformer.py:22-43) — the B200 visual frontend + encoder with the UNMODIFIED reference bidirectional
    decoder (oracle/_ref) on top — over a batch sweep, next to the all-reference fp32 CUDA model (cuDNN / cuBLAS, TF32
    off) on the same inputs.  One rank per GPU, the batch sharded across ranks (no collective: every rank decodes its own
    clips).  Prints ONE JSON line; wall-clock timing with synchronize on both sides, max over ranks."""
    import random

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/sblk_bench_nccl_%h_%p.log")
        dist.init_process_group("nccl", device_id=dev)
    from oracle import ref_runtime
    from sbl_for_multilingual_lip_reading_b200 import dropin, ops, sharding, synth
    ops.init()
    ref_runtime.fp32_exact()
    R = ref_runtime.load_reference("sbl")
    sd = dict(synth.frontend_state_dict(1, prefix="visual_frontend."))
    sd.update(synth.encoder_state_dict(2, 6, prefix="encoder."))
    ref = ref_runtime.build_sbl_reference(R, sd).to(dev).eval()
    with dropin.patched_reference(R.dir):
        import transformer.encoder as tenc
        import transformer.transformer as ttr
        torch.manual_seed(7)
        enc = tenc.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        dec = R.Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                        pe_maxlen=5000)
        ours = ttr.Transformer(enc, dec, None)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(dev).eval()
    # row f.1: the SBL decoder on libsblk as well (decoder.py) — the whole model behind the reference's Transformer class
    with dropin.patched_reference(R.dir, decoder=True):
        import transformer.decoder as tdec
        torch.manual_seed(7)
        enc2 = tenc.Encoder(512, 6, 8, 64, 64, 512, 2048, dropout=0.1, pe_maxlen=5000)
        dec2 = tdec.Decoder(0, 1, 58, 512, 6, 8, 64, 64, 512, 2048, dropout=0.1, tgt_emb_prj_weight_sharing=1,
                            pe_maxlen=5000)
        full = ttr.Transformer(enc2, dec2, None)
    full.load_state_dict(ref.state_dict())
    full = full.to(dev).eval()
    T = 30
    rows = []
    for gb in [int(v) for v in args.config4_batches.split(",")]:
        n = max(1, gb // world)
        g = torch.Generator().manual_seed(11 + rank)
        x = synth.synthetic_clips(n, T, seed=900 + rank)[:, 0].to(dev)            # [n,T,88,88] as train.py feeds it
        tgt = torch.full((n, 14), -1, dtype=torch.long)
        for i in range(n):   # data_gen.py:297-302
            ln = int(torch.randint(3, 12, (1,), generator=g))
            tgt[i, :ln] = torch.randint(2, 58, (ln,), generator=g)
        tgt_r = tgt.clone()
        for i in range(n):
            ln = int((tgt[i] >= 0).sum())
            tgt_r[i, :ln] = tgt[i, :ln].flip(0)
        tgt, tgt_r = tgt.to(dev), tgt_r.to(dev)

        def timed(model, reps):
            with torch.no_grad():
                random.seed(7); torch.manual_seed(5)
                out = model(x, tgt, tgt_r)
                torch.cuda.synchronize(dev)
                if world > 1:
                    dist.barrier()
                t0 = time.perf_counter()
                for _ in range(reps):
                    out = model(x, tgt, tgt_r)
                torch.cuda.synchronize(dev)
                return sharding.max_over_ranks((time.perf_counter() - t0) / reps, dev), out

        def timed_encoder(model, reps):
            with torch.no_grad():
                xi = x.unsqueeze(4).permute(0, 4, 1, 2, 3)
                f = model.visual_frontend(xi); model.encoder(f, [T] * n)
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                for _ in range(reps):
                    f = model.visual_frontend(xi)
                    model.encoder(f, [T] * n)
                torch.cuda.synchronize(dev)
                return sharding.max_over_ranks((time.perf_counter() - t0) / reps, dev)

        reps = args.steps
        t_full, o0 = timed(full, reps)
        t_ours, o1 = timed(ours, reps)
        t_ref, o2 = timed(ref, reps)
        e_ours, e_ref = timed_encoder(ours, reps), timed_encoder(ref, reps)
        rows.append({"global_batch": n * world, "clips_per_gpu": n,
                     "b200_full_model_clips_per_s": n * world / t_full,
                     "b200_dropins_clips_per_s": n * world / t_ours, "reference_cuda_fp32_clips_per_s": n * world / t_ref,
                     "ms_per_forward": {"b200_full_model": 1e3 * t_full, "b200_dropins": 1e3 * t_ours,
                                        "reference_cuda_fp32": 1e3 * t_ref},
                     "visual_encoder_ms": {"b200_dropins": 1e3 * e_ours, "reference_cuda_fp32": 1e3 * e_ref},
                     "decoder_share_of_forward_b200": 1.0 - e_ours / t_ours,
                     "logits_rel_err_full_vs_reference": {
                         "l2r": float(((o0[0] - o2[0]).norm() / o2[0].norm())),
                         "r2l": float(((o0[2] - o2[2]).norm() / o2[2].norm()))}})
    if rank == 0:
        line = {"metric": "sbl_full_model_teacher_forced_forward_clips_per_sec", "unit": UNIT, "n_gpus": world,
                "config": {"workload": "BASELINE configs[4]: full SBL multilingual model teacher-forced forward (B200 visual "
                                       "frontend + encoder, reference bidirectional decoder from oracle/_ref on top), "
                                       f"{T}-frame clips, batch sweep, batch sharded over {world} GPU(s)",
                           "arms": "b200_full_model = frontend + encoder + SBL decoder on libsblk (decoder.py); b200_dropins = "
                                   "libsblk frontend + encoder under the UNMODIFIED reference decoder; reference_cuda_fp32 = "
                                   "all-reference model (cuDNN / cuBLAS fp32, TF32 off)",
                           "decoder": "Decoder.forward (decoder.py:79-191): 16 steps x 2 directions x 6 layers, full-prefix "
                                      "recompute each step",
                           "always_on_dropout": True},
                "sweep": rows, "data": "synthetic", "timing": "wall clock, synchronize both sides, max over ranks"}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_config3(args):
    """BASELINE configs[3]: 1500-class frontend pre-training (stage-1 classify model), forward + backward + Adam step,
    global batch 256 (strong scaling: 256 / world clips per GPU), 31-frame clips, 3-layer encoder; gradients all-reduced
    by DistributedDataParallel (bucketed NCCL, overlapped with the libsblk backward).  Device-timed with CUDA events around
    each step, max over ranks.  The all-reference fp32 CUDA model (cuDNN / cuBLAS, TF32 off) runs the same step beside it
    for context.  Prints ONE JSON line."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/sblk_bench_nccl_%h_%p.log")
        dist.init_process_group("nccl", device_id=dev)
    from sbl_for_multilingual_lip_reading_b200 import ops, sharding, stage1, synth
    ops.init()
    gb, T, L = args.config3_batch, 31, 3
    n = max(1, gb // world)
    torch.manual_seed(7)
    model = stage1.Stage1Classifier(n_layers_enc=L, dropout=0.1).load_synthetic(1, 3).to(dev).train()
    net = (torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], broadcast_buffers=False)
           if world > 1 else model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
    x = synth.synthetic_clips(n, T, seed=40 + rank, pad_frames=2).to(dev)
    y = torch.randint(0, 1500, (n,), generator=torch.Generator().manual_seed(rank)).to(dev)
    lang = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(100 + rank)).to(dev)

    def step(m, o):
        v_t, v_l = m(x)
        loss = F.cross_entropy(v_t, y) + 0.1 * F.cross_entropy(v_l, lang)     # train.py:129-132
        o.zero_grad()
        loss.backward()
        o.step()
        return loss

    def timed(m, o, steps, warmup):
        for _ in range(warmup):
            step(m, o)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        evs = []
        before = ops.launch_count()
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = step(m, o)
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize(dev)
        launches = ops.launch_count() - before
        ms = sharding.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), dev) / steps
        return ms, float(loss.detach()), launches

    steps, warmup = args.steps, args.warmup
    ms, loss, launches = timed(net, opt, steps, warmup)
    ref_ms = None
    if not args.no_cpu_baseline:
        # context arm: the unmodified reference modules under the same step on the same GPU(s) (fp32, cuDNN / cuBLAS)
        from oracle import ref_runtime
        ref_runtime.fp32_exact()
        R = ref_runtime.load_reference("cls")
        sd = dict(synth.frontend_state_dict(1, prefix="visual_frontend."))
        sd.update(synth.encoder_state_dict(3, L, prefix="encoder_v."))
        rmodel = ref_runtime.build_cls_reference(R, sd, n_layers_enc=L).to(dev).train()

        class RefStage1(torch.nn.Module):
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, xx):
                feat = self.m.visual_frontend(xx)
                out, *_ = self.m.encoder_v(feat, [feat.size(1)] * feat.size(0))
                return self.m.fc_1500(out.mean(dim=1)), self.m.fc_2(out[:, 30, :])
        rnet = RefStage1(rmodel)
        if world > 1:
            rnet = torch.nn.parallel.DistributedDataParallel(rnet, device_ids=[local_rank], broadcast_buffers=False)
        ropt = torch.optim.Adam(rmodel.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
        ref_ms, _, _ = timed(rnet, ropt, max(2, steps // 2), 1)
    if rank == 0:
        # 2*MACs of the forward x3 (dgrad + wgrad) is the usual training estimate; the stem has no dgrad
        fpc = flops_per_clip(T, L)
        peaks = load_peaks()
        tf = 3.0 * n * fpc / (ms * 1e-3) / 1e12
        line = {"metric": "stage1_pretraining_clips_per_sec_fwd_bwd", "value": n * world / (ms * 1e-3), "unit": UNIT,
                "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "BASELINE configs[3]: 1500-class frontend pre-training (stage-1 classify model: Conv3d "
                                       "frontend + ResNet-18 + 3-layer encoder + fc_1500 / fc_2), forward + backward + Adam "
                                       f"step, global batch {n * world} = {n} clips x {T} frames per GPU, "
                                       "batch-statistics BatchNorm, dropout 0.1, DistributedDataParallel NCCL gradient "
                                       "all-reduce" + ("" if world > 1 else " (single GPU: no collective)"),
                           "global_batch": n * world, "clips_per_gpu": n, "frames": T, "encoder_layers": L,
                           "parallelism": f"ddp{world}"},
                "loss": loss, "gpu_launches_per_step": launches // steps,
                "approx_tflops_per_gpu": tf, "approx_frac_of_bf16_peak": tf / float(peaks["bf16_tflops"]),
                "reference_cuda_fp32": None if ref_ms is None else
                {"ms_per_step": ref_ms, "clips_per_s": n * world / (ref_ms * 1e-3),
                 "what": "unmodified reference modules (oracle/_ref), same step, fp32 cuDNN / cuBLAS with TF32 off"}}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="clips per GPU (BASELINE configs[1]: 32)")
    ap.add_argument("--frames", type=int, default=29)
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="time the one-batch plan instead of the two-stage software pipeline")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU output gathering inside the step: one-shot peer-memory kernel (default) or NCCL")
    ap.add_argument("--inline-gather", action="store_true",
                    help="multi-GPU, pipelined plan: gather each step's output in stream after the replay instead of on a "
                         "side stream next to the following step's replay")
    ap.add_argument("--workload", default="visual_encoder", choices=["visual_encoder", "config3", "config4"],
                    help="config4 = BASELINE configs[4] sweep: full SBL model (reference decoder on the drop-ins)")
    ap.add_argument("--config4-batches", default="16,32,64,128,256,512")
    ap.add_argument("--config3-batch", type=int, default=256, help="global batch of the configs[3] training step")
    ap.add_argument("--no-u8", action="store_true", help="skip the fused uint8-input end-to-end measurement (e2e_u8)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config2", action="store_true", help="skip the BASELINE configs[2] (8 clips x 40 frames per GPU) leg")
    ap.add_argument("--cool-down-seconds", type=float, default=1.0,
                    help="idle pause in front of every burst leg after the first (e2e, e2e_u8, latency)")
    ap.add_argument("--sustained-seconds", type=float, default=2.5,
                    help="length of the back-to-back sustained-regime run (0 = skip)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-clips", type=int, default=0,
                    help="clips per reference-arm step (0 = the whole --batch, bounded only on very slow hosts)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the encoder output of the last timed step, gathered over the "
                         "ranks ([gpus*batch,T,512]), as DIR/encoder_output.npy (float32; a seeded sample of clips above "
                         "64 MiB); "
                         "inputs and the dropout seed are fixed, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "visual_encoder"):
        ap.error("--dump-outputs is supported for the visual_encoder workload of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "b200" and args.gpus != world:
        if args.gpus > 1 and world == 1:
            raise SystemExit(f"bench.py --gpus {args.gpus}: launch with torch.distributed.run "
                             f"--nproc-per-node {args.gpus} (one rank per GPU)")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "config4":
        return run_config4_sweep(args)
    if args.workload == "config3":
        return run_config3(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
