"""Static-shape execution plans for the visual-encoder path: CUDA-graph replay + pipelined host I/O.

The reference runs the path eagerly (`Transformer.forward`, transformer/transformer.py:34-38: frontend, then
encoder with `input_lengths = [T]*N`).  Eagerly the B200 path is ~70 short kernels, so the host launch rate,
not the GPU, bounds it.  `VisualEncoderPlan` captures `encoder(frontend(x), [T]*N)` for one (N, T) into a CUDA
graph per input slot (streams + graphs instead of a tracing compiler) and exposes:

  * `forward_device(slot)`   replay on a pre-filled device input slot (bench `value`: inputs resident in HBM)
  * `submit_host(x, out)`    pinned-host -> H2D (copy stream) -> graph (compute stream) -> D2H (copy-out stream),
                             double-buffered so the PCIe copy of clip batch i+1 overlaps the compute of batch i
                             (bench `e2e`)

`PipelinedVisualEncoderPlan` is the throughput form of the same plan: a two-stage software pipeline in which the
(latency-bound, 64-SM) encoder stack of batch i-1 runs next to the clip prep + Conv3d stem of batch i.

The modules stay ordinary drop-ins: a plan is an optional accelerator around them, owning only torch tensors,
streams and graphs.  It passes its schedule to them as arguments (`Lipreading._frontend_forward`,
`Encoder._forward_eval`) and never changes their attributes.
"""
from __future__ import annotations

import torch

from . import ops


class VisualEncoderPlan:
    def __init__(self, frontend, encoder, n, t, device=None, slots=2, pdl=True, lengths=None, u8_input=None):
        self.frontend, self.encoder = frontend, encoder
        self.n, self.t, self.slots = int(n), int(t), int(slots)
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("VisualEncoderPlan needs a CUDA (B200) device; there is no CPU path")
        self.lengths = [self.t] * self.n if lengths is None else [int(v) for v in lengths]
        self.d_model = encoder.d_model
        with torch.cuda.device(self.device):
            ops.init()
            self._prev_pdl = ops.set_pdl(bool(pdl))
            self.compute = torch.cuda.Stream()
            self.copy_in = torch.cuda.Stream()
            self.copy_out = torch.cuda.Stream()
            # u8_input = (T_in, H0, W0): the plan takes the loader's raw uint8 frames and runs the fused input pipeline
            # (Lipreading.forward_u8: /255, normalise, centre-crop, pad to t frames) instead of fp32 clips
            self.u8_input = None if u8_input is None else tuple(int(v) for v in u8_input)
            if self.u8_input is None:
                self.x = [torch.zeros((self.n, 1, self.t, 88, 88), dtype=torch.float32, device=self.device)
                          for _ in range(self.slots)]
            else:
                t_in, h0, w0 = self.u8_input
                self.x = [torch.zeros((self.n, t_in, h0, w0), dtype=torch.uint8, device=self.device)
                          for _ in range(self.slots)]
            self.out = [None] * self.slots
            self.graphs = [None] * self.slots
            self.ev_in = [torch.cuda.Event() for _ in range(self.slots)]
            self.ev_done = [torch.cuda.Event() for _ in range(self.slots)]
            self.ev_out = [torch.cuda.Event() for _ in range(self.slots)]
            self.launches_per_forward = 0
            self._capture()
            self._pin_captured_state()
        self._i = 0

    # -------------------------------------------------------------------------------------------
    def _pin_captured_state(self):
        """A captured graph bakes in raw pointers to tensors the MODULES own as caches: packed weights, the zero-haloed
        flat workspaces, staged lengths vectors, the uint8 normalisation table.  The plan keeps strong references to all
        of them (a cache eviction or a re-pack after `load_state_dict` can then never free memory a replay still reads
        or writes) and records the weight versions it was captured with; `_check_weights` refuses to replay stale ones."""
        fe, enc = self.frontend, self.encoder
        self._pinned = (fe._packed, enc._packed, dict(fe._flat_ws), dict(enc._len_cache), dict(fe._lut))
        # the parameter / buffer OBJECTS are fixed for a module's life (load_state_dict, .to() and optimizers update them
        # in place), so the per-replay check walks a cached flat list instead of the module tree (~20 us)
        self._wtensors = [t for m in (fe, enc) for t in list(m.parameters()) + list(m.buffers())]
        self._weights_key = self._weights_now()

    def _weights_now(self):
        return tuple([(t.data_ptr(), t._version) for t in self._wtensors])

    def _check_weights(self):
        if self._weights_now() != self._weights_key:
            raise RuntimeError("the frontend / encoder weights changed after this plan was captured (load_state_dict or an "
                               "in-place update): its CUDA graphs still hold the old packed weights — call recapture()")

    def recapture(self):
        """Re-pack the weights and capture the graphs again (after load_state_dict / an optimizer step)."""
        self.synchronize()
        with torch.cuda.device(self.device):
            self._capture()
            self._pin_captured_state()

    # -------------------------------------------------------------------------------------------
    def _u8_crop(self):
        """The loader's 88x88 centre crop of the raw frames (CenterCrop, data_gen.py)."""
        _, h0, w0 = self.u8_input
        return (h0 - 88) // 2, (w0 - 88) // 2

    def _frontend_eager(self, x):
        if self.u8_input is not None:
            return self.frontend.forward_u8(x, frames=self.t, crop=self._u8_crop())
        return self.frontend(x)

    def _forward_eager(self, x):
        out, = self.encoder(self._frontend_eager(x), self.lengths)
        return out

    def _trunk(self, x, **schedule):
        """The frontend of the input slot `x` with the plan's schedule (Lipreading._frontend_forward)."""
        if self.u8_input is None:
            return self.frontend._frontend_forward(x, **schedule)
        x, frames, prep = self.frontend._u8_prep(x, self.t, self._u8_crop())
        return self.frontend._frontend_forward(x, prep=prep, frames=frames, **schedule)

    def _draw_dropout(self, drawn, out=None):
        """Forks the draw of the always-on dropout's factor F.dropout(ones, p=0.5) (Lipreading.forward, reference :122: the
        same generator draw as the module's F.dropout(features)) onto the tail stream and records `drawn` there once it
        is done.  Returns the factor (`out` when given: the draw is copied into it)."""
        fork = torch.cuda.Event()
        fork.record(torch.cuda.current_stream())
        self._tail_stream.wait_event(fork)
        with torch.cuda.stream(self._tail_stream):
            scale = torch.nn.functional.dropout(self._ones, p=0.5)
            if out is not None:
                scale = out.copy_(scale)
            drawn.record(self._tail_stream)
        return scale

    def _forward_fused_tail(self, s):
        """encoder(frontend(x[s])) with the dropout factor drawn off the critical path and the pooling launch writing the
        encoder's operand (capture-time only; see _capture)."""
        main = torch.cuda.current_stream()
        scale, join = None, None
        if self.frontend.always_on_dropout:
            drawn = torch.cuda.Event()
            scale = self._draw_dropout(drawn)
            join = lambda: main.wait_event(drawn)   # noqa: E731  (called right before the pooling launch)
        self._trunk(self.x[s], prefetch_extra=self._prefetch, scale=scale, out16=self.feat16[s], before_pool=join)
        out, = self.encoder._forward_eval(self.feat, self.lengths, x16=self.feat16[s])
        return out

    def _capture(self):
        torch.cuda.synchronize(self.device)
        fe, enc = self.frontend, self.encoder
        with torch.no_grad():
            # the frontend pulls the encoder's packed weights into L2 while its last layer runs (side stream)
            self._prefetch = []
            if fe.l2_prefetch:
                with torch.cuda.device(self.device):
                    stk = enc._get_packed().stacked
                self._prefetch = [stk[k] for k in ("w_in", "w_heads", "w_fc", "w_1", "w_2")]
            # warm-up on the capture stream: packs weights, sizes kernels, stages the lengths vector
            with torch.cuda.stream(self.compute):
                for _ in range(2):
                    self._forward_eager(self.x[0])
            self.compute.synchronize()
            # One private memory pool PER graph: with a shared pool the static output of one slot may alias an
            # intermediate buffer of the other slot's graph, and submit_host lets the device->host copy of slot s overlap
            # the replay of slot s^1 (a few hundred MB per pool; HBM is not the constraint here).
            # Fused tail (same as the pipelined plan): the always-on dropout factor of Lipreading.forward (reference :122)
            # is drawn on a side stream while the trunk runs and applied by the pooling launch, which writes the encoder's
            # 16-bit operand directly — no dropout / cast launches between the last conv and the encoder stack.
            # Bit-identical to the module path (same generator draw, same single rounding).
            fused_tail = not fe.training and not enc.training and enc._use_fused_stack(self.n, self.t, False)
            if fused_tail:
                dev = self.device
                self.feat16 = [torch.zeros((self.n * self.t, fe.inputDim), dtype=ops.enc16_dtype(), device=dev)
                               for _ in range(self.slots)]
                self.feat = torch.empty((self.n, self.t, fe.inputDim), dtype=torch.float32, device=dev)
                self._ones = torch.ones((self.n * self.t, fe.inputDim), dtype=torch.float32, device=dev)
                self._tail_stream = torch.cuda.Stream(device=dev)
            for s in range(self.slots):
                g = torch.cuda.CUDAGraph()
                before = ops.launch_count()
                with torch.cuda.graph(g, stream=self.compute):
                    if fused_tail:
                        self.out[s] = self._forward_fused_tail(s)
                    else:
                        self.out[s] = self._forward_eager(self.x[s])
                self.launches_per_forward = ops.launch_count() - before
                self.graphs[s] = g
        torch.cuda.synchronize(self.device)
        for ev in self.ev_out + self.ev_done:
            ev.record(torch.cuda.current_stream(self.device))

    # -------------------------------------------------------------------------------------------
    def forward_device(self, slot=0):
        """Replay on the compute stream of the plan; returns the static output tensor [N,T,d_model] fp32."""
        self._check_weights()
        with torch.cuda.stream(self.compute):
            self.graphs[slot].replay()
        return self.out[slot]

    def submit_host(self, x_host, out_host):
        """One pipelined step: x_host pinned fp32 [N,1,T,88,88] -> out_host pinned fp32 [N,T,d_model].
        Asynchronous; returns the event that marks out_host complete."""
        self._check_weights()
        s = self._i % self.slots
        self._i += 1
        # slot s is reusable once its previous replay finished (input consumed) and its output left the device
        self.copy_in.wait_event(self.ev_done[s])
        with torch.cuda.stream(self.copy_in):
            self.x[s].copy_(x_host, non_blocking=True)
            self.ev_in[s].record(self.copy_in)
        self.compute.wait_event(self.ev_in[s])
        self.compute.wait_event(self.ev_out[s])
        with torch.cuda.stream(self.compute):
            self.graphs[s].replay()
            self.ev_done[s].record(self.compute)
        self.copy_out.wait_event(self.ev_done[s])
        with torch.cuda.stream(self.copy_out):
            out_host.copy_(self.out[s], non_blocking=True)
            self.ev_out[s].record(self.copy_out)
        return self.ev_out[s]

    def synchronize(self):
        self.copy_in.synchronize()
        self.compute.synchronize()
        self.copy_out.synchronize()

    def close(self):
        ops.set_pdl(bool(self._prev_pdl))


class PipelinedVisualEncoderPlan(VisualEncoderPlan):
    """Two-stage software pipeline over consecutive clip batches (steady-state throughput; one batch of extra latency).

    The one-launch encoder stack is a dependent chain of 25 small GEMM stages: at the BASELINE batch it holds 8 clusters
    of 8 CTAs (64 of the 148 SMs) for ~0.2 ms at 10 % of the tensor peak, while the frontend kernels fill the machine.
    Replay i of this plan therefore runs

        encoder(features of batch i-1)   on a side stream, 8-CTA clusters           ||
        clip prep + Conv3d stem (+ the first `head_blocks` residual blocks) of batch i, persistent grids sized for the
        SMs the encoder leaves free (`head_sm_limit`)

    joins, and runs the rest of the trunk of batch i at full width.  A one-thread gate kernel (`ops.gate_wait`) holds
    the head back until every encoder cluster has been placed, so the two chains never fight over SM placement.
    Results are bit-identical to the unpipelined plan (same kernels; the grid size of a persistent kernel does not change
    any tile's arithmetic).  `forward_device(slot)` / `submit_host` return the output of the PREVIOUS batch; `drain()`
    finishes the last one."""

    def __init__(self, frontend, encoder, n, t, device=None, pdl=True, lengths=None, u8_input=None,
                 head_sm_limit=None, head_blocks=None, gate=True, gate_timeout_us=300, enc_cluster=None,
                 head_frac=None, enc_gpc=None, l2_prefetch=False):
        # head_frac: fraction of the frames of the first conv after the head that still runs inside the head (limited
        # width) — fills the time by which the encoder outlasts prep + stem; None = automatic, 0 = off
        self.head_frac = head_frac
        # l2_prefetch: keep the frontend's L2 weight-prefetch launches inside the step.  They pay for themselves in the
        # one-batch-per-replay plan (the encoder's weight chain starts cold: 746 vs 883 us) but not here, where the encoder
        # runs at the START of the step and the hints compete with the head for HBM (tools/exp/l2_prefetch_ab.py: 622.7 ->
        # 608-610 us with the L2 flushed between steps, 661-665 -> 654-657 us back to back; 42 -> 18 launches per step)
        self.l2_prefetch = bool(l2_prefetch)
        # head_blocks: residual blocks (after prep + stem) that run next to the encoder on `head_sm_limit` SMs; None =
        # automatic (see _capture).  enc_cluster: CTAs per encoder cluster (8 or 16), None = 8.
        self.enc_cluster = enc_cluster
        # enc_gpc: clip groups per encoder cluster (1, or 2 = interleaved: half the SMs for ~1.5x the time); None = 1
        self.enc_gpc = enc_gpc
        self.head_sm_limit, self.head_blocks = head_sm_limit, head_blocks
        self.use_gate, self.gate_timeout_us = bool(gate), int(gate_timeout_us)
        super().__init__(frontend, encoder, n, t, device=device, slots=2, pdl=pdl, lengths=lengths, u8_input=u8_input)

    def _capture(self):
        fe, enc = self.frontend, self.encoder
        dev = self.device
        g_clips = max(1, 128 // self.t)
        groups = -(-self.n // g_clips)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        if self.enc_cluster is None:
            # 8-CTA clusters leave the most SMs to the co-running frontend (measured at 8 clips x 40 frames: 375 us per
            # step with clusters of 8 against 401 us with 16, 511 us unpipelined)
            self.enc_cluster = 8
        cl = int(self.enc_cluster)
        if self.enc_gpc is None:
            # BASELINE-sized batches: two clip groups interleaved per encoder cluster — 4 clusters of 8 CTAs hold 32 SMs
            # for ~310 us instead of 64 SMs for ~215 us, and the frontend of the next batch gets 116 SMs (measured,
            # tools/exp/head_frac_probe.py: 688.1 -> 657.4 us per step); small batches (configs[2] shard, 3 groups): one
            # group per cluster is faster (360.4 vs 368.6 us)
            self.enc_gpc = 2 if (self.n * self.t > 512 and groups >= 6) else 1
        gpc = int(self.enc_gpc)
        groups = -(-groups // gpc)   # clusters
        if cl not in (8, 16) or gpc not in (1, 2) or not enc._use_fused_stack(self.n, self.t, False) or cl * groups > sms - 16:
            raise RuntimeError("PipelinedVisualEncoderPlan needs the one-launch encoder stack in one wave of clusters "
                               f"({groups} clip groups x {cl} CTAs on {sms} SMs); use VisualEncoderPlan for this shape")
        enc_ctas = cl * groups
        if self.head_sm_limit is None:
            self.head_sm_limit = (sms - enc_ctas) & ~1
        if self.head_blocks is None:
            # BASELINE-sized batches: prep + the (tensor-memory-filter) stem + the first residual block fit next to the
            # ~0.2 ms one-group-per-cluster encoder (measured, tools/exp/head_frac_probe.py: 712.7 us with half a conv in
            # the head, 700.4 with a whole conv, 675.8 with the whole block, 706.6 with two blocks); next to the ~0.3 ms
            # two-groups-per-cluster encoder: layers 1 and 2 (741 / 698 / 657 / 678 us with 2 / 3 / 4 / 5 blocks); small
            # latency-bound batches: the whole frontend co-runs with it
            self.head_blocks = (4 if gpc == 2 else 1) if self.n * self.t > 512 else 8
        self.head_blocks = int(self.head_blocks)
        if self.head_frac is None:
            # share of the frames of the first conv AFTER the head that still runs inside it: 675.8 us (0) / 679.9 (0.1) /
            # 677.9 (0.2) / 682.0 (0.4) per step at the BASELINE batch with one block in the head
            self.head_frac = 0.0
        self.head_frac = float(self.head_frac)
        torch.cuda.synchronize(dev)
        self.enc_stream = torch.cuda.Stream(device=dev, priority=-1)
        self.gate = torch.zeros(2, dtype=torch.int32, device=dev)
        # features cross the pipeline stages as the bf16 GEMM operand the encoder stack reads (written by the frontend's
        # last launch — average pool x dropout factor — so the encoder branch of the next replay is the stack kernel
        # alone); `feat` only carries the shape
        self.feat16 = [torch.zeros((self.n * self.t, fe.inputDim), dtype=ops.enc16_dtype(), device=dev) for _ in range(2)]
        self.feat = torch.empty((self.n, self.t, fe.inputDim), dtype=torch.float32, device=dev)
        self._ones = torch.ones((self.n * self.t, fe.inputDim), dtype=torch.float32, device=dev)
        self._tail_stream = torch.cuda.Stream(device=dev)
        self._scale = [torch.empty_like(self._ones) for _ in range(2)]
        stack = dict(cluster_size=cl, groups_per_cluster=gpc)
        prefetch = fe.l2_prefetch and self.l2_prefetch
        with torch.no_grad():
            stk = enc._get_packed().stacked
            self._prefetch = [stk[k] for k in ("w_in", "w_heads", "w_fc", "w_1", "w_2")] if prefetch else []
            with torch.cuda.stream(self.compute):   # warm-up: packs weights, sizes kernels, stages the lengths
                for _ in range(2):
                    enc._forward_eval(self._frontend_eager(self.x[0]), self.lengths, **stack)
            self.compute.synchronize()
            for s in range(2):   # one private pool per graph (see VisualEncoderPlan._capture)
                g = torch.cuda.CUDAGraph()
                before = ops.launch_count()
                with torch.cuda.graph(g, stream=self.compute):
                    main = torch.cuda.current_stream()
                    fork, done = torch.cuda.Event(), torch.cuda.Event()
                    fork.record(main)
                    self.enc_stream.wait_event(fork)
                    with torch.cuda.stream(self.enc_stream):
                        self.out[s ^ 1], = enc._forward_eval(self.feat, self.lengths, x16=self.feat16[s ^ 1],
                                                             resident_counter=self.gate if self.use_gate else None,
                                                             **stack)
                        done.record(self.enc_stream)
                    if self.use_gate:
                        ops.gate_wait(self.gate, enc_ctas, self.gate_timeout_us)
                    # the always-on dropout of Lipreading.forward (reference :122): its factor mask / (1 - p) is drawn
                    # on a side stream and applied by the pooling launch that ends the trunk.  The draw is forked right
                    # before layer 4 (residual block 6) is enqueued: its two small launches cost 10-12 us of the step at
                    # the start of the replay (in stream OR on a side stream: they take SMs while the encoder's clusters
                    # and the gated stem are being placed, tools/exp/pipeline_switches_probe.py), while the 132-CTA
                    # grids of layer 4 leave 16 SMs idle anyway.
                    scale, draw, join = None, None, None
                    if fe.always_on_dropout:
                        scale, drawn = self._scale[s], torch.cuda.Event()
                        draw = lambda: self._draw_dropout(drawn, out=scale)   # noqa: E731
                        join = lambda: main.wait_event(drawn)   # noqa: E731
                    self._trunk(self.x[s], head_sm_limit=self.head_sm_limit, head_blocks=self.head_blocks,
                                head_join=lambda: main.wait_event(done), head_frac=self.head_frac,
                                hook=draw, hook_block=6, scale=scale, out16=self.feat16[s], before_pool=join,
                                prefetch=prefetch, prefetch_extra=self._prefetch)
                self.launches_per_forward = ops.launch_count() - before
                self.graphs[s] = g
        torch.cuda.synchronize(dev)
        for ev in self.ev_out + self.ev_done:
            ev.record(torch.cuda.current_stream(dev))

    def forward_device(self, slot=0):
        """Replay step `slot`: frontend of x[slot] next to the encoder of the batch replayed before it (the other slot).
        Returns that PREVIOUS batch's static output tensor [N,T,d_model] fp32."""
        self._check_weights()
        with torch.cuda.stream(self.compute):
            self.graphs[slot].replay()
        return self.out[slot ^ 1]

    def submit_host(self, x_host, out_host):
        """One pipelined step: x_host (pinned) -> device; out_host (pinned) receives the output of the batch submitted
        by the PREVIOUS call (of the warm-up / zero features on the first call).  Returns the completion event."""
        self._check_weights()
        s = self._i % 2
        self._i += 1
        self.copy_in.wait_event(self.ev_done[s])
        with torch.cuda.stream(self.copy_in):
            self.x[s].copy_(x_host, non_blocking=True)
            self.ev_in[s].record(self.copy_in)
        self.compute.wait_event(self.ev_in[s])
        self.compute.wait_event(self.ev_out[s])   # out[s ^ 1] of this graph's previous replay has left the device
        with torch.cuda.stream(self.compute):
            self.graphs[s].replay()
            self.ev_done[s].record(self.compute)
        self.copy_out.wait_event(self.ev_done[s])
        with torch.cuda.stream(self.copy_out):
            out_host.copy_(self.out[s ^ 1], non_blocking=True)
            self.ev_out[s].record(self.copy_out)
        return self.ev_out[s]

    def drain(self, out_host=None):
        """Encoder of the last submitted batch (eager, on the compute stream).  Returns its device output; also copies it
        to `out_host` when given."""
        s = (self._i - 1) % 2
        with torch.no_grad(), torch.cuda.stream(self.compute):
            self.compute.wait_event(self.ev_out[s ^ 1])
            # nothing co-runs with this last encoder pass: the module's own (full-width, fastest) launch form instead
            # of the 32-SM interleaved one the steady state uses — 195 vs 313 us at the BASELINE batch, same bits
            out, = self.encoder._forward_eval(self.feat, self.lengths, x16=self.feat16[s], cluster_size=0,
                                              groups_per_cluster=1)
            if out_host is not None:
                out_host.copy_(out, non_blocking=True)
        return out
