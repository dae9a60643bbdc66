"""Drop-in replacement for the reference visual frontend (transformer/video_frontend.py).

Same public names, constructor arguments, attributes and state-dict keys/shapes as the reference
(`Lipreading`, `ResNet`, `BasicBlock`, `conv3x3`, `visual_frontend`), so checkpoints load unchanged and
`Transformer` (transformer/transformer.py:11,34,57) runs on top of it.  The torch.nn submodules below are
parameter HOLDERS only (they give identical initialisation, key names and pickling); the forward pass
never calls them — it runs the hand-written sm_100a kernels of libsblk through `ops`:

    prep_clip -> conv3d+BN+ReLU+maxpool (tcgen05) -> 8 BasicBlocks as implicit-GEMM convs (tcgen05, TMA im2col,
    folded BN, fused residual/ReLU) -> global average pool -> always-on dropout(0.5) -> view [N,T,512]

Reference line citations are relative to SBL_Multilingual_Lip_reading/transformer/video_frontend.py.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


def conv3x3(in_planes, out_planes, stride=1):
    """Parameter holder identical to reference conv3x3 (:10-12)."""
    return nn.Conv2d(in_planes, out_planes, kernel_size=3, stride=stride, padding=1, bias=False)


class BasicBlock(nn.Module):
    """State-dict-compatible holder of reference BasicBlock (:15-41)."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = conv3x3(inplanes, planes, stride)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = conv3x3(planes, planes)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):  # pragma: no cover - the fused path in Lipreading is the only forward
        raise RuntimeError("BasicBlock is a parameter holder; call Lipreading.forward (libsblk kernels)")


class ResNet(nn.Module):
    """State-dict-compatible holder of reference ResNet trunk without stem (:44-89)."""

    def __init__(self, block, layers):
        self.inplanes = 64
        super().__init__()
        self.layer1 = self._make_layer(block, 64, layers[0])
        self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
        self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
        self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        for m in self.modules():  # same init as reference :54-63
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
            elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def _make_layer(self, block, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(
                nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride, bias=False),
                nn.BatchNorm2d(planes * block.expansion),
            )
        layers = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        for _ in range(1, blocks):
            layers.append(block(self.inplanes, planes))
        return nn.Sequential(*layers)

    def forward(self, x):  # pragma: no cover
        raise RuntimeError("ResNet is a parameter holder; call Lipreading.forward (libsblk kernels)")


class _PackedFrontend:
    """BN-folded, bf16, K-major copies of the frontend weights (a cache, never part of the state dict)."""
    __slots__ = ("key", "c3w", "c3b", "blocks")


class Lipreading(nn.Module):
    """Drop-in for reference Lipreading (:91-157): forward(x[N,1,T,88,88] fp32) -> [N,T,512] fp32.

    `always_on_dropout` (default True) reproduces the reference quirk `F.dropout(x, p=0.5)` with the functional
    default training=True (:122): the dropout is active even under model.eval().  It is applied with the very
    same torch call on the pooled features so a seeded CUDA reference run draws the identical mask; set it to
    False for deterministic parity runs (the reference side is then compared through `_frontend_forward`).
    """

    def __init__(self, hiddenDim=512, embedSize=256):
        super().__init__()
        self.inputDim = 512
        self.hiddenDim = hiddenDim
        self.embedSize = embedSize
        self.nLayers = 3
        self.frontend3D = nn.Sequential(
            nn.Conv3d(1, 64, kernel_size=(5, 7, 7), stride=(1, 2, 2), padding=(2, 3, 3), bias=False),
            nn.BatchNorm3d(64),
            nn.ReLU(True),
            nn.MaxPool3d(kernel_size=(1, 3, 3), stride=(1, 2, 2), padding=(0, 1, 1)),
        )
        self.resnet18 = ResNet(BasicBlock, [2, 2, 2, 2])
        self._initialize_weights()
        self.always_on_dropout = True
        self._packed = None
        self._flat_ws = {}
        self._streams = {}
        self._lut = {}
        # L2 weight prefetch on a side stream (see _frontend_forward): layers 1-2 while the stem runs, layers 3-4 when
        # layer 3 starts.  The eager default; the CUDA-graph plans pass their own choice per call.
        self.l2_prefetch = True
        # eval path: clip prep fused into the stem kernel (sblk_stem_fused_fwd: the stem's producer warps build the
        # row-Toeplitz entries from the fp32 clip, no prepped copy of the clip in HBM, one launch less; bit-identical).
        # Measured (tools/exp/stem_fused_probe.py, head_frac_probe.py): fp32 clips 91.1 -> 86.7 us alone, pipelined step
        # 661.5 -> 651.3 us; raw uint8 frames 93.2 -> 122.9 us (16 byte loads + 16 table look-ups per work item), so the
        # uint8 path keeps the separate prep launch unless fuse_prep_u8 is set
        self.fuse_prep = True
        self.fuse_prep_u8 = False
        # eval path, layers 3-4: the block head's 1x1 downsample branch is folded into the block's conv2 as a K-extension
        # (sblk_conv2d_igemm_ext_fwd): conv1 then runs as a plain stride-2 conv on 256-wide pair tiles (the dual kernel
        # is limited to 128-wide tiles by its second accumulator, i.e. 1.5x the operand bytes per FLOP of a path that is
        # bound by L2->SM operand delivery), and the branch is added in fp32 inside conv2's accumulator instead of
        # being rounded to bf16 and read back as a residual.  False = the dual head kernel of round 1.
        self.fold_downsample = True
        # layers 1-2: consecutive flat convs walk their tiles in alternating directions (ops.conv3x3_flat reverse=):
        # each conv starts on the rows the previous launch touched last, the part of a 65.6 MB tensor that is still in
        # L2 (bit-identical; measured in DESIGN.md "[r2d] Alternating tile direction")
        self.alternate_tile_order = True
        # eval path, layers 3-4: a whole residual block as ONE launch (ops.conv_block: pair tiles of whole frames go through
        # conv1 and conv2 without any dependency on other frames) — one launch boundary less per block; bit-identical
        # to the two launches.  fuse_blocks_max: widest block that is fused.  256 = layer 3 only: a layer-4 block (512
        # channels = two column tiles per frame group on neighbouring CTA pairs) has ONE work unit per pair at the BASELINE
        # batch, so the conv1 -> conv2 hand-over is exposed and the single launch is no faster than two (measured:
        # 45.7 vs 45.7 us and 58.0 vs 56.7 us per block, tools/exp/fuse_blocks_probe.py)
        self.fuse_blocks = True
        self.fuse_blocks_max = 256

    # ---- pickling / state: the packed cache holds plain tensors but is cheap to rebuild; drop it ----------
    def __getstate__(self):
        st = self.__dict__.copy()
        st["_packed"] = None
        st["_flat_ws"] = {}
        st["_streams"] = {}
        st["_lut"] = {}
        return st

    # attributes of modules pickled by earlier versions that nothing reads any more (the plans' former hooks, the
    # retired multi-chain frontend)
    _RETIRED = ("parallel_chains", "chain_sm_limit", "l2_prefetch_extra", "_overlap", "_tail", "_block_hook")

    def __setstate__(self, st):
        self.__dict__.update({k: v for k, v in st.items() if k not in self._RETIRED})
        self.__dict__.setdefault("_flat_ws", {})
        self.__dict__.setdefault("_streams", {})
        self.__dict__.setdefault("_lut", {})
        self.__dict__.setdefault("l2_prefetch", True)
        self.__dict__.setdefault("fuse_prep", True)
        self.__dict__.setdefault("fuse_prep_u8", False)
        self.__dict__.setdefault("fold_downsample", True)
        self.__dict__.setdefault("alternate_tile_order", True)
        self.__dict__.setdefault("fuse_blocks", True)
        self.__dict__.setdefault("fuse_blocks_max", 256)

    def _initialize_weights(self):  # same as reference :127-157
        for m in self.modules():
            if isinstance(m, nn.Conv3d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.kernel_size[2] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, nn.Conv1d):
                n = m.kernel_size[0] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, (nn.BatchNorm3d, nn.BatchNorm2d, nn.BatchNorm1d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    # ------------------------------------------------------------------------------------------
    def _cache_key(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def invalidate_packed(self):
        """Drop the packed (bf16 / enc16, BN-folded) weight cache.  The cache key is (data_ptr, tensor._version) of every
        parameter and buffer, which `load_state_dict`, optimizer steps and `.to()` all change; edits THROUGH `.data`
        (`p.data.copy_()`, `m.weight.data.normal_()`) do not bump the version counter, so call this after them."""
        self._packed = None

    def _apply(self, fn, *args, **kwargs):
        self._packed = None
        return super()._apply(fn, *args, **kwargs)

    def _get_packed(self):
        key = self._cache_key()
        pk = self._packed
        if pk is not None and pk.key == key:
            return pk
        pk = _PackedFrontend()
        pk.key = key
        conv, bn = self.frontend3D[0], self.frontend3D[1]
        pk.c3w, pk.c3b = ops.pack_conv3d(conv.weight.detach().contiguous(), bn.weight.detach(), bn.bias.detach(),
                                         bn.running_mean, bn.running_var, bn.eps)

        def fold(c, b):
            return ops.pack_conv2d(c.weight.detach().contiguous(), b.weight.detach(), b.bias.detach(),
                                   b.running_mean, b.running_var, b.eps)

        pk.blocks = []
        for layer in (self.resnet18.layer1, self.resnet18.layer2, self.resnet18.layer3, self.resnet18.layer4):
            for blk in layer:
                w1, b1 = fold(blk.conv1, blk.bn1)
                w2, b2 = fold(blk.conv2, blk.bn2)
                ds = fold(blk.downsample[0], blk.downsample[1]) if blk.downsample is not None else None
                if ds is not None:   # (filter, shift, bn2 shift + downsample shift: bias of the folded form)
                    ds = (ds[0], ds[1], (b2 + ds[1]).contiguous())
                # layer1 / layer2 run on the zero-haloed flat layout (shifted-window kernels): [C, 10*C] packing
                flat = layer is self.resnet18.layer1 or layer is self.resnet18.layer2
                if flat and blk.stride == 1:
                    w1 = ops.pack_flat_weight(w1)
                if flat:
                    w2 = ops.pack_flat_weight(w2)
                pk.blocks.append((blk.stride, w1, b1, w2, b2, ds))
        self._packed = pk
        return pk

    def _flat_workspace(self, a, cout, stride):
        """Two zero-initialised flat buffers for the outputs of a strided block head.  Only pixel rows are ever written
        (sblk_conv2d_dual_igemm_fwd, flat_out), so the halo rows stay zero across calls; cached per (device, shape)."""
        f, h, w_ = (a.f, a.h, a.w) if isinstance(a, ops.FlatActs) else a.shape[:3]
        p, q = (h - 1) // stride + 1, (w_ - 1) // stride + 1
        key = (str(a.data.device if isinstance(a, ops.FlatActs) else a.device), f, p, q, cout)
        ws = self._flat_ws.get(key)
        if ws is None:
            if len(self._flat_ws) > 16:   # (plans pin the entries their graphs use: runner._pin_captured_state)
                self._flat_ws.clear()
            dev = a.data.device if isinstance(a, ops.FlatActs) else a.device
            ws = tuple(torch.zeros((ops.flat_rows(f, p, q), cout), dtype=torch.bfloat16, device=dev) for _ in range(2))
            self._flat_ws[key] = ws
        return ws

    def _check_input(self, x):
        if x.dim() != 5 or x.size(1) != 1 or x.size(3) != 88 or x.size(4) != 88:
            raise RuntimeError(f"Lipreading expects [N,1,T,88,88], got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("Lipreading (libsblk) runs on a B200 CUDA device only; no CPU fallback exists")
        if x.dtype != torch.float32:
            x = x.float()
        x = x.contiguous()
        if x.data_ptr() % 16:     # a contiguous view at an odd storage offset: the kernels read 16-byte vectors
            x = x.clone()
        return x

    def _prefetch_stream(self, device):
        key = str(device)
        if key not in self._streams:
            self._streams[key] = torch.cuda.Stream(device=device)
        return self._streams[key]

    def _frontend_forward(self, x, prep=ops.prep_clip, frames=None, *, head_sm_limit=None, out16=None, **schedule):
        """reference :111-117 — prep -> Conv3d stem -> ResNet-18 trunk -> average pool on the current stream; returns the
        pooled features [N*T,512] fp32 (before the always-on dropout).  `prep` turns `x` into the stem's prepped layout
        (fp32 clips: ops.prep_clip; raw uint8 frames with `frames` output frames: the closure of _u8_prep).

        The keyword arguments (these two and those of _trunk) are the schedule of the CUDA-graph plans (runner.py);
        unset, they mean the eager path.
        * head_sm_limit (0 = all SMs): the clip prep, the stem and the first `head_blocks` residual blocks size their
          persistent grids for that many SMs because another kernel chain (the previous batch's encoder stack) co-runs
          on the other SMs; `head_join()` is called once the head is enqueued and makes the current stream wait for that
          chain before the full-width kernels start.  head_frac > 0: that share of the frames of the first conv after
          the head still runs inside it.
        * out16: the pooling launch writes mean * `scale` (the always-on dropout's factor drawn ahead of time, or None)
          straight into this 16-bit encoder operand instead of the fp32 features (bit-identical), after `before_pool()`
          has been called; returns None.
        * hook(): called on the current stream right before residual block `hook_block` is enqueued.
        * prefetch (default: the module's l2_prefetch): L2 weight hints on a side stream; the tensors of `prefetch_extra`
          (the encoder's packed weights) are hinted when layer 4 starts."""
        if frames is None:
            x = self._check_input(x)
            n, t = x.shape[0], x.shape[2]
        else:           # raw uint8 frames, already validated by _u8_prep
            n, t = x.shape[0], frames
        pk = self._get_packed()
        with torch.cuda.device(x.device):
            feat = None if out16 is not None else torch.empty((n * t, self.inputDim), dtype=torch.float32,
                                                               device=x.device)
            head = [] if head_sm_limit is None else [ops.set_sm_limit(head_sm_limit)]   # the limit to restore
            try:
                self._trunk(x, pk, prep, feat, out16, head, **schedule)
            finally:
                if head:
                    ops.set_sm_limit(head.pop())
        return feat

    def _trunk(self, x, pk, prep, feat, out16, head, *, head_blocks=0, head_join=None, head_frac=0.0, scale=None,
               before_pool=None, hook=None, hook_block=0, prefetch=None, prefetch_extra=()):
        if hook is not None and not 0 <= hook_block < len(pk.blocks):
            raise RuntimeError(f"hook_block={hook_block}: the trunk has residual blocks 0..{len(pk.blocks) - 1}")
        if prefetch is None:
            prefetch = self.l2_prefetch

        def end_head():   # back to full-width grids; the co-running chain must be finished before they start
            ops.set_sm_limit(head.pop())
            head_join()

        # fuse_prep: the stem's producer warps build the row-Toeplitz entries themselves (ops.RawClip) instead of reading
        # a prepped copy of the clip written by a separate launch (bit-identical)
        xp = ops.raw_clip(x) if (self.fuse_prep and prep is ops.prep_clip) else prep(x)
        # layer1 / layer2 run on the zero-haloed flat layout (flat shifted-window kernels);
        # from layer3 on, activations are dense NHWC and the convs are TMA-im2col implicit GEMMs
        a = ops.conv3d_bn_relu_pool(xp, pk.c3w, pk.c3b, flat=True)
        pf_stream = None
        rev = [False]   # direction of the previous flat launch (the stem writes its output front to back)

        def flip():
            rev[0] = (not rev[0]) if self.alternate_tile_order else False
            return rev[0]
        for bi, (stride, w1, b1, w2, b2, ds) in enumerate(pk.blocks):
            split = 0
            if head and bi == head_blocks:
                # head_frac > 0: the first conv of this block is run in two frame ranges — the first one still inside
                # the head (limited width, next to the other chain), the rest at full width — to use the time by which
                # the other chain outlasts the head.  Frame ranges of the flat layout are independent (ops.flat_frames).
                if head_frac > 0 and isinstance(a, ops.FlatActs) and stride == 1 and ds is None and a.f >= 2:
                    split = min(a.f - 1, max(1, int(round(a.f * float(head_frac)))))
                    y = ops.FlatActs(torch.empty_like(a.data), a.f, a.h, a.w)
                    split_rev = flip()
                    ops.conv3x3_flat(ops.flat_frames(a, 0, split), w1, b1, relu=True,
                                     out=ops.flat_frames(y, 0, split).data, reverse=split_rev)
                end_head()
            if hook is not None and bi == hook_block:
                hook()
            if prefetch and bi in (0, 4, 6):
                # Weights of the layers still to come are pulled into L2 by a tiny kernel on a side stream while the
                # current layer computes (layers 3-4 move few activation bytes, so the lines survive).  Benchmarks flush
                # L2 between forwards and a serving loop evicts the 61 MB of weights with ~600 MB of activations per
                # batch: without this, every kernel's first weight tiles and the encoder stack's whole dependent chain
                # of weight loads pay DRAM latency.
                if bi == 6:
                    tensors = list(prefetch_extra)
                else:   # layers 1-2 (1.5 MB) while the stem runs, layers 3-4 (28 MB) when layer 3 starts
                    tensors = [t_ for blk in (pk.blocks[:4] if bi == 0 else pk.blocks[4:])
                               for t_ in (blk[1], blk[3]) + (tuple(blk[5][:1]) if blk[5] else ())]
                if tensors:
                    main = torch.cuda.current_stream()
                    if pf_stream is None:
                        pf_stream = self._prefetch_stream(x.device)
                    ev = torch.cuda.Event()
                    ev.record(main)
                    pf_stream.wait_event(ev)
                    with torch.cuda.stream(pf_stream):
                        ops.l2_prefetch(tensors)
            if isinstance(a, ops.FlatActs) and stride == 1 and ds is None:
                if split:
                    ops.conv3x3_flat(ops.flat_frames(a, split, a.f), w1, b1, relu=True,
                                     out=ops.flat_frames(y, split, a.f).data, reverse=split_rev)
                else:
                    y = ops.conv3x3_flat(a, w1, b1, relu=True, reverse=flip())
                a = ops.conv3x3_flat(y, w2, b2, relu=True, residual=a, reverse=flip())
                continue
            if ds is not None:   # conv1 and the 1x1 downsample branch share one pass over the block input
                if w2.dim() == 2:  # layer2: the block stays in the flat layout (conv2 is a flat stride-1 conv)
                    y, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=stride, relu=True,
                                             flat_ws=self._flat_workspace(a, w1.shape[0], stride))
                    rev[0] = False   # the dual head writes its tiles front to back
                    a = ops.conv3x3_flat(y, w2, b2, relu=True, residual=res, reverse=flip())
                    continue
                if self.fold_downsample and self.fuse_blocks and w1.shape[0] in (256, 512) and w1.shape[0] <= self.fuse_blocks_max:
                    fused = ops.conv_block(a, w1, b1, w2, ds[2], w_ds=ds[0], stride=stride)
                    if fused is not None:
                        a = fused
                        continue
                if self.fold_downsample:
                    # y = relu(bn1(conv1 x)); out = relu(bn2(conv2 y) + bn_ds(ds x)) in one fp32 accumulator
                    y = ops.conv2d(a, w1, b1, stride=stride, relu=True)
                    a = ops.conv2d(y, w2, ds[2], stride=1, relu=True, ext=(a, ds[0], stride))
                    continue
                y, res = ops.conv2d_dual(a, w1, b1, ds[0], ds[1], stride=stride, relu=True)
            else:
                if (self.fuse_blocks and w1.shape[0] in (256, 512) and w1.shape[0] <= self.fuse_blocks_max and stride == 1
                        and not isinstance(a, ops.FlatActs) and a.shape[-1] == w1.shape[0]):
                    fused = ops.conv_block(a, w1, b1, w2, b2, stride=1)
                    if fused is not None:
                        a = fused
                        continue
                y, res = ops.conv2d(a, w1, b1, stride=stride, relu=True), a
            a = ops.conv2d(y, w2, b2, stride=1, relu=True, residual=res)
        if head:   # the whole trunk ran inside the head
            end_head()
        if out16 is not None:
            if before_pool is not None:
                before_pool()
            ops.avgpool(a, want_f32=False, out_bf16=out16, scale=scale, enc16=True)
        else:
            ops.avgpool(a, out_f32=feat)
        if pf_stream is not None:   # join (graph capture needs every forked stream back; no data dependency)
            ev = torch.cuda.Event()
            ev.record(pf_stream)
            torch.cuda.current_stream().wait_event(ev)

    def _u8_prep(self, x_u8, frames, crop):
        """Checks forward_u8's arguments; returns (x_u8, output frames, the prep closure for _frontend_forward)."""
        if self.training:
            raise RuntimeError("Lipreading.forward_u8 (libsblk) is the evaluation / serving input path; training runs "
                               "through forward() on the loader's augmented fp32 clips")
        if not torch.is_tensor(x_u8) or x_u8.dtype != torch.uint8 or x_u8.dim() != 4:
            raise RuntimeError("forward_u8 expects a uint8 tensor [N, T, H0, W0]")
        if not x_u8.is_cuda:
            raise RuntimeError("Lipreading (libsblk) runs on a B200 CUDA device only; no CPU fallback exists")
        x_u8 = x_u8.contiguous()
        t_out = x_u8.shape[1] if frames is None else int(frames)
        if t_out < x_u8.shape[1]:
            raise RuntimeError(f"forward_u8: frames={t_out} < clip length {x_u8.shape[1]}")
        key = str(x_u8.device)
        lut = self._lut.get(key)
        if lut is None:
            from . import synth
            lut = self._lut[key] = synth.normalize_lut().to(x_u8.device)
        if torch.is_tensor(crop):
            crop = crop.to(device=x_u8.device, dtype=torch.int32).contiguous()

        def prep(xs):
            if self.fuse_prep_u8:
                return ops.raw_clip_u8(xs, lut, t_out, crop)
            return ops.prep_clip_u8(xs, lut, t_out, crop)
        return x_u8, t_out, prep

    def forward_u8(self, x_u8, frames=None, crop=(4, 4)):
        """Fused input pipeline (SURVEY.md §8f.3): raw uint8 gray frames [N, T_in, H0, W0] (the loader's .npy layout,
        H0 = W0 = 96 for LRW) -> the same [N, frames, 512] features `forward` returns for the clip the reference loader
        would have built on the CPU (/255, ColorNormalize, 88x88 crop at `crop`, zero-padding to `frames` frames:
        data_gen.py:122-125,276-296; cvtransforms.py:7-48).  `crop`: (y1, x1) or an int32 CUDA tensor [N*T_in, 2] of
        per-frame offsets (RandomCrop).  Bit-identical to forward(reference-normalised fp32 clip); 4x fewer host->device
        bytes."""
        x_u8, t_out, prep = self._u8_prep(x_u8, frames, crop)
        feat = self._frontend_forward(x_u8, prep=prep, frames=t_out)
        if self.always_on_dropout:
            feat = F.dropout(feat, p=0.5)  # functional default training=True, exactly as reference :122
        return feat.view(-1, t_out, self.inputDim)

    def train(self, mode=True):
        # training updates the BatchNorm running statistics in place from a kernel (no torch version bump): the
        # BN-folded evaluation weights are re-packed whenever the mode changes
        self._packed = None
        return super().train(mode)

    def forward(self, x):
        """reference :119-125.  model.train(): BatchNorm on batch statistics + autograd through libsblk
        (training.py); model.eval(): running statistics folded into the kernels, output detached from autograd."""
        frameLen = x.size(2)
        if x.size(0) == 0:   # empty batch (the reference returns an empty tensor as well): nothing to launch
            self._check_input(x)
            return x.new_zeros((0, frameLen, self.inputDim), dtype=torch.float32)
        if self.training:
            from . import training
            feat = training.frontend_forward_train(self, self._check_input(x))
            feat = F.dropout(feat, p=0.5)  # reference :122 (functional default training=True); torch autograd
            return feat.view(-1, frameLen, self.inputDim)
        feat = self._frontend_forward(x)
        if self.always_on_dropout:
            feat = F.dropout(feat, p=0.5)  # functional default training=True, exactly as reference :122
        return feat.view(-1, frameLen, self.inputDim)


device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')  # reference :174


def visual_frontend(pt=None):
    """Factory identical to reference visual_frontend (:176-190): optional partial state-dict load."""
    model = Lipreading(hiddenDim=512, embedSize=256)
    if pt is not None:
        model_dict = model.state_dict()
        pretrained_dict = torch.load(pt, map_location=device)
        print(len(pretrained_dict))
        pretrained_dict = {k: v for k, v in pretrained_dict.items()
                           if k in model_dict.keys() and v.size() == model_dict[k].size()}
        print('loaded params/tot params:{}/{}'.format(len(pretrained_dict), len(model_dict)))
        model_dict.update(pretrained_dict)
        model.load_state_dict(model_dict)
    return model
