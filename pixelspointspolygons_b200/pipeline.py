"""Host-fed serving loop of the hot path: pinned staging slots -> H2D -> LAS arithmetic -> encoder -> result.

The reference feeds the encoder from a DataLoader: laspy decodes a tile, `P3Dataset.load_lidar_points`
(R:pixelspointspolygons/datasets/p3_coco.py:74-101) turns it into fp32 pixel-space points on the CPU, the collate
function builds the jagged batch (R:pixelspointspolygons/datasets/collate_funcs.py:108) and the trainer / predictor moves
it to the device before `encoder(x_image, x_lidar)`.  `HostPipeline` is that loop for a GPU whose kernels are an order of
magnitude faster than the PCIe link: the loader writes what the LAS file holds (integer coordinates as uint16 deltas + an
int32 base per tile, 6 bytes per point; the tile headers; optionally the fp32 image) straight into a pinned staging slot,
and per batch the host issues

    copy stream     H2D(slot s + 1)          one copy of the slot's whole arena
    compute stream  compute(slot s)          ONE CUDA-graph launch: las_packed_to_pixels -> voxelize -> PFN (-> patch embed,
                                             concat, fusion_layer) (-> the caller's reduction -> pinned result)
    return stream   D2H(result of slot s-1)  optional, the full output tensor

ordered by events only where data flows, so that both copy engines and the SMs are busy at the same time (the step time is
the longest of the three: at B = 16 x 100 k points the 9.6 MB copy, 177 us at 54 GB/s) and the host spends ~30 us per batch.
Results are bit-identical to calling `las_packed_to_pixels` + the module on the same batch
(tests/test_gpu_pipeline.py).  Batches have a fixed shape (B tiles, `total` points in all; the split of the points over the
tiles is data and may change from batch to batch), as a captured graph demands.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence

import torch

from . import _lib
from ._lib import P3P_LAYOUT_NLC
from .encoder import PointPillarsEncoder
from .las import LasPackedFrontEnd, tile_meta_bytes


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


class Slot:
    """Pinned host views of one staging slot (what the loader fills) and the device tensors its results land in."""

    def __init__(self, index):
        self.index = index
        self.deltas: torch.Tensor = None   # (total, 3) uint16   X - base (pack_las)
        self.base: torch.Tensor = None     # (B, 3) int32
        self.offsets: torch.Tensor = None  # (B + 1) int64
        self.meta: torch.Tensor = None     # (B * sizeof(p3p_las_tile)) uint8: written by set_tiles
        self.image: Optional[torch.Tensor] = None  # (B, 3, H, W) float32 (fusion workloads)
        self.out: torch.Tensor = None      # device: the module's output for this slot
        self.host_out: Optional[torch.Tensor] = None    # pinned: full copy of `out` (host_result = "full")
        self.host_value: Optional[torch.Tensor] = None  # pinned: reduce(out) (host_result = callable)
        self.done: torch.cuda.Event = None  # recorded after the graph that produced out / host_value
        self.host_done: torch.cuda.Event = None  # recorded after the graph that filled host_out


class HostPipeline:
    """module: a `PointPillarsEncoder` (LiDAR-only; output (B, ny nx, C) token rows) or an `EarlyFusionFrontEnd`
    (`mode` = "concat": (B, 2C, ny, nx); "tokens": through `fusion_layer`, (B, ny nx, C); "vit_tokens": the ViT's input
    sequence (B, 1 + ny nx, C) with `cls_token` (1, 1, C) and `pos_embed` (1, 1 + ny nx, C), see
    `EarlyFusionFrontEnd.forward_tokens`), in eval mode on a CUDA device.

    In "vit_tokens" mode the captured graphs read `cls_token` and `pos_embed` where they are in device memory (they must
    be contiguous float32 on the module's device): an in-place update -- an optimizer step, `load_state_dict`, `.copy_()`
    -- is seen by the next batch computed, a tensor put in their place (a new `nn.Parameter`, `.to()` elsewhere) is not;
    build a new pipeline for that.

    Use:
        s = pipe.staging()        # the slot to fill next (blocks only if its previous copy is still in flight)
        s.deltas[...] = ...; s.base[...] = ...; s.offsets[...] = ...; pipe.set_tiles(s, headers); s.image[...] = ...
        prev = pipe.submit()      # launches compute(previous batch) ‖ H2D(this batch); returns the previous batch's slot
        prev.done.synchronize(); prev.out / prev.host_value ...
        last = pipe.flush()       # computes the batch submitted last
    """

    def __init__(self, module, B: int, total: int, slots: int = 3, mode: str = "tokens", image_hw: Sequence[int] = (224, 224),
                 host_result=None, z_hi: float = 100.0, variant: str = "dataset", cls_token: Optional[torch.Tensor] = None,
                 pos_embed: Optional[torch.Tensor] = None):
        if slots < 2:
            raise ValueError("at least two slots (one in compute, one in copy)")
        p = next(module.parameters())
        if not p.is_cuda:
            raise RuntimeError("HostPipeline runs on CUDA only (sm_100a); the module is on " + str(p.device))
        if module.training:
            raise RuntimeError("HostPipeline captures the eval-mode kernels: call module.eval() first")
        self.module, self.B, self.total, self.n, self.variant = module, int(B), int(total), int(slots), variant
        self.device = dev = p.device
        self.fusion = not isinstance(module, PointPillarsEncoder)
        self.mode = mode if self.fusion else "lidar"
        if self.fusion and mode not in ("concat", "tokens", "vit_tokens"):
            raise ValueError("mode must be 'concat', 'tokens' or 'vit_tokens'")
        enc = module.lidar_embed if self.fusion else module
        hw, Cc = enc.ny * enc.nx, enc.channels
        self._cls = self._pos = None
        if self.mode == "vit_tokens":
            if cls_token is None or pos_embed is None:
                raise ValueError("mode 'vit_tokens' needs cls_token and pos_embed")
            for name, t in (("cls_token", cls_token), ("pos_embed", pos_embed)):
                if t.dtype != torch.float32 or t.device != dev or not t.is_contiguous():
                    raise TypeError(f"{name} must be a contiguous float32 tensor on {dev} (the graphs read it in place)")
            self._cls, self._pos = cls_token, pos_embed
        elif cls_token is not None or pos_embed is not None:
            raise ValueError("cls_token / pos_embed belong to mode 'vit_tokens'")
        self._full = host_result == "full"
        self._reduce: Optional[Callable] = host_result if callable(host_result) else None
        if host_result is not None and not (self._full or self._reduce):
            raise ValueError("host_result must be None, 'full' or a callable")

        # ---- one arena per slot: [deltas | base | offsets | meta | image], the same layout on both sides -----------------
        tile_bytes = C.sizeof(_lib.LasTile)
        H, W = int(image_hw[0]), int(image_hw[1])
        sizes = [("deltas", self.total * 6), ("base", self.B * 12), ("offsets", (self.B + 1) * 8), ("meta", self.B * tile_bytes)]
        if self.fusion:
            sizes.append(("image", self.B * 3 * H * W * 4))
        self._off, pos = {}, 0
        for name, nb in sizes:
            self._off[name] = (pos, nb)
            pos += _align(nb)
        self.arena_bytes = pos

        def views(arena, slot: Optional[Slot]):
            def v(name, dtype, shape):
                o, nb = self._off[name]
                return arena[o:o + nb].view(dtype).view(*shape)
            d = dict(deltas=v("deltas", torch.uint16, (self.total, 3)), base=v("base", torch.int32, (self.B, 3)),
                     offsets=v("offsets", torch.int64, (self.B + 1,)), meta=v("meta", torch.uint8, (self.B * tile_bytes,)),
                     image=v("image", torch.float32, (self.B, 3, H, W)) if self.fusion else None)
            if slot is not None:
                for k, t in d.items():
                    setattr(slot, k, t)
            return d

        self.slots: List[Slot] = []
        self._host, self._dev, self._dviews = [], [], []
        for i in range(self.n):
            s = Slot(i)
            host = torch.zeros(self.arena_bytes, dtype=torch.uint8).pin_memory()
            devt = torch.empty(self.arena_bytes, dtype=torch.uint8, device=dev)
            views(host, s)
            s.offsets.copy_(torch.arange(self.B + 1, dtype=torch.int64) * (self.total // max(self.B, 1)))
            s.offsets[self.B] = self.total
            if self.mode == "concat":
                s.out = torch.empty(self.B, 2 * Cc, enc.ny, enc.nx, dtype=torch.float32, device=dev)
            elif self.mode == "vit_tokens":
                s.out = torch.empty(self.B, 1 + hw, Cc, dtype=torch.float32, device=dev)
            else:
                s.out = torch.empty(self.B, hw, Cc, dtype=torch.float32, device=dev)
            if self._full:
                s.host_out = torch.empty(s.out.shape, dtype=torch.float32).pin_memory()
            s.done, s.host_done = torch.cuda.Event(), torch.cuda.Event()
            self.slots.append(s)
            self._host.append(host)
            self._dev.append(devt)
            self._dviews.append(views(devt, None))
        self._x16 = None
        if self.mode in ("tokens", "vit_tokens"):
            self._x16 = torch.empty(self.B, enc.ny, enc.nx, 2 * Cc, dtype=module.fusion_layer.operand_dtype, device=dev)
        # the LAS arithmetic's per-tile constants come from the slot's own arena (set_tiles), not from a fixed table
        self._fe = LasPackedFrontEnd([], self.total, dev, z_hi, variant, B=self.B)
        self._x = [torch.nested.nested_tensor_from_jagged(self._fe.out, d["offsets"]) for d in self._dviews]
        self.stream = torch.cuda.Stream(dev)      # compute: one graph launch per batch
        self._copy = torch.cuda.Stream(dev)       # H2D of the slots' arenas
        self._back = torch.cuda.Stream(dev)       # D2H of the full outputs (host_result = "full")
        self._copied = [torch.cuda.Event() for _ in range(self.n)]  # slot's arena has reached the device
        self._used = [torch.cuda.Event() for _ in range(self.n)]    # slot's device arena has been consumed by its compute
        self._graphs: List[Optional[torch.cuda.CUDAGraph]] = [None] * self.n
        self._filled = -1     # slot handed out by staging() and not yet submitted
        self._pending = -1    # slot submitted last: on the device (or on its way), not yet computed
        self._next = 0
        self.launches = 0
        # a warm-up pass outside capture (lazy allocations: workspace, weight blobs), then one compute graph per slot
        for s in self.slots:
            self.set_tiles(s, [dict(scales=(1.0, 1.0, 1.0), offsets=(0.0, 0.0, 0.0), top_left=(0.0, 0.0), height=H, width=W)] * self.B)
        with torch.cuda.stream(self.stream):
            self._dev[0].copy_(self._host[0], non_blocking=True)
            self._compute(0)
        self.stream.synchronize()
        for i in range(self.n):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                self._compute(i)
            self._graphs[i] = g
        torch.cuda.synchronize(dev)

    # ------------------------------------------------------------------ pieces
    def set_tiles(self, slot: Slot, tiles: Sequence[dict]):
        """Write the tiles' LAS headers / image geometry (the dicts `las_to_pixels` takes) into the slot's arena."""
        if len(tiles) != self.B:
            raise ValueError(f"{len(tiles)} tile headers for a pipeline of {self.B} tiles")
        raw = tile_meta_bytes(tiles, self.variant)
        slot.meta.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))

    def _compute(self, i: int):
        d, s, m = self._dviews[i], self.slots[i], self.module
        self._fe(d["deltas"], d["base"], d["offsets"], meta=d["meta"])
        x = self._x[i]  # (the jagged view of the front end's output buffer with this slot's offsets)
        if self.mode == "lidar":
            m.encode_into(x, s.out, P3P_LAYOUT_NLC)
        elif self.mode == "concat":
            m.forward_into(d["image"], x, s.out, lidar_zero=False)
        elif self.mode == "tokens":
            m.forward_tokens_into(d["image"], x, self._x16, s.out, lidar_zero=False)
        else:
            m.forward_tokens_into(d["image"], x, self._x16, s.out, lidar_zero=False, cls_token=self._cls, pos_embed=self._pos)
        if self._reduce is not None:
            r = self._reduce(s.out)
            if s.host_value is None:
                s.host_value = torch.empty(r.shape, dtype=r.dtype).pin_memory()
            s.host_value.copy_(r, non_blocking=True)

    # ------------------------------------------------------------------ the loop
    def staging(self) -> Slot:
        """The slot to fill next.  Its previous contents have reached the device before this returns."""
        if self._filled >= 0:
            raise RuntimeError("staging() called twice without submit()")
        i = self._next
        self._copied[i].synchronize()  # (no-op unless the ring is shorter than the work in flight)
        self._filled = i
        return self.slots[i]

    def _launch_compute(self, k: int) -> Slot:
        s = self.slots[k]
        self.stream.wait_event(self._copied[k])
        if self._full:
            self.stream.wait_event(s.host_done)  # (the previous ring cycle's copy of this slot's `out`, about to be rewritten)
        with torch.cuda.stream(self.stream):
            self._graphs[k].replay()
        self.launches += 1
        self._used[k].record(self.stream)
        s.done.record(self.stream)
        if self._full:  # the whole output goes back on its own stream, next to the following batches' copies and kernels
            self._back.wait_event(s.done)
            with torch.cuda.stream(self._back):
                s.host_out.copy_(s.out, non_blocking=True)
            s.host_done.record(self._back)
        return s

    def submit(self) -> Optional[Slot]:
        """The staged slot is complete: its copy is enqueued, and next to it the compute of the batch submitted before it.
        Returns that previous batch's slot (its `done` event says when `out` / `host_value` are ready, `host_done` when
        `host_out` is), or None for the first batch."""
        if self._filled < 0:
            raise RuntimeError("submit() without a staged slot")
        i, prev = self._filled, self._pending
        if prev >= 0 and i != (prev + 1) % self.n:
            raise RuntimeError("slots are submitted in ring order")
        self._filled, self._next = -1, (i + 1) % self.n
        self._copy.wait_event(self._used[i])  # the compute that read this slot's device arena one ring cycle ago
        with torch.cuda.stream(self._copy):
            self._dev[i].copy_(self._host[i], non_blocking=True)
        self._copied[i].record(self._copy)
        self._pending = i
        return self._launch_compute(prev) if prev >= 0 else None

    def flush(self) -> Optional[Slot]:
        """Compute the batch submitted last (nothing left to prefetch)."""
        prev = self._pending
        if prev < 0:
            return None
        self._pending = -1
        return self._launch_compute(prev)

    @property
    def h2d_bytes_per_step(self) -> int:
        return self.arena_bytes

    @property
    def d2h_bytes_per_step(self) -> int:
        s = self.slots[0]
        if self._full:
            return s.out.numel() * 4
        return 0 if s.host_value is None else s.host_value.numel() * s.host_value.element_size()
