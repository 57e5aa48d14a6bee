#!/usr/bin/env python
"""bench.py -- throughput of the LiDAR pillar-encode (+ early-fusion) hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload lidar|fusion]
                    [--dump-outputs DIR]

A step is one pass of the hot path over one batch of synthetic tiles (BASELINE.json configs[1]: Pix2Poly
LiDAR-only, 224 px tiles, 100k points per tile, batch 16 per GPU).  Under torchrun (N > 1) every rank encodes its
own batch (tiles are independent units: no collective on the data path, weak scaling), the step time is the MAX
over ranks and `value` is the whole-job tiles/s.  One JSON line is printed by rank 0.

  value         device-timed (CUDA events) over exactly K steps issued right after W warm-up steps (from the completion
                of the last warm-up step to that of the last timed step), inputs resident in HBM, rotating over
                input/output sets larger than L2
  sustained     the same loop held for >= --min-seconds (clocks sampled inside)
  e2e           same metric through the public module API with HOST pinned inputs: H2D copy of the step's points +
                offsets and a D2H read of the step's result checksum inside the timed region
  roofline      the dominant kernel (PFN tensor-core kernel): algorithmic FLOPs / its CUDA-event duration
  hbm_roofline  whole-path algorithmic bytes * tiles/s over the measured copy bandwidth (BASELINE's "% HBM roofline")
  cpu_baseline  the oracle (CPU restatement of the reference path) timed on the host cores on a bounded sample

`--impl reference` times the reference's CPU implementation of the path: the oracle port (open3d==0.19.0, which
holds the reference's arithmetic, is not installable offline -- DESIGN.md), all host threads, bounded sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "pillar_encode_tiles_per_sec"
UNIT = "tiles/s"
HW = 28 * 28
C_FEAT = 384


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps `value` is taken from (default 20000, ~1 s at B = 16; 200 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="lidar", choices=["lidar", "fusion", "fusion_layer"],
                    help="lidar: voxelize + PFN + scatter -> tokens; fusion: + patch embed -> concat (B, 768, 28, 28); "
                         "fusion_layer: + conv3x3 768 -> 384 + BN + ReLU -> tokens (SURVEY 8f rank 1)")
    ap.add_argument("--batch", type=int, default=16, help="tiles per GPU per step")
    ap.add_argument("--points", type=int, default=100_000, help="points per tile")
    ap.add_argument("--precision", default="fp16", choices=["fp32", "tf32", "fp16", "bf16"])
    ap.add_argument("--max-points-per-voxel", type=int, default=64)
    ap.add_argument("--sets", type=int, default=8, help="rotating input/output sets (must exceed L2 in total)")
    ap.add_argument("--in-flight", type=int, default=2, help="batches in flight: consecutive steps alternate between this many "
                    "streams / workspaces (1 = every step waits for the previous one)")
    ap.add_argument("--no-graph", action="store_true", help="launch through the C ABI every step instead of CUDA graphs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-results", action="store_true", help="skip the secondary configurations (tf32, fusion, density points)")
    ap.add_argument("--min-seconds", type=float, default=2.0, help="length of the sustained timed region (and bound of the e2e ones)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32, rank 0; "
                         "a seeded sample of the tiles when the output exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20_000 if args.impl == "ours" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def algorithmic_bytes_per_tile(n_points, workload):
    """SURVEY 8(d): LiDAR-only 12 N + 4 C ny nx; early fusion 12 N + 4*3*224*224 + 4*768*784 (fp32 I/O)."""
    if workload == "fusion":
        return 12 * n_points + 4 * 3 * 224 * 224 + 4 * 768 * HW
    if workload == "fusion_layer":  # points + image in, fused tokens out (the concat is not an algorithmic output)
        return 12 * n_points + 4 * 3 * 224 * 224 + 4 * C_FEAT * HW
    return 12 * n_points + 4 * C_FEAT * HW


def algorithmic_flops(tiles, M):
    """SURVEY 8(d) minimal exact form: 2*8*32*(K + [Pp>0]) + 2*32*384*(K + Pp) + 2*32*384*P over the batch."""
    K = P = Pp = 0
    for t in tiles:
        cx = np.minimum((t[:, 0] * np.float32(0.125)).astype(np.int64), 28)
        cy = np.minimum((t[:, 1] * np.float32(0.125)).astype(np.int64), 28)
        ok = (cx < 28) & (cy < 28) & (t[:, 2] < 100.0)
        cnt = np.bincount((cy * 28 + cx)[ok], minlength=HW)
        kept = np.minimum(cnt, M)
        K += int(kept.sum())
        P += int((cnt > 0).sum())
        Pp += int(((cnt > 0) & (cnt < M)).sum())
    return 2 * 8 * 32 * (K + (1 if Pp else 0)) + 2 * 32 * C_FEAT * (K + Pp) + 2 * 32 * C_FEAT * P, K, P


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (profiling recipe's clocks line).

    NVML is polled in-process every ~2 ms (the timed region of the default run lasts tens of milliseconds, shorter than
    one `nvidia-smi -lms` period); `nvidia-smi` is the fallback when the NVML binding is missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.stop_flag, self.thread = None, None, False, None
        self.sm, self.mx, self.reason_bits = [], None, 0
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if visible:
                ids = [v.strip() for v in visible.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample(self):
        """One NVML reading (polling thread; it runs while the main thread waits in the closing synchronize of the timed
        region, i.e. while the queued steps execute -- an inline call from the launch loop would stall the launches: an
        NVML query takes milliseconds)."""
        n = self.nvml
        if n is None:
            return
        try:
            self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
            self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            try:
                self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass

    def _poll(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            n = self.nvml
            names = (("hw_slowdown", getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                     ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                     ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                     ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)))
            reasons = sorted(name for name, bit in names if self.reason_bits & int(bit))
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def cpu_oracle_modules(M):
    from oracle import pillars_oracle as po

    grid = po.GridSpec(max_num_points=M)
    enc = po.OraclePointPillarsEncoder(grid).eval()
    sd, sdi = po.synth_weights(0)
    enc.load_state_dict(sd)
    pe = po.OraclePatchEmbed().eval()
    pe.load_state_dict(sdi)
    return po, enc, pe


def cpu_step(po, enc, pe, tiles, images, workload):
    with torch.no_grad():
        if workload == "fusion":
            return po.early_fusion_front(pe, enc, images, tiles)
        return enc(tiles, return_flattened=True)


def run_reference(args, rank, world):
    """Reference arm: the CPU restatement of the reference path on all host threads, bounded sample per step."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    po, enc, pe = cpu_oracle_modules(args.max_points_per_voxel)
    tiles_all = [po.synth_tile(args.points, 1000 + i, clustered=(i % 2 == 1)) for i in range(min(args.batch, 4))]
    img_all = torch.rand(len(tiles_all), 3, 224, 224)
    t0 = time.perf_counter()
    cpu_step(po, enc, pe, tiles_all[:1], img_all[:1], args.workload)
    t_tile = time.perf_counter() - t0
    budget = 150.0
    n = int(max(1, min(len(tiles_all), budget / max(t_tile, 1e-3) / max(args.steps + args.warmup, 1))))
    tiles, images = tiles_all[:n], img_all[:n]
    for _ in range(args.warmup):
        cpu_step(po, enc, pe, tiles, images, args.workload)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(po, enc, pe, tiles, images, args.workload)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = f"{n} of {args.batch} tiles per step ({args.points} pts/tile), {args.steps} steps, tiles/s scales per tile"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "mpoints_per_s": value * args.points / 1e6,
        "note": "reference CPU path, restated (open3d 0.19.0 not installable offline); ONE CPU process on rank 0 whatever N is: compare with the N = 1 line only",
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    name = {"lidar": "Pix2Poly LiDAR-only (PointPillars front end of lidar_pp_vit)",
            "fusion": "Pix2Poly early fusion (image patch embed + LiDAR pillars -> concat)",
            "fusion_layer": "Pix2Poly early fusion through fusion_layer (patch embed + LiDAR pillars + conv3x3 768->384 + BN + ReLU -> tokens)"}[args.workload]
    return {"workload": f"{name}, synthetic 224px tiles, {args.points} pts/tile, batch {args.batch} per GPU",
            "tiles_per_gpu": args.batch, "points_per_tile": args.points, "max_points_per_voxel": args.max_points_per_voxel,
            "precision": args.precision, "in_flight": args.in_flight,
            "l2": f"rotating input+output sets per GPU (> 126 MB L2 in total; default {args.sets})",
            "parallelism": f"tiles sharded batch-wise over {args.gpus} GPU(s), no collective"}


def bind_to_gpu_numa(local_rank):
    """Best effort: run this rank's host threads on the CPUs of its GPU's NUMA node, so that the pinned buffers allocated
    afterwards (first touch) and the copy-issuing thread sit next to the GPU's PCIe root.  Returns a description."""
    try:
        import pynvml

        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = local_rank
        if visible:
            ids = [v.strip() for v in visible.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                phys = int(ids[local_rank])
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa node unknown (single node or virtualised)"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"bound to NUMA node {node} ({len(allowed)} cpus)"
        return f"NUMA node {node} has no allowed cpus"
    except Exception as e:  # noqa: BLE001
        return f"not bound ({type(e).__name__})"


def synth_las_batch(tiles, rng):
    """Raw LAS integers whose loader arithmetic (p3_coco.py:74-101) lands near the given pixel-space tiles: 1 mm scale,
    56 m tiles.  -> (deltas (sum N, 3) uint16, base (B, 3) int32, per-tile header dicts)."""
    from pixelspointspolygons_b200 import pack_las

    deltas, bases, metas = [], [], []
    for i, t in enumerate(tiles):
        left, top = 2_600_000.0 + 56.0 * i, 1_200_000.0
        X = np.clip(np.rint(t[:, 0].astype(np.float64) * 250.0), 0, 56_000).astype(np.int32)
        Y = np.clip(np.rint((224.0 - t[:, 1].astype(np.float64)) * 250.0), 0, 56_000).astype(np.int32)
        Z = np.rint(t[:, 2].astype(np.float64) * 300.0).astype(np.int32) + 400_000  # 30 m of relief at 1 mm
        d, b = pack_las(X, Y, Z)
        deltas.append(d); bases.append(b)
        metas.append(dict(scales=(0.001, 0.001, 0.001), offsets=(left, top, 0.0), top_left=(left, top), height=224, width=224))
    return np.concatenate(deltas), np.stack(bases), metas


class Workload:
    """One configuration of the hot path on this rank's GPU: modules, rotating input / output sets resident in HBM, and one
    CUDA graph per set (the steady-state serving loop replays them)."""

    def __init__(self, dev, rank, workload, precision, B, N, M, sets, use_graph=True, keep_host=False, lanes=2):
        from pixelspointspolygons_b200 import PointPillarsEncoder, _lib, default_cfg
        from tools import synth

        self.dev, self.workload, self.precision, self.B, self.N, self.M = dev, workload, precision, B, N, M
        # batches in flight: consecutive steps alternate between `lanes` streams (one workspace each), so that the voxelizer
        # of step i + 1 runs on the SMs the PFN of step i has not claimed yet / has already left
        self.lanes = max(1, int(lanes))
        self.streams = [torch.cuda.Stream(dev) for _ in range(self.lanes)]
        cfg = default_cfg(device=str(dev), max_num_points_per_voxel=M, p3p_precision=precision)
        self.enc = PointPillarsEncoder(cfg, voxel_encoder={"in_channels": 3, "feat_channels": [64, C_FEAT]},
                                       scatter={"in_channels": C_FEAT, "output_shape": [28, 28]}).to(dev).eval()
        sd, sdi = synth.synth_weights(0)
        self.enc.load_state_dict(sd)
        self.fusion = None
        if workload in ("fusion", "fusion_layer"):
            from pixelspointspolygons_b200.fusion import EarlyFusionFrontEnd

            self.fusion = EarlyFusionFrontEnd(cfg).to(dev).eval()
            self.fusion.lidar_embed.load_state_dict(sd)
            self.fusion.image_embed.load_state_dict(sdi)
            with torch.no_grad():  # seeded fusion_layer weights (conv ~ N(0, 1/fan_in), BN like synth_weights)
                g = torch.Generator().manual_seed(1)
                fl = self.fusion.fusion_layer
                fl[0].weight.copy_((torch.randn(fl[0].weight.shape, generator=g) / (9 * 768) ** 0.5).to(dev))
                fl[0].bias.copy_((torch.randn(C_FEAT, generator=g) * 0.1).to(dev))
                fl[1].weight.copy_((torch.rand(C_FEAT, generator=g) + 0.5).to(dev))
                fl[1].running_var.copy_((torch.rand(C_FEAT, generator=g) + 0.5).to(dev))
        # enough rotating sets that consecutive uses of a set are > L2 apart
        per_set = 12 * N * B + (4 * 768 * HW * B + 4 * 3 * 224 * 224 * B if self.fusion is not None else 4 * C_FEAT * HW * B)
        sets = max(2, sets, -(-(160 << 20) // per_set))
        self.sets = sets = -(-sets // self.lanes) * self.lanes  # a multiple of the lanes: set s always runs on lane s % lanes
        host_tiles = [[synth.synth_tile(N, 1000 * (1 + rank) + 16 * s + i, clustered=(i % 2 == 1)) for i in range(B)]
                      for s in range(min(sets, 8))]
        self.tiles0 = host_tiles[0]
        self.host_tiles = host_tiles if keep_host else None
        vals = [torch.from_numpy(np.concatenate(t)) for t in host_tiles]
        self.offs = torch.arange(B + 1, dtype=torch.int64) * N
        self.pinned_vals = [v.pin_memory() for v in vals] if keep_host else None
        self.pinned_offs = self.offs.clone().pin_memory() if keep_host else None
        # (beyond 8 distinct batches the sets re-use the point data in fresh buffers: what matters is that they are not in L2)
        self.dev_vals = [vals[s % len(vals)].to(dev) for s in range(sets)]
        self.dev_offs = self.offs.to(dev)
        self.dev_x = [torch.nested.nested_tensor_from_jagged(v, self.dev_offs) for v in self.dev_vals]
        self.pinned_img = self.dev_img = None
        if self.fusion is not None:
            imgs = [torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(1000 * (1 + rank) + s))
                    for s in range(min(sets, 8))]
            self.pinned_img = [p.pin_memory() for p in imgs] if keep_host else None
            self.dev_img = [imgs[s % len(imgs)].to(dev) for s in range(sets)]
            if workload == "fusion_layer":
                self.x16 = [torch.empty(B, 28, 28, 2 * C_FEAT, dtype=self.fusion.fusion_layer.operand_dtype, device=dev) for _ in range(sets)]
                self.outs = [torch.empty(B, HW, C_FEAT, device=dev) for _ in range(sets)]
            else:
                self.outs = [torch.empty(B, 2 * C_FEAT, 28, 28, device=dev) for _ in range(sets)]
        else:
            self.outs = [torch.empty(B, HW, C_FEAT, device=dev) for _ in range(sets)]
        self._lib = _lib
        for i in range(sets):
            self.step(i)
        torch.cuda.synchronize()
        self.graphs = None
        if use_graph:
            self.graphs = []
            for s in range(sets):
                st = self.streams[s % self.lanes]
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=st):
                    self.step(s)
                self.graphs.append(g)
            torch.cuda.synchronize()

    def step(self, i, lane=None):
        s = i % self.sets
        lane = s % self.lanes if lane is None else lane
        if self.workload == "fusion_layer":
            self.fusion.forward_tokens_into(self.dev_img[s], self.dev_x[s], self.x16[s], self.outs[s], lidar_zero=False, lane=lane)
        elif self.fusion is not None:
            self.fusion.forward_into(self.dev_img[s], self.dev_x[s], self.outs[s], lane=lane)
        else:
            self.enc.encode_into(self.dev_x[s], self.outs[s], self._lib.P3P_LAYOUT_NLC, lane=lane)

    def run_step(self, i, single=False):
        """Step i on its lane's stream (enqueue only); single: every step on ONE stream (a step starts when the previous ends)."""
        s = i % self.sets
        with torch.cuda.stream(self.streams[0 if single else s % self.lanes]):
            if self.graphs is not None:
                self.graphs[s].replay()
            else:
                self.step(i)

    @property
    def launches_per_step(self):
        # voxelize + PFN (+ patch embed (+ fusion convolution)); the counter memset is not a kernel
        return 2 if self.fusion is None else (4 if self.workload == "fusion_layer" else 3)

    def time_steps(self, steps, first=0, single=False, warmup=0):
        """Device time (ms) of steps first .. first + steps - 1 issued back to back; the end event follows the last step of
        every lane.  Without warm-up the start event precedes the first step on every lane.  With `warmup` steps (first -
        warmup .. first - 1) issued right before them, it follows the last warm-up step on its stream: the window holds
        `steps` step completions of a full pipeline, whose fill stays in the warm-up."""
        cur = torch.cuda.current_stream(self.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if warmup:
            for i in range(first - warmup, first):
                self.run_step(i, single)
            e0.record(self.streams[0 if single else (first - 1) % self.sets % self.lanes])
        else:
            e0.record(cur)
            for st in self.streams:
                st.wait_event(e0)
        for i in range(steps):
            self.run_step(first + i, single)
        for st in self.streams:
            cur.wait_stream(st)
        e1.record(cur)
        e1.synchronize()
        return e0.elapsed_time(e1)

    def time_for(self, seconds, chunk=256, single=False):
        """Steps and device milliseconds of a loop of at least `seconds` (chunks of `chunk` steps between two events)."""
        total_ms, total_steps = 0.0, 0
        while total_ms < seconds * 1e3:
            total_ms += self.time_steps(chunk, total_steps, single)
            total_steps += chunk
        return total_steps, total_ms


DUMP_LIMIT = 64 << 20


def dump_outputs(w, i, directory):
    """Write what step i (completed) handed its caller as `directory`/<name>.npy, fp32: the tokens (B, ny*nx, C) of the
    lidar and fusion_layer workloads, the concatenated features (B, 2C, ny, nx) of the fusion workload.  Above
    DUMP_LIMIT bytes a fixed, seeded sample of the tiles is written (ascending tile order).  Returns a description."""
    out = w.outs[i % w.sets].cpu().numpy()
    name = "features" if w.workload == "fusion" else "tokens"
    tiles = np.arange(out.shape[0])
    if out.nbytes > DUMP_LIMIT:
        keep = max(1, DUMP_LIMIT // (out.nbytes // out.shape[0]))
        tiles = np.sort(np.random.default_rng(0).choice(out.shape[0], keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(out[tiles], dtype=np.float32))
    return {"dir": directory, "step": i, "files": {name: list(out[tiles].shape)},
            "tiles": "all" if len(tiles) == out.shape[0] else tiles.tolist()}


def conv_roofline(w, peaks):
    """The fusion convolution alone (resident 16-bit input of the last step of every set): FLOPs / CUDA-event time."""
    fl = w.fusion.fusion_layer
    B = w.B
    for i in range(3):
        fl.forward_nhwc(w.x16[i % w.sets], w.outs[i % w.sets], 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 40
    e0.record()
    for i in range(n):
        fl.forward_nhwc(w.x16[i % w.sets], w.outs[i % w.sets], 1)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / n
    flops = 2.0 * B * HW * C_FEAT * 9 * 2 * C_FEAT
    peak = float(peaks.get("bf16_tflops", 1590.0))
    return {"kernel": "conv3x3_tc_kernel", "bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
            "frac": flops / (ms * 1e-3) / 1e12 / peak, "ms_per_launch": ms, "flops_per_launch": flops,
            "what": "implicit GEMM 784 B x 6912 x 384 (16-bit operands, fp32 accumulate), launched back to back"}


def sub_result(dev, rank, workload, precision, B, N, M, seconds=0.4):
    """A secondary configuration, device-timed for ~`seconds` after a warm-up (CUDA-graph replay, rotating sets)."""
    try:
        w = Workload(dev, rank, workload, precision, B, N, M, sets=2)
        w.time_steps(20)
        steps, ms = w.time_for(seconds, chunk=64)
        out = {"workload": workload, "precision": precision, "tiles_per_gpu": B, "points_per_tile": N, "max_points_per_voxel": M,
               "ms_per_step": ms / steps, "tiles_per_s_per_gpu": B * steps / (ms * 1e-3), "steps": steps, "sets": w.sets,
               "in_flight": w.lanes}
        if workload == "fusion_layer":
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            out["conv_roofline"] = conv_roofline(w, peaks)
        del w
        torch.cuda.empty_cache()
        return out
    except Exception as e:  # a secondary line must not take the headline down
        return {"workload": workload, "precision": precision, "tiles_per_gpu": B, "points_per_tile": N,
                "max_points_per_voxel": M, "error": repr(e)[:300]}


def train_sub_result(dev, rank, B, N, M, with_dense):
    """The optional training step (SURVEY 8f-4): forward + backward of the LiDAR encoder in train mode through the fused
    kernels (pixelspointspolygons_b200/train.py), device-timed; next to it, on one GPU, the dense autograd formulation the
    reference runs (nn.Linear + BatchNorm1d + ReLU + max over (V, M, *) tensors) on the same pillars."""
    try:
        from pixelspointspolygons_b200 import PointPillarsEncoder, default_cfg
        from tools.synth import synth_tile, synth_weights

        enc = PointPillarsEncoder(default_cfg(device=str(dev), max_num_points_per_voxel=M),
                                  voxel_encoder={"in_channels": 3, "feat_channels": [64, 384]},
                                  scatter={"in_channels": 384, "output_shape": [28, 28]}).to(dev).train()
        enc.load_state_dict(synth_weights(0)[0])
        x = torch.from_numpy(np.stack([synth_tile(N, 1000 * (rank + 1) + i, clustered=(i % 2 == 1)) for i in range(B)])).to(dev)
        wgt = torch.randn(B, 784, 384, device=dev)

        def timed(fn, warm, iters):
            def step():
                enc.zero_grad(set_to_none=True)
                (fn(x) * wgt).sum().backward()
            for _ in range(warm):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(iters):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / iters

        fused = timed(lambda t: enc(t), 3, 30)
        out = {"workload": "train_step", "what": "forward + backward of the LiDAR encoder in train mode (BatchNorm batch statistics, "
               "gradients of the six PFN parameters), exact fp32, eager launches", "tiles_per_gpu": B, "points_per_tile": N,
               "max_points_per_voxel": M, "ms_per_step": fused, "tiles_per_s_per_gpu": B / (fused * 1e-3)}
        if with_dense:
            out["dense_autograd_ms_per_step"] = timed(lambda t: enc.forward_dense_reference(t), 1, 3)
        del enc, x, wgt
        torch.cuda.empty_cache()
        return out
    except Exception as e:
        return {"workload": "train_step", "tiles_per_gpu": B, "points_per_tile": N, "max_points_per_voxel": M, "error": repr(e)[:300]}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    import torch.distributed as dist

    from pixelspointspolygons_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    numa = bind_to_gpu_numa(local_rank)
    B, N, M = args.batch, args.points, args.max_points_per_voxel
    W = Workload(dev, rank, args.workload, args.precision, B, N, M, args.sets, use_graph=not args.no_graph, keep_host=True,
                 lanes=args.in_flight)
    enc, fusion, sets = W.enc, W.fusion, W.sets
    flops, kept, pillars = algorithmic_flops(W.tiles0, M)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the timed region: device time of exactly K steps right after W warm-up steps, max over ranks ----------------
    barrier()
    ms_region = W.time_steps(args.steps, first=args.warmup, warmup=args.warmup)
    barrier()
    ms = torch.tensor([ms_region], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_k = float(ms.item())
    ms_per_step = ms_k / args.steps
    value = B * world / (ms_per_step * 1e-3)
    dumped = dump_outputs(W, args.warmup + args.steps - 1, args.dump_outputs) if (args.dump_outputs and rank == 0) else None
    # ---- the same loop held for >= --min-seconds (sustained clocks / power), clocks sampled inside ---------------------
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    sus_steps, sus_ms = W.time_for(args.min_seconds)
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([sus_ms / sus_steps], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sustained = {"steps": sus_steps, "seconds": sus_ms * 1e-3, "ms_per_step": float(t.item()),
                 "value": B * world / (float(t.item()) * 1e-3), "unit": UNIT,
                 "what": f"the same step loop held for >= {args.min_seconds} s (max over ranks of the per-step time; clocks "
                         "sampled inside): the power-limited serving loop"}
    one_steps, one_ms = W.time_for(min(0.5, args.min_seconds), single=True)
    t1 = torch.tensor([one_ms / one_steps], device=dev)
    if world > 1:
        dist.all_reduce(t1, op=dist.ReduceOp.MAX)
    one_in_flight = {"ms_per_step": float(t1.item()), "value": B * world / (float(t1.item()) * 1e-3), "unit": UNIT, "steps": one_steps,
                     "what": "the same graphs replayed on ONE stream: a step starts when the previous one has ended (the latency-"
                             "oriented number; `value` keeps `in_flight` batches in flight on as many streams / workspaces)"}

    # ---- end to end through the module API with host buffers ------------------------------------------------------
    # Every step copies its inputs from pinned host memory and reads its result back; the copy of step i + 1 runs on a
    # side stream while step i computes (two device input buffers), as a serving loop would prefetch its next batch.
    nbuf = 2
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d_vals = [torch.empty_like(W.dev_vals[0]) for _ in range(nbuf)]
    d_offs = [torch.empty_like(W.dev_offs) for _ in range(nbuf)]
    d_img = [torch.empty_like(W.dev_img[0]) for _ in range(nbuf)] if fusion is not None else None
    h_sum = [torch.empty(B, dtype=torch.float32).pin_memory() for _ in range(nbuf)]
    out_numel = W.outs[0].numel()
    h_full = [torch.empty(out_numel, dtype=torch.float32).pin_memory() for _ in range(nbuf)]
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)
    copied = [torch.cuda.Event() for _ in range(nbuf)]
    consumed = [torch.cuda.Event() for _ in range(nbuf)]
    nh = len(W.pinned_vals)

    def e2e_copy(i):
        s, b = i % nh, i % nbuf
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])  # the buffer's previous step has finished reading it
            d_vals[b].copy_(W.pinned_vals[s], non_blocking=True)
            d_offs[b].copy_(W.pinned_offs, non_blocking=True)
            if fusion is not None:
                d_img[b].copy_(W.pinned_img[s], non_blocking=True)
            copied[b].record(copy_stream)

    def e2e_compute(i, full):
        b = i % nbuf
        main_stream.wait_event(copied[b])
        x = torch.nested.nested_tensor_from_jagged(d_vals[b], d_offs[b])
        if args.workload == "fusion_layer":
            y = fusion.forward_tokens(d_img[b], x, lidar_zero=False)
        else:
            y = fusion(d_img[b], x) if fusion is not None else enc(x, return_flattened=True)
        consumed[b].record(main_stream)
        if full:
            h_full[b].copy_(y.reshape(-1), non_blocking=True)
        else:
            h_sum[b].copy_(y.reshape(B, -1).sum(dim=1), non_blocking=True)

    def e2e_run(n, full):
        e2e_copy(0)
        for i in range(n):
            if i + 1 < n:
                e2e_copy(i + 1)
            e2e_compute(i, full)

    def e2e_measure(full, seconds):
        for b in range(nbuf):
            consumed[b].record(main_stream)
        e2e_run(3, full)
        barrier()
        n, tot = 0, 0.0
        while tot < seconds * 1e3:
            e0.record()
            e2e_run(32, full)
            e1.record()
            e1.synchronize()
            tot += e0.elapsed_time(e1)
            n += 32
        barrier()
        m = torch.tensor([tot / n], device=dev)
        if world > 1:
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
        return B * world / (float(m.item()) * 1e-3), n

    h2d = W.pinned_vals[0].numel() * 4 + W.pinned_offs.numel() * 8 + (W.pinned_img[0].numel() * 4 if fusion is not None else 0)
    e2e_value, e2e_steps = e2e_measure(False, min(1.0, args.min_seconds))

    # ---- the serving loop of the package (HostPipeline): the loader's output is what a LAS file holds -- integer
    #      coordinates as uint16 deltas + an int32 base per tile (6 bytes per point over PCIe instead of 12), the tile headers,
    #      the fp32 image -- in pinned staging slots; per batch the host issues H2D(batch i + 1) on a copy stream, ONE CUDA-graph
    #      launch compute(batch i) (‖ D2H(result i - 1) on a third stream).  The loader arithmetic of p3_coco.py:74-101 (float64 scale / offset, MinMaxScaler on z, clip)
    #      runs on the GPU in front of the encoder, bit-exact (tests/test_gpu_parity.py, tests/test_gpu_pipeline.py) ----------
    from pixelspointspolygons_b200 import HostPipeline

    las_sets = [synth_las_batch(t, None) for t in W.host_tiles]
    module = fusion if fusion is not None else enc
    mode = "tokens" if args.workload == "fusion_layer" else "concat"

    def pipeline_measure(host_result, seconds):
        pipe = HostPipeline(module, B, B * N, slots=len(las_sets), mode=mode, host_result=host_result)
        for i, (d, b, metas) in enumerate(las_sets):  # every slot holds its own batch: the timed loop re-sends them in turn
            s = pipe.slots[i]
            s.deltas.copy_(torch.from_numpy(d)); s.base.copy_(torch.from_numpy(b)); s.offsets.copy_(W.offs)
            pipe.set_tiles(s, metas)
            if s.image is not None:
                s.image.copy_(W.pinned_img[i % len(W.pinned_img)])

        def run(n):
            for _ in range(n):
                pipe.staging()
                pipe.submit()

        run(2 * pipe.n)
        pipe.stream.synchronize()
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n, tot = 0, 0.0
        while tot < seconds * 1e3:
            p0.record(pipe.stream)
            run(64)
            p1.record(pipe.stream)
            p1.synchronize()
            tot += p0.elapsed_time(p1)
            n += 64
        last = pipe.flush()
        pipe.stream.synchronize()
        check = float(last.out.float().abs().sum().item())
        barrier()
        m = torch.tensor([tot / n], device=dev)
        if world > 1:
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
        res = (B * world / (float(m.item()) * 1e-3), n, pipe.h2d_bytes_per_step, pipe.d2h_bytes_per_step, check)
        del pipe
        torch.cuda.empty_cache()
        return res

    e2e_las_value, n_las, h2d_las, d2h_las, chk = pipeline_measure(lambda y: y.reshape(B, -1).sum(dim=1), min(1.5, args.min_seconds))
    e2e_full_value, e2e_full_steps, _, d2h_full, _ = pipeline_measure("full", min(1.0, args.min_seconds))
    if not (chk > 0.0 and np.isfinite(chk)):
        raise SystemExit("the pipeline's last result is empty or not finite")
    e2e = {"value": e2e_las_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_las), "d2h_bytes_per_step": int(d2h_las),
           "steps": n_las, "api": "pixelspointspolygons_b200.HostPipeline (staging() / submit() per batch)",
           "input": "pinned host slots holding LAS integer coordinates as uint16 deltas + int32 base per tile (6 B/point), tile "
                    "headers, offsets (+ fp32 images); the reference loader's coordinate arithmetic runs on the GPU "
                    "(p3p_las_packed_to_pixels) in front of the encoder",
           "fp32_points_input": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "steps": e2e_steps,
                                 "what": "eager module calls fed with ready-made fp32 pixel-space points (12 B/point), two device "
                                         "buffers, H2D on a copy stream, as in round 1"},
           "host_numa": numa,
           "result_read": "one float per tile (sum of the tile's output) copied to pinned memory inside every batch's graph: the "
                          "consumer of this path is the ViT on the same GPU, the host only needs a completion / sanity value",
           "full_result_d2h": {"value": e2e_full_value, "unit": UNIT, "d2h_bytes_per_step": int(d2h_full), "steps": e2e_full_steps,
                               "what": "the same pipeline copying the whole output tensor of batch i - 1 back to pinned host memory "
                                       "on a third stream"},
           "pipeline": "per batch: H2D(i + 1) on the copy stream ‖ one CUDA-graph launch compute(i) ‖ D2H(i - 1) on the return stream"}

    # ---- per-kernel durations (CUDA events recorded inside p3p_encode on the launching stream) ----------------
    prof_steps = 100
    l = _lib.lib()
    _lib.check(l.p3p_profile_begin(prof_steps), "p3p_profile_begin")
    for i in range(prof_steps):
        W.step(i, lane=0)
    arr = [(C.c_float * prof_steps)() for _ in range(2)]
    cnt = C.c_int32(0)
    _lib.check(l.p3p_profile_end(arr[0], arr[1], prof_steps, C.byref(cnt)), "p3p_profile_end")
    stage_ms = {n: (statistics.mean(list(a)[:cnt.value]) if cnt.value else None) for n, a in zip(("voxelize", "pfn"), arr)}

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    which = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    bf16_burst = float(peaks.get("bf16_tflops", 1590.0))
    bf16_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    half = args.precision not in ("bf16", "fp16")  # tf32 dense = half the 16-bit rate
    tensor_peak = bf16_burst / (2.0 if half else 1.0)
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "pfn_traffic.json")))
        traffic, traffic_src = tj.get(args.precision), tj.get("source")
    except Exception:
        pass
    pfn_s = (stage_ms["pfn"] or 0.0) * 1e-3
    achieved_tf = flops / pfn_s / 1e12 if pfn_s > 0 else None
    roofline = {"kernel": "pfn_tc_kernel" if (args.precision != "fp32" and M <= 512) else "pfn_simt_kernel",
                "bound": "tensor", "achieved": achieved_tf, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": (achieved_tf / tensor_peak) if achieved_tf else None, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": which + " burst figure (the kernel is timed alone between two events)" + ("; tf32 peak taken as bf16/2" if half else ""),
                "frac_of_sustained_peak": (achieved_tf / (bf16_sus / (2.0 if half else 1.0))) if achieved_tf else None,
                "flops_per_launch": flops, "ms_per_launch": stage_ms["pfn"], "kept_points": kept, "pillars": pillars}
    bytes_tile = algorithmic_bytes_per_tile(N, args.workload)
    per_gpu_gbs = bytes_tile * (value / world) / 1e9
    hbm = {"bound": "hbm", "achieved": per_gpu_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": per_gpu_gbs / hbm_peak,
           "bytes_per_tile": bytes_tile, "peak_source": which, "scope": "whole path, per GPU, timed region (`value`)",
           "whole_path_tflops": flops * (value / world / B) / 1e12,
           # the sustained loop's rate against the sustained peak
           "whole_path_frac_of_sustained_tensor_peak": flops * (sustained["value"] / world / B) / 1e12 / (bf16_sus / (2.0 if half else 1.0))}

    # ---- secondary configurations, so that the driver's line carries them (BASELINE configs 2-5) -----------------------
    subs = []
    if not args.no_sub_results:
        del d_vals, d_offs, d_img, h_full
        torch.cuda.empty_cache()
        plan = [("lidar", "tf32", B, N, M), ("lidar", "bf16", B, N, M), ("fusion", args.precision, 16, N, M),
                ("fusion", args.precision, 8, N, M), ("fusion", "tf32", 16, N, M), ("fusion_layer", args.precision, 16, N, M),
                ("fusion_layer", args.precision, 8, N, M), ("lidar", args.precision, 32, N, M),
                ("lidar", args.precision, 16, 10_000, M), ("lidar", args.precision, 16, 400_000, M),
                ("lidar", args.precision, 16, N, 128)]
        for wl, prec, b, n, m in plan:
            if (wl, prec, b, n, m) == (args.workload, args.precision, B, N, M):
                continue
            barrier()
            subs.append(sub_result(dev, rank, wl, prec, b, n, m))
        barrier()
        subs.append(train_sub_result(dev, rank, 16, N, M, with_dense=(world == 1)))

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        po2, cenc, cpe = cpu_oracle_modules(M)
        n = min(B, 4)
        tiles = W.tiles0[:n]
        imgs = torch.rand(n, 3, 224, 224)
        cpu_step(po2, cenc, cpe, tiles[:1], imgs[:1], args.workload)
        t0 = time.perf_counter()
        reps = 0
        while reps < 3 or (time.perf_counter() - t0 < 10.0 and reps < 50):
            cpu_step(po2, cenc, cpe, tiles, imgs, args.workload)
            reps += 1
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": n * reps / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"{n} of {B} tiles x {reps} repetitions ({N} pts/tile); oracle = CPU restatement of the "
                                  "reference path (open3d 0.19.0 not installable offline); one process"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16", "fp16": "f16 operands, f32 accumulate, f32 in/out"}[args.precision], "data": "synthetic",
            "config": workload_config(args), "mpoints_per_s": value * N / 1e6,
            "timed_region": {"steps_timed": args.steps, "warmup_steps": args.warmup, "seconds": ms_k * 1e-3,
                             "what": "`value` / `ms_per_step`: exactly --steps steps issued right after --warmup warm-up steps, "
                                     "from the completion of the last warm-up step to that of the last timed step (max over ranks)"},
            "sustained": sustained, "one_batch_in_flight": one_in_flight, "dump_outputs": dumped,
            "e2e": e2e, "gpu_launches": W.launches_per_step * (args.steps + sus_steps), "launch_mode": "cuda_graph" if W.graphs else "c_abi_per_step",
            "roofline": roofline, "hbm_roofline": hbm, "stage_ms": stage_ms, "sub_results": subs, "cpu_baseline": cpu_baseline, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
