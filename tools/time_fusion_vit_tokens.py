#!/usr/bin/env python
"""Device time of the early-fusion ViT input: EarlyFusionFrontEnd.forward_tokens(..., cls_token=, pos_embed=) -- the class
token and pos_embed written by the fusion convolution's epilogue -- against forward_tokens + torch.cat + add, at B = 16 and
B = 8 (config 3's share of a batch), N = 100 k points per tile, fp16 and bf16 operands, eager launches, one and two batches
in flight (two streams, two lanes).

Inputs and outputs rotate over 4 sets (> 126 MB in all: each set is read from HBM, not from L2).  The two routes alternate
twice per configuration, each measurement 2000 steps between two CUDA events.  One step of each route is also traced with
torch.profiler (a run of its own) to count its kernels.

usage (GPU box): python tools/time_fusion_vit_tokens.py [--out FILE.json] [--steps 2000]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth  # (neutral generators: measurement tools do not touch oracle/)
from pixelspointspolygons_b200 import EarlyFusionFrontEnd, default_cfg

C, HW, SETS = 384, 784, 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def setup(prec, B, dev):
    fe = EarlyFusionFrontEnd(default_cfg(device=str(dev), p3p_precision=prec))
    sd, sdi = synth.synth_weights(0)
    fe.lidar_embed.load_state_dict(sd)
    fe.image_embed.load_state_dict(sdi)
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        w = fe.fusion_layer[0].weight
        w.copy_(torch.randn(w.shape, generator=g) / (9 * 768) ** 0.5)
    fe = fe.to(dev).eval()
    tiles = [synth.synth_tile(100_000, 1000 + i, clustered=(i % 2 == 1)) for i in range(B)]
    pts = torch.from_numpy(np.stack(tiles))
    sets = []
    for s in range(SETS):  # same values, separate memory
        sets.append(dict(x=pts.to(dev), img=torch.rand(B, 3, 224, 224, generator=g).to(dev),
                         x16=torch.empty(B, 28, 28, 2 * C, dtype=fe.fusion_layer.operand_dtype, device=dev),
                         out=torch.empty(B, 1 + HW, C, device=dev), rows=torch.empty(B, HW, C, device=dev)))
    cls = torch.randn(1, 1, C, generator=g).to(dev) * 0.02
    pos = torch.randn(1, 1 + HW, C, generator=g).to(dev) * 0.02
    return fe, sets, cls, pos


def fused(fe, s, cls, pos, lane):
    return fe.forward_tokens_into(s["img"], s["x"], s["x16"], s["out"], lidar_zero=False, lane=lane, cls_token=cls, pos_embed=pos)


def unfused(fe, s, cls, pos, lane):
    t = fe.forward_tokens_into(s["img"], s["x"], s["x16"], s["rows"], lidar_zero=False, lane=lane)
    return torch.cat((cls.expand(t.shape[0], -1, -1), t), dim=1) + pos


def time_route(route, fe, sets, cls, pos, streams, steps):
    """us per step; steps alternate over the streams (lane = stream index)."""
    cur = torch.cuda.current_stream()
    def issue(n, first=0):
        for i in range(first, first + n):
            k = i % len(streams)
            with torch.cuda.stream(streams[k]):
                route(fe, sets[i % SETS], cls, pos, k)
    issue(20)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for st in streams:
        st.wait_event(e0)
    issue(steps, 20)
    for st in streams:
        cur.wait_stream(st)
    e1.record(cur)
    e1.synchronize()
    return e0.elapsed_time(e1) / steps * 1e3


def kernels_per_step(route, fe, sets, cls, pos):
    from torch.profiler import ProfilerActivity, profile

    route(fe, sets[0], cls, pos, 0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        route(fe, sets[0], cls, pos, 0)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
             and not e.name.lower().startswith(("memset", "memcpy"))]
    return len(names), names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=2000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    result = {"card": card(), "N": 100_000, "sets": SETS, "steps": args.steps, "rows": []}
    print(json.dumps(result["card"]))
    routes = {"fused": fused, "forward_tokens+cat+add": unfused}
    with torch.no_grad():
        for prec in ("fp16", "bf16"):
            for B in (16, 8):
                fe, sets, cls, pos = setup(prec, B, dev)
                # same values from both routes (the epilogue's add is the same fp32 add as torch's)
                a, b = fused(fe, sets[0], cls, pos, 0), unfused(fe, sets[0], cls, pos, 0)
                torch.cuda.synchronize()
                assert torch.equal(a, b), "the two routes differ"
                counts = {name: kernels_per_step(r, fe, sets, cls, pos) for name, r in routes.items()}
                for lanes in (1, 2):
                    streams = [torch.cuda.Stream(dev) for _ in range(lanes)]
                    t = {name: [] for name in routes}
                    for _ in range(2):
                        for name, r in routes.items():
                            t[name].append(time_route(r, fe, sets, cls, pos, streams, args.steps))
                    row = {"precision": prec, "B": B, "in_flight": lanes,
                           "us_per_step": {k: [round(x, 1) for x in v] for k, v in t.items()},
                           "kernels_per_step": {k: v[0] for k, v in counts.items()}}
                    row["gain_us"] = round(min(t["forward_tokens+cat+add"]) - min(t["fused"]), 1)
                    result["rows"].append(row)
                    print(json.dumps(row), flush=True)
                result.setdefault("kernel_names", {k: v[1] for k, v in counts.items()})
                del fe, sets
                torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
