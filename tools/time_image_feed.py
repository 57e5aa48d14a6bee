#!/usr/bin/env python
"""The early-fusion serving loop fed with the fp32 image against the uint8 image: HostPipeline(mode = concat / tokens,
image_dtype = float32 / uint8) at B = 16 tiles x 100 k points, fp16 operands, and the patch embedding alone on either input.

Pipelines: the same LAS batches and the same images in both (the fp32 image is the uint8 one expanded through the pixel
table, so both compute the same values: checked bit for bit on every slot).  Per mode the two feeds alternate three
times, each window >= --seconds of back-to-back batches timed by CUDA events on the compute stream, as bench.py times its
e2e leg.  Kernel: `PatchEmbed.forward_into` alone, one CUDA graph with a launch per image set, 64 sets (> 126 MB of L2
for either format), replayed 32 times between two CUDA events per measurement; into the concat buffer (fp32 NCHW) and the
fusion convolution's 16-bit channels-last input (tokens mode); fp32 and uint8 alternated three times.

usage (GPU box): python tools/time_image_feed.py [--out profiles/FILE.json] [--seconds 2.0]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import bind_to_gpu_numa, synth_las_batch  # noqa: E402
from tools import synth  # noqa: E402  (neutral generators: measurement tools do not touch oracle/)
from pixelspointspolygons_b200 import EarlyFusionFrontEnd, HostPipeline, default_cfg  # noqa: E402
from pixelspointspolygons_b200._lib import P3P_LAYOUT_NCHW, P3P_LAYOUT_NLC  # noqa: E402

B, N, C, SLOTS, KSETS = 16, 100_000, 384, 3, 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def front_end(dev):
    fe = EarlyFusionFrontEnd(default_cfg(device=str(dev), p3p_precision="fp16"))
    sd, sdi = synth.synth_weights(0)
    fe.lidar_embed.load_state_dict(sd)
    fe.image_embed.load_state_dict(sdi)
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        w = fe.fusion_layer[0].weight
        w.copy_(torch.randn(w.shape, generator=g) / (9 * 768) ** 0.5)
    return fe.to(dev).eval()


def make_pipeline(fe, mode, image_dtype, las_sets, imgs8):
    pipe = HostPipeline(fe, B, B * N, slots=SLOTS, mode=mode, image_dtype=image_dtype,
                        host_result=lambda y: y.reshape(B, -1).sum(dim=1))
    offs = torch.arange(B + 1, dtype=torch.int64) * N
    for i, (d, b, metas) in enumerate(las_sets):  # every slot holds its own batch: the timed loop re-sends them in turn
        s = pipe.slots[i]
        s.deltas.copy_(torch.from_numpy(d)); s.base.copy_(torch.from_numpy(b)); s.offsets.copy_(offs)
        pipe.set_tiles(s, metas)
        s.image.copy_(imgs8[i] if image_dtype == torch.uint8 else fe.image_embed.expand_pixels(imgs8[i]))
    return pipe


def measure(pipe, seconds):
    """tiles/s of back-to-back batches (staging() + submit() per batch) over >= `seconds`, timed on the compute stream."""
    def run(n):
        for _ in range(n):
            pipe.staging()
            pipe.submit()

    run(2 * pipe.n)
    pipe.stream.synchronize()
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
    last.done.synchronize()
    return {"tiles_per_s": round(B / (tot / n * 1e-3), 1), "us_per_step": round(tot / n * 1e3, 1), "steps": n,
            "seconds": round(tot * 1e-3, 2)}


def time_kernel(fe, images, out, layout, c_total, replays=32):
    """us per PatchEmbed.forward_into launch: one CUDA graph of a launch per image set (the host's ctypes call stays out of
    the timing), replayed `replays` times between two events."""
    pe = fe.image_embed
    for x in images:  # warm-up outside capture (prepared weights, the table's device copy)
        pe.forward_into(x, out, c_total, 0, layout=layout)
    torch.cuda.synchronize()
    graph, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=st):
        for x in images:
            pe.forward_into(x, out, c_total, 0, layout=layout)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    e1.synchronize()
    return round(e0.elapsed_time(e1) / (replays * len(images)) * 1e3, 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=2.0)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    numa = bind_to_gpu_numa(0)
    result = {"card": card(), "host_numa": numa, "tiles": B, "points_per_tile": N, "precision": "fp16", "slots": SLOTS,
              "window_seconds": args.seconds, "pipeline": {}, "patch_embed_kernel_us": {}}
    print(json.dumps(result["card"]), flush=True)
    fe = front_end(dev)
    las_sets = [synth_las_batch([synth.synth_tile(N, 1000 + 16 * s + i, clustered=(i % 2 == 1)) for i in range(B)], None)
                for s in range(SLOTS)]
    g = torch.Generator().manual_seed(2)
    imgs8 = [torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g) for _ in range(SLOTS)]
    feeds = {"fp32": torch.float32, "uint8": torch.uint8}
    with torch.no_grad():
        for mode in ("concat", "tokens"):
            pipes = {k: make_pipeline(fe, mode, dt, las_sets, imgs8) for k, dt in feeds.items()}
            runs = {k: [] for k in feeds}
            for _ in range(3):
                for k in feeds:
                    r = measure(pipes[k], args.seconds)
                    runs[k].append(r)
                    print(mode, k, json.dumps(r), flush=True)
            torch.cuda.synchronize()
            # every slot keeps its own batch, so slot i of either pipeline holds the result of batch i
            same = all(torch.equal(a.out.view(torch.int32), b.out.view(torch.int32))
                       for a, b in zip(pipes["fp32"].slots, pipes["uint8"].slots))
            assert same, f"{mode}: the uint8 feed computed something else than the fp32 feed"
            result["pipeline"][mode] = {
                k: {"h2d_bytes_per_step": pipes[k].h2d_bytes_per_step, "runs": runs[k],
                    "tiles_per_s_median": sorted(r["tiles_per_s"] for r in runs[k])[1]} for k in feeds}
            result["pipeline"][mode]["outputs_bit_identical"] = same
            del pipes
            torch.cuda.empty_cache()
        # the patch embedding alone
        g = torch.Generator().manual_seed(3)
        sets8 = [torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g).to(dev) for _ in range(KSETS)]
        sets32 = [fe.image_embed.expand_pixels(x) for x in sets8]
        outs = {"concat (fp32 NCHW, c_total 2C)": (torch.empty(B, 2 * C, 28, 28, device=dev), P3P_LAYOUT_NCHW),
                "tokens (16-bit NLC, c_total 2C)": (torch.empty(B, 28, 28, 2 * C, dtype=fe.fusion_layer.operand_dtype, device=dev),
                                                    P3P_LAYOUT_NLC)}
        for name, (out, layout) in outs.items():
            t = {"fp32": [], "uint8": []}
            for _ in range(3):
                t["fp32"].append(time_kernel(fe, sets32, out, layout, 2 * C))
                t["uint8"].append(time_kernel(fe, sets8, out, layout, 2 * C))
            result["patch_embed_kernel_us"][name] = t
            print("patch embed", name, json.dumps(t), flush=True)
    print(json.dumps(result["pipeline"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
