"""bench.py --dump-outputs: the file holds what the last timed step handed its caller, float32, within the size cap."""
import importlib.util
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_writes_the_step_output_and_samples_tiles_above_the_cap(tmp_path, monkeypatch):
    bench = load_bench()
    outs = [torch.rand(6, 5, 4, generator=torch.Generator().manual_seed(s)) for s in range(3)]
    w = types.SimpleNamespace(outs=outs, sets=3, workload="lidar")
    d = bench.dump_outputs(w, 4, str(tmp_path / "all"))  # step 4 ran on set 1
    got = np.load(tmp_path / "all" / "tokens.npy")
    assert got.dtype == np.float32 and d["tiles"] == "all" and np.array_equal(got, outs[1].numpy())
    # above the cap: a fixed, seeded sample of whole tiles, the same one every time
    monkeypatch.setattr(bench, "DUMP_LIMIT", 2 * 5 * 4 * 4)
    w.workload = "fusion"
    d1 = bench.dump_outputs(w, 4, str(tmp_path / "a"))
    d2 = bench.dump_outputs(w, 4, str(tmp_path / "b"))
    a, b = np.load(tmp_path / "a" / "features.npy"), np.load(tmp_path / "b" / "features.npy")
    assert len(d1["tiles"]) == 2 and d1["tiles"] == sorted(d1["tiles"]) == d2["tiles"]
    assert a.nbytes <= bench.DUMP_LIMIT and np.array_equal(a, b) and np.array_equal(a, outs[1].numpy()[d1["tiles"]])


def test_reference_arm_rejects_dump_outputs(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 2 and "--dump-outputs" in p.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["lidar", "fusion"])
def test_dump_matches_the_module_on_the_last_step_inputs(cuda_device, tmp_path, workload):
    from pixelspointspolygons_b200 import PointPillarsEncoder, default_cfg
    from pixelspointspolygons_b200.fusion import EarlyFusionFrontEnd
    from tools.synth import synth_tile, synth_weights

    B, N, warmup, steps = 2, 3000, 2, 3
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--batch", str(B), "--points", str(N),
                        "--warmup", str(warmup), "--steps", str(steps), "--no-sub-results", "--no-cpu-baseline", "--min-seconds", "0.05",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["timed_region"]["steps_timed"] == steps and line["dump_outputs"]["step"] == warmup + steps - 1
    name = "features" if workload == "fusion" else "tokens"
    assert sorted(os.listdir(tmp_path)) == [name + ".npy"]
    got = np.load(tmp_path / (name + ".npy"))
    assert got.dtype == np.float32

    # the inputs of that step: bench.py's Workload keeps >= 8 rotating sets and step i < 8 reads set i, whose tiles and image
    # are seeded 1000 + 16 i + tile and 1000 + i on rank 0
    s = warmup + steps - 1
    tiles = [synth_tile(N, 1000 + 16 * s + i, clustered=(i % 2 == 1)) for i in range(B)]
    x = torch.nested.nested_tensor([torch.from_numpy(t) for t in tiles], layout=torch.jagged).to(cuda_device)
    cfg = default_cfg(device=str(cuda_device), max_num_points_per_voxel=64, p3p_precision="fp16")
    sd, sdi = synth_weights(0)
    with torch.no_grad():
        if workload == "fusion":
            fe = EarlyFusionFrontEnd(cfg).to(cuda_device).eval()
            fe.lidar_embed.load_state_dict(sd)
            fe.image_embed.load_state_dict(sdi)
            img = torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(1000 + s)).to(cuda_device)
            want = fe(img, x)
        else:
            enc = PointPillarsEncoder(cfg, voxel_encoder={"in_channels": 3, "feat_channels": [64, 384]},
                                      scatter={"in_channels": 384, "output_shape": [28, 28]}).to(cuda_device).eval()
            enc.load_state_dict(sd)
            want = enc(x, return_flattened=True)
    assert np.array_equal(got, want.cpu().numpy())
