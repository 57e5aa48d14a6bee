"""GPU tests of the fused training step (csrc/pfn_train.cu, pixelspointspolygons_b200/train.py) at its edges, against the
same checker and bars as tests/test_gpu_train.py: the float64 dense autograd step (encoder.forward_dense_reference) on the
same pillars; forward within 1e-4 of scale, gradients through assert_grad_close, running buffers within rtol 1e-4 and
num_batches_tracked exact.

Edges: the C / M limits of the contract (C = 512 with M = 512, C not a multiple of 32, M = 1, M not a power of two);
pillars cut by max_voxels and pillars that lose their canvas cell (they count in the batch statistics but get no gradient
through `out`); empty tiles, first, in the middle and alone; the skewed batches the moment scheme is most sensitive to;
other canvases; the full 8 x 100 k batch; buffers that start as NaN / 0xFF; SyncBatchNorm with an empty or nearly empty
rank; and shapes outside the contract, refused before anything changes."""
import threading

import numpy as np
import pytest
import torch

from oracle import pillars_oracle as po
from p3p_cases import edge_cases, pillar_block
from pixelspointspolygons_b200 import PointPillarsEncoder, default_cfg
from pixelspointspolygons_b200 import train as p3p_train
from test_gpu_train import PARAMS, assert_grad_close, build, dense_step, grad_errors, nested, rel

pytestmark = pytest.mark.gpu

F = np.float32


def build_on(dev, M=64, C=384, seed=21, center_alias=True, max_voxels=(784, 784), drop_overflow=False, in_width=224,
             in_height=224, output_shape=(28, 28)):
    """build() of test_gpu_train on another grid (max_voxels: (train, test); output_shape: (ny, nx))."""
    cfg = default_cfg(device=str(dev), in_size=in_width, max_num_points_per_voxel=M, max_num_voxels=max_voxels,
                      patch_feature_dim=C, p3p_center_alias=center_alias, p3p_drop_overflow=drop_overflow,
                      in_height=in_height, in_width=in_width)
    enc = PointPillarsEncoder(cfg, voxel_encoder={"in_channels": 3, "feat_channels": [64, C]},
                              scatter={"in_channels": C, "output_shape": list(output_shape)}).to(dev)
    sd, _ = po.synth_weights(seed, feat_channels=(64, C))
    enc.load_state_dict(sd)
    return enc.train()


def check_step(enc, tiles, what, seed=17):
    """One fused training step against the float64 dense step on the same batch; -> the fused output."""
    dev = next(enc.parameters()).device
    x = nested(tiles, dev)
    C, hw = enc.channels, enc.ny * enc.nx
    weight = torch.randn(len(tiles), hw, C, generator=torch.Generator().manual_seed(seed)).to(dev)
    ref_out, ref_grads, ref_bufs = dense_step(enc, x, weight)

    out = enc(x)
    assert out.shape == (len(tiles), hw, C) and out.requires_grad
    (out * weight).sum().backward()
    assert rel(out.detach(), ref_out) <= 1e-4, (what, "forward", rel(out.detach(), ref_out))
    named = dict(enc.voxel_encoder.named_parameters())
    t32 = None  # torch's own fp32 dense step: only needed where the strict bound does not hold
    for n in PARAMS:
        got = named[n].grad
        assert got is not None and torch.isfinite(got).all(), (what, n)
        q99, rms, mx = grad_errors(got, ref_grads[n])
        if not (q99 <= 2e-4 and rms <= 1e-3 and mx <= 2e-2) and t32 is None:
            _, t32, _ = dense_step(enc, x, weight, torch.float32)
        assert_grad_close(got, ref_grads[n], t32[n] if t32 is not None else ref_grads[n], (what, n))
    for n, b in enc.voxel_encoder.named_buffers():
        if b.dtype.is_floating_point:
            assert torch.isfinite(b).all(), (what, n)
            assert torch.allclose(b.double(), ref_bufs[n], rtol=1e-4, atol=1e-6), (what, n)
        else:
            assert int(b) == int(ref_bufs[n]), (what, n)
    return out.detach()


def planted(M, seed, others):
    """One tile with pillars of exactly M (no padded row), M - 1 (one padded row) and M + 5 (cut to M) points, and the
    points of `others` outside those three cells."""
    cells = ((3, 3, M), (10, 12, M - 1), (20, 5, M + 5))
    keep = np.ones(len(others), bool)
    for cx, cy, _ in cells:
        keep &= ~((np.floor(others[:, 0] / 8) == cx) & (np.floor(others[:, 1] / 8) == cy))
    blocks = [pillar_block(cx, cy, n, seed + i) for i, (cx, cy, n) in enumerate(cells)]
    return np.concatenate(blocks + [others[keep]])


# ---------------------------------------------------------------------------------------------------------------- limits
@pytest.mark.parametrize("case", ["c512_m512", "c512_m64", "c200", "m1", "m100"])
def test_limits_match_dense_autograd(cuda_device, case):
    """C = 512 with M = 512 is the largest CTA of backward pass 1 (229 776 bytes of shared memory for its dW1 block);
    C = 200 leaves idle lanes in the last warp of the thread-per-channel kernels; M = 1 has no padded row anywhere;
    M = 100 is not a power of two, with pillars of exactly M and M - 1 points."""
    if case == "c512_m512":
        M, C, tiles = 512, 512, [planted(512, 1, po.synth_tile(3000, 2)), po.synth_tile(30000, 3, clustered=True)]
    elif case == "c512_m64":
        M, C, tiles = 64, 512, [planted(64, 4, po.synth_tile(3000, 5)), po.synth_tile(20000, 6, clustered=True)]
    elif case == "c200":
        M, C, tiles = 64, 200, [po.synth_tile(20000, 7, clustered=True), po.synth_tile(3000, 8)]
    elif case == "m1":
        M, C, tiles = 1, 384, [po.synth_tile(9000, 9), po.synth_tile(500, 10)]
    else:
        M, C, tiles = 100, 384, [planted(100, 11, po.synth_tile(3000, 12)), po.synth_tile(20000, 13, clustered=True)]
    enc = build(cuda_device, M=M, C=C, seed=21)
    check_step(enc, tiles, case)
    assert int(enc.voxel_encoder.pfn_layers[1].norm.num_batches_tracked) == 1


# ---------------------------------------------------------------------------------------- cut and overwritten pillars
@pytest.mark.parametrize("name", ["vmax_cut", "vmax_cut_with_alias"])
def test_max_voxels_cut_matches_dense_autograd(cuda_device, name):
    """Train-mode max_voxels (max_voxels[0]) cuts every tile of the batch, the normal one too."""
    tiles, kw = edge_cases()[name]
    enc = build_on(cuda_device, max_voxels=kw["max_voxels"])
    check_step(enc, tiles + [po.synth_tile(3000, 41)], name)


@pytest.mark.parametrize("drop_overflow", [False, True])
def test_pillars_that_lose_their_cell_match_dense_autograd(cuda_device, drop_overflow):
    """A z-layer-1 pillar overwrites its cell (z = 100), an x = 224 point aliases the next row's first cell, and the
    overflowing hashes of `drop_overflow`, in one batch with a normal tile.  The pillars without a canvas cell count in
    both BatchNorms' statistics but get no gradient through `out`."""
    cases = edge_cases()
    tiles = [t for name in ("z100_overwrites_cell", "x224_then_alias", "drop_overflow") for t in cases[name][0]]
    tiles.append(po.synth_tile(5000, 42))
    enc = build_on(cuda_device, drop_overflow=drop_overflow)
    check_step(enc, tiles, ("overwritten", drop_overflow))


# ------------------------------------------------------------------------------------------------------- empty tiles
@pytest.mark.parametrize("case", ["empty_first", "empty_middle_and_one_point"])
def test_empty_tiles_match_dense_autograd(cuda_device, case):
    """An empty first tile moves the sample the layer-1 centre is taken from (the first 128 entries of the pillar list)."""
    empty = np.zeros((0, 3), F)
    if case == "empty_first":
        tiles = [empty, po.synth_tile(5000, 43), po.synth_tile(800, 44)]
    else:
        tiles = [po.synth_tile(4000, 45), empty, po.synth_tile(1, 46)]
    check_step(build(cuda_device, seed=21), tiles, case)


def test_all_empty_batch(cuda_device):
    """No pillar at all: the output is zero and the gradients are zero.  The running statistics keep their values and
    num_batches_tracked counts the batch -- what torch's BatchNorm1d does with an empty input (its batch statistics are
    0 / 0, and it skips the update; tests/test_train_protocol.py checks update_running_stats against it) -- so no NaN
    reaches them."""
    enc = build(cuda_device, seed=21)
    before = {n: b.clone() for n, b in enc.voxel_encoder.named_buffers()}
    x = nested([np.zeros((0, 3), F), np.zeros((0, 3), F)], cuda_device)
    out = enc(x)
    assert out.shape == (2, 784, 384) and out.requires_grad
    assert torch.equal(out.detach(), torch.zeros_like(out))
    weight = torch.randn(2, 784, 384, generator=torch.Generator().manual_seed(5)).to(cuda_device)
    (out * weight).sum().backward()
    for n, p in enc.voxel_encoder.named_parameters():
        assert p.grad is not None and torch.equal(p.grad, torch.zeros_like(p)), n
    for n, b in enc.voxel_encoder.named_buffers():
        if n.endswith("num_batches_tracked"):
            assert int(b) == int(before[n]) + 1, n
        else:
            assert torch.equal(b, before[n]), n


# --------------------------------------------------------------------------------------------------- skewed batches
def plateau_tile(n, seed):
    """What MinMaxScaler makes of a tile with one low-noise return: z in [97, 100], one point at 0 and one at 100."""
    rng = np.random.default_rng(seed)
    pts = np.concatenate([rng.uniform(0.0, 224.0, (n, 2)), rng.uniform(97.0, 100.0, (n, 1))], 1).astype(F)
    pts[:, :2] = np.minimum(pts[:, :2], np.nextafter(F(224), F(0)))
    pts[:, 2] = np.minimum(pts[:, 2], np.nextafter(F(100), F(0)))
    pts[rng.integers(0, n), 2] = 0.0
    pts[rng.integers(0, n), 2] = 100.0
    return pts


@pytest.mark.parametrize("center_alias", [True, False])
def test_z_plateau_batch_matches_dense_autograd(cuda_device, center_alias):
    """100 k points per tile: every pillar is full, so no padded zero row dilutes the layer-0 variance of channel 2
    (absolute z, about 98.5 with a spread of 0.9), where E[y^2] - E[y]^2 cancels; without center_alias channels 0 and 1
    carry absolute x and y as well."""
    enc = build(cuda_device, seed=21, center_alias=center_alias)
    check_step(enc, [plateau_tile(100_000, 47), plateau_tile(100_000, 48)], ("plateau", center_alias))


def test_atypical_first_pillars_match_dense_autograd(cuda_device):
    """The layer-1 centre is taken from the first 128 pillars of the list: here all of them sit in a sparse tile of low
    z, far from the batch's mean (two dense tiles of high z)."""
    rng = np.random.default_rng(49)
    low = np.concatenate([rng.uniform(0.0, 224.0, (300, 2)), rng.uniform(0.0, 3.0, (300, 1))], 1).astype(F)
    high = []
    for seed in (50, 51):
        t = po.synth_tile(60000, seed, clustered=True)
        t[:, 2] = F(90.0) + t[:, 2] * F(0.1)
        high.append(t)
    check_step(build(cuda_device, seed=21), [low] + high, "atypical_first")


# ------------------------------------------------------------------------------------------------------- other grids
def test_odd_canvas_matches_dense_autograd(cuda_device):
    """216-px tiles -> 27 x 27 = 729 cells (not a multiple of 8), as test_odd_canvas_takes_the_general_path in eval mode."""
    enc = build_on(cuda_device, in_width=216, in_height=216, output_shape=(27, 27), max_voxels=(729, 729))
    tiles = []
    for i, n in enumerate((9000, 40, 20000)):
        t = po.synth_tile(n, 700 + i, clustered=(i == 2))
        t[:, :2] *= F(216.0 / 224.0)
        tiles.append(t)
    check_step(enc, tiles, "odd_canvas")


def test_non_square_canvas_matches_dense_autograd(cuda_device):
    """224 x 160 px -> ny = 20 rows of nx = 28 cells: train_list_kernel rebuilds each pillar's cell from its packed
    coordinates with nx, so a transposed axis would put features in the wrong cells."""
    enc = build_on(cuda_device, in_width=224, in_height=160, output_shape=(20, 28), max_voxels=(560, 560))
    assert (enc.ny, enc.nx) == (20, 28)
    tiles = []
    for i, n in enumerate((12000, 3000)):
        t = po.synth_tile(n, 710 + i, clustered=(i == 0))
        t[:, 1] *= F(160.0 / 224.0)
        tiles.append(t)
    out = check_step(enc, tiles, "non_square")
    # the occupied cells are those of the points: rows y // 8 < 20, columns x // 8 < 28
    occupied = out[0].abs().amax(1) > 0
    pts = tiles[0]
    cells = np.unique((np.floor(pts[:, 1] / 8).astype(int) * 28 + np.floor(pts[:, 0] / 8).astype(int)))
    assert set(torch.nonzero(occupied).flatten().tolist()) <= set(cells.tolist())


# --------------------------------------------------------------------------------------------------------- full size
def test_full_batch_matches_dense_autograd(cuda_device):
    """8 tiles x 100 k points, M = 64, C = 384: every pillar full, every tile cut at max_voxels by its z = 100 pillar."""
    tiles = [po.synth_tile(100_000, 60 + i) for i in range(8)]
    check_step(build(cuda_device, seed=21), tiles, "full")


# ------------------------------------------------------------------------------------------------- unwritten buffers
class _PoisonedTorch:
    """torch, except that empty / empty_like return NaN-filled floating and 0xFF-filled integer buffers."""

    def __init__(self, real):
        self._real = real

    def __getattr__(self, name):
        return getattr(self._real, name)

    @staticmethod
    def _poison(t):
        return t.fill_(float("nan")) if t.is_floating_point() else t.fill_(-1 if t.dtype != torch.uint8 else 255)

    def empty(self, *args, **kwargs):
        return self._poison(self._real.empty(*args, **kwargs))

    def empty_like(self, *args, **kwargs):
        return self._poison(self._real.empty_like(*args, **kwargs))


def test_unwritten_buffers_are_never_read(cuda_device, monkeypatch):
    """Every buffer the training step allocates (workspace, state, out, route = du + amax, the gradients) starts as NaN /
    0xFF: the step must give what it gives on fresh allocations.  du is written only for pillars that own their canvas
    cell, so this also checks that backward pass 2 reads it for no other pillar (z = 100 pillars overwrite cells here).
    The backward's fp32 shared-memory atomics are not order-stable: the comparison is within 1e-5, not bit for bit."""
    tiles = [po.synth_tile(20000, 70, clustered=True), po.synth_tile(3000, 71), po.synth_tile(40, 72)]
    weight = torch.randn(3, 784, 384, generator=torch.Generator().manual_seed(7)).to(cuda_device)

    def step():
        enc = build(cuda_device, seed=21)
        out = enc(nested(tiles, cuda_device))
        (out * weight).sum().backward()
        torch.cuda.synchronize()
        return out.detach(), dict(enc.voxel_encoder.named_parameters()), dict(enc.voxel_encoder.named_buffers())

    out_c, par_c, buf_c = step()
    monkeypatch.setattr(p3p_train, "torch", _PoisonedTorch(torch))
    out_p, par_p, buf_p = step()
    monkeypatch.undo()
    assert torch.isfinite(out_p).all()
    assert rel(out_p, out_c) <= 1e-5
    for n in PARAMS:
        assert torch.isfinite(par_p[n].grad).all(), n
        assert rel(par_p[n].grad, par_c[n].grad) <= 1e-5, (n, rel(par_p[n].grad, par_c[n].grad))
    for n, b in buf_p.items():
        assert torch.allclose(b.double(), buf_c[n].double(), rtol=1e-6, atol=1e-9), n


# ------------------------------------------------------------------------------------ SyncBatchNorm, unequal ranks
def two_ranks(dev, tiles0, tiles1, weight):
    """The two-threads-one-GPU reducer of test_training_two_simulated_ranks_match_whole_batch: -> [(out, grads)] x 2."""
    ranks = [build(dev, seed=9), build(dev, seed=9)]
    barrier = threading.Barrier(2)
    slots, lock = {}, threading.Lock()

    def reducer(rank):
        def red(t, what):
            torch.cuda.synchronize()
            with lock:
                slots[(what, rank)] = t.clone()
            barrier.wait()
            total = slots[(what, 0)] + slots[(what, 1)]
            barrier.wait()
            t.copy_(total)
        return red

    results, errors = {}, []
    parts = [(tiles0, weight[:len(tiles0)]), (tiles1, weight[len(tiles0):])]

    def run(rank):
        try:
            with torch.cuda.device(dev):
                enc = ranks[rank]
                values, offsets, B = enc._pack(nested(parts[rank][0], dev))
                tensors = [dict(enc.voxel_encoder.named_parameters())[n] for n in PARAMS]
                out, ctx = p3p_train.train_forward(enc, values, offsets, B, tensors, reduce_fn=reducer(rank))
                grads = p3p_train.train_backward(ctx, parts[rank][1], reduce_fn=reducer(rank))
                torch.cuda.synchronize()
                results[rank] = (out, grads)
        except Exception as e:  # pragma: no cover
            errors.append(e)
            barrier.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    return [results[0], results[1]], ranks


@pytest.mark.parametrize("case", ["empty_rank", "unequal_ranks"])
def test_sync_batchnorm_with_an_empty_rank_matches_whole_batch(cuda_device, case):
    """Rank 1 holds only empty tiles, or a few points against rank 0's 70 k: the concatenated outputs and the summed
    gradients are those of the whole batch on one rank."""
    empty = np.zeros((0, 3), F)
    tiles0 = [po.synth_tile(40000, 80, clustered=True), po.synth_tile(30000, 81)]
    tiles1 = [empty, empty] if case == "empty_rank" else [po.synth_tile(50, 82), po.synth_tile(1, 83)]
    weight = torch.randn(4, 784, 384, generator=torch.Generator().manual_seed(3)).to(cuda_device)

    whole = build(cuda_device, seed=9)
    out_w = whole(nested(tiles0 + tiles1, cuda_device))
    (out_w * weight).sum().backward()
    torch.cuda.synchronize()

    results, ranks = two_ranks(cuda_device, tiles0, tiles1, weight)
    out_s = torch.cat([results[0][0], results[1][0]], 0)
    assert rel(out_s, out_w.detach()) <= 1e-5
    if case == "empty_rank":
        assert torch.equal(results[1][0], torch.zeros_like(results[1][0]))
    named = dict(whole.voxel_encoder.named_parameters())
    for i, n in enumerate(PARAMS):
        assert torch.isfinite(results[1][1][i]).all(), n
        e = rel(results[0][1][i] + results[1][1][i], named[n].grad)
        assert e <= 1e-5, (n, e)
    for r in ranks:
        for (n, b), (_, bw) in zip(whole.voxel_encoder.named_buffers(), r.voxel_encoder.named_buffers()):
            assert torch.allclose(b.double(), bw.double(), rtol=1e-6, atol=1e-9), n


# --------------------------------------------------------------------------------------------------------- rejection
@pytest.mark.parametrize("C, M, words", [(513, 64, "1..512 channels"), (384, 1024, "max_points <= 512"),
                                         (513, 1024, "1..512 channels")], ids=["c513", "m1024", "c513_m1024"])
def test_unsupported_shapes_are_refused_before_anything_changes(cuda_device, C, M, words):
    """Outside C <= 512, M <= 512 the forward raises, and no running buffer, num_batches_tracked or gradient has moved."""
    enc = build(cuda_device, M=M, C=C, seed=1)
    before = {n: b.clone() for n, b in enc.voxel_encoder.named_buffers()}
    x = nested([po.synth_tile(2000, 1)], cuda_device)
    with pytest.raises(Exception, match=words):
        enc(x)
    torch.cuda.synchronize()
    for n, b in enc.voxel_encoder.named_buffers():
        assert torch.equal(b, before[n]), n
    assert all(p.grad is None for p in enc.voxel_encoder.parameters())
