"""CPU tests of the training protocol of SURVEY 8f rank 4 (host logic + the algebra the kernels of csrc/pfn_train.cu use).

`fused_math` restates, in float64 torch on dense (V, M, 8) decorated rows, exactly what the kernels compute: BatchNorm
batch statistics from input moments, the backward through both maxima and both BatchNorms as sparse rows + the batch
constants kvec / Q, parameter gradients from the stored moments -- with the four packed exchanges of the SyncBatchNorm
protocol as a `reduce` callback.  It is checked against autograd over the dense modules of encoder.py (nn.Linear +
nn.BatchNorm1d in train mode), single process and as two gloo ranks through train.exchange / train.sync_group."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from pixelspointspolygons_b200 import train as p3p_train
from pixelspointspolygons_b200.encoder import PFNLayer

EPS = 1e-3


def make_case(V, M, C, seed):
    g = torch.Generator().manual_seed(seed)
    n = torch.randint(1, M + 1, (V,), generator=g)
    n[0] = M
    d = torch.randn(V, M, 8, generator=g, dtype=torch.float64) * 3.0
    d = d * (torch.arange(M).view(1, M, 1) < n.view(V, 1, 1))
    l0, l1 = PFNLayer(8, 64, False).double().train(), PFNLayer(64, C, True).double().train()
    with torch.no_grad():
        for l in (l0, l1):
            l.linear.weight.copy_(torch.randn(l.linear.weight.shape, generator=g, dtype=torch.float64) * 0.2)
            l.norm.weight.copy_(torch.rand(l.norm.weight.shape, generator=g, dtype=torch.float64) + 0.5)
            l.norm.bias.copy_(torch.randn(l.norm.bias.shape, generator=g, dtype=torch.float64) * 0.1)
        l1.norm.weight[0] = -0.7  # a negative BatchNorm scale: the winning row is the minimum of the linear output
    gout = torch.randn(V, C, generator=g, dtype=torch.float64)
    gout[1] = 0.0  # a pillar that lost its canvas cell
    return d, n, l0, l1, gout


def dense_autograd(d, l0, l1, gout):
    for l in (l0, l1):
        l.zero_grad()
    out = l1(l0(d)).squeeze(1)
    (out * gout).sum().backward()
    return out.detach(), [l0.linear.weight.grad, l0.norm.weight.grad, l0.norm.bias.grad,
                          l1.linear.weight.grad, l1.norm.weight.grad, l1.norm.bias.grad]


def fused_math(d, l0, l1, gout, reduce=lambda t: None):
    W0, g0, b0 = l0.linear.weight.detach(), l0.norm.weight.detach(), l0.norm.bias.detach()
    W1, g1, b1 = l1.linear.weight.detach(), l1.norm.weight.detach(), l1.norm.bias.detach()
    V, M, _ = d.shape
    C = W1.shape[0]
    rows = torch.tensor([float(V * M)], dtype=torch.float64)
    s, S = d.sum((0, 1)), torch.einsum("vmi,vmj->ij", d, d)
    sums0 = torch.cat([W0 @ s, torch.einsum("ki,ij,kj->k", W0, S, W0), rows])
    reduce(sums0)
    R = sums0[-1]
    mu0 = sums0[:32] / R
    rs0 = 1.0 / torch.sqrt(sums0[32:64] / R - mu0 ** 2 + EPS)
    yh0 = (d @ W0.T - mu0) * rs0
    x0 = torch.relu(g0 * yh0 + b0)
    hmax, am0 = x0.max(1)
    z = torch.cat([x0, hmax[:, None, :].expand(-1, M, -1)], -1)
    sz, Z = z.sum((0, 1)), torch.einsum("vmi,vmj->ij", z, z)
    sums1 = torch.cat([W1 @ sz, torch.einsum("ci,ij,cj->c", W1, Z, W1), rows])
    reduce(sums1)
    mu1 = sums1[:C] / R
    rs1 = 1.0 / torch.sqrt(sums1[C:2 * C] / R - mu1 ** 2 + EPS)
    a1 = g1 * rs1
    y1 = z @ W1.T
    u_all = a1 * (y1 - mu1) + b1
    u, am1 = u_all.max(1)
    out = torch.relu(u)
    # backward pass 1
    du = gout * (u > 0)
    ystar = y1.gather(1, am1[:, None, :]).squeeze(1)
    zstar = z[torch.arange(V)[:, None], am1]                      # (V, C, 64)
    dbeta1, dgamma1 = du.sum(0), (du * (ystar - mu1) * rs1).sum(0)
    A1 = torch.einsum("vc,vcj->cj", du, zstar)
    back1g = torch.cat([dbeta1, dgamma1]).clone()
    reduce(back1g)
    coefk = a1 / R * (-back1g[:C] + back1g[C:] * rs1 * mu1)
    coefq = a1 / R * back1g[C:] * rs1
    kvec, Q = coefk @ W1, torch.einsum("c,cj,ci->ji", coefq, W1, W1)
    # backward pass 2
    G = torch.zeros(V, M, 64, dtype=torch.float64)
    G.index_put_((torch.arange(V)[:, None].expand(V, C), am1), (a1 * du)[:, :, None] * W1[None], accumulate=True)
    dz = G + kvec - z @ Q.T
    dx0 = dz[:, :, :32].clone()
    dx0[torch.arange(V)[:, None].expand(V, 32), am0, torch.arange(32)[None].expand(V, 32)] += dz[:, :, 32:].sum(1)
    du0 = dx0 * (x0 > 0)
    dbeta0, dgamma0 = du0.sum((0, 1)), (du0 * yh0).sum((0, 1))
    A0 = torch.einsum("vmk,vmi->ki", du0, d)
    back0g = torch.cat([dbeta0, dgamma0]).clone()
    reduce(back0g)
    a0 = g0 * rs0
    dW1 = a1[:, None] * (A1 - (back1g[:C] / R)[:, None] * sz - (back1g[C:] / R * rs1)[:, None] * (W1 @ Z - mu1[:, None] * sz))
    dW0 = a0[:, None] * (A0 - (back0g[:32] / R)[:, None] * s - (back0g[32:] / R * rs0)[:, None] * (W0 @ S - mu0[:, None] * s))
    return out, [dW0, dgamma0, dbeta0, dW1, dgamma1, dbeta1]


def close(a, b, tol=1e-9):
    return (a - b).abs().max().item() <= tol * max(b.abs().max().item(), 1e-30)


@pytest.mark.parametrize("V,M,C", [(12, 8, 16), (40, 16, 48), (3, 64, 8)])
def test_moment_statistics_and_closed_form_backward_match_dense_autograd(V, M, C):
    d, n, l0, l1, gout = make_case(V, M, C, seed=V + M)
    ref_out, ref_grads = dense_autograd(d, l0, l1, gout)
    out, grads = fused_math(d, l0, l1, gout)
    assert close(out, ref_out)
    for g, r in zip(grads, ref_grads):
        assert close(g, r, 1e-8)


def test_state_layout_matches_the_header():
    total, offs = p3p_train.state_layout(384)
    keys = list(offs)
    assert keys == list(p3p_train._STATE_FIELDS) and offs["mom0"] == 0
    sizes = dict(mom0=73, sums0=65, bn0=64, mom1=64 + 4096, sums1=769, bn1=768, cen=65, back1=768, back1g=768, A1=384 * 64, kq=64 + 4096,
                 back0=64, back0g=64, A0=256)
    for a, b in zip(keys[:-1], keys[1:]):
        assert offs[b] - offs[a] >= sizes[a] and offs[a] % 2 == 0
    assert total >= offs["A0"] + 256
    with pytest.raises(Exception):
        p3p_train.state_layout(4096)


def test_update_running_stats_is_batchnorm1d_train_mode():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(50, 6, generator=g) * 2 + 1
    ref = nn.BatchNorm1d(6, eps=1e-3, momentum=0.01).train()
    ref(x)
    bn = nn.BatchNorm1d(6, eps=1e-3, momentum=0.01).train()
    p3p_train.update_running_stats(bn, x.mean(0), x.var(0, unbiased=False), torch.tensor(50.0, dtype=torch.float64))
    assert torch.allclose(bn.running_mean, ref.running_mean, atol=1e-7) and torch.allclose(bn.running_var, ref.running_var, atol=1e-7)
    assert int(bn.num_batches_tracked) == 1
    assert p3p_train.sync_group(bn) is None and p3p_train.sync_group(nn.SyncBatchNorm(6)) is None  # no process group here


@pytest.mark.parametrize("momentum", [0.01, None])
def test_update_running_stats_on_an_empty_batch_is_batchnorm1d_train_mode(momentum):
    """No row in the batch: torch's BatchNorm1d counts the batch but keeps its running statistics (and writes no NaN)."""
    g = torch.Generator().manual_seed(1)
    ref = nn.BatchNorm1d(6, eps=1e-3, momentum=momentum).train()
    bn = nn.BatchNorm1d(6, eps=1e-3, momentum=momentum).train()
    for m in (ref, bn):
        m.running_mean.copy_(torch.randn(6, generator=g))
        m.running_var.copy_(torch.rand(6, generator=g) + 0.5)
    bn.load_state_dict(ref.state_dict())
    ref(torch.zeros(0, 6))
    p3p_train.update_running_stats(bn, torch.zeros(6), torch.zeros(6), torch.tensor(0.0, dtype=torch.float64))
    assert torch.equal(bn.running_mean, ref.running_mean) and torch.equal(bn.running_var, ref.running_var)
    assert int(bn.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    x = torch.randn(30, 6, generator=g)  # and the next, non-empty batch is counted as the second
    ref(x)
    p3p_train.update_running_stats(bn, x.mean(0), x.var(0, unbiased=False), torch.tensor(30.0, dtype=torch.float64))
    assert torch.allclose(bn.running_mean, ref.running_mean, atol=1e-7) and torch.allclose(bn.running_var, ref.running_var, atol=1e-7)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        d, n, l0, l1, gout = make_case(20, 8, 24, seed=5)
        lo, hi = rank * 10, rank * 10 + 10
        group = p3p_train.sync_group(nn.SyncBatchNorm(4))  # the layer's group: the default one
        assert group is not None and p3p_train.sync_group(nn.BatchNorm1d(4)) is None
        out, grads = fused_math(d[lo:hi], l0, l1, gout[lo:hi], reduce=lambda t: p3p_train.exchange(t, group))
        for g in grads:  # what DDP's gradient all-reduce does (sum here; DDP divides by the world size)
            dist.all_reduce(g)
        outs = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(outs, out)
        if rank == 0:
            torch.save((torch.cat(outs), grads), out_path)
    finally:
        dist.destroy_process_group()


def test_two_rank_syncbn_exchange_equals_whole_batch(tmp_path):
    path = str(tmp_path / "r.pt")
    mp.spawn(_worker, args=(2, _free_port(), path), nprocs=2, join=True)
    out, grads = torch.load(path)
    d, n, l0, l1, gout = make_case(20, 8, 24, seed=5)
    ref_out, ref_grads = dense_autograd(d, l0, l1, gout)
    assert close(out, ref_out)
    for g, r in zip(grads, ref_grads):
        assert close(g, r, 1e-8)
