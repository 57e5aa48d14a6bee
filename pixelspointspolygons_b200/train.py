"""Training step of the LiDAR encoder on the fused kernels (SURVEY 8f rank 4).

The reference trains the encoder through autograd over Open3D-ML's dense PillarFeatureNet
(R:pixelspointspolygons/models/pointpillars/pointpillars_o3d.py:92-95, voxelize under no_grad) inside DDP, its
BatchNorm1d layers converted to SyncBatchNorm (R:pixelspointspolygons/models/pix2poly/model_pix2poly.py:326-328).
`FusedPFNTrain` is that graph as one autograd node over libp3p.so (csrc/pfn_train.cu): batch statistics from input
moments (two passes over the kept points), an exact-fp32 forward that keeps the winning row of every (pillar, channel), and
a backward that routes through both maxima and both BatchNorms without a (V, M, *) tensor.

Multi-GPU: under SyncBatchNorm the ranks exchange, per step, four small all-reduces (65 and 2C + 1 doubles forward,
2C and 64 doubles backward; SURVEY 8e) -- `exchange` below; the parameter gradients returned are this rank's share and
DDP averages them, exactly as for the reference module.  There is no CPU or eager fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib

_STATE_FIELDS = ("mom0", "sums0", "bn0", "mom1", "sums1", "bn1", "cen", "back1", "back1g", "A1", "kq", "back0", "back0g", "A0")


def state_layout(channels: int):
    """(total doubles, {field: offset}) of the training state buffer (p3p_pfn_train_state_doubles)."""
    offs = (C.c_int64 * len(_STATE_FIELDS))()
    total = _lib.lib().p3p_pfn_train_state_doubles(channels, offs)
    if total <= 0:
        _lib.check(-2, "p3p_pfn_train_state_doubles")
    return int(total), {k: int(offs[i]) for i, k in enumerate(_STATE_FIELDS)}


def sync_group(norm: nn.Module):
    """The process group to exchange BatchNorm sums over, or None: a SyncBatchNorm layer in an initialised job."""
    if isinstance(norm, nn.SyncBatchNorm) and dist.is_available() and dist.is_initialized():
        group = norm.process_group if norm.process_group is not None else dist.group.WORLD
        if dist.get_world_size(group) > 1:
            return group
    return None


def exchange(t: torch.Tensor, group) -> None:
    """Sum `t` (a view of the state buffer) over the ranks of `group` in place; no-op without a group."""
    if group is not None:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def update_running_stats(norm: nn.Module, mean: torch.Tensor, var_biased: torch.Tensor, rows: torch.Tensor) -> None:
    """What nn.BatchNorm1d.forward does to its buffers in train mode (momentum update with the unbiased variance).  A batch
    without a single row (no pillar on any rank) counts in num_batches_tracked but leaves the running statistics as they
    are, as torch's batch_norm does for an empty input; `rows` stays on the device, so this costs no synchronisation."""
    if not getattr(norm, "track_running_stats", True) or norm.running_mean is None:
        return
    with torch.no_grad():
        norm.num_batches_tracked += 1
        m = norm.momentum if norm.momentum is not None else 1.0 / norm.num_batches_tracked.to(torch.float64)
        m = (rows > 0).to(torch.float64) * m
        unbiased = var_biased.to(torch.float64) * (rows / torch.clamp(rows - 1.0, min=1.0))
        norm.running_mean.mul_(1.0 - m).add_((mean.to(torch.float64) * m).to(norm.running_mean.dtype))
        norm.running_var.mul_(1.0 - m).add_((unbiased * m).to(norm.running_var.dtype))


class _Ctx:
    """Everything one training forward leaves behind for its backward."""
    __slots__ = ("grid", "B", "total", "ws", "state", "offs", "params", "keep", "group", "channels", "route", "out")


def _params(enc, tensors) -> _lib.PfnParams:
    p = _lib.PfnParams()
    w0, g0, b0, w1, g1, b1 = tensors
    p.linear0_weight, p.norm0_weight, p.norm0_bias = w0.data_ptr(), g0.data_ptr(), b0.data_ptr()
    p.linear1_weight, p.norm1_weight, p.norm1_bias = w1.data_ptr(), g1.data_ptr(), b1.data_ptr()
    p.norm0_mean = p.norm0_var = p.norm1_mean = p.norm1_var = None
    p.eps = float(enc.voxel_encoder.pfn_layers[0].norm.eps)
    p.channels, p.center_alias = enc.channels, int(enc.center_alias)
    return p


def train_forward(enc, values: torch.Tensor, offsets: torch.Tensor, B: int, tensors, reduce_fn: Optional[Callable] = None):
    """Voxelize + batch statistics + PFN + scatter.  -> (out (B, ny nx, C) fp32, ctx).  `reduce_fn(tensor, what)` replaces
    the SyncBatchNorm all-reduce (tests drive several simulated ranks through it)."""
    l = _lib.lib()
    device = values.device
    norms = [enc.voxel_encoder.pfn_layers[0].norm, enc.voxel_encoder.pfn_layers[1].norm]
    group = sync_group(norms[0])
    red = reduce_fn if reduce_fn is not None else (lambda t, what: exchange(t, group))
    grid, total, Cc, hw = enc._grid(True), values.shape[0], enc.channels, enc.ny * enc.nx
    keep = [t.detach().contiguous() for t in tensors]
    for t in keep:
        if t.device != device or t.dtype != torch.float32:
            raise RuntimeError("PFN parameters must be float32 on the device of x_lidar")
    params = _params(enc, keep)
    n_state, offs = state_layout(Cc)
    stream = torch.cuda.current_stream(device).cuda_stream
    with torch.cuda.device(device):
        # this batch's own workspace: the pillar table must outlive the forward (the backward re-reads the kept points)
        ws = torch.empty(max(l.p3p_workspace_bytes(C.byref(grid), B, total), 1), dtype=torch.uint8, device=device)
        state = torch.empty(n_state, dtype=torch.float64, device=device)
        _lib.check(l.p3p_voxelize(values.data_ptr(), values.shape[1], offsets.data_ptr(), B, total, C.byref(grid), None,
                                  ws.data_ptr(), ws.numel(), stream), "p3p_voxelize")
        _lib.check(l.p3p_pfn_train_stats0(C.byref(grid), B, total, C.byref(params), state.data_ptr(), ws.data_ptr(), ws.numel(),
                                          stream), "p3p_pfn_train_stats0")
        red(state[offs["sums0"]:offs["sums0"] + 65], "sums0")
        _lib.check(l.p3p_pfn_train_stats1(C.byref(grid), B, total, C.byref(params), state.data_ptr(), ws.data_ptr(), ws.numel(),
                                          stream), "p3p_pfn_train_stats1")
        red(state[offs["sums1"]:offs["sums1"] + 2 * Cc + 1], "sums1")
        stats = torch.empty(2 * 32 + 2 * Cc, dtype=torch.float32, device=device)
        mean0, var0, mean1, var1 = stats[:32], stats[32:64], stats[64:64 + Cc], stats[64 + Cc:]
        _lib.check(l.p3p_pfn_train_stats2(C.byref(params), state.data_ptr(), mean0.data_ptr(), var0.data_ptr(), mean1.data_ptr(),
                                          var1.data_ptr(), stream), "p3p_pfn_train_stats2")
        route = torch.empty(max(l.p3p_pfn_train_route_bytes(C.byref(grid), B, Cc), 1), dtype=torch.uint8, device=device)
        out = torch.empty(B, hw, Cc, dtype=torch.float32, device=device)
        _lib.check(l.p3p_pfn_train_forward(C.byref(grid), B, total, C.byref(params), state.data_ptr(), out.data_ptr(),
                                           route.data_ptr(), ws.data_ptr(), ws.numel(), stream), "p3p_pfn_train_forward")
    rows0 = state[offs["sums0"] + 64]
    update_running_stats(norms[0], mean0, var0, rows0)
    update_running_stats(norms[1], mean1, var1, state[offs["sums1"] + 2 * Cc])
    ctx = _Ctx()
    ctx.grid, ctx.B, ctx.total, ctx.ws, ctx.state, ctx.offs = grid, B, total, ws, state, offs
    ctx.params, ctx.keep, ctx.group, ctx.channels, ctx.route, ctx.out = params, keep, group, Cc, route, out
    return out, ctx


def train_backward(ctx: _Ctx, grad_out: torch.Tensor, reduce_fn: Optional[Callable] = None):
    """Gradients of (linear0.weight, norm0.weight, norm0.bias, linear1.weight, norm1.weight, norm1.bias) -- this rank's share."""
    l = _lib.lib()
    device = ctx.state.device
    red = reduce_fn if reduce_fn is not None else (lambda t, what: exchange(t, ctx.group))
    g = grad_out.detach().to(torch.float32).contiguous()
    Cc, offs, state, ws, grid = ctx.channels, ctx.offs, ctx.state, ctx.ws, ctx.grid
    stream = torch.cuda.current_stream(device).cuda_stream
    with torch.cuda.device(device):
        route = ctx.route
        _lib.check(l.p3p_pfn_backward1(C.byref(grid), ctx.B, ctx.total, C.byref(ctx.params), state.data_ptr(), g.data_ptr(),
                                       ctx.out.data_ptr(), route.data_ptr(), ws.data_ptr(), ws.numel(), stream), "p3p_pfn_backward1")
        b1g = state[offs["back1g"]:offs["back1g"] + 2 * Cc]
        b1g.copy_(state[offs["back1"]:offs["back1"] + 2 * Cc])
        red(b1g, "back1")
        _lib.check(l.p3p_pfn_backward2(C.byref(grid), ctx.B, ctx.total, C.byref(ctx.params), state.data_ptr(), route.data_ptr(),
                                       ws.data_ptr(), ws.numel(), stream), "p3p_pfn_backward2")
        b0g = state[offs["back0g"]:offs["back0g"] + 64]
        b0g.copy_(state[offs["back0"]:offs["back0"] + 64])
        red(b0g, "back0")
        grads = [torch.empty_like(t) for t in ctx.keep]
        _lib.check(l.p3p_pfn_backward3(C.byref(ctx.params), state.data_ptr(), *[t.data_ptr() for t in grads], stream),
                   "p3p_pfn_backward3")
    return grads


class FusedPFNTrain(torch.autograd.Function):
    """out (B, ny nx, C) = scatter(PFN_train(voxelize(points))) with gradients to the six PFN parameters."""

    @staticmethod
    def forward(ctx, enc, values, offsets, B, w0, g0, b0, w1, g1, b1):
        out, c = train_forward(enc, values, offsets, B, (w0, g0, b0, w1, g1, b1))
        c.out = None  # (the output is saved through autograd: no reference cycle, in-place edits are detected)
        ctx.p3p = c
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        c = ctx.p3p  # (kept: with retain_graph=True the node may run again; every pass re-zeroes its accumulators)
        c.out = ctx.saved_tensors[0]
        grads = train_backward(c, grad_out)
        c.out = None
        return (None, None, None, None, *grads)
