"""CPU tests of the training step's shape contract at the C-ABI boundary (C <= 512 channels, max_points <= 512): every
training entry refuses a shape outside it with a negative code and a message naming the limit, before it launches or
writes anything -- fake, aligned device addresses, never dereferenced: no CUDA call is made."""
import ctypes as C

import pytest

FAKE = 1 << 20  # 16-byte aligned, never dereferenced
P3P_ERR_INVALID_ARGUMENT, P3P_ERR_UNSUPPORTED = -1, -2


def grid(M):
    from pixelspointspolygons_b200 import _lib

    return _lib.make_grid((0, 0, 0), (224, 224, 100), (8, 8, 100), M, 784, 28, 28)


def params(channels):
    from pixelspointspolygons_b200 import _lib

    p = _lib.PfnParams()
    for name in ("linear0_weight", "norm0_weight", "norm0_bias", "linear1_weight", "norm1_weight", "norm1_bias"):
        setattr(p, name, FAKE)
    p.eps, p.channels, p.center_alias = 1e-3, channels, 1
    return p


def grid_entries(l, channels, M, ws):
    """-> {entry: return code} of the five entries that take the grid (workspace `ws`, or None)."""
    g, p, n = C.byref(grid(M)), C.byref(params(channels)), (1 << 40) if ws else 0
    return {
        "p3p_pfn_train_stats0": l.p3p_pfn_train_stats0(g, 2, 1000, p, FAKE, ws, n, None),
        "p3p_pfn_train_stats1": l.p3p_pfn_train_stats1(g, 2, 1000, p, FAKE, ws, n, None),
        "p3p_pfn_train_forward": l.p3p_pfn_train_forward(g, 2, 1000, p, FAKE, FAKE, FAKE, ws, n, None),
        "p3p_pfn_backward1": l.p3p_pfn_backward1(g, 2, 1000, p, FAKE, FAKE, FAKE, FAKE, ws, n, None),
        "p3p_pfn_backward2": l.p3p_pfn_backward2(g, 2, 1000, p, FAKE, FAKE, ws, n, None),
    }


def params_entries(l, channels):
    """-> {entry: return code} of the entries that see only the parameters (called here for refused channel counts only:
    with a valid one they would launch)."""
    p = C.byref(params(channels))
    return {
        "p3p_pfn_train_stats2": l.p3p_pfn_train_stats2(p, FAKE, FAKE, FAKE, FAKE, FAKE, None),
        "p3p_pfn_backward3": l.p3p_pfn_backward3(p, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None),
    }


@pytest.mark.parametrize("channels, M, words", [
    (513, 64, b"1..512 channels, got 513"),
    (1024, 64, b"1..512 channels, got 1024"),
    (0, 64, b"1..512 channels, got 0"),
    (384, 1024, b"max_points <= 512, got 1024"),
    (513, 1024, b"1..512 channels, got 513"),  # the channel count is checked first
])
def test_training_entries_refuse_shapes_outside_the_contract(built_lib, channels, M, words):
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    codes = grid_entries(l, channels, M, FAKE)
    if not 1 <= channels <= 512:
        codes.update(params_entries(l, channels))
        assert l.p3p_pfn_train_state_doubles(channels, None) == 0
    assert len(codes) in (5, 7)
    for name, rc in codes.items():
        assert rc == P3P_ERR_UNSUPPORTED, (name, rc)
        assert words in l.p3p_last_error(), (name, l.p3p_last_error())


@pytest.mark.parametrize("channels, M", [(512, 512), (512, 488), (512, 64), (200, 100), (1, 1), (384, 512)])
def test_shapes_inside_the_contract_pass_the_shape_checks(built_lib, channels, M):
    """Every (C, M) of the contract fits the shared memory of every kernel of the step (the dW1 block of backward pass 1 is
    the largest: 229 776 bytes at C = M = 512, within sm_100's 227 KB).  Without a workspace each entry gets past the shape
    checks and stops at its null-pointer check, still before any CUDA call."""
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    for name, rc in grid_entries(l, channels, M, None).items():
        assert rc == P3P_ERR_INVALID_ARGUMENT, (name, rc, l.p3p_last_error())
        assert b"null" in l.p3p_last_error(), (name, l.p3p_last_error())
    assert l.p3p_pfn_train_state_doubles(channels, None) > 0
