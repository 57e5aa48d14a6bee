"""CPU tests of the conv3x3 shape contract at the C-ABI boundary: p3p_conv3x3 and p3p_conv3x3_vit_tokens refuse what the
strip planner cannot tile (widths above 256, no strip of whole rows that is a multiple of 16 positions, accumulators beyond
the 512 TMEM columns) and non-16-bit operands with P3P_ERR_UNSUPPORTED and a message naming the limit, before any CUDA
call (fake, aligned device addresses, never dereferenced)."""
import pytest

FAKE = 1 << 20  # 16-byte aligned, never dereferenced
P3P_ERR_UNSUPPORTED = -2


def conv(l, B, H, W, Cin, Cout, precision):
    return l.p3p_conv3x3(FAKE, B, H, W, Cin, FAKE, Cout, precision, 1, FAKE, 1, Cout, 0, None)


def vit_tokens(l, B, H, W, Cin, Cout, precision):
    return l.p3p_conv3x3_vit_tokens(FAKE, B, H, W, Cin, FAKE, Cout, precision, FAKE, FAKE, FAKE, None)


@pytest.mark.parametrize("entry", [conv, vit_tokens], ids=["p3p_conv3x3", "p3p_conv3x3_vit_tokens"])
@pytest.mark.parametrize("H, W, Cout, precision, words", [
    (4, 257, 64, 3, b"widths up to 256"),
    (8, 200, 64, 3, b"no strip of whole rows of width 200"),   # 200 % 16 = 8 and 2 rows are over 256 positions
    (2, 20, 64, 2, b"no strip of whole rows of width 20"),     # 20 and 40 positions: neither a multiple of 16
    (28, 224, 384, 3, b"within TMEM (3 channel tiles)"),       # 3 x 256 accumulator columns > 512
    (28, 28, 384, 1, b"16-bit"),                               # tf32
])
def test_unsupported_shapes_are_refused(built_lib, entry, H, W, Cout, precision, words):
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    rc = entry(l, 2, H, W, 64, Cout, precision)
    assert rc == P3P_ERR_UNSUPPORTED, (rc, l.p3p_last_error())
    assert words in l.p3p_last_error(), l.p3p_last_error()
