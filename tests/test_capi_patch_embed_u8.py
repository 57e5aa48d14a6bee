"""CPU tests of p3p_patch_embed_u8 at the C-ABI boundary: the symbol is exported and bound, and every refusal comes back as
a negative code with a message naming the limit before anything is launched (fake device addresses: no CUDA call is made)."""
import ctypes as C

import pytest

FAKE = 1 << 20  # 16-byte aligned, never dereferenced: every call below fails on the host


def call(l, images=FAKE, lut=FAKE, B=1, in_chans=3, H=224, W=224, P=8, blob=FAKE, weight=FAKE, bias=FAKE, channels=384,
         precision=3, out=FAKE, out_dtype=0, out_layout=0, c_total=384, c_offset=0):
    return l.p3p_patch_embed_u8(images, lut, B, in_chans, H, W, P, blob, weight, bias, channels, precision, out, out_dtype,
                                out_layout, c_total, c_offset, None)


def test_u8_entry_is_exported(built_lib):
    from pixelspointspolygons_b200 import _lib

    assert "p3p_patch_embed_u8" in _lib.EXPORTED
    assert hasattr(C.CDLL(built_lib), "p3p_patch_embed_u8")
    assert _lib.lib().p3p_patch_embed_u8.restype is C.c_int
    assert len(_lib.lib().p3p_patch_embed_u8.argtypes) == 18


@pytest.mark.parametrize("kwargs, code, words", [
    (dict(images=None), -1, b"null images"),
    (dict(lut=None), -1, b"pixel_lut"),
    (dict(lut=None, B=0), -1, b"pixel_lut"),           # checked even for an empty batch
    (dict(in_chans=0), -2, b"1..4"),
    (dict(in_chans=5), -2, b"1..4"),
    (dict(H=220), -1, b"whole number of 8-px patches"),
    (dict(W=100, P=16), -1, b"whole number of 16-px patches"),
    (dict(images=FAKE + 4), -1, b"8-byte aligned"),
    (dict(images=FAKE + 1), -1, b"8-byte aligned"),
    (dict(blob=None, weight=None), -1, b"null weight and blob"),
    (dict(out=None), -1, b"null"),
    (dict(out=FAKE + 8), -1, b"misaligned"),
    # what p3p_patch_embed refuses, with its messages
    (dict(out_layout=7), -1, b"layout"),
    (dict(out_dtype=9), -1, b"dtype"),
    (dict(precision=4), -1, b"precision"),
    (dict(c_offset=1), -1, b"outside c_total"),
    (dict(channels=0), -1, b"positive"),
    (dict(B=-1), -1, b"num_tiles"),
])
def test_u8_argument_errors(built_lib, kwargs, code, words):
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    rc = call(l, **kwargs)
    assert rc == code, (rc, l.p3p_last_error())
    assert words in l.p3p_last_error(), l.p3p_last_error()


def test_u8_refusals_match_p3p_patch_embed(built_lib):
    """The checks shared with p3p_patch_embed give the same codes and messages."""
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    for kw in (dict(out_layout=7), dict(out_dtype=9), dict(precision=-1), dict(c_offset=5), dict(H=100)):
        a = dict(B=1, in_chans=3, H=224, W=224, P=8, channels=384, precision=3, out_dtype=0, out_layout=0, c_total=384, c_offset=0)
        a.update(kw)
        rc_u8 = call(l, **a)
        msg_u8 = l.p3p_last_error()
        rc = l.p3p_patch_embed(FAKE, a["B"], a["in_chans"], a["H"], a["W"], a["P"], FAKE, FAKE, a["channels"], a["precision"], FAKE,
                               a["out_dtype"], a["out_layout"], a["c_total"], a["c_offset"], None)
        assert rc == rc_u8 < 0 and l.p3p_last_error() == msg_u8, kw


def test_empty_batch_is_a_no_op(built_lib):
    from pixelspointspolygons_b200 import _lib

    assert call(_lib.lib(), B=0, images=None, out=None) == 0
