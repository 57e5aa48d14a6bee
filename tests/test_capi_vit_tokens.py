"""CPU tests of p3p_conv3x3_vit_tokens at the C-ABI boundary: the symbol is exported and bound, and its argument errors come
back as negative codes with a message before anything is launched (fake, aligned device addresses: no CUDA call is made)."""
import ctypes as C

import pytest

FAKE = 1 << 20  # 16-byte aligned, never dereferenced: every call below fails on the host


def call(l, x=FAKE, B=1, H=28, W=28, Cin=768, blob=FAKE, Cout=384, precision=3, cls=FAKE, pos=FAKE, out=FAKE):
    return l.p3p_conv3x3_vit_tokens(x, B, H, W, Cin, blob, Cout, precision, cls, pos, out, None)


def test_vit_tokens_entry_is_exported(built_lib):
    from pixelspointspolygons_b200 import _lib

    assert "p3p_conv3x3_vit_tokens" in _lib.EXPORTED
    assert hasattr(C.CDLL(built_lib), "p3p_conv3x3_vit_tokens")
    assert _lib.lib().p3p_conv3x3_vit_tokens.restype is C.c_int


@pytest.mark.parametrize("kwargs, code, words", [
    (dict(cls=None), -1, b"cls_token"),
    (dict(pos=None), -1, b"pos_embed"),
    (dict(cls=None, B=0), -1, b"cls_token"),      # checked even for an empty batch
    (dict(x=None), -1, b"null"),
    (dict(out=None), -1, b"null"),
    (dict(out=FAKE + 4), -1, b"misaligned"),
    (dict(H=0), -1, b"bad sizes"),
    (dict(Cout=385), None, b"384"),
    (dict(Cin=96), None, b"multiple of 64"),
    (dict(precision=1), None, b"16-bit"),
])
def test_vit_tokens_argument_errors(built_lib, kwargs, code, words):
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    rc = call(l, **kwargs)
    assert rc < 0 and (code is None or rc == code), rc
    assert words in l.p3p_last_error(), l.p3p_last_error()


def test_vit_tokens_unsupported_shapes_match_p3p_conv3x3(built_lib):
    """The same error codes as p3p_conv3x3 for the same unsupported shapes."""
    from pixelspointspolygons_b200 import _lib

    l = _lib.lib()
    for Cin, Cout in ((96, 384), (768, 385)):
        rc_tokens = call(l, Cin=Cin, Cout=Cout)
        rc_conv = l.p3p_conv3x3(FAKE, 1, 28, 28, Cin, FAKE, Cout, 3, 1, FAKE, 1, Cout, 0, None)
        assert rc_tokens == rc_conv < 0


def test_empty_batch_is_a_no_op(built_lib):
    from pixelspointspolygons_b200 import _lib

    assert call(_lib.lib(), B=0) == 0
