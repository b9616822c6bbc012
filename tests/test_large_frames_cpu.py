"""Frame-size bounds of the long-range attention entry point (csrc/lra.cu): the row pass takes W <= 1280 (one CTA up to 704 columns,
a 2-CTA cluster above), the bf16 column pass H <= 768.  Shapes past them are refused with CDFO_ERR_UNSUPPORTED and a message naming
the bound, before any CUDA call (this runs without a device) -- so a refused call never writes into the caller's workspace."""
import ctypes

import pytest

CDFO_ERR_UNSUPPORTED = -4


def _lra(lib, B, H, W):
    buf = ctypes.create_string_buffer(64)
    f = ctypes.c_float(0.0)
    return lib.cdfo_lra_fwd(buf, buf, buf, buf, None, buf, f, f, buf, buf, buf, buf, B, H, W, None)


@pytest.mark.parametrize("H,W,bound", [(8, 1288, b"W <= 1280"), (400, 1344, b"W <= 1280"), (776, 64, b"H <= 768"),
                                       (1088, 960, b"H <= 768"), (776, 1288, b"W <= 1280")])
def test_lra_rejects_frames_past_the_bounds(cdfo_so, H, W, bound):
    lib = ctypes.CDLL(cdfo_so)
    lib.cdfo_last_error.restype = ctypes.c_char_p
    assert _lra(lib, 1, H, W) == CDFO_ERR_UNSUPPORTED
    assert bound in lib.cdfo_last_error()


def test_lra_c8_entry_point_applies_the_same_bounds(cdfo_so):
    lib = ctypes.CDLL(cdfo_so)
    lib.cdfo_last_error.restype = ctypes.c_char_p
    buf = ctypes.create_string_buffer(64)
    f = ctypes.c_float(0.0)
    rc = lib.cdfo_lra_c8_fwd(buf, buf, buf, buf, None, buf, f, f, buf, buf, buf, 128, 0, buf, 1, 776, 64, None)
    assert rc == CDFO_ERR_UNSUPPORTED and b"H <= 768" in lib.cdfo_last_error()


def test_lra_shape_checks_still_come_first(cdfo_so):
    """Sizes that are not multiples of the 8x8 window stay a shape error, whatever their width."""
    lib = ctypes.CDLL(cdfo_so)
    lib.cdfo_last_error.restype = ctypes.c_char_p
    assert _lra(lib, 1, 12, 1288) == -1
    assert b"multiples of the window size 8" in lib.cdfo_last_error()
