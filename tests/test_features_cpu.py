"""Argument checks of the feature extraction on c8 bf16 (cdfo_b200/features.py, csrc/features_c8.cu): sizes the kernels cannot handle are
refused with a message naming the bound, before any CUDA call (this runs without a device)."""
import ctypes

import pytest
import torch

CDFO_ERR_SHAPE = -1


@pytest.mark.parametrize("H,W", [(10, 16), (16, 6), (2, 8), (0, 16)])
def test_side_branch_rejects_sizes_that_are_not_multiples_of_4(H, W):
    """The two stride-2 convolutions and their transposes bring back only multiples of 4 (10 -> 6 -> 4 -> 5 -> 8)."""
    from cdfo_b200 import _lib, features
    from cdfo_b200.model import _SideBranch
    s8 = torch.zeros(1, 8, H, W, 8, dtype=torch.bfloat16)
    with pytest.raises(_lib.CdfoError, match=r"multiples of 4, at least 4 \(got %d x %d\)" % (H, W)):
        features.side_branch_c8(_SideBranch(64, 16), s8, s8)


def _so(cdfo_so):
    lib = ctypes.CDLL(cdfo_so)
    lib.cdfo_last_error.restype = ctypes.c_char_p
    return lib


@pytest.mark.parametrize("Hi,Wi,Ho,Wo,transposed,msg", [
    (272, 480, 136, 241, 0, b"output must be (in + 4 - 3) / 2 + 1"),
    (272, 480, 137, 240, 0, b"output must be (in + 4 - 3) / 2 + 1"),
    (137, 241, 273, 480, 1, b"transposed output must be"),
    (137, 241, 272, 478, 1, b"transposed output must be"),
])
def test_conv16_c8_rejects_wrong_output_sizes(cdfo_so, Hi, Wi, Ho, Wo, transposed, msg):
    lib = _so(cdfo_so)
    buf = ctypes.create_string_buffer(64)
    assert lib.cdfo_conv16_c8_fwd(buf, buf, buf, buf, 1, Hi, Wi, Ho, Wo, 16, transposed, None) == CDFO_ERR_SHAPE
    assert msg in lib.cdfo_last_error()


def test_mdta_c8_entry_points_reject_missing_channels(cdfo_so):
    """The Gram reads q and k from chunks 0..15 (C >= 128); apply reads v from the 64 channels at v_channel0."""
    lib = _so(cdfo_so)
    buf = ctypes.create_string_buffer(64)
    assert lib.cdfo_mdta_gram_c8_fwd(buf, buf, 1, 120, 16, 16, 1, None) == CDFO_ERR_SHAPE
    assert b"cdfo_mdta_gram_c8_fwd: bad shape" in lib.cdfo_last_error()
    for C, v0 in ((192, 136), (64, 8), (128, 128)):
        assert lib.cdfo_mdta_apply_c8_fwd(buf, C, v0, buf, buf, None, buf, None, 1, 16, 16, None) == CDFO_ERR_SHAPE
        assert b"cdfo_mdta_apply_c8_fwd: bad shape" in lib.cdfo_last_error()


def test_dwconv3x3_c8_rejects_too_many_row_strips(cdfo_so):
    """Grid y = (C / 8) x ceil(H / 16) strips must stay <= 65535: 24 chunks x 2731 strips is 65544."""
    lib = _so(cdfo_so)
    buf = ctypes.create_string_buffer(64)
    assert lib.cdfo_dwconv3x3_c8_fwd(buf, buf, buf, 1, 192, 16 * 2731, 1, None) == CDFO_ERR_SHAPE
    assert b"too many row strips" in lib.cdfo_last_error()
