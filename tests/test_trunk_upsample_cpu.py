"""The index arithmetic of the UP2 A-operand builder (csrc/conv3x3_pair_sm100.cu) restated in numpy: a tile's 18 x 10 halo of
bilinear_x2(x), rebuilt from the edge-clamped 10 x 6 source window, equals F.interpolate's values with zero padding outside the 2x frame.
Inputs are multiples of 16 below 2^12, so every blend is exact and the comparison is exact too.  Argument checks of the C entry point
and of hotpath.cross_scale_block."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

TILE_H, TILE_W = 16, 8


def build_halo(x, h0, w0):
    """x [Hi, Wi] float32 -> the A stage of the 2x tile at (h0, w0): [18, 10], as the builder warps compute it."""
    Hi, Wi = x.shape
    rr = np.clip(h0 // 2 - 1 + np.arange(TILE_H // 2 + 2), 0, Hi - 1)
    cc = np.clip(w0 // 2 - 1 + np.arange(TILE_W // 2 + 2), 0, Wi - 1)
    raw = x[np.ix_(rr, cc)]
    out = np.zeros((TILE_H + 2, TILE_W + 2), np.float32)

    def blend(nb, x):
        return np.float32(0.25) * nb + np.float32(0.75) * x

    for j in range(TILE_W + 2):                          # one (chunk, halo column) per lane, walked down the raw rows
        C = w0 - 1 + j
        if not 0 <= C < 2 * Wi:
            continue
        c0 = (C >> 1) - (w0 >> 1) + 1
        cn = c0 + (1 if C & 1 else -1)
        prev = blend(raw[0, cn], raw[0, c0])
        for rr in range(1, TILE_H // 2 + 2):
            cur = blend(raw[rr, cn], raw[rr, c0])
            R = h0 + 2 * rr - 3
            if 0 <= R < 2 * Hi:
                out[2 * rr - 2, j] = blend(cur, prev)
            if R + 1 < 2 * Hi:
                out[2 * rr - 1, j] = blend(prev, cur)
            prev = cur
    return out


@pytest.mark.parametrize("Hi,Wi", [(2, 2), (3, 5), (13, 21), (17, 9), (8, 12)])
def test_builder_halo_matches_interpolate(Hi, Wi):
    rng = np.random.default_rng(Hi * 100 + Wi)
    x = (rng.integers(-256, 256, size=(Hi, Wi)) * 16).astype(np.float32)
    up = F.interpolate(torch.from_numpy(x)[None, None], scale_factor=2.0, mode="bilinear", align_corners=False)[0, 0].numpy()
    padded = np.zeros((2 * Hi + TILE_H + 2, 2 * Wi + TILE_W + 2), np.float32)      # zero padding of the 3x3 convolution
    padded[1:2 * Hi + 1, 1:2 * Wi + 1] = up
    for h0 in range(0, 2 * Hi, TILE_H):
        for w0 in range(0, 2 * Wi, TILE_W):
            ref = padded[h0:h0 + TILE_H + 2, w0:w0 + TILE_W + 2]
            assert np.array_equal(build_halo(x, h0, w0), ref), (h0, w0)


def test_up2_entry_point_rejects_bad_arguments(cdfo_so):
    lib = ctypes.CDLL(cdfo_so)
    lib.cdfo_last_error.restype = ctypes.c_char_p
    buf = ctypes.create_string_buffer(64)
    fn = lib.cdfo_conv3x3_pair_sm100_up2_fwd
    assert fn(None, buf, None, None, buf, 1, 64, 256, 16, 16, 2, 0, None) != 0
    assert b"NULL" in lib.cdfo_last_error()
    assert fn(buf, buf, None, None, buf, 1, 256, 64, 16, 16, 2, 0, None) != 0
    assert b"64 -> 256 only" in lib.cdfo_last_error()
    assert fn(buf, buf, None, None, buf, 1, 64, 256, 15, 16, 2, 0, None) != 0
    assert b"even" in lib.cdfo_last_error()
    assert fn(buf, buf, None, None, buf, 1, 64, 256, 16, 16, 2, 2, None) != 0
    assert b"y_planes" in lib.cdfo_last_error()


@pytest.mark.parametrize("H,W", [(15, 16), (16, 9), (2, 16), (16, 2), (3, 3)])
def test_cross_scale_block_rejects_odd_or_small_frames(H, W):
    """The block's kernels need even sides (x0.5, parity planes) and a half-size image of at least 2 x 2 (border-class bias): other sizes
    are refused with a message naming the bound, before any CUDA call (this runs without a device)."""
    from cdfo_b200 import _lib, hotpath
    from cdfo_b200.model import _CrossScaleBlock
    x8 = torch.zeros(1, 8, H, W, 8, dtype=torch.bfloat16)
    with pytest.raises(_lib.CdfoError, match=r"even and >= 4 \(got %d x %d\)" % (H, W)):
        hotpath.cross_scale_block(_CrossScaleBlock(), x8, want_half=True)
