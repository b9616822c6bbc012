"""conv3x3_up2 (body.0 of Block_'s down(body(up(x))) branch with the bilinear x2 evaluated while the A operand is built) against the
two-kernel form conv3x3(resample(x, 1)): equal bit for bit, kernel by kernel and over the whole reconstruction trunk."""
import pytest
import torch

import golden_util as G

pytestmark = pytest.mark.gpu

# (B, H, W) of the 1x input: the c3 trunk (272 x 480) and half of it; 2H % 16 != 0 and 2W % 8 != 0 (ragged tiles); an odd number of
# tiles (16 x 24 -> 3, 48 x 40 -> 15); 2 x 2 and 3 x 5 images in which every pixel is a border pixel
SHAPES = [(1, 272, 480), (4, 136, 240), (2, 13, 21), (4, 17, 9), (1, 8, 12), (1, 24, 20), (4, 2, 2), (1, 3, 5)]


@pytest.mark.parametrize("B,H,W", SHAPES)
def test_conv3x3_up2_equals_resample_then_conv(cuda_dev, B, H, W):
    from cdfo_b200 import conv
    g = torch.Generator().manual_seed(B * 1000 + H * 7 + W)
    x8 = conv.to_c8(torch.randn(B, 64, H, W, generator=g).to(cuda_dev))
    w = (torch.randn(256, 64, 3, 3, generator=g) * 0.05).to(cuda_dev)
    b = torch.randn(256, generator=g).to(cuda_dev)
    edge = torch.randn(9, 256, generator=g).to(cuda_dev)
    xu = conv.resample(x8, 1)
    for planes in (False, True):
        for be in (None, edge):
            ref = conv.conv3x3(xu, w, b, conv.ACT_LRELU, parity_planes=planes, bias_edge=be)
            got = conv.conv3x3_up2(x8, w, b, conv.ACT_LRELU, parity_planes=planes, bias_edge=be)
            assert got.shape == ref.shape
            assert torch.equal(got, ref), "planes=%s bias_edge=%s: %d of %d values differ" % (
                planes, be is not None, int((got != ref).sum()), ref.numel())
    ref = conv.conv3x3(xu, w, None, conv.ACT_NONE)
    assert torch.equal(conv.conv3x3_up2(x8, w, None, conv.ACT_NONE), ref)


def _block_with_resample(blk, x8, x8_half, want_half):
    """hotpath.cross_scale_block with body.0 at 2x reading the output of the x2 resample kernel instead of building it in its producer."""
    from cdfo_b200 import conv, hotpath
    b0, b2 = blk.body._modules["0"], blk.body._modules["2"]
    wts = hotpath._block_weights(blk)
    wd0, bd0, ed0 = wts["body0_dn"]
    wu0, bu0, eu0 = wts["body0_up"]
    y = conv.conv3x3(conv.conv3x3(x8, b0.weight, b0.bias, conv.ACT_LRELU), b2.weight, b2.bias, conv.ACT_NONE, resid8=x8)
    xh = x8_half if x8_half is not None else conv.resample(x8, 0)
    cu = conv.conv3x3(conv.conv3x3(xh, wd0, bd0, conv.ACT_LRELU, bias_edge=ed0), wts["up_body2"][0], wts["up_body2"][1], conv.ACT_NONE)
    t2 = conv.conv3x3(conv.resample(x8, 1), wu0, bu0, conv.ACT_LRELU, parity_planes=True, bias_edge=eu0)
    return conv.conv3x3_then_half(t2, wts["dn_body2"][0], wts["dn_body2"][1], resid8=y, up8=cu, want_half=want_half)


def test_recon_trunk_upsample_in_body0_is_bit_exact(cuda_dev):
    """The whole trunk (21 cross-scale blocks) at the c3 size with the upsample inside body.0 and with the resample kernel."""
    from cdfo_b200 import conv, hotpath
    from cdfo_b200.model import CVSR_V8
    m = CVSR_V8()
    m.load_state_dict(G.seeded_weights("O1"), strict=True)
    m = m.to(cuda_dev).eval()
    g = torch.Generator().manual_seed(7)
    x8 = conv.to_c8(torch.randn(1, 64, 272, 480, generator=g).to(cuda_dev))
    with torch.no_grad():
        ref = x8
        for grp in m.recon_trunk.body._modules.values():               # hotpath.recon_trunk's loop
            r, r_half = ref, None
            blocks = list(grp.body._modules.values())
            for k, blk in enumerate(blocks):
                if k + 1 < len(blocks):
                    r, r_half = _block_with_resample(blk, r, r_half, want_half=True)
                else:
                    r = _block_with_resample(blk, r, r_half, want_half=False)
            ref = conv.conv3x3(r, grp.conv.weight, grp.conv.bias, conv.ACT_NONE, resid8=ref)
        ref = ref + x8
    got = hotpath.recon_trunk(m.recon_trunk, x8)
    assert torch.equal(got, ref)
