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


def test_recon_trunk_fused_upsample_is_bit_exact(cuda_dev):
    """The whole trunk (21 cross-scale blocks) at the c3 size with the upsample inside body.0 and with the resample kernel."""
    from cdfo_b200 import config, conv, hotpath
    from cdfo_b200.model import CVSR_V8
    m = CVSR_V8()
    m.load_state_dict(G.seeded_weights("O1"), strict=True)
    m = m.to(cuda_dev).eval()
    g = torch.Generator().manual_seed(7)
    x8 = conv.to_c8(torch.randn(1, 64, 272, 480, generator=g).to(cuda_dev))
    keep = config.trunk_fused_upsample
    try:
        config.trunk_fused_upsample = False
        ref = hotpath.recon_trunk(m.recon_trunk, x8)
        config.trunk_fused_upsample = True
        got = hotpath.recon_trunk(m.recon_trunk, x8)
    finally:
        config.trunk_fused_upsample = keep
    assert torch.equal(got, ref)
