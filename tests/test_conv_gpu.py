"""tcgen05 3x3 convolution (TMA halo, implicit GEMM) against torch conv2d in fp32 on bf16-rounded operands."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

CASES = [
    # B, Cin, Cout, H, W, act, resid
    (1, 64, 64, 16, 8, 0, False),       # exactly one tile
    (2, 64, 64, 33, 21, 1, True),       # ragged tiles, ReLU, residual
    (1, 64, 432, 24, 40, 0, False),     # conv_offset.2: three N tiles of 144
    (1, 128, 64, 24, 40, 2, False),     # conv_expand_fea_r: two 64-channel K blocks
    (1, 64, 256, 20, 24, 2, False),     # trunk body.0: two N tiles of 128
    (1, 256, 64, 20, 24, 0, True),      # trunk body.2: four K blocks, weights streamed with the A stages (N tile 64)
    (2, 448, 64, 40, 24, 2, False),     # tsa_fusion-shaped K (7 blocks), streamed weights, several tiles per CTA
    (1, 256, 32, 20, 24, 0, False),     # wide input, resident N tile of 32
    (1, 64, 48, 18, 10, 0, False),      # N tile of 16
    (3, 64, 64, 64, 64, 0, False),      # many tiles per CTA (pipeline wrap-around)
]


@pytest.mark.parametrize("case", CASES)
def test_conv3x3_sm100(cuda_dev, case):
    from cdfo_b200 import conv
    B, Cin, Cout, H, W, act, use_res = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, Cin, H, W, generator=g).to(torch.bfloat16).float()
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g) * 0.1
    r = torch.randn(B, Cout, H, W, generator=g).to(torch.bfloat16).float() if use_res else None
    ref = F.conv2d(x, w, b, 1, 1)
    ref = F.relu(ref) if act == 1 else (F.leaky_relu(ref, 0.1) if act == 2 else ref)
    if use_res:
        ref = ref + r
    d = lambda t: None if t is None else t.to(cuda_dev)
    x8 = conv.to_c8(d(x))
    r8 = conv.to_c8(d(r)) if use_res else None
    wd = d(w)
    y = conv.conv3x3(x8, wd, d(b), act, r8, out_nchw=True)
    err = (y.cpu() - ref).abs().max().item()
    print("conv3x3 %s: max err %.3g (max|ref| %.3g)" % (case, err, ref.abs().max().item()))
    assert err <= 2e-3 * max(1.0, ref.abs().max().item())
    y8 = conv.conv3x3(x8, wd, d(b), act, r8, out_nchw=False)
    assert (conv.from_c8(y8).cpu() - ref).abs().max().item() <= 1.2e-2 * max(1.0, ref.abs().max().item())  # bf16 output rounding


PAIR_CASES = [
    # B, Cin, Cout, H, W, act, resid
    (1, 256, 64, 16, 8, 0, False),      # one tile: the pair's second CTA recomputes tile 0 and stores nothing
    (1, 256, 64, 16, 16, 2, True),      # exactly one tile per CTA of one pair
    (2, 256, 64, 33, 21, 1, True),      # ragged tiles, odd tile count
    (1, 128, 64, 24, 40, 0, False),     # two K blocks (conv_expand_fea_r's shape)
    (1, 192, 64, 20, 24, 2, False),     # three K blocks = the stage count
    (3, 256, 64, 136, 240, 0, True),    # the trunk's half-resolution call: ~10 tiles per CTA (ring and accumulator wrap-around)
    (1, 64, 256, 16, 8, 2, False),      # N = 256: each CTA holds 128 output channels, the accumulators fill all 512 TMEM columns
    (2, 64, 256, 40, 56, 2, False),     # trunk body.0 shape, several tiles per CTA
    (3, 64, 256, 136, 240, 0, False),
    (2, 64, 64, 33, 21, 1, True),       # 64 -> 64 layers (one K block per tile)
    (6, 64, 64, 64, 64, 2, True),
]


@pytest.mark.parametrize("case", PAIR_CASES)
def test_conv3x3_pair_sm100(cuda_dev, case):
    """Two-SM kernel (tcgen05.mma cta_group::2, weights resident in a CTA pair) against torch conv2d, and against the single-SM
    kernel (same bf16 operands, fp32 accumulation in a different order)."""
    import cdfo_b200
    from cdfo_b200 import conv
    B, Cin, Cout, H, W, act, use_res = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, Cin, H, W, generator=g).to(torch.bfloat16).float()
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(torch.bfloat16).float()
    w[Cout // 2 + 8:] *= 3.0                        # the two halves of the output channels live in different CTAs: make them differ
    b = torch.randn(Cout, generator=g) * 0.1
    r = torch.randn(B, Cout, H, W, generator=g).to(torch.bfloat16).float() if use_res else None
    d = lambda t: None if t is None else t.to(cuda_dev)
    xd, wd, bd = d(x), d(w), d(b)
    ref = F.conv2d(xd, wd, bd, 1, 1)
    ref = F.relu(ref) if act == 1 else (F.leaky_relu(ref, 0.1) if act == 2 else ref)
    if use_res:
        ref = ref + d(r)
    x8 = conv.to_c8(xd)
    r8 = conv.to_c8(d(r)) if use_res else None
    assert cdfo_b200._lib.lib().cdfo_conv3x3_pair_sm100_supported(Cout, Cin) == 1
    try:
        cdfo_b200.config.conv_pair = True
        y_pair = conv.from_c8(conv.conv3x3(x8, wd, bd, act, r8))
        y_again = conv.from_c8(conv.conv3x3(x8, wd, bd, act, r8))
        cdfo_b200.config.conv_pair = False
        y_single = conv.from_c8(conv.conv3x3(x8, wd, bd, act, r8))
    finally:
        cdfo_b200.config.conv_pair = True
    scale = max(1.0, ref.abs().max().item())
    err = (y_pair - ref).abs().max().item()
    print("conv3x3 pair %s: max err %.3g vs torch, %.3g vs single-SM (max|ref| %.3g)" % (case, err, (y_pair - y_single).abs().max().item(), scale))
    assert torch.equal(y_pair, y_again)
    assert err <= 1.2e-2 * scale                    # bf16 output rounding
    assert (y_pair - y_single).abs().max().item() <= 8e-3 * scale


@pytest.mark.parametrize("case", [(1, 256, 32, 16, False), (2, 256, 66, 42, True), (1, 64, 34, 18, True), (3, 256, 136, 240, True),
                                  (1, 256, 544, 960, False)])
def test_conv3x3_then_half_as_4x4_stride2(cuda_dev, case):
    """bilinear x0.5 (align_corners=False: 2x2 mean) of a 3x3 convolution as one 4x4 / stride-2 convolution on a CTA pair, against
    the torch composition F.interpolate(F.conv2d(...), scale_factor=0.5) on bf16-rounded operands (arch:324-333, :401-406)."""
    from cdfo_b200 import conv
    B, Cin, Hi, Wi, use_res = case
    g = torch.Generator().manual_seed(sum(case))
    d = lambda t: None if t is None else t.to(cuda_dev)
    x = d(torch.randn(B, Cin, Hi, Wi, generator=g).to(torch.bfloat16).float())
    w = d((torch.randn(64, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(torch.bfloat16).float())
    w[40:] *= 3.0
    b = d(torch.randn(64, generator=g) * 0.1)
    r = d(torch.randn(B, 64, Hi // 2, Wi // 2, generator=g).to(torch.bfloat16).float()) if use_res else None
    ref = F.interpolate(F.conv2d(x, w, b, 1, 1), scale_factor=0.5, mode="bilinear", align_corners=False)
    if use_res:
        ref = ref + r
    x8 = conv.to_c8(x)
    y = conv.from_c8(conv.conv3x3_then_half(x8, w, b, conv.to_c8(r) if use_res else None))
    y2 = conv.from_c8(conv.conv3x3_then_half(x8, w, b, conv.to_c8(r) if use_res else None))
    scale = max(1.0, ref.abs().max().item())
    err = (y - ref).abs().max().item()
    print("conv4x4s2 %s: max err %.3g (max|ref| %.3g)" % (case, err, scale))
    assert torch.equal(y, y2)
    assert err <= 1.2e-2 * scale          # bf16 rounding of the output and of the folded weights (sums of up to four bf16 values / 4)
    # the same input stored as its four parity planes (dense TMA boxes instead of stride-2 loads): bit-identical result
    xp = x8.view(B, Cin // 8, Hi // 2, 2, Wi // 2, 2, 8).permute(0, 1, 3, 5, 2, 4, 6).contiguous()
    y3 = conv.from_c8(conv.conv3x3_then_half(xp, w, b, conv.to_c8(r) if use_res else None))
    assert torch.equal(y, y3)


@pytest.mark.parametrize("case", [(1, 256, 32, 16, True), (2, 256, 72, 44, True), (1, 64, 40, 24, False), (2, 256, 544, 960, True)])
def test_conv4x4s2_block_epilogue_vs_torch_and_half_kernel(cuda_dev, case):
    """The folded convolution closing a cross-scale block in its epilogue (cdfo_conv4x4s2_pair_sm100_block_fwd): + bilinear x2 of the
    half-resolution branch and the x0.5 of the sum, against torch on the same bf16 operands (Block_.forward, arch:401-406; ragged tiles
    included), and the x0.5 against the resampling kernel applied to the bf16 sum (which rounds once more)."""
    from cdfo_b200 import conv
    B, Cin, Hi, Wi, use_res = case
    g = torch.Generator().manual_seed(sum(case[:4]) + 1)
    d = lambda t: t.to(cuda_dev)
    x = d(torch.randn(B, Cin, Hi, Wi, generator=g).to(torch.bfloat16).float())
    w = d((torch.randn(64, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(torch.bfloat16).float())
    b = d(torch.randn(64, generator=g) * 0.1)
    r = d(torch.randn(B, 64, Hi // 2, Wi // 2, generator=g).to(torch.bfloat16).float()) if use_res else None
    low = d(torch.randn(B, 64, Hi // 4, Wi // 4, generator=g).to(torch.bfloat16).float())
    ref = F.interpolate(F.conv2d(x, w, b, 1, 1), scale_factor=0.5, mode="bilinear", align_corners=False) + \
        F.interpolate(low, scale_factor=2.0, mode="bilinear", align_corners=False)
    if use_res:
        ref = ref + r
    ref_half = F.interpolate(ref, scale_factor=0.5, mode="bilinear", align_corners=False)
    x8, r8, low8 = conv.to_c8(x), (conv.to_c8(r) if use_res else None), conv.to_c8(low)
    y8, h8 = conv.conv3x3_then_half(x8, w, b, r8, up8=low8, want_half=True)
    y, h = conv.from_c8(y8), conv.from_c8(h8)
    scale = max(1.0, ref.abs().max().item())
    err, err_h = (y - ref).abs().max().item(), (h - ref_half).abs().max().item()
    print("conv4x4s2 block epilogue %s: max err %.3g, half %.3g (max|ref| %.3g)" % (case, err, err_h, scale))
    assert err <= 1.2e-2 * scale and err_h <= 1.2e-2 * scale
    # the x0.5 of the epilogue (from the fp32 sum) against the resampling kernel on the bf16 sum
    assert (h - conv.from_c8(conv.resample(y8, 0))).abs().max().item() <= 2 ** -7 * scale
    # only one of the two options, and reruns are bit-identical
    assert torch.equal(conv.conv3x3_then_half(x8, w, b, r8, up8=low8), y8)
    y_b, h_b = conv.conv3x3_then_half(x8, w, b, r8, want_half=True)
    assert torch.equal(y_b, conv.conv3x3_then_half(x8, w, b, r8))
    assert (conv.from_c8(h_b) - conv.from_c8(conv.resample(y_b, 0))).abs().max().item() <= 2 ** -7 * scale


@pytest.mark.parametrize("B,H,W,planes", [(1, 16, 8, False), (2, 34, 50, False), (1, 40, 24, True), (2, 2, 2, False)])
def test_conv3x3_with_composed_1x1_and_border_bias(cuda_dev, B, H, W, planes):
    """A 1x1 convolution composed into the following zero-padded 3x3 one (hotpath._compose_3x3_after_1x1: Block_'s down / up 1x1 + body.0,
    arch:388-406): composed weights + the border-class bias table of cdfo_conv3x3_pair_sm100_edge_fwd against the torch chain
    conv2d(conv2d(x, w1, b1), w3, b3, padding=1), borders and corners included."""
    from cdfo_b200 import conv, hotpath
    g = torch.Generator().manual_seed(B * 100 + H)
    d = lambda t: t.to(cuda_dev)
    x = d(torch.randn(B, 64, H, W, generator=g).to(torch.bfloat16).float())
    w1 = d(torch.randn(64, 64, 1, 1, generator=g) / 8)
    b1 = d(torch.randn(64, generator=g))                       # a large 1x1 bias: the border classes differ visibly
    w3 = d(torch.randn(256, 64, 3, 3, generator=g) / 24)
    b3 = d(torch.randn(256, generator=g) * 0.1)
    ref = F.leaky_relu(F.conv2d(F.conv2d(x, w1, b1), w3, b3, padding=1), 0.1)
    w, b, be = hotpath._compose_3x3_after_1x1(w3, b3, w1, b1)
    assert (be[0] - be[4]).abs().max().item() > 0.1
    y = conv.conv3x3(conv.to_c8(x), w, b, conv.ACT_LRELU, parity_planes=planes, bias_edge=be)
    if planes:
        y = y.permute(0, 1, 4, 2, 5, 3, 6).reshape(B, 32, H, W, 8).contiguous()
    y = conv.from_c8(y)
    scale = max(1.0, ref.abs().max().item())
    err = (y - ref).abs().max().item()
    border = torch.ones_like(ref, dtype=torch.bool)
    border[:, :, 1:-1, 1:-1] = False
    print("composed 1x1 o 3x3 %dx%dx%d: max err %.3g (border %.3g), max|ref| %.3g" % (B, H, W, err, (y - ref)[border].abs().max().item(), scale))
    assert err <= 1.2e-2 * scale          # bf16 rounding of the composed weights and of the output
    # without the table the border pixels are wrong by the 1x1 bias seen through the missing taps
    y0 = conv.from_c8(conv.conv3x3(conv.to_c8(x), w, b, conv.ACT_LRELU))
    assert (y0 - ref)[border].abs().max().item() > 5 * err


@pytest.mark.parametrize("B,Cin,Cout,H,W", [(1, 64, 256, 32, 16), (2, 64, 256, 66, 42), (1, 256, 64, 34, 18), (1, 64, 256, 544, 960)])
def test_conv3x3_pair_parity_plane_output(cuda_dev, B, Cin, Cout, H, W):
    """The CTA-pair convolution writing its output as four parity planes [B, C/8, 2, 2, H/2, W/2, 8] (the layout the folded
    4x4 / stride-2 convolution reads) = a permutation of its plain c8 output, bit for bit."""
    from cdfo_b200 import conv
    g = torch.Generator().manual_seed(B + Cin + H)
    x8 = conv.to_c8(torch.randn(B, Cin, H, W, generator=g).to(cuda_dev))
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(cuda_dev)
    b = (torch.randn(Cout, generator=g) * 0.1).to(cuda_dev)
    y = conv.conv3x3(x8, w, b, conv.ACT_LRELU)
    yp = conv.conv3x3(x8, w, b, conv.ACT_LRELU, parity_planes=True)
    assert tuple(yp.shape) == (B, Cout // 8, 2, 2, H // 2, W // 2, 8)
    assert torch.equal(yp, y.view(B, Cout // 8, H // 2, 2, W // 2, 2, 8).permute(0, 1, 3, 5, 2, 4, 6).contiguous())


def test_pixel_shuffle_epilogue_and_conv_last_skip(cuda_dev):
    """upconv (1x1 as a centre-tap 3x3) + PixelShuffle(2) + lrelu in the conv epilogue, and conv_last + bilinear x4 skip,
    against the plain torch composition of arch/SIDECVSR_our.py:4473-4480 on bf16-rounded operands."""
    import torch.nn.functional as F
    from cdfo_b200 import conv
    g = torch.Generator().manual_seed(11)
    B, H, W = 2, 24, 40
    t = torch.randn(B, 64, H, W, generator=g).to(torch.bfloat16).float()
    w1 = (torch.randn(256, 64, 1, 1, generator=g) * 0.1).to(torch.bfloat16).float()
    b1 = torch.randn(256, generator=g) * 0.1
    ref = F.leaky_relu(F.pixel_shuffle(F.conv2d(t, w1, b1), 2), 0.1)
    d = lambda v: v.to(cuda_dev)
    w3 = conv.ps_order(d(w1))                                        # 1x1 weight, PixelShuffle row order
    y8 = conv.conv3x3(conv.to_c8(d(t)), w3, conv.ps_order(d(b1)), conv.ACT_LRELU, pixel_shuffle=True)
    assert tuple(y8.shape) == (B, 8, 2 * H, 2 * W, 8)
    got = conv.from_c8(y8).cpu()
    assert (got - ref).abs().max().item() <= 1e-2 * ref.abs().max().item()
    # conv_last + skip on the 2x grid (any H, W multiple of 4 works): 64 -> 1, 3x3
    wl = (torch.randn(1, 64, 3, 3, generator=g) * 0.05).to(torch.bfloat16).float()
    bl = torch.randn(1, generator=g)
    lr = torch.rand(B, 1, 2 * H // 4, 2 * W // 4, generator=g)
    x2 = conv.from_c8(y8).cpu()       # bf16-exact input
    ref2 = F.conv2d(x2, wl, bl, padding=1) + F.interpolate(lr, scale_factor=4.0, mode="bilinear", align_corners=False)
    wl_d, bl_d = d(wl), d(bl)
    got2 = conv.conv_last_skip(y8, wl_d, bl_d, d(lr)).cpu()
    err = (got2 - ref2).abs().max().item()
    print("conv_last+skip max err %.3g" % err)
    assert err <= 2e-3


@pytest.mark.parametrize("B,Cin,Cout,H,W", [(2, 64, 64, 33, 21), (1, 448, 64, 40, 24), (1, 64, 256, 20, 24), (1, 128, 48, 18, 10)])
def test_conv1x1_sm100(cuda_dev, B, Cin, Cout, H, W):
    """Kernel size 1 on the tcgen05 convolution kernel (tsa_fusion, upconv, the trunk's down / up convs)."""
    import torch.nn.functional as F
    from cdfo_b200 import conv
    g = torch.Generator().manual_seed(B + Cin + Cout)
    x = torch.randn(B, Cin, H, W, generator=g).to(torch.bfloat16).float()
    w = (torch.randn(Cout, Cin, 1, 1, generator=g) / Cin ** 0.5).to(torch.bfloat16).float()
    b = torch.randn(Cout, generator=g)
    ref = F.leaky_relu(F.conv2d(x, w, b), 0.1)
    d = lambda v: v.to(cuda_dev)
    y = conv.conv3x3(conv.to_c8(d(x)), d(w), d(b), conv.ACT_LRELU, out_nchw=True).cpu()
    err = (y - ref).abs().max().item()
    print("conv1x1 %s: max err %.3g (max|ref| %.3g)" % ((B, Cin, Cout, H, W), err, ref.abs().max().item()))
    assert err <= 2e-5 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("B,Cin,Cout,H,W", [(2, 128, 64, 33, 21), (1, 64, 256, 24, 40), (3, 64, 64, 64, 64)])
def test_conv3x3_pair_nchw_output_equals_single_sm(cuda_dev, B, Cin, Cout, H, W):
    """NCHW fp32 output of the CTA-pair convolution (conv_expand_fea_r feeds the MDTA statistics kernel in fp32) = the single-SM
    kernel's, bit for bit (same fp32 accumulation order)."""
    from cdfo_b200 import config, conv
    g = torch.Generator().manual_seed(B * Cin + H)
    x8 = conv.to_c8(torch.randn(B, Cin, H, W, generator=g).to(cuda_dev))
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).to(cuda_dev)
    b = (torch.randn(Cout, generator=g) * 0.1).to(cuda_dev)
    y_pair = conv.conv3x3(x8, w, b, conv.ACT_LRELU, out_nchw=True)
    config.conv_pair = False
    try:
        y_one = conv.conv3x3(x8, w, b, conv.ACT_LRELU, out_nchw=True)
    finally:
        config.conv_pair = True
    assert y_pair.dtype == torch.float32 and torch.equal(y_pair, y_one)
