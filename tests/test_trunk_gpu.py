"""Resample kernels and the c8 reconstruction trunk (SURVEY 8f rank 1) against torch / the oracle."""
import pytest
import torch
import torch.nn.functional as F

import golden_util as G
from oracle import torch_ref

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("H,W", [(8, 8), (24, 40), (34, 50)])
def test_resample_c8_half_and_double_vs_interpolate(cuda_dev, H, W):
    from cdfo_b200 import conv
    g = torch.Generator().manual_seed(H * W)
    x = torch.randn(2, 64, H, W, generator=g).to(torch.bfloat16).float().to(cuda_dev)
    x8 = conv.to_c8(x)
    up = conv.from_c8(conv.resample(x8, 1))
    ref_up = F.interpolate(x, scale_factor=2.0, mode="bilinear", align_corners=False)
    assert (up - ref_up).abs().max().item() <= 2 ** -8 * ref_up.abs().max().item()      # bf16 output rounding only
    dn = conv.from_c8(conv.resample(x8, 0))
    ref_dn = F.interpolate(x, scale_factor=0.5, mode="bilinear", align_corners=False)
    assert (dn - ref_dn).abs().max().item() <= 2 ** -8 * ref_dn.abs().max().item()


# the model's 24 x 40 test size; two samples at 16 x 24; 18 x 30, whose half-size images (9 x 15) are odd, with ragged tiles at every scale
@pytest.mark.parametrize("B,H,W", [(1, 24, 40), (2, 16, 24), (1, 18, 30)])
def test_trunk_vs_oracle(cuda_dev, B, H, W):
    """SCNet_ (21 cross-scale blocks) on c8 bf16 with composed 1x1 convolutions and the block sums in the folded convolution's epilogue
    vs the fp32 oracle (arch:378-480).  Observed on the B200 at 1 x 24 x 40: 7.2e-3 of max|ref| (21 blocks of bf16 activations); the
    bound is 1e-2."""
    from cdfo_b200 import conv, hotpath
    from cdfo_b200.model import CVSR_V8
    sd = G.seeded_weights("O1")
    m = CVSR_V8()
    m.load_state_dict(sd, strict=True)
    m = m.to(cuda_dev).eval()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, 64, H, W, generator=g)
    with torch.no_grad():
        ref = torch_ref.trunk(sd, x)
    got = conv.from_c8(hotpath.recon_trunk(m.recon_trunk, conv.to_c8(x.to(cuda_dev)))).cpu()
    err = (got - ref).abs().max().item()
    print("trunk %d x %d x %d max err %.3g (max|ref| %.3g)" % (B, H, W, err, ref.abs().max().item()))
    assert err <= 1e-2 * ref.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm_and_dwconv_vs_torch(cuda_dev, dtype):
    """Channel LayerNorm (arch:1169-1198) and the depthwise 3x3 of the MDTA attention (arch:1545-1576)."""
    from cdfo_b200 import hotpath
    g = torch.Generator().manual_seed(8)
    x = torch.randn(2, 64, 19, 37, generator=g).to(dtype)
    gamma, beta = torch.randn(64, generator=g), torch.randn(64, generator=g)
    xf = x.float()
    mu, var = xf.mean(1, keepdim=True), xf.var(1, keepdim=True, unbiased=False)
    ref = (xf - mu) * torch.rsqrt(var + 1e-5) * gamma.view(1, -1, 1, 1) + beta.view(1, -1, 1, 1)
    got = hotpath.layernorm_c(x.to(cuda_dev), gamma.to(cuda_dev), beta.to(cuda_dev)).float().cpu()
    tol = 1e-5 if dtype == torch.float32 else 2 ** -7
    assert (got - ref).abs().max().item() <= tol * ref.abs().max().item()
    x3 = torch.randn(2, 192, 19, 37, generator=g).to(dtype)
    w = torch.randn(192, 1, 3, 3, generator=g)
    ref = F.conv2d(x3.float(), w, None, 1, 1, 1, 192)
    got = hotpath.dwconv3x3(x3.to(cuda_dev), w.to(cuda_dev)).float().cpu()
    assert (got - ref).abs().max().item() <= tol * ref.abs().max().item()
    x4 = torch.randn(1, 24, 11, 40, generator=g).to(dtype)            # W % 8 == 0: vectorised bf16 path
    w4 = torch.randn(24, 1, 3, 3, generator=g)
    ref = F.conv2d(x4.float(), w4, None, 1, 1, 1, 24)
    got = hotpath.dwconv3x3(x4.to(cuda_dev), w4.to(cuda_dev)).float().cpu()
    assert (got - ref).abs().max().item() <= tol * ref.abs().max().item()


@pytest.mark.parametrize("dtype,H,W", [(torch.float32, 24, 40), (torch.bfloat16, 24, 40), (torch.float32, 9, 7), (torch.bfloat16, 40, 36)])
def test_self_mdta_gram_path_vs_torch_chain(cuda_dev, dtype, H, W):
    """Feature-extraction MDTA (Attention.forward, arch:1545-1576): Gram kernel + folded 64x64 matrix against the plain torch chain
    (normalize, q k^T over H*W, softmax, attn v, project_out) on the same depthwise-convolved qkv."""
    import torch.nn.functional as F
    from cdfo_b200 import hotpath
    from cdfo_b200.model import _SelfMDTA
    torch.manual_seed(3)
    m = _SelfMDTA(64, 8).to(cuda_dev)
    m.temperature.data = torch.rand(8, 1, 1, device=cuda_dev) + 0.5
    B = 2
    qkv = (torch.randn(B, 192, H, W, device=cuda_dev) * 0.7).to(dtype)
    G, nq, nk = hotpath.mdta_gram(qkv)
    q, k, v = qkv.float().chunk(3, dim=1)
    sh = (B, 8, 8, H * W)
    Gr = q.reshape(sh) @ k.reshape(sh).transpose(-2, -1)
    assert (G - Gr).abs().max().item() <= 1e-3 * Gr.abs().max().item()
    assert torch.allclose(nq, q.reshape(B, 64, -1).pow(2).sum(-1), rtol=1e-4) and torch.allclose(nk, k.reshape(B, 64, -1).pow(2).sum(-1), rtol=1e-4)
    qn, kn = F.normalize(q.reshape(sh), dim=-1), F.normalize(k.reshape(sh), dim=-1)
    attn = ((qn @ kn.transpose(-2, -1)) * m.temperature.float()).softmax(dim=-1)
    ref = F.conv2d((attn @ v.reshape(sh)).reshape(B, 64, H, W), m.project_out.weight.float())
    # the module itself (qkv conv + depthwise conv in front): compare through its own forward on an input x
    x = torch.randn(B, 64, H, W, device=cuda_dev).to(dtype)
    with torch.no_grad():
        mm = m.to(dtype)
        out = mm(x)
        qkv2 = hotpath.dwconv3x3(mm.qkv(x), mm.qkv_dwconv.weight)
        q2, k2, v2 = qkv2.float().chunk(3, dim=1)
        a2 = ((F.normalize(q2.reshape(sh), dim=-1) @ F.normalize(k2.reshape(sh), dim=-1).transpose(-2, -1)) * mm.temperature.float()).softmax(dim=-1)
        ref2 = F.conv2d((a2 @ v2.reshape(sh)).reshape(B, 64, H, W), mm.project_out.weight.float())
    tol = 2e-2 if dtype == torch.bfloat16 else 3e-3       # fp32: cuDNN's project_out convolution of the reference chain runs in TF32
    err = (out.float() - ref2).abs().max().item()
    print("self-MDTA %s %dx%d: max err %.3g (max|ref| %.3g)" % (dtype, H, W, err, ref2.abs().max().item()))
    assert err <= tol * max(1.0, ref2.abs().max().item())
    # and the fp64-free check of the folded matrix itself on the first qkv
    Mref = torch.einsum("ohi,bhij->bohj", m.project_out.weight.float().view(64, 8, 8), attn).reshape(B, 64, 64)
    assert (torch.bmm(Mref, v.reshape(B, 64, -1)).view(B, 64, H, W) - ref).abs().max().item() <= 3e-3 * max(1.0, ref.abs().max().item())
