"""Frames larger than 704 x 384 LR: JCT-VC Class A (2560x1600 HR = 640x400 LR) and 2160p UHD (3840x2160 HR = 960x540 LR, run on
544 rows).  The long-range attention row pass splits rows wider than 704 columns over a 2-CTA cluster, the column pass above 384
rows is the bf16 mma.sync kernel, and the texture DCN kernels split an x batch of more than 65 000 texture rows into slices.
The oracle runs on the GPU in fp32 (TF32 off) with torchvision's own deform_conv2d."""
import contextlib

import numpy as np
import pytest
import torch

import golden_util as G
from oracle import torch_ref

pytestmark = pytest.mark.gpu

TOL_ABS, TOL_PSNR = 1e-2, 0.02      # model-level bounds (BASELINE.json north star)


@contextlib.contextmanager
def _fp32_oracle():
    """Plain fp32 convolutions / matmuls, and torchvision's CUDA deform_conv2d rather than this library's override."""
    from cdfo_b200 import torchvision_override as tvo
    was = tvo.installed()
    tvo.uninstall()
    flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
        if was:
            tvo.install()


def _sd(variant, dev, sd=None):
    return {k: v.to(dev) for k, v in (sd or G.seeded_weights(variant)).items()}


def _model(variant, dev, sd=None, lowp=None):
    from cdfo_b200.model import CVSR_V8
    m = CVSR_V8(alignment="dual_att" if variant == "O1" else "mv_dcn")
    m.load_state_dict(sd if sd is not None else G.seeded_weights(variant), strict=True)
    m = m.to(dev).eval()
    m.lowp = lowp
    return m


def _lra_inputs(B, H, W, seed, dev):
    g = torch.Generator().manual_seed(seed)
    res = torch.randn(B, 64, H, W, generator=g) * 0.3
    x = torch.randn(B, 64, H, W, generator=g) * 0.5
    u = torch.rand(B, 64, H, W, generator=g).clamp_min(1e-12)
    return res.to(dev), x.to(dev), u.to(dev)


# ------------------------------------------------------------------------------------------------ long-range attention
# (1, 8, 1280): the widest row the cluster pass takes (and past the TMA ring's room: the cp.async load phase)
@pytest.mark.parametrize("B,H,W", [(1, 400, 640), (1, 544, 960), (2, 16, 1024), (1, 8, 1280)])
def test_lra_large_vs_oracle(cuda_dev, B, H, W):
    res, x, u = _lra_inputs(B, H, W, H * 1000 + W, cuda_dev)
    sd = _sd("O1", cuda_dev)
    with _fp32_oracle():
        ref = torch_ref.long_range_attention(sd, "RDAB.", res, x, u)
        mask = torch_ref.lra_mask(sd, "RDAB.", res, u)
    out = _model("O1", cuda_dev).RDAB(res, x, u)
    err = (out - ref).abs().max().item()
    print("LRA B%d %dx%d: max err %.3g, masked tokens %.1f%%" % (B, H, W, err, 100 * mask.sum(1).clamp(max=1).float().mean().item()))
    assert err <= 2e-3


def test_lra_dense_mask_wide_row(cuda_dev):
    """test_lra_dense_mask's construction at W = 960: > 90 % of the tokens masked, so almost every query's flash tile reads the key
    blocks of the other CTA of the cluster."""
    B, H, W = 1, 16, 960
    res, x, u = _lra_inputs(B, H, W, 5, torch.device("cpu"))
    sd = dict(G.seeded_weights("O1"))
    sd["RDAB.conv_du_re2.0.bias"] = sd["RDAB.conv_du_re2.0.bias"].clone()
    sd["RDAB.conv_du_re2.0.bias"][10] += 30.0
    u = u.clone()
    u[:, 13, :, ::3] = 1.0 - 1e-7
    sd["RDAB.conv_du_re2.0.bias"][13] += 16.0
    res, x, u = res.to(cuda_dev), x.to(cuda_dev), u.to(cuda_dev)
    sdd = _sd("O1", cuda_dev, sd)
    with _fp32_oracle():
        ref = torch_ref.long_range_attention(sdd, "RDAB.", res, x, u)
        mask = torch_ref.lra_mask(sdd, "RDAB.", res, u)
    out = _model("O1", cuda_dev, sd).RDAB(res, x, u)
    frac = mask.sum(1).clamp(max=1).float().mean().item()
    err = (out - ref).abs().max().item()
    print("LRA dense mask W=960: masked tokens %.1f%%, max err %.3g" % (100 * frac, err))
    assert frac > 0.9
    assert err <= 2e-3


def test_lra_cluster_rows_are_deterministic(cuda_dev):
    res, x, u = _lra_inputs(1, 544, 960, 11, cuda_dev)
    m = _model("O1", cuda_dev)
    a = m.RDAB(res, x, u)
    b = m.RDAB(res, x, u)
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ texture DCN slices
def _dcn_inputs(B, H, W, xB, dev, seed=3):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(2 * B, 64, H, W, generator=g) * 0.5
    c2 = torch.nn.Conv2d(64, 432, 3, 1, 1)
    with torch.no_grad():
        c2.weight.copy_(torch.randn(432, 64, 3, 3, generator=g) * 0.03)
        c2.bias.copy_(torch.randn(432, generator=g) * 0.2)
    x = torch.randn(xB, 64, H, W, generator=g)
    mv = torch.randint(-192, 192, (B, 2, H, W), generator=g).float() / 128.0
    wd = torch.randn(64, 64, 3, 3, generator=g) * 0.05
    bd = torch.randn(64, generator=g)
    from cdfo_b200 import dcn_sm100 as S
    f = torch.zeros(S.fields_shape(B, 16, H, W))
    f[..., :2] = torch.randn(f[..., :2].shape, generator=g) * 2.0
    f[..., 2] = torch.rand(f[..., 2].shape, generator=g)
    return z.to(dev), c2.to(dev), x.to(dev), mv.to(dev), wd.to(dev), bd.to(dev), f.half().to(dev)


def test_dcn_texture_slices_equal_separate_calls(cuda_dev):
    """x_batch = 8 at H = 544: 8 * 16 * 547 = 70 016 texture rows, two slices.  Every output sample equals, bit for bit, the same call
    made on each half of the sequences alone (plain and stacked entry points of both kernels; two neighbour groups, so that the
    slices enumerate b = k * x_batch + j for k > 0 too)."""
    from cdfo_b200 import conv, dcn_sm100 as S, hotpath
    xB, n_grp, H, W = 8, 2, 544, 64
    B = xB * n_grp
    z, c2, x, mv, wd, bd, fields = _dcn_inputs(B, H, W, xB, cuda_dev)
    z8, wd16 = conv.to_c8(z), S.pack_weight_f16(wd)
    hw, hb = hotpath._head_weights_fused(c2, 16)
    chunks = [0, 16]

    def run(js):
        sel = [k * xB + j for k in range(n_grp) for j in js]
        xq = S.pack_q4t(x[js].contiguous())
        zz = conv.to_c8(torch.cat([z[sel], z[[b + B for b in sel]]], 0))
        f, m = fields[sel].contiguous(), mv[sel].contiguous()
        st_t = torch.zeros((len(js), 40, H, W, 8), dtype=torch.bfloat16, device=cuda_dev)
        S.dcn_tex_stacked(xq, f, wd16, bd, m, st_t, chunks)
        st_f = torch.zeros_like(st_t)
        S.mv_head_dcn_fused(zz, hw, hb, 10.0, xq, m, wd16, bd, stack=st_f, group_chunk=chunks)
        return sel, S.dcn_tex(xq, f, wd16, bd, mv=m), S.mv_head_dcn_fused(zz, hw, hb, 10.0, xq, m, wd16, bd), st_t, st_f

    everything = list(range(xB))
    _, y_t, y_f, st_t, st_f = run(everything)
    assert xB * 16 * (H + 3) > 65000
    for js in (everything[:4], everything[4:]):
        sel, h_t, h_f, hs_t, hs_f = run(js)
        assert torch.equal(y_t[sel], h_t)
        assert torch.equal(y_f[sel], h_f)
        assert torch.equal(st_t[js], hs_t)
        assert torch.equal(st_f[js], hs_f)
    assert torch.isfinite(y_t).all() and y_t.abs().max() > 0


# ------------------------------------------------------------------------------------------------ the whole model
@pytest.mark.parametrize("variant,H,W", [("O2", 544, 960), ("O1", 400, 640)])
def test_full_model_large_frame_vs_oracle(cuda_dev, variant, H, W):
    from cdfo_b200 import synthetic
    from oracle import priors_ref
    clip = synthetic.make_clip(41, H, W, 1)
    mvs = torch.from_numpy(priors_ref.mv2mvs_model_layout(clip["mv_l0"][0].numpy()))
    n0, n1 = synthetic.gumbel_uniforms(4, 2, 0, 1, H, W), synthetic.gumbel_uniforms(4, 2, 1, 1, H, W)
    c = {k: v.to(cuda_dev) for k, v in clip.items() if k in ("x", "pms", "rms", "ufs")}
    mvs = mvs.to(cuda_dev)
    n0, n1 = [u.to(cuda_dev) for u in n0], [u.to(cuda_dev) for u in n1]
    sd = _sd(variant, cuda_dev)
    with _fp32_oracle():
        ref0, l1_ref = torch_ref.cvsr_v8_forward(sd, c["x"], mvs, c["pms"], c["rms"], c["ufs"], None, n0, variant)
        ref1, _ = torch_ref.cvsr_v8_forward(sd, c["x"], mvs, c["pms"], c["rms"], c["ufs"], l1_ref, n1, variant)
        ref0, ref1 = ref0.cpu(), ref1.cpu()
        del l1_ref
    m = _model(variant, cuda_dev, lowp=torch.bfloat16)
    sr0, l1 = m(c["x"], None, mvs, c["pms"], c["rms"], c["ufs"], None, noise=n0)
    sr1, _ = m(c["x"], None, mvs, c["pms"], c["rms"], c["ufs"], l1, noise=n1)
    rng = np.random.default_rng(2)
    for name, sr, ref in (("first", sr0, ref0), ("cached", sr1, ref1)):
        out, r = sr.float().cpu().numpy(), ref.numpy()
        err = np.abs(out - r).max()
        target = np.clip(r + rng.normal(0, 0.02, r.shape), 0, 1)
        dpsnr = abs(G.psnr(np.clip(out, 0, 1), target) - G.psnr(np.clip(r, 0, 1), target))
        print("CVSR_V8 %s %dx%d %s frame: max abs err %.3g, dPSNR %.4f dB" % (variant, H, W, name, err, dpsnr))
        assert err <= TOL_ABS and dpsnr <= TOL_PSNR


def test_2160p_step_of_eight_sequences_is_batching_invariant(cuda_dev):
    """2160p with 8 sequences per step (sliced DCN textures; the trunk's 256-channel 2x tensor holds 4.3e9 elements, past 2^31):
    each sequence's SR frames are within one uint8 level of the same sequence run alone, and the trunk on the batch equals the
    per-sample trunk bit for bit."""
    from cdfo_b200 import conv, driver, hotpath
    from test_driver_gpu import _sequence
    T, h, W, S = 2, 540, 960, 8
    seqs = [_sequence(50 + s, T, h, W, with_gt=False) for s in range(S)]
    m = _model("O2", cuda_dev, lowp=torch.bfloat16)
    both = {}
    driver.FrameDriver(m, seed=3).run(seqs, seq_ids=list(range(S)), sink=lambda s, i, img: both.__setitem__((s, i), img))
    for s in range(S):
        alone = {}
        driver.FrameDriver(m, seed=3).run([seqs[s]], seq_ids=[s], sink=lambda _, i, img: alone.__setitem__(i, img))
        for i in range(T):
            assert both[(s, i)].shape == (4 * h, 4 * W)
            d = np.abs(both[(s, i)].astype(np.int64) - alone[i].astype(np.int64))
            assert d.max() <= 1 and (d > 0).mean() < 0.08, (s, i, d.max(), (d > 0).mean())
    g = torch.Generator(device=cuda_dev).manual_seed(4)
    x8 = conv.to_c8(torch.randn((S, 64, 544, W), device=cuda_dev, generator=g) * 0.5)
    y = hotpath.recon_trunk(m.recon_trunk, x8)
    for s in range(S):
        assert torch.equal(y[s:s + 1], hotpath.recon_trunk(m.recon_trunk, x8[s:s + 1].contiguous())), s


def test_driver_2160p_matches_naive_loop(cuda_dev):
    """FrameDriver on 540-row, 960-column sequences (run on 544 rows): 2160 x 3840 SR frames after the crop, within one uint8 level of
    the window-by-window loop."""
    from cdfo_b200 import driver
    from test_driver_gpu import _naive_loop, _sequence
    T, h, W = 3, 540, 960
    seqs = [_sequence(60, T, h, W, with_gt=False), _sequence(61, T, h, W, with_gt=False)]
    m = _model("O2", cuda_dev)
    got = {}
    driver.FrameDriver(m, seed=9).run(seqs, seq_ids=[5, 6], sink=lambda s, i, img: got.__setitem__((s, i), img))
    for s, q in enumerate(seqs):
        ref = _naive_loop(m, q, 5 + s, 9, cuda_dev)
        for i in range(T):
            assert got[(s, i)].shape == (2160, 3840)
            d = np.abs(got[(s, i)].astype(np.int64) - ref[i].astype(np.int64))
            assert d.max() <= 1 and (d > 0).mean() < 0.08, (s, i, d.max(), (d > 0).mean())
