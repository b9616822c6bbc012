"""Each c8 kernel of the feature extraction (csrc/features_c8.cu), run alone through its C entry point, against a float64 reference
written here, at the shapes of the c3 step (4 new frames of 272 x 480 per step, 28 on the first one, 24 samples of conv_expand_ufs) and
at the edges of each kernel's tiling.  Every input is rounded to bf16 first, so that only the kernel's own rounding counts, and every
output is filled with NaN before the call, so that an element the kernel never writes fails.  The bound is per element:

    |got - ref| <= rel |ref| + (1 + rel) e

rel = 2^-8, half a bf16 ulp, for bf16 outputs and 0 for fp32 ones.  e is the fp32 arithmetic of the kernel, derived in each test with
u = 2^-24: a chain of n roundings over terms t_k is off by at most n u sum |t_k|; a bf16 output rounds an fp32 value that is already
off by e, by at most rel (|ref| + e).  Each check prints the largest error / bound; the docstrings give the range seen on a B200.

Then the chains (self attention, side branch, the whole extraction) at the c3 shape against oracle/torch_ref in float64, and the
extraction's bit-exactness across batch sizes (first step vs later steps) and reruns."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import golden_util as G
from oracle import torch_ref

pytestmark = pytest.mark.gpu

U = 2.0 ** -24           # fp32 unit roundoff
HALF_BF16 = 2.0 ** -8    # half a bf16 ulp, relative


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _randn(g, *shape, scale=1.0, offset=0.0):
    """bf16-rounded normal samples on the generator's device."""
    return (torch.randn(*shape, generator=g, device=g.device) * scale + offset).to(torch.bfloat16)


def _to_c8(x):
    """[B, C, H, W] -> c8 bf16 [B, C/8, H, W, 8], by plain torch.  Keep the result in a variable until the kernel has been launched: a
    temporary whose only reference is the ctypes pointer is freed at once, and the allocator may hand its block to the next argument."""
    B, C, H, W = x.shape
    return x.to(torch.bfloat16).reshape(B, C // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


def _from_c8(x8):
    """c8 [B, C/8, H, W, 8] -> [B, C, H, W] float64, by plain torch."""
    B, C8, H, W, _ = x8.shape
    return x8.permute(0, 1, 4, 2, 3).reshape(B, C8 * 8, H, W).double()


def _nan_c8(B, C, H, W, dev):
    return torch.full((B, C // 8, H, W, 8), float("nan"), dtype=torch.bfloat16, device=dev)


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _check(name, got, ref, e, rel=HALF_BF16):
    """Assert |got - ref| <= rel |ref| + (1 + rel) e element by element (the value rounded to bf16 is within e of ref, so its half ulp is
    within rel (|ref| + e)); no element may be NaN (never written).  Returns the largest ratio."""
    got = got.double()
    assert got.shape == ref.shape, (name, tuple(got.shape), tuple(ref.shape))
    unwritten = int(torch.isnan(got).sum())
    err = (got - ref).abs()
    bound = rel * ref.abs() + (1 + rel) * e
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    worst = float(torch.nan_to_num(ratio, nan=float("inf")).max())
    print("%s: max error / bound %.3g" % (name, worst))
    assert unwritten == 0, "%s: %d elements not written" % (name, unwritten)
    assert worst <= 1.0, "%s: error %.3g x the bound (max error %.3g)" % (name, worst, float(err.max()))
    return worst


def _lrelu(x):
    return F.leaky_relu(x, 0.1)


# ------------------------------------------------------------------------------------------------------------------- prior_conv_c8
def _prior_conv_ref(x, w, b):
    """Conv2d(1, Co, 3, 1, 1) in float64 -> (value, sum of |terms| including the bias)."""
    x, w, b = x.double(), w.double(), b.double()
    return F.conv2d(x, w, b, padding=1), F.conv2d(x.abs(), w.abs(), b.abs(), padding=1)


# conv_expand_ufs on 6 B = 24 samples, conv_first / conv_second on the 4 new frames, a ragged size, a single pixel
@pytest.mark.parametrize("B,H,W", [(24, 272, 480), (4, 272, 480), (3, 19, 37), (1, 1, 1)])
@pytest.mark.parametrize("lrelu", [0, 1])
def test_prior_conv_c8_vs_fp64(cuda_dev, B, H, W, lrelu):
    """y = bias + 9 taps, one fmaf chain from the bias: 9 roundings, e = 9 u (|b| + sum |w x|).  With lrelu the negative side is one more
    product by 0.1f, which is 0.1 to within u / 4: e += 2 u |ref|.  With lrelu off, the output is bit for bit the bf16 rounding of
    cdfo_prior_conv_fwd's fp32 output (same taps, same fmaf order).  Observed on a B200: error / bound 0.85 - 0.996 (the bf16 rounding
    dominates: the bound is reached when a value rounds by almost half an ulp)."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 100 + B + H + lrelu)
    x = _randn(g, B, 1, H, W).float()
    w = torch.randn(64, 1, 3, 3, generator=g, device=cuda_dev) * 0.5
    b = torch.randn(64, generator=g, device=cuda_dev) * 0.2
    y = _nan_c8(B, 64, H, W, cuda_dev)
    _lib.call("cdfo_prior_conv_c8_fwd", _lib.ptr(x), _lib.ptr(w), _lib.ptr(b), _lib.ptr(y), B, 64, H, W, lrelu, _lib.stream_ptr(cuda_dev))
    acc, mag = _prior_conv_ref(x, w, b)
    ref = _lrelu(acc) if lrelu else acc
    e = 9 * U * mag + (2 * U * ref.abs() if lrelu else 0.0)
    _check("prior_conv_c8 %dx%dx%d lrelu=%d" % (B, H, W, lrelu), _from_c8(y), ref, e)
    if not lrelu:
        y32 = torch.empty((B, 64, H, W), dtype=torch.float32, device=cuda_dev)
        _lib.call("cdfo_prior_conv_fwd", _lib.ptr(x), _lib.ptr(w), _lib.ptr(b), _lib.ptr(y32), B, 64, H, W, _lib.stream_ptr(cuda_dev))
        assert torch.equal(_bits(y.permute(0, 1, 4, 2, 3).reshape(B, 64, H, W)), _bits(y32.to(torch.bfloat16)))


# ------------------------------------------------------------------------------------------------------------------- layernorm_c8
def _layernorm_ref(x, gamma, beta, eps=1e-5):
    """WithBias LayerNorm over channels in float64 -> (value, e).  The kernel's fp32 steps and what each costs:
      mean: 64 sequential adds, times 1/64 (exact)                  dmu = u sum |x|
      d = x - mean (rounded)                                         |dd| <= dmu + u |d|
      q = sum d^2 (fmaf chain of 64), / 64 (exact), + eps (rounded)  relative to var + eps: (66 u var + dmu^2) / (var + eps) + u
      r = rsqrtf (2 ulp = 4 u)                                       rho_r = that / 2 + 4 u
      o = (d r) gamma + beta (two roundings)                         e = |gamma| r (dmu + |d| (rho_r + 4 u)) + u |beta|
    The two-pass variance keeps dmu^2 / var small when the mean is large; E[x^2] - mean^2 in fp32 would not."""
    x = x.double()
    gamma, beta = gamma.double().view(1, -1, 1, 1), beta.double().view(1, -1, 1, 1)
    mu = x.mean(1, keepdim=True)
    d = x - mu
    var = (d * d).mean(1, keepdim=True)
    r = 1.0 / torch.sqrt(var + eps)
    ref = d * r * gamma + beta
    dmu = U * x.abs().sum(1, keepdim=True)
    rho_r = ((66 * U * var + dmu * dmu) / (var + eps) + U) / 2 + 4 * U
    e = gamma.abs() * r * (dmu + d.abs() * (rho_r + 4 * U)) + U * beta.abs()
    return ref, e


@pytest.mark.parametrize("B,H,W,mean,std", [(4, 272, 480, 0.0, 1.0), (2, 9, 7, 0.0, 1.0), (4, 272, 480, 30.0, 0.1)])
def test_layernorm_c8_vs_fp64(cuda_dev, B, H, W, mean, std):
    """Per-pixel LayerNorm over 64 channels; the (mean 30, std 0.1) input guards the two-pass variance.  e: see _layernorm_ref.  Observed
    on a B200: error / bound 0.93 (mean 30) - 0.995."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 200 + H)
    x = _randn(g, B, 64, H, W, scale=std, offset=mean)
    gamma = 1.0 + 0.2 * torch.randn(64, generator=g, device=cuda_dev)
    beta = 0.2 * torch.randn(64, generator=g, device=cuda_dev)
    x8, y = _to_c8(x), _nan_c8(B, 64, H, W, cuda_dev)
    _lib.call("cdfo_layernorm_c8_fwd", _lib.ptr(x8), _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(y), B, H, W, ctypes.c_float(1e-5),
              _lib.stream_ptr(cuda_dev))
    ref, e = _layernorm_ref(x, gamma, beta)
    _check("layernorm_c8 %dx%dx%d mean %g std %g" % (B, H, W, mean, std), _from_c8(y), ref, e)


# ------------------------------------------------------------------------------------------------------------------- dwconv3x3_c8
# The kernel tiles columns in blocks of 128 threads and rows in strips of 16: W = 127 / 128 is one block, 129 two (the last one column
# wide), 480 four (the last 96 wide); H = 1 / 15 / 16 is one strip, 17 two (the last one row), 272 seventeen.
@pytest.mark.parametrize("B,C,H,W", [(4, 192, 272, 480), (2, 192, 17, 129), (1, 192, 16, 128), (2, 192, 15, 127), (1, 192, 1, 129),
                                     (3, 8, 272, 129), (2, 8, 17, 480), (1, 8, 1, 127)])
def test_dwconv3x3_c8_vs_fp64(cuda_dev, B, C, H, W):
    """Depthwise 3x3, padding 1, no bias: one fmaf chain of 9 taps from 0, e = 9 u sum |w x|.  Observed on a B200: error / bound
    0.95 - 0.996."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 300 + C + H + W)
    x = _randn(g, B, C, H, W)
    w = torch.randn(C, 9, generator=g, device=cuda_dev) * 0.3
    x8, y = _to_c8(x), _nan_c8(B, C, H, W, cuda_dev)
    _lib.call("cdfo_dwconv3x3_c8_fwd", _lib.ptr(x8), _lib.ptr(w), _lib.ptr(y), B, C, H, W, _lib.stream_ptr(cuda_dev))
    xd, wd = x.double(), w.double().view(C, 1, 3, 3)
    ref = F.conv2d(xd, wd, padding=1, groups=C)
    e = 9 * U * F.conv2d(xd.abs(), wd.abs(), padding=1, groups=C)
    _check("dwconv3x3_c8 %dx%dx%dx%d" % (B, C, H, W), _from_c8(y), ref, e)


# ------------------------------------------------------------------------------------------------------------------- Gram and fold
def _qkv(dev, B, H, W, seed):
    """qkv [B, 192, H, W] bf16 whose k is, per head, a mix of q plus noise: normalised q k^T entries of order 1 (logits that depend on the
    temperature), channels of different scales (norms that matter)."""
    g = _gen(dev, seed)
    scale = torch.exp(torch.randn(64, generator=g, device=dev) * 0.5).view(1, 64, 1, 1)
    q = torch.randn(B, 64, H, W, generator=g, device=dev) * scale
    mix = torch.randn(8, 8, 8, generator=g, device=dev) / 8 ** 0.5
    k = torch.einsum("hij,bhjp->bhip", mix, q.view(B, 8, 8, H * W)).reshape(B, 64, H, W)
    k = k + 0.5 * torch.randn(B, 64, H, W, generator=g, device=dev)
    v = torch.randn(B, 64, H, W, generator=g, device=dev)
    return torch.cat((q, k, v), 1).to(torch.bfloat16)


def _gram_ref(qkv):
    """qkv [B, 192, H, W] -> (S, A) [B, 640] float64 in the partial layout (G [8 heads][8][8] | |q|^2 [64] | |k|^2 [64]): the exact sums S
    and the sums of |terms| A."""
    B = qkv.size(0)
    q = qkv[:, :64].double().reshape(B, 8, 8, -1)
    k = qkv[:, 64:128].double().reshape(B, 8, 8, -1)
    S = torch.cat((torch.matmul(q, k.transpose(-1, -2)).reshape(B, 512), (q * q).sum(-1).reshape(B, 64), (k * k).sum(-1).reshape(B, 64)), 1)
    A = torch.cat((torch.matmul(q.abs(), k.abs().transpose(-1, -2)).reshape(B, 512), S[:, 512:]), 1)
    return S, A


def _gram_depth(HW, parts):
    """Roundings on the way from a pixel to its part's sum: the thread's fmaf chain over every 256th pixel of the longest range, five
    shuffle levels, the 8 warps in order."""
    longest = -(-HW // parts)
    return -(-longest // 256) + 5 + 8


def _run_gram(qkv, parts):
    from cdfo_b200 import _lib
    B, C, H, W = qkv.shape
    partial = torch.full((B, parts, 640), float("nan"), dtype=torch.float32, device=qkv.device)
    qkv8 = _to_c8(qkv)
    _lib.call("cdfo_mdta_gram_c8_fwd", _lib.ptr(qkv8), _lib.ptr(partial), B, C, H, W, parts, _lib.stream_ptr(qkv.device))
    return partial


def _run_fold(partial, temperature, proj):
    from cdfo_b200 import _lib
    B, parts, _ = partial.shape
    M = torch.full((B, 64, 64), float("nan"), dtype=torch.float32, device=partial.device)
    _lib.call("cdfo_mdta_fold_fwd", _lib.ptr(partial), _lib.ptr(temperature), _lib.ptr(proj), _lib.ptr(M), B, parts,
              _lib.stream_ptr(partial.device))
    return M


def _fold_ref(S, dS, temperature, proj):
    """M = project_out . blockdiag_h softmax_j(G_h / (|q_i| |k_j|) T_h) in float64 from the sums S [B, 640], and its bound e given dS, the
    absolute error of the sums the kernel starts from.  The kernel's fp32 steps after that:
      |q|, |k| = sqrtf: relative dS / 2S + u;  l = G / (|q| |k|) * T: 3 roundings
          dl = |T| (dG + |G| (rho_q + rho_k + 3 u)) / (|q| |k|)
      z = l - max l (rounded: u |z|); __expf: 2 + 1.173 |z| ulp (ulp <= 2 u relative)      rho_exp = (2 + 1.173 |z|) 2 u + u |z|
      softmax: sum of 8, one division                       rho_attn_j = dl_j + max dl + rho_exp_j + max rho_exp + 8 u
      M[o][8h + j] = fmaf chain of 8 over i                 e = sum_i |P[o][8h + i]| attn[h][i][j] (rho_attn + 8 u)"""
    B = S.size(0)
    Gm, sq, sk = S[:, :512].view(B, 8, 8, 8), S[:, 512:576].view(B, 8, 8), S[:, 576:].view(B, 8, 8)
    dG, dsq, dsk = dS[:, :512].view(B, 8, 8, 8), dS[:, 512:576].view(B, 8, 8), dS[:, 576:].view(B, 8, 8)
    nq, nk = sq.sqrt().clamp_min(1e-12), sk.sqrt().clamp_min(1e-12)
    rq, rk = dsq / sq.clamp_min(1e-300) / 2 + U, dsk / sk.clamp_min(1e-300) / 2 + U
    den = nq[..., :, None] * nk[..., None, :]
    T = temperature.double().view(1, 8, 1, 1)
    l = Gm / den * T
    dl = T.abs() * (dG + Gm.abs() * (rq[..., :, None] + rk[..., None, :] + 3 * U)) / den
    z = l - l.amax(-1, keepdim=True)
    attn = torch.softmax(l, -1)
    rexp = (2 + 1.173 * z.abs()) * 2 * U + U * z.abs()
    rattn = dl + dl.amax(-1, keepdim=True) + rexp + rexp.amax(-1, keepdim=True) + 8 * U
    P = proj.double().view(64, 8, 8)
    M = torch.einsum("ohi,bhij->bohj", P, attn).reshape(B, 64, 64)
    e = torch.einsum("ohi,bhij->bohj", P.abs(), attn * (rattn + 8 * U)).reshape(B, 64, 64)
    return M, e


def _fold_weights(dev):
    g = _gen(dev, 400)
    temperature = torch.linspace(0.5, 4.0, 8, device=dev)          # a different temperature per head
    proj = torch.randn(64, 64, generator=g, device=dev) / 8.0
    return temperature, proj


# the c3 step (32 ranges of 4080 pixels), one sample with 7 ranges that do not divide H W, ranges shorter than 256 pixels, one range
GRAM_CASES = [(4, 272, 480, 32), (1, 272, 480, 7), (3, 17, 23, 32), (3, 17, 23, 7), (2, 9, 7, 1)]


@pytest.mark.parametrize("B,H,W,parts", GRAM_CASES)
def test_mdta_gram_c8_vs_fp64(cuda_dev, B, H, W, parts):
    """Sum of the fp32 partials (taken in float64) against the float64 q k^T and squared norms: e = depth u A, with depth the roundings of
    _gram_depth and A the sums of |terms|.  fp32 output: rel = 0.  Observed on a B200: error / bound 0.021 - 0.12."""
    qkv = _qkv(cuda_dev, B, H, W, 500 + parts)
    partial = _run_gram(qkv, parts)
    assert not torch.isnan(partial).any(), "a (sample, part, head) was not written"
    S, A = _gram_ref(qkv)
    _check("mdta_gram_c8 %dx%dx%d parts %d" % (B, H, W, parts), partial.double().sum(1), S, _gram_depth(H * W, parts) * U * A, rel=0.0)


@pytest.mark.parametrize("B,H,W,parts", GRAM_CASES)
def test_mdta_fold_on_kernel_partials_vs_fp64(cuda_dev, B, H, W, parts):
    """The fold alone: the Gram kernel's own partials in, float64 softmax . project_out on the same partials as the reference.  The fold
    sums the parts in fp32 in order: dS = parts u sum_parts |partial|; the rest in _fold_ref.  Observed on a B200: error / bound
    0.046 - 0.091."""
    temperature, proj = _fold_weights(cuda_dev)
    partial = _run_gram(_qkv(cuda_dev, B, H, W, 600 + parts), parts)
    M = _run_fold(partial, temperature, proj)
    pd = partial.double()
    ref, e = _fold_ref(pd.sum(1), parts * U * pd.abs().sum(1), temperature, proj)
    _check("mdta_fold %dx%dx%d parts %d" % (B, H, W, parts), M, ref, e, rel=0.0)


@pytest.mark.parametrize("B,H,W,parts", GRAM_CASES)
def test_mdta_gram_and_fold_vs_fp64(cuda_dev, B, H, W, parts):
    """Gram + fold end to end against float64 from the bf16 qkv, per-head temperatures 0.5 .. 4: dS = (depth + parts) u A.  Observed on a
    B200: error / bound 0.019 - 0.051."""
    temperature, proj = _fold_weights(cuda_dev)
    qkv = _qkv(cuda_dev, B, H, W, 700 + parts)
    M = _run_fold(_run_gram(qkv, parts), temperature, proj)
    S, A = _gram_ref(qkv)
    ref, e = _fold_ref(S, (_gram_depth(H * W, parts) + parts) * U * A, temperature, proj)
    _check("mdta_gram + fold %dx%dx%d parts %d" % (B, H, W, parts), M, ref, e, rel=0.0)


# ------------------------------------------------------------------------------------------------------------------- apply
# 5 tiles of 16 pixels per warp at the step's 4 frames, 33 at the first step's 28; H W = 63 and 391 end in a partial tile
@pytest.mark.parametrize("B,H,W", [(4, 272, 480), (28, 272, 480), (2, 9, 7), (3, 17, 23)])
@pytest.mark.parametrize("with_x2", [True, False])
def test_mdta_apply_c8_vs_fp64(cuda_dev, B, H, W, with_x2):
    """out1 = x1 + M v against x1 + bf16(M) v in float64 (the kernel rounds M to bf16 on purpose: the reference uses the same operand).
    The products are exact in fp32; the tensor cores add 16 of them per k step to the accumulator, four steps, and may truncate, so
    count 2 u per addition: e = 2 (64 + 4 + 1) u (sum |M v| + |x1|).  out2 must be bf16(bf16(out1) + x2) bit for bit, as a separate add
    kernel reading out1 would give.  Observed on a B200: error / bound 0.98 - 0.993."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 800 + B + H)
    HW = H * W
    qkv8 = _randn(g, B, 24, H, W, 8)
    M = torch.randn(B, 64, 64, generator=g, device=cuda_dev) * 0.2
    x1 = _randn(g, B, 64, H, W)
    x2 = _randn(g, B, 64, H, W) if with_x2 else None
    out1 = _nan_c8(B, 64, H, W, cuda_dev)
    out2 = _nan_c8(B, 64, H, W, cuda_dev) if with_x2 else None
    x1_8, x2_8 = _to_c8(x1), (_to_c8(x2) if with_x2 else None)
    _lib.call("cdfo_mdta_apply_c8_fwd", _lib.ptr(qkv8), 192, 128, _lib.ptr(M), _lib.ptr(x1_8), _lib.ptr(x2_8), _lib.ptr(out1), _lib.ptr(out2), B, H, W,
              _lib.stream_ptr(cuda_dev))
    v = _from_c8(qkv8[:, 16:]).reshape(B, 64, HW)
    Mq = M.to(torch.bfloat16).double()
    ref = x1.double() + torch.bmm(Mq, v).view(B, 64, H, W)
    e = 2 * 69 * U * (torch.bmm(Mq.abs(), v.abs()).view(B, 64, H, W) + x1.double().abs())
    del v
    _check("mdta_apply_c8 %dx%dx%d x2=%d" % (B, H, W, with_x2), _from_c8(out1), ref, e)
    if with_x2:
        want = (out1.float() + x2_8.float()).to(torch.bfloat16)
        assert torch.equal(_bits(out2), _bits(want))


# ------------------------------------------------------------------------------------------------------------------- conv16_c8
# (B, Hi, Wi, Ho, Wo, transposed, y_channels): the side branch at c3 (body.2, body.4, body.7, body.9 into the 64-channel buffer of body.11),
# ragged odd sizes, the smallest legal sizes of each mode, and a transposed convolution with output padding 0 in H and 1 in W
CONV16_CASES = [(4, 272, 480, 137, 241, 0, 16), (4, 137, 241, 70, 122, 0, 16), (4, 70, 122, 137, 241, 1, 16), (4, 137, 241, 272, 480, 1, 64),
                (4, 137, 241, 272, 480, 1, 16), (3, 5, 7, 4, 5, 0, 16), (2, 1, 1, 2, 2, 0, 16), (2, 2, 2, 1, 1, 1, 16),
                (2, 2, 2, 2, 2, 1, 64), (3, 3, 5, 3, 8, 1, 16)]


@pytest.mark.parametrize("B,Hi,Wi,Ho,Wo,transposed,y_channels", CONV16_CASES)
def test_conv16_c8_vs_fp64(cuda_dev, B, Hi, Wi, Ho, Wo, transposed, y_channels):
    """16 -> 16, 3x3, stride 2, padding 2 (+ lrelu 0.1) against F.conv2d / F.conv_transpose2d in float64: one fmaf chain from the bias
    over at most 9 taps x 16 channels, e = 144 u (|b| + sum |w x|), + 2 u |ref| for the lrelu product.  With y_channels = 64, chunks 2..7 of
    the output are prefilled with a canary and must come back untouched: side_branch_c8 keeps channels 16..63 of that buffer zero across
    calls.  Observed on a B200: error / bound 0.75 - 0.993."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 900 + Hi * Wi + Ho)
    x = _randn(g, B, 16, Hi, Wi)
    w = torch.randn(16, 16, 3, 3, generator=g, device=cuda_dev) * 0.2
    b = torch.randn(16, generator=g, device=cuda_dev) * 0.1
    y = torch.empty((B, y_channels // 8, Ho, Wo, 8), dtype=torch.bfloat16, device=cuda_dev)
    y[:, :2] = float("nan")
    canary = _randn(g, B, y_channels // 8 - 2, Ho, Wo, 8)
    y[:, 2:] = canary
    x8 = _to_c8(x)
    _lib.call("cdfo_conv16_c8_fwd", _lib.ptr(x8), _lib.ptr(w), _lib.ptr(b), _lib.ptr(y), B, Hi, Wi, Ho, Wo, y_channels, transposed,
              _lib.stream_ptr(cuda_dev))
    xd, wd, bd = x.double(), w.double(), b.double()
    if transposed:
        op = (Ho - (2 * Hi - 3), Wo - (2 * Wi - 3))
        acc = F.conv_transpose2d(xd, wd, bd, stride=2, padding=2, output_padding=op)
        mag = F.conv_transpose2d(xd.abs(), wd.abs(), bd.abs(), stride=2, padding=2, output_padding=op)
    else:
        acc = F.conv2d(xd, wd, bd, stride=2, padding=2)
        mag = F.conv2d(xd.abs(), wd.abs(), bd.abs(), stride=2, padding=2)
    ref = _lrelu(acc)
    _check("conv16_c8 %dx%dx%d -> %dx%d transposed=%d y_channels=%d" % (B, Hi, Wi, Ho, Wo, transposed, y_channels),
           _from_c8(y[:, :2].contiguous()), ref, 144 * U * mag + 2 * U * ref.abs())
    assert torch.equal(_bits(y[:, 2:]), _bits(canary)), "conv16_c8 wrote past channel 15"


# ------------------------------------------------------------------------------------------------------------------- spatial gate
@pytest.mark.parametrize("B,H,W", [(4, 70, 122), (2, 6, 4), (3, 3, 7), (1, 1, 1)])
def test_spatial_gate_c8_vs_fp64(cuda_dev, B, H, W):
    """y = x sigmoid(b + conv7x7([max_c x, mean_c x])) against float64.  The kernel's fp32 steps:
      mean: 16 sequential adds, times 1/16 (exact)                  dmean = 15 u mean |x|
      acc: fmaf chain of 98 taps from the bias                      dacc = sum |w_mean| dmean + 98 u (|b| + sum |w pooled|)
      gate = 1 / (1 + __expf(-acc)): __expf 2 + 1.173 |acc| ulp     dgate = g (1 - g) (dacc + (2 + 1.173 |acc|) 2 u) + 2 u g
      y = x gate (rounded)                                           e = |x| (dgate + u g)
    Below 7 x 7 every window crosses the border.  Observed on a B200: error / bound 0.63 - 0.995."""
    from cdfo_b200 import _lib
    g = _gen(cuda_dev, 1000 + H * W)
    x = _randn(g, B, 16, H, W)
    w = torch.randn(1, 2, 7, 7, generator=g, device=cuda_dev) * 0.3
    b = torch.randn(1, generator=g, device=cuda_dev) * 0.1
    pooled_ws = torch.empty((B, H, W, 2), dtype=torch.float32, device=cuda_dev)
    x8, y = _to_c8(x), _nan_c8(B, 16, H, W, cuda_dev)
    _lib.call("cdfo_spatial_gate_c8_fwd", _lib.ptr(x8), _lib.ptr(w), _lib.ptr(b), _lib.ptr(pooled_ws), _lib.ptr(y), B, H, W,
              _lib.stream_ptr(cuda_dev))
    xd, wd, bd = x.double(), w.double(), b.double()
    pooled = torch.cat((xd.amax(1, keepdim=True), xd.mean(1, keepdim=True)), 1)
    acc = F.conv2d(pooled, wd, bd, padding=3)
    gate = torch.sigmoid(acc)
    ref = xd * gate
    dmean = 15 * U * xd.abs().mean(1, keepdim=True)
    dacc = F.conv2d(torch.cat((torch.zeros_like(dmean), dmean), 1), wd.abs(), padding=3) + 98 * U * F.conv2d(pooled.abs(), wd.abs(), bd.abs(), padding=3)
    dgate = gate * (1 - gate) * (dacc + (2 + 1.173 * acc.abs()) * 2 * U) + 2 * U * gate
    _check("spatial_gate_c8 %dx%dx%d" % (B, H, W), _from_c8(y), ref, xd.abs() * (dgate + U * gate))


# ------------------------------------------------------------------------------------------------------------------- chains at c3
@pytest.fixture(scope="module")
def model(cuda_dev):
    from cdfo_b200.model import CVSR_V8
    m = CVSR_V8(alignment="mv_dcn")
    m.load_state_dict(G.seeded_weights("O2"), strict=True)
    m = m.to(cuda_dev).eval()
    return m, {k: v.detach().double() for k, v in m.state_dict().items()}


def _chain_error(name, got8, ref):
    got = _from_c8(got8)
    err = float((got - ref).abs().max()) / float(ref.abs().max())
    rel = float((got - ref).norm() / ref.norm())
    print("%s: max error %.3g of max|ref| (%.3g), relative L2 %.3g" % (name, err, float(ref.abs().max()), rel))
    return err, rel


PATH = "transformer_feature_extraction.path1"


def test_self_mdta_c8_vs_oracle_at_c3(cuda_dev, model):
    """qkv 1x1 (tcgen05, bf16 weights) -> depthwise -> Gram (32 parts) -> fold -> apply at 4 x 272 x 480 against torch_ref in float64.
    Observed on a B200: max error 3.0e-3 (out1) and 4.0e-3 (out2) of max|ref|, relative L2 2.0e-3 and 2.3e-3; the bounds are about twice
    that."""
    from cdfo_b200 import features
    m, sd = model
    g = _gen(cuda_dev, 1100)
    n, x1, x2 = (_randn(g, 4, 64, 272, 480) for _ in range(3))
    o1, o2 = features.self_mdta_c8(m.transformer_feature_extraction.path1.attn, _to_c8(n), _to_c8(x1), _to_c8(x2))
    with torch.no_grad():
        ref = x1.double() + torch_ref._self_mdta(sd, PATH + ".attn", n.double())
    e1, r1 = _chain_error("self_mdta_c8 out1", o1, ref)
    e2, r2 = _chain_error("self_mdta_c8 out2", o2, ref + x2.double())
    assert e1 <= 6e-3 and e2 <= 8e-3 and r1 <= 4e-3 and r2 <= 5e-3


@pytest.mark.parametrize("B,H,W", [(4, 272, 480), (2, 4, 4), (1, 4, 12), (2, 8, 4)])
def test_side_branch_c8_vs_oracle(cuda_dev, model, B, H, W):
    """The whole 16-channel branch + residual at the c3 shape and at the smallest sizes it accepts, against torch_ref in float64.  Observed
    on a B200: max error 2.0e-3 - 2.8e-3 of max|ref|, relative L2 1.6e-3 - 1.7e-3; the bounds are about twice that."""
    from cdfo_b200 import features
    m, sd = model
    g = _gen(cuda_dev, 1200 + H + W)
    s, r = _randn(g, B, 64, H, W, scale=0.5), _randn(g, B, 64, H, W, scale=0.5)
    out = features.side_branch_c8(m.transformer_feature_extraction.path1.side_to_feaoneUDSA, _to_c8(s), _to_c8(r))
    with torch.no_grad():
        ref = torch_ref._side_branch(sd, PATH + ".side_to_feaoneUDSA", s.double()) + r.double()
    err, rel = _chain_error("side_branch_c8 %dx%dx%d" % (B, H, W), out, ref)
    assert err <= 6e-3 and rel <= 3.5e-3


def _frames(n_seq, H, W):
    """The 7-frame windows of n_seq sequences as [7 n_seq, 1, H, W] fp32 frames and partition maps."""
    from cdfo_b200 import synthetic
    clip = synthetic.make_clip(3, H, W, n_seq)
    return clip["x"].reshape(-1, 1, H, W), clip["pms"].reshape(-1, 1, H, W)


def test_feature_extraction_c8_vs_oracle_at_c3(cuda_dev, model):
    """conv_first / conv_second + side branch + 3 transformer iterations on the step's 4 new frames at 272 x 480, against torch_ref in
    float64.  Observed on a B200: max error 1.21e-2 of max|ref| (13.6), relative L2 4.6e-3: bf16 activations through three iterations of
    four bf16 convolutions each.  The bounds are about twice that."""
    from cdfo_b200 import features
    m, sd = model
    x, pms = _frames(4, 272, 480)
    x, pms = x[3::7].to(cuda_dev), pms[3::7].to(cuda_dev)
    out = features.feature_extraction_c8(m, x, pms)
    with torch.no_grad():
        l1 = _lrelu(F.conv2d(x.double(), sd["conv_first.weight"], sd["conv_first.bias"], padding=1))
        s0 = F.conv2d(pms.double(), sd["conv_second.weight"], sd["conv_second.bias"], padding=1)
        ref = torch_ref.feature_extraction(sd, l1, s0)
    err, rel = _chain_error("feature_extraction_c8 4x272x480", out, ref)
    assert err <= 2.5e-2 and rel <= 1e-2


def test_feature_extraction_c8_batch_invariant_and_rerun(cuda_dev, model):
    """The first step extracts the 28 frames of the window, later steps the 4 new ones: a frame's features must not depend on which
    batch it came in.  Frame 25 alone, inside the last 4 and inside all 28 give the same bits; a rerun of the 4 gives the same bits."""
    from cdfo_b200 import features
    m, _ = model
    x, pms = _frames(4, 272, 480)
    x, pms = x.to(cuda_dev), pms.to(cuda_dev)
    all28 = features.feature_extraction_c8(m, x, pms)
    last4 = features.feature_extraction_c8(m, x[24:], pms[24:])
    one = features.feature_extraction_c8(m, x[25:26], pms[25:26])
    assert torch.equal(_bits(last4), _bits(all28[24:]))
    assert torch.equal(_bits(one), _bits(all28[25:26]))
    assert torch.equal(_bits(features.feature_extraction_c8(m, x[24:], pms[24:])), _bits(last4))
