"""Host-side mirror of the reference model `CVSR_V8` (arch/SIDECVSR_our.py:4371-4481).

Same constructor signature, same `forward(x, mvs0, mvs1, pms, rms, ufs, pre_L1_fea=None) -> (sr, L1_fea)`,
same parameter names and shapes (reference state_dicts load with strict=True), but a different execution plan:

  * the six neighbour iterations of the reference's Python loop (arch:4443-4460) are independent, so every
    hot-path module runs ONCE on a batch of 6*B (neighbour-major) instead of six times;
  * the hot path -- prior-guided attention (RDAB), MV-guided alignment (DualAttAlignment /
    MVDualAttAlignment + DCN), fusion and the upsampling tail -- runs in the CUDA kernels of libcdfo_b200
    (see hotpath.py); CUDA only, no CPU fallback;
  * the parts SURVEY.md 8(f) ranks as "next" (feature extraction, reconstruction trunk) run in this repo's c8 bf16 kernels when
    `self.lowp` is torch.bfloat16 (features.py, hotpath.recon_trunk); with lowp = None the feature extraction is the plain fp32 torch
    chain (used by the fp32 parity tests) and `trunk_backend = "cudnn"` selects torch convolutions for A/B runs.

`alignment="dual_att"` is the model as shipped (O1); `alignment="mv_dcn"` swaps in the DCN alignment the
reference carries commented out at arch:4396 (O2, the variant BASELINE.json's DCN roofline is quoted on).

Gumbel noise: the reference draws torch.rand_like inside LLongRangAttention (arch:2169). Here the six uniform
tensors are an explicit input (`noise=`); when omitted they are drawn from `self.noise_generator`
(device RNG), in the reference's neighbour order.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import config, hotpath

_NB = (0, 1, 2, 4, 5, 6)


def _lrelu(x):
    return F.leaky_relu(x, 0.1)


class _Holder(nn.Module):
    """A module that only owns parameters / sub-modules; the compute lives in functions."""


def _seq(*mods_by_index):
    """nn.Sequential-like container with explicit integer names (reference uses nn.Sequential indices)."""
    h = _Holder()
    for idx, m in mods_by_index:
        h.add_module(str(idx), m)
    return h


# ------------------------------------------------------------------------------------------ "next" rows: parameter holders + fp32 torch chain
class _ChannelLayerNorm(_Holder):
    """LayerNorm(dim, WithBias) over channels per pixel, arch:1169-1198; parameters live at `.body`."""

    def __init__(self, dim):
        super().__init__()
        self.body = _Holder()
        self.body.weight = nn.Parameter(torch.ones(dim))
        self.body.bias = nn.Parameter(torch.zeros(dim))

    def forward(self, x):
        if x.is_cuda and x.dtype in (torch.float32, torch.bfloat16) and x.size(1) == 64:
            return hotpath.layernorm_c(x, self.body.weight, self.body.bias)
        mu = x.mean(1, keepdim=True)
        var = x.var(1, keepdim=True, unbiased=False)
        return (x - mu) * torch.rsqrt(var + 1e-5) * self.body.weight.view(1, -1, 1, 1) + self.body.bias.view(1, -1, 1, 1)


class _SelfMDTA(_Holder):
    """Attention (MDTA), arch:1545-1576."""

    def __init__(self, dim, heads):
        super().__init__()
        self.num_heads = heads
        self.temperature = nn.Parameter(torch.ones(heads, 1, 1))
        self.qkv = nn.Conv2d(dim, dim * 3, 1, bias=False)
        self.qkv_dwconv = nn.Conv2d(dim * 3, dim * 3, 3, 1, 1, groups=dim * 3, bias=False)
        self.project_out = nn.Conv2d(dim, dim, 1, bias=False)

    def forward(self, x):
        b, c, h, w = x.shape
        qkv = self.qkv(x)
        if qkv.is_cuda and qkv.dtype in (torch.float32, torch.bfloat16):
            qkv = hotpath.dwconv3x3(qkv, self.qkv_dwconv.weight)
        else:
            qkv = self.qkv_dwconv(qkv)
        if qkv.is_cuda and qkv.dtype in (torch.float32, torch.bfloat16) and c == 64 and self.num_heads == 8 and qkv.is_contiguous():
            # the attention is one 64 x 64 matrix per sample: softmax(G / (|q| |k|) T) folded with project_out, applied to v as a batched GEMM
            G, nq, nk = hotpath.mdta_gram(qkv)
            nq = nq.sqrt().clamp_min(1e-12).view(b, 8, 8, 1)          # F.normalize: x / max(|x|, eps)
            nk = nk.sqrt().clamp_min(1e-12).view(b, 8, 1, 8)
            attn = (G / (nq * nk) * self.temperature.float().view(1, 8, 1, 1)).softmax(dim=-1)
            M = torch.einsum("ohi,bhij->bohj", self.project_out.weight.float().view(64, 8, 8), attn).reshape(b, 64, 64)
            v = qkv[:, 128:].reshape(b, 64, h * w)
            return torch.bmm(M.to(v.dtype), v).view(b, 64, h, w)
        q, k, v = qkv.chunk(3, dim=1)
        sh = (b, self.num_heads, c // self.num_heads, h * w)
        q = F.normalize(q.reshape(sh).float(), dim=-1)
        k = F.normalize(k.reshape(sh).float(), dim=-1)
        attn = ((q @ k.transpose(-2, -1)) * self.temperature.float()).softmax(dim=-1)
        out = (attn.to(v.dtype) @ v.reshape(sh)).reshape(b, c, h, w)
        return self.project_out(out)


class _SpatialGate(_Holder):
    """SpatialAttention, arch:1883-1899."""

    def __init__(self):
        super().__init__()
        self.spatial = nn.Conv2d(2, 1, 7, 1, 3)

    def forward(self, x):
        pooled = torch.cat((x.amax(1, keepdim=True), x.mean(1, keepdim=True)), dim=1)
        return x * torch.sigmoid(self.spatial(pooled))


class _SideBranch(_Holder):
    """side_to_feaoneUDSA_2, arch:1815-1875 (Sequential indices 0,2,4 conv; 6 gate; 7,9 transposed conv; 11 conv)."""

    def __init__(self, in_f, nf):
        super().__init__()
        self.body = _seq(
            (0, nn.Conv2d(in_f, nf, 3, 1, 1)), (2, nn.Conv2d(nf, nf, 3, 2, 2)), (4, nn.Conv2d(nf, nf, 3, 2, 2)),
            (6, _SpatialGate()), (7, nn.ConvTranspose2d(nf, nf, 3, 2, 2)),
            (9, nn.ConvTranspose2d(nf, nf, 3, 2, 2, output_padding=1)), (11, nn.Conv2d(nf, in_f, 3, 1, 1)))

    def forward(self, s):
        b = self.body._modules
        x = _lrelu(b["0"](s))
        x = _lrelu(b["2"](x))
        x = _lrelu(b["4"](x))
        x = b["6"](x)
        x = _lrelu(b["7"](x))
        x = _lrelu(b["9"](x))
        return _lrelu(b["11"](x))


class _PartitionTransformer(_Holder):
    """PartitionTransformerSA_2, arch:1441-1475."""

    def __init__(self, dim=64, heads=8):
        super().__init__()
        self.norm1 = _ChannelLayerNorm(dim)
        self.attn = _SelfMDTA(dim, heads)
        self.norm2 = _ChannelLayerNorm(dim)
        self.conv = nn.Conv2d(dim, dim, 3, 1, 1)
        self.side_to_feaoneUDSA = _SideBranch(dim, 16)

    def forward(self, x1, x2):
        x2 = self.side_to_feaoneUDSA(x2) + x1
        for it in range(3):
            if it:
                x2 = self.side_to_feaoneUDSA(x2) + x2
            x1 = x1 + self.attn(self.norm1(x1))
            x1 = x1 + self.conv(self.norm2(x1)) + x2
        return x1


class _FeatureExtraction(_Holder):
    """PAItransformerSA_2, arch:1643-1653 (its adaptiveWeight tuple is not registered -> no state_dict keys)."""

    def __init__(self):
        super().__init__()
        self.path1 = _PartitionTransformer(64, 8)

    def forward(self, x1, x2):
        return self.path1(x1, x2)


class _CrossScaleBlock(_Holder):
    """Block_, arch:378-406."""

    def __init__(self, nf=64, mult=4):
        super().__init__()
        self.body = _seq((0, nn.Conv2d(nf, nf * mult, 3, padding=1)), (2, nn.Conv2d(nf * mult, nf, 3, padding=1)))
        self.down = _seq((0, nn.Conv2d(nf, nf, 1)))
        self.up = _seq((0, nn.Conv2d(nf, nf, 1)))

    def _body(self, z):
        b = self.body._modules
        return b["2"](_lrelu(b["0"](z)))

    def forward(self, x):
        dn = lambda z: F.interpolate(self.down._modules["0"](z), scale_factor=0.5, mode="bilinear", align_corners=False)  # noqa: E731
        up = lambda z: F.interpolate(self.up._modules["0"](z), scale_factor=2.0, mode="bilinear", align_corners=False)  # noqa: E731
        return x + self._body(x) + up(self._body(dn(x))) + dn(self._body(up(x)))


class _CrossScaleGroup(_Holder):
    """SCGroup_, arch:430-444."""

    def __init__(self, nf=64):
        super().__init__()
        self.conv = nn.Conv2d(nf, nf, 3, padding=1)
        self.body = _seq(*[(k, _CrossScaleBlock(nf)) for k in range(3)])

    def forward(self, x):
        r = x
        for k in range(3):
            r = self.body._modules[str(k)](r)
        return x + self.conv(r)


class _Trunk(_Holder):
    """SCNet_(SCGroupN=7), arch:468-480."""

    def __init__(self, nf=64, groups=7):
        super().__init__()
        self.body = _seq(*[(g, _CrossScaleGroup(nf)) for g in range(groups)])

    def forward(self, x):
        y = x
        for m in self.body._modules.values():
            y = m(y)
        return y + x


# ------------------------------------------------------------------------------------------ hot-path parameter holders
class LLongRangAttention(_Holder):
    """Parameters of arch:2141-2162; forward = hotpath.long_range_attention (arch:2179-2249)."""

    def __init__(self, in_dim=64):
        super().__init__()
        self.input_conv = nn.Conv2d(in_dim, in_dim * 2, 1)
        self.conv_du_re = _seq((0, nn.Conv2d(in_dim, in_dim, 1)), (2, nn.Conv2d(in_dim, in_dim, 3, 2, 2)))
        self.conv_du_re2 = _seq((0, nn.Conv2d(in_dim, in_dim, 1)))
        self.fuse = nn.Conv2d(in_dim * 2, in_dim, 1)
        self.directW1_conv = nn.Conv2d(1, 1, (1, 9), 1, (0, 4))
        self.directH1_conv = nn.Conv2d(1, 1, (9, 1), 1, (4, 0))
        self.window_size = 8

    def forward(self, res, x, noise):
        return hotpath.long_range_attention(self, res, x, noise)


class _ResBlock(_Holder):
    def __init__(self, nf):
        super().__init__()
        self.conv1 = nn.Conv2d(nf, nf, 3, 1, 1)
        self.conv2 = nn.Conv2d(nf, nf, 3, 1, 1)


class _CAParams(_Holder):
    def __init__(self, c):
        super().__init__()
        self.conv_du = _seq((0, nn.Conv2d(c, c, 1)), (2, nn.Conv2d(c, c, 1)))


class DualAttAlignment(_Holder):
    """Parameters of arch:3427-3453 (fusion_in is owned but unused, like the reference); forward arch:3455-3496."""

    def __init__(self):
        super().__init__()
        dim = 64
        self.out_channels, self.num_heads = dim, 4
        self.conv_du = _seq((0, nn.Conv2d(dim, dim // 16, 1)), (2, nn.Conv2d(dim // 16, dim, 1)))
        self.temperature = nn.Parameter(torch.ones(self.num_heads, 1, 1))
        self.project_out = nn.Conv2d(dim, dim, 1, bias=False)
        self.fusion_in = _seq((0, nn.Conv2d(dim * 2, dim, 1)), (2, nn.Conv2d(dim, dim, 1)))
        self.fusion_out = _seq((0, nn.Conv2d(dim * 2, dim, 1, bias=False)))
        self.CALayer = _CAParams(dim)
        self.ResidualBlock = _ResBlock(dim)
        self.ResidualBlock1 = _ResBlock(dim)

    def forward(self, x, extra_feat, pred_feat, flow_1):
        return hotpath.dual_att_alignment(self, x, extra_feat, pred_feat, flow_1)


class MVDualAttAlignment(_Holder):
    """Parameters of arch:3265-3301 (a ModulatedDeformConv base: weight [64,64,3,3], bias [64]); forward :3303-3352."""

    def __init__(self, in_channels=64, out_channels=64, kernel_size=3, stride=1, padding=1, dilation=1, groups=1,
                 deformable_groups=16, bias=True, max_residue_magnitude=10):
        super().__init__()
        assert (in_channels, out_channels, kernel_size, stride, padding, dilation, groups) == (64, 64, 3, 1, 1, 1, 1)
        self.max_residue_magnitude = max_residue_magnitude
        self.in_channels, self.out_channels, self.deformable_groups = in_channels, out_channels, deformable_groups
        self.stride, self.padding, self.dilation, self.groups = stride, padding, dilation, groups
        self.num_heads = 8
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels, 3, 3).uniform_(-1 / 24.0, 1 / 24.0))
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.conv_offset = _seq((0, nn.Conv2d(out_channels, out_channels, 3, 1, 1)),
                                (2, nn.Conv2d(out_channels, 27 * deformable_groups, 3, 1, 1)))
        self.conv_du = _seq((0, nn.Conv2d(out_channels, out_channels // 16, 1)),
                            (2, nn.Conv2d(out_channels // 16, out_channels, 1)))
        self.fusion_out = nn.Conv2d(128, 64, 1, bias=False)
        self.temperature = nn.Parameter(torch.ones(self.num_heads, 1, 1))
        self.project_out = nn.Conv2d(64, 64, 1, bias=False)
        nn.init.zeros_(self.conv_offset._modules["2"].weight)   # arch:3293-3301
        nn.init.zeros_(self.conv_offset._modules["2"].bias)

    def forward(self, x, extra_feat, pred_feat, flow_1):
        return hotpath.mv_dual_att_alignment(self, x, extra_feat, pred_feat, flow_1)


class FeatureRing:
    """The sliding window's L1 features (arch:4417-4427 keeps them as `pre_L1_fea` and rebuilds the [B*N] tensor with a cat per
    frame) as a frame-major ring in HBM: 2N slots of [B, C, H, W] fp32, frame t stored at t % N and t % N + N, so the window is
    always ONE contiguous view buf[head : head + N] -- a step writes the new frame twice (2 x B x 33 MB at c3) instead of copying
    all N frames, the centre frame and the two neighbour runs (frames 0-2 and 4-6) are contiguous views."""

    def __init__(self, l1_bn, B, N):
        C, H, W = l1_bn.shape[1:]
        self.B, self.N, self.head, self.serial = B, N, 0, 0
        self.buf = torch.empty((2 * N, B, C, H, W), dtype=torch.float32, device=l1_bn.device)
        fm = l1_bn.view(B, N, C, H, W).transpose(0, 1)
        self.buf[:N].copy_(fm)
        self.buf[N:].copy_(fm)

    def push(self, new):
        self.buf[self.head].copy_(new)
        self.buf[self.head + self.N].copy_(new)
        self.head = (self.head + 1) % self.N
        self.serial += 1

    def window(self):
        return self.buf[self.head:self.head + self.N]

    def load(self, b, frames):
        """Window positions 1 .. len(frames) of batch sample b (both copies) := frames, each [C, H, W]: the features a sample needs
        before the next push to hold a new window (frame driver admission; position 0 is pushed out by that step)."""
        for p, f in enumerate(frames, 1):
            t = (self.head + p) % self.N
            self.buf[t, b].copy_(f)
            self.buf[t + self.N, b].copy_(f)

    def handle(self):
        """What forward() returns as L1_fea in ring mode: a view of the window (FRAME-major [N*B, C, H, W]; equal to the
        reference's tensor for B = 1) tagged with the ring, valid until the next step."""
        w = self.window()
        t = w.view(self.N * self.B, *w.shape[2:])
        t._cdfo_ring = (self, self.serial)
        return t


# ------------------------------------------------------------------------------------------ the model
class CVSR_V8(nn.Module):
    def __init__(self, nf=64, nframes=7, fea_ext_RBs=7, SCGs=4, istraining=False, alignment="dual_att"):
        super().__init__()
        assert nf == 64 and nframes == 7, "the kernels are specialised for the shipped configuration (nf=64, 7 frames)"
        self.nf, self.center, self.istraining, self.stride = nf, nframes // 2, istraining, 4
        self.conv_first = nn.Conv2d(1, nf, 3, 1, 1)
        self.conv_second = nn.Conv2d(1, nf, 3, 1, 1)
        self.transformer_feature_extraction = _FeatureExtraction()
        self.conv_expand_fea_r = nn.Conv2d(2 * nf, nf, 3, 1, 1)
        self.conv_expand_ufs = nn.Conv2d(1, nf, 3, 1, 1)
        self.conv_expand_rms = nn.Conv2d(1, nf, 3, 1, 1)
        self.tsa_fusion = nn.Conv2d(nframes * nf, nf, 1, 1)
        self.recon_trunk = _Trunk(nf, 7)
        self.upconv1 = nn.Conv2d(nf, nf * 4, 1, 1, 0)
        self.upconv2 = nn.Conv2d(nf, nf * 4, 1, 1, 0)
        self.conv_last = nn.Conv2d(nf, 1, 3, 1, 1)
        if alignment == "dual_att":
            self.MV_deform_align = DualAttAlignment()
        elif alignment == "mv_dcn":
            self.MV_deform_align = MVDualAttAlignment(64, 64, 3, padding=1, deformable_groups=16, max_residue_magnitude=10)
        else:
            raise ValueError("alignment must be 'dual_att' (as shipped) or 'mv_dcn' (arch:4396)")
        self.alignment = alignment
        self.RDAB = LLongRangAttention(64)
        self.lowp = None            # torch dtype for the non-hot-path convolutions (None: fp32)
        self.noise_generator = None
        self.trunk_backend = "cuda"   # "cuda": tcgen05 convs + resample kernels on c8 bf16; "cudnn": torch convolutions
        self.feature_ring = False     # True: the returned L1_fea is a FeatureRing handle (no per-frame copies of the window's features)

    # -- feature extraction of `n` frames ("next" row f2): own c8 bf16 kernels with lowp = bf16
    def _features(self, x, pms):
        dt = self.lowp
        if dt is torch.bfloat16 and config.features_c8 and x.is_cuda:
            from . import conv, features
            return conv.from_c8(features.feature_extraction_c8(self, x, pms))
        if dt is not None:
            with torch.autocast("cuda", dtype=dt):
                l1 = _lrelu(self.conv_first(x))
                l1 = self.transformer_feature_extraction(l1, self.conv_second(pms))
            return l1.float()
        l1 = _lrelu(self.conv_first(x))
        return self.transformer_feature_extraction(l1, self.conv_second(pms))

    def _trunk(self, x8):
        """c8 bf16 in -> c8 bf16 out on the tcgen05 kernels ("next" row f1); NCHW fp32 out on the torch A/B backend."""
        from . import conv
        if self.trunk_backend == "cuda":
            return hotpath.recon_trunk(self.recon_trunk, x8)      # c8 bf16 out: the tail takes it as is
        x = conv.from_c8(x8)
        dt = self.lowp
        if dt is not None:
            with torch.autocast("cuda", dtype=dt):
                return self.recon_trunk(x.contiguous(memory_format=torch.channels_last)).float()
        return self.recon_trunk(x)

    @torch.no_grad()
    def load_window_features(self, l1, b, x, pms, order):
        """Starts a new window in batch sample b of a running sequence of steps: computes the L1 features of the distinct frames
        x, pms [n, 1, H, W] and writes feature order[p] to window position p + 1 (p = 0..5) of `l1`, the L1_fea the previous step
        returned (a FeatureRing handle or the batch-major [B*N, C, H, W] tensor).  The next step's push of its new frame then leaves
        sample b with the features of the whole new window, as if it had started with it."""
        f = self._features(x, pms)
        ring = getattr(l1, "_cdfo_ring", None)
        if ring is not None:
            ring[0].load(b, [f[k] for k in order])
            return
        win = l1.view(-1, 2 * self.center + 1, *l1.shape[1:])[b]
        for p, k in enumerate(order, 1):
            win[p].copy_(f[k])

    @torch.no_grad()
    def forward(self, x, mvs0, mvs1, pms, rms, ufs, pre_L1_fea=None, noise=None):
        if not x.is_cuda:
            raise NotImplementedError("cdfo_b200.CVSR_V8 is CUDA-only (no CPU fallback); use the reference for CPU runs")
        B, N, C, H, W = x.shape
        assert N == 7 and C == 1 and H % 8 == 0 and W % 8 == 0
        ctr = self.center
        ring = None
        if pre_L1_fea is None:
            l1 = self._features(x.reshape(-1, C, H, W), pms.reshape(-1, C, H, W))
            if self.feature_ring:
                ring = FeatureRing(l1, B, N)
        elif getattr(pre_L1_fea, "_cdfo_ring", None) is not None:
            ring, serial = pre_L1_fea._cdfo_ring
            if serial != ring.serial or ring.B != B or tuple(ring.buf.shape[3:]) != (H, W):
                raise hotpath._lib.CdfoError("CVSR_V8: stale or mismatched feature-ring handle (pass the L1_fea of the previous step)")
            ring.push(self._features(x[:, -1], pms[:, -1]))
        else:
            new = self._features(x[:, -1], pms[:, -1])
            l1 = torch.cat([pre_L1_fea.view(B, N, -1, H, W)[:, 1:], new.unsqueeze(1)], 1).reshape(B * N, -1, H, W)
        if ring is not None:
            win = ring.window()                                                      # [N, B, 64, H, W], frame-major
            l1 = ring.handle()
            center = win[ctr]
            fea_nb = (win[:ctr].reshape(ctr * B, -1, H, W), win[ctr + 1:].reshape((N - 1 - ctr) * B, -1, H, W))   # two contiguous views
        else:
            fea = l1.view(B, N, -1, H, W)
        if ufs.shape[1] != N:  # reference accepts [B,1,N,H,W] as well (arch:4434-4437)
            ufs, rms = ufs.transpose(1, 2), rms.transpose(1, 2)
        if noise is None:
            noise = [torch.rand((B, 64, H, W), device=x.device, generator=self.noise_generator).clamp_min_(1e-12)
                     for _ in _NB]
        # neighbour-major batch of 6*B: index n*B + b (slices + cat: a list index would build a CPU index tensor, i.e. a
        # host-to-device copy per call, which also cannot be captured in a CUDA graph)
        def neighbours(t):
            return torch.cat([t[:, :ctr], t[:, ctr + 1:]], 1).transpose(0, 1)
        if ring is None:
            fea_nb = neighbours(fea).reshape(6 * B, -1, H, W)
            center = fea[:, ctr]
        ufs_nb = neighbours(ufs).reshape(6 * B, 1, H, W)
        rms_nb = neighbours(rms).reshape(6 * B, 1, H, W)
        mv_nb = neighbours(mvs1).reshape(6 * B, 2, H, W).contiguous()
        if torch.is_tensor(noise):       # already neighbour-major [6 * B, 64, H, W]
            u_nb = noise
        else:
            u_nb = torch.cat([u.to(x.device, torch.float32) for u in noise], 0)
        fused8 = hotpath.align_and_fuse(self, center, fea_nb, ufs_nb, rms_nb, mv_nb, u_nb, B)   # c8 bf16 [B,8,H,W,8]
        t = self._trunk(fused8)
        out = hotpath.tail(self, t, x[:, ctr])
        return out, l1
