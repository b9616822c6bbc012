"""Feature extraction of CVSR_V8 (conv_first / conv_second + PAItransformerSA_2, arch/SIDECVSR_our.py:4416-4419, :1441-1475, :1643-1653)
on the device in c8 bf16: the 64-channel 1x1 / 3x3 convolutions on the tcgen05 kernel (csrc/conv3x3_sm100.cu), everything else in
csrc/features_c8.cu.  No cuDNN / cuBLAS / ATen kernel in the steady state, every reduction in a fixed order (bit-identical reruns).

    l1 = lrelu(conv_first(x));  s = conv_second(pms)
    x2 = side(s) + l1
    3 x:  [x2 = side(x2) + x2]   x1 = x1 + attn(norm1(x1))   x1 = x1 + conv(norm2(x1)) + x2          (arch:1455-1475)
side = the 16-channel branch side_to_feaoneUDSA_2 (arch:1815-1832): 3x3 64->16, two stride-2 convolutions, the 7x7 spatial gate, two
stride-2 transposed convolutions, 3x3 16->64, each followed by lrelu 0.1.
"""
import torch

from . import _lib, conv

_zero_pad = {}      # (device, B, H, W) -> c8 [B, 8, H, W, 8] whose channels 16.. stay zero (input of the 16 -> 64 convolution)


def _f32(t):
    return t.detach().contiguous().float()


def _padded_ci(weight):
    """[Co, 16, 3, 3] -> [Co, 64, 3, 3] with zero input channels 16..63: the tcgen05 kernel takes multiples of 64 input channels."""
    def build(w):
        out = torch.zeros((w.size(0), 64, 3, 3), dtype=torch.float32, device=w.device)
        out[:, :w.size(1)] = w.float()
        return out
    return conv.derived(weight, "ci64", build)


def prior_conv_c8(mod, x, lrelu):
    """Conv2d(1, 64, 3, 1, 1) on [B, 1, H, W] fp32 -> c8 bf16 [B, 8, H, W, 8]."""
    B, C, H, W = x.shape
    if C != 1:
        raise _lib.CdfoError("prior_conv_c8: one-channel input expected")
    x = _f32(x)
    Co = mod.weight.size(0)
    y = torch.empty((B, Co // 8, H, W, 8), dtype=torch.bfloat16, device=x.device)
    _lib.call("cdfo_prior_conv_c8_fwd", _lib.ptr(x), _lib.ptr(_f32(mod.weight)), _lib.ptr(_f32(mod.bias)), _lib.ptr(y), B, Co, H, W, int(bool(lrelu)),
              _lib.stream_ptr(x.device))
    return y


def layernorm_c8(norm, x8, eps=1e-5):
    import ctypes
    B, _, H, W, _ = x8.shape
    y = torch.empty_like(x8)
    _lib.call("cdfo_layernorm_c8_fwd", _lib.ptr(x8), _lib.ptr(_f32(norm.body.weight)), _lib.ptr(_f32(norm.body.bias)), _lib.ptr(y), B, H, W,
              ctypes.c_float(eps), _lib.stream_ptr(x8.device))
    return y


def side_branch_c8(side, s8, resid8):
    """lrelu(body.11(...)) + resid8 for a c8 bf16 [B, 8, H, W, 8] input: six convolutions + the spatial gate, 8 launches.  H and W must be
    multiples of 4: the two stride-2 convolutions take H to H / 2 + 1 and H / 4 + 2, and the transposed ones bring only those sizes back
    to H (a side of 10 would come back as 8)."""
    b = side.body._modules
    B, _, H, W, _ = s8.shape
    if H < 4 or W < 4 or H % 4 or W % 4:
        raise _lib.CdfoError("side_branch_c8: H and W must be multiples of 4, at least 4 (got %d x %d)" % (H, W))
    dev = s8.device
    st = _lib.stream_ptr(dev)
    t = conv.conv3x3(s8, b["0"].weight, b["0"].bias, conv.ACT_LRELU)                         # [B, 2, H, W, 8]
    H1, W1 = (H + 1) // 2 + 1, (W + 1) // 2 + 1
    H2, W2 = (H1 + 1) // 2 + 1, (W1 + 1) // 2 + 1

    def c16(x8, mod, Hi, Wi, Ho, Wo, transposed, out=None):
        y = torch.empty((B, 2, Ho, Wo, 8), dtype=torch.bfloat16, device=dev) if out is None else out
        _lib.call("cdfo_conv16_c8_fwd", _lib.ptr(x8), _lib.ptr(_f32(mod.weight)), _lib.ptr(_f32(mod.bias)), _lib.ptr(y), B, Hi, Wi, Ho, Wo,
                  int(y.size(1)) * 8, int(transposed), st)
        return y
    t = c16(t, b["2"], H, W, H1, W1, 0)
    t = c16(t, b["4"], H1, W1, H2, W2, 0)
    gate = b["6"].spatial
    pooled = torch.empty((B, H2, W2, 2), dtype=torch.float32, device=dev)
    g = torch.empty_like(t)
    _lib.call("cdfo_spatial_gate_c8_fwd", _lib.ptr(t), _lib.ptr(_f32(gate.weight)), _lib.ptr(_f32(gate.bias)), _lib.ptr(pooled), _lib.ptr(g), B, H2,
              W2, st)
    t = c16(g, b["7"], H2, W2, H1, W1, 1)
    key = (str(dev), B, H, W)
    pad = _zero_pad.get(key)
    if pad is None:
        pad = _zero_pad[key] = torch.zeros((B, 8, H, W, 8), dtype=torch.bfloat16, device=dev)
    c16(t, b["9"], H1, W1, H, W, 1, out=pad)                                                   # writes channels 0..15; 16..63 stay zero
    return conv.conv3x3(pad, _padded_ci(b["11"].weight), b["11"].bias, conv.ACT_LRELU, resid8=resid8)


def self_mdta_c8(attn, n8, x1, x2=None, parts=32):
    """x1 + attn(n8) [and that + x2]: qkv 1x1 -> depthwise 3x3 -> per-head Gram -> folded 64x64 matrix -> apply (arch:1545-1576)."""
    B, _, H, W, _ = n8.shape
    dev = n8.device
    st = _lib.stream_ptr(dev)
    qkv = conv.conv3x3(n8, attn.qkv.weight, None, conv.ACT_NONE)                               # 1x1, 64 -> 192: [B, 24, H, W, 8]
    dw = torch.empty_like(qkv)
    _lib.call("cdfo_dwconv3x3_c8_fwd", _lib.ptr(qkv), _lib.ptr(_f32(attn.qkv_dwconv.weight).reshape(192, 9)), _lib.ptr(dw), B, 192, H, W, st)
    # 32 pixel ranges per (sample, head): ~16 pixels per thread, so the 80-value block reduction of the Gram kernel is amortised
    parts = max(1, min(parts, (H * W + 255) // 256))
    partial = torch.empty((B, parts, 640), dtype=torch.float32, device=dev)
    _lib.call("cdfo_mdta_gram_c8_fwd", _lib.ptr(dw), _lib.ptr(partial), B, 192, H, W, parts, st)
    M = torch.empty((B, 64, 64), dtype=torch.float32, device=dev)
    _lib.call("cdfo_mdta_fold_fwd", _lib.ptr(partial), _lib.ptr(_f32(attn.temperature).reshape(-1)), _lib.ptr(_f32(attn.project_out.weight).reshape(64, 64)),
              _lib.ptr(M), B, parts, st)
    out1 = torch.empty_like(x1)
    out2 = None if x2 is None else torch.empty_like(x1)
    _lib.call("cdfo_mdta_apply_c8_fwd", _lib.ptr(dw), 192, 128, _lib.ptr(M), _lib.ptr(x1), _lib.ptr(x2), _lib.ptr(out1), _lib.ptr(out2), B, H, W, st)
    return out1, out2


@torch.no_grad()
def feature_extraction_c8(model, x, pms):
    """x, pms [n, 1, H, W] fp32 -> L1 features as c8 bf16 [n, 8, H, W, 8]."""
    path = model.transformer_feature_extraction.path1
    side = path.side_to_feaoneUDSA
    x1 = prior_conv_c8(model.conv_first, x, lrelu=True)
    s = prior_conv_c8(model.conv_second, pms, lrelu=False)
    x2 = side_branch_c8(side, s, x1)                                   # side(s) + l1
    for it in range(3):
        if it:
            x2 = side_branch_c8(side, x2, x2)                          # side(x2) + x2
        a, t = self_mdta_c8(path.attn, layernorm_c8(path.norm1, x1), x1, x2)        # a = x1 + attn;  t = a + x2
        n2 = layernorm_c8(path.norm2, a)
        x1 = conv.conv3x3(n2, path.conv.weight, path.conv.bias, conv.ACT_NONE, resid8=t)   # conv(norm2(a)) + a + x2
    return x1
