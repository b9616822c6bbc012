"""Host side of the tcgen05 3x3 convolution (cdfo_conv3x3_sm100_fwd) and of the c8 layout adapters."""
import torch

from . import _lib, config

ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2
_wcache = _lib.TensorCache()


@torch.no_grad()
def to_c8(x: torch.Tensor, out: torch.Tensor = None, channel0: int = 0) -> torch.Tensor:
    """NCHW fp32 -> [B, C/8, H, W, 8] bf16; with `out` ([B, Cout/8, H, W, 8], contiguous) into its channels [channel0, channel0 + C)."""
    B, C, H, W = x.shape
    x = x.contiguous().float()
    if out is None:
        out = torch.empty((B, C // 8, H, W, 8), dtype=torch.bfloat16, device=x.device)
        _lib.call("cdfo_pack_c8", _lib.ptr(x), _lib.ptr(out), B, C, H, W, _lib.stream_ptr(x.device))
        return out
    if out.dtype != torch.bfloat16 or not out.is_contiguous() or out.dim() != 5 or (out.size(0), out.size(2), out.size(3), out.size(4)) != (B, H, W, 8):
        raise _lib.CdfoError("to_c8: out must be a contiguous bf16 c8 tensor of the same batch and size")
    _lib.call("cdfo_pack_c8_into", _lib.ptr(x), _lib.ptr(out), B, C, H, W, out.size(1) * 8, int(channel0), _lib.stream_ptr(x.device))
    return out


@torch.no_grad()
def from_c8(x8: torch.Tensor) -> torch.Tensor:
    """[B, C/8, H, W, 8] bf16 -> NCHW fp32."""
    B, C8, H, W, _ = x8.shape
    out = torch.empty((B, C8 * 8, H, W), dtype=torch.float32, device=x8.device)
    _lib.call("cdfo_unpack_c8", _lib.ptr(x8), _lib.ptr(out), B, C8 * 8, H, W, _lib.stream_ptr(x8.device))
    return out


@torch.no_grad()
def pack_weight(weight: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, k, k] (k = 1 or 3) -> packed bf16 B operand (cached per parameter / version)."""
    return _wcache.get(weight, lambda: _pack_weight(weight))


def _pack_weight(weight):
    Cout, Cin, ks = weight.shape[:3]
    if ks not in (1, 3) or weight.shape[3] != ks:
        raise _lib.CdfoError("conv_sm100: kernel size 1 or 3 expected, got %s" % (tuple(weight.shape[2:]),))
    nbytes = _lib.lib().cdfo_conv_sm100_weight_bytes(Cout, Cin, ks)
    if nbytes == 0 or Cin % 64 or Cout % 16:
        raise _lib.CdfoError("conv_sm100: unsupported channels %d -> %d" % (Cin, Cout))
    w = weight.detach().contiguous().float()
    out = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=w.device)
    _lib.call("cdfo_conv_sm100_pack_weight", _lib.ptr(w), _lib.ptr(out), Cout, Cin, int(ks), _lib.stream_ptr(w.device))
    return out


_wcache_pair = _lib.TensorCache()


@torch.no_grad()
def pack_weight_pair(weight: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> the CTA-pair kernel's B operand [2 halves][9][Cin/8][Cout/2][8] bf16 (cached per parameter / version)."""
    return _wcache_pair.get(weight, lambda: _pack_weight_pair(weight))


def _pack_weight_pair(weight):
    Cout, Cin = weight.shape[:2]
    nbytes = _lib.lib().cdfo_conv3x3_pair_sm100_weight_bytes(Cout, Cin)
    if nbytes == 0:
        raise _lib.CdfoError("conv3x3 (CTA pair): unsupported channels %d -> %d" % (Cin, Cout))
    w = weight.detach().contiguous().float()
    out = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=w.device)
    _lib.call("cdfo_conv3x3_pair_sm100_pack_weight", _lib.ptr(w), _lib.ptr(out), Cout, Cin, _lib.stream_ptr(w.device))
    return out


_wcache_4x4 = _lib.TensorCache()


@torch.no_grad()
def conv3x3_then_half(x8, weight, bias=None, resid8=None, up8=None, want_half=False):
    """bilinear_x0.5(conv3x3(x8, weight) + bias) + resid8 as ONE 4x4 / stride-2 convolution on a CTA pair (cdfo_conv4x4s2_pair_sm100_fwd).
    x8 [B, Cin/8, 2H, 2W, 8] bf16 -- or its parity planes [B, Cin/8, 2, 2, H, W, 8] as conv3x3(..., parity_planes=True) writes them
    (dense TMA boxes instead of stride-2 loads) -- weight [64, Cin, 3, 3] -> [B, 8, H, W, 8] bf16; resid8 at the output size.
    up8 [B, 8, H/2, W/2, 8]: its bilinear x2 is added in the epilogue; want_half: also returns bilinear_x0.5 of the result
    [B, 8, H/2, W/2, 8] (taken from the fp32 values) -- the two resampling passes that close / open a cross-scale block."""
    planes = x8.dim() == 7
    if planes:
        B, C8, _, _, Ho, Wo, _ = x8.shape
        Hi, Wi = 2 * Ho, 2 * Wo
        if tuple(x8.shape[2:4]) != (2, 2):
            raise _lib.CdfoError("conv3x3_then_half: parity planes must be [B, Cin/8, 2, 2, H, W, 8]")
    else:
        B, C8, Hi, Wi, _ = x8.shape
    Cout, Cin = weight.shape[:2]
    if C8 * 8 != Cin or tuple(weight.shape[2:]) != (3, 3) or not _lib.lib().cdfo_conv4x4s2_pair_sm100_supported(Cout, Cin) or Hi % 2 or Wi % 2:
        raise _lib.CdfoError("conv3x3_then_half: unsupported shape %s on %s" % (tuple(weight.shape), tuple(x8.shape)))
    if x8.dtype != torch.bfloat16 or not x8.is_contiguous():
        raise _lib.CdfoError("conv3x3_then_half: input must be a contiguous bf16 c8 tensor")
    def pack():
        w = weight.detach().contiguous().float()
        out = torch.empty(_lib.lib().cdfo_conv4x4s2_pair_sm100_weight_bytes(Cin) // 2, dtype=torch.bfloat16, device=w.device)
        _lib.call("cdfo_conv4x4s2_pair_sm100_pack_weight", _lib.ptr(w), _lib.ptr(out), Cin, _lib.stream_ptr(w.device))
        return out
    wpk = _wcache_4x4.get(weight, pack)
    y = torch.empty((B, Cout // 8, Hi // 2, Wi // 2, 8), dtype=torch.bfloat16, device=x8.device)
    if resid8 is not None and (tuple(resid8.shape) != tuple(y.shape) or resid8.dtype != torch.bfloat16 or not resid8.is_contiguous()):
        raise _lib.CdfoError("conv3x3_then_half: residual must be a contiguous bf16 c8 tensor of the output shape")
    b = None if bias is None else bias.detach().contiguous().float()
    half = None
    if up8 is not None or want_half:
        hs = (B, Cout // 8, Hi // 4, Wi // 4, 8)
        if Hi % 4 or Wi % 4 or (up8 is not None and (tuple(up8.shape) != hs or up8.dtype != torch.bfloat16 or not up8.is_contiguous())):
            raise _lib.CdfoError("conv3x3_then_half: up8 must be a contiguous bf16 c8 tensor of half the output size (output size even)")
        if want_half:
            half = torch.empty(hs, dtype=torch.bfloat16, device=x8.device)
    _lib.call("cdfo_conv4x4s2_pair_sm100_block_fwd", _lib.ptr(x8), _lib.ptr(wpk), _lib.ptr(b), _lib.ptr(resid8), _lib.ptr(up8), _lib.ptr(y),
              _lib.ptr(half), B, Cin, Hi, Wi, 1 if planes else 0, _lib.stream_ptr(x8.device))
    return (y, half) if want_half else y


_derived = _lib.TensorCache()


@torch.no_grad()
def derived(param, kind, fn):
    """fn(param) cached per (parameter, version, kind): weights re-laid-out for a kernel (PixelShuffle channel
    order, padded output channels, composed 1x1 o 3x3 ...).  The result then has its own pack_weight entry."""
    return _derived.get(param, lambda: fn(param.detach()), kind)


def centre_tap(w):
    """[Cout, Cin, 1, 1] -> [Cout, Cin, 3, 3] with the 1x1 weight at the centre tap."""
    out = torch.zeros((w.size(0), w.size(1), 3, 3), dtype=torch.float32, device=w.device)
    out[:, :, 1, 1] = w.float().reshape(w.size(0), w.size(1))
    return out


def ps_order(t):
    """Rows of a weight / bias reordered for the pixel-shuffle epilogue: new row (2i+j)*(Cout/4) + c <- row 4c + 2i + j."""
    cout = t.size(0)
    c = torch.arange(cout // 4, device=t.device)
    idx = torch.cat([4 * c + q for q in range(4)])
    return t.index_select(0, idx).contiguous()


@torch.no_grad()
def conv3x3(x8, weight, bias=None, act=ACT_NONE, resid8=None, out_nchw=False, pixel_shuffle=False, parity_planes=False, bias_edge=None):
    """Convolution with a [Cout, Cin, k, k] weight, k = 1 or 3, stride 1, "same" padding, on the tcgen05 kernel.
    x8 [B, Cin/8, H, W, 8] bf16 -> [B, Cout/8, H, W, 8] bf16 (or [B, Cout, H, W] fp32 when out_nchw, or
    [B, Cout/32, 2H, 2W, 8] bf16 = PixelShuffle(2) when pixel_shuffle and the weight rows are in ps_order, or the four parity
    planes [B, Cout/8, 2, 2, H/2, W/2, 8] when parity_planes: CTA-pair shapes only, the input layout of conv3x3_then_half).
    bias_edge [9, Cout] fp32: per-class bias of the border pixels (cdfo_conv3x3_pair_sm100_edge_fwd; CTA-pair shapes only)."""
    B, C8, H, W, _ = x8.shape
    Cout, Cin, ks = weight.shape[:3]
    if C8 * 8 != Cin or ks not in (1, 3) or weight.shape[3] != ks:
        raise _lib.CdfoError("conv3x3: weight %s does not match input with %d channels" % (tuple(weight.shape), C8 * 8))
    if x8.dtype != torch.bfloat16 or not x8.is_contiguous():
        raise _lib.CdfoError("conv3x3: input must be a contiguous bf16 c8 tensor")
    b = None if bias is None else bias.detach().contiguous().float()
    if resid8 is not None and (resid8.shape != (B, Cout // 8, H, W, 8) or resid8.dtype != torch.bfloat16 or not resid8.is_contiguous()):
        raise _lib.CdfoError("conv3x3: residual must be a contiguous bf16 c8 tensor of the output shape")
    # 64 -> 64 has one K block per tile: the single-SM kernel is faster there (795 vs 621 TFLOP/s); parity_planes forces the pair kernel
    pair_shape = _lib.lib().cdfo_conv3x3_pair_sm100_supported(Cout, Cin) and (parity_planes or not (Cin == 64 and Cout == 64))
    pair_ok = ks == 3 and not pixel_shuffle and not out_nchw and pair_shape
    if bias_edge is not None:
        if not (config.conv_pair and pair_ok) or b is None or tuple(bias_edge.shape) != (9, Cout) or bias_edge.dtype != torch.float32 \
                or not bias_edge.is_contiguous() or H < 2 or W < 2:
            raise _lib.CdfoError("conv3x3: bias_edge needs a CTA-pair shape, a bias and a contiguous fp32 [9, %d] table" % Cout)
        if parity_planes and (resid8 is not None or H % 2 or W % 2):
            raise _lib.CdfoError("conv3x3: parity_planes needs an even size and no residual")
        shape = (B, Cout // 8, 2, 2, H // 2, W // 2, 8) if parity_planes else (B, Cout // 8, H, W, 8)
        y = torch.empty(shape, dtype=torch.bfloat16, device=x8.device)
        _lib.call("cdfo_conv3x3_pair_sm100_edge_fwd", _lib.ptr(x8), _lib.ptr(pack_weight_pair(weight)), _lib.ptr(b), _lib.ptr(bias_edge),
                  _lib.ptr(resid8), _lib.ptr(y), B, Cin, Cout, H, W, int(act), 1 if parity_planes else 0, _lib.stream_ptr(x8.device))
        return y
    if parity_planes:
        if not pair_ok or resid8 is not None or H % 2 or W % 2:
            raise _lib.CdfoError("conv3x3: parity_planes needs a CTA-pair shape (3x3, %d -> %d), an even size and no residual" % (Cin, Cout))
        y = torch.empty((B, Cout // 8, 2, 2, H // 2, W // 2, 8), dtype=torch.bfloat16, device=x8.device)
        _lib.call("cdfo_conv3x3_pair_sm100_planes_fwd", _lib.ptr(x8), _lib.ptr(pack_weight_pair(weight)), _lib.ptr(b), _lib.ptr(None),
                  _lib.ptr(y), B, Cin, Cout, H, W, int(act), 1, _lib.stream_ptr(x8.device))
        return y
    if config.conv_pair and out_nchw and ks == 3 and not pixel_shuffle and resid8 is None and pair_shape:
        y = torch.empty((B, Cout, H, W), dtype=torch.float32, device=x8.device)
        _lib.call("cdfo_conv3x3_pair_sm100_planes_fwd", _lib.ptr(x8), _lib.ptr(pack_weight_pair(weight)), _lib.ptr(b), _lib.ptr(None),
                  _lib.ptr(y), B, Cin, Cout, H, W, int(act), 2, _lib.stream_ptr(x8.device))
        return y
    if config.conv_pair and pair_ok:
        y = torch.empty((B, Cout // 8, H, W, 8), dtype=torch.bfloat16, device=x8.device)
        _lib.call("cdfo_conv3x3_pair_sm100_fwd", _lib.ptr(x8), _lib.ptr(pack_weight_pair(weight)), _lib.ptr(b), _lib.ptr(resid8),
                  _lib.ptr(y), B, Cin, Cout, H, W, int(act), _lib.stream_ptr(x8.device))
        return y
    wpk = pack_weight(weight)
    if pixel_shuffle:
        y = torch.empty((B, Cout // 32, 2 * H, 2 * W, 8), dtype=torch.bfloat16, device=x8.device)
    elif out_nchw:
        y = torch.empty((B, Cout, H, W), dtype=torch.float32, device=x8.device)
    else:
        y = torch.empty((B, Cout // 8, H, W, 8), dtype=torch.bfloat16, device=x8.device)
    _lib.call("cdfo_conv_sm100_fwd", _lib.ptr(x8), _lib.ptr(wpk), _lib.ptr(b), _lib.ptr(resid8), _lib.ptr(y),
              B, Cin, Cout, H, W, int(ks), int(act), 2 if pixel_shuffle else (0 if out_nchw else 1), _lib.stream_ptr(x8.device))
    return y


@torch.no_grad()
def conv3x3_up2(x8, weight, bias, act=ACT_NONE, parity_planes=False, bias_edge=None):
    """conv3x3(resample(x8, 1), weight, bias, act, parity_planes=..., bias_edge=...) bit for bit, with the bilinear x2 evaluated while the
    convolution's A operand is built: x8 [B, 8, H, W, 8] bf16 (the 1x image), weight [256, 64, 3, 3] -> [B, 32, 2H, 2W, 8] bf16 (or its
    parity planes [B, 32, 2, 2, H, W, 8]); bias_edge [9, 256] fp32 as in conv3x3."""
    B, C8, H, W, _ = x8.shape
    Cout, Cin = weight.shape[:2]
    if C8 * 8 != Cin or (Cout, Cin) != (256, 64) or tuple(weight.shape[2:]) != (3, 3):
        raise _lib.CdfoError("conv3x3_up2: 64 -> 256 3x3 only, got weight %s on input %s" % (tuple(weight.shape), tuple(x8.shape)))
    if x8.dtype != torch.bfloat16 or not x8.is_contiguous():
        raise _lib.CdfoError("conv3x3_up2: input must be a contiguous bf16 c8 tensor")
    b = None if bias is None else bias.detach().contiguous().float()
    if bias_edge is not None and (b is None or tuple(bias_edge.shape) != (9, Cout) or bias_edge.dtype != torch.float32
                                  or not bias_edge.is_contiguous()):
        raise _lib.CdfoError("conv3x3_up2: bias_edge needs a bias and a contiguous fp32 [9, %d] table" % Cout)
    shape = (B, Cout // 8, 2, 2, H, W, 8) if parity_planes else (B, Cout // 8, 2 * H, 2 * W, 8)
    y = torch.empty(shape, dtype=torch.bfloat16, device=x8.device)
    _lib.call("cdfo_conv3x3_pair_sm100_up2_fwd", _lib.ptr(x8), _lib.ptr(pack_weight_pair(weight)), _lib.ptr(b), _lib.ptr(bias_edge), _lib.ptr(y),
              B, Cin, Cout, 2 * H, 2 * W, int(act), 1 if parity_planes else 0, _lib.stream_ptr(x8.device))
    return y


@torch.no_grad()
def conv_last_skip(x8, weight, bias, lr):
    """conv_last (Cin -> 1, 3x3) + bias + bilinear x4 skip of the 1-channel LR image lr [B,1,H/4,W/4] (arch:4477-4480).
    x8 [B, Cin/8, H, W, 8] bf16 -> [B, 1, H, W] fp32."""
    B, C8, H, W, _ = x8.shape
    w16 = derived(weight, "pad16", lambda w: torch.cat([w.float(), torch.zeros((15,) + tuple(w.shape[1:]), device=w.device)], 0).contiguous())
    wpk = pack_weight(w16)
    y = torch.empty((B, 1, H, W), dtype=torch.float32, device=x8.device)
    b = bias.detach().float().contiguous()
    lr = lr.contiguous().float()
    if lr.shape != (B, 1, H // 4, W // 4):
        raise _lib.CdfoError("conv_last_skip: LR image %s does not match the %dx%d output" % (tuple(lr.shape), H, W))
    _lib.call("cdfo_conv_last_skip_sm100_fwd", _lib.ptr(x8), _lib.ptr(wpk), _lib.ptr(b), _lib.ptr(lr), _lib.ptr(y), B, C8 * 8, H, W,
              _lib.stream_ptr(x8.device))
    return y


@torch.no_grad()
def resample(a, mode, b=None, base=None):
    """c8 bf16 bilinear resampling (align_corners=False): mode 0 = x0.5 of a, 1 = x2 of a, 2 = base + x0.5(a) + x2(b),
    3 = base + x2(b) (a is ignored)."""
    if mode == 3:
        B, C8, Ho, Wo, _ = base.shape
        if tuple(b.shape) != (B, C8, Ho // 2, Wo // 2, 8) or Ho % 2 or Wo % 2 or not base.is_contiguous() or not b.is_contiguous() \
                or base.dtype != torch.bfloat16 or b.dtype != torch.bfloat16:
            raise _lib.CdfoError("resample: base / b shapes do not match")
        y = torch.empty_like(base)
        _lib.call("cdfo_resample_c8", _lib.ptr(None), _lib.ptr(b), _lib.ptr(base), _lib.ptr(y), B, C8 * 8, Ho, Wo, 3, _lib.stream_ptr(base.device))
        return y
    B, C8, Ha, Wa, _ = a.shape
    Ho, Wo = (Ha // 2, Wa // 2) if mode in (0, 2) else (2 * Ha, 2 * Wa)
    if a.dtype != torch.bfloat16 or not a.is_contiguous() or (mode != 1 and (Ha % 2 or Wa % 2)):
        raise _lib.CdfoError("resample: contiguous bf16 c8 input with even size expected")
    if mode == 2 and (tuple(base.shape) != (B, C8, Ho, Wo, 8) or tuple(b.shape) != (B, C8, Ho // 2, Wo // 2, 8)
                      or not base.is_contiguous() or not b.is_contiguous()):
        raise _lib.CdfoError("resample: base / b shapes do not match")
    y = torch.empty((B, C8, Ho, Wo, 8), dtype=torch.bfloat16, device=a.device)
    _lib.call("cdfo_resample_c8", _lib.ptr(a), _lib.ptr(b), _lib.ptr(base), _lib.ptr(y), B, C8 * 8, Ho, Wo, int(mode),
              _lib.stream_ptr(a.device))
    return y
