"""Execution of the hot-path modules of CVSR_V8 on the device.

Each function takes the parameter-holder module (cdfo_b200/model.py) plus activations and runs the path the
reference runs at the cited lines in the hand-written kernels of libcdfo_b200; DESIGN.md section 4 lists the ATen
copies that are left in a step (no cuDNN / cuBLAS launch).  Everything is CUDA-only.
"""
import ctypes

import torch
import torch.nn.functional as F

from . import _lib, config, conv, dcn_sm100


def _lrelu(x):
    return F.leaky_relu(x, 0.1)


def _c(mod, x, **kw):
    return F.conv2d(x, mod.weight, mod.bias, **kw)


def _pkey(*params):
    """Identity of a set of parameters for a derived-tensor cache: storage address, device and in-place version of each.  The cache
    itself hangs on the OWNING MODULE (never on id(): CPython reuses the addresses of freed objects, and every parameter of a
    freshly loaded checkpoint has the same _version), so it dies with the model and cannot be hit by another one."""
    return tuple((p.data_ptr(), str(p.device), p._version, p.dtype) for p in params)


def _module_cache(mod, slot, key, build):
    """mod.__dict__['_cdfo_derived'][slot] = (key, value); rebuilt when the key (see _pkey) changes -- load_state_dict, .to(device),
    optimizer steps.  A write through `.data` that keeps address and version is invisible: call clear_derived(model) after one."""
    store = mod.__dict__.setdefault("_cdfo_derived", {})
    hit = store.get(slot)
    if hit is not None and hit[0] == key:
        return hit[1]
    val = build()
    store[slot] = (key, val)
    return val


def clear_derived(model):
    """Drop every derived tensor (composed trunk weights, permuted head weights, LRA tables) cached on the modules of `model`."""
    for m in model.modules():
        m.__dict__.pop("_cdfo_derived", None)


# ------------------------------------------------------------------------------------------ MDTA (A4 / A5 shared)
def _f32(t):
    return t.detach().contiguous().float()


def _is_c8(t):
    return t.dim() == 5 and t.dtype == torch.bfloat16 and t.size(1) == 8 and t.size(4) == 8


def dual_mdta(mod, x, extra_feat, pred_feat, flow, mode):
    """warp + fusion_out + the two MDTA passes + project_out (arch:3304-3337 / :3456-3492) in csrc/mdta.cu.
    mode 0 (MVDualAttAlignment): returns c8 bf16 [2B, 8, H, W, 8] = cat([o1, o2], 0), the input of conv_offset.0.
    mode 1 (DualAttAlignment): returns (ReLU(fusion_out(cat[o1 + o2, x])) [B,64,H,W] fp32, per-part channel sums of it).
    `x` may hold fewer samples than the others (sample b uses x[b % x.size(0)]).
    Mode 0 also takes x, extra_feat and pred_feat as c8 bf16 [., 8, H, W, 8] (all three): cdfo_mdta_c8_fwd."""
    if mode == 0 and _is_c8(extra_feat):
        if not (_is_c8(x) and _is_c8(pred_feat)) or pred_feat.shape != extra_feat.shape or extra_feat.size(0) % x.size(0) \
                or x.shape[2:4] != extra_feat.shape[2:4]:
            raise _lib.CdfoError("dual_mdta: x, extra_feat and pred_feat must all be c8 bf16 tensors of one size")
        B, _, H, W, _ = extra_feat.shape
        x, extra_feat, pred_feat, flow = x.contiguous(), extra_feat.contiguous(), pred_feat.contiguous(), _f32(flow)
        dev = x.device
        du0, du2 = mod.conv_du._modules["0"], mod.conv_du._modules["2"]
        ws = torch.empty(_lib.lib().cdfo_mdta_workspace_bytes(B, H, W, mod.num_heads), dtype=torch.uint8, device=dev)
        out = torch.empty((2 * B, 8, H, W, 8), dtype=torch.bfloat16, device=dev)
        _lib.call("cdfo_mdta_c8_fwd", _lib.ptr(x), int(x.size(0)), _lib.ptr(extra_feat), _lib.ptr(pred_feat), _lib.ptr(flow),
                  _lib.ptr(_f32(mod.fusion_out.weight)), _lib.ptr(_f32(du0.weight)), _lib.ptr(_f32(du0.bias)), _lib.ptr(_f32(du2.weight)),
                  _lib.ptr(_f32(du2.bias)), _lib.ptr(_f32(mod.temperature)), _lib.ptr(_f32(mod.project_out.weight)), int(mod.num_heads),
                  _lib.ptr(out), _lib.ptr(ws), B, H, W, _lib.stream_ptr(dev))
        return out
    B, C, H, W = extra_feat.shape
    if C != 64 or x.size(1) != 64 or pred_feat.shape != extra_feat.shape or B % x.size(0):
        raise _lib.CdfoError("dual_mdta: 64-channel inputs of one size expected")
    heads = mod.num_heads
    fo = mod.fusion_out._modules["0"] if mode == 1 else mod.fusion_out
    du0, du2 = mod.conv_du._modules["0"], mod.conv_du._modules["2"]
    x, extra_feat, pred_feat, flow = _f32(x), _f32(extra_feat), _f32(pred_feat), _f32(flow)
    dev = x.device
    ws = torch.empty(_lib.lib().cdfo_mdta_workspace_bytes(B, H, W, heads), dtype=torch.uint8, device=dev)
    ca = None
    if mode == 0:
        out = torch.empty((2 * B, 8, H, W, 8), dtype=torch.bfloat16, device=dev)
    else:
        out = torch.empty((B, 64, H, W), dtype=torch.float32, device=dev)
        ca = torch.empty((B, _lib.lib().cdfo_mdta_parts(B), 64), dtype=torch.float32, device=dev)
    _lib.call("cdfo_mdta_fwd", _lib.ptr(x), int(x.size(0)), _lib.ptr(extra_feat), _lib.ptr(pred_feat), _lib.ptr(flow),
              _lib.ptr(_f32(fo.weight)), _lib.ptr(_f32(du0.weight)), _lib.ptr(_f32(du0.bias)), _lib.ptr(_f32(du2.weight)),
              _lib.ptr(_f32(du2.bias)), _lib.ptr(_f32(mod.temperature)), _lib.ptr(_f32(mod.project_out.weight)), int(heads),
              int(mode), _lib.ptr(out), _lib.ptr(ca), _lib.ptr(ws), B, H, W, _lib.stream_ptr(dev))
    return out if mode == 0 else (out, ca)


@torch.no_grad()
def dual_att_alignment(mod, x, extra_feat, pred_feat, flow):
    """DualAttAlignment.forward, arch:3455-3496 (flow [B,2,H,W]): MDTA kernels -> CALayer gate -> two residual
    blocks on the tcgen05 3x3 convolution (c8 bf16, residual adds in its epilogue) -> + x."""
    B, _, H, W = extra_feat.shape
    out, ca = dual_mdta(mod, x, extra_feat, pred_feat, flow, mode=1)
    dev = out.device
    c0, c2 = mod.CALayer.conv_du._modules["0"], mod.CALayer.conv_du._modules["2"]
    gate = torch.empty((B, 64), dtype=torch.float32, device=dev)
    _lib.call("cdfo_channel_gate_fwd", _lib.ptr(ca), int(ca.size(1)), _lib.ptr(_f32(c0.weight)), _lib.ptr(_f32(c0.bias)),
              _lib.ptr(_f32(c2.weight)), _lib.ptr(_f32(c2.bias)), _lib.ptr(gate), B, 64, int(c0.weight.size(0)), H * W,
              _lib.stream_ptr(dev))
    y8 = torch.empty((B, 8, H, W, 8), dtype=torch.bfloat16, device=dev)
    _lib.call("cdfo_pack_c8_scaled", _lib.ptr(out), _lib.ptr(gate), _lib.ptr(y8), B, 64, H, W, _lib.stream_ptr(dev))
    for rb in (mod.ResidualBlock, mod.ResidualBlock1):
        t = conv.conv3x3(y8, rb.conv1.weight, rb.conv1.bias, conv.ACT_RELU)
        y8 = conv.conv3x3(t, rb.conv2.weight, rb.conv2.bias, conv.ACT_NONE, resid8=y8)
    xf = _f32(x)
    res = torch.empty((B, 64, H, W), dtype=torch.float32, device=dev)
    _lib.call("cdfo_unpack_c8_add", _lib.ptr(y8), _lib.ptr(xf), int(xf.size(0)), _lib.ptr(res), B, 64, H, W, _lib.stream_ptr(dev))
    return res


def _expand_batch(x, B):
    """x [xB, ...] shared by B = k * xB samples (sample b uses x[b % xB])."""
    return x if x.size(0) == B else x.repeat(B // x.size(0), 1, 1, 1)


def _head_weights(c2, dg):
    """conv_offset[-1] with its output channels permuted into (dy, dx, m) triples in the order k' = tap*dg + g (reference
    channels 2k, 2k+1, dg*18 + k with k = g*9 + tap: the chunk/cat of arch:3341-3345), packed for the tcgen05 conv."""
    def build():
        kp = torch.arange(dg * 9, device=c2.weight.device)
        k = (kp % dg) * 9 + kp // dg
        perm = torch.stack([2 * k, 2 * k + 1, dg * 18 + k], dim=1).reshape(-1)
        w = c2.weight.detach().index_select(0, perm).contiguous()
        wpk = conv.pack_weight(w)
        bias = c2.bias.detach().index_select(0, perm).contiguous().float()
        return wpk, bias, w          # w keeps conv.pack_weight's weak reference alive
    out = _module_cache(c2, "head_%d" % dg, _pkey(c2.weight, c2.bias), build)
    return out[0], out[1]


def _head_weights_fused(c2, dg):
    """conv_offset[-1] permuted and packed for the fused head + DCN kernel (dcn_sm100.fused_head_permutation)."""
    def build():
        perm = dcn_sm100.fused_head_permutation(dg, c2.weight.device)
        w = c2.weight.detach().index_select(0, perm).contiguous()
        return conv.pack_weight(w), c2.bias.detach().index_select(0, perm).contiguous().float(), w
    out = _module_cache(c2, "head_fused_%d" % dg, _pkey(c2.weight, c2.bias), build)
    return out[0], out[1]


@torch.no_grad()
def mv_hidden_maps(mod, x, extra_feat, pred_feat, flow):
    """lrelu(conv_offset[0](o_k)) of the two MDTA outputs (arch:3304-3340, first layer of conv_offset): c8 bf16 [2B, 8, H, W, 8]."""
    c0 = mod.conv_offset._modules["0"]
    return conv.conv3x3(dual_mdta(mod, x, extra_feat, pred_feat, flow, mode=0), c0.weight, c0.bias, conv.ACT_LRELU)


@torch.no_grad()
def mv_offset_fields(mod, x, extra_feat, pred_feat, flow):
    """Learned offset residual and mask of MVDualAttAlignment WITHOUT the MV prior (arch:3339-3350 minus the
    `+ flow.flip(1).repeat(...)` term, which the DCN kernel adds itself), as packed fields
    [B, 9, dg/gp, H, W, gp, 4] fp16 = (10*tanh(dy1) + 10*tanh(dy2), same for dx, sigmoid(m1 + m2), 0) per (tap, pixel, group).
    Both conv_offset layers run in the tcgen05 convolution kernel; tanh / sum / sigmoid are its epilogue."""
    B = extra_feat.size(0)
    c0, c2 = mod.conv_offset._modules["0"], mod.conv_offset._modules["2"]
    z = mv_hidden_maps(mod, x, extra_feat, pred_feat, flow)   # [2B, 8, H, W, 8]
    H, W = z.shape[2:4]
    dg = mod.deformable_groups
    wpk, bias = _head_weights(c2, dg)
    fields = torch.empty(dcn_sm100.fields_shape(B, dg, H, W), dtype=torch.float16, device=z.device)
    args = (B, 64, dg, H, W, ctypes.c_float(float(mod.max_residue_magnitude)), _lib.stream_ptr(z.device))
    if config.head_dual:
        # both evaluations in one launch: the first stays in the epilogue's registers (bit-identical to the two-launch path)
        _lib.call("cdfo_mv_offset_head_dual_sm100_fwd", _lib.ptr(z), _lib.ptr(wpk), _lib.ptr(bias), _lib.ptr(fields), *args)
        return fields
    first = torch.empty_like(fields)
    _lib.call("cdfo_mv_offset_head_sm100_fwd", _lib.ptr(z[:B]), _lib.ptr(wpk), _lib.ptr(bias), _lib.ptr(None),
              _lib.ptr(first), *args)
    _lib.call("cdfo_mv_offset_head_sm100_fwd", _lib.ptr(z[B:]), _lib.ptr(wpk), _lib.ptr(bias), _lib.ptr(first),
              _lib.ptr(fields), *args)
    return fields


unpack_fields = dcn_sm100.unpack_fields   # (residual [B, dg*18, H, W], mask [B, dg*9, H, W]) in the reference's channel order


@torch.no_grad()
def mv_dual_att_alignment(mod, x, extra_feat, pred_feat, flow, stack=None, group_chunk=None, x8=None):
    """MVDualAttAlignment.forward, arch:3303-3352: DCN with offset = residual + decoded MV prior.
    `x` may hold fewer samples than the other arguments (sample b uses x[b % x.size(0)]): the model's six
    neighbour calls share the centre-frame feature (arch:4456).  With `stack` ([n_seq, chunks, H, W, 8] bf16) the DCN
    epilogue writes group g of the group-major batch into chunks [group_chunk[g], +8) of it and None is returned.
    extra_feat / pred_feat may be c8 bf16 (then x8 = the c8 copy of x is required: the MDTA kernels read c8, the DCN samples x)."""
    if config.dcn_gather == "tex" and config.fused_head_dcn and mod.deformable_groups == 16:
        # ONE kernel from the hidden maps to the aligned feature: the offset / mask fields stay on the SM
        z = mv_hidden_maps(mod, x8 if _is_c8(extra_feat) else x, extra_feat, pred_feat, flow)
        hw, hb = _head_weights_fused(mod.conv_offset._modules["2"], 16)
        return dcn_sm100.mv_head_dcn_fused(z, hw, hb, mod.max_residue_magnitude, dcn_sm100.pack_q4t(x), flow,
                                           dcn_sm100.pack_weight_f16(mod.weight), mod.bias, stack=stack, group_chunk=group_chunk)
    fields = mv_offset_fields(mod, x, extra_feat, pred_feat, flow)
    if config.dcn_gather == "tex":
        if stack is not None:
            return dcn_sm100.dcn_tex_stacked(dcn_sm100.pack_q4t(x), fields, dcn_sm100.pack_weight_f16(mod.weight), mod.bias, flow,
                                             stack, group_chunk)
        return dcn_sm100.dcn_tex(dcn_sm100.pack_q4t(x), fields, dcn_sm100.pack_weight_f16(mod.weight), mod.bias, mv=flow)
    xq = dcn_sm100.pack_q4p(x)
    return dcn_sm100.dcn_sm100(xq, None, None, dcn_sm100.pack_weight(mod.weight), mod.bias, mv=flow, fused_fields=fields)


# ------------------------------------------------------------------------------------------ A8
def _lra_tap_tables(mod):
    """kw[9], kh[9], K1[64], R[64,64] of csrc/lra.cu from directW1_conv / directH1_conv (cached on the module per weight version)."""
    def build():
        kw = mod.directW1_conv.weight.detach().reshape(9).double()
        kh = mod.directH1_conv.weight.detach().reshape(9).double()
        c = torch.arange(64, device=kw.device)
        tix = c.view(64, 1) - c.view(1, 64) + 4                 # tix[c_star][c] = tap index of a bump centred at c_star
        tapm = torch.where((tix >= 0) & (tix <= 8), kw[tix.clamp(0, 8)], torch.zeros((), dtype=kw.dtype, device=kw.device))
        k1 = tapm.sum(dim=1)                                     # K1[c_star]
        r = tapm @ tapm.t()                                      # R[c1][c2]
        tab = torch.cat([kw, kh, k1, r.reshape(-1)]).float().contiguous()
        # the two scalar biases are read back ONCE per weight version (a .item() per call would be a host sync per step and
        # would make the step impossible to capture in a CUDA graph)
        return tab, float(mod.directW1_conv.bias.detach()), float(mod.directH1_conv.bias.detach())
    return _module_cache(mod, "lra_tables", _pkey(mod.directW1_conv.weight, mod.directH1_conv.weight, mod.directW1_conv.bias,
                                                   mod.directH1_conv.bias), build)


@torch.no_grad()
def mask_logits(mod, v):
    """v_max [B, 64] = ReLU(conv_du_re2(mean ReLU(conv_du_re.2(v)))) (arch:2183-2186) from v = ReLU(conv_du_re.0(res)) [B, 64, H, W] fp32:
    the stride-2 convolution on the tensor cores with ReLU + spatial sum in its epilogue, then the pooled 64 x 64 product (csrc/lra_mask_logits.cu)."""
    B, C, H, W = v.shape
    if C != 64:
        raise _lib.CdfoError("mask_logits: 64 channels expected")
    c2, c3 = mod.conv_du_re._modules["2"], mod.conv_du_re2._modules["0"]
    ws = torch.empty(_lib.lib().cdfo_lra_mask_logits_workspace_bytes(B, H, W), dtype=torch.uint8, device=v.device)
    vmax = torch.empty((B, 64), dtype=torch.float32, device=v.device)
    _lib.call("cdfo_lra_mask_logits_fwd", _lib.ptr(_f32(v)), _lib.ptr(_f32(c2.weight)), _lib.ptr(_f32(c2.bias)), _lib.ptr(_f32(c3.weight).reshape(64, 64)),
              _lib.ptr(_f32(c3.bias)), _lib.ptr(vmax), _lib.ptr(ws), B, H, W, _lib.stream_ptr(v.device))
    return vmax


def _pointwise(in1, in2, weight, bias, act, mode=0, resid1=None, resid2=None):
    """cdfo_pointwise_conv_fwd: tensor-core 1x1 convolution on NCHW fp32 (mode 0: x = in1 + in2; mode 1: pixel-major cat)."""
    B, K, H, W = in1.shape
    Co = weight.size(0)
    out = torch.empty((B, Co, H, W), dtype=torch.float32, device=in1.device)
    _lib.call("cdfo_pointwise_conv_fwd", _lib.ptr(in1), _lib.ptr(in2), _lib.ptr(_f32(weight).reshape(Co, -1)), _lib.ptr(None if bias is None else _f32(bias)),
              _lib.ptr(resid1), _lib.ptr(resid2), _lib.ptr(out), B, K, Co, H, W, int(act), int(mode), _lib.stream_ptr(in1.device))
    return out


@torch.no_grad()
def long_range_attention(mod, res, x, u, x2=None, out8=None, channel0=0, res_prior=None):
    """LLongRangAttention.forward, arch:2179-2249, on the input x (+ x2: the model's `fea + rms_prior`, arch:4449, is formed
    inside the kernels and never written); u = uniform noise of gumbel_softmax (arch:2169).
    The 1x1 convolutions (conv_du_re.0, input_conv, fuse) are tensor-core pointwise kernels, the mask / row / column /
    window attentions csrc/lra.cu / csrc/lra_col_sm100.cu, the mask logits csrc/lra_mask_logits.cu: every launch is this library's.
    With out8 (contiguous bf16 c8 [B, C8, H, W, 8]) the result leaves as bf16 in its channels [channel0, channel0 + 64) instead of a
    new fp32 tensor (the fuse kernel's epilogue packs it).  res_prior = (conv module, one-channel map [B, 1, H, W]) says that res IS
    that prior convolution's output (the model: res = conv_expand_rms(rms), arch:4447): v = ReLU(conv_du_re.0(res)) is then one direct
    1 -> 64 convolution of the one-channel map with composed weights (`res` is not read for the mask logits)."""
    B, C, H, W = x.shape
    x = _f32(x)
    x2 = None if x2 is None else _f32(x2)
    du0 = mod.conv_du_re._modules["0"]
    if res_prior is not None:
        pc, rms1 = res_prior

        def build():
            w1 = du0.weight.detach().float().reshape(64, 64)
            return (w1 @ pc.weight.detach().float().reshape(64, 9)).contiguous(), (w1 @ pc.bias.detach().float() + du0.bias.detach().float()).contiguous()
        wv, bv = _module_cache(mod, "du0_after_prior", _pkey(du0.weight, du0.bias, pc.weight, pc.bias), build)
        rms1 = _f32(rms1)
        v = torch.empty((B, 64, H, W), dtype=torch.float32, device=x.device)
        _lib.call("cdfo_prior_conv_act_fwd", _lib.ptr(rms1), _lib.ptr(wv), _lib.ptr(bv), _lib.ptr(v), B, 64, H, W, 1, _lib.stream_ptr(x.device))
    else:
        v = _pointwise(_f32(res), None, du0.weight, du0.bias, act=1)
    vmax = mask_logits(mod, v)                                                          # bilinear up of a 1x1 map = broadcast
    qv = _pointwise(x, x2, mod.input_conv.weight, mod.input_conv.bias, act=0)
    nbytes = _lib.lib().cdfo_lra_workspace_bytes(B, H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    tab, beta, bh = _lra_tap_tables(mod)
    if out8 is not None:
        if out8.dtype != torch.bfloat16 or not out8.is_contiguous() or out8.dim() != 5 or (out8.size(0), out8.size(2), out8.size(3), out8.size(4)) != (B, H, W, 8):
            raise _lib.CdfoError("long_range_attention: out8 must be a contiguous bf16 c8 tensor of the same batch and size")
        _lib.call("cdfo_lra_c8_fwd", _lib.ptr(qv), _lib.ptr(u.contiguous()), _lib.ptr(vmax), _lib.ptr(x), _lib.ptr(x2), _lib.ptr(tab),
                  ctypes.c_float(beta), ctypes.c_float(bh),
                  _lib.ptr(_f32(mod.fuse.weight).reshape(64, 128)), _lib.ptr(_f32(mod.fuse.bias)),
                  _lib.ptr(out8), out8.size(1) * 8, int(channel0), _lib.ptr(ws), B, H, W, _lib.stream_ptr(x.device))
        return out8
    out = torch.empty_like(x)
    _lib.call("cdfo_lra_fwd", _lib.ptr(qv), _lib.ptr(u.contiguous()), _lib.ptr(vmax), _lib.ptr(x), _lib.ptr(x2), _lib.ptr(tab),
              ctypes.c_float(beta), ctypes.c_float(bh),
              _lib.ptr(_f32(mod.fuse.weight).reshape(64, 128)), _lib.ptr(_f32(mod.fuse.bias)),
              _lib.ptr(out), _lib.ptr(ws), B, H, W, _lib.stream_ptr(x.device))
    return out


# ------------------------------------------------------------------------------------------ model-level stages
@torch.no_grad()
def prior_conv(conv_mod, x):
    """conv_expand_ufs / conv_expand_rms (arch:4446-4447): Conv2d(1, 64, 3, 1, 1) on a one-channel prior map, fp32."""
    B, C, H, W = x.shape
    if C != 1:
        raise _lib.CdfoError("prior_conv: one-channel input expected")
    x = _f32(x)
    Co = conv_mod.weight.size(0)
    y = torch.empty((B, Co, H, W), dtype=torch.float32, device=x.device)
    _lib.call("cdfo_prior_conv_fwd", _lib.ptr(x), _lib.ptr(_f32(conv_mod.weight)), _lib.ptr(_f32(conv_mod.bias)), _lib.ptr(y), B, Co, H, W,
              _lib.stream_ptr(x.device))
    return y


_SLOT = (0, 1, 2, 4, 5, 6)   # frame slot of neighbour n in the stacked tensor (arch:4463: frames in temporal order)


@torch.no_grad()
def align_and_fuse(model, center, fea_nb, ufs_nb, rms_nb, mv_nb, u_nb, B):
    """Body of the reference's neighbour loop (arch:4445-4456) for all six neighbours at once (batch index n*B + b,
    `center` [B,64,H,W] shared by the six), then stack + tsa_fusion 1x1 + lrelu (arch:4463-4466).
    Returns the fused feature as c8 bf16 [B, 8, H, W, 8].  The 448-channel stack is written once, in bf16, directly by the
    DCN epilogue (O2) and read by the tcgen05 convolution kernel (kernel size 1)."""
    H, W = center.shape[2:]
    c8_align = (config.mdta_c8 and model.alignment == "mv_dcn" and config.dcn_gather == "tex" and config.fused_head_dcn
                and model.MV_deform_align.deformable_groups == 16)
    if c8_align:
        from . import features
        ufs_prior = features.prior_conv_c8(model.conv_expand_ufs, ufs_nb, lrelu=False)
    else:
        ufs_prior = prior_conv(model.conv_expand_ufs, ufs_nb)
    rms_prior = prior_conv(model.conv_expand_rms, rms_nb)
    # fea_nb: [6B, 64, H, W], or the contiguous runs of it (model.FeatureRing: frames 0-2 and 4-6); cat([fea, x_n]) (arch:4454) is
    # two packs into one c8 tensor
    runs = fea_nb if isinstance(fea_nb, (tuple, list)) else (fea_nb,)
    cat8 = torch.empty((6 * B, 16, H, W, 8), dtype=torch.bfloat16, device=center.device)
    off = 0
    for run in runs:
        sl = slice(off, off + run.size(0))
        long_range_attention(model.RDAB, rms_prior[sl], run, u_nb[sl], x2=rms_prior[sl], out8=cat8[sl], channel0=64,
                             res_prior=(model.conv_expand_rms, rms_nb[sl]) if config.lra_logits_from_prior else None)
        conv.to_c8(run, out=cat8[sl], channel0=0)
        off += run.size(0)
    fr = model.conv_expand_fea_r
    stack = torch.empty((B, 56, H, W, 8), dtype=torch.bfloat16, device=center.device)
    center8 = conv.to_c8(center)
    stack[:, 24:32] = center8
    al = model.MV_deform_align
    if c8_align:
        # the alignment's MDTA kernels read conv_expand_fea_r's c8 bf16 output, the c8 prior features and the packed centre feature as
        # they are (no fp32 NCHW copies of any of them)
        fea_i = conv.conv3x3(cat8, fr.weight, fr.bias, conv.ACT_NONE)
        mv_dual_att_alignment(al, center, fea_i, ufs_prior, mv_nb, stack=stack, group_chunk=[8 * f for f in _SLOT], x8=center8)
        return conv.conv3x3(stack, model.tsa_fusion.weight, model.tsa_fusion.bias, conv.ACT_LRELU)   # 1x1, 448 -> 64
    fea_i = conv.conv3x3(cat8, fr.weight, fr.bias, conv.ACT_NONE, out_nchw=True)
    if model.alignment == "mv_dcn" and config.dcn_gather == "tex":
        mv_dual_att_alignment(al, center, fea_i, ufs_prior, mv_nb, stack=stack, group_chunk=[8 * f for f in _SLOT])
    else:
        a8 = conv.to_c8(al(center, fea_i, ufs_prior, mv_nb)).view(6, B, 8, H, W, 8)
        for n, f in enumerate(_SLOT):
            stack[:, 8 * f:8 * f + 8] = a8[n]
    return conv.conv3x3(stack, model.tsa_fusion.weight, model.tsa_fusion.bias, conv.ACT_LRELU)   # 1x1, 448 -> 64


@torch.no_grad()
def tail(model, t, x_center):
    """arch:4473-4480 in three launches of the tcgen05 convolution: upconv1 + PixelShuffle + lrelu, upconv2 + PixelShuffle
    + lrelu (the shuffle is the store address of the epilogue; the 64-channel HR tensor exists once, in bf16), and
    conv_last + bias + bilinear x4 skip.  t: [B,64,H,W] fp32 or c8 bf16 [B,8,H,W,8]."""
    t8 = t if t.dim() == 5 else conv.to_c8(t)
    for up in (model.upconv1, model.upconv2):
        w = conv.derived(up.weight, "ps", lambda v: conv.ps_order(v.float()))
        b = conv.derived(up.bias, "ps", conv.ps_order)
        t8 = conv.conv3x3(t8, w, b, conv.ACT_LRELU, pixel_shuffle=True)
    return conv.conv_last_skip(t8, model.conv_last.weight, model.conv_last.bias, x_center)


# ------------------------------------------------------------------------------------------ reconstruction trunk (8f rank 1)
def _compose_1x1_after_3x3(w1, b1, w3, b3):
    """conv1x1(w1, b1) o conv3x3(w3, b3) == conv3x3(w, b): exact (the 1x1 comes after, no border effect)."""
    m = w1.float().reshape(w1.size(0), w1.size(1))
    w = torch.einsum("om,mikl->oikl", m, w3.float()).contiguous()
    b = m @ b3.float() + b1.float()
    return w, b


def _compose_3x3_after_1x1(w3, b3, w1, b1):
    """conv3x3(w3, b3, zero padding) o conv1x1(w1, b1) == conv3x3(w, .) with a bias that depends on the border class: the 1x1's bias is
    seen only by the taps that lie inside the frame.  Returns (w [O, I, 3, 3], interior bias [O], bias_edge [9, O]) with class =
    (row: top 0 / middle 1 / bottom 2) * 3 + (column: left 0 / middle 1 / right 2)."""
    m = w1.float().reshape(w1.size(0), w1.size(1))
    w = torch.einsum("omkl,mi->oikl", w3.float(), m).contiguous()
    tapb = torch.einsum("omkl,m->okl", w3.float(), b1.float())                  # [O, 3, 3]: the 1x1 bias through each tap
    rows = (slice(1, 3), slice(0, 3), slice(0, 2))                              # taps inside the frame for a top / middle / bottom row
    be = torch.stack([b3.float() + tapb[:, rows[r], rows[c]].sum(dim=(1, 2)) for r in range(3) for c in range(3)], 0).contiguous()
    return w, be[4].contiguous(), be


def _block_weights(blk):
    """Per cross-scale block: the 1x1 convs that FOLLOW a body, composed into the body's second 3x3, and the 1x1 convs that PRECEDE a
    body (they commute with the bilinear resampling), composed into the body's first 3x3 with a border-aware bias (cached on the block)."""
    b0, b2 = blk.body._modules["0"], blk.body._modules["2"]
    dn, up = blk.down._modules["0"], blk.up._modules["0"]

    def build():
        wu2, bu2 = _compose_1x1_after_3x3(up.weight.detach(), up.bias.detach(), b2.weight.detach(), b2.bias.detach())
        wd2, bd2 = _compose_1x1_after_3x3(dn.weight.detach(), dn.bias.detach(), b2.weight.detach(), b2.bias.detach())
        return {"up_body2": (wu2, bu2), "dn_body2": (wd2, bd2),
                "body0_dn": _compose_3x3_after_1x1(b0.weight.detach(), b0.bias.detach(), dn.weight.detach(), dn.bias.detach()),
                "body0_up": _compose_3x3_after_1x1(b0.weight.detach(), b0.bias.detach(), up.weight.detach(), up.bias.detach())}
    return _module_cache(blk, "composed", _pkey(b0.weight, b0.bias, b2.weight, b2.bias, dn.weight, dn.bias, up.weight, up.bias), build)


@torch.no_grad()
def cross_scale_block(blk, x8, x8_half=None, want_half=False):
    """Block_.forward, arch:401-406, on c8 bf16 [B, 8, H, W, 8] with H and W even and >= 4.  Bilinear x0.5 / x2 commute with the 1x1
    convs (per-pixel linear maps whose bias passes through weights that sum to 1), so each 1x1 of down / up is composed into the body's
    first 3x3 (border-class bias table) and the 1x1 that follows a body into the body's second 3x3:
        x + body(x)                         two convs at 1x (residual add in the epilogue)
        up(body(down(x)))                   x0.5 -> conv o down-1x1 -> conv o up-1x1 at 1/2x, then x2
        down(body(up(x)))                   conv o up-1x1 at 2x, its input the bilinear x2 of x built in the kernel's producer and its output
                                            the four parity planes -> conv o down-1x1 and x0.5 as one 4x4 / stride-2 convolution at 1x
    The last kernel also adds the other two branches in its epilogue.  x8_half: bilinear x0.5 of x8 if the producer of x8 already
    wrote it; want_half: return (out, x0.5 of out), the x0.5 taken in the same epilogue."""
    H, W = x8.shape[2:4]
    if H % 2 or W % 2 or H < 4 or W < 4:
        raise _lib.CdfoError("cross_scale_block: H and W must be even and >= 4 (got %d x %d)" % (H, W))
    b0, b2 = blk.body._modules["0"], blk.body._modules["2"]
    wts = _block_weights(blk)
    wd0, bd0, ed0 = wts["body0_dn"]
    wu0, bu0, eu0 = wts["body0_up"]
    y = conv.conv3x3(conv.conv3x3(x8, b0.weight, b0.bias, conv.ACT_LRELU), b2.weight, b2.bias, conv.ACT_NONE, resid8=x8)
    xh = x8_half if x8_half is not None else conv.resample(x8, 0)
    cu = conv.conv3x3(conv.conv3x3(xh, wd0, bd0, conv.ACT_LRELU, bias_edge=ed0), wts["up_body2"][0], wts["up_body2"][1], conv.ACT_NONE)
    t2 = conv.conv3x3_up2(x8, wu0, bu0, conv.ACT_LRELU, parity_planes=True, bias_edge=eu0)
    return conv.conv3x3_then_half(t2, wts["dn_body2"][0], wts["dn_body2"][1], resid8=y, up8=cu, want_half=want_half)


@torch.no_grad()
def recon_trunk(trunk, x8):
    """SCNet_(7 x SCGroup_(3 x Block_)), arch:430-480, c8 bf16 in and out; H and W even and >= 4 (cross_scale_block)."""
    y = x8
    for grp in trunk.body._modules.values():
        r, r_half = y, None
        blocks = list(grp.body._modules.values())
        for k, blk in enumerate(blocks):
            if k + 1 < len(blocks):
                r, r_half = cross_scale_block(blk, r, r_half, want_half=True)
            else:
                r = cross_scale_block(blk, r, r_half)
        y = conv.conv3x3(r, grp.conv.weight, grp.conv.bias, conv.ACT_NONE, resid8=y)
    return y + x8


# ------------------------------------------------------------------------------------------ feature extraction pieces (8f rank 2)
@torch.no_grad()
def layernorm_c(x, gamma, beta, eps=1e-5):
    """LayerNorm over the channels of each pixel (WithBias, arch:1169-1198) on NCHW fp32 / bf16, fp32 arithmetic."""
    B, C, H, W = x.shape
    x = x.contiguous()
    y = torch.empty_like(x)
    _lib.call("cdfo_layernorm_c_fwd", _lib.ptr(x), _lib.ptr(_f32(gamma)), _lib.ptr(_f32(beta)), _lib.ptr(y), B, C, H, W,
              ctypes.c_float(eps), _lib.dtype_code(x), _lib.stream_ptr(x.device))
    return y


@torch.no_grad()
def dwconv3x3(x, weight):
    """Depthwise 3x3 / stride 1 / padding 1 without bias (qkv_dwconv, arch:1545-1576) on NCHW fp32 / bf16."""
    B, C, H, W = x.shape
    x = x.contiguous()
    y = torch.empty_like(x)
    _lib.call("cdfo_dwconv3x3_fwd", _lib.ptr(x), _lib.ptr(_f32(weight).reshape(C, 9)), _lib.ptr(y), B, C, H, W, _lib.dtype_code(x),
              _lib.stream_ptr(x.device))
    return y


@torch.no_grad()
def mdta_gram(qkv, parts=256):
    """Per-head Gram q k^T over H*W and the squared norms of the rows of q and k (8 heads x 8 channels) of the depthwise-convolved
    qkv tensor [B, 192, H, W] (arch:1545-1576): (G [B, 8, 8, 8], |q|^2 [B, 64], |k|^2 [B, 64]) fp32, q and k read once."""
    B, C, H, W = qkv.shape
    if C < 128 or not qkv.is_contiguous():
        raise _lib.CdfoError("mdta_gram: contiguous [B, >=128, H, W] tensor expected")
    parts = max(1, min(parts, (H * W + 63) // 64))
    partial = torch.empty((B, parts, 640), dtype=torch.float32, device=qkv.device)
    _lib.call("cdfo_mdta_gram_fwd", _lib.ptr(qkv), _lib.ptr(partial), B, C, H, W, parts, _lib.dtype_code(qkv), _lib.stream_ptr(qkv.device))
    s = partial.sum(1)
    return s[:, :512].view(B, 8, 8, 8), s[:, 512:576], s[:, 576:640]
