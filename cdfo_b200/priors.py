"""Coding-prior decoding on the device: MV field -> 7 flows, end-of-sequence fix-up, flow_warp.

Mirrors (same names / argument meaning) the reference's host helpers
`mv2mvs` (test_LD_37.py:83-105), `modify_mv_for_end_frames`
(test_LD_37.py:209-234) and `flow_warp` (arch/SIDECVSR_our.py:3068-3099),
but runs them as CUDA kernels through the C ABI.
"""
import torch

from . import _lib


@torch.no_grad()
def mv2mvs(mv: torch.Tensor) -> torch.Tensor:
    """mv: CUDA int8 or int32 tensor [H, W, 3] (mv_a, mv_b, ref-distance).
    Returns fp32 flows [1, 7, 2, H, W] -- the tensor the reference obtains after
    `mv2mvs(...)`, `unsqueeze(0)` and `permute(0,1,4,2,3)` (test_LD_37.py:159-161)."""
    _lib.require_cuda(mv)
    if mv.dim() != 3 or mv.size(2) != 3:
        raise ValueError("mv must be [H, W, 3], got %s" % (tuple(mv.shape),))
    if mv.dtype not in (torch.int8, torch.int32):
        raise TypeError("mv must be int8 or int32, got %s" % mv.dtype)
    mv = mv.contiguous()
    H, W = mv.shape[:2]
    out = torch.empty((1, 7, 2, H, W), dtype=torch.float32, device=mv.device)
    _lib.call("cdfo_mv2mvs", _lib.ptr(mv), int(mv.dtype == torch.int32), _lib.ptr(out), H, W,
                                _lib.stream_ptr(mv.device))
    return out


@torch.no_grad()
def mv2mvs_ra(mv_l0: torch.Tensor, mv_l1: torch.Tensor) -> torch.Tensor:
    """RA configuration: an (l0, l1) pair of CUDA int8 / int32 MV fields [H, W, 3] (ref-distance -99 = list missing) ->
    fp32 flows [1, 7, 2, H, W]: frames 0-2 from l0, 4-6 from l1, each list complemented from the other where it is missing
    (opt/data_RA_bi.py:419-424, :496-533, and the / 32 of train_RA_37.py:383-386)."""
    _lib.require_cuda(mv_l0, mv_l1)
    if mv_l0.shape != mv_l1.shape or mv_l0.dim() != 3 or mv_l0.size(2) != 3:
        raise ValueError("mv_l0 / mv_l1 must both be [H, W, 3]")
    if mv_l0.dtype != mv_l1.dtype or mv_l0.dtype not in (torch.int8, torch.int32):
        raise TypeError("mv_l0 / mv_l1 must both be int8 or int32")
    mv_l0, mv_l1 = mv_l0.contiguous(), mv_l1.contiguous()
    H, W = mv_l0.shape[:2]
    out = torch.empty((1, 7, 2, H, W), dtype=torch.float32, device=mv_l0.device)
    _lib.call("cdfo_mv2mvs_ra", _lib.ptr(mv_l0), _lib.ptr(mv_l1), int(mv_l0.dtype == torch.int32), _lib.ptr(out), H, W,
              _lib.stream_ptr(mv_l0.device))
    return out


@torch.no_grad()
def modify_mv_for_end_frames(i: int, mvs: torch.Tensor, max_idx: int) -> torch.Tensor:
    """In place on mvs [B, 7, 2, H, W] fp32 (contiguous CUDA); returns mvs."""
    _lib.require_cuda(mvs)
    if mvs.dim() != 5 or mvs.size(1) != 7 or mvs.size(2) != 2 or mvs.dtype != torch.float32:
        raise ValueError("mvs must be fp32 [B, 7, 2, H, W]")
    if not mvs.is_contiguous():
        raise RuntimeError("mvs has to be contiguous")
    B, _, _, H, W = mvs.shape
    _lib.call("cdfo_mv_end_fix", _lib.ptr(mvs), B, H, W, int(i), int(max_idx), _lib.stream_ptr(mvs.device))
    return mvs


@torch.no_grad()
def modify_mv_for_end_frames_batched(mvs: torch.Tensor, i_max: torch.Tensor) -> torch.Tensor:
    """The same fix-up with its own (i, max_idx) per sample: i_max is a CUDA int32 [B, 2] table on the device of mvs (frame
    driver slots sit at different frames of different sequences).  One launch, in place on mvs [B, 7, 2, H, W]; returns mvs."""
    _lib.require_cuda(mvs, i_max)
    if mvs.dim() != 5 or mvs.size(1) != 7 or mvs.size(2) != 2 or mvs.dtype != torch.float32:
        raise ValueError("mvs must be fp32 [B, 7, 2, H, W]")
    if not mvs.is_contiguous():
        raise RuntimeError("mvs has to be contiguous")
    B, _, _, H, W = mvs.shape
    if i_max.dtype != torch.int32 or tuple(i_max.shape) != (B, 2) or not i_max.is_contiguous() or i_max.device != mvs.device:
        raise ValueError("i_max must be a contiguous int32 [B, 2] tensor on the device of mvs")
    _lib.call("cdfo_mv_end_fix_batched", _lib.ptr(mvs), B, H, W, _lib.ptr(i_max), _lib.stream_ptr(mvs.device))
    return mvs


@torch.no_grad()
def flow_warp(x, flow, interp_mode="bilinear", padding_mode="zeros", align_corners=True, return_index=False):
    """x [B,C,H,W] fp32, flow [B,H,W,2] (the reference's argument layout, last dim = (x, y))."""
    if interp_mode != "bilinear" or padding_mode != "zeros" or not align_corners:
        raise NotImplementedError("flow_warp: only the mode the model uses (bilinear, zeros, align_corners=True)")
    _lib.require_cuda(x, flow)
    assert x.size()[-2:] == flow.size()[1:3]
    B, C, H, W = x.shape
    x = x.contiguous().float()
    flow_chw = flow.permute(0, 3, 1, 2).contiguous().float()  # a no-copy view round trip when the model permuted it
    return flow_warp_chw(x, flow_chw, return_index)


@torch.no_grad()
def flow_warp_chw(x, flow_chw, return_index=False):
    """Same op with flow held as [B,2,H,W] (the layout CVSR_V8 keeps, arch/SIDECVSR_our.py:4445)."""
    B, C, H, W = x.shape
    y = torch.empty_like(x)
    idx = torch.empty((B, H, W, 2), dtype=torch.int32, device=x.device) if return_index else None
    _lib.call("cdfo_flow_warp_fwd", _lib.ptr(x), _lib.ptr(flow_chw), _lib.ptr(y), B, C, H, W, _lib.ptr(idx),
                                       _lib.stream_ptr(x.device))
    return (y, idx) if return_index else y
