"""Deterministic synthetic clips, coding priors and weights (no dataset / checkpoint ships with the reference).

Everything is drawn from seeded *CPU* torch generators so that the build container (golden fixtures made
from the real reference) and the GPU box regenerate bit-identical inputs.  Shapes and value ranges follow the
reference's data contract (test_LD_37.py:19-105,143-161): LR luma / partition map / unfiltered frame in
[0,1] on a k/255 grid, residual map = int/255, MV field int8 [H,W,3] = (mv_a, mv_b, ref-distance) in
quarter-pel units, constant on 8x8 blocks, decoded with mv2mvs.
"""
import math

import torch

N_FRAMES = 7


def _gen(seed):
    return torch.Generator().manual_seed(int(seed))


def make_clip(seed, H, W, B=1, config="LD"):
    """Returns dict of CPU tensors: x, pms, rms, ufs [B,7,1,H,W] fp32; mv_l0 int8 [B,H,W,3]
    (config 'RA' adds mv_l1 with positive ref-distances and -99 sentinels, opt/data_RA_bi.py:501-528)."""
    assert H % 8 == 0 and W % 8 == 0, "H and W must be multiples of 8 (window attention, arch:2235)"
    g = _gen(20240000 + seed)
    out = {}
    x = torch.randint(0, 256, (B, N_FRAMES, 1, H, W), generator=g).float()
    # smooth the LR frames a little so that they look like images rather than white noise
    k = torch.ones(1, 1, 5, 5) / 25.0
    x = torch.nn.functional.conv2d(x.reshape(-1, 1, H, W), k, padding=2).reshape(B, N_FRAMES, 1, H, W)
    x = torch.round(x * 2.0 - 127.0).clamp(0, 255)
    out["x"] = x / 255.0
    # partition map: piece-wise constant on 8/16/32-px blocks
    pm = torch.zeros(B, N_FRAMES, 1, H, W)
    for bs in (32, 16, 8):
        hb, wb = math.ceil(H / bs), math.ceil(W / bs)
        lvl = torch.randint(0, 256, (B, N_FRAMES, 1, hb, wb), generator=g).float()
        use = (torch.rand(B, N_FRAMES, 1, hb, wb, generator=g) < 0.5).float()
        up = lambda t: t.repeat_interleave(bs, -2).repeat_interleave(bs, -1)[..., :H, :W]  # noqa: E731
        pm = torch.where(up(use) > 0, up(lvl), pm)
    out["pms"] = pm / 255.0
    # residual map: rounded N(0, 6), 70 % of the 8x8 blocks zero
    res = torch.round(torch.randn(B, N_FRAMES, 1, H, W, generator=g) * 6.0).clamp(-128, 127)
    keep = (torch.rand(B, N_FRAMES, 1, H // 8, W // 8, generator=g) >= 0.7).float()
    out["rms"] = res * keep.repeat_interleave(8, -2).repeat_interleave(8, -1) / 255.0
    # unfiltered frame: x + U(-4, 4)/255, clipped
    noise = torch.randint(-4, 5, (B, N_FRAMES, 1, H, W), generator=g).float()
    out["ufs"] = (x + noise).clamp(0, 255) / 255.0
    # motion vectors: quarter-pel, block constant, ref-distance in {-1,-2,-4}
    def mv_field(sign):
        blk = torch.randint(-64, 64, (B, H // 8, W // 8, 2), generator=g)
        rd = torch.tensor([1, 2, 4])[torch.randint(0, 3, (B, H // 8, W // 8, 1), generator=g)] * sign
        f = torch.cat([blk, rd], dim=-1).repeat_interleave(8, 1).repeat_interleave(8, 2)
        return f.to(torch.int8)
    out["mv_l0"] = mv_field(-1)
    if config == "RA":
        l1 = mv_field(+1).clone()
        sentinel = (torch.rand(B, H // 8, W // 8, generator=g) < 0.15).repeat_interleave(8, 1).repeat_interleave(8, 2)
        l1[..., 2][sentinel] = -99
        out["mv_l1"] = l1
    return out


def gumbel_uniforms(seed, sequence, frame, B, H, W, C=64):
    """The six uniform draws of LLongRangAttention.gumbel_softmax for one output frame (arch:2169), keyed by
    (sequence, frame, neighbour) rather than by device RNG state -> sharding-invariant results."""
    us = []
    for nb in (0, 1, 2, 4, 5, 6):
        g = _gen(70000000 + ((seed * 4099 + sequence) * 4099 + frame) * 7 + nb)
        u = torch.rand(B, C, H, W, generator=g)
        us.append(u.clamp_min(1e-12))  # the reference redraws while any u == 0 (arch:2170-2171)
    return us


def _fan_in(shape):
    n = 1
    for s in shape[1:]:
        n *= s
    return max(n, 1)


def seeded_state_dict(template, seed=4):
    """Deterministic non-degenerate weights for every key of `template` (a state_dict giving names and shapes).
    Scales follow the reference's initialisers (kaiming fan-in; x0.1 for residual trunks, arch:275-292); the
    zero-initialised head of the DCN alignment (arch:3301) gets small non-zero values so that parity exercises
    it (SURVEY.md 8c), temperatures / LayerNorm gains are perturbed around 1."""
    sd = {}
    for idx, key in enumerate(sorted(template.keys())):
        shape = tuple(template[key].shape)
        g = _gen(seed * 1000003 + idx)
        leaf = key.rsplit(".", 1)[-1]
        if leaf == "temperature":
            t = 1.0 + 0.25 * torch.randn(shape, generator=g)
        elif ".norm" in key and leaf == "weight":
            t = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif leaf == "bias":
            std = 0.1 if "conv_offset.2" in key else 0.02
            t = std * torch.randn(shape, generator=g)
        else:  # convolution weights
            std = math.sqrt(1.0 / _fan_in(shape))
            if key.startswith("recon_trunk") or "ResidualBlock" in key:
                std *= 0.1 * math.sqrt(2.0)
            if "conv_offset.2" in key:
                std = 0.01
            if "directW1_conv" in key or "directH1_conv" in key:
                std = 0.3
            if key.startswith("conv_last"):
                std *= 0.02   # keeps SR = bilinear base + a small residual, i.e. outputs stay near [0, 1]
            t = std * torch.randn(shape, generator=g)
        sd[key] = t.to(template[key].dtype)
    return sd


class SyntheticSequences:
    """Lazy list of `n` synthetic coded sequences in the reference's on-disk data contract (driver.Sequence: uint8 LR / partition /
    unfiltered planes, integer residual maps, int8 MV fields [T, h, W, 3], uint8 ground truth at x4), each a pure function of its
    sequence id -- a rank generates only the sequences it owns, and every sharding sees identical data (BASELINE.json configs[3]:
    64 independent 1080p x4 sequences).  `frames`, `h`, `w` are one value for every sequence or one per sequence (a job of mixed sizes
    and lengths, tools/bench_job.py)."""

    def __init__(self, n, frames=16, h=270, w=480, seed=0, with_gt=True):
        self.n, self.seed, self.with_gt = int(n), int(seed), bool(with_gt)
        per = lambda v: [int(x) for x in v] if hasattr(v, "__len__") else [int(v)] * self.n   # noqa: E731
        self.frames, self.h, self.w = per(frames), per(h), per(w)
        if not len(self.frames) == len(self.h) == len(self.w) == self.n:
            raise ValueError("SyntheticSequences: one frames / h / w value per sequence")
        self._cache = {}

    def __len__(self):
        return self.n

    def shape_of(self, sid):
        """(T, h, W) of sequence `sid` without generating it."""
        if not 0 <= sid < self.n:
            raise IndexError(sid)
        return self.frames[sid], self.h[sid], self.w[sid]

    def __getitem__(self, sid):
        import numpy as np
        from .driver import Sequence
        if not 0 <= sid < self.n:
            raise IndexError(sid)
        if sid in self._cache:
            return self._cache[sid]
        T, h, w = self.shape_of(sid)
        rng = np.random.default_rng(900000 + 7919 * self.seed + sid)
        # a slowly drifting smooth image: low-resolution noise upsampled x8, shifted by one pixel per frame
        base = rng.integers(0, 256, (h // 8 + 3, w // 8 + 3 + T)).astype(np.float32)
        big = np.kron(base, np.ones((8, 8), np.float32))
        k = np.ones(9, np.float32) / 9.0
        big = np.apply_along_axis(lambda r: np.convolve(r, k, mode="same"), 1, big)
        big = np.apply_along_axis(lambda c: np.convolve(c, k, mode="same"), 0, big)
        lr = np.stack([big[8:8 + h, 8 + t:8 + t + w] for t in range(T)])
        lr = np.clip(np.round(lr + rng.normal(0, 2.0, lr.shape)), 0, 255).astype(np.uint8)
        unflt = np.clip(lr.astype(np.int16) + rng.integers(-4, 5, lr.shape), 0, 255).astype(np.uint8)
        hb, wb = -(-h // 16), -(-w // 16)
        pm = np.kron(rng.integers(0, 256, (T, hb, wb)).astype(np.uint8), np.ones((1, 16, 16), np.uint8))[:, :h, :w]
        keep = np.kron((rng.random((T, -(-h // 8), -(-w // 8))) >= 0.7).astype(np.int16), np.ones((1, 8, 8), np.int16))[:, :h, :w]
        res = (np.clip(np.round(rng.normal(0, 6.0, (T, h, w))), -128, 127).astype(np.int16) * keep).astype(np.int16)
        blk = rng.integers(-64, 64, (T, -(-h // 8), -(-w // 8), 2))
        rd = -np.array([1, 2, 4])[rng.integers(0, 3, (T, -(-h // 8), -(-w // 8), 1))]
        mv = np.kron(np.concatenate([blk, rd], -1), np.ones((1, 8, 8, 1), np.int64))[:, :h, :w].astype(np.int8)
        gt = None
        if self.with_gt:
            up = np.kron(lr, np.ones((1, 4, 4), np.uint8)).astype(np.int16)
            gt = np.clip(up + rng.integers(-3, 4, up.shape), 0, 255).astype(np.uint8)
        q = Sequence(lr, pm, res, unflt, mv, gt, name="synthetic_%03d" % sid)
        if len(self._cache) > 8:
            self._cache.clear()
        self._cache[sid] = q
        return q
