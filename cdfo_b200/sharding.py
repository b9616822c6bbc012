"""Multi-GPU plan of the hot path: independent units, no exchange step (SURVEY.md 8e).

Every output frame depends only on its own 7-frame window of LR frames + priors (test_LD_37.py:143-160) and per-frame
features depend only on that frame (arch/SIDECVSR_our.py:4417-4419), so the work list of (sequence, frame) items is
partitioned statically: one process per GPU, weights replicated, no collective on the data path.  The only collective
is the end-of-job gather of the metric sums (the reference computes PSNR/SSIM per sequence on the host,
metric/psnr_ssim.py:446-484): one all_reduce(SUM) of an [n_seq, 3] fp64 tensor (sum of per-frame PSNR, sum of per-frame
SSIM, frame count -- what metrics.psnr_ssim(accum=) accumulates), NCCL on the GPU box, gloo in the CPU tests.

Work items (`WorkItem`, `partition_items`): output frames [lo, hi) of one sequence.  Sequence mode gives one item per sequence in
`sequence_shard` blocks; split mode cuts sequences into frame ranges and balances their cost (frames x padded LR pixels) over the
ranks.  The metric rows are kept per item, so per-sequence PSNR / SSIM do not depend on how the job was cut or scheduled.

Nothing here touches CUDA: the functions are plain host logic and are tested with world_size-2 gloo groups.
"""
from typing import NamedTuple

import torch
import torch.distributed as dist

HALO = 3   # frames of temporal context on each side of an output frame (nframes // 2, arch:4377)
MIN_ITEM_FRAMES = 16   # an item start recomputes the features of 6 window frames: split no item shorter than this


def partition(n_items, world, rank):
    """Contiguous block [lo, hi) of `n_items` owned by `rank`; sizes differ by at most one, earlier ranks get the extra."""
    if world <= 0 or not 0 <= rank < world or n_items < 0:
        raise ValueError("partition: bad arguments")
    base, extra = divmod(n_items, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def sequence_shard(n_seq, world, rank):
    """Sequence ids owned by `rank` (config c4: 64 sequences over 2/4/8 GPUs -> blocks of 32/16/8)."""
    lo, hi = partition(n_seq, world, rank)
    return list(range(lo, hi))


def frame_shard(n_frames, world, rank):
    """Within one sequence (load balance of long clips): output frames [lo, hi) owned by `rank` and the frame range
    [read_lo, read_hi) it must read (a HALO-frame halo each side, clipped like generate_input_index, test_LD_37.py:13-16).
    The first window of a shard recomputes the per-frame features of its halo: the L1_fea cache is a pure optimisation."""
    lo, hi = partition(n_frames, world, rank)
    return (lo, hi), (max(lo - HALO, 0), min(hi + HALO, n_frames))


class WorkItem(NamedTuple):
    """Output frames lo .. hi-1 of sequence `seq`."""
    seq: int
    lo: int
    hi: int

    def read_range(self, n_frames):
        """Frames [lo', hi') the item reads: its frames and a HALO-frame halo each side, clipped to the sequence (frame_shard)."""
        return max(self.lo - HALO, 0), min(self.hi + HALO, n_frames)


def padded_pixels(h, w):
    """LR pixels the model runs on per frame (rows padded to a multiple of 8, driver.padded_rows)."""
    return (h + 7) // 8 * 8 * w


def item_cost(item, shape):
    """Work of an item: output frames x padded LR pixels of its sequence (shape = (T, h, W))."""
    return (item.hi - item.lo) * padded_pixels(shape[1], shape[2])


def sequence_items(n_seq, world, rank, n_frames_of):
    """Sequence mode, one rank: one whole-sequence item per sequence of its sequence_shard block (`n_frames_of(k)` = T of sequence k
    is asked only for those)."""
    return [WorkItem(k, 0, int(n_frames_of(k))) for k in sequence_shard(n_seq, world, rank)]


def partition_items(shapes, world, slots=1, split=False):
    """Work items of a job and the rank of each: (items, ranks), a pure function of the arguments (every rank computes the same).

    shapes: (T, h, W) of every sequence.  Sequence mode (split=False): one item per sequence, in sequence order, rank = its
    sequence_shard block.  Split mode: every sequence is cut into near-equal frame ranges so that the job has at least
    world x slots items where the lengths allow it (no item shorter than MIN_ITEM_FRAMES unless its sequence is), items never
    cross a sequence boundary, and the items go, largest cost first, to the rank with the least cost so far: every rank's cost
    ends within one item's cost of the mean.  Items are listed in (sequence, lo) order."""
    shapes = [tuple(int(v) for v in s) for s in shapes]
    if world <= 0 or slots <= 0 or any(len(s) != 3 or min(s) <= 0 for s in shapes):
        raise ValueError("partition_items: bad arguments")
    n = len(shapes)
    if not split:
        items, ranks = [], []
        for r in range(world):
            own = sequence_items(n, world, r, lambda k: shapes[k][0])
            items += own
            ranks += [r] * len(own)
        return items, ranks
    costs = [T * padded_pixels(h, w) for T, h, w in shapes]
    target = sum(costs) / float(world * slots)
    items = []
    for k, (T, h, w) in enumerate(shapes):
        pieces = min(max(1, -(-costs[k] // max(int(target), 1))), max(1, T // MIN_ITEM_FRAMES))
        for p in range(pieces):
            lo, hi = partition(T, pieces, p)
            items.append(WorkItem(k, lo, hi))
    load = [0] * world
    ranks = [0] * len(items)
    order = sorted(range(len(items)), key=lambda j: (-item_cost(items[j], shapes[items[j].seq]), j))
    for j in order:
        r = min(range(world), key=lambda q: (load[q], q))
        ranks[j] = r
        load[r] += item_cost(items[j], shapes[items[j].seq])
    return items, ranks


def rank_costs(items, ranks, shapes, world):
    """Cost (item_cost) each rank of a partition carries."""
    load = [0] * world
    for it, r in zip(items, ranks):
        load[r] += item_cost(it, shapes[it.seq])
    return load


def sequence_sums(item_sums, item_seqs, n_seq):
    """Per-sequence [n_seq, 3] fp64 metric sums (host) from the reduced per-item rows [n_items, 3]; item_seqs[j] = sequence of item
    j.  Each sequence's items are added in item order onto zero, whatever rank or slot ran them: the result depends only on the
    per-frame values."""
    rows = item_sums.detach().cpu()
    out = torch.zeros((n_seq, 3), dtype=torch.float64)
    for j, k in enumerate(item_seqs):
        out[k] += rows[j]
    return out


def window_indices(i, n_frames, radius=HALO):
    """Frame indices of the 7-frame window of output frame i, clipped at the sequence ends (test_LD_37.py:13-16)."""
    return [min(max(j, 0), n_frames - 1) for j in range(i - radius, i + radius + 1)]


def noise_key(seed, sequence, frame, neighbour):
    """Seed of the Gumbel uniforms of (sequence, frame, neighbour): a function of the work item, not of the device RNG state
    or of the rank that runs it -> outputs are identical for every sharding (same formula as synthetic.gumbel_uniforms)."""
    return 70000000 + ((seed * 4099 + sequence) * 4099 + frame) * 7 + neighbour


def gather_metrics(local, group=None):
    """Sum of the per-rank [n_rows, 3] fp64 metric sums over all ranks (in place; identity without a process group).  A row is a
    sequence or a work item; rows a rank does not own must be zero, so every row has one contributing rank and the reduction is
    exact.  Returns the reduced tensor (see mean_metrics_per_sequence, sequence_sums)."""
    if local.dtype != torch.float64 or local.dim() != 2 or local.size(1) != 3:
        raise ValueError("gather_metrics: expected an [n_seq, 3] float64 tensor")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(local, op=dist.ReduceOp.SUM, group=group)
    return local


def mean_metrics_per_sequence(sums):
    """(mean PSNR [dB], mean SSIM) of each sequence from the reduced [n_seq, 3] sums = (sum of per-frame PSNR, sum of per-frame
    SSIM, frames) that metrics.psnr_ssim(accum=) / FrameDriver.run accumulate: the per-sequence average of per-frame values, which is
    what the reference's cal_psnr_ssim reports (metric/psnr_ssim.py:477-481)."""
    n = sums[:, 2].clamp_min(1.0)
    return sums[:, 0] / n, sums[:, 1] / n