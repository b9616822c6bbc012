"""Host logic of the job scheduler: work-item partition (sharding.partition_items), the driver's slot schedule
(driver.slot_schedule), per-item metric rows reduced over a world-size-2 gloo group, argument checks of the batched MV fix-up.
No GPU."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cdfo_b200 import driver, sharding, synthetic

JCT_LD = [(240, 270, 480), (600, 270, 480), (500, 120, 208), (300, 60, 104), (600, 180, 320), (500, 60, 104)]
MIXES = [
    [(23, 270, 480)],
    [(600, 270, 480)],
    [(5, 24, 40), (2, 24, 40), (9, 24, 40)],
    [(16, 64, 64)] * 7,
    [(17, 32, 48), (31, 32, 48), (1, 64, 64), (64, 64, 64)],
    JCT_LD,
    [(8, 60, 104)] * 3 + [(240, 270, 480)],
]


def _check_partition(shapes, world, slots, split):
    items, ranks = sharding.partition_items(shapes, world, slots, split)
    assert len(items) == len(ranks) and all(0 <= r < world for r in ranks)
    covered = {}
    for it in items:
        T = shapes[it.seq][0]
        assert 0 <= it.lo < it.hi <= T                                        # never crosses a sequence boundary
        if T >= sharding.MIN_ITEM_FRAMES:
            assert it.hi - it.lo >= sharding.MIN_ITEM_FRAMES
        rlo, rhi = it.read_range(T)
        for i in range(it.lo, it.hi):
            covered[(it.seq, i)] = covered.get((it.seq, i), 0) + 1
            w = sharding.window_indices(i, T)
            assert min(w) >= rlo and max(w) < rhi                             # the read range holds every window of its frames
    assert covered == {(k, i): 1 for k, (T, _, _) in enumerate(shapes) for i in range(T)}
    assert items == sorted(items)                                              # (sequence, lo) order
    return items, ranks


@pytest.mark.parametrize("world", range(1, 9))
def test_partition_sequence_mode_is_sequence_shard(world):
    for shapes in MIXES:
        items, ranks = _check_partition(shapes, world, 4, split=False)
        assert [(it.lo, it.hi) for it in items] == [(0, T) for T, _, _ in shapes]
        for r in range(world):
            assert [it.seq for it, q in zip(items, ranks) if q == r] == sharding.sequence_shard(len(shapes), world, r)


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("slots", [1, 4])
def test_partition_split_mode_balances_cost(world, slots):
    for shapes in MIXES:
        items, ranks = _check_partition(shapes, world, slots, split=True)
        assert (items, ranks) == sharding.partition_items(shapes, world, slots, split=True)    # pure function of its arguments
        load = sharding.rank_costs(items, ranks, shapes, world)
        mean = sum(load) / world
        biggest = max(sharding.item_cost(it, shapes[it.seq]) for it in items)
        assert all(abs(c - mean) <= biggest for c in load), (shapes, load, biggest)
        possible = sum(max(1, T // sharding.MIN_ITEM_FRAMES) for T, _, _ in shapes)
        assert len(items) >= min(world * slots, possible)                      # enough items for every slot where lengths allow


def test_partition_one_long_sequence_fills_every_slot():
    items, ranks = sharding.partition_items([(600, 270, 480)], 8, 4, split=True)
    assert len(items) == 32 and all(ranks.count(r) == 4 for r in range(8))
    assert max(it.hi - it.lo for it in items) - min(it.hi - it.lo for it in items) <= 1


def test_partition_rejects_bad_arguments():
    for bad in (([(0, 8, 8)], 1, 1), ([(4, 8, 8)], 0, 1), ([(4, 8, 8)], 1, 0), ([(4, 8)], 1, 1)):
        with pytest.raises(ValueError):
            sharding.partition_items(*bad, split=True)


def _run_schedule(ranges, slots):
    steps = driver.slot_schedule(ranges, slots)
    issued = {k: [] for k in range(len(ranges))}
    holder = {}
    assert steps[0].first
    for t, st in enumerate(steps):
        if st.first:
            assert all(e is not None and not e[2] for e in st.slots)          # a batch starts with every slot live
        for s, e in enumerate(st.slots):
            if e is None:
                continue
            k, i, admitted = e
            issued[k].append((t, s, i))
            if admitted:
                assert not st.first and i == ranges[k][0]
    for k, (lo, hi) in enumerate(ranges):
        frames = [i for _, _, i in issued[k]]
        assert frames == list(range(lo, hi))                                   # every frame once, in order
        ts = [t for t, _, _ in issued[k]]
        assert ts == list(range(ts[0], ts[0] + hi - lo))                       # consecutive steps
        assert len({s for _, s, _ in issued[k]}) == 1                          # on one slot
        holder[k] = (issued[k][0][1], ts[0], ts[-1])
    return steps, holder


@pytest.mark.parametrize("slots", [1, 2, 3, 4])
def test_slot_schedule_invariants(slots):
    for ranges in ([(0, 2), (0, 5), (0, 9)], [(0, 23)], [(0, 7), (7, 23), (3, 4), (0, 1), (10, 30), (0, 16)],
                   [(0, 5)] * 6, [(0, 3), (0, 3), (0, 9), (0, 4), (0, 4)]):
        steps, holder = _run_schedule(ranges, slots)
        for t, st in enumerate(steps):
            held = [k for k, (s, a, b) in holder.items() if a <= t <= b]
            assert len(held) == len({holder[k][0] for k in held})            # a slot holds one item at a time
            assert len(held) == sum(e is not None for e in st.slots)
        # a slot refills in the step after its item ends (while the queue has items and other slots still run)
        for k, (s, a, b) in holder.items():
            nxt = [j for j, (s2, a2, _) in holder.items() if s2 == s and a2 > b]
            if nxt and not steps[min(holder[j][1] for j in nxt)].first:
                assert min(holder[j][1] for j in nxt) == b + 1
        for st in steps:
            assert len(st.slots) <= slots


def test_slot_schedule_refills_next_step_and_idles():
    steps = driver.slot_schedule([(0, 2), (0, 5), (0, 9)], 2)
    assert len(steps) == 11
    assert steps[0] == driver.Step(True, ((0, 0, False), (1, 0, False)))
    assert steps[2] == driver.Step(False, ((2, 0, True), (1, 2, False)))     # slot 0 admits item 2 the step after item 0 ended
    assert steps[5].slots[1] is None and steps[10] == driver.Step(False, ((2, 8, False), None))
    idle = sum(e is None for st in steps for e in st.slots)
    assert idle == 2 * 11 - (2 + 5 + 9)


@pytest.mark.parametrize("n,slots", [(1, 4), (4, 4), (8, 4), (7, 4), (3, 2), (64, 8)])
def test_slot_schedule_equal_lengths_are_todays_batches(n, slots):
    T = 6
    steps = driver.slot_schedule([(0, T)] * n, slots)
    want = []
    for b0 in range(0, n, slots):
        ids = list(range(b0, min(b0 + slots, n)))
        for i in range(T):
            want.append(driver.Step(i == 0, tuple((k, i, False) for k in ids)))
    assert steps == want                                                       # no admission, no idle slot


def test_synthetic_shape_of_needs_no_generation():
    lazy = synthetic.SyntheticSequences(3, frames=[5, 9, 2], h=[24, 24, 60], w=[40, 40, 104], with_gt=False)
    assert [lazy.shape_of(k) for k in range(3)] == [(5, 24, 40), (9, 24, 40), (2, 60, 104)] and not lazy._cache
    assert lazy[2].shape == (2, 60, 104)
    assert synthetic.SyntheticSequences(2, frames=4, h=16, w=24).shape_of(1) == (4, 16, 24)


# ------------------------------------------------------------------------------------------------ per-item metric rows
def _fake_frame_metrics(seq, frame):
    g = torch.Generator().manual_seed(1000 * seq + frame)
    err = torch.randn(16, 16, generator=g, dtype=torch.float64)
    return torch.tensor([float(30.0 + (err * err).mean()), float(err.abs().mean()), 1.0], dtype=torch.float64)


SHAPES = [(40, 24, 40), (17, 24, 40), (33, 60, 104), (5, 24, 40)]


def _item_rows(items, mine):
    rows = torch.zeros(len(items), 3, dtype=torch.float64)
    for j in mine:                                          # frame order within an item, as the slot accumulator adds them
        for i in range(items[j].lo, items[j].hi):
            rows[j] += _fake_frame_metrics(items[j].seq, i)
    return rows


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        items, ranks = sharding.partition_items(SHAPES, world, 2, split=True)
        rows = sharding.gather_metrics(_item_rows(items, [j for j, r in enumerate(ranks) if r == rank]))
        total = sharding.sequence_sums(rows, [it.seq for it in items], len(SHAPES))
        dist.barrier()
        if rank == 0:
            torch.save(total, out)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_item_metric_rows_world2_gloo(tmp_path):
    """Split items over two ranks, rows all-reduced, items summed per sequence == the same items all run in one process."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "total.pt")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    total = torch.load(out)
    items, ranks = sharding.partition_items(SHAPES, 2, 2, split=True)
    assert len(set(ranks)) == 2 and any(it.lo > 0 for it in items)
    ref = sharding.sequence_sums(_item_rows(items, range(len(items))), [it.seq for it in items], len(SHAPES))
    assert torch.equal(total, ref)
    assert total[:, 2].tolist() == [float(T) for T, _, _ in SHAPES]


def test_sequence_sums_one_item_per_sequence_is_the_row():
    rows = torch.tensor([[31.25, 0.5, 3.0], [0.1 + 0.2, 1 / 3.0, 7.0]], dtype=torch.float64)
    assert torch.equal(sharding.sequence_sums(rows, [0, 1], 2), rows)


# ------------------------------------------------------------------------------------------------ C entry point, argument checks
def test_mv_end_fix_batched_rejects_bad_arguments(cdfo_so):
    import cdfo_b200._lib as L
    lib = L.lib()
    buf = ctypes.create_string_buffer(64)
    assert lib.cdfo_mv_end_fix_batched(None, 1, 8, 8, buf, None) == -2 and b"NULL" in lib.cdfo_last_error()
    assert lib.cdfo_mv_end_fix_batched(buf, 1, 8, 8, None, None) == -2
    for B, H, W in ((0, 8, 8), (1, 0, 8), (1, 8, -1), (70000, 8, 8), (1, 1 << 16, 1 << 15)):
        assert lib.cdfo_mv_end_fix_batched(buf, B, H, W, buf, None) == -1 and b"bad shape" in lib.cdfo_last_error()
