"""GPU checks of the job scheduler: the batched end-of-sequence MV fix-up (csrc/priors.cu) against the per-batch kernel and the
reference, a slot admission's feature window, sequences of different lengths on fewer slots than sequences, two frame sizes in one
run_sharded call, one sequence split over every slot."""
import numpy as np
import pytest
import torch

from cdfo_b200 import driver, priors
from oracle import metrics_ref as R, priors_ref
from test_driver_gpu import _model, _naive_loop, _sequence

pytestmark = pytest.mark.gpu


def test_mv_end_fix_batched_matches_per_sample(cuda_dev):
    """(i, T) mixed across the batch: every fix-up branch, short sequences where several conditions hold at once, both ends."""
    cases = [(i, T) for T in (1, 2, 5, 7) for i in range(T)] + [(0, 9), (1, 9), (2, 9), (4, 9), (6, 9), (7, 9), (8, 9), (3, 600)]
    B, H, W = len(cases), 16, 24
    g = torch.Generator().manual_seed(5)
    flows = torch.randn(B, 7, 2, H, W, generator=g)
    i_max = torch.tensor(cases, dtype=torch.int32, device=cuda_dev)
    got = priors.modify_mv_for_end_frames_batched(flows.to(cuda_dev), i_max).cpu()
    for b, (i, T) in enumerate(cases):
        one = priors.modify_mv_for_end_frames(i, flows[b:b + 1].to(cuda_dev).contiguous(), T).cpu()
        ref = priors_ref.modify_mv_for_end_frames(i, flows[b:b + 1].numpy().copy(), T)
        assert torch.equal(got[b:b + 1], one), (i, T)
        assert np.array_equal(got[b:b + 1].numpy(), ref), (i, T)


def test_mv_end_fix_batched_rejects_bad_tables(cuda_dev):
    mvs = torch.zeros(2, 7, 2, 8, 8, device=cuda_dev)
    for bad in (torch.zeros(2, 2, dtype=torch.int64, device=cuda_dev), torch.zeros(3, 2, dtype=torch.int32, device=cuda_dev)):
        with pytest.raises(ValueError):
            priors.modify_mv_for_end_frames_batched(mvs, bad)
    with pytest.raises(NotImplementedError):
        priors.modify_mv_for_end_frames_batched(mvs, torch.zeros(2, 2, dtype=torch.int32))


def _window_planes(q, lo, H, dev):
    T = q.shape[0]
    o = driver.generate_input_index(lo, 7, T - 1)
    x = torch.from_numpy(R.planes_to_unit(q.lr[o], H))[:, None].to(dev)
    pms = torch.from_numpy(R.planes_to_unit(q.pm[[driver.side_info_index(j) for j in o]], H))[:, None].to(dev)
    return x, pms


@pytest.mark.parametrize("ring", [True, False])
def test_admission_loads_the_slot_window(cuda_dev, ring):
    """Admission of sequence c at frame lo into slot 0 of a running batch of two: after load_window_features and the next step (which
    pushes the features of W(lo)[6]), slot 0's feature window equals the features of W(lo) computed alone, and slot 1's window only
    shifted.  ring=True: the eager FeatureRing; ring=False: the batch-major L1_fea that a graphed step copies in."""
    h, W = 24, 40
    H = driver.padded_rows(h)
    model = _model(cuda_dev)
    a, b, c = _sequence(31, 9, h, W, False), _sequence(32, 12, h, W, False), _sequence(33, 9, h, W, False)

    def window(l1):                                                          # [2, 7, 64, H, W] copy, sample-major
        if ring:
            return l1._cdfo_ring[0].window().transpose(0, 1).clone()
        return l1.view(2, 7, 64, H, W).clone()
    model.feature_ring = ring
    try:
        mvs = torch.zeros(2, 7, 2, H, W, device=cuda_dev)
        xa, pa = _window_planes(a, 0, H, cuda_dev)
        for step, lo in enumerate((0, 4, 8)):                                # W(0) repeats frame 0, W(8) repeats frame 8
            xb, pb = _window_planes(b, step, H, cuda_dev)
            if step == 0:
                x, pms = torch.stack([xa, xb]), torch.stack([pa, pb])
                _, l1 = model(x, None, mvs, pms, pms, pms, None, noise=driver.noise_for(0, [0, 1], 0, H, W, cuda_dev))
            before = window(l1)
            xc, pc = _window_planes(c, lo, H, cuda_dev)
            o = driver.generate_input_index(lo, 7, 8)[:6]
            distinct = sorted(set(o))
            pick = [o.index(j) for j in distinct]
            model.load_window_features(l1, 0, xc[pick], pc[pick], [distinct.index(j) for j in o])
            assert torch.equal(window(l1)[1], before[1])                      # the other slot is untouched
            xb, pb = _window_planes(b, step + 1, H, cuda_dev)
            x, pms = torch.stack([xc, xb]), torch.stack([pc, pb])
            _, l1 = model(x, None, mvs, pms, pms, pms, l1, noise=driver.noise_for(0, [0, 1], step + 1, H, W, cuda_dev))
            after = window(l1)
            alone = model._features(xc, pc)                                   # [7, 64, H, W]: W(lo) as a first window
            err = float((after[0] - alone).abs().max())
            assert err <= 5e-3 * max(1.0, float(alone.abs().max())), (lo, err)   # batch 2 vs 7: reduction orders only
            assert torch.equal(after[1, :6], before[1, 1:])                    # slot 1 only shifted by one frame
    finally:
        model.feature_ring = False


@pytest.mark.parametrize("graph", [False, True])
def test_driver_lengths_2_5_9_on_two_slots(cuda_dev, graph):
    """Three sequences of different lengths on two slots (admission and idle slot): every frame within one uint8 level of the
    window-by-window loop on < 8 % of the pixels, PSNR / SSIM equal to the oracle on the delivered frames."""
    h, W = 28, 40
    lengths = (2, 5, 9)
    seqs = [_sequence(40 + k, T, h, W) for k, T in enumerate(lengths)]
    model = _model(cuda_dev)
    got = {}

    def sink(s, i, img):
        assert (s, i) not in got
        got[(s, i)] = img
    res = driver.FrameDriver(model, seed=3, graph=graph).run(seqs, seq_ids=[7, 8, 9], sink=sink, slots=2)
    assert len(got) == sum(lengths) and res["frames"] == 9
    assert res["admissions"] == 1 and res["steps"] == 11 and res["idle_slot_steps"] == 2 * 11 - sum(lengths)
    for s, q in enumerate(seqs):
        ref = _naive_loop(model, q, 7 + s, 3, cuda_dev)
        p = sm = 0.0
        for i in range(q.shape[0]):
            d = np.abs(got[(s, i)].astype(np.int64) - ref[i].astype(np.int64))
            assert d.max() <= 1 and (d > 0).mean() < 0.08, (s, i, d.max(), (d > 0).mean())
            p += R.psnr_y(got[(s, i)], q.gt[i]) / q.shape[0]
            sm += R.ssim_y(got[(s, i)], q.gt[i]) / q.shape[0]
        assert abs(res["psnr"][s] - p) < 1e-9 and abs(res["ssim"][s] - sm) < 1e-10


def test_run_sharded_two_frame_sizes(cuda_dev):
    seqs = [_sequence(50, 4, 24, 40), _sequence(51, 3, 32, 48), _sequence(52, 6, 24, 40)]
    model = _model(cuda_dev)
    seen = []
    r = driver.run_sharded(model, seqs, batch=2, seed=4, sink=lambda k, i, img: seen.append((k, i, img.shape)))
    assert r["frames"] == [4.0, 3.0, 6.0] and sorted((k, i) for k, i, _ in seen) == [(k, i) for k, q in enumerate(seqs) for i in range(q.shape[0])]
    assert all(shape == (4 * seqs[k].shape[1], 4 * seqs[k].shape[2]) for k, _, shape in seen)
    one = driver.FrameDriver(model, seed=4).run([seqs[1]], seq_ids=[1])
    assert abs(one["psnr"][0] - r["psnr"][1]) < 5e-3 and abs(one["ssim"][0] - r["ssim"][1]) < 1e-4


@pytest.mark.parametrize("T", [23, 40])
def test_run_sharded_split_one_sequence(cuda_dev, T):
    """One sequence with split=True on four slots: 23 frames stay one item (16-frame minimum), 40 frames become two items of 20,
    the second starting at frame 20 with a fresh window (first-frame path at lo = 20)."""
    q = _sequence(60, T, 24, 40)
    model = _model(cuda_dev)
    got, whole = {}, {}

    def sink(k, i, img):
        assert (k, i) not in got
        got[(k, i)] = img
    r = driver.run_sharded(model, [q], batch=4, seed=5, sink=sink, split=True)
    assert r["items"] == T // 16 and r["frames"] == [float(T)] and sorted(got) == [(0, i) for i in range(T)]
    one = driver.FrameDriver(model, seed=5).run([q], seq_ids=[0], sink=lambda s, i, img: whole.__setitem__(i, img))
    for i in range(T):
        d = np.abs(got[(0, i)].astype(np.int64) - whole[i].astype(np.int64))
        assert d.max() <= 1 and (d > 0).mean() < 0.08, (i, d.max(), (d > 0).mean())
    assert abs(one["psnr"][0] - r["psnr"][0]) < 5e-3 and abs(one["ssim"][0] - r["ssim"][0]) < 1e-4
