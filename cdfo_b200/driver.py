"""Frame driver: the reference's evaluation loop (`eval_seq`, test_LD_37.py:118-181) as a device-resident pipeline.

What the reference does per output frame i of a sequence with T frames (all on the host, one frame at a time):
  o_list = clip(i-3 .. i+3, 0, T-1)                                   generate_input_index   test_LD_37.py:13-16
  LR / partition-map planes: uint8 / 255, 270-row frames + 2 zero rows generate_input / _PM    :19-46  (side info of frame max(1, j))
  residual / unfiltered planes / 255                                    generate_RM / _UF       :49-74
  mvs = mv2mvs(mvl0[max(1, i)]); modify_mv_for_end_frames(i, mvs, T)    :83-105, :157-163, :209-234
  sr, L1_fea = model(..., L1_fea)  (cached features after frame 0)      :165-169
  crop the padded rows, clamp * 255 -> uint8 -> PNG                     :172-180
  PSNR / SSIM of the PNGs against the ground truth, averaged per frame  metric/psnr_ssim.py:446-484

Here: S sequences of equal shape are batched; only the NEW frame of each window crosses PCIe (uint8 planes + the int MV
field from double-buffered pinned staging, on a copy stream that runs one step ahead of the compute stream); the
7-frame windows, the decoded flows, the feature cache and the SR frame stay in HBM; the uint8 SR frame returns through
pinned memory one step later; PSNR / SSIM are computed on the GPU (csrc/metrics.cu) into a per-sequence [n, 3] fp64
accumulator that `sharding.gather_metrics` reduces over ranks at the end of the job.  The Gumbel noise of
LLongRangAttention is keyed by (seed, sequence id, frame, neighbour), so results do not depend on batching or sharding.
"""
import os
from typing import NamedTuple

import numpy as np
import torch

from . import metrics, priors, sharding
from .graph import GraphedStep

NEIGHBOURS = (0, 1, 2, 4, 5, 6)


def generate_input_index(center_index, frame_number, max_index):
    """Window of `frame_number` frame indices centred on `center_index`, clipped to [0, max_index] (test_LD_37.py:13-16)."""
    lo = center_index - frame_number // 2
    return [min(max(j, 0), max_index) for j in range(lo, lo + frame_number)]


def side_info_index(j):
    """The reference reads the side information of frame max(1, j): frame 0 has none (test_LD_37.py:36,54,67,155)."""
    return max(1, j)


def new_frame_of_step(i, n_frames):
    """Index of the one frame that enters the window at step i >= 1 (= last entry of generate_input_index)."""
    return min(i + 3, n_frames - 1)


class Sequence:
    """One coded sequence as the reference stores it on disk, held as integer arrays.

    lr, pm, unflt: uint8 [T, h, W];  res: integer [T, h, W] (first channel of *_res.npy);  mvl0: int8 / int32 [T, h, W, 3]
    (mv_a, mv_b, ref-distance);  gt: uint8 [T, 4h, 4W] or None.  Entry 0 of the side-information arrays is never read."""

    def __init__(self, lr, pm, res, unflt, mvl0, gt=None, name="seq"):
        self.lr = np.ascontiguousarray(lr, dtype=np.uint8)
        self.pm = np.ascontiguousarray(pm, dtype=np.uint8)
        self.unflt = np.ascontiguousarray(unflt, dtype=np.uint8)
        res = np.asarray(res)
        if not np.issubdtype(res.dtype, np.integer) or res.min(initial=0) < -32768 or res.max(initial=0) > 32767:
            raise ValueError("Sequence: residual maps must be integers within int16")
        self.res = np.ascontiguousarray(res, dtype=np.int16)
        mv = np.asarray(mvl0)
        if not np.issubdtype(mv.dtype, np.integer):
            raise ValueError("Sequence: mvl0 must be an integer array [T, h, W, 3]")
        small = mv.min(initial=0) >= -128 and mv.max(initial=0) <= 127
        self.mvl0 = np.ascontiguousarray(mv, dtype=np.int8 if small else np.int32)
        self.gt = None if gt is None else np.ascontiguousarray(gt, dtype=np.uint8)
        self.name = name
        T, h, W = self.lr.shape
        for a, what in ((self.pm, "pm"), (self.res, "res"), (self.unflt, "unflt")):
            if a.shape != (T, h, W):
                raise ValueError("Sequence: %s has shape %s, expected %s" % (what, a.shape, (T, h, W)))
        if self.mvl0.shape != (T, h, W, 3):
            raise ValueError("Sequence: mvl0 has shape %s, expected %s" % (self.mvl0.shape, (T, h, W, 3)))
        if self.gt is not None and self.gt.shape != (T, 4 * h, 4 * W):
            raise ValueError("Sequence: gt has shape %s, expected %s" % (self.gt.shape, (T, 4 * h, 4 * W)))

    @property
    def shape(self):
        return self.lr.shape

    @classmethod
    def from_directory(cls, lr_dir, side_dir, gt_dir=None, name=None):
        """Reads the reference's on-disk layout (test_LD_37.py:131-160): `lr_dir/<sorted frames>.png`,
        `side_dir/{part_m/%05d_M_mask.png, res/%05d_res.npy, unfiltered/%05d_unflt.png, mvl0/%05d_mvl0.npy}` and, optionally,
        `gt_dir/%05d.png` (metric/psnr_ssim.py:456-458).  Frame 0 has no side information; its slots repeat frame 1's."""
        import cv2
        files = sorted(f for f in os.listdir(lr_dir) if f.lower().endswith(".png"))
        if not files:
            raise FileNotFoundError("no PNG frames under %s" % lr_dir)

        def grey(path):
            img = cv2.imread(path, 0)
            if img is None:
                raise FileNotFoundError(path)
            return img

        lr = np.stack([grey(os.path.join(lr_dir, f)) for f in files])
        T = len(files)
        idx = ["%05d" % side_info_index(i) for i in range(T)]
        pm = np.stack([grey(os.path.join(side_dir, "part_m", k + "_M_mask.png")) for k in idx])
        unflt = np.stack([grey(os.path.join(side_dir, "unfiltered", k + "_unflt.png")) for k in idx])
        res = np.stack([np.load(os.path.join(side_dir, "res", k + "_res.npy"))[:, :, 0] for k in idx])
        mv = np.stack([np.load(os.path.join(side_dir, "mvl0", k + "_mvl0.npy")) for k in idx])
        gt = None
        if gt_dir is not None:
            gt = np.stack([grey(os.path.join(gt_dir, "%05d.png" % i)) for i in range(T)])
            gt = gt[:, :4 * lr.shape[1], :4 * lr.shape[2]]          # cal_psnr_ssim crops both to the common size (:460-466)
        return cls(lr, pm, res, unflt, mv, gt, name or os.path.basename(os.path.normpath(lr_dir)))


def padded_rows(h):
    """LR rows the model runs on: the reference appends 2 zero rows to 270-row frames (test_LD_37.py:24-26); in general
    the next multiple of 8 (CVSR_V8 needs H % 8 == 0)."""
    return (h + 7) // 8 * 8


def noise_for(seed, seq_ids, frame, H, W, device):
    """Six [S, 64, H, W] uniform tensors (neighbour order 0,1,2,4,5,6) keyed by (seed, sequence id, frame, neighbour); `frame` is
    one index for every sequence or one per sequence."""
    frames = [frame] * len(seq_ids) if isinstance(frame, int) else list(frame)
    g = torch.Generator(device=device)
    out = []
    for nb in NEIGHBOURS:
        per_seq = []
        for sid, f in zip(seq_ids, frames):
            g.manual_seed(sharding.noise_key(seed, sid, f, nb))
            per_seq.append(torch.rand((64, H, W), device=device, generator=g))
        out.append(torch.stack(per_seq).clamp_min_(1e-12))   # the reference redraws while any u == 0 (arch:2170-2171)
    return out


class Step(NamedTuple):
    """One model step of a slot schedule: `first` = the step runs the first-frame path (pre_L1_fea=None) on every slot; `slots` =
    per slot (item index, output frame, admitted) or None for an idle slot."""
    first: bool
    slots: tuple


def slot_schedule(ranges, slots):
    """The steps that run the items with output frame ranges `ranges` = [(lo, hi), ...] (queue order) on `slots` slots.

    A batch of min(slots, queued) items starts together through the first-frame path.  A slot whose item ended takes the next queued
    item at the next step (an admission: its window is loaded with W(lo)'s frames and features, and the step runs as a steady-state
    one); with the queue empty it idles (keeps stepping its last window, its output is dropped).  When every slot's item ends at the
    same step, the next batch starts through the first-frame path again: items of equal length give exactly the batches of
    `slots` items, in order, that running them batch by batch gives."""
    ranges = [(int(lo), int(hi)) for lo, hi in ranges]
    if slots <= 0 or any(not 0 <= lo < hi for lo, hi in ranges):
        raise ValueError("slot_schedule: bad arguments")
    steps, queue, n = [], 0, len(ranges)
    while queue < n:
        S = min(slots, n - queue)
        cur = list(range(queue, queue + S))
        queue += S
        frame = [ranges[k][0] for k in cur]
        admitted = [False] * S
        first = True
        while True:
            steps.append(Step(first, tuple(None if cur[s] is None else (cur[s], frame[s], admitted[s]) for s in range(S))))
            first = False
            ended = []
            for s in range(S):
                admitted[s] = False
                if cur[s] is not None:
                    frame[s] += 1
                    if frame[s] == ranges[cur[s]][1]:
                        cur[s] = None
                        ended.append(s)
            if all(c is None for c in cur):
                break
            for s in ended:
                if queue < n:
                    cur[s], frame[s], admitted[s] = queue, ranges[queue][0], True
                    queue += 1
    return steps


_PLANES = (("x", "lr"), ("pms", "pm"), ("rms", "res"), ("ufs", "unflt"))


class _Staging:
    """One slot of pinned host staging + device landing buffers for the new frames of a step: the new frame of every batch slot, and
    the six window frames W(lo)[0:6] of the slots that admit an item at that step (`adm`, copied only for those slots)."""

    def __init__(self, S, h, H, W, mv_dtype, with_gt, device):
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()   # noqa: E731
        self.host = {"lr": pin((S, h, W), torch.uint8), "pm": pin((S, h, W), torch.uint8), "unflt": pin((S, h, W), torch.uint8),
                     "res": pin((S, h, W), torch.int16), "mv": pin((S, H, W, 3), mv_dtype), "imax": pin((S, 2), torch.int32)}
        self.host["mv"].zero_()                                    # padded rows: mv = refdist = 0 -> 0 / -0 = NaN -> flow 0
        if with_gt:
            self.host["gt"] = pin((S, 4 * h, 4 * W), torch.uint8)
        self.dev = {k: torch.empty_like(v, device=device) for k, v in self.host.items()}
        self.adm_host = {"lr": pin((S, 6, h, W), torch.uint8), "pm": pin((S, 6, h, W), torch.uint8),
                         "unflt": pin((S, 6, h, W), torch.uint8), "res": pin((S, 6, h, W), torch.int16)}
        self.adm_dev = {k: torch.empty_like(v, device=device) for k, v in self.adm_host.items()}
        self.ready = torch.cuda.Event()      # recorded on the copy stream after the H2D copies
        self.consumed = torch.cuda.Event()   # recorded on the compute stream after the landing buffers were read
        self.used = False


class FrameDriver:
    """driver = FrameDriver(model); result = driver.run(sequences, seq_ids)

    `model` is a cdfo_b200.model.CVSR_V8 on a CUDA device in eval mode.  `run` processes sequences of equal frame size (h, W), of any
    lengths, frame by frame on `slots` batch slots (default: one per sequence) and returns {"psnr": [..], "ssim": [..], "frames": T of
    the longest sequence, "sums": float64 [S, 3] (device), and the slot counts of run_items}; `sink`, when given, is called as
    sink(batch_index, frame_index, uint8 ndarray [4h, 4W]) for every SR frame, one step late, in frame order per sequence.
    `run_items` runs a queue of work items (sharding.WorkItem) with the slot schedule of `slot_schedule`."""

    def __init__(self, model, seed=0, crop_border=4, graph=False):
        self.model, self.seed, self.crop_border, self.use_graph = model, int(seed), int(crop_border), bool(graph)
        self.device = next(model.parameters()).device
        if self.device.type != "cuda":
            raise NotImplementedError("cdfo_b200.FrameDriver is CUDA-only (no CPU fallback)")
        self.copy_stream = torch.cuda.Stream(self.device)
        self._graphed = None

    # ------------------------------------------------------------------ host side of one step
    @staticmethod
    def _fill(buf, state, items, qs, h):
        """Host staging of one step: per slot the new frame of its window, the MV field / GT of its output frame, its (i, T) for the
        end-of-sequence fix-up and, on an admission, the six window frames W(lo)[0:6]."""
        for s, (k, i, admit, _live) in enumerate(state):
            q = qs[items[k].seq]
            T = q.shape[0]
            f = new_frame_of_step(i, T)
            m = side_info_index(f)
            buf.host["lr"][s].copy_(torch.from_numpy(q.lr[f]))
            buf.host["pm"][s].copy_(torch.from_numpy(q.pm[m]))
            buf.host["res"][s].copy_(torch.from_numpy(q.res[m]))
            buf.host["unflt"][s].copy_(torch.from_numpy(q.unflt[m]))
            buf.host["mv"][s, :h].copy_(torch.from_numpy(q.mvl0[side_info_index(i)]))
            buf.host["imax"][s, 0], buf.host["imax"][s, 1] = i, T
            if "gt" in buf.host:
                buf.host["gt"][s].copy_(torch.from_numpy(q.gt[i]))
            if admit:
                for p, j in enumerate(generate_input_index(i, 7, T - 1)[:6]):
                    buf.adm_host["lr"][s, p].copy_(torch.from_numpy(q.lr[j]))
                    for key in ("pm", "res", "unflt"):
                        buf.adm_host[key][s, p].copy_(torch.from_numpy(getattr(q, key)[side_info_index(j)]))

    def _upload(self, buf, admitted):
        cs = self.copy_stream
        if buf.used:
            cs.wait_event(buf.consumed)
        with torch.cuda.stream(cs):
            for k, v in buf.host.items():
                buf.dev[k].copy_(v, non_blocking=True)
            for s in admitted:
                for k, v in buf.adm_host.items():
                    buf.adm_dev[k][s].copy_(v[s], non_blocking=True)
            buf.ready.record(cs)
        buf.used = True

    # ------------------------------------------------------------------ the loop
    @torch.no_grad()
    def run(self, sequences, seq_ids=None, sink=None, slots=None):
        seqs = list(sequences)
        S = len(seqs)
        if S == 0:
            raise ValueError("FrameDriver.run: no sequences")
        h, W = seqs[0].shape[1:]
        if any(tuple(q.shape[1:]) != (h, W) for q in seqs):
            raise ValueError("FrameDriver.run: the sequences of one run must share the frame size (rows, columns)")
        seq_ids = list(range(S)) if seq_ids is None else list(seq_ids)
        items = [sharding.WorkItem(k, 0, q.shape[0]) for k, q in enumerate(seqs)]
        r = self.run_items(seqs, items, S if slots is None else int(slots), sink=sink, noise_ids=seq_ids)
        sums = r.pop("item_sums")                       # one item per sequence, in sequence order
        res = dict(r, frames=max(q.shape[0] for q in seqs), sums=sums, psnr=None, ssim=None)
        if all(q.gt is not None for q in seqs):
            host = sums.cpu()
            res["psnr"] = (host[:, 0] / host[:, 2]).tolist()       # mean of the per-frame values (metric/psnr_ssim.py:477-481)
            res["ssim"] = (host[:, 1] / host[:, 2]).tolist()
        return res

    @torch.no_grad()
    def run_items(self, sequences, items, slots, sink=None, noise_ids=None):
        """Runs the work items `items` (sharding.WorkItem, all of one frame size; `sequences[item.seq]` is the sequence) on `slots`
        batch slots in queue order (slot_schedule).  sink(item.seq, frame, img) is called once per output frame, in frame order
        within an item.  The Gumbel noise of a frame is keyed by noise_ids[item.seq] (default item.seq).  Returns {"item_sums":
        float64 [len(items), 3] (device) = (sum of per-frame PSNR, SSIM, frames) per item (zero without ground truth), "steps",
        "slot_steps", "idle_slot_steps", "admissions"}."""
        items = [sharding.WorkItem(*it) for it in items]
        if not items:
            raise ValueError("FrameDriver.run_items: no items")
        qs = {}
        for it in items:
            if it.seq not in qs:
                qs[it.seq] = sequences[it.seq]
        h, W = qs[items[0].seq].shape[1:]
        if any(tuple(q.shape[1:]) != (h, W) for q in qs.values()):
            raise ValueError("FrameDriver.run_items: the items of one run must share the frame size (rows, columns)")
        if W % 8:
            raise ValueError("FrameDriver.run: frame width must be a multiple of 8 (got %d)" % W)
        if any(not 0 <= it.lo < it.hi <= qs[it.seq].shape[0] for it in items):
            raise ValueError("FrameDriver.run_items: an item's frame range lies outside its sequence")
        noise_ids = {k: (k if noise_ids is None else noise_ids[k]) for k in qs}
        with_gt = all(q.gt is not None for q in qs.values())
        # int32 staging if any sequence carries int32 MVs; int8 fields are widened by the staging copy itself (the caller's
        # Sequence objects are never modified)
        mv_dtype = torch.int32 if any(q.mvl0.dtype == np.int32 for q in qs.values()) else torch.int8
        item_sums = torch.zeros((len(items), 3), dtype=torch.float64, device=self.device)
        stats = {"steps": 0, "slot_steps": 0, "idle_slot_steps": 0, "admissions": 0}
        steps = slot_schedule([(it.lo, it.hi) for it in items], slots)
        ring_before = self.model.feature_ring
        self.model.feature_ring = not self.use_graph      # eager steps keep the window's L1 features in a ring (model.FeatureRing)
        try:
            b0 = 0
            for b1 in range(1, len(steps) + 1):
                if b1 == len(steps) or steps[b1].first:
                    self._batch(steps[b0:b1], items, qs, noise_ids, sink, item_sums, with_gt, mv_dtype, h, W, stats)
                    b0 = b1
        finally:
            self.model.feature_ring = ring_before       # also on an exception mid-sequence: later plain callers must not get ring handles
        return dict(stats, item_sums=item_sums)

    def _batch(self, steps, items, qs, noise_ids, sink, item_sums, with_gt, mv_dtype, h, W, stats):
        """One batch of the schedule: steps[0] is its first-frame step, the slot count is fixed."""
        S = len(steps[0].slots)
        state, last = [], [None] * S          # per step and slot: (item, frame, admitted, live); an idle slot repeats its last entry
        for st in steps:
            row = []
            for s, e in enumerate(st.slots):
                if e is not None:
                    last[s] = e
                row.append((e[0], e[1], e[2], True) if e is not None else (last[s][0], last[s][1], False, False))
            state.append(row)
        dev, H = self.device, padded_rows(h)
        main = torch.cuda.current_stream(dev)
        bufs = [_Staging(S, h, H, W, mv_dtype, with_gt, dev) for _ in range(2)]
        out_u8 = [torch.empty((S, 4 * h, 4 * W), dtype=torch.uint8, device=dev) for _ in range(2)]
        out_host = [torch.empty((S, 4 * h, 4 * W), dtype=torch.uint8).pin_memory() for _ in range(2)]
        out_done = [torch.cuda.Event() for _ in range(2)]
        out_ready = [torch.cuda.Event() for _ in range(2)]
        acc = torch.zeros((S, 3), dtype=torch.float64, device=dev)     # metric sums of the item each slot holds

        # ---- first window: frames W(lo) of every plane (test_LD_37.py:143-155), converted on the device
        windows = [generate_input_index(i, 7, qs[items[k].seq].shape[0] - 1) for k, i, _, _ in state[0]]

        def window_of(get):
            host = torch.from_numpy(np.stack([np.stack([get(qs[items[k].seq], j) for j in o])
                                              for (k, _, _, _), o in zip(state[0], windows)]))
            return metrics.planes_to_unit(host.to(dev), H).unsqueeze(2)          # [S, 7, 1, H, W]

        win = {"x": window_of(lambda q, j: q.lr[j]), "pms": window_of(lambda q, j: q.pm[side_info_index(j)]),
               "rms": window_of(lambda q, j: q.res[side_info_index(j)]), "ufs": window_of(lambda q, j: q.unflt[side_info_index(j)])}
        self._fill(bufs[0], state[0], items, qs, h)       # step 0 needs only the MV field (+ GT) and (i, T) from its staging
        self._upload(bufs[0], [])
        l1, pending = None, None
        for t in range(len(steps)):
            buf = bufs[t % 2]
            if t + 1 < len(steps):                          # stage step t+1 while step t computes
                nxt = bufs[(t + 1) % 2]
                if nxt.used:
                    nxt.ready.synchronize()                 # its previous H2D finished: the pinned buffers may be rewritten
                self._fill(nxt, state[t + 1], items, qs, h)
                self._upload(nxt, [s for s, e in enumerate(state[t + 1]) if e[2]])
            main.wait_event(buf.ready)
            if t > 0:
                for s, (k, i, admit, _) in enumerate(state[t]):
                    if admit:
                        self._admit(win, l1, s, buf, generate_input_index(i, 7, qs[items[k].seq].shape[0] - 1)[:6], H)
                        acc[s].zero_()
                new = {key: metrics.planes_to_unit(buf.dev[plane], H) for key, plane in _PLANES}
                for key in win:
                    win[key] = torch.cat([win[key][:, 1:], new[key].view(S, 1, 1, H, W)], 1)
            mvs = torch.cat([priors.mv2mvs(buf.dev["mv"][s]) for s in range(S)], 0)
            priors.modify_mv_for_end_frames_batched(mvs, buf.dev["imax"])
            noise = noise_for(self.seed, [noise_ids[items[k].seq] for k, _, _, _ in state[t]], [i for _, i, _, _ in state[t]], H, W, dev)
            if l1 is None:
                sr, l1 = self.model(win["x"], None, mvs, win["pms"], win["rms"], win["ufs"], None, noise=noise)
            elif self.use_graph:
                if self._graphed is None or self._graphed.static_in[0].shape != win["x"].shape:
                    self._graphed = GraphedStep(self.model, win["x"], mvs, win["pms"], win["rms"], win["ufs"], l1, noise)
                sr, l1 = self._graphed(win["x"], mvs, win["pms"], win["rms"], win["ufs"], l1, noise)
            else:
                sr, l1 = self.model(win["x"], None, mvs, win["pms"], win["rms"], win["ufs"], l1, noise=noise)
            o = t % 2
            if t >= 2 and sink is not None:
                main.wait_event(out_done[o])                      # the D2H of step t-2 has left this buffer
            metrics.sr_to_u8(sr.reshape(S, 4 * H, 4 * W), 4 * h, out=out_u8[o])
            if with_gt:
                metrics.psnr_ssim(out_u8[o], buf.dev["gt"], self.crop_border, accum=acc)
            live = [(s, items[k].seq, i) for s, (k, i, _, alive) in enumerate(state[t]) if alive]
            for s, (k, i, _, alive) in enumerate(state[t]):
                if alive and i == items[k].hi - 1:
                    item_sums[k].copy_(acc[s])
            stats["steps"] += 1
            stats["slot_steps"] += S
            stats["idle_slot_steps"] += S - len(live)
            stats["admissions"] += sum(1 for e in state[t] if e[2])
            buf.consumed.record(main)
            out_ready[o].record(main)
            if sink is not None:
                cs = self.copy_stream
                cs.wait_event(out_ready[o])
                with torch.cuda.stream(cs):
                    out_host[o].copy_(out_u8[o], non_blocking=True)
                    out_done[o].record(cs)
                if pending is not None:                 # deliver the previous frame while this one computes
                    self._deliver(sink, pending, out_host, out_done)
                pending = (o, live)
        if sink is not None and pending is not None:
            self._deliver(sink, pending, out_host, out_done)
        torch.cuda.current_stream(dev).synchronize()

    def _admit(self, win, l1, s, buf, frames, H):
        """Admission into slot s before the step shifts in frame W(lo)[6]: the planes of W(lo)[0:6] go to window positions 1..6 and
        their L1 features (computed once per distinct frame: W(0) repeats frame 0) to the pre-push window positions 1..6."""
        for key, plane in _PLANES:
            win[key][s, 1:] = metrics.planes_to_unit(buf.adm_dev[plane][s], H).unsqueeze(1)
        distinct = sorted(set(frames))
        first = [frames.index(j) for j in distinct]
        pick = lambda t: torch.cat([t[s, 1 + p:2 + p] for p in first], 0)   # noqa: E731   [n, 1, H, W] (slices: no index tensor)
        self.model.load_window_features(l1, s, pick(win["x"]), pick(win["pms"]), [distinct.index(j) for j in frames])

    @staticmethod
    def _deliver(sink, pending, out_host, out_done):
        o, live = pending
        out_done[o].synchronize()
        for s, seq, i in live:
            sink(seq, i, out_host[o][s].numpy().copy())


def run_sharded(model, sequences, batch=4, seed=0, crop_border=4, graph=False, sink=None, group=None, split=False, shapes=None):
    """Evaluates `sequences` (the full, rank-independent list; sequences of any frame sizes and lengths) over all ranks of the process
    group and returns the per-sequence PSNR / SSIM on every rank.  No collective on the data path.

    The job is a list of work items (sharding.partition_items): by default one per sequence, rank r owning the contiguous block
    sharding.sequence_shard gives it; with split=True, sequences are cut into frame ranges balanced by cost over every slot of every
    rank (one long sequence then runs on all of them), which needs the (T, h, W) of every sequence: `shapes`, else
    `sequences.shape_of(k)` when the list has it, else `sequences[k].shape`.  A rank loads only the sequences its items touch.  Its
    items run in groups of one frame size, one group after another, each on `batch` slots of a FrameDriver (run_items), longest item
    first (items of equal length keep their order, so equal sequences run in today's batches).  One
    all_reduce of the [n_items, 3] fp64 per-item sums (sharding.gather_metrics) and a sum of each sequence's items in item order give
    results that do not depend on the world size or the slot assignment.

    sink(seq_id, frame, img) is called exactly once per output frame.  Frames of one item arrive in order; the items of a split
    sequence run on different slots and ranks, so across items a sequence's frames may arrive out of order."""
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    n = len(sequences)
    if split:
        if shapes is None:
            shape_of = getattr(sequences, "shape_of", None) or (lambda k: sequences[k].shape)
            shapes = [shape_of(k) for k in range(n)]
        items, ranks = sharding.partition_items(shapes, world, batch, split=True)
        mine = [j for j, r in enumerate(ranks) if r == rank]
        item_seqs = [it.seq for it in items]
    else:
        own = sharding.sequence_items(n, world, rank, lambda k: sequences[k].shape[0])
        items = [None] * n
        for it in own:
            items[it.seq] = it
        mine = [it.seq for it in own]                  # item j is sequence j
        item_seqs = list(range(n))
    drv = FrameDriver(model, seed=seed, crop_border=crop_border, graph=graph)
    sums = torch.zeros((len(items), 3), dtype=torch.float64, device=drv.device)
    stats = {"steps": 0, "slot_steps": 0, "idle_slot_steps": 0, "admissions": 0}
    groups = {}
    for j in mine:
        groups.setdefault(tuple(sequences[items[j].seq].shape[1:]), []).append(j)
    for js in groups.values():
        js.sort(key=lambda j: items[j].lo - items[j].hi)   # longest first (stable): a short item refills the slot that frees first
        r = drv.run_items(sequences, [items[j] for j in js], batch, sink=sink)
        for row, j in enumerate(js):
            sums[j] = r["item_sums"][row]
        for k in stats:
            stats[k] += r[k]
    sums = sharding.gather_metrics(sums, group)
    host = sharding.sequence_sums(sums, item_seqs, n)
    cnt = host[:, 2].clamp_min(1.0)
    return dict(stats, psnr=(host[:, 0] / cnt).tolist(), ssim=(host[:, 1] / cnt).tolist(), frames=host[:, 2].tolist(),
                sums=host.to(drv.device), items=len(items))
