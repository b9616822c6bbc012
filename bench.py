#!/usr/bin/env python
"""Benchmark of the CDFO hot path on B200: HR frames/s of CVSR_V8 (DCN alignment variant) at 1080p x4.

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host CPU cores

A step = one HR output frame for each of the `--seqs` independent sequences resident on a GPU: the sliding
7-frame window advances by one frame (steady state: cached L1 features, one new frame of feature extraction,
six neighbour alignments, fusion, trunk, x4 tail).  Workload = BASELINE.json configs[2]: JCT-VC Class-B-shaped
clips, 7 x (480x270 LR, zero-padded to 272 rows) -> 1920x1080(+8) HR, LD priors, synthetic data, seeded weights.
N > 1 shards independent sequences over the ranks (weak scaling, no collective on the data path; one NCCL
all_reduce of the per-rank frame counts / checksums at the end = the PSNR/SSIM gather of the real pipeline).

One JSON line on rank 0:
  value     whole-job HR frames/s with inputs resident in HBM (device-timed, max over ranks)
  e2e       the same through the public API from pinned HOST buffers: H2D of the new LR frame + priors of the
            step, forward, D2H of the uint8 SR frame, all inside the timed region
  roofline  the tcgen05 DCN kernel: algorithmic bytes (SURVEY 8d: x + offset + mask + y per LR pixel and
            neighbour call, at the I/O widths the kernel was given) / live CUDA-event duration vs measured HBM peak
  cpu_baseline  oracle port (oracle/torch_ref.py) of the same forward on the host cores, bounded sample
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "HR frames/sec, 1080p x4 LD-QP37"
UNIT = "frames/s"
LR_H, LR_W = 272, 480            # 270 rows + 2 zero rows (test_LD_37.py:24-26)
ALGO_BYTES_PER_PX_BF16 = 1120    # SURVEY.md 8(d): x 128 + offset 576 + mask 288 + y 128 (2-byte I/O)  [DCN-only kernel]
FUSED_FLOP_PER_PX = 2 * 497664 + 73728   # SURVEY.md 8(d) row 3: last head conv x 2 + offset assembly + DCN, fused
FUSED_BYTES_PER_PX = 516                 # 2 hidden maps 256 + x 128 + flow 4 + y 128


def workload(args):
    """config.workload: identical in both arms (ours and --impl reference) -- BASELINE.json configs[2]."""
    return ("CVSR_V8+MVDualAttAlignment (%s), 7x(480x270->272 rows) LR -> 1920x1080 HR, %s priors, steady state (cached L1_fea)"
            % (args.variant, args.priors))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower() == "active"})
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_frames(hw, steps, warmup, budget_s, variant="O2"):
    """The reference's algorithm (oracle/torch_ref.py: fp32 torch CPU ops + torchvision's CPU deform_conv2d, 0-diff against the real
    reference at this very configuration, tests/golden/model_c3_golden.npz `port_err`) on the host cores: FULL steady-state frames
    of one sequence at LR size `hw` -- nothing is cropped or extrapolated.  One untimed first frame builds the L1 cache, then up to
    `warmup` untimed and `steps` timed cached frames, stopping early once `budget_s` seconds are spent (at least one timed frame).
    Returns (list of seconds per timed frame, warm-ups done, cores)."""
    import torch
    from cdfo_b200 import synthetic
    from oracle import priors_ref, torch_ref
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    H, W = hw
    from cdfo_b200.model import CVSR_V8
    tmpl = CVSR_V8(alignment="mv_dcn" if variant == "O2" else "dual_att").state_dict()
    sd = synthetic.seeded_state_dict(tmpl, seed=4)
    clip = synthetic.make_clip(1, H, W, 1)
    mvs = torch.from_numpy(priors_ref.mv2mvs_model_layout(clip["mv_l0"][0].numpy()))
    noise = synthetic.gumbel_uniforms(4, 0, 0, 1, H, W)
    t_start = time.perf_counter()
    times, warm_done = [], 0
    with torch.no_grad():
        _, l1 = torch_ref.cvsr_v8_forward(sd, clip["x"], mvs, clip["pms"], clip["rms"], clip["ufs"], None, noise, variant)
        first = time.perf_counter() - t_start
        est = first
        while len(times) < steps:
            spent = time.perf_counter() - t_start
            timed = warm_done >= warmup or spent + 2.0 * est > budget_s     # out of budget for more warm-up: time this one
            if times and spent + est > budget_s:
                break
            t0 = time.perf_counter()
            _, l1 = torch_ref.cvsr_v8_forward(sd, clip["x"], mvs, clip["pms"], clip["rms"], clip["ufs"], l1, noise, variant)
            est = time.perf_counter() - t0
            if timed:
                times.append(est)
            else:
                warm_done += 1
    return times, warm_done, cores, first


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H, W = args.lr_h, args.lr_w
    times, warm_done, cores, first = cpu_reference_frames((H, W), max(1, args.steps), max(0, args.warmup), args.cpu_budget_s, args.variant)
    sec = sum(times) / len(times)
    fps = 1.0 / sec
    capped = len(times) < args.steps or warm_done < args.warmup
    sample = ("oracle port (oracle/torch_ref.py, fp32, torch CPU ops + torchvision deform_conv2d; equals the real reference to 0 diff at "
              "this configuration) of the steady-state forward on FULL %dx%d LR frames of one sequence: %d timed frame(s) after %d "
              "warm-up(s) (+ one cache-building first frame, %.1f s), %.2f s per frame (min %.2f, max %.2f)%s"
              % (H, W, len(times), warm_done, first, sec, min(times), max(times),
                 "; --steps %d / --warmup %d were cut by the %d s time cap (--cpu-budget-s)" % (args.steps, args.warmup, args.cpu_budget_s) if capped else ""))
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": warm_done, "steps_requested": args.steps, "warmup_requested": args.warmup, "time_capped": capped,
        "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload(args), "lr": [H, W], "host": "CPU",
                   "step": "one HR frame of one sequence (the CPU path has no batch to amortise; ours steps %d sequences at once)" % args.seqs},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.gpus > 1:
        line["config"]["note"] = "the CPU arm runs on rank 0's host only: value is ONE host, not multiplied by n_gpus"
    print(json.dumps(line), flush=True)


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per LR pixel of the roofline kernel, read from the newest per-round capture summary
    profiles/r??_roofline_kernel_traffic.json (written by tools/ncu_traffic.py from an `ncu --set full` .ncu-rep).  No constant in
    this file: a missing summary fails loudly."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r??_roofline_kernel_traffic.json")))
    if not files:
        raise SystemExit("bench.py: no profiles/r??_roofline_kernel_traffic.json (run tools/ncu_traffic.py on this round's ncu capture)")
    d = json.load(open(files[-1]))
    return d, os.path.relpath(files[-1], ROOT)


# --dump-outputs: at most 56 MB in all, so that two builds can be compared file by file
DUMP_CAP_BYTES = {"sr": 40_000_000, "l1_features": 16_000_000}


def dump_outputs(out_dir, arrays):
    """Writes each tensor of `arrays` as out_dir/<name>.npy in float32.  A tensor larger than its DUMP_CAP_BYTES entry is written
    as a 1-D sample instead: the elements at the sorted flat indices numpy.random.default_rng(0) draws without replacement, which
    depend only on the tensor's size and so are the same in every run with the same arguments."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.float()
        cap = DUMP_CAP_BYTES[name] // 4
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import cdfo_b200
    from cdfo_b200 import dcn_sm100, synthetic
    from cdfo_b200.model import CVSR_V8

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL writes its version banner (NCCL_DEBUG=VERSION / WARN) to STDOUT: send its log to stderr, stdout is the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    assert cdfo_b200._lib.lib().cdfo_device_ok(local) == 1, "not an sm_100 device"

    H, W, S = args.lr_h, args.lr_w, args.seqs
    model = CVSR_V8(alignment="mv_dcn" if args.variant == "O2" else "dual_att")
    model.load_state_dict(synthetic.seeded_state_dict(model.state_dict(), seed=4), strict=True)
    model = model.to(dev).eval()
    model.lowp = torch.bfloat16

    # a pool of distinct windows per rank (sequence ids are global: rank r owns sequences r*S .. r*S+S-1)
    pool = []
    for wdx in range(args.pool):
        clip = synthetic.make_clip(1000 * (rank * S) + wdx, H, W, S, config=args.priors)
        host = {k: clip[k].pin_memory() for k in ("x", "pms", "rms", "ufs")}
        host["mv"] = clip["mv_l0"].pin_memory()
        if args.priors == "RA":
            host["mv1"] = clip["mv_l1"].pin_memory()
        pool.append(host)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    noise = [torch.rand((S, 64, H, W), device=dev, generator=g).clamp_min_(1e-12) for _ in range(6)]
    if not args.graph:
        # eager steps: the window's L1 features live in a frame-major ring (model.FeatureRing: no per-frame copy of the 7-frame cache)
        # and the six noise tensors are handed over as one neighbour-major batch
        model.feature_ring = True
        noise = torch.cat(noise, 0)

    def decode_mv(mv_dev, mv1_dev=None):
        if mv1_dev is not None:      # config c5: bidirectional decoding of the (l0, l1) pair (opt/data_RA_bi.py:496-533)
            return torch.cat([cdfo_b200.mv2mvs_ra(mv_dev[s], mv1_dev[s]) for s in range(S)], 0)
        return torch.cat([cdfo_b200.mv2mvs(mv_dev[s]) for s in range(S)], 0)

    resident = []
    for host in pool:
        d = {k: host[k].to(dev) for k in ("x", "pms", "rms", "ufs")}
        d["mvs"] = decode_mv(host["mv"].to(dev), host["mv1"].to(dev) if "mv1" in host else None)
        resident.append(d)
    _, l1 = model(resident[0]["x"], None, resident[0]["mvs"], resident[0]["pms"], resident[0]["rms"], resident[0]["ufs"],
                  None, noise=noise)

    # the steady-state step replayed as ONE CUDA graph (cdfo_b200/graph.py: bit-identical outputs, no host work between the ~330
    # launches of a step); --graph 0 times the eager launch sequence instead
    graphed = None
    if args.graph:
        from cdfo_b200.graph import GraphedStep
        d0 = resident[0]
        graphed = GraphedStep(model, d0["x"], d0["mvs"], d0["pms"], d0["rms"], d0["ufs"], l1, noise)

    def forward(x, mvs, pms, rms, ufs, l1):
        if graphed is not None:
            return graphed(x, mvs, pms, rms, ufs, l1)
        return model(x, None, mvs, pms, rms, ufs, l1, noise=noise)

    def step_resident(i, l1):
        d = resident[i % len(resident)]
        return forward(d["x"], d["mvs"], d["pms"], d["rms"], d["ufs"], l1)

    # e2e: per step only the NEW frame of the window and its priors cross PCIe (the other six are already resident,
    # exactly like the reference's sliding window would allow); SR leaves as uint8 like cv2.imwrite gets it.
    win = {k: resident[0][k].clone() for k in ("x", "pms", "rms", "ufs")}
    sr_host = torch.empty((S, 1, 4 * H - 8, 4 * W), dtype=torch.uint8).pin_memory()
    h2d = sum(pool[0][k][:, -1:].numel() * 4 for k in ("x", "pms", "rms", "ufs")) + pool[0]["mv"].numel() * (2 if args.priors == "RA" else 1)
    d2h = sr_host.numel()

    # Double-buffered like cdfo_b200.driver.FrameDriver: the H2D copies of step i + 1 run on a copy stream underneath the kernels of step i
    # (contiguous pinned sources, device staging buffers guarded by events), the uint8 SR frame of step i leaves on a third stream while
    # step i + 1 computes.  Every timed step still issues one H2D set and one D2H inside the timed region (the final synchronize waits
    # for all of them).
    main_s, copy_s, d2h_s = torch.cuda.current_stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    new_host = []
    for host in pool:
        nh = {k: host[k][:, -1:].contiguous().pin_memory() for k in ("x", "pms", "rms", "ufs")}
        nh["mv"] = host["mv"]
        if "mv1" in host:
            nh["mv1"] = host["mv1"]
        new_host.append(nh)
    stage = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in new_host[0].items()} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    sr_hosts = [sr_host, torch.empty_like(sr_host).pin_memory()]
    issued = [None]

    def issue(i):
        j = i % 2
        copy_s.wait_event(consumed[j])            # the kernels that read this staging buffer two steps ago are done
        with torch.cuda.stream(copy_s):
            for k, v in new_host[i % len(pool)].items():
                stage[j][k].copy_(v, non_blocking=True)
            ready[j].record(copy_s)
        issued[0] = i

    def step_e2e(i, l1):
        if issued[0] != i:                        # first step of a run: nothing was prefetched for it
            issue(i)
        j = i % 2
        main_s.wait_event(ready[j])
        st = stage[j]
        for k in ("x", "pms", "rms", "ufs"):
            win[k] = torch.cat([win[k][:, 1:], st[k]], 1)
        mvs = decode_mv(st["mv"], st.get("mv1"))
        consumed[j].record(main_s)
        issue(i + 1)
        sr, l1 = forward(win["x"], mvs, win["pms"], win["rms"], win["ufs"], l1)
        out8 = cdfo_b200.sr_to_u8(sr, 4 * H - 8)                        # crop 1088 -> 1080 rows, clamp, x255, truncate (test_LD_37.py:172-178)
        done = torch.cuda.Event()
        done.record(main_s)
        d2h_s.wait_event(done)
        with torch.cuda.stream(d2h_s):
            sr_hosts[j].copy_(out8, non_blocking=True)
        out8.record_stream(d2h_s)
        return sr, l1

    last_sr = [None]

    def timed(step_fn, steps, warmup, l1, log_dcn):
        for i in range(warmup):
            _, l1 = step_fn(i, l1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if log_dcn:
            dcn_sm100.event_log = []
        launches0 = cdfo_b200._lib.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            last_sr[0], l1 = step_fn(warmup + i, l1)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        log, dcn_sm100.event_log = dcn_sm100.event_log, None
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, l1, cdfo_b200._lib.launch_count - launches0, log

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, l1, launches, dcn_log = timed(step_resident, args.steps, args.warmup, l1, True)
    if args.dump_outputs and rank == 0:
        # what forward() returned in the last timed step, before the runs below overwrite the graph's static outputs; the feature
        # ring hands out its window frame-major, the cat path batch-major: written batch-major [seqs, 7, 64, H, W] either way
        feats = l1.reshape(7, S, *l1.shape[1:]).transpose(0, 1) if getattr(l1, "_cdfo_ring", None) else l1.reshape(S, 7, *l1.shape[1:])
        dump_outputs(args.dump_outputs, {"sr": last_sr[0], "l1_features": feats})
    if graphed is not None:
        # inside a replayed graph neither the ctypes launch counter nor the per-launch events exist: take both from eager steps
        keep, graphed = graphed, None
        _, l1, launches, dcn_log = timed(step_resident, args.steps, 1, l1, True)
        graphed = keep
    ms_e2e, l1, _, _ = timed(step_e2e, args.steps, max(1, args.warmup // 2), l1, False)
    clocks = sampler.stop() if rank == 0 else None

    # the end-of-job metric gather of the real pipeline (PSNR/SSIM sums, cdfo_b200/sharding.py): one tiny all_reduce of
    # [n_seq, 3] fp64 = (sum of squares of the last SR frame as the error stand-in, 0, frames produced) per owned sequence
    from cdfo_b200 import sharding
    sums = torch.zeros((world * S, 3), device=dev, dtype=torch.float64)
    own = sharding.sequence_shard(world * S, world, rank)
    sums[own[0]:own[-1] + 1, 0] = last_sr[0].double().pow(2).sum(dim=(1, 2, 3))
    sums[own[0]:own[-1] + 1, 2] = float(args.steps)
    sums = sharding.gather_metrics(sums)
    total_frames = float(sums[:, 2].sum().item())

    if rank == 0:
        hbm_peak, peak_src = peaks()
        traffic, traffic_src = ncu_traffic()
        durs = [a.elapsed_time(b) * 1e-3 for a, b, _, _ in dcn_log]           # seconds per launch
        px = dcn_log[0][2] if dcn_log else 0
        fused = bool(dcn_log) and dcn_log[0][3] == "fused"
        if ("fused" in traffic["kernel"]) != fused:      # a capture of another kernel says nothing about this one
            raise SystemExit("bench.py: %s holds the traffic of %s, not of the kernel this run reports; capture it (tools/ncu_traffic.py)"
                             % (traffic_src, traffic["kernel"]))
        avg = sum(durs) / max(1, len(durs))
        if fused:
            # the fused head + DCN alignment kernel: tensor-bound (SURVEY 8d row 3: 1 069 056 FLOP and 516 B per LR pixel and call)
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.isfile(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
            peak_tf = float(pk.get("bf16_tflops_sustained", 1400.0))
            achieved = FUSED_FLOP_PER_PX * px / avg / 1e12 if durs else 0.0
            roof = {
                "kernel": "mv_head_dcn_fused_sm100_kernel (conv_offset[-1] on both hidden maps 64->432 3x3 bf16 tcgen05 + tanh/sigmoid + MV prior "
                          "+ texture-gather DCNv2 64->64 3x3 dg=16 fp16 tcgen05 TS-form; offset/mask fields never in HBM)",
                "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": traffic["dram_bytes_per_px"] * px, "traffic_source": traffic_src,
                "peak_source": ("measured cuBLAS bf16, sustained figure for a kernel timed inside a long step (MEASURED_PEAKS.json); burst %.1f"
                                % pk["bf16_tflops"]) if pk else "fallback sustained figure (B200_PROFILING.md)",
                "frac_of_burst_peak": achieved / float(pk["bf16_tflops"]) if pk else None,
                "avg_launch_us": avg * 1e6, "launches_timed": len(durs), "algorithmic_flops_per_launch": FUSED_FLOP_PER_PX * px,
                "algorithmic_bytes_per_launch": FUSED_BYTES_PER_PX * px,
                "hbm_frac_of_same_launch": FUSED_BYTES_PER_PX * px / avg / 1e9 / hbm_peak if durs else None,
                "note": "algorithmic work = SURVEY 8d row 3: 2 x 497 664 (two evaluations of the 64->432 3x3 head) + 73 728 (DCN) FLOP and 516 B "
                        "(2 hidden maps 256 + x 128 + flow 4 + y 128) per LR pixel and neighbour call x %d px per launch; traffic = dram bytes per "
                        "px of this round's ncu --set full capture scaled to this launch; DESIGN.md 3.1" % px,
            }
        else:
            per_px = ALGO_BYTES_PER_PX_BF16
            achieved = per_px * px / avg / 1e9 if durs else 0.0
            kname = ("dcn_tex_sm100_kernel (tcgen05 implicit-GEMM DCNv2 64->64 3x3 dg=16, texture-unit gather)"
                     if cdfo_b200.config.dcn_gather == "tex" else "dcn_sm100_kernel (tcgen05 implicit-GEMM DCNv2, LDG gather)")
            roof = {
                "kernel": kname, "bound": "hbm",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic["dram_bytes_per_px"] * px,
                "traffic_source": traffic_src, "peak_source": peak_src, "avg_launch_us": avg * 1e6, "launches_timed": len(durs),
                "algorithmic_bytes_per_launch": per_px * px,
                "note": "two-kernel path (CDFO_FUSED_HEAD_DCN=0): algorithmic bytes = SURVEY 8d's 1120 B per LR pixel and neighbour call (x 128 + "
                        "offset 576 + mask 288 + y 128) x %d px per launch; the binding resource is the L1TEX data stage, DESIGN.md 3.1" % px,
            }
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            times, warm_done, cores, first = cpu_reference_frames((H, W), 3, 1, args.cpu_baseline_budget_s, args.variant)
            med = sorted(times)[len(times) // 2]
            cpu = {"value": 1.0 / med, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "oracle port (oracle/torch_ref.py, fp32 torch CPU) of the steady-state forward on FULL %dx%d LR frames of ONE "
                             "sequence: median of %d timed frame(s) after %d warm-up(s) (+ one cache-building first frame, %.1f s): %.2f s "
                             "per frame, nothing cropped or scaled" % (H, W, len(times), warm_done, first, med)}
        value = total_frames / (ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload(args), "lr": [H, W], "seqs_per_gpu": S, "cuda_graph": bool(args.graph), "parallelism": "sequence-sharded x%d, no data-path collective" % world,
                       "l2": "inputs larger than L2 (per step > 1 GB of offsets/masks/activations; %d rotating windows)" % len(pool),
                       "stages": "feature extraction / alignment / attention / fusion / trunk (CTA-pair tcgen05 convs) / tail: this repo's CUDA kernels only (no cuDNN / cuBLAS launch in the step; DESIGN.md 4 lists the ATen copies left)"},
            "e2e": {"value": total_frames / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config c4 (and c5 at scale)
def run_c4(args):
    """BASELINE.json configs[3] literally: `--c4-seqs` (64) independent 1080p x4 sequences of `--c4-frames` (16) frames each through the
    public pipeline cdfo_b200.driver.run_sharded -- sliding 7-frame window with clipped ends (test_LD_37.py:13-16), MV decode +
    end-of-sequence fix-ups on the device (:83-105, :209-234), uint8 planes H2D from pinned staging, uint8 SR frames D2H, on-GPU PSNR / SSIM
    (metric/psnr_ssim.py:278-399) and ONE NCCL all_reduce of the real [n_seq, 3] metric sums at the end.  The job is fixed, the ranks
    split it (contiguous blocks of sequences): STRONG scaling.  Everything -- first frames included -- is inside the timed region; the
    sequences sit decoded in host memory when it starts (a rank generates only the ones it owns)."""
    import torch
    import torch.distributed as dist
    import cdfo_b200
    from cdfo_b200 import driver, sharding, synthetic
    from cdfo_b200.model import CVSR_V8
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    model = CVSR_V8(alignment="mv_dcn" if args.variant == "O2" else "dual_att")
    model.load_state_dict(synthetic.seeded_state_dict(model.state_dict(), seed=4), strict=True)
    model = model.to(dev).eval()
    model.lowp = torch.bfloat16
    n, T, S = args.c4_seqs, args.c4_frames, args.seqs
    lazy = synthetic.SyntheticSequences(n, frames=T, h=270, w=480, seed=0, with_gt=True)
    own = sharding.sequence_shard(n, world, rank)
    t0 = time.perf_counter()
    held = {k: lazy[k] for k in own}

    class Owned:                      # run_sharded indexes only the sequences this rank owns
        def __len__(self):
            return n

        def __getitem__(self, k):
            return held[k]
    gen_s = time.perf_counter() - t0
    # untimed warm-up on a short clip of the same shape (module load, allocator, cuDNN heuristics)
    warm = synthetic.SyntheticSequences(S, frames=8, h=270, w=480, seed=1, with_gt=True)
    driver.FrameDriver(model, seed=7).run([warm[k] for k in range(S)], sink=lambda s, i, img: None)
    delivered = [0]

    def sink(sid, i, img):
        delivered[0] += 1
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    res = driver.run_sharded(model, Owned(), batch=S, seed=0, sink=sink)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - w0
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0].item()), float(t[1].item()) * 1e-3
    assert delivered[0] == len(own) * T, (delivered[0], len(own), T)
    frames = sum(res["frames"])
    assert frames == n * T, (frames, n, T)
    if rank == 0:
        per_frame_h2d = 3 * 270 * 480 + 2 * 270 * 480 + 272 * 480 * 3 + 1080 * 1920     # uint8 lr/pm/unflt, int16 res, int8 mv, uint8 gt
        line = {
            "metric": METRIC, "value": frames / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": T, "warmup": 1,
            "ms_per_step": ms / T, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "c4: %d independent 1080p x4 sequences x %d frames (7x(480x270->272 rows) LR -> 1920x1080 HR, LD priors) "
                                   "through driver.run_sharded: sliding window with clipped ends, MV end fix-ups, on-GPU PSNR/SSIM, NCCL gather of "
                                   "the metric sums" % (n, T), "variant": args.variant, "seqs_per_batch": S,
                       "parallelism": "sequence-sharded x%d (contiguous blocks), no data-path collective" % world,
                       "l2": "inputs larger than L2", "timed_region": "whole job incl. every sequence's first (7-frame) window, H2D, D2H, metrics, all_reduce",
                       "host_generation_s_untimed": gen_s, "wall_s": wall},
            "e2e": {"value": frames / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": per_frame_h2d * S, "d2h_bytes_per_step": 1080 * 1920 * S},
            "gpu_launches": cdfo_b200._lib.launch_count, "psnr": res["psnr"], "ssim": res["ssim"],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % v)
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seqs", type=int, default=4, help="independent sequences resident per GPU (batched per step).  8 measured 89.2 / 85.5 HR fps on one GPU and 677 on eight against 85.6 and 699 with 4: about +4 %% per SM clock, less than the spread between power-capped boxes")
    ap.add_argument("--pool", type=int, default=3, help="distinct input windows rotated through")
    ap.add_argument("--variant", default="O2", choices=["O1", "O2"])
    ap.add_argument("--priors", default="LD", choices=["LD", "RA"], help="LD (configs c3/c4) or RA = bidirectional (l0, l1) MV pairs (config c5)")
    ap.add_argument("--lr-h", type=int, default=LR_H)
    ap.add_argument("--lr-w", type=int, default=LR_W)
    ap.add_argument("--workload", default="c3", choices=["c3", "c4"], help="c3 (default): steady-state step of resident windows (BASELINE configs[2]); "
                    "c4: 64 whole sequences through driver.run_sharded (configs[3], strong scaling)")
    ap.add_argument("--c4-seqs", type=int, default=64)
    ap.add_argument("--c4-frames", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget-s", type=int, default=400, help="--impl reference: wall-clock cap of the CPU run (full frames; steps / warm-ups beyond it are dropped and the line says so)")
    ap.add_argument("--cpu-baseline-budget-s", type=int, default=80, help="cap of the in-arm cpu_baseline leg (full frames, rank 0, N = 1)")
    ap.add_argument("--graph", type=int, default=0, help="1: replay the steady-state step as a CUDA graph (+1.7 %%); 0 (default): eager "
                    "launches, which is what lets the DCN kernel be timed live with CUDA events inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="c3: after the timed steps, write what the last one returned as DIR/sr.npy (the HR "
                    "frames [seqs, 1, 4H, 4W]) and DIR/l1_features.npy (the window's L1 features [seqs, 7, 64, H, W]), float32; an output "
                    "over its size cap is written as a fixed seeded 1-D sample (bench.dump_outputs).  Rank 0's sequences only")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "c4"):
        ap.error("--dump-outputs writes the outputs of the c3 steps of our arm only")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c4":
        run_c4(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
