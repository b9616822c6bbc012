"""Throughput of a whole evaluation job of mixed sequences through driver.run_sharded, one process per GPU:

  torchrun --nproc_per_node N tools/bench_job.py [--job ld|long] [--modes b1,seq,split] [--frames-scale F] [--seqs S]

The job is synthetic (synthetic.SyntheticSequences) with the LR sizes and frame counts of the JCT-VC LD test set under the common
test conditions (--job ld: Classes B 480x270, C 208x120, D 104x60, E 320x180; 16 sequences, 7180 frames), or one long 1080p x4
sequence (--job long).  --frames-scale shrinks every length (at least 1 frame).  Modes, each timed over the whole job:
  b1     run_sharded(batch=1): one sequence per step, sequence blocks
  seq    run_sharded(batch=S): sequence blocks, S slots per GPU, sequences of one size and different lengths share a batch
  split  run_sharded(batch=S, split=True): sequences cut into frame ranges balanced by cost over every slot of every GPU
Prints one JSON line: per mode HR frames/s and HR Mpixel/s (CUDA events, slowest rank), the partition's per-rank cost imbalance
(max / mean), slot occupancy (live slot-steps / slot-steps over all ranks) and per-sequence PSNR / SSIM; GPU name and power limit
are read in the same call.  Sequences a rank needs are generated before the timed region; every shape is warmed up untimed."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# (name, LR width, LR height, frames): JCT-VC LD sequences at x4 (Class B 1920x1080 -> 480x270, C 832x480 -> 208x120,
# D 416x240 -> 104x60, E 1280x720 -> 320x180); frame counts of the common test conditions
JCT_LD = [
    ("Kimono", 480, 270, 240), ("ParkScene", 480, 270, 240), ("Cactus", 480, 270, 500), ("BasketballDrive", 480, 270, 500),
    ("BQTerrace", 480, 270, 600),
    ("BasketballDrill", 208, 120, 500), ("BQMall", 208, 120, 600), ("PartyScene", 208, 120, 500), ("RaceHorsesC", 208, 120, 300),
    ("BasketballPass", 104, 60, 500), ("BQSquare", 104, 60, 600), ("BlowingBubbles", 104, 60, 500), ("RaceHorses", 104, 60, 300),
    ("FourPeople", 320, 180, 600), ("Johnny", 320, 180, 600), ("KristenAndSara", 320, 180, 600),
]
LONG = [("Long1080p", 480, 270, 600)]


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except (OSError, ValueError, subprocess.SubprocessError):
        return {"name": None, "power_limit": None, "sm_max_clock": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--job", default="ld", choices=["ld", "long"])
    ap.add_argument("--modes", default="b1,seq,split")
    ap.add_argument("--frames-scale", type=float, default=1.0)
    ap.add_argument("--seqs", type=int, default=4, help="slots per GPU (batch of run_sharded) in modes seq and split")
    ap.add_argument("--variant", default="O2", choices=["O1", "O2"])
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
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
    info = gpu_info(local)
    model = CVSR_V8(alignment="mv_dcn" if args.variant == "O2" else "dual_att")
    model.load_state_dict(synthetic.seeded_state_dict(model.state_dict(), seed=4), strict=True)
    model = model.to(dev).eval()
    model.lowp = torch.bfloat16

    table = JCT_LD if args.job == "ld" else LONG
    frames = [max(1, int(round(T * args.frames_scale))) for _, _, _, T in table]
    lazy = synthetic.SyntheticSequences(len(table), frames=frames, h=[h for _, _, h, _ in table], w=[w for _, w, _, _ in table],
                                        seed=0, with_gt=True)
    shapes = [lazy.shape_of(k) for k in range(len(table))]
    modes = [m for m in args.modes.split(",") if m]
    plans = {}
    for m in modes:
        if m not in ("b1", "seq", "split"):
            raise SystemExit("unknown mode %r" % m)
        slots = 1 if m == "b1" else args.seqs
        plans[m] = (slots,) + sharding.partition_items(shapes, world, slots, split=(m == "split"))
    need = sorted({it.seq for _, items, ranks in plans.values() for it, r in zip(items, ranks) if r == rank})
    held = {k: lazy[k] for k in need}

    class Held:                       # run_sharded reads shapes of every sequence, frames of the ones this rank's items touch
        def __len__(self):
            return len(table)

        def __getitem__(self, k):
            return held[k]

        def shape_of(self, k):
            return lazy.shape_of(k)

    # untimed warm-up of every frame size at every batch the modes use (module load, allocator, cuDNN heuristics, packed weights)
    for h, w in sorted({(h, w) for _, h, w in shapes}):
        for slots in sorted({p[0] for p in plans.values()}):
            warm = synthetic.SyntheticSequences(slots, frames=4, h=h, w=w, seed=1, with_gt=True)
            driver.FrameDriver(model, seed=7).run([warm[k] for k in range(slots)], sink=lambda s, i, img: None)
    delivered = [0]

    def sink(k, i, img):
        delivered[0] += 1
    result = {}
    for m in modes:
        slots, items, ranks = plans[m]
        delivered[0] = 0
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = driver.run_sharded(model, Held(), batch=slots, seed=0, sink=sink, split=(m == "split"))
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, res["slot_steps"], res["idle_slot_steps"], delivered[0]], device=dev, dtype=torch.float64)
        if world > 1:
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms = float(tmax[0])
        n_frames, hr_px = sum(T for T, _, _ in shapes), sum(T * 16 * h * w for T, h, w in shapes)
        assert int(t[3]) == n_frames and res["frames"] == [float(T) for T, _, _ in shapes], (int(t[3]), n_frames)
        cost = sharding.rank_costs(items, ranks, shapes, world)
        result[m] = {
            "hr_fps": n_frames / (ms * 1e-3), "hr_mpix_s": hr_px / (ms * 1e-3) / 1e6, "ms": ms, "slots_per_gpu": slots,
            "items": len(items), "cost_imbalance": max(cost) / (sum(cost) / world),
            "slot_occupancy": 1.0 - float(t[2]) / float(t[1]), "admissions_rank0": res["admissions"],
            "psnr": dict(zip([n for n, _, _, _ in table], res["psnr"])), "ssim": dict(zip([n for n, _, _, _ in table], res["ssim"])),
        }
    if rank == 0:
        print(json.dumps({"tool": "bench_job", "job": args.job, "n_gpus": world, "frames_scale": args.frames_scale,
                          "sequences": len(table), "frames": sum(T for T, _, _ in shapes), "variant": args.variant, "dtype": "bf16",
                          "gpu": info, "timed_region": "whole run_sharded call incl. first windows, admissions, H2D / D2H, metrics, all_reduce",
                          "modes": result}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
