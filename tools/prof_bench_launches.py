"""Steady-state launch list of bench.py from torch.profiler (CUDA activities): runs `bench.py ARGS` in this process under the profiler and
writes a markdown table of the kernels of the timed steps, cut between occurrences of a kernel that runs once per step (as
launch_summary.py does for ncu lists).  Example:
    python tools/prof_bench_launches.py OUT.md --first 5 --last 7 -- --steps 2 --warmup 3 --no-cpu-baseline"""
import argparse
import collections
import os
import runpy
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--marker", default="mv_head_dcn_fused_sm100_kernel", help="a kernel that runs once per step")
    ap.add_argument("--first", type=int, default=5, help="keep launches from the first-th marker launch (1-based) ...")
    ap.add_argument("--last", type=int, default=7, help="... to just before the last-th one")
    ap.add_argument("--title", default="torch.profiler launch list of bench.py")
    a, rest = ap.parse_known_args()
    rest = [r for r in rest if r != "--"]
    sys.argv = [os.path.join(ROOT, "bench.py")] + rest
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        try:
            runpy.run_path(sys.argv[0], run_name="__main__")
        except SystemExit as e:
            if e.code:
                raise
    torch.cuda.synchronize()
    kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy")
                   and not e.name.startswith("Memset")), key=lambda e: e.time_range.start)
    hits = [i for i, e in enumerate(kern) if a.marker in e.name]
    kern = kern[hits[a.first - 1]:hits[a.last - 1] if a.last <= len(hits) else None]
    steps = a.last - a.first
    agg = collections.OrderedDict()
    for e in kern:
        t = agg.setdefault(e.name, [0.0, 0])
        t[0] += e.time_range.elapsed_us()
        t[1] += 1
    tot = sum(v[0] for v in agg.values())
    lines = ["# " + a.title, "", "Command: `python tools/prof_bench_launches.py OUT.md --first %d --last %d -- %s`; shown: the %d steps between "
             "the %d-th and the %d-th launch of `%s` (one per step).  Kernel sum %.1f us per step over %d launches per step." %
             (a.first, a.last, " ".join(rest), steps, a.first, a.last, a.marker, tot / steps, len(kern) // steps), "",
             "| us per step | launches per step | share | kernel |", "|---|---|---|---|"]
    for name, (t, n) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
        lines.append("| %.1f | %g | %.1f%% | `%s` |" % (t / steps, n / steps, 100.0 * t / tot, name[:110]))
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines[:12]))


if __name__ == "__main__":
    main()
