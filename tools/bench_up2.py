"""Body.0 of the x2 branch at c3 trunk shapes: resample(x, 1) + conv3x3 (the 2x input through HBM) against conv3x3_up2 (the bilinear x2
built in the convolution's producer).  CUDA-event timing, the two forms alternated in one run, inputs rotated over enough copies that the
working set exceeds the 126 MB L2.  Prints the card name and power limit with the result."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cdfo_b200 import conv  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
        return q.stdout.strip()
    except OSError:
        return torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--h", type=int, default=272, help="1x height of the trunk (c3: 272 x 480)")
    ap.add_argument("--w", type=int, default=480)
    ap.add_argument("--iters", type=int, default=20, help="launches per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the two forms")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    B, H, W = a.frames, a.h, a.w
    xs = [conv.to_c8(torch.randn(B, 64, H, W, device=dev, generator=g)) for _ in range(4)]     # 4 x 67 MB at c3, 4 frames
    w = torch.randn(256, 64, 3, 3, device=dev, generator=g) * 0.05
    b = torch.randn(256, device=dev, generator=g)
    edge = torch.randn(9, 256, device=dev, generator=g)
    forms = {
        "resample+conv": lambda x: conv.conv3x3(conv.resample(x, 1), w, b, conv.ACT_LRELU, parity_planes=True, bias_edge=edge),
        "conv3x3_up2": lambda x: conv.conv3x3_up2(x, w, b, conv.ACT_LRELU, parity_planes=True, bias_edge=edge),
    }
    same = torch.equal(forms["resample+conv"](xs[0]), forms["conv3x3_up2"](xs[0]))
    times = {k: [] for k in forms}
    for k, f in forms.items():                 # warm-up: module load, cudaFuncSetAttribute, weight packing
        for i in range(3):
            f(xs[i % len(xs)])
    for _ in range(a.rounds):
        for k, f in forms.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            for i in range(a.iters):
                f(xs[i % len(xs)])
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.iters * 1e3)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    flops = 2.0 * B * (2 * H) * (2 * W) * 64 * 256 * 9
    print(json.dumps({"card": card(), "shape_1x": [B, 64, H, W], "bit_identical": same,
                      "us": {k: [round(t, 1) for t in v] for k, v in times.items()},
                      "median_us": {k: round(v, 1) for k, v in med.items()},
                      "conv_TFLOPs": {k: round(flops / v / 1e6, 1) for k, v in med.items()},
                      "saved_us": round(med["resample+conv"] - med["conv3x3_up2"], 1)}))


if __name__ == "__main__":
    main()
