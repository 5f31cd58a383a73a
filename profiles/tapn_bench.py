"""Kernel time of the grouped 3x3 conv at the pyramid's 128- and 64-wide levels (C2 frame shapes), tc32 and bf16.

python profiles/tapn_bench.py [label]   -> one JSON line per shape / precision: mean us per launch over CUDA events around graph replays.
Six inputs are rotated so the working set (> 126 MB of L2 at the 128 level) is not served from L2 alone.  profiles/tapn_ab.sh
alternates two library builds on one box."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from heal_b200 import ops  # noqa: E402

SHAPES = [("L1_128", 5, 256, 128, 128), ("L2_64", 5, 512, 64, 64)]
ROT, WARM, ITERS, REPLAYS = 6, 20, 200, 5


def main():
    label = sys.argv[1] if len(sys.argv) > 1 else ""
    torch.manual_seed(0)
    for name, N, C, H, W in SHAPES:
        conv = torch.nn.Conv2d(C, C, 3, padding=1, groups=32, bias=True)
        for prec, fmt in (("tc32", "split"), ("bf16", "bf16")):
            pc = ops.pack_conv_tc(conv, None, True, planes=2).to("cuda")
            xs = [ops.convert(ops.to_act(torch.randn(N, C, H, W, device="cuda")), fmt) for _ in range(ROT)]
            outs = [ops.conv2d_tc(x, pc)[0] for x in xs]
            for i in range(WARM):
                ops.conv2d_tc(xs[i % ROT], pc, out=outs[i % ROT])
            torch.cuda.synchronize()
            # replayed as one CUDA graph, as in the frame: the host cost of a launch is not in the number
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(ITERS):
                    ops.conv2d_tc(xs[i % ROT], pc, out=outs[i % ROT])
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(REPLAYS):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (ITERS * REPLAYS)
            flops = 2.0 * N * H * W * C * (C // 32) * 9
            print(json.dumps({"label": label, "shape": name, "N": N, "C": C, "H": H, "W": W, "precision": prec,
                              "us_per_launch": round(us, 2), "algorithmic_tflops": round(flops / us / 1e6, 1)}))


if __name__ == "__main__":
    main()
