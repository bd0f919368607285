"""The Mask R-CNN post-backbone step (bench.py's engine and inputs) on a block of N images: stage times (CUDA events,
eager), one-graph latency, and -- with --once -- a single eager step for an ncu launch list.  The per-rank block of
the strong-scaling leg is N = 16 / world.

    python tools/step_probe.py --images 2,8,16
    ncu --metrics gpu__time_duration.sum --clock-control none --csv ... python tools/step_probe.py --images 2 --once
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench

ap = argparse.ArgumentParser()
ap.add_argument("--images", default="2,8,16")
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--once", action="store_true")
args = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
hp = bench.make_engine()
for n in [int(v) for v in args.images.split(",")]:
    x = bench.to_torch(bench.make_host_inputs(n), dev=dev)
    for _ in range(3):
        hp(x)
    torch.cuda.synchronize()
    if args.once:
        hp(x)
        torch.cuda.synchronize()
        continue
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.iters)]
    for i in range(args.iters):
        hp(x, events=ev[i])
    torch.cuda.synchronize()
    stages = [float(np.median([ev[i][s].elapsed_time(ev[i][s + 1]) for i in range(args.iters)])) for s in range(4)]
    out = {"images": n, "stages_ms": dict(zip(("rpn_proposals", "box_roi_align", "fast_rcnn_post", "mask_roi_align"), stages)),
           "eager_ms": float(sum(stages))}
    for chunks in (1, 2, 4):
        if chunks > n:
            continue
        g = hp.capture(x, chunks=chunks)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g.replay(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        out[f"graph_ms_{chunks}_blocks"] = float(np.median(ts))
        out["kernels"] = g.kernels_per_replay // chunks
        del g
    print(json.dumps(out), flush=True)
