"""Probe (image blocks per graphed step) x (steps in flight) for the device-resident step.  One JSON line."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench

dev = torch.device("cuda", 0)
x = bench.to_torch(bench.make_host_inputs(16), dev=dev)
eng = bench.make_engine()
res = {}
for chunks, depth in ((1, 3), (1, 4), (2, 2), (2, 3), (2, 4), (4, 1), (4, 2), (4, 3), (4, 4), (4, 6), (8, 2), (8, 3)):
    pipe = eng.pipeline(x, chunks=chunks, depth=depth)
    pipe.run(2 * depth)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.run(60)
    e1.record()
    torch.cuda.synchronize()
    res[f"chunks{chunks}_inflight{depth}"] = round(e0.elapsed_time(e1) / 60, 4)
    del pipe
    torch.cuda.empty_cache()
print(json.dumps(res))
