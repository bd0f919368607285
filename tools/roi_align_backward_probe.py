"""ROIPooler.backward: the atomic (default) and the deterministic mode, timed alternately in one process.

    python tools/roi_align_backward_probe.py [--reps 50] [--out profiles/roi_align_backward_probe.json]

Workloads (FPN P2..P5 of 16 synthetic 800x1333 images, C = 256, ROIs from utils.synthetic.rois):
  a        16 x 1000 ROIs, 7x7, sampling_ratio 0 (the ROI heads' box pooler at inference-size proposal counts)
  box_sr*  16 x 512 ROIs, 7x7 (training box head)
  mask_sr* 16 x 128 ROIs, 14x14 (training mask head)
Each call is timed with CUDA events (the gradient buffers are zeroed outside the timed window); the medians of
both modes come from the same alternating loop.  The per-phase split of the deterministic mode (bin, partition,
accumulate + fold) comes from a separate torch.profiler pass.  The card's name and power limit are read in the
same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from detectron2_tensorflow_b200.modeling import ROIPooler  # noqa: E402
from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList  # noqa: E402
from detectron2_tensorflow_b200.utils import synthetic as syn  # noqa: E402

SCALES = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]
WORKLOADS = [("a", 1000, 7, 0), ("box_sr0", 512, 7, 0), ("box_sr2", 512, 7, 2), ("mask_sr0", 128, 14, 0),
             ("mask_sr2", 128, 14, 2)]
PHASES = {"roi_align_grad_bin_kernel": "bin", "roi_align_grad_partition_kernel": "partition",
          "roi_align_grad_accum_kernel": "accumulate+fold", "roi_align_backward_kernel": "atomic"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def setup(dev, n_images, rois, crop, sr, channels=256):
    boxes, idx = syn.rois(n_images, rois, seed=3)
    shapes = [(n_images,) + syn.level_hw(s) + (channels,) for s in syn.FPN_STRIDES]
    g = torch.randn((n_images * rois, crop, crop, channels), device=dev, generator=torch.Generator(dev).manual_seed(4))
    inst = SparseBoxList(torch.from_numpy(idx).to(dev), BoxList(torch.from_numpy(boxes).to(dev)), (n_images, rois))
    bufs = [torch.zeros(s, dtype=torch.float32, device=dev) for s in shapes]
    return ROIPooler((crop, crop), SCALES, sr, "ROIAlignV2"), g, shapes, inst, bufs


def run(pooler, g, shapes, inst, bufs, det):
    pooler.backward(g, shapes, inst, grad_x=bufs, deterministic=det)


def phase_split(pooler, g, shapes, inst, bufs, det, calls=10):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            run(pooler, g, shapes, inst, bufs, det)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k, name in PHASES.items():
            if k in e.key:
                out[name] = out.get(name, 0.0) + e.device_time_total / 1e3 / calls  # ms per call
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--images", type=int, default=16)
    ap.add_argument("--out", default=os.path.join("profiles", "roi_align_backward_probe.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this probe measures the GPU kernels")
    dev = torch.device("cuda", 0)
    result = {"card": card(), "images": args.images, "channels": 256, "reps": args.reps, "workloads": {}}
    for name, rois, crop, sr in WORKLOADS:
        pooler, g, shapes, inst, bufs = setup(dev, args.images, rois, crop, sr)
        for det in (False, True, False, True):  # warm-up: module load, workspace allocation
            run(pooler, g, shapes, inst, bufs, det)
        times = {False: [], True: []}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.reps):
            for det in (False, True):
                for b in bufs:
                    b.zero_()
                ev[0].record()
                run(pooler, g, shapes, inst, bufs, det)
                ev[1].record()
                ev[1].synchronize()
                times[det].append(ev[0].elapsed_time(ev[1]))
        a_ms, d_ms = float(np.median(times[False])), float(np.median(times[True]))
        w = {"rois": args.images * rois, "crop": crop, "sampling_ratio": sr,
             "atomic_ms_median": a_ms, "deterministic_ms_median": d_ms, "ratio": d_ms / a_ms,
             "atomic_ms_p10_p90": [float(np.percentile(times[False], q)) for q in (10, 90)],
             "deterministic_ms_p10_p90": [float(np.percentile(times[True], q)) for q in (10, 90)],
             "deterministic_phases_ms": phase_split(pooler, g, shapes, inst, bufs, True),
             "atomic_phases_ms": phase_split(pooler, g, shapes, inst, bufs, False)}
        result["workloads"][name] = w
        print(json.dumps({name: w}), flush=True)
        del pooler, g, inst, bufs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], "out": args.out}))


if __name__ == "__main__":
    main()
