"""Timing of the RPN proposal stage alone (d2b_rpn_proposals: select / sort / decode -> capped walk in merge order ->
NMS masks + sweep-merge for the images the walk does not finish) at config-2 sizes (2000 pre / 1000 post), for N = 16,
4 and 1 images (the walk runs from 4 images on); CUDA events, median, L2 flushed or warm.  Variant "whole-image": the
gaussian logits with every box grown past the image (clamped size deltas), so that all boxes clip to the whole image
and each level keeps one box: the walk visits every candidate, spends its budget, and every image goes to masks +
sweep-merge (its worst case).

    python tools/rpn_probe.py [--images 16,4,1] [--variants gaussian,clustered,ties,whole-image]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import Box2BoxTransform, RPNOutputs
from detectron2_tensorflow_b200.structures import ImageList
from detectron2_tensorflow_b200.utils import synthetic as syn

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--images", default="16,4,1")
ap.add_argument("--variants", default="gaussian,clustered,ties,whole-image")
ap.add_argument("--once", action="store_true", help="one call per case, no timing (ncu launch lists)")
args = ap.parse_args()
dev = torch.device("cuda", 0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
anchors = syn.rpn_anchors()
ta = [torch.from_numpy(a).to(dev) for a in anchors]


def timeit(fn, cold):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.iters):
        if cold:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


for variant in args.variants.split(","):
    seed = {"gaussian": 2, "clustered": 3, "ties": 4, "whole-image": 2}[variant]
    logits, deltas = syn.rpn_inputs(16, seed=seed, variant=variant.replace("whole-image", "gaussian"), anchors=anchors)
    if variant == "whole-image":
        for d in deltas:
            d[..., 2:] = 8.0  # above the scale clamp: every box 62x its anchor, clipped to the image
    for N in [int(v) for v in args.images.split(",")]:
        tl = [torch.from_numpy(x[:N]).to(dev) for x in logits]
        td = [torch.from_numpy(x[:N]).to(dev) for x in deltas]
        images = ImageList(None, torch.from_numpy(syn.image_shapes(N)).to(dev))
        outs = RPNOutputs(Box2BoxTransform((1., 1., 1., 1.)), images, tl, td, ta)
        run = lambda: outs.find_top_proposals(0.7, 2000, 1000, 0.0)
        if args.once:
            run()
            torch.cuda.synchronize()
            continue
        l0 = nv.kernel_launch_count()
        r = run()
        launches = nv.kernel_launch_count() - l0
        nms_in = N * sum(min(2000, a.shape[0]) for a in anchors)
        cold, warm = timeit(run, True), timeit(run, False)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            run()
        torch.cuda.current_stream().wait_stream(s)
        with torch.cuda.graph(g):
            run()
        gcold, gwarm = timeit(g.replay, True), timeit(g.replay, False)
        print(json.dumps({"case": f"RPN proposal stage, {variant}, N={N}", "launches": launches, "eager_ms_cold": cold,
                          "eager_ms_warm": warm, "graph_ms_cold": gcold, "graph_ms_warm": gwarm,
                          "boxes_into_nms": nms_in, "boxes_per_s": nms_in / gcold * 1e3,
                          "valid": int(r.get_field("is_valid").sum())}), flush=True)
