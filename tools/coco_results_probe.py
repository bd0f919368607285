"""Times COCO-ready masks for a batch of 16 images, each at its own original size, on one GPU:

  (a) today's per-image loop: SparseBoxList.from_dense (a host sync), the "fixed" pasting boxes of
      detector_postprocess, reframe_box_masks_to_rle with exact sizing (a second sync), rle_to_coco -- 16 times;
  (b) one detector_postprocess_rle call with exact sizing (one sync), then rle_to_coco with per-mask sizes;
  (c) the same call at a fixed capacity captured in a CUDA graph and replayed.

Each is timed with and without bringing the strings to the host (rle_to_coco); coco_results (the whole COCO results
list) is timed after (b) and (c).  Detections come from the engine geometry: 800x1333 resized inputs (the shortest
edge resized to 800, the longest capped at 1,333), 100 slots per image, about 60 % valid, 28x28 masks; the 16
original sizes are seeded and COCO-like (longest side 640, the other 240-640).  The three paths must produce identical
strings.  A host clock around work that ends in a device synchronise (the per-image path syncs inside), 3 warm-up
runs, median of 20.  Writes one JSON object (with the card name and power limit read in the same run) to --out and
stdout.

    python tools/coco_results_probe.py --out profiles/coco_results_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from detectron2_tensorflow_b200.modeling import coco_results, detector_postprocess_rle  # noqa: E402
from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList, reframe_box_masks_to_rle, rle_to_coco  # noqa: E402


def timed(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def inputs(dev, N=16, R=100, seed=0):
    rng = np.random.default_rng(seed)
    long_side = 640
    short = rng.integers(240, 641, N)
    outs = np.array([[s, long_side] if rng.random() < 0.7 else [long_side, s] for s in short], np.int64)
    ins = np.zeros((N, 2), np.int64)
    for n, (h, w) in enumerate(outs):
        sc = 800.0 / min(h, w)
        if max(h, w) * sc > 1333:
            sc = 1333.0 / max(h, w)
        ins[n] = [int(h * sc + 0.5), int(w * sc + 0.5)]
    boxes = np.zeros((N, R, 4), np.float32)
    for n, (h, w) in enumerate(ins):
        cy, cx = rng.uniform(0, h, R), rng.uniform(0, w, R)
        bh = np.exp(rng.uniform(np.log(20), np.log(500), R)); bw = np.exp(rng.uniform(np.log(20), np.log(500), R))
        boxes[n] = np.stack([np.clip(cy - bh / 2, 0, h), np.clip(cx - bw / 2, 0, w), np.clip(cy + bh / 2, 0, h),
                             np.clip(cx + bw / 2, 0, w)], 1)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    bl = BoxList(T(boxes))
    bl.add_field("pred_masks", T(rng.random((N, R, 28, 28)).astype(np.float32)))
    bl.add_field("is_valid", T(rng.random((N, R)) < 0.6))
    bl.add_field("scores", T(rng.random((N, R)).astype(np.float32)))
    bl.add_field("pred_classes", T(rng.integers(0, 80, (N, R))))
    bl.set_tracking("image_shape", T(ins.astype(np.int32)))
    return bl, outs


def per_image(bl, outs, host):
    """Today's path, image by image (the from_dense + "fixed" boxes of detector_postprocess, then the RLE paste)."""
    N = bl.boxes.shape[0]
    res = []
    for n in range(N):
        one = BoxList(bl.boxes[n:n + 1])
        one.add_field("pred_masks", bl.get_field("pred_masks")[n:n + 1])
        one.add_field("is_valid", bl.get_field("is_valid")[n:n + 1])
        sp = SparseBoxList.from_dense(one)
        out = torch.tensor([float(outs[n][0]), float(outs[n][1])], dtype=torch.float64, device=bl.boxes.device)
        s = (out / bl.get_tracking("image_shape")[n].to(torch.float64)).to(torch.float32)
        b = sp.data.boxes
        b = torch.stack([s[0] * b[:, 0], s[1] * b[:, 1], s[0] * b[:, 2], s[1] * b[:, 3]], 1)
        rle = reframe_box_masks_to_rle(sp.data.get_field("pred_masks"), b, tuple(outs[n]))
        res.append(rle_to_coco(*rle, tuple(outs[n])) if host else rle)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res["gpu"] = q.stdout.strip()
    bl, outs = inputs(dev)
    N, R = bl.boxes.shape[:2]
    sizes = np.repeat(outs, R, 0)
    os_dev = torch.from_numpy(outs.astype(np.int32)).to(dev)
    cats = list(range(1, 81))
    ids = list(range(N))

    rle, boxes = detector_postprocess_rle(bl, outs)
    need = int(rle[1][-1])
    cap = 2 * need
    valid = int(bl.get_field("is_valid").sum())

    # (c): captured once at a fixed capacity, sizes from a device tensor
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        detector_postprocess_rle(bl, os_dev, capacity=cap)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rle_g, boxes_g = detector_postprocess_rle(bl, os_dev, capacity=cap)

    want = [d["counts"] for img in per_image(bl, outs, True) for d in img]
    got_b = [d["counts"] for d in rle_to_coco(*rle, sizes=sizes) if d is not None]
    g.replay()
    torch.cuda.synchronize()
    got_c = [d["counts"] for d in rle_to_coco(*rle_g, sizes=sizes) if d is not None]
    res["setup"] = {"images": int(N), "slots_per_image": int(R), "valid_detections": valid,
                    "input_shapes": bl.get_tracking("image_shape").cpu().tolist(), "output_shapes": outs.tolist(),
                    "rle_bytes": need, "graph_capacity": cap,
                    "batched_equals_per_image": got_b == want, "graph_equals_per_image": got_c == want}

    def b_host():
        r, _ = detector_postprocess_rle(bl, outs)
        rle_to_coco(*r, sizes=sizes)

    def c_host():
        g.replay()
        rle_to_coco(*rle_g, sizes=sizes)

    def b_coco():
        r, bx = detector_postprocess_rle(bl, outs)
        coco_results(bl, r, bx, outs, ids, cats)

    def c_coco():
        g.replay()
        coco_results(bl, rle_g, boxes_g, outs, ids, cats)

    res["ms"] = {
        "a_per_image_device": timed(lambda: per_image(bl, outs, False)),
        "a_per_image_strings_on_host": timed(lambda: per_image(bl, outs, True)),
        "b_batched_exact_device": timed(lambda: detector_postprocess_rle(bl, outs)),
        "b_batched_exact_strings_on_host": timed(b_host),
        "c_graph_fixed_capacity_device": timed(g.replay),
        "c_graph_fixed_capacity_strings_on_host": timed(c_host),
        "b_batched_exact_coco_results": timed(b_coco),
        "c_graph_fixed_capacity_coco_results": timed(c_coco),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
