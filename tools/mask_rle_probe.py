"""Times COCO RLE output of the mask ops against image-mask planes copied to the host, on one GPU:

  * Mask R-CNN: 16 images x 100 detections, 28x28 masks pasted on 800x1333 (the boxes of tools/paste_probe.py):
    d2b_paste_masks to uint8 planes, planes + pinned copy to the host, fused paste -> RLE, RLE + copy of the offsets
    and strings to the host;
  * SOLOv2: 16 x 100 kept masks at 200x336 upsampled to 800x1333, the same four variants;
  * the host encoder the tests compare against (tests/coco_rle.py: pycocotools rleEncode + rleToString in numpy, one
    host thread) over the same Mask R-CNN planes: host work the fused encoder removes.

CUDA events around each variant, 3 warm-up calls, median of 20.  Writes one JSON object (with the card name and power
limit read in the same run) to --out and stdout.

    python tools/mask_rle_probe.py --out profiles/mask_rle_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import coco_rle  # noqa: E402
from detectron2_tensorflow_b200.modeling import solo_upsample_masks  # noqa: E402
from detectron2_tensorflow_b200.structures import reframe_box_masks_to_image_masks, reframe_box_masks_to_rle  # noqa: E402
from detectron2_tensorflow_b200.utils import synthetic as syn  # noqa: E402


def timed(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res["gpu"] = q.stdout.strip()

    # ---- Mask R-CNN paste (tools/paste_probe.py inputs)
    rng = np.random.default_rng(0)
    M, H, W = 1600, 800, 1333
    masks_np = rng.random((M, 28, 28)).astype(np.float32)
    cy, cx = rng.uniform(0, H, M), rng.uniform(0, W, M)
    h = np.exp(rng.uniform(np.log(20), np.log(500), M)); w = np.exp(rng.uniform(np.log(20), np.log(500), M))
    boxes_np = np.stack([np.clip(cy - h / 2, 0, H), np.clip(cx - w / 2, 0, W), np.clip(cy + h / 2, 0, H),
                         np.clip(cx + w / 2, 0, W)], 1).astype(np.float32)
    masks, boxes = torch.from_numpy(masks_np).to(dev), torch.from_numpy(boxes_np).to(dev)
    planes_host = torch.empty((M, H, W), dtype=torch.uint8, pin_memory=True)
    chars, offsets = reframe_box_masks_to_rle(masks, boxes, (H, W))
    cap = chars.numel()
    chars_host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    off_host = torch.empty(M + 1, dtype=torch.int64, pin_memory=True)

    def planes_copy():
        planes_host.copy_(reframe_box_masks_to_image_masks(masks, boxes, (H, W)), non_blocking=True)

    def rle_copy():
        c, o = reframe_box_masks_to_rle(masks, boxes, (H, W), capacity=cap)
        off_host.copy_(o, non_blocking=True)
        chars_host.copy_(c, non_blocking=True)

    res["maskrcnn"] = {
        "masks": M, "image": [H, W], "plane_bytes": M * H * W, "rle_bytes": cap,
        "paste_planes_ms": timed(lambda: reframe_box_masks_to_image_masks(masks, boxes, (H, W))),
        "paste_planes_copy_ms": timed(planes_copy),
        "paste_rle_ms": timed(lambda: reframe_box_masks_to_rle(masks, boxes, (H, W), capacity=cap)),
        "paste_rle_copy_ms": timed(rle_copy),
    }
    planes_copy()
    torch.cuda.synchronize()
    planes_np = planes_host.numpy()
    t0 = time.perf_counter()
    want = coco_rle.encode(planes_np)
    res["maskrcnn"]["host_encode_ms_one_thread"] = (time.perf_counter() - t0) * 1e3
    rle_copy()
    torch.cuda.synchronize()
    off = off_host.tolist()
    data = chars_host.numpy().tobytes()
    res["maskrcnn"]["rle_equals_host_encode"] = all(data[off[i]:off[i + 1]] == want[i] for i in range(M))
    del planes_np, want

    # ---- SOLOv2 upsample (tools/upsample_probe.py inputs)
    B, D, h, w = 16, 100, 200, 336
    obj = np.stack([syn.solo_masks(D, hw=(h, w), seed=70 + i)[0] for i in range(B)]).reshape(B, D, -1).astype(np.uint8)
    obj = np.concatenate([obj, np.zeros((B, D, (-obj.shape[-1]) % 64), np.uint8)], -1)
    kept = torch.from_numpy(np.packbits(obj, axis=-1, bitorder="little").view(np.int64)).to(dev)
    s_chars, _ = solo_upsample_masks(kept, (h, w), (H, W), 0.5, False, return_masks=False, return_rle=True)["rle"]
    s_cap = s_chars.numel()
    s_chars_host = torch.empty(s_cap, dtype=torch.uint8, pin_memory=True)
    s_off_host = torch.empty(B * D + 1, dtype=torch.int64, pin_memory=True)
    planes_host = planes_host.view(B, D, H, W)

    def solo_planes_copy():
        planes_host.copy_(solo_upsample_masks(kept, (h, w), (H, W), 0.5, False)["pred_masks"], non_blocking=True)

    def solo_rle():
        return solo_upsample_masks(kept, (h, w), (H, W), 0.5, False, return_masks=False, return_rle=True,
                                   rle_capacity=s_cap)["rle"]

    def solo_rle_copy():
        c, o = solo_rle()
        s_off_host.copy_(o, non_blocking=True)
        s_chars_host.copy_(c, non_blocking=True)

    res["solov2"] = {
        "masks": B * D, "source": [h, w], "image": [H, W], "plane_bytes": B * D * H * W, "rle_bytes": s_cap,
        "upsample_planes_ms": timed(lambda: solo_upsample_masks(kept, (h, w), (H, W), 0.5, False)),
        "upsample_planes_copy_ms": timed(solo_planes_copy),
        "upsample_boxes_only_ms": timed(lambda: solo_upsample_masks(kept, (h, w), (H, W), 0.5, False, return_masks=False)),
        "upsample_rle_ms": timed(solo_rle),
        "upsample_rle_copy_ms": timed(solo_rle_copy),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
