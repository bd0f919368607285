"""Times COCO-ready SOLOv2 masks for a batch of 16 images, each at its own original size, on one GPU:

  (a) a per-image loop of the single-size `solo_upsample_masks(..., return_rle=True)` with exact sizing (a host sync
      per image); it cannot crop, so (a), (b) and (c) resize the whole mask (mask_shapes=None);
  (b) one batched `solo_upsample_rle` call with exact sizing (one sync);
  (c) the same call at a fixed capacity captured in a CUDA graph and replayed;
  (d) the whole `SOLOv2Inference.inference_rle` from raw head outputs (select, dynamic conv + tail, batched RLE), with
      crops, eagerly with exact sizing and as a graph replay at a fixed capacity.
(b) and (c) are also timed with the crops.  Each path is timed on the device alone and with the strings and boxes
brought to the host (rle_to_coco).  (a), (b) and (c) must give identical strings and boxes on the valid slots.

Inputs: 16 images x 100 slots of 200x336 object-like packed masks (the mask features of an 800x1344 padded canvas at
stride 4), about 90 % of the slots valid; the 16 original sizes are seeded and COCO-like (landscape, longest side 640,
the other 300-640); each image is resized into the canvas as the input pipeline does it (shortest edge 800, longest
capped at 1,333) and its crop is ceil(size in the canvas / 4).  A host clock around work that ends in a device
synchronise, 3 warm-up runs, median of 20.  Writes one JSON object (with the card name and power limit read in the same run) to
--out and stdout.

    python tools/solo_coco_probe.py --out profiles/solo_coco_probe.json
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

from detectron2_tensorflow_b200.modeling import SOLOv2Inference, solo_upsample_masks, solo_upsample_rle  # noqa: E402
from detectron2_tensorflow_b200.structures import rle_to_coco  # noqa: E402

B, D, H, W, E = 16, 100, 200, 336, 256


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


def sizes(rng):
    """COCO-like original sizes (landscape, so that every resize fits the 800x1344 canvas) and the crop of each
    image's resize in that canvas."""
    outs, crops = [], []
    for s in rng.integers(300, 641, B):
        hw = (int(s), 640)
        sc = min(800.0 / min(hw), 1333.0 / max(hw))
        crop = (-(-int(hw[0] * sc + 0.5) // 4), -(-int(hw[1] * sc + 0.5) // 4))
        assert crop[0] <= H and crop[1] <= W
        outs.append(hw)
        crops.append(crop)
    return np.array(outs, np.int64), np.array(crops, np.int64)


def packed_masks(rng, dev, crops):
    """Object-like ellipses inside each image's crop, bit-packed as d2b_solo_postprocess emits them."""
    cy = torch.from_numpy(rng.uniform(0, 1, (B, D)) * crops[:, :1]).float().to(dev)
    cx = torch.from_numpy(rng.uniform(0, 1, (B, D)) * crops[:, 1:]).float().to(dev)
    ry = torch.from_numpy(np.exp(rng.uniform(np.log(3), np.log(60), (B, D)))).float().to(dev)
    rx = torch.from_numpy(np.exp(rng.uniform(np.log(3), np.log(60), (B, D)))).float().to(dev)
    yy = torch.arange(H, device=dev, dtype=torch.float32)[None, None, :, None]
    xx = torch.arange(W, device=dev, dtype=torch.float32)[None, None, None, :]
    m = ((yy - cy[..., None, None]) / ry[..., None, None]) ** 2 + ((xx - cx[..., None, None]) / rx[..., None, None]) ** 2 <= 1
    bits = m.reshape(B, D, -1, 64).to(torch.int64) << torch.arange(64, device=dev, dtype=torch.int64)
    return bits.sum(-1)  # H * W is a multiple of 64; bit 63 wraps to the sign bit, as in the packed format


def head_outputs(dev):
    """Raw SOLOv2 head outputs at configs[3] scale (tools/solo_inference_probe.py): ~500 candidates per image."""
    g = torch.Generator(device=dev).manual_seed(0)
    grids = (40, 36, 24, 16, 12)
    probs = [torch.where(torch.rand((B, g_, g_, 80), device=dev, generator=g) < 0.0016,
                         torch.rand((B, g_, g_, 80), device=dev, generator=g) * 0.8 + 0.15,
                         torch.zeros((), device=dev)) for g_ in grids]
    kerns = [torch.randn((B, g_, g_, E), device=dev, generator=g) / 16 for g_ in grids]
    yy = torch.arange(H, device=dev, dtype=torch.float32)[None, :, None, None]
    xx = torch.arange(W, device=dev, dtype=torch.float32)[None, None, :, None]
    cy = torch.rand((B, 1, 1, E), device=dev, generator=g) * H
    cx = torch.rand((B, 1, 1, E), device=dev, generator=g) * W
    sg = torch.rand((B, 1, 1, E), device=dev, generator=g) * 35 + 5
    feat = torch.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * sg * sg)).contiguous()
    feat[..., 0] = 1.0
    for k_ in kerns:
        k_.mul_(0.01)
        pick = torch.randint(1, E, k_.shape[:-1] + (1,), device=dev, generator=g)
        k_.scatter_(-1, pick, 8.0)
        k_[..., 0] = -4.0
    head = SOLOv2Inference(0.5, 500, "gaussian", 2.0, 0.05, D, score_threshold=0.1, num_grids=grids,
                           strides=(8, 8, 16, 32, 32), max_candidates=1024)
    return head, probs, kerns, feat


def graphed(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res["gpu"] = q.stdout.strip()
    rng = np.random.default_rng(0)
    outs, crops = sizes(rng)
    pk = packed_masks(rng, dev, crops)
    valid_h = rng.random((B, D)) < 0.9
    valid = torch.from_numpy(valid_h).to(dev)
    os_dev = torch.from_numpy(outs.astype(np.int32)).to(dev)
    cs_dev = torch.from_numpy(crops.astype(np.int32)).to(dev)
    per_mask = np.repeat(outs, D, 0)

    def a(host):
        got = []
        for b in range(B):
            r = solo_upsample_masks(pk[b:b + 1], (H, W), tuple(outs[b]), return_masks=False, return_rle=True)
            got.append((rle_to_coco(*r["rle"], tuple(outs[b])), r["boxes"].cpu()) if host else r)
        return got

    def b(crop):
        return solo_upsample_rle(pk, (H, W), outs, crops if crop else None, valid)

    def on_host(rle, boxes):
        return rle_to_coco(*rle, sizes=per_mask), boxes.cpu()

    rle_b, boxes_b = b(False)
    cap = 2 * int(rle_b[1][-1])
    g_c, (rle_c, boxes_c) = graphed(lambda: solo_upsample_rle(pk, (H, W), os_dev, None, valid, capacity=cap))
    g_cc, (rle_cc, _) = graphed(lambda: solo_upsample_rle(pk, (H, W), os_dev, cs_dev, valid, capacity=cap))
    g_c.replay()
    g_cc.replay()
    torch.cuda.synchronize()

    # (a), (b), (c) agree: strings and boxes of the valid slots; (b) and (c) give the others empty strings, zero boxes
    want_s, want_b = [], []
    for (coco, bx), v in zip(a(True), valid_h):
        want_s += [d["counts"] if x else None for d, x in zip(coco, v)]
        want_b.append(np.where(v[:, None], bx[0].numpy(), 0))
    want_b = np.stack(want_b)
    for name, (rle, bx) in (("b", (rle_b, boxes_b)), ("c", (rle_c, boxes_c))):
        got = [d and d["counts"] for d in rle_to_coco(*rle, sizes=per_mask)]
        assert got == want_s, f"({name}) strings differ from the per-image loop"
        assert np.array_equal(bx.cpu().numpy(), want_b), f"({name}) boxes differ from the per-image loop"

    head, probs, kerns, feat = head_outputs(dev)
    res_d, rle_d = head.inference_rle(probs, kerns, feat, outs, crops)
    cap_d = 2 * int(rle_d[1][-1])
    g_d, (res_dg, rle_dg) = graphed(lambda: head.inference_rle(probs, kerns, feat, os_dev, cs_dev, capacity=cap_d))
    g_d.replay()
    torch.cuda.synchronize()
    assert torch.equal(rle_dg[1], rle_d[1]) and torch.equal(rle_dg[0][:int(rle_d[1][-1])], rle_d[0])
    assert torch.equal(res_dg.boxes, res_d.boxes)

    res["setup"] = {"images": B, "slots_per_image": D, "mask_hw": [H, W], "valid_slots": int(valid_h.sum()),
                    "output_shapes": outs.tolist(), "crops": crops.tolist(),
                    "rle_bytes_full_mask": int(rle_b[1][-1]), "rle_bytes_cropped": int(rle_cc[1][-1]),
                    "graph_capacity": cap, "a_b_c_identical": True,
                    "inference_detections": int(res_d.get_field("is_valid").sum()),
                    "inference_rle_bytes": int(rle_d[1][-1]), "inference_graph_equals_eager": True}

    def d_eager():
        return head.inference_rle(probs, kerns, feat, outs, crops)

    def d_eager_host():
        r, rle = d_eager()
        on_host(rle, r.boxes)

    def replay_host(g, rle, boxes):
        def run():
            g.replay()
            on_host(rle, boxes)
        return run

    res["ms"] = {
        "a_per_image_device": timed(lambda: a(False)),
        "a_per_image_strings_on_host": timed(lambda: a(True)),
        "b_batched_exact_device": timed(lambda: b(False)),
        "b_batched_exact_strings_on_host": timed(lambda: on_host(*b(False))),
        "c_graph_fixed_capacity_device": timed(g_c.replay),
        "c_graph_fixed_capacity_strings_on_host": timed(replay_host(g_c, rle_c, boxes_c)),
        "b_cropped_batched_exact_device": timed(lambda: b(True)),
        "b_cropped_batched_exact_strings_on_host": timed(lambda: on_host(*b(True))),
        "c_cropped_graph_fixed_capacity_device": timed(g_cc.replay),
        "d_inference_rle_eager_device": timed(d_eager),
        "d_inference_rle_eager_strings_on_host": timed(d_eager_host),
        "d_inference_rle_graph_device": timed(g_d.replay),
        "d_inference_rle_graph_strings_on_host": timed(replay_host(g_d, rle_dg, res_dg.boxes)),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
