"""CPU only: what the capped walk in merge order (rpn_lazy_merge_kernel) does on the seeded RPN inputs, against the
suppression-mask pairs of per-level bitmask NMS.  Per image: candidates visited until `post` boxes are kept (and the
64-candidate blocks that takes), IoU tests of the walk (a candidate's tests against the kept boxes of its level stop
at the first suppressor), and the mask pairs n (n - 1) / 2 of every level.  The numbers behind kRpnLazyMaxBlocks.

    python tools/rpn_lazy_visits.py [--variants gaussian,clustered,ties] [--images 16,4,4]

"gaussian" is bench.py's input (bench.make_host_inputs); the other variants are syn.rpn_inputs(seed=2, variant=...).
Top-k and decode come from the oracle; clip and the TF IoU rule are restated here in numpy."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import bench
import oracle
from detectron2_tensorflow_b200.utils import synthetic as syn

PRE, POST, THR = 2000, 1000, 0.7


def iou_row(a, B):
    """TF NonMaxSuppression IoU of box a against the rows of B (fp32, division form; 0 for degenerate boxes)."""
    ya0, xa0, ya1, xa1 = min(a[0], a[2]), min(a[1], a[3]), max(a[0], a[2]), max(a[1], a[3])
    yb0, xb0 = np.minimum(B[:, 0], B[:, 2]), np.minimum(B[:, 1], B[:, 3])
    yb1, xb1 = np.maximum(B[:, 0], B[:, 2]), np.maximum(B[:, 1], B[:, 3])
    aa = (ya1 - ya0) * (xa1 - xa0)
    ab = (yb1 - yb0) * (xb1 - xb0)
    inter = np.maximum(np.minimum(ya1, yb1) - np.maximum(ya0, yb0), np.float32(0)) * \
        np.maximum(np.minimum(xa1, xb1) - np.maximum(xa0, xb0), np.float32(0))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = inter / ((aa + ab) - inter)
    r[(aa <= 0) | (ab <= 0)] = 0
    return r


def walk_image(levels):
    """levels: [(boxes [k,4] in candidate order, logits [k])] of one image -> (visited, IoU tests, mask pairs)."""
    order = sorted((-float(v), l, p) for l, (_, vals) in enumerate(levels) for p, v in enumerate(vals))
    kept = [[] for _ in levels]
    nk = visited = tests = 0
    for _, l, p in order:
        if nk >= POST:
            break
        visited += 1
        K = levels[l][0][kept[l]]
        if len(K):
            hit = np.nonzero(iou_row(levels[l][0][p], K) > THR)[0]
            tests += int(hit[0]) + 1 if len(hit) else len(K)  # kept boxes in kept order, stop at the first suppressor
            if len(hit):
                continue
        kept[l].append(p)
        nk += 1
    pairs = sum(len(v) * (len(v) - 1) // 2 for _, v in levels)
    return visited, tests, pairs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", default="gaussian,clustered,ties")
    ap.add_argument("--images", default="16,4,4", help="images per variant (same order)")
    args = ap.parse_args()
    oracle.build()
    anchors = syn.rpn_anchors()
    for variant, N in zip(args.variants.split(","), [int(v) for v in args.images.split(",")]):
        if variant == "gaussian":
            host = bench.make_host_inputs(N)
            logits, deltas, shapes = host["logits"], host["deltas"], host["shapes"]
        else:
            logits, deltas = syn.rpn_inputs(N, seed=2, variant=variant, anchors=anchors)
            shapes = syn.image_shapes(N)
        rows = []
        for n in range(N):
            h, w = np.float32(shapes[n][0]), np.float32(shapes[n][1])
            levels = []
            for d, a, lg in zip(deltas, anchors, logits):
                vals, idx = oracle.top_k(lg[n].reshape(-1), min(PRE, lg.shape[1]))
                b = oracle.rpn_predict_proposals(d[n:n + 1], a)[0][idx]
                b = np.stack([np.maximum(np.minimum(b[:, 0], h), 0), np.maximum(np.minimum(b[:, 1], w), 0),
                              np.maximum(np.minimum(b[:, 2], h), 0), np.maximum(np.minimum(b[:, 3], w), 0)],
                             1).astype(np.float32)
                levels.append((b, vals))
            rows.append(walk_image(levels))
        v, t, p = (np.array(c) for c in zip(*rows))
        print(json.dumps({"variant": variant, "images": N,
                          "visited_per_image": [int(v.min()), int(v.max())],
                          "blocks_per_image": [int(-(-v.min() // 64)), int(-(-v.max() // 64))],
                          "iou_tests_per_image": [int(t.min()), int(t.max())], "iou_tests_total": int(t.sum()),
                          "mask_pairs_per_image": int(p.max()), "mask_pairs_total": int(p.sum()),
                          "pairs_saved_x": round(float(p.sum()) / float(t.sum()), 1)}), flush=True)


if __name__ == "__main__":
    main()
