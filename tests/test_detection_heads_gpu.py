"""GPU: Fast R-CNN (d2b_fast_rcnn_postprocess: clip, score threshold, class-offset NMS, top-k, fused decode) and
YOLOv4 (d2b_yolo_postprocess: max / first argmax over classes, threshold, one class-agnostic NMS) post-processing
against oracle.fast_rcnn_inference / oracle.yolo_inference on full batches, adversarial inputs and both sides of
every size-selected branch of their shared tail.

Bar: boxes bit-exact with NaN == NaN, scores bit-exact (compared as int32 bit patterns), pred_classes int64 and
is_valid equal, Fast R-CNN kept indices equal to the oracle's ROI slots, out_num equal to the oracle's count, and
out_nms_boxes_in equal to the number of candidates counted here in numpy.  The Python wrappers pass NULL for the last
two, so the entries are called through their params structs.  Every case runs inside the canary bands of
test_canary_gpu, so a write one element past an output or workspace fails even when the values match.  Seeds are
fixed: every case reproduces from its id.

The three atomic paths of frcnn_prep_kernel (one per CTA when all 8 warps hold one image, one per warp, one per
thread) are chosen inside the kernel by the order of the index rows; a trace cannot show them, so the row-order case
says why each order reaches them."""
import math

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.utils import synthetic as syn

from test_canary_gpu import Guard
from test_dispatch_boundaries_gpu import K as kname, Launch, reach, traced
import test_fuzz_gpu as fz
import test_postprocess_gpu as pp

pytestmark = pytest.mark.gpu

WEIGHTS = (10.0, 10.0, 5.0, 5.0)  # ROI_BOX_HEAD.BBOX_REG_WEIGHTS
SCALE_CLAMP = math.log(1000.0 / 16)

# Host-side thresholds of the tail (csrc/nms.cu use_lazy, reached through nms_lazy_applies(stride, T) in
# d2b_fast_rcnn_postprocess / d2b_yolo_postprocess, with stride = Rmax * K or n: the capacity, not the live count)
LAZY_MAX_OUT = 8192          # kLazyMaxOut: caps above it never take det_tail_kernel
BITMASK_MAX_N = 65536        # kBitmaskMaxN: strides above it always take det_tail_kernel
SWEEP_CLUSTER_MIN_W = 128    # kSweepClusterMinW (nms_sorted): W = ceil(stride / 64) above it sweeps in a cluster
TAIL_SMEM_DEFAULT = 40 * 1024  # det_tail: 20 * T bytes of shared memory, opt-in attribute above this
SORT_TILE = 8192             # kTile (sort_segments_desc): sort_big runs when pad_pow2(stride) exceeds one tile


@pytest.fixture
def guard(monkeypatch):
    return Guard(monkeypatch)


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def pad_pow2(x):
    p = 1
    while p < x:
        p <<= 1
    return p


def tail_launches(stride, T_det):
    """nms_lazy_applies(stride, T): det_tail_kernel with 20 T bytes of shared memory, else det_gather + bitmask NMS
    (nms_mask_kernel, then the column sweep -- in a cluster past W = kSweepClusterMinW words) + det_emit."""
    if T_det <= LAZY_MAX_OUT and (stride > BITMASK_MAX_N or 8 * T_det <= stride):
        return [Launch(kname("det_tail_kernel"), dyn_smem=20 * T_det)], [kname("det_gather_kernel"),
                                                                          kname("nms_mask_kernel")]
    sweeps = [kname("nms_sweep_cols_kernel"), kname("nms_sweep_cols_cluster_kernel")]
    if (stride + 63) // 64 > SWEEP_CLUSTER_MIN_W:
        sweeps.reverse()
    return ([Launch(kname("det_gather_kernel")), Launch(kname("nms_mask_kernel")), Launch(sweeps[0]),
             Launch(kname("det_emit_kernel"))], [kname("det_tail_kernel"), sweeps[1]])


def sort_launches(stride):
    if pad_pow2(stride) > SORT_TILE:
        return [Launch(kname("sort_local")), Launch(kname("sort_big"))], []
    return [Launch(kname("sort_local"))], [kname("sort_big")]


def check_common(got, want):
    """got / want: (boxes, scores, classes, valid, ...) with classes int64."""
    assert got[2].dtype == np.int64
    assert np.array_equal(got[3], want[3])
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[1].view(np.int32), want[1].view(np.int32))
    assert np.array_equal(got[0], want[0], equal_nan=True)


def same_bytes(a, b):
    return all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(a, b))


# ------------------------------------------------------------------ Fast R-CNN through d2b_fast_rcnn_params
def frcnn_call(cuda, scores, idx, N, Rmax, shapes, score_thr, nms_thr, T_det, agnostic, boxes=None, deltas=None,
               props=None):
    """One d2b_fast_rcnn_postprocess call; boxes [M, Kb*4], or deltas [M, Kb*4] + props [M, 4] (fused decode).
    Returns numpy (boxes, scores, classes, valid, roi, num, nms_boxes_in)."""
    M, K1 = scores.shape
    K = K1 - 1
    b = boxes if boxes is not None else deltas
    Kb = b.shape[1] // 4
    keep = [T(scores, cuda), T(idx, cuda), T(shapes, cuda), T(b, cuda)]
    ob = torch.empty((N, T_det, 4), dtype=torch.float32, device=cuda)
    os_ = torch.empty((N, T_det), dtype=torch.float32, device=cuda)
    oc = torch.empty((N, T_det), dtype=torch.int64, device=cuda)
    ov = torch.empty((N, T_det), dtype=torch.bool, device=cuda)
    orr = torch.empty((N, T_det), dtype=torch.int32, device=cuda)
    on = torch.empty((N,), dtype=torch.int32, device=cuda)
    nin = torch.empty((1,), dtype=torch.int64, device=cuda)
    p = nv.FastRcnnParams()
    p.scores, p.indices, p.image_shapes = keep[0].data_ptr(), keep[1].data_ptr(), keep[2].data_ptr()
    if boxes is not None:
        p.boxes = keep[3].data_ptr()
    else:
        keep.append(T(props, cuda))
        p.boxes, p.deltas, p.proposal_boxes = None, keep[3].data_ptr(), keep[4].data_ptr()
        for i in range(4):
            p.weights[i] = WEIGHTS[i]
        p.scale_clamp = SCALE_CLAMP
    p.num_preds, p.num_images, p.rmax = M, N, Rmax
    p.num_bbox_reg_classes, p.num_classes = Kb, K
    p.score_thresh, p.nms_thresh, p.topk_per_image = float(score_thr), float(nms_thr), T_det
    p.nms_cls_agnostic = int(bool(agnostic))
    p.out_boxes, p.out_scores, p.out_classes, p.out_valid = ob.data_ptr(), os_.data_ptr(), oc.data_ptr(), ov.data_ptr()
    p.out_roi_index, p.out_num, p.out_nms_boxes_in = orr.data_ptr(), on.data_ptr(), nin.data_ptr()
    nv.call("fast_rcnn_postprocess", p, cuda)
    return tuple(t.cpu().numpy() for t in (ob, os_, oc, ov, orr, on, nin))


def frcnn_live(scores, idx, N, Rmax, thr):
    """Candidates per image, counted on the zero-filled dense scores of SparseBoxList.to_dense."""
    K = scores.shape[1] - 1
    d = np.zeros((N, Rmax, K), np.float32)
    ok = (idx[:, 0] >= 0) & (idx[:, 0] < N) & (idx[:, 1] >= 0) & (idx[:, 1] < Rmax)
    d[idx[ok, 0], idx[ok, 1]] = scores[ok, :K]
    return (d > np.float32(thr)).sum(axis=(1, 2))


def frcnn_check(got, want, live):
    check_common(got, want)
    assert np.array_equal(got[4], want[4])  # kept indices (ROI slots)
    assert np.array_equal(got[5], want[5])  # out_num
    assert int(got[6][0]) == int(live.sum())  # out_nms_boxes_in


def frcnn_run(cuda, oracle_lib, boxes, scores, idx, N, Rmax, shapes, thr, nms_thr, T_det, agnostic, deltas=None,
              props=None, trace=False):
    """Oracle and kernel on the same case (with the boxes, or fused-decode from deltas + props whose decode the
    oracle does with apply_deltas); asserts equality; returns (got, oracle outputs, trace)."""
    if deltas is not None:
        boxes = oracle_lib.apply_deltas(deltas, props, WEIGHTS)
    want = oracle_lib.fast_rcnn_inference(boxes, scores, idx, (N, Rmax), shapes, thr, nms_thr, T_det, agnostic)
    live = frcnn_live(scores, idx, N, Rmax, thr)
    call = (lambda: frcnn_call(cuda, scores, idx, N, Rmax, shapes, thr, nms_thr, T_det, agnostic, deltas=deltas,
                               props=props)) if deltas is not None else \
        (lambda: frcnn_call(cuda, scores, idx, N, Rmax, shapes, thr, nms_thr, T_det, agnostic, boxes=boxes))
    got, tr = traced(call) if trace else (call(), None)
    frcnn_check(got, want, live)
    return got, want, tr


# ------------------------------------------------------------------ a. Fast R-CNN randomized differential
SCORE_MODES = ("softmax", "rounded", "at_thresh", "nonfinite", "below")


def softmax_scores(rng, M, K):
    lg = rng.standard_normal((M, K + 1)) * 3.0
    e = np.exp(lg - lg.max(1, keepdims=True))
    return (e / e.sum(1, keepdims=True)).astype(np.float32)


def frcnn_scores(rng, M, K, mode, thr):
    s = softmax_scores(rng, M, K)
    if mode == "rounded":  # ties across classes and ROIs: class-major, then slot order
        s = np.round(s * 16) / 16
    elif mode == "at_thresh":  # exactly the threshold: `>` does not pass it
        s = np.where(rng.random(s.shape) < 0.3, np.float32(thr), s)
    elif mode == "nonfinite":
        flat = s.reshape(-1)
        for v, frac in ((np.nan, 0.05), (np.inf, 0.01), (-np.inf, 0.05)):
            flat[rng.integers(0, flat.size, max(int(flat.size * frac), 1))] = v
    elif mode == "below":  # nothing passes
        s = np.float32(thr) - np.float32(0.001) - np.abs(rng.standard_normal(s.shape))
    return s.astype(np.float32)


def frcnn_deltas(rng, M, Kb):
    """Deltas beyond scale_clamp, +-1e4 centre offsets and a few inf / NaN values."""
    d = (rng.standard_normal((M, Kb, 4)) * 0.5).astype(np.float32)
    f = d.reshape(-1, 4)
    rows = rng.integers(0, f.shape[0], max(f.shape[0] // 20, 1))
    f[rows, 2:] = rng.choice([-1.0, 1.0], (rows.size, 2)) * rng.uniform(5.0 * SCALE_CLAMP, 300.0, (rows.size, 2))
    rows = rng.integers(0, f.shape[0], max(f.shape[0] // 50, 1))
    f[rows, :2] = rng.choice([-1.0, 1.0], (rows.size, 2)) * 1e5  # x 1/10 by the weights: +-1e4 centre offsets
    rows = rng.integers(0, f.shape[0], 3)
    f[rows[0], rng.integers(0, 4)] = np.inf
    f[rows[1], rng.integers(0, 4)] = -np.inf
    f[rows[2], rng.integers(0, 4)] = np.nan
    return d.reshape(M, Kb * 4)


def ragged_rows(rng, N, R, order):
    """Index rows of a ragged batch: per image all R slots, a random subset, or none (and the last image empty on
    some seeds); a few rows with n < 0, n >= N or r >= Rmax; image-major, reversed or permuted.  No duplicate
    (n, r) among the in-range rows."""
    rows = []
    for n in range(N):
        kind = rng.choice(["full", "subset", "empty"], p=[0.35, 0.5, 0.15])
        if kind == "full":
            r = np.arange(R)
        elif kind == "subset":
            r = np.sort(rng.choice(R, int(rng.integers(1, R + 1)), replace=False))
        else:
            r = np.zeros(0, np.int64)
        rows.append(np.stack([np.full(r.size, n), r], 1))
    if N > 1 and rng.random() < 0.3:
        rows[-1] = rows[-1][:0]
    if sum(len(x) for x in rows) == 0:
        rows[0] = np.array([[0, R - 1]])
    idx = np.concatenate(rows).astype(np.int64)
    bad = np.array([[-1, 0], [N, 0], [N + 3, R - 1], [0, R], [N - 1, R + 7], [0, -1]], np.int64)
    idx = np.concatenate([idx, bad[rng.choice(len(bad), int(rng.integers(0, 4)), replace=False)]])
    if order == "reversed":
        idx = idx[::-1]
    elif order == "permuted":
        idx = idx[rng.permutation(len(idx))]
    return np.ascontiguousarray(idx)


def frcnn_boxes(rng, M, Kb, H=400, W=500):
    b = fz.fuzz_boxes(rng, M * Kb, H, W)
    z = rng.integers(0, M * Kb, max(M * Kb // 30, 1))
    b[z] = np.array([-60.0, -50.0, -10.0, -4.0], np.float32)  # clips to a zero box
    return b.reshape(M, Kb * 4)


def run_frcnn_fuzz(cuda, oracle_lib, seed):
    rng = np.random.default_rng(9000 + seed)
    N = int(rng.integers(1, 17))
    R = int(rng.choice([1, 7, 200, 1000]))
    K = int(rng.choice([1, 2, 20, 80]))
    Kb = K if rng.random() < 0.6 else 1
    agnostic = bool(rng.random() < 0.3)
    T_det = int(rng.choice([1, 10, 100, 1000]))
    thr = float(rng.choice([0.05, 0.0, 0.5, -1.0]))
    nms_thr = float(rng.choice([0.0, 0.5, 1.0]))
    if R * K > 16000:  # keeps the oracle's NMS at seconds: (Rmax * K) candidates x T kept per image
        N, T_det = min(N, 4), min(T_det, 100)
    order = str(rng.choice(["image", "reversed", "permuted"]))
    idx = ragged_rows(rng, N, R, order)
    M = idx.shape[0]
    modes = [SCORE_MODES[int(rng.integers(0, len(SCORE_MODES)))] for _ in range(N)]
    scores = softmax_scores(rng, M, K)
    for n in range(N):
        sel = idx[:, 0] == n
        if sel.any():
            scores[sel] = frcnn_scores(rng, int(sel.sum()), K, modes[n], thr)
    shapes = np.stack([rng.integers(100, 400, N), rng.integers(100, 500, N)], 1).astype(np.int32)
    boxes = frcnn_boxes(rng, M, Kb)
    got, _, _ = frcnn_run(cuda, oracle_lib, boxes, scores, idx, N, R, shapes, thr, nms_thr, T_det, agnostic)
    if seed % 2:  # fused decode: the same case from deltas + proposals, against apply_deltas + the oracle
        deltas, props = frcnn_deltas(rng, M, Kb), fz.fuzz_boxes(rng, M, 400, 500)
        fused, _, _ = frcnn_run(cuda, oracle_lib, None, scores, idx, N, R, shapes, thr, nms_thr, T_det, agnostic,
                                deltas=deltas, props=props)
        decoded = frcnn_call(cuda, scores, idx, N, R, shapes, thr, nms_thr, T_det, agnostic,
                             boxes=oracle_lib.apply_deltas(deltas, props, WEIGHTS))
        assert same_bytes(fused, decoded)


@pytest.mark.parametrize("seed", range(48))
def test_fast_rcnn_fuzz(cuda, oracle_lib, guard, seed):
    run_frcnn_fuzz(cuda, oracle_lib, seed)
    guard.check()


def test_fast_rcnn_negative_threshold_absent_slots(cuda, oracle_lib, guard):
    """score_thresh < 0 on a ragged batch: every slot that no index row fills is a zero row of the dense tensors
    (SparseBoxList.to_dense), so its K classes are candidates with score 0, a zero box and kept index = the slot --
    and they are the only candidates of an image whose rows all score below the threshold."""
    rng = np.random.default_rng(77)
    N, R, K = 3, 40, 3
    idx = np.array([[0, r] for r in range(0, R, 3)] + [[2, r] for r in range(R - 5)], np.int64)  # image 1 empty
    M = idx.shape[0]
    scores = softmax_scores(rng, M, K)
    scores[idx[:, 0] == 2] = -2.0  # image 2: only its 5 absent slots can be kept
    shapes = np.array([[300, 400], [200, 250], [350, 300]], np.int32)
    boxes = frcnn_boxes(rng, M, K)
    for agnostic in (False, True):
        _, want, _ = frcnn_run(cuda, oracle_lib, boxes, scores, idx, N, R, shapes, -1.0, 0.5, 100, agnostic)
        # zero boxes have no area, so none suppresses another: (score 0, class-major, slot) order up to the cap
        assert want[5][1] == 100 and want[5][2] == 15
        assert np.array_equal(want[4][1], np.concatenate([np.arange(R), np.arange(R), np.arange(20)]))
        assert np.array_equal(want[2][1], np.repeat([0, 1, 2], [R, R, 20]))
        assert np.array_equal(want[4][2, :15], np.tile(np.arange(R - 5, R), 3))
        assert not want[0][1:].any() and not want[1][1:].any()
    frcnn_run(cuda, oracle_lib, None, scores, idx, N, R, shapes, -1.0, 0.5, 100, False,
              deltas=frcnn_deltas(rng, M, K), props=fz.fuzz_boxes(rng, M, 400, 500))
    guard.check()


# ------------------------------------------------------------------ b. Fast R-CNN: row order is irrelevant
@pytest.mark.parametrize("ragged", [False, True], ids=["full", "partial_cta"])
def test_fast_rcnn_row_order(cuda, oracle_lib, guard, ragged):
    """N = 16, R = 1000, K = 80 in four row orders; every output byte-identical across them and equal to the oracle.
    frcnn_prep_kernel gives a CTA 256 (row, class) threads = 3.2 rows: image-major rows put all 8 warps of almost
    every CTA in one image (one atomic per CTA); r-major rows (slot 0 of every image, then slot 1, ...) change image
    every 80 threads, so most warps hold one image (one atomic per warp) and the warps across a row boundary hold
    two (one atomic per thread); reversed and permuted orders mix all three.  partial_cta drops rows so that
    M * K is not a multiple of 256 and the last CTA is partial."""
    rng = np.random.default_rng(31 + ragged)
    N, R, K = 16, 1000, 80
    valid = np.ones((N, R), bool)
    if ragged:
        valid &= rng.random((N, R)) < 0.9
        valid[5] = False
    idx = np.argwhere(valid).astype(np.int64)
    M = idx.shape[0]
    assert (M * K % 256 != 0) == ragged
    scores, deltas = syn.fast_rcnn_inputs(1, M, K, seed=12)
    props = fz.fuzz_boxes(rng, M, 800, 1333)
    boxes = oracle_lib.apply_deltas(deltas, props, WEIGHTS)
    shapes = np.tile(np.array([[800, 1333]], np.int32), (N, 1))
    want = oracle_lib.fast_rcnn_inference(boxes, scores, idx, (N, R), shapes, 0.05, 0.5, 100, False)
    live = frcnn_live(scores, idx, N, R, 0.05)
    orders = {"image": np.arange(M), "reversed": np.arange(M)[::-1], "permuted": rng.permutation(M),
              "r_major": np.lexsort((idx[:, 0], idx[:, 1]))}
    first = None
    for name, o in orders.items():
        got = frcnn_call(cuda, scores[o], idx[o], N, R, shapes, 0.05, 0.5, 100, False, boxes=boxes[o])
        frcnn_check(got, want, live)
        assert first is None or same_bytes(got, first), name
        first = first or got
    guard.check()


# ------------------------------------------------------------------ c. YOLOv4 randomized differential
def yolo_call(cuda, boxes, probs, score_thr, nms_thr, T_det):
    """One d2b_yolo_postprocess call -> numpy (boxes, scores, classes, valid, num, nms_boxes_in)."""
    N, n, K = probs.shape
    tb, tp = T(boxes, cuda), T(probs, cuda)
    ob = torch.empty((N, T_det, 4), dtype=torch.float32, device=cuda)
    os_ = torch.empty((N, T_det), dtype=torch.float32, device=cuda)
    oc = torch.empty((N, T_det), dtype=torch.int64, device=cuda)
    ov = torch.empty((N, T_det), dtype=torch.bool, device=cuda)
    on = torch.empty((N,), dtype=torch.int32, device=cuda)
    nin = torch.empty((1,), dtype=torch.int64, device=cuda)
    p = nv.YoloParams()
    p.boxes, p.probs = tb.data_ptr(), tp.data_ptr()
    p.num_images, p.num_boxes, p.num_classes = N, n, K
    p.score_thresh, p.nms_thresh, p.post_nms_topk = float(score_thr), float(nms_thr), T_det
    p.out_boxes, p.out_scores, p.out_classes, p.out_valid = ob.data_ptr(), os_.data_ptr(), oc.data_ptr(), ov.data_ptr()
    p.out_num, p.out_nms_boxes_in = on.data_ptr(), nin.data_ptr()
    nv.call("yolo_postprocess", p, cuda)
    return tuple(t.cpu().numpy() for t in (ob, os_, oc, ov, on, nin))


def yolo_live(probs, thr):
    """Boxes kept by the threshold: reduce_max propagates NaN, and NaN > thr is false."""
    if probs.shape[1] == 0:
        return np.zeros(probs.shape[0], np.int64)
    return (probs.max(-1) > np.float32(thr)).sum(1)


def yolo_run(cuda, oracle_lib, boxes, probs, thr, nms_thr, T_det, trace=False):
    want = oracle_lib.yolo_inference(boxes, probs, thr, nms_thr, T_det)
    call = lambda: yolo_call(cuda, boxes, probs, thr, nms_thr, T_det)
    got, tr = traced(call) if trace else (call(), None)
    check_common(got, want)
    assert np.array_equal(got[4], want[4])
    assert int(got[5][0]) == int(yolo_live(probs, thr).sum())
    return got, want, tr


PROB_MODES = ("random", "ties", "zeros", "inf", "nan", "at_thresh", "below")


def yolo_probs(rng, n, K, mode, thr):
    p = (rng.random((n, K)) ** 3).astype(np.float32)
    if n == 0:
        return p
    rows = rng.random(n) < 0.3
    if mode == "ties":  # the first maximal class wins
        p = np.round(p * 8) / 8
        p[rows] = np.float32(0.5)
    elif mode == "zeros":  # +0.0 against -0.0 in the maximal position, both orders
        z = np.where(rng.random((n, K)) < 0.5, np.float32(0.0), np.float32(-0.0))
        p = np.where(rows[:, None], z, p - np.float32(1.5))
    elif mode == "inf":
        p[rng.random((n, K)) < 0.02] = np.inf
        p[rng.random((n, K)) < 0.1] = -np.inf
        p[rows] = -np.inf
    elif mode == "nan":  # NaN in class 0, a middle class, the last class; all-NaN rows
        where = rng.integers(0, 4, n)
        for w, col in ((0, 0), (1, K // 2), (2, K - 1)):
            p[rows & (where == w), col] = np.nan
        p[rows & (where == 3)] = np.nan
    elif mode == "at_thresh":  # the maximum exactly at the threshold does not pass
        p = np.minimum(p, np.float32(thr))
        p[rows, int(rng.integers(0, K))] = np.float32(thr)
    elif mode == "below":
        p = np.float32(thr) - np.float32(0.001) - p
    return p.astype(np.float32)


def run_yolo_fuzz(cuda, oracle_lib, seed):
    rng = np.random.default_rng(9500 + seed)
    N = int(rng.integers(1, 9))
    n = int(rng.choice([0, 1, 31, 100, 5000, 22743]))
    K = int(rng.choice([1, 31, 32, 33, 80]))
    T_det = int(rng.choice([1, 20, 100, 1000]))
    thr = float(rng.choice([0.2, 0.0, -1.0]))
    nms_thr = float(rng.choice([0.45, 0.0, 1.0]))
    if n * K * N > 4_000_000:
        N = max(1, 4_000_000 // (n * K))
    boxes = np.stack([fz.fuzz_boxes(rng, n, 300, 400) for _ in range(N)]) if n else np.zeros((N, 0, 4), np.float32)
    if n > 1:
        boxes[:, rng.integers(0, n, max(n // 100, 1))] = np.nan  # passed through, never compared against
    probs = np.stack([yolo_probs(rng, n, K, PROB_MODES[int(rng.integers(0, len(PROB_MODES)))], thr)
                      for _ in range(N)]) if n else np.zeros((N, 0, K), np.float32)
    yolo_run(cuda, oracle_lib, boxes, probs, thr, nms_thr, T_det)


@pytest.mark.parametrize("seed", range(40))
def test_yolo_fuzz(cuda, oracle_lib, guard, seed):
    run_yolo_fuzz(cuda, oracle_lib, seed)
    guard.check()


@pytest.mark.parametrize("thr", [0.2, 0.0, -1.0])
def test_yolo_nan_rows_dropped(cuda, oracle_lib, guard, thr):
    """A NaN probability in any class -- the first, a middle, the last, or all of them -- drops the box whatever
    the threshold (TF's reduce_max propagates NaN and NaN > thr is false); the other rows keep the first maximum,
    with +0.0 and -0.0 equal."""
    K = 5
    probs = np.array([[np.nan, 0.9, 0.1, 0.0, 0.3],
                      [0.9, 0.2, np.nan, 0.1, 0.3],
                      [0.3, 0.9, 0.1, 0.2, np.nan],
                      [np.nan] * K,
                      [0.4, 0.95, 0.95, 0.1, 0.2],
                      [-0.0, 0.0, -0.0, 0.0, -0.0],
                      [0.0, -0.0, -1.5, -0.0, 0.0],
                      [0.6, 0.1, 0.0, 0.0, 0.6]], np.float32)[None]
    boxes = np.array([[10 + 40 * i, 10, 40 + 40 * i, 40] for i in range(probs.shape[1])], np.float32)[None]
    _, want, _ = yolo_run(cuda, oracle_lib, boxes, probs, thr, 0.5, 10)
    v = want[3][0]
    cls = dict(zip([(int(b[0]) - 10) // 40 for b in want[0][0][v]], want[2][0][v]))  # row of a kept box: class
    want_cls = {4: 1, 7: 0}
    if thr < 0:
        want_cls.update({5: 0, 6: 0})
    assert cls == want_cls
    guard.check()


# ------------------------------------------------------------------ d. both sides of every size-selected branch
def frcnn_boundary(cuda, oracle_lib, R, K, T_det, live=None, every=False, seed=0):
    """One image plus a short second one, R slots x K classes: stride = R * K.  live: exactly that many candidates
    in image 0 (scores 0 elsewhere); every: every (slot, class) of image 0 is a candidate."""
    rng = np.random.default_rng(R * K + T_det + seed)
    N = 2
    idx = np.concatenate([np.stack([np.zeros(R), np.arange(R)], 1),
                          np.stack([np.ones(R // 3), np.arange(R // 3)], 1)]).astype(np.int64)
    M = idx.shape[0]
    scores = softmax_scores(rng, M, K)
    if every:
        scores[:R, :K] = rng.uniform(0.1, 1.0, (R, K)).astype(np.float32)
    if live is not None:
        s0 = np.zeros(R * K, np.float32)
        s0[rng.choice(R * K, live, replace=False)] = rng.uniform(0.1, 1.0, live).astype(np.float32)
        scores[:R, :K] = s0.reshape(R, K)
    shapes = np.array([[800, 1333], [600, 900]], np.int32)
    boxes = fz.fuzz_boxes(rng, M * K, 800, 1333).reshape(M, K * 4)
    _, want, tr = frcnn_run(cuda, oracle_lib, boxes, scores, idx, N, R, shapes, 0.05, 0.5, T_det, False, trace=True)
    assert want[3].any()
    return tr, frcnn_live(scores, idx, N, R, 0.05)


def yolo_boundary(cuda, oracle_lib, n, T_det, live=None, seed=0):
    rng = np.random.default_rng(n + T_det + seed)
    N, K = 2, 4
    boxes = np.stack([pp.clustered_boxes(rng, n, k=60) for _ in range(N)])
    probs = (rng.random((N, n, K)) * 0.9 + 0.05).astype(np.float32)
    if live is not None:  # image 0: exactly `live` boxes above the threshold 0.05
        probs[0] = 0.0
        probs[0, rng.choice(n, live, replace=False), 0] = rng.uniform(0.1, 1.0, live).astype(np.float32)
    _, want, tr = yolo_run(cuda, oracle_lib, boxes, probs, 0.05, 0.5, T_det, trace=True)
    assert want[3].any()
    return tr


# (id, Fast R-CNN (R, K) or None, YOLO n or None, T): the stride is R * K for Fast R-CNN and n for YOLO
TAIL_CASES = [
    # use_lazy: 8 T <= stride -> det_tail_kernel, 8 T = stride + 8 -> the bitmask chain
    ("lazy-8T=stride", (500, 8), 4000, 500),
    ("bitmask-8T=stride+8", (500, 8), 4000, 501),
    # bitmask chain: W = 128 words -> nms_sweep_cols_kernel, W = 129 -> nms_sweep_cols_cluster_kernel
    ("sweep-W128", (1024, 8), 8192, 1100),
    ("sweep-W129-cluster", (1032, 8), 8256, 1100),
    # det_tail's 20 T bytes of shared memory: 40,960 (default) vs 40,980 (opt-in attribute)
    ("tail-smem-40960", (1000, 20), 20000, TAIL_SMEM_DEFAULT // 20),
    ("tail-smem-optin", (1000, 20), 20000, TAIL_SMEM_DEFAULT // 20 + 1),
    # stride > kBitmaskMaxN: the lazy tail at any cap it accepts
    ("tail-stride-above-bitmask-limit", (1000, 80), 70000, 100),
]


@pytest.mark.parametrize("head", ["fast_rcnn", "yolo"])
@pytest.mark.parametrize("case", [c[1:] for c in TAIL_CASES], ids=[c[0] for c in TAIL_CASES])
def test_tail_branch(cuda, oracle_lib, guard, head, case):
    (R, K), n, T_det = case
    stride = R * K if head == "fast_rcnn" else n
    tr = frcnn_boundary(cuda, oracle_lib, R, K, T_det)[0] if head == "fast_rcnn" else \
        yolo_boundary(cuda, oracle_lib, n, T_det)
    tl, ta = tail_launches(stride, T_det)
    reach(tr, tl + [Launch(kname("frcnn_prep_kernel" if head == "fast_rcnn" else "yolo_prep_kernel"))], ta)
    guard.check()


@pytest.mark.parametrize("live", [SORT_TILE, SORT_TILE + 1])
def test_sort_tile_boundary(cuda, oracle_lib, guard, live):
    """Live candidate count at one sort tile (kTile = 8,192 keys: sort_local alone sorts them) and one past it
    (sort_big merges two tiles).  YOLO with every box live: n = stride = live, so sort_big also shows in the trace
    only for 8,193; Fast R-CNN at stride 16,400 launches sort_big in both cases and takes the live count inside."""
    tr = yolo_boundary(cuda, oracle_lib, live, 100, live=live)
    reach(tr, *sort_launches(live))
    tr, lv = frcnn_boundary(cuda, oracle_lib, 1025, 16, 100, live=live)
    assert lv[0] == live
    reach(tr, *sort_launches(1025 * 16))
    guard.check()


def test_fast_rcnn_capacity_not_live_count(cuda, oracle_lib, guard):
    """The tail is chosen on the capacity Rmax * K, not on the live count: 80,000 slots with 30 live candidates take
    det_tail_kernel, 480 slots with every one live and T = 100 (8 T > 480) take the bitmask chain."""
    tr, lv = frcnn_boundary(cuda, oracle_lib, 1000, 80, 100, live=30)
    assert lv[0] == 30
    reach(tr, *tail_launches(80000, 100))
    tr, lv = frcnn_boundary(cuda, oracle_lib, 60, 8, 100, every=True)
    assert lv[0] == 480
    reach(tr, *tail_launches(480, 100))
    guard.check()


# ------------------------------------------------------------------ e. configs[1] at its batch size
def test_fast_rcnn_config2_batch16(cuda, oracle_lib, guard):
    """BASELINE.json configs[1]'s fast_rcnn_post stage: 16 images x 1,000 ROIs x 80 classes, thresholds 0.05 / 0.5,
    top-100, with boxes and with fused decode: every image against the oracle, and images 0, 7 and 15 run alone give
    the rows of the batch byte for byte."""
    N, R, K = 16, 1000, 80
    rng = np.random.default_rng(16)
    scores, deltas = syn.fast_rcnn_inputs(N, R, K)
    idx = np.stack([np.repeat(np.arange(N), R), np.tile(np.arange(R), N)], 1).astype(np.int64)
    props = np.concatenate([pp.clustered_boxes(rng, R, k=40) for _ in range(N)])
    shapes = syn.image_shapes(N)
    got, want, _ = frcnn_run(cuda, oracle_lib, None, scores, idx, N, R, shapes, 0.05, 0.5, 100, False,
                             deltas=deltas, props=props)
    assert (want[5] > 0).all()
    boxes = oracle_lib.apply_deltas(deltas, props, WEIGHTS)
    got_b, _, _ = frcnn_run(cuda, oracle_lib, boxes, scores, idx, N, R, shapes, 0.05, 0.5, 100, False)
    assert same_bytes(got, got_b)
    for n in (0, 7, 15):
        sl = slice(n * R, (n + 1) * R)
        one_idx = np.stack([np.zeros(R), np.arange(R)], 1).astype(np.int64)
        one = frcnn_call(cuda, scores[sl], one_idx, 1, R, shapes[n:n + 1], 0.05, 0.5, 100, False,
                         deltas=deltas[sl], props=props[sl])
        assert same_bytes(one[:6], [x[n:n + 1] for x in got[:6]]), n
    guard.check()


def test_yolo_batch16(cuda, oracle_lib, guard):
    """YOLOv4 at 16 images x 22,743 boxes x 80 classes (608 x 608 input), top-100: every image against the oracle,
    and images 0, 7 and 15 run alone give the rows of the batch byte for byte."""
    N, n, K = 16, 22743, 80
    rng = np.random.default_rng(22743)
    boxes = np.stack([pp.clustered_boxes(rng, n, k=40) for _ in range(N)])
    probs = (rng.random((N, n, K), dtype=np.float32) ** 6).astype(np.float32)
    probs[:, ::5] = np.round(probs[:, ::5] * 8) / 8
    got, want, _ = yolo_run(cuda, oracle_lib, boxes, probs, 0.25, 0.45, 100)
    assert (want[4] > 0).all()
    for i in (0, 7, 15):
        one = yolo_call(cuda, boxes[i:i + 1], probs[i:i + 1], 0.25, 0.45, 100)
        assert same_bytes(one[:5], [x[i:i + 1] for x in got[:5]]), i
    guard.check()
