"""GPU: RetinaNet post-processing (d2b_retinanet_postprocess: sigmoid top-k, level offsets, decode, merge of the level
runs, class-offset NMS) against oracle.retinanet_inference on batches, adversarial inputs and both sides of every
size-selected branch.

Bar: boxes bit-exact with NaN == NaN (inf / NaN deltas legitimately give NaN boxes in both), scores bit-exact
(compared as int32 bit patterns), pred_classes int32 and is_valid equal.  Every case runs inside the canary bands of
test_canary_gpu, so a write one element past an output or workspace fails even when the values match.  Seeds are
fixed: every case reproduces from its id.

Several paths of the top-k are chosen per row inside the kernels (sampled logit cutoff, the `redo` repeat of pass 0,
the re-read of the row by topk_finish_kernel, candidate-list overflow, scalar code for rows that do not start on a
16-byte boundary).  A trace cannot show which one a row took, so the cases that target them say why their input
forces the path."""
import math

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import (Box2BoxTransform, DefaultAnchorGenerator, RetinaNetInference,
                                                 YOLOv4Inference, fast_rcnn_inference)
from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList
from detectron2_tensorflow_b200.utils import synthetic as syn

from test_canary_gpu import Guard
from test_dispatch_boundaries_gpu import K as kname, Launch, _rejected, reach, traced
import test_fuzz_gpu as fz

pytestmark = pytest.mark.gpu

SCALE_CLAMP = math.log(1000.0 / 16)


@pytest.fixture
def guard(monkeypatch):
    return Guard(monkeypatch)


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def T_misaligned(x, dev):
    """x on the device starting 4 bytes past a 16-byte boundary (a contiguous view at storage offset 1)."""
    flat = np.concatenate([np.zeros(1, np.float32), np.ascontiguousarray(x, np.float32).reshape(-1)])
    return torch.from_numpy(flat).to(dev)[1:].view(x.shape)


def run(cuda, oracle_lib, cls, dl, anchors, K, topk, score_thr, nms_thr, T_det, dev_anchors=None, dev_cls=None):
    """Runs the head and the oracle on the same inputs, asserts equality; returns (trace, oracle outputs)."""
    wb, ws, wc, wv, wn = oracle_lib.retinanet_inference(cls, dl, anchors, K, topk, score_thr, nms_thr, T_det)
    head = RetinaNetInference(num_classes=K, topk_candidates=topk, score_threshold=score_thr, nms_threshold=nms_thr,
                              max_detections_per_image=T_det)
    tc = dev_cls if dev_cls is not None else [T(x, cuda) for x in cls]
    td = [T(x, cuda) for x in dl]
    ta = dev_anchors if dev_anchors is not None else [T(a, cuda) for a in anchors]
    res, trace = traced(lambda: head.inference(tc, td, ta))
    check(res, (wb, ws, wc, wv))
    return trace, (wb, ws, wc, wv, wn)


def check(res, want, rows=slice(None)):
    wb, ws, wc, wv = want
    assert res.get_field('pred_classes').dtype == torch.int32
    assert np.array_equal(res.get_field('is_valid').cpu().numpy(), wv[rows])
    assert np.array_equal(res.get_field('pred_classes').cpu().numpy(), wc[rows])
    assert np.array_equal(res.get_field('scores').cpu().numpy().view(np.int32), ws[rows].view(np.int32))
    assert np.array_equal(res.boxes.cpu().numpy(), wb[rows], equal_nan=True)


def table_anchors(rng, hwa, H=600, W=800):
    return fz.fuzz_boxes(rng, hwa, H, W)


def normal_deltas(rng, N, hwa, sd=0.3):
    return (rng.standard_normal((N, hwa, 4)) * sd).astype(np.float32)


# ------------------------------------------------------------------ a. randomized differential cases
LOGIT_MODES = ("prior", "rounded", "saturated", "zeros", "nonfinite", "below")


def fuzz_logits(rng, shape, mode):
    x = (rng.standard_normal(shape) * 1.5 - 4.6).astype(np.float32)  # the prior (retinanet.py:425)
    if mode == "rounded":  # ties within and across levels and classes
        x = np.round((rng.standard_normal(shape) * 2.0 - 1.0) * 8) / 8
    elif mode == "saturated":  # >= 17: the computed sigmoid is exactly 1.0
        x = np.where(rng.random(shape) < 0.4, 17.0 + np.abs(rng.standard_normal(shape)) * 20, x)
    elif mode == "zeros":  # p == 0.5 exactly, for both signs of zero
        z = rng.random(shape) < 0.5
        x = np.where(z, np.where(rng.random(shape) < 0.5, np.float32(0.0), np.float32(-0.0)), x + 4.0)
    elif mode == "nonfinite":
        x = (rng.standard_normal(shape) * 2.0 - 1.0)
        flat = x.reshape(-1)
        for v, frac in ((np.nan, 0.05), (np.inf, 0.02), (-np.inf, 0.05)):
            flat[rng.integers(0, flat.size, max(int(flat.size * frac), 1))] = v
    elif mode == "below":  # every score below 0.05: zero detections
        x = np.minimum(rng.standard_normal(shape) - 8.0, -4.0)
    return x.astype(np.float32)


def fuzz_deltas(rng, N, hwa, nonfinite):
    d = normal_deltas(rng, N, hwa)
    if hwa:
        f = d.reshape(-1, 4)
        rows = rng.integers(0, f.shape[0], max(f.shape[0] // 20, 1))
        f[rows, 2:] = rng.choice([-1.0, 1.0], (rows.size, 2)) * rng.uniform(SCALE_CLAMP, 50.0, (rows.size, 2))
        rows = rng.integers(0, f.shape[0], max(f.shape[0] // 50, 1))
        f[rows, :2] = rng.choice([-1.0, 1.0], (rows.size, 2)) * 1e4
        if nonfinite:  # max_coord becomes inf or stays finite while some boxes are NaN
            rows = rng.integers(0, f.shape[0], 2)
            f[rows[0], rng.integers(0, 4)] = rng.choice([np.inf, -np.inf])
            f[rows[1], rng.integers(0, 4)] = np.nan
    return d


def run_fuzz(cuda, oracle_lib, seed):
    rng = np.random.default_rng(7000 + seed)
    N = int(rng.integers(1, 7))
    L = int(rng.integers(1, 9))  # 8 = D2B_MAX_LEVELS
    K = int(rng.choice([1, 2, 7, 80]))
    topk = int(rng.choice([1, 7, 100, 1000, 2049]))
    score_thr = float(rng.choice([0.05, 0.0, 0.5, 0.999, -1.0]))
    nms_thr = float(rng.choice([0.0, 0.5, 1.0]))
    T_det = int(rng.choice([1, 50, 100, 1000]))
    modes = [LOGIT_MODES[int(rng.integers(0, len(LOGIT_MODES)))] for _ in range(N)]
    if "zeros" in modes and rng.random() < 0.5:
        score_thr = 0.5  # p == 0.5 does not pass: the comparison is strict (retinanet.py:329-331)
    big = 5000 if K <= 7 else 1500  # keeps the oracle at milliseconds
    grid = rng.random() < 0.4
    if grid:  # in-kernel anchors: hwa = h * w * A with A = 3
        hws = [[(1, 1), (1, 3), (10, 10), (20, 25)][int(rng.choice(4, p=[0.2, 0.3, 0.3, 0.2]))] for _ in range(L)]
        strides = [8 * 2 ** l for l in range(L)]
        gen = DefaultAnchorGenerator([[32.0 * 2 ** l] for l in range(L)], [list(syn.ASPECT_RATIOS)], strides,
                                     device=cuda)
        desc = gen.grid_descriptors(hws)
        anchors = [a.cpu().numpy() for a in gen.grid_anchors(hws)]
        dev_anchors = desc
    else:
        hwa = [int(rng.choice([1, 7, 300, big], p=[0.15, 0.2, 0.35, 0.3])) for _ in range(L)]
        anchors = [table_anchors(rng, h) for h in hwa]
        dev_anchors = None
    hwa = [a.shape[0] for a in anchors]
    cls = [np.stack([fuzz_logits(rng, (h, K), modes[n]) for n in range(N)]) for h in hwa]
    nonfinite = rng.random() < 0.25
    dl = [fuzz_deltas(rng, N, h, nonfinite) for h in hwa]
    run(cuda, oracle_lib, cls, dl, anchors, K, topk, score_thr, nms_thr, T_det, dev_anchors=dev_anchors)


@pytest.mark.parametrize("seed", range(48))
def test_retinanet_fuzz(cuda, oracle_lib, guard, seed):
    run_fuzz(cuda, oracle_lib, seed)
    guard.check()


# ------------------------------------------------------------------ b. long rows, a different top-k regime per image
def regime_logits(rng, shape, regime):
    """Logits of one image's level.  The rows are longer than 2^20 elements: chunks of kChunkLong = 65,536 elements,
    and topk_prehist takes the cutoff from a sample of the first 1,024 elements of every chunk."""
    n = int(np.prod(shape))
    if regime == "typical":  # the prior: a usable sampled cutoff and a complete candidate list
        x = rng.standard_normal(n) * 1.5 - 4.6
    elif regime == "saturated":  # k-th logit far above 8: no usable cutoff, topk_finish_kernel re-reads the row
        x = rng.standard_normal(n) * 40.0
    elif regime == "misleads":
        # 8 large logits in the sampled window of every chunk: the sample ranks them first, so the cutoff lands at
        # their binade [2, 4) -- but the whole row holds only 8 per chunk (< k) above it, so the exact count of pass 0
        # fails and the `redo` launch repeats pass 0 without a cutoff
        x = rng.standard_normal(n) * 1.5 - 4.6
        for c0 in range(0, n, 65536):
            x[c0 + rng.choice(min(1024, n - c0), 8, replace=False)] = 3.0 + rng.random(8)
    elif regime == "plateau":
        # every logit 1.0 but a few 3.0: the cutoff lands just below 1.0 and the whole row (> kCandCap = 65,536
        # elements) is above it, so the candidate list overflows and the row is re-read
        x = np.full(n, 1.0)
        x[rng.integers(0, n, 500)] = 3.0
    elif regime == "nan":  # all NaN: one pre-histogram bin, no finite cutoff, nothing passes the score threshold
        x = np.full(n, np.nan)
    else:  # "below": every score below 0.05
        x = np.minimum(rng.standard_normal(n) - 8.0, -4.0)
    return x.astype(np.float32).reshape(shape)


REGIMES = ("typical", "saturated", "misleads", "plateau", "nan", "below")


@pytest.mark.parametrize("aligned", [True, False], ids=["aligned", "unaligned"])
def test_retinanet_long_rows_mixed_regimes(cuda, oracle_lib, guard, aligned):
    """Two levels of more than 2^20 elements per row, N = 6, image i in regime REGIMES[i], in the same launches.
    aligned: K = 80, hwa 16,400 and 13,200 (1,312,000 and 1,056,000 elements): every row starts on a 16-byte boundary.
    unaligned: K = 3, hwa 400,002 and 360,002 (rows of 2 mod 4 elements) and the logits placed 4 bytes past a
    16-byte boundary: every row of every image starts misaligned, so topk_prehist samples with scalar loads and
    topk_scan_cut_kernel takes its scalar scan."""
    rng = np.random.default_rng(11 if aligned else 12)
    K, hwa = (80, (16400, 13200)) if aligned else (3, (400002, 360002))
    N = len(REGIMES)
    anchors = [table_anchors(rng, h, 1000, 1300) for h in hwa]
    cls = [np.stack([regime_logits(rng, (h, K), r) for r in REGIMES]) for h in hwa]
    dl = [normal_deltas(rng, N, h) for h in hwa]
    dev_cls = None if aligned else [T_misaligned(x, cuda) for x in cls]
    if not aligned:
        assert all(t.data_ptr() % 16 == 4 for t in dev_cls) and all(h * K % 4 == 2 for h in hwa)
    trace, (_, _, _, wv, _) = run(cuda, oracle_lib, cls, dl, anchors, K, 1000, 0.05, 0.5, 100, dev_cls=dev_cls)
    assert wv[[0, 1, 2, 3]].any(axis=1).all() and not wv[[4, 5]].any()
    # one CTA per kChunkLong chunk of each row: the long-row path
    ctas = N * sum(-(-h * K // 65536) for h in hwa)
    reach(trace, [Launch(kname("topk_scan_cut_kernel"), grid_x=ctas), Launch(kname("topk_finish_kernel"))])
    guard.check()


# ------------------------------------------------------------------ c. branch boundaries
def boundary_inputs(rng, N, hwa, K, loc=-1.0, sd=2.0):
    anchors = [table_anchors(rng, h, 1500, 2000) for h in hwa]
    cls = [(rng.standard_normal((N, h, K)) * sd + loc).astype(np.float32) for h in hwa]
    cls[0][:, ::5] = np.round(cls[0][:, ::5] * 4) / 4  # ties
    dl = [normal_deltas(rng, N, h) for h in hwa]
    return cls, dl, anchors


def run_boundary(cuda, oracle_lib, hwa, K, topk, T_det, N=2, score_thr=0.05, loc=-1.0):
    rng = np.random.default_rng(sum(hwa) + K + topk + T_det)
    cls, dl, anchors = boundary_inputs(rng, N, hwa, K, loc)
    trace, want = run(cuda, oracle_lib, cls, dl, anchors, K, topk, score_thr, 0.5, T_det)
    assert want[3].any()
    return trace, want


def merge_launches(L, k):
    """retina_merge_rank_kernel while the merged keys fit 96 KB of shared memory (stride * 8, stride = L * k), else
    the segment sort of P3 = pad_pow2(stride) keys (sort_local, + sort_big past one 8,192-key tile)."""
    stride = L * k
    if stride * 8 <= 96 * 1024:
        return [Launch(kname("retina_merge_rank_kernel"), dyn_smem=stride * 8)], [kname("sort_big")]
    return [Launch(kname("sort_local")), Launch(kname("sort_big"))], [kname("retina_merge_rank_kernel")]


def tail_launches(stride, T_det):
    """use_lazy(stride, T): det_tail_kernel (20 T bytes of shared memory) else gather + bitmask NMS + emit."""
    if T_det <= 8192 and (stride > 65536 or 8 * T_det <= stride):
        return [Launch(kname("det_tail_kernel"), dyn_smem=20 * T_det)], [kname("nms_mask_kernel"),
                                                                          kname("det_gather_kernel")]
    sweeps = [kname("nms_sweep_cols_kernel"), kname("nms_sweep_cols_cluster_kernel")]
    if (stride + 63) // 64 > 128:  # kSweepClusterMinW
        sweeps.reverse()
    return ([Launch(kname("retina_maxcoord_kernel")), Launch(kname("det_gather_kernel")),
             Launch(kname("nms_mask_kernel")), Launch(sweeps[0]), Launch(kname("det_emit_kernel"))],
            [kname("det_tail_kernel"), sweeps[1]])


def check_branches(trace, L, k, T_det):
    ml, ma = merge_launches(L, k)
    tl, ta = tail_launches(L * k, T_det)
    reach(trace, ml + tl, ma + ta)


BOUNDARY = []
# merge of the level runs: 96 KB of keys (opt-in shared memory above 48 KB) vs the segment sort
for _hwa, _k in (((5000, 4500, 4200), 4096), ((5000, 4500, 4200), 4097),
                 ((2500, 2300, 2100, 2060, 900, 300), 2048), ((2500, 2300, 2100, 2060, 900, 300), 2049)):
    BOUNDARY.append((f"merge-L{len(_hwa)}-k{_k}", dict(hwa=_hwa, K=2, topk=_k, T_det=100)))
# NMS tail: lazy (8 T <= stride) vs the bitmask chain; cluster sweep past W = 128 words; det_tail's attribute
for _hwa, _k, _T in (((6000,), 5000, 625), ((6000,), 5000, 626), ((6000, 5500), 5000, 2000),
                     ((9000, 8500), 8200, 2048), ((9000, 8500), 8200, 2049)):
    BOUNDARY.append((f"tail-stride{len(_hwa) * _k}-T{_T}", dict(hwa=_hwa, K=2, topk=_k, T_det=_T)))
# n above the bitmask limit: lazy at the largest cap
BOUNDARY.append(("tail-stride81920-T8192", dict(hwa=(20000, 18000, 17000, 16500, 16384), K=1, topk=16384,
                                                 T_det=8192, score_thr=0.5, loc=-1.5)))


@pytest.mark.parametrize("params", [p for _, p in BOUNDARY], ids=[i for i, _ in BOUNDARY])
def test_retinanet_boundary(cuda, oracle_lib, guard, params):
    trace, _ = run_boundary(cuda, oracle_lib, **params)
    k = min(params["topk"], max(params["hwa"]))
    check_branches(trace, len(params["hwa"]), k, params["T_det"])
    guard.check()


@pytest.mark.parametrize("hwa", [1 << 20, (1 << 20) + 1])
def test_retinanet_row_length_boundary(cuda, oracle_lib, guard, hwa):
    """K = 1, N = 3: rows of 2^20 elements run in kChunk = 8,192-element chunks (the pre-histogram samples 1,024 of
    every 8,192), rows of 2^20 + 1 in kChunkLong = 65,536-element chunks (1,024 of every 65,536).  The odd length also
    starts the rows of images 1 and 2 off a 16-byte boundary."""
    rng = np.random.default_rng(hwa)
    N = 3
    cls, dl, anchors = boundary_inputs(rng, N, [hwa], 1, loc=-4.6, sd=1.5)
    trace, want = run(cuda, oracle_lib, cls, dl, anchors, 1, 1000, 0.05, 0.5, 100)
    assert want[3].any(axis=1).all()
    chunk = 65536 if hwa > (1 << 20) else 8192
    reach(trace, [Launch(kname("topk_scan_cut_kernel"), grid_x=N * -(-hwa // chunk)),
                  Launch(kname("topk_prehist"), grid_x=N * -(-hwa // (8 * chunk)))])
    guard.check()


@pytest.mark.parametrize("topk", [2048, 2049])
def test_retinanet_topk_sort_boundary(cuda, oracle_lib, guard, topk):
    """Padded k <= kFinSortMax = 2,048: the winners are sorted inside topk_finish_kernel; above it by sort_local.  One
    level, so the merge is the rank kernel and sort_local can only come from the top-k."""
    trace, _ = run_boundary(cuda, oracle_lib, (3000,), 4, topk, 100)
    if topk <= 2048:
        reach(trace, [Launch(kname("topk_finish_kernel")), Launch(kname("retina_merge_rank_kernel"))],
              [kname("sort_local")])
    else:
        reach(trace, [Launch(kname("topk_finish_kernel")), Launch(kname("sort_local"), dyn_smem=12 * 4096)],
              [kname("sort_big")])
    guard.check()


# ------------------------------------------------------------------ d. configs[2] at its batch size
def test_retinanet_config3_batch32(cuda, oracle_lib, guard):
    """BASELINE.json configs[2]: 32 images, K = 80, P3-P7 (201,600 anchors, 16.1 M logits per image), top-1000 per
    level: every image against the oracle, and images 0, 17 and 31 run alone equal their rows of the batch."""
    N, K = 32, 80
    anchors = syn.retinanet_anchors()
    cls, dl = syn.retinanet_inputs(N, K, seed=6, anchors=anchors)
    ta = [T(a, cuda) for a in anchors]
    head = RetinaNetInference(num_classes=K)
    tc, td = [T(x, cuda) for x in cls], [T(x, cuda) for x in dl]
    res = head.inference(tc, td, ta)
    got = {f: res.get_field(f).cpu() for f in ("scores", "pred_classes", "is_valid")}
    got["boxes"] = res.boxes.cpu()
    del res
    wb, ws, wc, wv, wn = oracle_lib.retinanet_inference(cls, dl, anchors, K, 1000, 0.05, 0.5, 100)
    assert (wn > 0).all()
    assert np.array_equal(got["is_valid"].numpy(), wv)
    assert np.array_equal(got["pred_classes"].numpy(), wc)
    assert np.array_equal(got["scores"].numpy().view(np.int32), ws.view(np.int32))
    assert np.array_equal(got["boxes"].numpy(), wb)
    for n in (0, 17, 31):
        one = head.inference([x[n:n + 1] for x in tc], [x[n:n + 1] for x in td], ta)
        assert torch.equal(one.boxes.cpu().view(torch.int32), got["boxes"][n:n + 1].view(torch.int32)), n
        assert torch.equal(one.get_field("scores").cpu().view(torch.int32), got["scores"][n:n + 1].view(torch.int32))
        for f in ("pred_classes", "is_valid"):
            assert torch.equal(one.get_field(f).cpu(), got[f][n:n + 1]), (n, f)
    guard.check()


# ------------------------------------------------------------------ e. rejected before any launch
def small_retina(cuda, L=2, hwa=50, K=3):
    rng = np.random.default_rng(L + hwa + K)
    cls = [T(rng.standard_normal((1, hwa, K)).astype(np.float32), cuda) for _ in range(L)]
    dl = [T(normal_deltas(rng, 1, hwa), cuda) for _ in range(L)]
    an = [T(table_anchors(rng, hwa), cuda) for _ in range(L)]
    return cls, dl, an


def small_frcnn(cuda, R=40, K=5):
    rng = np.random.default_rng(R * K)
    idx = np.stack([np.zeros(R, np.int64), np.arange(R, dtype=np.int64)], 1)
    boxes = fz.fuzz_boxes(rng, R * K, 300, 400).reshape(R, K * 4)
    sc = rng.random((R, K + 1)).astype(np.float32)
    props = SparseBoxList(T(idx, cuda), BoxList(T(fz.fuzz_boxes(rng, R, 300, 400), cuda)), (1, R))
    props.set_tracking("image_shape", T(np.array([[300, 400]], np.int32), cuda))
    return T(boxes, cuda), T(sc, cuda), props


def small_yolo(cuda, n=200, K=4):
    rng = np.random.default_rng(n + K)
    return T(fz.fuzz_boxes(rng, n, 300, 400)[None], cuda), T(rng.random((1, n, K)).astype(np.float32), cuda)


BAD_THRESHOLDS = [1.5, -0.1, float("nan")]


@pytest.mark.parametrize("thr", BAD_THRESHOLDS, ids=["1.5", "-0.1", "nan"])
def test_rejects_nms_threshold_before_launch(cuda, guard, thr):
    """nms_threshold outside [0, 1] (NaN included), as tf.image.non_max_suppression: rejected by the plans of the three
    detection heads before top-k / prep / sort launch, not by the NMS after them."""
    msg = "nms_thresh must be in"
    cls, dl, an = small_retina(cuda)
    _rejected(guard, lambda: RetinaNetInference(3, 100, 0.05, thr, 20).inference(cls, dl, an), msg)
    boxes, sc, props = small_frcnn(cuda)
    _rejected(guard, lambda: fast_rcnn_inference(boxes, sc, props, 0.05, thr, 20, False), msg)
    _rejected(guard, lambda: fast_rcnn_inference(None, sc, props, 0.05, thr, 20, False, pred_proposal_deltas=boxes,
                                                 box2box_transform=Box2BoxTransform((10., 10., 5., 5.))), msg)
    yb, yp = small_yolo(cuda)
    _rejected(guard, lambda: YOLOv4Inference(0.2, thr, 20).inference(yb, yp), msg)


def test_rejects_unsupported_nms_sizes_in_heads(cuda, guard):
    """n > kBitmaskMaxN = 65,536 candidates per image with a cap > kLazyMaxOut = 8,192 (nms.cu nms_check_sizes):
    RetinaNet L * k = 5 * 16,384, Fast R-CNN Rmax * K = 1,000 * 80, YOLOv4 n = 65,537."""
    cls, dl, an = small_retina(cuda, L=5, hwa=16384, K=1)
    _rejected(guard, lambda: RetinaNetInference(1, 16384, 0.05, 0.5, 8193).inference(cls, dl, an),
              "n=81920 with max_output_size=8193 is not supported")
    boxes, sc, props = small_frcnn(cuda, R=1000, K=80)
    _rejected(guard, lambda: fast_rcnn_inference(boxes, sc, props, 0.05, 0.5, 8193, False),
              "n=80000 with max_output_size=8193 is not supported")
    yb, yp = small_yolo(cuda, n=65537, K=2)
    _rejected(guard, lambda: YOLOv4Inference(0.2, 0.5, 8193).inference(yb, yp),
              "n=65537 with max_output_size=8193 is not supported")
