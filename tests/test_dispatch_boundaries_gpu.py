"""GPU: every kernel path that the host code selects from the input sizes, run on both sides of its threshold and
compared with the oracle at the bar of the other GPU files (integers, orders and fp32 values bit-exact; a bf16 output
equals the oracle's fp32 result, computed on the bf16-rounded inputs, rounded to bf16).

The thresholds are compile-time constants in csrc/ (template instantiations, opt-in shared memory above 48 KB,
grid limits, the fused/generic split).  Each case of CASES names the branch, the constant and the host function that
selects it, and a reach check runs the call under torch.profiler and asserts that the branch's kernel -- and, where the
branch is a launch parameter, its dynamic shared memory or grid -- was launched.  A moved threshold or a re-tuned knob
then fails here instead of silently dropping the coverage.  Two branches live inside one kernel: paste_boxes_kernel
reads the mask from shared or global memory, which shows as its shared memory size; the fallback of rpn_select_kernel
does not show in a trace, so its case says why the input forces it.  Every case runs inside the canary bands of
test_canary_gpu, so a write one element past an output or workspace fails even when the values match."""
import collections
import json
import os
import re
import tempfile
import warnings

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.layers import batch_nms, matrix_nms, segmented_top_k
from detectron2_tensorflow_b200.layers.functional import _roi_align_call
from detectron2_tensorflow_b200.modeling import Box2BoxTransform, Matcher, ROIPooler, find_top_rpn_proposals, label_boxes
from detectron2_tensorflow_b200.structures import BoxList, ImageList, SparseBoxList, reframe_box_masks_to_image_masks
from detectron2_tensorflow_b200.utils import synthetic as syn

from test_canary_gpu import Guard
import test_fuzz_gpu as fz

pytestmark = pytest.mark.gpu

# A trace reports static + dynamic shared memory per block.  The static part (the kernel's own arrays and the 1 KB
# the system reserves per block) is below this for every kernel checked here; the largest, 12 KB, is the sweep state
# of nms_sweep_columns in rpn_sweep_merge_kernel.
STATIC_SMEM_MAX = 16 * 1024


# ------------------------------------------------------------------ reach check
def traced(fn):
    """Run fn() under torch.profiler; returns (fn's result, [(kernel name, kernel args)]), or (result, None) when the
    profiler cannot trace CUDA activity here (the values are still compared; only the reach check is skipped)."""
    acts = torch.profiler.supported_activities()
    if torch.profiler.ProfilerActivity.CUDA not in acts:
        warnings.warn("torch.profiler has no CUDA activity: reach checks skipped")
        return fn(), None
    with tempfile.TemporaryDirectory() as d:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return out, [(e["name"], e.get("args", {})) for e in events if e.get("cat") == "kernel"]


class Launch(object):
    """A kernel the case must launch, by name pattern.  Optional checks on every launch of it: the dynamic shared memory
    it was given (bytes; 0 = none) and grid.x; and on all of them: the sorted list of their grid.y."""

    def __init__(self, pattern, dyn_smem=None, grid_x=None, grid_ys=None):
        self.pattern, self.dyn_smem, self.grid_x, self.grid_ys = pattern, dyn_smem, grid_x, grid_ys

    def check(self, trace):
        hits = [a for n, a in trace if re.search(self.pattern, n)]
        assert hits, f"no launch of {self.pattern}; launched: {sorted({n for n, _ in trace})}"
        for a in hits:
            s = a["shared memory"]
            assert self.dyn_smem is None or self.dyn_smem <= s <= self.dyn_smem + STATIC_SMEM_MAX, \
                (self.pattern, s, self.dyn_smem)
            assert self.grid_x is None or a["grid"][0] == self.grid_x, (self.pattern, a["grid"], self.grid_x)
        if self.grid_ys is not None:
            assert sorted(a["grid"][1] for a in hits) == sorted(self.grid_ys), (self.pattern, [a["grid"] for a in hits])


def reach(trace, launches=(), absent=()):
    if trace is None:
        return
    for l in launches:
        l.check(trace)
    for pat in absent:
        bad = sorted({n for n, _ in trace if re.search(pat, n)})
        assert not bad, f"{pat} must not run here; launched {bad}"


def K(name):
    """Pattern for a kernel by its unqualified name (template arguments may follow)."""
    return r"(?<!\w)" + name + r"(?!\w)"


@pytest.fixture
def guard(monkeypatch):
    return Guard(monkeypatch)


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


# ------------------------------------------------------------------ ROIAlign forward, bf16 features
RA_GROUPS = {64: 0, 256: 1, 512: 2}  # C / 8 bf16 per 16-byte group: 32 -> GROUPS 1, 64 -> GROUPS 2, else generic
RA_S1 = {0: 1, 2: 2, 3: 0}           # sampling_ratio 0/1 -> S1 1, 2 -> S1 2, else runtime loop


def run_roi_align_bf16(cuda, oracle_lib, C, sr, out):
    N, R = 2, 80
    feats = syn.fpn_features(N, C, seed=C + sr, padded_hw=(128, 192))
    boxes, idx = syn.rois(N, R, seed=sr + 1, image_hw=(120, 190))
    scales = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]
    tb = [torch.from_numpy(f).to(cuda).to(torch.bfloat16) for f in feats]
    ref_in = [t.float().cpu().numpy() for t in tb]
    want, _ = oracle_lib.roi_pooler(ref_in, scales, boxes, idx[:, 0], (7, 7), sr)
    odt = torch.bfloat16 if out == "bf16" else torch.float32
    bt, it = T(boxes, cuda), T(idx[:, 0], cuda)
    got, trace = traced(lambda: _roi_align_call(tb, scales, bt, it, 1, (7, 7), sr, True, True, min_level=2,
                                                 canonical_box_size=224, canonical_level=4, out_dtype=odt))
    assert got.dtype == odt
    if out == "bf16":
        want = torch.from_numpy(want).to(torch.bfloat16).float().numpy()
    assert np.array_equal(got.float().cpu().numpy(), want)
    g, s = RA_GROUPS[C], RA_S1[sr] if RA_GROUPS[C] else 0
    tout = "__nv_bfloat16" if out == "bf16" else "float"
    reach(trace, [Launch(r"roi_align_kernel<__nv_bfloat16,\s*%s,\s*%d,\s*%d>" % (tout, g, s))])


# ------------------------------------------------------------------ label_boxes
def run_label_boxes(cuda, oracle_lib, G, lq):
    rng = np.random.default_rng(G + 7 * lq)
    N, P = 2, 3000
    pred = np.stack([fz.fuzz_boxes(rng, P, 300, 400) for _ in range(N)])
    gt = np.stack([fz.fuzz_boxes(rng, G, 300, 400) for _ in range(N)])
    gt[:, 0] = pred[:, 5]  # exact matches
    gt[:, G - 1] = pred[:, 9]  # ... also in the last staged slot
    valid, crowd, diff = rng.random((N, G)) < 0.8, rng.random((N, G)) < 0.1, rng.random((N, G)) < 0.1
    counts = np.array([P, P - 123], np.int32)
    shapes = np.array([[280, 390], [300, 400]], np.int32)
    th, lab, w = [0.3, 0.7], [0, -1, 1], (10., 10., 5., 5.)
    wm, wl, wd = oracle_lib.label_boxes(pred, gt, valid, th, lab, lq, gt_crowd=crowd, gt_difficult=diff,
                                        pred_counts=counts, boundary_threshold=0.0, image_shapes=shapes, weights=w)
    args = [T(a, cuda) for a in (pred, gt, valid, crowd, diff, counts, shapes)]
    (gm, gl, gd), trace = traced(lambda: label_boxes(
        args[0], args[1], args[2], Matcher(th, lab, lq), gt_crowd=args[3], gt_difficult=args[4], pred_counts=args[5],
        boundary_threshold=0.0, image_shapes=args[6], box2box_transform=Box2BoxTransform(w)))
    assert np.array_equal(gl.cpu().numpy(), wl)
    assert np.array_equal(gm.cpu().numpy(), wm)
    assert np.array_equal(gd.cpu().numpy(), wd, equal_nan=True)
    smem = 76 * G + 48  # label_smem_bytes; above 48 KB from G = 647
    launches = [Launch(K("label_kernel"), dyn_smem=smem)]
    if lq:
        launches.append(Launch(K("label_gtmax_kernel"), dyn_smem=smem))
    reach(trace, launches, absent=() if lq else (K("label_gtmax_kernel"),))


# ------------------------------------------------------------------ paste_masks
def run_paste_big_masks(cuda, oracle_lib, mh, mw):
    rng = np.random.default_rng(mh * mw)
    H, W, M = 800, 1333, 36
    yy, xx = np.mgrid[0:mh, 0:mw].astype(np.float32)
    cy, cx, r = (rng.uniform(0.3, 0.7, (M, 1, 1)) * mh, rng.uniform(0.3, 0.7, (M, 1, 1)) * mw,
                 rng.uniform(0.2, 0.5, (M, 1, 1)) * min(mh, mw))
    masks = (1.0 / (1.0 + np.exp(np.hypot(yy - cy, xx - cx) - r)) + rng.uniform(-0.05, 0.05, (M, mh, mw)))
    masks = masks.astype(np.float32)
    boxes, _ = syn.rois(1, M, seed=mh + mw, image_hw=(H, W))
    boxes[0] = [-20, -30, H + 10, W + 5]
    boxes[1] = [400, 700, 300, 500]  # reversed
    want = oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W), 0.5)
    tm, tb = T(masks, cuda), T(boxes, cuda)
    got, trace = traced(lambda: reframe_box_masks_to_image_masks(tm, tb, (H, W), 0.5))
    assert np.array_equal(got.cpu().numpy(), want)
    assert want.sum() > 0
    # kMaxMaskSmem: up to 16,384 floats the mask is staged in shared memory (above 48 KB from 12,289), else read from
    # global memory
    reach(trace, [Launch(K("paste_boxes_kernel"), dyn_smem=4 * mh * mw if mh * mw <= 16384 else 0)])


def run_paste_many_masks(cuda, oracle_lib, M):
    rng = np.random.default_rng(M)
    H = W = 8
    masks = rng.random((M, 7, 7)).astype(np.float32)
    y0, x0 = rng.uniform(-3, 8, M), rng.uniform(-3, 8, M)
    boxes = np.stack([y0, x0, y0 + rng.uniform(-1, 9, M), x0 + rng.uniform(-1, 9, M)], 1).astype(np.float32)
    want = oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W), 0.5)
    tm, tb = T(masks, cuda), T(boxes, cuda)
    got, trace = traced(lambda: reframe_box_masks_to_image_masks(tm, tb, (H, W), 0.5))
    assert np.array_equal(got.cpu().numpy(), want)
    chunks = [min(65535, M - m0) for m0 in range(0, M, 65535)]  # one launch per grid.y chunk
    reach(trace, [Launch(K("paste_boxes_kernel"), grid_ys=chunks)])


# ------------------------------------------------------------------ Matrix-NMS
def blob_masks(rng, n, H, W, classes=4):
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    m = np.zeros((n, H, W), np.float32)
    for i in range(n):
        cy, cx = rng.uniform(0, H), rng.uniform(0, W)
        ry, rx = rng.uniform(0.05, 0.5) * H, rng.uniform(0.05, 0.5) * W
        m[i] = (((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0)
    m[n // 2:n // 2 + n // 8] = m[:n // 8]  # exact duplicates
    cls = rng.integers(0, classes, n).astype(np.int64)
    sc = np.sort(rng.random(n).astype(np.float32))[::-1].copy()
    return m, cls, sc


def run_matrix_nms(cuda, oracle_lib, n, H, W, kernel):
    rng = np.random.default_rng(n + H * W)
    if H * W > 1000:
        m, cls, sc = blob_masks(rng, n, H, W)
    else:
        m = (rng.random((n, H, W)) < rng.uniform(0.1, 0.6, (n, 1, 1))).astype(np.float32)
        m[n // 2:n // 2 + n // 8] = m[:n // 8]
        cls = rng.integers(0, 5, n).astype(np.int64)
        sc = np.sort(rng.random(n).astype(np.float32))[::-1].copy()
    want = oracle_lib.matrix_nms(m, cls, sc, None, kernel, 2.0)
    tm, tc, ts = T(m, cuda), T(cls, cuda), T(sc, cuda)
    got, trace = traced(lambda: matrix_nms(tm, tc, ts, kernel=kernel, sigma=2.0))
    assert np.array_equal(got.cpu().numpy(), want, equal_nan=True)
    iou_row = 8 * ((H * W + 63) // 64)  # one packed mask row, staged up to 160 KB, else re-read from L2 per pair
    launches = [Launch(K("mnms_iou_kernel"), dyn_smem=iou_row if iou_row <= 160 * 1024 else 0)]
    if n <= 4096:  # kDecayStageMax: the per-row table fits shared memory
        launches.append(Launch(r"mnms_decay_kernel<true>", dyn_smem=20 * n))
        absent = (r"mnms_decay_kernel<false>",)
    else:
        launches.append(Launch(r"mnms_decay_kernel<false>"))
        absent = (r"mnms_decay_kernel<true>",)
    reach(trace, launches, absent)


# ------------------------------------------------------------------ segmented top-k
def run_topk(cuda, oracle_lib, k, sigmoid):
    rng = np.random.default_rng(k + sigmoid)
    N = 2
    rows = [(rng.standard_normal((N, ln)) * 3).astype(np.float32) for ln in (k + 1, 3 * k + 5)]
    rows[1][:, ::7] = np.round(rows[1][:, ::7])  # ties
    (vals, idx, cnt), trace = traced(lambda: segmented_top_k([T(r, cuda) for r in rows], k, sigmoid=sigmoid))
    vals, idx, cnt = vals.cpu().numpy(), idx.cpu().numpy(), cnt.cpu().numpy()
    for n in range(N):
        for l, r in enumerate(rows):
            x = oracle_lib.sigmoid_array(r[n]) if sigmoid else r[n]
            wv, wi = oracle_lib.top_k(x, k)
            assert cnt[n, l] == len(wi) == k
            assert np.array_equal(idx[n, l], wi), (n, l)
            assert np.array_equal(vals[n, l], wv)
    P = 1 << (k - 1).bit_length()  # topk_padded_k
    if sigmoid and P <= 2048:  # kFinSortMax: sorted inside topk_finish_kernel
        launches, absent = [Launch(K("topk_finish_kernel"))], [K("sort_local")]
    else:
        tile = min(P, 8192)  # sort.cu kTile; 1.5 keys of shared memory per key
        launches, absent = [Launch(K("sort_local"), dyn_smem=12 * tile)], []
    if P > 8192:  # segments longer than one tile
        launches.append(Launch(K("sort_big")))
    else:
        absent.append(K("sort_big"))
    reach(trace, launches, absent)


def run_topk_long_rows(cuda, oracle_lib, length):
    rng = np.random.default_rng(length)
    N, k = 2, 1000
    x = (rng.standard_normal((N, length)) * 2).astype(np.float32)
    x[:, -1] = 100.0  # the last element of the row wins
    x[:, ::3] = np.round(x[:, ::3] * 4) / 4
    (vals, idx, cnt), trace = traced(lambda: segmented_top_k([T(x, cuda)], k))
    for n in range(N):
        wv, wi = oracle_lib.top_k(x[n], k)
        assert np.array_equal(idx[n, 0].cpu().numpy(), wi)
        assert np.array_equal(vals[n, 0].cpu().numpy(), wv)
        assert wi[0] == length - 1
    chunk = 65536 if length > (1 << 20) else 8192  # kChunkLong / kChunk
    reach(trace, [Launch(K("topk_hist"), grid_x=N * -(-length // chunk))])  # one CTA per chunk of each row


# ------------------------------------------------------------------ batched NMS
def run_nms(cuda, oracle_lib, n, max_out, B):
    rng = np.random.default_rng(n + max_out)
    boxes = np.stack([fz.fuzz_boxes(rng, n, 2000, 3000) for _ in range(B)])
    scores = np.stack([fz.fuzz_scores(rng, (n,)) for _ in range(B)])
    (keep, num), trace = traced(lambda: batch_nms(T(boxes, cuda), T(scores, cuda), max_out, axis=1, iou_threshold=0.5))
    keep, num = keep.cpu().numpy(), num.cpu().numpy()
    for b in range(B):
        want = oracle_lib.nms(boxes[b], scores[b], max_out, 0.5)
        assert num[b] == len(want), b
        assert np.array_equal(keep[b, :len(want)], want), b
        assert np.all(keep[b, len(want):] == -1)
    if n <= 512:  # kSmallMaxN
        reach(trace, [Launch(K("nms_small_kernel"))], [K("nms_prep_kernel")])
        return
    lazy = max_out <= 8192 and (n > 65536 or max_out * 8 <= n)  # use_lazy: kLazyMaxOut, kBitmaskMaxN
    if lazy:
        reach(trace, [Launch(K("nms_prep_kernel")), Launch(K("nms_lazy_kernel"), dyn_smem=16 * max_out)],
              [K("nms_mask_kernel")])
        return
    sweeps = [K("nms_sweep_cols_kernel"), K("nms_sweep_cols_cluster_kernel")]
    if (n + 63) // 64 > 128:  # kSweepClusterMinW
        sweeps.reverse()
    reach(trace, [Launch(K("nms_mask_kernel")), Launch(sweeps[0])], [K("nms_lazy_kernel"), K("nms_small_kernel"), sweeps[1]])


# ------------------------------------------------------------------ RPN proposals
def run_rpn(cuda, oracle_lib, pre, post=1000, hwa=None):
    """hwa=None: the full-size P2 level (201,600 anchors), one image, every logit the same."""
    rng = np.random.default_rng(pre + post)
    thr = 0.7
    if hwa is None:
        anchors = syn.rpn_anchors()[0]
        d = (rng.standard_normal((1, anchors.shape[0], 4)) * np.array([0.3, 0.3, 0.2, 0.2])).astype(np.float32)
        props = [oracle_lib.rpn_predict_proposals(d, anchors)]
        logits = [np.full((1, anchors.shape[0]), 0.25, np.float32)]
        shapes = syn.image_shapes(1)
        hwa = [anchors.shape[0]]
    else:
        N = 2
        props = [np.stack([fz.fuzz_boxes(rng, h, 300, 400) for _ in range(N)]) for h in hwa]
        logits = [(np.round(rng.standard_normal((N, h)) * 16) / 16).astype(np.float32) for h in hwa]
        shapes = np.array([[300, 400], [280, 390]], np.int32)
    wb, wl, wv, _ = oracle_lib.find_top_rpn_proposals(props, logits, shapes, thr, pre, post, 0.0)
    tp, tl, ts = [T(p, cuda) for p in props], [T(x, cuda) for x in logits], T(shapes, cuda)
    res, trace = traced(lambda: find_top_rpn_proposals(tp, tl, ImageList(None, ts), thr, pre, post, 0.0))
    assert np.array_equal(res.get_field("is_valid").cpu().numpy(), wv)
    assert np.array_equal(res.boxes.cpu().numpy(), wb)
    assert np.array_equal(res.get_field("objectness_logits").cpu().numpy(), wl)
    assert wv.any()
    if pre > 4096:  # kRpnFusedMaxK
        reach(trace, [Launch(K("topk_hist"))], [K("rpn_select_kernel"), K("rpn_sweep_merge_kernel")])
        return
    # pipelines.cu: the fused sweep + merge runs when NMS uses the bitmask and L * 4 + 2 bytes per survivor fit
    L, k = len(hwa), min(pre, max(hwa))
    cap = min(post, k)
    lazy = post <= 8192 and (k > 65536 or post * 8 <= k)
    if not lazy and (4 * L + 2) * cap + 16 <= 200 * 1024:
        dyn = L * cap * 4 + -(-2 * cap // 16) * 16  # rpn_sweep_merge_fused
        reach(trace, [Launch(K("rpn_select_kernel")), Launch(K("rpn_sweep_merge_kernel"), dyn_smem=dyn)],
              [K("topk_hist"), K("rpn_merge_rank_kernel")])
    else:
        reach(trace, [Launch(K("rpn_select_kernel"))], [K("topk_hist"), K("rpn_sweep_merge_kernel")])


# ------------------------------------------------------------------ ROIPooler, 8 levels
def run_pooler_8_levels(cuda, oracle_lib):
    rng = np.random.default_rng(8)
    N, C, img = 2, 8, 512
    scales = [2.0 ** -l for l in range(1, 9)]  # levels 1..8 = D2B_MAX_LEVELS
    feats = [rng.standard_normal((N, img >> l, img >> l, C)).astype(np.float32) for l in range(1, 9)]
    M = 400
    side = np.exp(rng.uniform(np.log(1.0), np.log(500.0), M))
    cy, cx = rng.uniform(0, img, M), rng.uniform(0, img, M)
    boxes = np.stack([cy - side / 2, cx - side / 2, cy + side / 2, cx + side / 2], 1).astype(np.float32)
    bidx = rng.integers(0, N, M).astype(np.int64)
    want, wc = oracle_lib.roi_pooler(feats, scales, boxes, bidx, (7, 7), 2, True, canonical_box_size=16,
                                     canonical_level=4)
    assert (wc > 0).all(), wc  # every level, the eighth included, receives boxes
    pooler = ROIPooler(7, scales, 2, "ROIAlignV2", canonical_box_size=16, canonical_level=4)
    idx = np.stack([bidx, np.arange(M, dtype=np.int64)], 1)
    inst = SparseBoxList(T(idx, cuda), BoxList(T(boxes, cuda)), (N, M))
    tf = [T(f, cuda) for f in feats]
    got, trace = traced(lambda: pooler(tf, inst))
    assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(pooler.last_level_counts.cpu().numpy(), wc)
    reach(trace, [Launch(r"roi_align_kernel<float,\s*float,\s*0,\s*0>")])


# ------------------------------------------------------------------ the table
Case = collections.namedtuple("Case", "id branch constant source run params")
CASES = []


def case(id, branch, constant, source, run, **params):
    CASES.append(Case(id, branch, constant, source, run, params))


for _C in (64, 256, 512):
    for _sr in (0, 2, 3):
        for _out in ("bf16", "fp32"):
            case(f"roi_align-bf16-C{_C}-sr{_sr}-{_out}",
                 f"roi_align_kernel<bf16, {_out}, GROUPS={RA_GROUPS[_C]}, S1={RA_S1[_sr] if RA_GROUPS[_C] else 0}>",
                 "C / 8 == 32 or 64 -> GROUPS 1 / 2; sampling_ratio 0, 1 / 2 -> S1 1 / 2", "roi_align.cu launch",
                 run_roi_align_bf16, C=_C, sr=_sr, out=_out)
for _G in (646, 647, 1024):
    for _lq in (False, True):
        case(f"label_boxes-G{_G}-lq{int(_lq)}", "label_kernel / label_gtmax_kernel staged GT above 48 KB",
             "label_smem_bytes(G) = 76 G + 48 > 48 KB (G >= 647); D2B_MATCH_MAX_GT = 1024", "matcher.cu d2b_label_boxes",
             run_label_boxes, G=_G, lq=_lq)
for _mh, _mw in ((110, 110), (111, 111), (128, 128), (128, 129)):
    case(f"paste-mask{_mh}x{_mw}", "paste_boxes_kernel: mask in default / opt-in shared memory, or read from global",
         "4 mh mw > 48 KB (mh mw > 12,288); kMaxMaskSmem = 16,384", "paste_masks.cu d2b_paste_masks",
         run_paste_big_masks, mh=_mh, mw=_mw)
for _M in (65535, 65536, 70000):
    case(f"paste-{_M}-masks", "paste_boxes_kernel: second grid.y chunk", "grid.y limit 65,535 (m0 += 65535)",
         "paste_masks.cu d2b_paste_masks", run_paste_many_masks, M=_M)
# 624 x 630: a 49,144-byte row is below 48 KB, but mnms_iou_kernel has 1 KB of static shared memory, so the row only
# fits after raising the kernel's limit (it failed to launch while the limit was raised above 48 KB only).
for _n, _H, _W, _kern in ((24, 624, 630, "gaussian"), (24, 640, 640, "linear"), (12, 1024, 1280, "gaussian"),
                          (12, 1152, 1152, "linear")):
    case(f"matrix_nms-iou-{_n}x{_H}x{_W}", "mnms_iou_kernel: row staged in default / opt-in smem, or unstaged",
         "8 ceil(hw / 64) > 48 KB (hw > 393,216); > 160 KB (hw > 1,310,720) unstaged", "matrix_nms.cu d2b_matrix_nms",
         run_matrix_nms, n=_n, H=_H, W=_W, kernel=_kern)
for _n in (1638, 1639, 2458, 4096, 4097):
    case(f"matrix_nms-decay-n{_n}", "mnms_decay_kernel<true> (table in smem, attribute above 32 KB) vs <false>",
         "20 n > 32 KB (n >= 1,639), > 48 KB (n >= 2,458); kDecayStageMax = 4,096", "matrix_nms.cu d2b_matrix_nms",
         run_matrix_nms, n=_n, H=6, W=10, kernel="gaussian" if _n % 2 else "linear")
for _k in (2048, 2049, 8192, 8193, 16384):
    for _sig in (False, True):
        case(f"topk-k{_k}-{'sigmoid' if _sig else 'identity'}",
             "winners sorted in topk_finish_kernel / sort_local / + sort_big",
             "padded k > kFinSortMax = 2,048; > kTile = 8,192; kTopkMaxK = 16,384", "topk.cu topk_run, sort.cu",
             run_topk, k=_k, sigmoid=_sig)
for _len in (1 << 20, (1 << 20) + 1):
    case(f"topk-identity-row{_len}", "row chunks of kChunk vs kChunkLong elements", "row_len > 2^20 -> kChunkLong",
         "topk.cu fill_args", run_topk_long_rows, length=_len)
# n = 400: nms_small_smem = 40,896 bytes is below 48 KB, but with the kernel's 12 KB of static shared memory it is above
# the default dynamic limit (48 KB minus the static size): it failed to launch in a process that had not yet raised the
# limit for a larger n.
for _n in (400, 512, 513, 8192, 8193):
    case(f"nms-n{_n}-uncapped", "nms_small_kernel / prep+sort+mask, sweep_cols vs sweep_cols_cluster",
         "kSmallMaxN = 512; nms_small_smem vs 48 KB - static; W = ceil(n / 64) > kSweepClusterMinW = 128",
         "boxes.cu d2b_batched_nms, nms.cu nms_small / nms_sorted",
         run_nms, n=_n, max_out=_n, B=2)
# cap 3,072: 49,152 bytes of kept boxes plus 1.5 KB of static shared memory in nms_lazy_kernel (failed to launch while
# the limit was raised above 48 KB only).
for _n, _mo, _B in ((800, 100, 2), (799, 100, 2), (24576, 3072, 1), (24584, 3073, 1), (65536, 8192, 1),
                    (65537, 100, 1)):
    case(f"nms-n{_n}-cap{_mo}", "nms_lazy_kernel (opt-in smem above 3,072 kept boxes) vs bitmask",
         "max_out * 8 <= n; 16 max_out > 48 KB; kLazyMaxOut = 8,192; n > kBitmaskMaxN = 65,536",
         "nms.cu use_lazy / nms_sorted", run_nms, n=_n, max_out=_mo, B=_B)
for _pre in (4096, 4097):
    case(f"rpn-pre{_pre}", "cluster-fused rpn_select_kernel vs generic top-k chain", "kRpnFusedMaxK = 4,096",
         "pipelines.cu (fused_select)", run_rpn, pre=_pre, hwa=[9000, 700])
# rpn_sweep_merge_kernel has 12 KB of static shared memory (nms_sweep_columns), so its default dynamic limit is
# 36,816 bytes, not 48 KB.  L * cap * 4 + 2 * cap bytes: 36,800 (below), 36,832 and 40,960 (between 36,816 and 48 KB:
# both failed to launch before the limit was read from the kernel), 90,112 (opt-in).
for _hwa, _post in (([9000, 700], 3680), ([9000, 700], 3682), ([9000, 700], 4096), ([9000, 3000, 700, 300, 120], 4096)):
    case(f"rpn-sweep-merge-L{len(_hwa)}-post{_post}", "rpn_sweep_merge_kernel dynamic shared memory vs its limit",
         "L * cap * 4 + align16(2 cap) vs 48 KB - static", "rpn_fused.cu rpn_sweep_merge_fused", run_rpn, pre=4096,
         post=_post, hwa=_hwa)
# rpn_select_kernel resolves the boundary bucket by ranking when it holds <= kCandCap = 256 elements and no warp's raw
# list overflowed; all logits equal => the boundary bucket is the whole row (201,600 > 256), so the in-kernel radix
# passes with tie quotas finish the selection.  The trace can only show rpn_select_kernel itself.
case("rpn-equal-logits-p2", "rpn_select_kernel fallback (radix passes + tie quotas)", "kCandCap = 256",
     "rpn_fused.cu rpn_select_kernel", run_rpn, pre=1000)
case("rpn-8-levels", "num_levels == D2B_MAX_LEVELS", "D2B_MAX_LEVELS = 8", "pipelines.cu, rpn_fused.cu", run_rpn,
     pre=300, hwa=[3000, 1500, 700, 300, 120, 50, 20, 9])
case("roi_pooler-8-levels", "num_levels == D2B_MAX_LEVELS", "D2B_MAX_LEVELS = 8", "roi_align.cu fill_args",
     run_pooler_8_levels)


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_dispatch_boundary(cuda, oracle_lib, guard, c):
    c.run(cuda, oracle_lib, **c.params)
    guard.check()


# ------------------------------------------------------------------ limits: rejected on the host, nothing launched
def _rejected(guard, fn, match):
    before = nv.lib().d2b_kernel_launch_count()
    # D2B_EINVAL: _native.call raises ValueError for it, as the reference raises ValueError / asserts on bad arguments;
    # D2BError is for CUDA and workspace failures.
    with pytest.raises(ValueError, match=match):
        fn()
    assert nv.lib().d2b_kernel_launch_count() == before, "a rejected call launched kernels"
    guard.check()


def test_rejects_max_gt_above_limit(cuda, guard):
    """D2B_MATCH_MAX_GT = 1024 (matcher.cu d2b_label_boxes)."""
    rng = np.random.default_rng(0)
    pred, gt = T(fz.fuzz_boxes(rng, 100, 300, 400), cuda), T(fz.fuzz_boxes(rng, 1025, 300, 400)[None], cuda)
    valid = torch.ones((1, 1025), dtype=torch.bool, device=cuda)
    _rejected(guard, lambda: label_boxes(pred, gt, valid, Matcher([0.5], [0, 1], True)), "max_gt=1025 > 1024")


def test_rejects_k_above_limit(cuda, guard):
    """kTopkMaxK = 16,384 (topk.cu topk_run)."""
    x = torch.randn((1, 20000), device=cuda)
    for sig in (False, True):
        _rejected(guard, lambda: segmented_top_k([x], 16385, sigmoid=sig), "k=16385 out of")


def test_rejects_unsupported_nms_sizes(cuda, guard):
    """n > kBitmaskMaxN = 65,536 with max_out > kLazyMaxOut = 8,192 (nms.cu nms_check_sizes): checked before the
    ordering launches of d2b_batched_nms, which used to run its memset, prep, sort and gather kernels (and ask for a
    540 MB mask workspace) before nms_sorted rejected the sizes."""
    rng = np.random.default_rng(1)
    n = 65537
    boxes, scores = T(fz.fuzz_boxes(rng, n, 300, 400)[None], cuda), torch.randn((1, n), device=cuda)
    _rejected(guard, lambda: batch_nms(boxes, scores, 8193, axis=1), "n=65537 with max_output_size=8193 is not supported")
