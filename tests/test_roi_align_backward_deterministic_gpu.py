"""GPU: the deterministic ROIAlign / ROIPooler backward (`deterministic=True`) against the CPU kernel, bit for bit.

The mode sums every padded-gradient pixel in the order TF's CPU CropAndResizeGradImage + MirrorPadGrad use (ROIs in
input order per level, crop rows, crop columns, TL/TR/BL/BR, then the border fold in raster order), so the result
must equal the oracle's float32 bits exactly -- including where NaN and inf land, which the order decides (inf - inf)
-- and must not change from call to call, with stream, or with how the batch is split into image blocks.  The default
mode stays the atomic kernel, with no workspace."""
import ctypes as C

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.layers import ROIAlign
from detectron2_tensorflow_b200.modeling import ROIPooler
from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList
from detectron2_tensorflow_b200.utils import synthetic as syn

from test_canary_gpu import Guard
from test_dispatch_boundaries_gpu import traced

pytestmark = pytest.mark.gpu

SCALES = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def bits(a):
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bits(got, want):
    """Equal float32 bits.  A NaN only has to be a NaN: its payload is not an IEEE result (x86 produces the negative
    default NaN for inf - inf, the GPU the canonical 0x7fffffff), so NaN positions are compared instead."""
    g, w = bits(got), bits(want)
    assert g.shape == w.shape
    gn, wn = np.isnan(g.view(np.float32)), np.isnan(w.view(np.float32))
    assert np.array_equal(gn, wn), f"NaN positions differ at {np.flatnonzero((gn != wn).ravel())[:5]}"
    bad = np.flatnonzero((g != w).ravel() & ~gn.ravel())
    assert bad.size == 0, f"{bad.size} of {g.size} words differ, first at flat index {bad[:5]}"


def adversarial_boxes(rng, N, H, W, stride, M):
    """Random boxes plus every corner case of the tap rule, in image pixels (feature map = image / stride)."""
    Hi, Wi = H * stride, W * stride
    cy, cx = rng.uniform(0, Hi, M), rng.uniform(0, Wi, M)
    h, w = rng.uniform(2, Hi / 2, M), rng.uniform(2, Wi / 2, M)
    b = np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], 1).astype(np.float32)
    bi = rng.integers(0, N, M).astype(np.int32)
    extra = [
        [Hi + 100, 10, Hi + 300, 50],                               # fully outside
        [-50, -80, 40, 30], [Hi - 20, Wi - 30, Hi + 60, Wi + 90],   # partly outside
        [30, 40, 30, 40], [5.5 * stride, 7.5 * stride] * 2,         # zero size: every sample on one point
        [100, 100, 100.3, 100.2], [10, 20, 10.5, 20.5],             # sub-pixel: many samples share a pixel
        [2.5 * stride, 3.5 * stride, 9.5 * stride, 12.5 * stride],  # half-integer edges: top == bot, left == right
        [-stride, -stride, (H + 1) * stride, (W + 1) * stride],     # the whole padded map: every fold
        [0, 0, Hi, Wi],
        [np.nan, 10, 50, 60], [10, np.inf, 50, 60], [-np.inf, 10, np.inf, 60], [10, 20, 50, np.nan],
        [40, 40, 80, 80], [40, 40, 80, 80],                         # box_ind -1 and N below
        [Hi - 8, 0, Hi - 7, Wi], [0, Wi - 8, Hi, Wi - 7],           # thin strips along the far edges
    ]
    e = np.array(extra, np.float32)
    ebi = rng.integers(0, N, len(e)).astype(np.int32)
    ebi[-4], ebi[-3] = -1, N
    return np.concatenate([b, e]), np.concatenate([bi, ebi])


def single_level_case(sr, aligned, Cc, crop, seed=0, M=60):
    rng = np.random.default_rng(seed + 31 * sr + 7 * Cc + crop)
    N, H, W, stride = 2, 13, 19, 16
    boxes, bi = adversarial_boxes(rng, N, H, W, stride, M)
    g = rng.standard_normal((boxes.shape[0], crop, crop, Cc)).astype(np.float32)
    return (N, H, W, Cc), boxes, bi, g, 1.0 / stride


# ------------------------------------------------------------------ 1. single level, bit parity
@pytest.mark.parametrize("crop", [7, 14, 1])
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 1, 2, 3])
def test_single_level_bit_parity(cuda, oracle_lib, sr, aligned, crop):
    for Cc in (4, 16, 256) if crop == 7 else (16,):
        shape, boxes, bi, g, scale = single_level_case(sr, aligned, Cc, crop)
        want = oracle_lib.roi_align_backward(g, shape, boxes, bi, scale, sr, aligned)
        layer = ROIAlign((crop, crop), scale, sr, aligned)
        got = layer.backward(T(g, cuda), shape, T(boxes, cuda), T(bi, cuda), deterministic=True)
        assert_bits(got, want)


@pytest.mark.parametrize("sr", [0, 2])
def test_identical_boxes_one_image(cuda, oracle_lib, sr):
    """2,000 copies of one box on one image: every destination pixel sums 2,000+ terms in ROI order."""
    rng = np.random.default_rng(5)
    shape = (2, 20, 24, 32)
    boxes = np.tile(np.array([[37.0, 51.0, 190.0, 260.0]], np.float32), (2000, 1))
    bi = np.ones(2000, np.int32)
    g = rng.standard_normal((2000, 7, 7, 32)).astype(np.float32)
    want = oracle_lib.roi_align_backward(g, shape, boxes, bi, 1 / 16., sr, True)
    got = ROIAlign((7, 7), 1 / 16., sr, True).backward(T(g, cuda), shape, T(boxes, cuda), T(bi, cuda),
                                                       deterministic=True)
    assert_bits(got, want)


def test_non_finite_grad_out(cuda, oracle_lib):
    """NaN / +inf / -inf in grad_out: which of inf - inf or inf + inf happens depends on the summation order."""
    rng = np.random.default_rng(6)
    shape, boxes, bi, g, scale = single_level_case(2, True, 16, 7, seed=3, M=80)
    idx = rng.integers(0, g.size, 300)
    g.ravel()[idx[:100]] = np.inf
    g.ravel()[idx[100:200]] = -np.inf
    g.ravel()[idx[200:]] = np.nan
    want = oracle_lib.roi_align_backward(g, shape, boxes, bi, scale, 2, True)
    got = ROIAlign((7, 7), scale, 2, True).backward(T(g, cuda), shape, T(boxes, cuda), T(bi, cuda),
                                                    deterministic=True)
    assert np.isinf(want).any() and np.isnan(want).any()
    assert_bits(got, want)


def test_int64_strided_batch_index(cuda, oracle_lib):
    """int64 batch indices (a column view of SparseBoxList.indices) give the same bits as int32 ones."""
    shape, boxes, bi, g, scale = single_level_case(0, True, 16, 7, seed=9)
    want = oracle_lib.roi_align_backward(g, shape, boxes, bi, scale, 0, True)
    idx = T(np.stack([bi.astype(np.int64), np.arange(bi.size)], 1), cuda)
    layer = ROIAlign((7, 7), scale, 0, True)
    got = layer.backward(T(g, cuda), shape, T(boxes, cuda), idx[:, 0], deterministic=True)
    assert_bits(got, want)


# ------------------------------------------------------------------ 2. multi-level ROIPooler, FPN shapes
def pooler_case(cuda, N, R, crop, Cc, seed):
    boxes, idx = syn.rois(N, R, seed=seed)
    shapes = [(N,) + syn.level_hw(s) + (Cc,) for s in syn.FPN_STRIDES]
    g = np.random.default_rng(seed).standard_normal((N * R, crop, crop, Cc)).astype(np.float32)
    inst = SparseBoxList(T(idx, cuda), BoxList(T(boxes, cuda)), (N, R))
    return shapes, boxes, idx, g, inst


@pytest.mark.parametrize("R,crop", [(1000, 7), (128, 14)])
@pytest.mark.parametrize("sr", [0, 2])
def test_pooler_bit_parity_fpn(cuda, oracle_lib, sr, R, crop):
    shapes, boxes, idx, g, inst = pooler_case(cuda, 2, R, crop, 256, seed=40 + R + sr)
    want = oracle_lib.roi_pooler_backward(g, shapes, SCALES, boxes, idx[:, 0], sr)
    pooler = ROIPooler((crop, crop), SCALES, sr, "ROIAlignV2")
    got = pooler.backward(T(g, cuda), shapes, inst, deterministic=True)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert_bits(a, b)


# ------------------------------------------------------------------ 3. accumulate into a non-zero gradient
# The oracle's C functions add the gradient onto the buffer they are given; these helpers call them, with the
# arguments the oracle's Python wrappers pass, on a copy of `init` instead of zeros.
def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def oracle_roi_align_backward_into(oracle_lib, init, grad_out, boxes, box_ind, spatial_scale, sampling_ratio, aligned):
    out = np.array(init, np.float32, order="C")
    g = np.ascontiguousarray(grad_out, np.float32)
    M, oh, ow, Cc = g.shape
    N, H, W, _ = out.shape
    b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 4)
    bi = np.ascontiguousarray(box_ind, np.int32)
    rc = oracle_lib.lib().orc_roi_align_backward(_ptr(g), N, H, W, Cc, _ptr(b), _ptr(bi), C.c_int64(M), oh, ow,
                                                 C.c_float(spatial_scale), int(sampling_ratio), int(aligned), _ptr(out))
    assert rc == 0
    return out


def oracle_roi_pooler_backward_into(oracle_lib, inits, grad_out, scales, boxes, batch_idx, sampling_ratio,
                                    aligned=True, canonical_box_size=224, canonical_level=4):
    outs = [np.array(x, np.float32, order="C") for x in inits]
    g = np.ascontiguousarray(grad_out, np.float32)
    M, oh, ow, Cc = g.shape
    L, N = len(outs), outs[0].shape[0]
    Hs = (C.c_int * L)(*[o.shape[1] for o in outs])
    Ws = (C.c_int * L)(*[o.shape[2] for o in outs])
    ptrs = (C.c_void_p * L)(*[o.ctypes.data for o in outs])
    sc = np.ascontiguousarray(scales, np.float32)
    b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 4)
    bi = np.ascontiguousarray(batch_idx, np.int64)
    rc = oracle_lib.lib().orc_roi_pooler_backward(_ptr(g), ptrs, Hs, Ws, L, N, Cc, _ptr(sc), _ptr(b), _ptr(bi),
                                                  C.c_int64(M), oh, ow, int(sampling_ratio), int(aligned),
                                                  int(canonical_box_size), int(canonical_level))
    assert rc == 0
    return outs


def test_accumulate_into(cuda, oracle_lib):
    rng = np.random.default_rng(12)
    shape, boxes, bi, g, scale = single_level_case(2, True, 16, 7, seed=12)
    init = rng.standard_normal(shape).astype(np.float32)
    want = oracle_roi_align_backward_into(oracle_lib, init, g, boxes, bi, scale, 2, True)
    buf = T(init, cuda)
    ROIAlign((7, 7), scale, 2, True).backward(T(g, cuda), shape, T(boxes, cuda), T(bi, cuda), grad_input=buf,
                                             deterministic=True)
    assert_bits(buf, want)

    shapes, pb, idx, pg, inst = pooler_case(cuda, 2, 200, 7, 32, seed=13)
    inits = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    want = oracle_roi_pooler_backward_into(oracle_lib, inits, pg, SCALES, pb, idx[:, 0], 0)
    bufs = [T(x, cuda) for x in inits]
    ROIPooler((7, 7), SCALES, 0, "ROIAlignV2").backward(T(pg, cuda), shapes, inst, grad_x=bufs, deterministic=True)
    for a, b in zip(bufs, want):
        assert_bits(a, b)


# ------------------------------------------------------------------ 4. reproducibility and invariance
def test_repeatable_and_stream_invariant(cuda):
    shapes, boxes, idx, g, inst = pooler_case(cuda, 2, 1000, 7, 256, seed=21)
    pooler = ROIPooler((7, 7), SCALES, 0, "ROIAlignV2")
    gt = T(g, cuda)
    first = [t.clone() for t in pooler.backward(gt, shapes, inst, deterministic=True)]
    second = pooler.backward(gt, shapes, inst, deterministic=True)
    for a, b in zip(first, second):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    # a concurrent backward on another stream (atomic and deterministic) while this one runs on a side stream
    side, other = torch.cuda.Stream(cuda), torch.cuda.Stream(cuda)
    torch.cuda.synchronize(cuda)
    with torch.cuda.stream(other):
        busy = pooler.backward(gt, shapes, inst)
        busy2 = pooler.backward(gt, shapes, inst, deterministic=True)
    with torch.cuda.stream(side):
        third = pooler.backward(gt, shapes, inst, deterministic=True)
    torch.cuda.synchronize(cuda)
    for a, b, c in zip(first, third, busy2):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        assert torch.equal(a.view(torch.int32), c.view(torch.int32))
    del busy


def test_image_blocks_equal_full_batch(cuda):
    """The backward of images [b, e) alone equals the full batch's gradient on those images (sharded training)."""
    N, R = 4, 300
    shapes, boxes, idx, g, inst = pooler_case(cuda, N, R, 7, 64, seed=22)
    pooler = ROIPooler((7, 7), SCALES, 0, "ROIAlignV2")
    full = pooler.backward(T(g, cuda), shapes, inst, deterministic=True)
    for b, e in ((0, 1), (1, 3), (3, 4)):
        keep = (idx[:, 0] >= b) & (idx[:, 0] < e)
        sub_idx = idx[keep].copy()
        sub_idx[:, 0] -= b
        sub = SparseBoxList(T(sub_idx, cuda), BoxList(T(boxes[keep], cuda)), (e - b, R))
        sub_shapes = [(e - b,) + tuple(s[1:]) for s in shapes]
        part = pooler.backward(T(g[keep], cuda), sub_shapes, sub, deterministic=True)
        for p, f in zip(part, full):
            assert torch.equal(p.view(torch.int32), f[b:e].view(torch.int32))


# ------------------------------------------------------------------ 5. the default path is unchanged
def _kernels(fn):
    """Names of the kernels fn() launches, from the same profiler set-up as the dispatch-boundary tests."""
    _, trace = traced(fn)
    assert trace is not None, "torch.profiler has no CUDA activity here"
    return {name for name, _ in trace}


def test_modes_select_their_kernels(cuda, oracle_lib, monkeypatch):
    shapes, boxes, idx, g, inst = pooler_case(cuda, 2, 200, 7, 32, seed=23)
    pooler = ROIPooler((7, 7), SCALES, 0, "ROIAlignV2")
    gt = T(g, cuda)
    requests = []
    real_call = nv.call

    def spy(op, params, device):
        if op == "roi_align_backward":
            L = nv._bind(op)
            requests.append((params.deterministic, L.d2b_roi_align_backward_workspace_bytes(C.byref(params))))
        return real_call(op, params, device)

    monkeypatch.setattr(nv, "call", spy)
    pooler.backward(gt, shapes, inst)  # warm-up (module load)
    pooler.backward(gt, shapes, inst, deterministic=True)
    atomic = _kernels(lambda: pooler.backward(gt, shapes, inst))
    det = _kernels(lambda: pooler.backward(gt, shapes, inst, deterministic=True))
    atomic_bw = [k for k in atomic if "roi_align" in k]
    det_bw = [k for k in det if "roi_align" in k]
    assert atomic_bw and all("roi_align_backward_kernel" in k for k in atomic_bw), atomic_bw
    assert not any("roi_align_backward_kernel" in k for k in det_bw), det_bw
    for name in ("roi_align_grad_bin_kernel", "roi_align_grad_partition_kernel", "roi_align_grad_accum_kernel"):
        assert any(name in k for k in det_bw), (name, det_bw)
    assert all(n == 0 for d, n in requests if d == 0) and any(d == 0 for d, _ in requests)
    assert all(n > 0 for d, n in requests if d == 1) and any(d == 1 for d, _ in requests)
    # both modes compute the same gradient up to fp32 summation order
    a = pooler.backward(gt, shapes, inst)
    d = pooler.backward(gt, shapes, inst, deterministic=True)
    bound = oracle_lib.roi_pooler_backward(np.abs(g), shapes, SCALES, boxes, idx[:, 0], 0)
    for x, y, bnd in zip(a, d, bound):
        err = np.abs(x.cpu().numpy() - y.cpu().numpy())
        assert (err <= 1e-5 * bnd + 1e-7).all()


# ------------------------------------------------------------------ 6. memory safety: outputs and exact workspace
def test_canary_bands(cuda, oracle_lib, monkeypatch):
    guard = Guard(monkeypatch)
    rng = np.random.default_rng(30)
    # C = 4, M not a multiple of anything, tiles reached by one ROI, maps smaller than a tile and of one pixel
    for (N, H, W, Cc, M, crop, sr) in ((3, 11, 17, 4, 37, 7, 2), (1, 1, 1, 4, 5, 3, 0), (2, 9, 2, 8, 1, 1, 3),
                                        (2, 30, 23, 132, 13, 5, 1)):
        boxes, bi = adversarial_boxes(rng, N, H, W, 8, M)
        g = rng.standard_normal((boxes.shape[0], crop, crop, Cc)).astype(np.float32)
        want = oracle_lib.roi_align_backward(g, (N, H, W, Cc), boxes, bi, 1 / 8., sr, True)
        got = ROIAlign((crop, crop), 1 / 8., sr, True).backward(T(g, cuda), (N, H, W, Cc), T(boxes, cuda),
                                                              T(bi, cuda), deterministic=True)
        assert_bits(got, want)
    empty = ROIAlign((7, 7), 1 / 8., 0, True).backward(T(np.zeros((0, 7, 7, 4), np.float32), cuda), (2, 5, 6, 4),
                                                       T(np.zeros((0, 4), np.float32), cuda),
                                                       T(np.zeros(0, np.int32), cuda), deterministic=True)
    assert not bool(empty.any())
    shapes, boxes, idx, g, inst = pooler_case(cuda, 2, 77, 7, 4, seed=31)
    want = oracle_lib.roi_pooler_backward(g, shapes, SCALES, boxes, idx[:, 0], 2)
    got = ROIPooler((7, 7), SCALES, 2, "ROIAlignV2").backward(T(g, cuda), shapes, inst, deterministic=True)
    for a, b in zip(got, want):
        assert_bits(a, b)
    assert guard.check() >= 8
