"""GPU: the batched, per-image-size RLE mode of d2b_solo_upsample (`solo_upsample_rle`, `SOLOv2Inference.inference_rle`):
the [B, D] SOLOv2 detection slots of a whole batch, each image's top-left crop of its masks resized to its own output
size and encoded in one call.  String bytes, offsets and boxes are checked bit for bit against the oracle
(`solo_upsample_boxes` on the crop, encoded by coco_rle.py), against the single-size GPU path on the crop, and against
the planes of the single-size path encoded on the host."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import SOLOv2Inference, coco_results, solo_upsample_masks, solo_upsample_rle

import coco_rle
from test_canary_gpu import PATTERN, guard  # noqa: F401  (fixture)
from test_mask_rle_gpu import strings
from test_solo_upsample_gpu import T, blobs, pack

pytestmark = pytest.mark.gpu

MAX_PLANE = (1 << 31) - 65536
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def packed(m):
    """`pack`, also for D = 0."""
    B, D, h, w = m.shape
    return pack(m) if m.size else np.zeros((B, D, (h * w + 63) // 64), np.int64)


def unpack(packed, h, w):
    """int64 [..., ceil(h*w/64)] -> fp32 0/1 [..., h, w] (the inverse of `pack`)."""
    bits = np.unpackbits(np.ascontiguousarray(packed).view(np.uint8), axis=-1, bitorder="little")
    return bits[..., :h * w].reshape(packed.shape[:-1] + (h, w)).astype(np.float32)


def live(H, W, hb, wb, h, w):
    return H >= 1 and W >= 1 and H * W < MAX_PLANE and 1 <= hb <= h and 1 <= wb <= w


def oracle_ref(oracle_lib, m, outs, crops, valid, ac, thr):
    """Per image: slice [:hb, :wb], oracle_lib.solo_upsample_boxes at outs[b], coco_rle; invalid slots b"" and 0 boxes."""
    B, D, h, w = m.shape
    want, boxes = [], np.zeros((B, D, 4), np.float32)
    for b in range(B):
        (H, W), (hb, wb) = outs[b], crops[b]
        v = np.ones(D, bool) if valid is None else valid[b].astype(bool)
        if not live(H, W, hb, wb, h, w) or not v.any():
            want += [b""] * D
            continue
        wm, wbx = oracle_lib.solo_upsample_boxes(np.ascontiguousarray(m[b][v][:, :hb, :wb]), (H, W), ac, thr)
        enc = iter(coco_rle.encode(wm))
        want += [next(enc) if x else b"" for x in v]
        boxes[b][v] = wbx
    return want, boxes


def single_ref(cuda, m, outs, crops, valid, ac, thr, with_planes):
    """Per image, the single-size mode on the crop (repacked): its strings and boxes for the valid slots; with_planes
    also encodes its uint8 planes on the host and checks them against its strings."""
    B, D, h, w = m.shape
    got, boxes = [], np.zeros((B, D, 4), np.float32)
    for b in range(B):
        (H, W), (hb, wb) = outs[b], crops[b]
        v = np.ones(D, bool) if valid is None else valid[b].astype(bool)
        if not live(H, W, hb, wb, h, w) or D == 0:
            got += [b""] * D
            continue
        crop = np.ascontiguousarray(m[b:b + 1, :, :hb, :wb])
        r = solo_upsample_masks(T(pack(crop), cuda), (hb, wb), (H, W), thr, ac, return_masks=with_planes,
                                return_rle=True)
        mine = strings(*r["rle"])
        if with_planes:
            assert mine == coco_rle.encode(r["pred_masks"][0].cpu().numpy()), b
        got += [s if x else b"" for s, x in zip(mine, v)]
        boxes[b][v] = r["boxes"][0].cpu().numpy()[v]
    return got, boxes


def check(cuda, oracle_lib, m, outs, crops=None, valid=None, ac=False, thr=0.5, with_planes=True, capacity=None,
          oracle=True):
    """The batched call with host sizes (crops None: the whole mask) against the three references."""
    B, D, h, w = m.shape
    full = [(h, w)] * B
    (chars, offsets), boxes = solo_upsample_rle(T(packed(m), cuda), (h, w), outs, crops, None if valid is None else
                                                T(valid, cuda), thr, ac, capacity)
    got, gb = strings(chars, offsets), boxes.cpu().numpy()
    want, wb = single_ref(cuda, m, outs, crops or full, valid, ac, thr, with_planes)
    if oracle:
        ow, ob = oracle_ref(oracle_lib, m, outs, crops or full, valid, ac, thr)
        assert want == ow
        assert np.array_equal(wb, ob)
    assert offsets.cpu().tolist() == np.cumsum([0] + [len(s) for s in want]).tolist()
    assert got == want
    assert np.array_equal(gb, wb)
    return got, gb


def special_masks(rng, B, D, h, w):
    """Object-like blobs plus the edge cases: empty, full, checkerboard (many runs), only row 0, only column 0."""
    m = blobs(rng, B, D, h, w)
    yy, xx = np.mgrid[0:h, 0:w]
    m[0, 0] = 0
    m[0, 1] = 1
    m[1 % B, 2 % D] = ((yy + xx) % 2).astype(np.float32)
    m[2 % B, 3 % D] = 0; m[2 % B, 3 % D, 0, :] = 1
    m[3 % B, 4 % D] = 0; m[3 % B, 4 % D, :, 0] = 1
    m[B - 1, D - 1] = (rng.random((h, w)) > 0.5).astype(np.float32)
    return m


h0, w0 = 20, 34
GEOMS = {  # (output sizes, crops) of four images with 20 x 34 masks
    # 1x1, 1xW, Hx1 outputs and 4x up of the full mask
    "degenerate": ([(1, 1), (1, 57), (43, 1), (80, 136)], [(20, 34), (13, 21), (7, 34), (20, 34)]),
    # a 1x1 crop, shrink below the crop, output equal to the crop, a one-row crop
    "crops": ([(24, 40), (9, 13), (17, 29), (5, 60)], [(1, 1), (13, 21), (17, 29), (1, 34)]),
    # a one-column crop, the full mask, odd crops
    "columns": ([(64, 3), (40, 80), (21, 35), (100, 100)], [(20, 1), (20, 34), (19, 33), (11, 7)]),
}


@pytest.mark.parametrize("geom", sorted(GEOMS))
@pytest.mark.parametrize("thr", [0.5, 0.0, -0.5, 1.0])
@pytest.mark.parametrize("ac", [False, True])
def test_batched_matches_references(cuda, oracle_lib, geom, thr, ac):
    rng = np.random.default_rng(sorted(GEOMS).index(geom) * 100 + int(thr * 10) + 10 + 50 * ac)
    m = special_masks(rng, 4, 6, h0, w0)
    valid = rng.random((4, 6)) < 0.75
    valid[:, :2] = True
    valid[2, :] = True
    outs, crops = GEOMS[geom]
    check(cuda, oracle_lib, m, outs, crops, valid.astype(np.uint8), ac, thr)


def test_full_crop_equals_single_size_path(cuda, oracle_lib):
    """mask_shapes None: every image at its own size from the whole mask, as the single-size mode gives it."""
    rng = np.random.default_rng(4)
    m = special_masks(rng, 3, 5, 24, 33)
    check(cuda, oracle_lib, m, [(96, 132), (31, 17), (24, 33)])


@pytest.mark.parametrize("B,D", [(1, 1), (1, 7), (3, 0), (2, 3)])
def test_small_batches_and_valid_null(cuda, oracle_lib, B, D):
    rng = np.random.default_rng(B * 10 + D)
    m = blobs(rng, B, D, 12, 18)
    outs = [(30 + 7 * b, 41 - 5 * b) for b in range(B)]
    crops = [(12 - b, 18 - 3 * b) for b in range(B)]
    got, _ = check(cuda, oracle_lib, m, outs, crops)
    assert len(got) == B * D and all(got)  # valid NULL: every slot holds a string


def test_all_slots_invalid(cuda, oracle_lib):
    rng = np.random.default_rng(2)
    m = blobs(rng, 4, 5, h0, w0)
    outs, crops = GEOMS["crops"]
    got, boxes = check(cuda, oracle_lib, m, outs, crops, np.zeros((4, 5), np.uint8))
    assert got == [b""] * 20 and not boxes.any()


def test_out_of_range_device_sizes(cuda, oracle_lib, guard):
    """Sizes the host never saw, between canary bands: every slot of an image whose output size or crop is out of range
    is an empty string with a zero box, and the other images are unaffected."""
    rng = np.random.default_rng(5)
    D, h, w = 4, 16, 24
    bad = [((0, 50), (16, 24)), ((50, -3), (16, 24)), ((46341, 46341), (16, 24)), ((65536, 65536), (16, 24)),
           ((-2147483648, -1), (16, 24)), ((2147483647, 2147483647), (16, 24)),
           ((30, 30), (0, 24)), ((30, 30), (17, 24)), ((30, 30), (16, 25)), ((30, 30), (-1, -1)),
           ((30, 30), (2147483647, 1))]
    good = [((40, 60), (16, 24)), ((1, 1), (9, 13))]
    cfg = good[:1] + bad + good[1:]
    B = len(cfg)
    outs = np.array([c[0] for c in cfg], np.int32)
    crops = np.array([c[1] for c in cfg], np.int32)
    m = blobs(rng, B, D, h, w)
    pk = torch.empty((B, D, (h * w + 63) // 64), dtype=torch.int64, device=cuda)
    pk.copy_(T(pack(m), cuda))
    os_ = torch.empty(outs.shape, dtype=torch.int32, device=cuda)
    os_.copy_(torch.from_numpy(outs))
    cs = torch.empty(crops.shape, dtype=torch.int32, device=cuda)
    cs.copy_(torch.from_numpy(crops))
    (chars, offsets), boxes = solo_upsample_rle(pk, (h, w), os_, cs)
    got, gb = strings(chars, offsets), boxes.cpu().numpy()
    assert got[D:D * (1 + len(bad))] == [b""] * (D * len(bad))
    assert not gb[1:1 + len(bad)].any()
    ends = [0, B - 1]
    want, wb = oracle_ref(oracle_lib, m[ends], outs[ends], crops[ends], None, False, 0.5)
    assert got[:D] + got[-D:] == want
    assert np.array_equal(gb[ends], wb)
    guard.check()
    with pytest.raises(ValueError, match=r"output_shapes\[1\]"):
        solo_upsample_rle(pk, (h, w), outs, None)  # the same sizes from the host are refused before any call
    with pytest.raises(ValueError, match=r"mask_shapes\[7\]"):
        solo_upsample_rle(pk, (h, w), [(5, 5)] * B, crops)


def test_capacity(cuda, oracle_lib, guard):
    """Capacity 0 (the sizing query), exactly offsets[-1], one byte short and generous, with every buffer between canary
    bands."""
    rng = np.random.default_rng(11)
    m = special_masks(rng, 4, 5, h0, w0)
    valid = np.ones((4, 5), np.uint8)
    valid[1, 1] = 0
    outs, crops = GEOMS["columns"]
    want, wb = oracle_ref(oracle_lib, m, outs, crops, valid, False, 0.5)
    cum = np.cumsum([0] + [len(s) for s in want]).tolist()

    def banded(a, dtype):
        t = torch.empty(a.shape, dtype=dtype, device=cuda)
        t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        return t
    pk = banded(pack(m), torch.int64)
    args = (pk, (h0, w0), banded(np.array(outs, np.int32), torch.int32), banded(np.array(crops, np.int32), torch.int32),
            banded(valid, torch.uint8))
    (chars, offsets), boxes = solo_upsample_rle(*args, capacity=0)
    assert chars.numel() == 0 and offsets.cpu().tolist() == cum
    assert np.array_equal(boxes.cpu().numpy(), wb)
    for cap in (cum[-1], cum[-1] + 4096):
        (chars, offsets), boxes = solo_upsample_rle(*args, capacity=cap)
        assert strings(chars, offsets) == want and np.array_equal(boxes.cpu().numpy(), wb)
    (chars, offsets), _ = solo_upsample_rle(*args, capacity=cum[-1] - 1)
    assert offsets.cpu().tolist() == cum
    data = chars.cpu().numpy().tobytes()
    assert data[:cum[-2]] == b"".join(want[:-1])
    assert set(data[cum[-2]:]) == {PATTERN}  # the last string did not fit: untouched
    guard.check()


def coco_batch(rng, B=16, D=100, h=200, w=336):
    """16 images x 100 slots of 200x336 object-like masks (a canvas of 800x1344 at stride 4), ~90 % valid, COCO-like
    output sizes (longest side 640) and crops ceil(size in the canvas / 4)."""
    m = blobs(rng, B, D, h, w)
    valid = (rng.random((B, D)) < 0.9).astype(np.uint8)
    outs, crops = [], []
    for _ in range(B):
        long_, short = 640, int(rng.integers(300, 641))
        H, W = (long_, short) if rng.random() < 0.3 else (short, long_)
        s = min(800 / min(H, W), 1333 / max(H, W))  # the resize of the input pipeline
        ch, cw = int(round(H * s)), int(round(W * s))
        outs.append((H, W))
        crops.append((min(h, -(-ch // 4)), min(w, -(-cw // 4))))
    return m, valid, outs, crops


def test_full_batch_coco_sizes(cuda, oracle_lib):
    """The 16 x 100 x 200x336 case: crops against the single-size path on each crop, the oracle on three images, and
    the uncropped call against the single-size path on the whole mask."""
    rng = np.random.default_rng(16)
    m, valid, outs, crops = coco_batch(rng)
    got, gb = check(cuda, oracle_lib, m, outs, crops, valid, with_planes=False, oracle=False)
    for b in (0, 7, 15):
        want, wb = oracle_ref(oracle_lib, m[b:b + 1], outs[b:b + 1], crops[b:b + 1], valid[b:b + 1], False, 0.5)
        assert got[b * 100:(b + 1) * 100] == want
        assert np.array_equal(gb[b:b + 1], wb)
    check(cuda, oracle_lib, m, outs, None, valid, with_planes=False, oracle=False)


PROFILED = """
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np, torch
from detectron2_tensorflow_b200.modeling import solo_upsample_rle
dev = torch.device("cuda", 0)
pk = torch.from_numpy(np.random.default_rng(1).integers(-2**62, 2**62, (2, 4, 11))).to(dev)
os_ = torch.tensor([[60, 90], [33, 47]], dtype=torch.int32, device=dev)
solo_upsample_rle(pk, (20, 34), os_, capacity=1 << 16)
torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    solo_upsample_rle(pk, (20, 34), os_, capacity=1 << 16)
    torch.cuda.synchronize()
for e in prof.key_averages():
    print(e.key.replace(" ", ""))
"""


def test_batched_path_runs_the_rle_kernels_only(cuda):
    """The batched mode is the three RLE launches: no solo_upsample_kernel (its shared memory grows with the shrink
    factor, which the host does not know here), no statistics kernels.  Profiled in a process of its own, so that no
    earlier profiler session of the test process can hide kernel activity."""
    out = subprocess.run([sys.executable, "-c", PROFILED, ROOT], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-4000:]
    names = [n.replace("(bool)0", "false").replace("(bool)1", "true") for n in out.stdout.split()]
    assert sorted(k for n in names for k in re.findall(r"solo_rle_kernel<[^>]*>", n)) == \
        ["solo_rle_kernel<false,true>", "solo_rle_kernel<true,true>"], names
    assert sum("rle_offsets_kernel" in n for n in names) == 1, names
    assert not any(k in n for n in names for k in ("solo_upsample_kernel", "up_boxes_kernel", "up_init_stats")), names


def test_graph_replay_with_new_sizes(cuda, oracle_lib):
    """A fixed capacity and device sizes make the call sync-free: captured once, replayed after new masks, validity,
    output sizes and crops are written in place, equal to the eager call and to the oracle."""
    rng = np.random.default_rng(9)
    ma, mb = special_masks(rng, 4, 6, h0, w0), blobs(rng, 4, 6, h0, w0)
    va, vb = (rng.random((4, 6)) < 0.7).astype(np.uint8), (rng.random((4, 6)) < 0.7).astype(np.uint8)
    (oa, ca), (ob, cb) = GEOMS["degenerate"], GEOMS["crops"]
    pk, vl = T(pack(ma), cuda), T(va, cuda)
    os_, cs = T(np.array(oa, np.int32), cuda), T(np.array(ca, np.int32), cuda)
    cap = 1 << 16
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        solo_upsample_rle(pk, (h0, w0), os_, cs, vl, capacity=cap)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        (chars_g, off_g), boxes_g = solo_upsample_rle(pk, (h0, w0), os_, cs, vl, capacity=cap)
    for src, os_v, cs_v, v, m in ((None, oa, ca, va, ma), (1, ob, cb, vb, mb)):
        pk.copy_(T(pack(m), cuda)); vl.copy_(T(v, cuda))
        os_.copy_(T(np.array(os_v, np.int32), cuda)); cs.copy_(T(np.array(cs_v, np.int32), cuda))
        g.replay()
        torch.cuda.synchronize()
        (chars_e, off_e), boxes_e = solo_upsample_rle(pk, (h0, w0), os_, cs, vl, capacity=cap)
        assert torch.equal(off_g, off_e) and strings(chars_g, off_g) == strings(chars_e, off_e)
        assert torch.equal(boxes_g, boxes_e)
        assert off_e[-1].item() <= cap
        want, wb = oracle_ref(oracle_lib, m, os_v, cs_v, v, False, 0.5)
        assert strings(chars_g, off_g) == want and np.array_equal(boxes_g.cpu().numpy(), wb)


def head_inputs(rng, B=3):
    grids, strides, K, E, (H, W) = (8, 6), (8, 16), 4, 32, (28, 40)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    feat = np.stack([np.stack([np.sin(yy * rng.uniform(0.05, 0.4) + xx * rng.uniform(0.05, 0.4) + rng.uniform(0, 6))
                               for _ in range(E)], -1) for _ in range(B)]).astype(np.float32)
    probs = [rng.random((B, g, g, K)).astype(np.float32) ** 3 for g in grids]
    kerns = [(rng.standard_normal((B, g, g, E)) * 0.6).astype(np.float32) for g in grids]
    head = SOLOv2Inference(0.5, 40, "gaussian", 2.0, 0.05, 15, score_threshold=0.2, num_grids=grids, strides=strides,
                           max_candidates=256)
    return head, probs, kerns, feat


def inference_want(cuda, oracle_lib, head, probs, kerns, feat, outs, crops):
    """select, tail, then the oracle on each image's crop of the tail's packed masks, encoded by coco_rle."""
    B, Hf, Wf, _ = feat.shape
    sc = torch.cat([T(p, cuda).reshape(B, -1, p.shape[-1]) for p in probs], 1)
    kn = torch.cat([T(k, cuda).reshape(B, -1, k.shape[-1]) for k in kerns], 1)
    cand = head.select_candidates(sc, kn)
    tail = head.postprocess(None, cand["scores"], cand["classes"], cand["strides"], cand["counts"], return_masks=False,
                            mask_features=T(feat, cuda), mask_kernels=cand["kernels"])
    m = unpack(tail["packed_masks"].cpu().numpy(), Hf, Wf)
    valid = tail["is_valid"].cpu().numpy()
    want, wb = oracle_ref(oracle_lib, m, outs, crops, valid, head.align_corners, head.mask_threshold)
    return tail, want, wb


def same_fields(res, want):
    """Classes and validity exact; scores to 1e-5, since the tail sums mask scores with fp32 atomics."""
    assert torch.equal(res.get_field("pred_classes"), want["pred_classes"])
    assert torch.equal(res.get_field("is_valid"), want["is_valid"])
    assert torch.allclose(res.get_field("scores"), want["scores"], rtol=1e-5, atol=1e-7)


def test_inference_rle_eager_and_graph(cuda, oracle_lib):
    rng = np.random.default_rng(21)
    head, probs, kerns, feat = head_inputs(rng)
    outs, crops = [(111, 158), (80, 124), (47, 31)], [(28, 40), (20, 31), (23, 15)]
    tail, want, wb = inference_want(cuda, oracle_lib, head, probs, kerns, feat, outs, crops)
    assert int(tail["num"].sum()) > 0
    tp, tk, tf = [T(p, cuda) for p in probs], [T(k, cuda) for k in kerns], T(feat, cuda)
    res, rle = head.inference_rle(tp, tk, tf, outs, crops)
    assert strings(*rle) == want and np.array_equal(res.boxes.cpu().numpy(), wb)
    same_fields(res, tail)

    # coco_results on the output equals the list built image by image
    cats = [1, 3, 7, 9]
    ids = [501, 502, 503]
    got = coco_results(res, rle, res.boxes, outs, ids, cats)
    sc, cl, va = (res.get_field(k).cpu().numpy() for k in ("scores", "pred_classes", "is_valid"))
    expect = []
    for b in range(3):
        for d in range(sc.shape[1]):
            if va[b, d]:
                y0, x0, y1, x1 = wb[b, d]
                expect.append({"image_id": ids[b], "category_id": cats[int(cl[b, d])],
                               "bbox": [float(x0), float(y0), float(x1 - x0), float(y1 - y0)],
                               "score": float(sc[b, d]),
                               "segmentation": {"size": list(outs[b]), "counts": want[b * sc.shape[1] + d]}})
    assert got == expect and len(got) == int(va.sum())

    # the whole chain from raw head outputs, captured at an int capacity with device sizes, replayed on new inputs
    os_, cs = T(np.array(outs, np.int32), cuda), T(np.array(crops, np.int32), cuda)
    cap = 1 << 16
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        head.inference_rle(tp, tk, tf, os_, cs, capacity=cap)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res_g, (chars_g, off_g) = head.inference_rle(tp, tk, tf, os_, cs, capacity=cap)
    _, probs2, kerns2, feat2 = head_inputs(np.random.default_rng(22))
    outs2, crops2 = [(64, 90), (200, 150), (28, 40)], [(27, 39), (28, 40), (28, 40)]
    for p, q in zip(tp, probs2):
        p.copy_(T(q, cuda))
    for k, q in zip(tk, kerns2):
        k.copy_(T(q, cuda))
    tf.copy_(T(feat2, cuda))
    os_.copy_(T(np.array(outs2, np.int32), cuda))
    cs.copy_(T(np.array(crops2, np.int32), cuda))
    g.replay()
    torch.cuda.synchronize()
    _, want2, wb2 = inference_want(cuda, oracle_lib, head, probs2, kerns2, feat2, outs2, crops2)
    assert strings(chars_g, off_g) == want2 and np.array_equal(res_g.boxes.cpu().numpy(), wb2)
    res_e, rle_e = head.inference_rle(tp, tk, tf, os_, cs, capacity=cap)
    assert torch.equal(off_g, rle_e[1]) and strings(chars_g, off_g) == strings(*rle_e)
    same_fields(res_g, {k: res_e.get_field(k) for k in ("scores", "pred_classes", "is_valid")})


def test_misuse_launches_nothing(cuda):
    """EINVAL before any launch: planes in the batched mode, offsets or boxes NULL, batched fields without the mode."""
    B, D, h, w = 2, 3, 8, 8
    pk = torch.zeros(B, D, 1, dtype=torch.int64, device=cuda)
    shapes = torch.full((B, 2), 8, dtype=torch.int32, device=cuda)
    offsets = torch.full((B * D + 1,), -7, dtype=torch.int64, device=cuda)
    boxes = torch.full((B, D, 4), -7.0, device=cuda)
    planes = torch.empty(B, D, 8, 8, dtype=torch.uint8, device=cuda)

    def params():
        p = nv.SoloUpsampleParams()
        p.packed_masks, p.batch, p.num_dets, p.mask_h, p.mask_w, p.mask_threshold = pk.data_ptr(), B, D, h, w, 0.5
        p.out_boxes, p.out_rle_offsets, p.output_shapes = boxes.data_ptr(), offsets.data_ptr(), shapes.data_ptr()
        return p
    cases = []
    p = params(); p.out_masks = planes.data_ptr(); cases.append(p)
    p = params(); p.out_rle_offsets = None; cases.append(p)
    p = params(); p.out_boxes = None; cases.append(p)
    p = params(); p.output_shapes = None; p.image_h = p.image_w = 8; p.valid = shapes.data_ptr(); cases.append(p)
    L = nv._bind("solo_upsample")
    torch.cuda.synchronize()
    before = nv.kernel_launch_count()
    for p in cases:
        assert L.d2b_solo_upsample(C.byref(p), None, 0, None) == -1
    assert nv.kernel_launch_count() == before
    torch.cuda.synchronize()
    assert offsets.cpu().tolist() == [-7] * (B * D + 1) and bool((boxes == -7).all())
