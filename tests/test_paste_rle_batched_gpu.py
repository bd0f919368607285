"""GPU: the batched, per-image-size RLE mode of d2b_paste_masks (`detector_postprocess_rle`): the [N, R] detection slots
of a whole batch, each image pasted and encoded at its own output size in one call.  Bytes and offsets are checked
against the per-image path (from_dense + the boxes of detector_postprocess + reframe_box_masks_to_rle), against the
planes of detector_postprocess itself and against coco_rle.py applied to the oracle's masks."""
import ctypes as C

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import coco_results, detector_postprocess, detector_postprocess_rle
from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList, reframe_box_masks_to_rle, rle_to_coco

import coco_rle
import test_paste_masks_gpu as pm
from test_canary_gpu import PATTERN, guard  # noqa: F401  (fixture)
from test_mask_rle_gpu import T, adversarial_boxes, strings

pytestmark = pytest.mark.gpu


def make_inputs(rng, in_shapes, R, mh=28, mw=28, p_valid=0.6, adversarial=False):
    """Dense [N, R] detections: boxes in each image's input (image_shape) coordinates, soft masks, validity."""
    N = len(in_shapes)
    boxes = np.zeros((N, R, 4), np.float32)
    for n, (h, w) in enumerate(in_shapes):
        y0, x0 = rng.uniform(-0.1 * h, h, R), rng.uniform(-0.1 * w, w, R)
        boxes[n] = np.stack([y0, x0, y0 + rng.uniform(0.5, 0.6 * h, R), x0 + rng.uniform(0.5, 0.6 * w, R)], 1)
        if adversarial:
            k = min(R, 10)
            boxes[n, :k] = adversarial_boxes(rng, h, w, 10)[:k]
    masks = pm._masks(rng, N * R, mh, mw).reshape(N, R, mh, mw)
    valid = rng.random((N, R)) < p_valid
    return boxes, masks, valid, np.asarray(in_shapes, np.int32).reshape(N, 2)


def boxlist(dev, boxes, masks, valid, in_shapes):
    bl = BoxList(T(boxes, dev))
    bl.add_field("pred_masks", T(masks, dev))
    bl.add_field("is_valid", T(valid, dev))
    bl.set_tracking("image_shape", T(in_shapes, dev))
    return bl


def scaled(boxes, in_shapes, out_shapes):
    """postprocessing.py:36-43 in numpy: float32(float64(out) / float64(in)), one fp32 multiply per coordinate."""
    s = (np.asarray(out_shapes, np.float64) / in_shapes.astype(np.float64)).astype(np.float32)
    return boxes * np.concatenate([s, s], 1)[:, None, :]


def oracle_strings(oracle_lib, boxes, masks, valid, in_shapes, out_shapes, fmt):
    pb = scaled(boxes, in_shapes, out_shapes) if fmt == "fixed" else boxes
    want = []
    for n, hw in enumerate(out_shapes):
        if not valid[n].any():
            want += [b""] * valid.shape[1]
            continue
        enc = iter(coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(masks[n][valid[n]], pb[n][valid[n]],
                                                                              tuple(hw))))
        want += [next(enc) if v else b"" for v in valid[n]]
    return want


def per_image_strings(dev, boxes, masks, valid, in_shapes, out_shapes, fmt, with_planes):
    """Image by image, today's path: from_dense (the slots detector_postprocess keeps), its pasting boxes,
    reframe_box_masks_to_rle; with_planes also encodes detector_postprocess's own planes on the host."""
    got = []
    for n, hw in enumerate(out_shapes):
        one = boxlist(dev, boxes[n:n + 1], masks[n:n + 1], valid[n:n + 1], in_shapes[n:n + 1])
        sp = SparseBoxList.from_dense(one)
        b = sp.data.boxes
        if fmt == "fixed":
            s = (torch.tensor([float(hw[0]), float(hw[1])], dtype=torch.float64, device=dev)[None]
                 / sp.get_tracking("image_shape").to(torch.float64))[sp.indices[:, 0]].to(torch.float32)
            b = torch.stack([s[:, 0] * b[:, 0], s[:, 1] * b[:, 1], s[:, 0] * b[:, 2], s[:, 1] * b[:, 3]], 1)
        enc = iter(strings(*reframe_box_masks_to_rle(sp.data.get_field("pred_masks"), b, tuple(hw))))
        mine = [next(enc) if v else b"" for v in valid[n]]
        if with_planes:
            planes = detector_postprocess(one, tuple(hw), fmt, image_shapes=one.get_tracking("image_shape"))
            planes = planes.get_field("pred_masks")[0].cpu().numpy()[valid[n]]
            enc = iter(coco_rle.encode(planes))
            assert mine == [next(enc) if v else b"" for v in valid[n]], n
        got += mine
    return got


def check(dev, oracle_lib, boxes, masks, valid, in_shapes, out_shapes, fmt="fixed", with_planes=True):
    bl = boxlist(dev, boxes, masks, valid, in_shapes)
    (chars, offsets), pb = detector_postprocess_rle(bl, out_shapes, mask_format=fmt)
    want = oracle_strings(oracle_lib, boxes, masks, valid, in_shapes, out_shapes, fmt)
    assert offsets.cpu().tolist() == np.cumsum([0] + [len(s) for s in want]).tolist()
    assert chars.numel() == offsets[-1].item()
    got = strings(chars, offsets)
    assert got == want
    assert got == per_image_strings(dev, boxes, masks, valid, in_shapes, out_shapes, fmt, with_planes)
    want_boxes = scaled(boxes, in_shapes, out_shapes) if fmt == "fixed" else boxes
    assert np.array_equal(pb.cpu().numpy(), want_boxes, equal_nan=True)
    return got


IN4 = [(60, 80), (50, 70), (97, 131), (120, 30)]
OUTS = {
    "degenerate": [(1, 1), (1, 97), (83, 1), (300, 7)],        # 1x1, 1xW, Hx1, tall and thin
    "scales": [(120, 160), (25, 35), (97, 131), (64, 33)],     # larger, smaller, equal to the input (scale 1), mixed
    "coco_like": [(427, 640), (480, 640), (640, 427), (333, 500)],
}


@pytest.mark.parametrize("outs", sorted(OUTS))
@pytest.mark.parametrize("fmt", ["fixed", "conventional"])
@pytest.mark.parametrize("adversarial", [False, True])
def test_batched_rle_matches_per_image(cuda, oracle_lib, outs, fmt, adversarial):
    rng = np.random.default_rng(len(outs) * 7 + (fmt == "fixed") * 3 + adversarial)
    boxes, masks, valid, ins = make_inputs(rng, IN4, 16, adversarial=adversarial)
    valid[1, :] = False                      # an image without a detection
    valid[0, -1] = True                      # so the last slot of image 0 is a string between two images
    check(cuda, oracle_lib, boxes, masks, valid, ins, OUTS[outs], fmt, with_planes=outs != "coco_like")


@pytest.mark.parametrize("N,R", [(1, 1), (1, 7), (3, 1), (2, 0)])
def test_batched_rle_small_batches(cuda, oracle_lib, N, R):
    rng = np.random.default_rng(N * 10 + R)
    boxes, masks, valid, ins = make_inputs(rng, IN4[:N], R, mh=14, mw=14, p_valid=1.0)
    check(cuda, oracle_lib, boxes, masks, valid, ins, OUTS["scales"][:N])


def test_batched_rle_all_invalid(cuda, oracle_lib):
    rng = np.random.default_rng(2)
    boxes, masks, valid, ins = make_inputs(rng, IN4, 5)
    valid[:] = False
    got = check(cuda, oracle_lib, boxes, masks, valid, ins, OUTS["scales"])
    assert got == [b""] * 20
    assert rle_to_coco(*detector_postprocess_rle(boxlist(cuda, boxes, masks, valid, ins), OUTS["scales"])[0],
                       sizes=np.repeat(OUTS["scales"], 5, 0)) == [None] * 20


def test_batched_rle_full_batch(cuda, oracle_lib):
    """16 images x 100 slots (~60 % valid) of 28x28 masks at the engine geometry (800x1333 input), pasted back at 16
    COCO-like original sizes in one call; equal to 16 per-image calls, and to the oracle on three images."""
    rng = np.random.default_rng(16)
    ins = [(800, 1333)] * 16
    outs = [(int(h), int(w)) for h, w in zip(rng.integers(240, 641, 16), rng.integers(320, 641, 16))]
    boxes, masks, valid, ins = make_inputs(rng, ins, 100)
    bl = boxlist(cuda, boxes, masks, valid, ins)
    (chars, offsets), _ = detector_postprocess_rle(bl, outs)
    got = strings(chars, offsets)
    assert got == per_image_strings(cuda, boxes, masks, valid, ins, outs, "fixed", with_planes=False)
    for n in (0, 7, 15):
        sl = slice(n, n + 1)
        assert got[n * 100:(n + 1) * 100] == oracle_strings(oracle_lib, boxes[sl], masks[sl], valid[sl], ins[sl],
                                                            outs[n:n + 1], "fixed")


def test_batched_rle_capacity(cuda, oracle_lib, guard):
    """Capacity 0 (the sizing query), exactly offsets[-1] and one byte short, with chars, offsets, the validity and
    both shape arrays between canary bands."""
    rng = np.random.default_rng(11)
    boxes, masks, valid, ins = make_inputs(rng, IN4, 9)
    valid[-1, -1] = True
    outs = OUTS["scales"]
    want = oracle_strings(oracle_lib, boxes, masks, valid, ins, outs, "fixed")
    cum = np.cumsum([0] + [len(s) for s in want]).tolist()

    def banded(a, dtype):
        t = torch.empty(a.shape, dtype=dtype, device=cuda)
        t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        return t
    bl = BoxList(T(boxes, cuda))
    bl.add_field("pred_masks", T(masks, cuda))
    bl.add_field("is_valid", banded(valid.astype(np.uint8), torch.uint8))
    bl.set_tracking("image_shape", banded(ins, torch.int32))
    os_ = banded(np.asarray(outs, np.int32), torch.int32)
    (chars, offsets), _ = detector_postprocess_rle(bl, os_, capacity=0)
    assert chars.numel() == 0 and offsets.cpu().tolist() == cum
    with pytest.raises(ValueError, match=f"need {cum[-1]} bytes"):
        rle_to_coco(chars, offsets, sizes=np.repeat(outs, 9, 0))
    (chars, offsets), _ = detector_postprocess_rle(bl, os_, capacity=cum[-1])
    assert strings(chars, offsets) == want
    (chars, offsets), _ = detector_postprocess_rle(bl, os_, capacity=cum[-1] - 1)
    assert offsets.cpu().tolist() == cum
    data = chars.cpu().numpy().tobytes()
    assert data[:cum[-2]] == b"".join(want[:-1])
    assert set(data[cum[-2]:]) == {PATTERN}  # the last string did not fit: untouched
    guard.check()


def test_batched_rle_out_of_range_device_shapes(cuda, oracle_lib, guard):
    """Sizes the host never saw: every slot of an image with h < 1, w < 1 or h * w >= 2^31 - 65536 is an empty string,
    nothing is read or written out of bounds, and the other images are unaffected."""
    rng = np.random.default_rng(5)
    bad = [(0, 50), (50, -3), (46341, 46341), (65536, 65536), (-2147483648, -1), (2147483647, 2147483647)]
    good = [(70, 90), (1, 1)]
    outs = np.array(good[:1] + bad + good[1:], np.int32)
    ins = [(60, 80)] * len(outs)
    boxes, masks, valid, ins = make_inputs(rng, ins, 6, p_valid=1.0)
    os_ = torch.empty(outs.shape, dtype=torch.int32, device=cuda)
    os_.copy_(torch.from_numpy(outs))
    bl = boxlist(cuda, boxes, masks, valid, ins)
    (chars, offsets), _ = detector_postprocess_rle(bl, os_)
    got = strings(chars, offsets)
    assert got[6:6 * (1 + len(bad))] == [b""] * (6 * len(bad))
    ends = [0, len(outs) - 1]
    want = oracle_strings(oracle_lib, boxes[ends], masks[ends], valid[ends], ins[ends], outs[ends], "fixed")
    assert got[:6] + got[-6:] == want
    guard.check()
    with pytest.raises(ValueError, match=r"output_shapes\[1\]"):
        detector_postprocess_rle(bl, outs)  # the same sizes from the host are refused before any call


def test_batched_rle_misuse_launches_nothing(cuda):
    """EINVAL before any launch: planes requested in the batched mode, output_shapes NULL, N x R != num_masks."""
    M = 6
    masks = torch.rand(M, 14, 14, device=cuda)
    boxes = torch.zeros(M, 4, device=cuda)
    shapes = torch.full((2, 2), 8, dtype=torch.int32, device=cuda)
    offsets = torch.full((M + 1,), -7, dtype=torch.int64, device=cuda)
    planes = torch.empty(M, 8, 8, dtype=torch.uint8, device=cuda)

    def params():
        p = nv.PasteMasksParams()
        p.box_masks, p.boxes, p.num_masks, p.mask_h, p.mask_w = masks.data_ptr(), boxes.data_ptr(), M, 14, 14
        p.mask_threshold = 0.5
        p.num_images, p.dets_per_image, p.output_shapes, p.out_rle_offsets = 2, 3, shapes.data_ptr(), offsets.data_ptr()
        return p
    cases = []
    p = params(); p.out = planes.data_ptr(); cases.append(p)
    p = params(); p.output_shapes = None; cases.append(p)
    p = params(); p.out_rle_offsets = None; cases.append(p)
    p = params(); p.dets_per_image = 4; cases.append(p)
    p = params(); p.num_images = 0; cases.append(p)   # batched fields without the batched mode
    L = nv._bind("paste_masks")
    torch.cuda.synchronize()
    before = nv.kernel_launch_count()
    for p in cases:
        assert L.d2b_paste_masks(C.byref(p), None, 0, None) == -1
    assert nv.kernel_launch_count() == before
    torch.cuda.synchronize()
    assert offsets.cpu().tolist() == [-7] * (M + 1)
    with pytest.raises(ValueError, match="batched mode"):
        p = params(); p.out = planes.data_ptr()
        nv.call("paste_masks", p, cuda)


def test_batched_rle_graph_replay(cuda, oracle_lib):
    """A fixed capacity and device output sizes make the call sync-free: captured once, replayed with new masks, new
    validity and new sizes written in place, equal to the eager call."""
    rng = np.random.default_rng(9)
    a = make_inputs(rng, IN4, 12)
    b = make_inputs(rng, IN4, 12)
    bl = boxlist(cuda, *a)
    outs_a, outs_b = np.array(OUTS["scales"], np.int32), np.array(OUTS["coco_like"], np.int32)
    os_ = T(outs_a, cuda)
    cap = 1 << 18
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        detector_postprocess_rle(bl, os_, capacity=cap)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        (chars_g, off_g), boxes_g = detector_postprocess_rle(bl, os_, capacity=cap)
    bl.boxes.copy_(T(b[0], cuda))
    bl.get_field("pred_masks").copy_(T(b[1], cuda))
    bl.get_field("is_valid").copy_(T(b[2], cuda))
    os_.copy_(T(outs_b, cuda))
    g.replay()
    torch.cuda.synchronize()
    (chars_e, off_e), boxes_e = detector_postprocess_rle(bl, os_, capacity=cap)
    assert torch.equal(off_g, off_e) and strings(chars_g, off_g) == strings(chars_e, off_e)
    assert torch.equal(boxes_g, boxes_e)
    assert off_e[-1].item() <= cap
    assert strings(chars_g, off_g) == oracle_strings(oracle_lib, *b, outs_b, "fixed")


def test_coco_results_on_device(cuda):
    """coco_results over a real batched call: one entry per valid slot, its string, size and the scaled box."""
    rng = np.random.default_rng(3)
    boxes, masks, valid, ins = make_inputs(rng, IN4, 8)
    bl = boxlist(cuda, boxes, masks, valid, ins)
    bl.add_field("scores", T(rng.random((4, 8)).astype(np.float32), cuda))
    bl.add_field("pred_classes", T(rng.integers(0, 80, (4, 8)), cuda))
    outs = OUTS["coco_like"]
    rle, pb = detector_postprocess_rle(bl, outs)
    cats = list(range(1, 91))[:80]
    res = coco_results(bl, rle, pb, outs, [101, 102, 103, 104], cats)
    got = strings(*rle)
    slots = np.flatnonzero(valid.reshape(-1))
    assert len(res) == len(slots)
    sb = scaled(boxes, ins, outs).reshape(-1, 4)
    cls = bl.get_field("pred_classes").cpu().numpy().reshape(-1)
    for r, i in zip(res, slots):
        n = i // 8
        assert r["image_id"] == 101 + n and r["category_id"] == cats[cls[i]]
        assert r["segmentation"] == {"size": list(outs[n]), "counts": got[i]}
        y0, x0, y1, x1 = sb[i]
        assert r["bbox"] == [float(x0), float(y0), float(x1 - x0), float(y1 - y0)]
