"""GPU: COCO run-length strings emitted by d2b_paste_masks and d2b_solo_upsample (csrc/mask_rle.cuh), bit-exact bytes
and offsets against the restatement of pycocotools in coco_rle.py applied to the oracle's masks."""
import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import solo_upsample_masks
from detectron2_tensorflow_b200.structures import reframe_box_masks_to_image_masks, reframe_box_masks_to_rle, rle_to_coco
from detectron2_tensorflow_b200.utils import synthetic as syn

import coco_rle
import test_paste_masks_gpu as pm
import test_solo_upsample_gpu as su
from test_canary_gpu import PATTERN, guard  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def strings(chars, offsets):
    off = offsets.cpu().numpy()
    data = chars.cpu().numpy().tobytes()
    return [data[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def check_paste(cuda, oracle_lib, masks, boxes, HW, thr=0.5):
    want = coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, HW, thr))
    chars, offsets = reframe_box_masks_to_rle(T(masks, cuda), T(boxes, cuda), HW, thr)
    assert offsets.cpu().tolist() == np.cumsum([0] + [len(s) for s in want]).tolist()
    assert chars.numel() == offsets[-1].item()
    assert strings(chars, offsets) == want
    return want


def adversarial_boxes(rng, H, W, M):
    y0 = rng.uniform(-30, H + 10, M); x0 = rng.uniform(-30, W + 10, M)
    boxes = np.stack([y0, x0, y0 + rng.uniform(-20, 60, M), x0 + rng.uniform(-20, 60, M)], 1).astype(np.float32)
    boxes[0] = [40, 60, 10, 5]                 # reversed on both axes: a mirrored mask
    boxes[1] = [-500, -500, -400, -300]        # far outside
    boxes[2] = [3, 3, 3, 3]                    # a point
    boxes[3] = [1e7, 2e7, 3e7, 4e7]
    boxes[4] = [np.nan, 0, 10, 10]
    boxes[5] = [0, 0, np.inf, 20]
    boxes[6] = [12.25, 7.5, 12.75, 8.0]        # sub-pixel
    boxes[7] = [0, 0, H, W]                    # whole image
    boxes[8] = [5, 5, 5, 20]                   # zero height
    boxes[9] = [-20, -30, H + 10, W + 5]       # larger than the image
    return boxes


@pytest.mark.parametrize("H,W,mh,mw", [(97, 131, 28, 28), (64, 96, 14, 14), (50, 75, 7, 9), (1, 40, 28, 28),
                                       (61, 83, 28, 28)])
@pytest.mark.parametrize("seed", [0, 1])
def test_paste_rle_adversarial(cuda, oracle_lib, H, W, mh, mw, seed):
    rng = np.random.default_rng(seed * 1000 + H * W)
    M = 40
    masks = pm._masks(rng, M, mh, mw)
    boxes = adversarial_boxes(rng, H, W, M)
    boxes[20:], _ = syn.rois(1, M - 20, seed=3 + seed, image_hw=(H, W))
    check_paste(cuda, oracle_lib, masks, boxes, (H, W))


@pytest.mark.parametrize("H,W", [(45, 70), (64, 33), (800, 1333)])
def test_paste_rle_image_edges(cuda, oracle_lib, H, W):
    """Whole-image boxes: pixel 0 and pixel H*W-1 set, ones in row H-1 running on into row 0 of the next column,
    a full mask, a mask of the last row only, thresholds that keep everything / nothing."""
    mh = mw = 28
    m = np.zeros((6, mh, mw), np.float32)
    m[0] = 1                                   # everything: "0" + H*W
    m[1, 0, :] = m[1, -1, :] = 1               # top and bottom rows: runs across column boundaries
    m[2, -1, :] = 1                            # bottom row only
    m[3, 0, 0] = m[3, -1, -1] = 1              # the two corner pixels (and their bilinear neighbourhoods)
    m[4] = np.indices((mh, mw)).sum(0) % 2     # checkerboard
    m[5, :, 0] = 1                             # first column
    boxes = np.tile(np.array([[0, 0, H, W]], np.float32), (6, 1))
    want = check_paste(cuda, oracle_lib, m, boxes, (H, W))
    assert want[0] == coco_rle.encode(np.ones((1, H, W), np.uint8))[0]
    img = oracle_lib.reframe_box_masks_to_image_masks(m, boxes, (H, W))
    assert img[1, 0, 0] and img[1, -1, 0] and img[3, 0, 0] and img[3, -1, -1]
    for thr in (-1.0, 1.0):
        check_paste(cuda, oracle_lib, m, boxes, (H, W), thr)


def test_paste_rle_unbounded_runs(cuda, oracle_lib):
    """An H x W checkerboard box mask on the whole-image box at 800 x 1333: about a million runs per mask."""
    H, W = 800, 1333
    cb = (np.indices((H, W)).sum(0) % 2).astype(np.float32)
    masks = np.stack([cb, 1 - cb])
    boxes = np.array([[0, 0, H, W], [0, 0, H, W]], np.float32)
    want = check_paste(cuda, oracle_lib, masks, boxes, (H, W))
    assert min(len(s) for s in want) > 1_000_000


def test_paste_rle_full_batch(cuda, oracle_lib):
    """16 images x 100 detections, 28x28 masks on 800x1333 (the boxes of tools/paste_probe.py), in one call."""
    rng = np.random.default_rng(0)
    M, H, W = 1600, 800, 1333
    masks = rng.random((M, 28, 28)).astype(np.float32)
    cy, cx = rng.uniform(0, H, M), rng.uniform(0, W, M)
    h = np.exp(rng.uniform(np.log(20), np.log(500), M)); w = np.exp(rng.uniform(np.log(20), np.log(500), M))
    boxes = np.stack([np.clip(cy - h / 2, 0, H), np.clip(cx - w / 2, 0, W), np.clip(cy + h / 2, 0, H),
                      np.clip(cx + w / 2, 0, W)], 1).astype(np.float32)
    chars, offsets = reframe_box_masks_to_rle(T(masks, cuda), T(boxes, cuda), (H, W))
    got = strings(chars, offsets)
    for i0 in range(0, M, 100):
        want = coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(masks[i0:i0 + 100], boxes[i0:i0 + 100], (H, W)))
        assert got[i0:i0 + 100] == want


def test_paste_planes_unchanged_with_rle(cuda, oracle_lib):
    """One call that writes the planes and the strings: planes byte-identical to the plane-only call."""
    rng = np.random.default_rng(7)
    H, W, M = 61, 83, 40
    masks = pm._masks(rng, M, 28, 28)
    boxes = adversarial_boxes(rng, H, W, M)
    tm, tb = T(masks, cuda), T(boxes, cuda)
    plain = reframe_box_masks_to_image_masks(tm, tb, (H, W))
    out = torch.full((M, H, W), 7, dtype=torch.uint8, device=cuda)
    offsets = torch.empty(M + 1, dtype=torch.int64, device=cuda)
    chars = torch.empty(1 << 16, dtype=torch.uint8, device=cuda)
    p = nv.PasteMasksParams()
    p.box_masks, p.boxes, p.num_masks, p.mask_h, p.mask_w, p.image_h, p.image_w = tm.data_ptr(), tb.data_ptr(), M, 28, 28, H, W
    p.mask_threshold = 0.5
    p.out, p.out_rle, p.rle_capacity, p.out_rle_offsets = out.data_ptr(), chars.data_ptr(), chars.numel(), offsets.data_ptr()
    nv.call("paste_masks", p, cuda)
    assert torch.equal(out, plain)
    want = coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W)))
    assert strings(chars, offsets) == want
    assert nv.lib().d2b_paste_masks_workspace_bytes(nv.C.byref(p)) == 0


def test_paste_rle_capacity(cuda, oracle_lib, guard):
    """Capacity 0 (the sizing query), exactly offsets[M], and one byte short (the last string is not written), with
    every output between canary bands; then M = 0."""
    rng = np.random.default_rng(11)
    H, W, M = 97, 131, 24
    masks = pm._masks(rng, M, 28, 28)
    boxes, _ = syn.rois(1, M, seed=3, image_hw=(H, W))
    want = coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W)))
    total = sum(len(s) for s in want)
    tm, tb = T(masks, cuda), T(boxes, cuda)
    cum = np.cumsum([0] + [len(s) for s in want]).tolist()
    chars, offsets = reframe_box_masks_to_rle(tm, tb, (H, W), capacity=0)
    assert chars.numel() == 0 and offsets.cpu().tolist() == cum
    with pytest.raises(ValueError, match=f"need {total} bytes"):
        rle_to_coco(chars, offsets, (H, W))
    chars, offsets = reframe_box_masks_to_rle(tm, tb, (H, W), capacity=total)
    assert [d["counts"] for d in rle_to_coco(chars, offsets, (H, W))] == want
    chars, offsets = reframe_box_masks_to_rle(tm, tb, (H, W), capacity=total - 1)
    assert offsets.cpu().tolist() == cum
    got = chars.cpu().numpy().tobytes()
    assert got[:cum[-2]] == b"".join(want[:-1])
    assert set(got[cum[-2]:]) == {PATTERN}  # the last string did not fit: untouched
    e_chars, e_off = reframe_box_masks_to_rle(tm[:0], tb[:0], (H, W), capacity=0)
    assert e_chars.numel() == 0 and e_off.cpu().tolist() == [0]
    assert rle_to_coco(*reframe_box_masks_to_rle(tm[:0], tb[:0], (H, W)), (H, W)) == []
    guard.check()


def test_paste_rle_graph_replay(cuda, oracle_lib):
    """A fixed capacity makes the call sync-free: captured once, replayed on new inputs, equal to the eager call."""
    rng = np.random.default_rng(5)
    H, W, M = 200, 300, 30
    a, b = pm._masks(rng, M, 28, 28), pm._masks(rng, M, 28, 28)
    boxes, _ = syn.rois(1, M, seed=8, image_hw=(H, W))
    tm, tb = T(a, cuda), T(boxes, cuda)
    cap = 1 << 16
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        reframe_box_masks_to_rle(tm, tb, (H, W), capacity=cap)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        chars_g, off_g = reframe_box_masks_to_rle(tm, tb, (H, W), capacity=cap)
    tm.copy_(T(b, cuda))
    g.replay()
    torch.cuda.synchronize()
    chars_e, off_e = reframe_box_masks_to_rle(tm, tb, (H, W), capacity=cap)
    assert torch.equal(off_g, off_e) and strings(chars_g, off_g) == strings(chars_e, off_e)
    assert strings(chars_g, off_g) == coco_rle.encode(oracle_lib.reframe_box_masks_to_image_masks(b, boxes, (H, W)))


def solo_want(oracle_lib, m, HW, ac, thr):
    return [s for b in range(m.shape[0]) for s in coco_rle.encode(oracle_lib.solo_upsample_boxes(m[b], HW, ac, thr)[0])]


@pytest.mark.parametrize("hw,HW,ac", [((20, 32), (80, 128), False), ((20, 32), (80, 128), True), ((25, 37), (101, 149), False),
                                      ((40, 64), (33, 50), True), ((3, 5), (64, 1), True), ((1, 1), (17, 19), False)])
def test_solo_rle(cuda, oracle_lib, hw, HW, ac):
    rng = np.random.default_rng(hw[0] * 100 + HW[1] + int(ac))
    B, D = 2, 7
    m = su.blobs(rng, B, D, *hw)
    m[0, 0] = 0                      # empty mask: padding rows encode as [H*W]
    m[0, 1] = 1
    m[1, 0] = 0; m[1, 0, 0, :] = 1
    m[1, 1] = 0; m[1, 1, :, 0] = 1
    m[1, 2] = (rng.random(hw) > 0.5).astype(np.float32)
    m[1, 3] = 0; m[1, 3, -1, -1] = 1  # the last source pixel only
    pk = T(su.pack(m), cuda)
    plain = solo_upsample_masks(pk, hw, HW, 0.5, ac, return_masks=True, return_packed=True)
    want = solo_want(oracle_lib, m, HW, ac, 0.5)
    for cap in (None, 1 << 20):
        got = solo_upsample_masks(pk, hw, HW, 0.5, ac, return_masks=True, return_packed=True, return_rle=True,
                                  rle_capacity=cap)
        for k in ("pred_masks", "packed_masks", "boxes"):
            assert torch.equal(got[k], plain[k]), k
        assert strings(*got["rle"]) == want
    only = solo_upsample_masks(pk, hw, HW, 0.5, ac, return_masks=False, return_rle=True)
    assert only["pred_masks"] is None and torch.equal(only["boxes"], plain["boxes"])
    assert strings(*only["rle"]) == want
    assert want[0] == coco_rle.encode(np.zeros((1,) + HW, np.uint8))[0]


@pytest.mark.parametrize("thr", [0.0, 0.3, 0.75, 1.0, -0.1, 1.5])
def test_solo_rle_thresholds(cuda, oracle_lib, thr):
    rng = np.random.default_rng(3)
    m = su.blobs(rng, 1, 9, 30, 44)
    m[0, 8] = 0
    got = solo_upsample_masks(T(su.pack(m), cuda), (30, 44), (121, 170), thr, False, return_masks=False, return_rle=True)
    assert strings(*got["rle"]) == solo_want(oracle_lib, m, (121, 170), False, thr)


def test_solo_rle_full_size(cuda, oracle_lib):
    """16 images x 100 kept masks at 200x336 -> 800x1333; half of the last image's rows are padding."""
    m = np.stack([syn.solo_masks(100, hw=(200, 336), seed=70 + i)[0] for i in range(16)]).astype(np.float32)
    m[15, 50:] = 0
    pk = T(su.pack(m), cuda)
    got = solo_upsample_masks(pk, (200, 336), (800, 1333), 0.5, False, return_masks=False, return_rle=True)
    plain = solo_upsample_masks(pk, (200, 336), (800, 1333), 0.5, False, return_masks=False)
    assert torch.equal(got["boxes"], plain["boxes"])
    s = strings(*got["rle"])
    for b in (0, 7, 15):
        assert s[b * 100:(b + 1) * 100] == solo_want(oracle_lib, m[b:b + 1], (800, 1333), False, 0.5)


def test_solo_rle_capacity_and_empty(cuda, oracle_lib, guard):
    rng = np.random.default_rng(4)
    m = su.blobs(rng, 2, 5, 20, 32)
    pk = T(su.pack(m), cuda)
    want = solo_want(oracle_lib, m, (80, 128), True, 0.5)
    cum = np.cumsum([0] + [len(s) for s in want]).tolist()
    got = solo_upsample_masks(pk, (20, 32), (80, 128), 0.5, True, return_masks=False, return_rle=True, rle_capacity=0)
    assert got["rle"][0].numel() == 0 and got["rle"][1].cpu().tolist() == cum
    got = solo_upsample_masks(pk, (20, 32), (80, 128), 0.5, True, return_masks=False, return_rle=True,
                              rle_capacity=cum[-1] - 1)
    data = got["rle"][0].cpu().numpy().tobytes()
    assert data[:cum[-2]] == b"".join(want[:-1]) and set(data[cum[-2]:]) == {PATTERN}
    e = solo_upsample_masks(pk[:, :0], (20, 32), (80, 128), 0.5, True, return_masks=False, return_rle=True)
    assert e["rle"][1].cpu().tolist() == [0]
    guard.check()
