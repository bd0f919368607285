"""GPU parity: mask paste-back (reframe_box_masks_to_image_masks, mask_ops.py:7-56) vs the oracle, bit-exact."""
import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200.structures import reframe_box_masks_to_image_masks
from detectron2_tensorflow_b200.utils import synthetic as syn

pytestmark = pytest.mark.gpu


def _masks(rng, M, mh, mw):
    # smooth blobs in (0,1) so the 0.5 level set crosses many pixels
    yy, xx = np.mgrid[0:mh, 0:mw].astype(np.float32)
    out = np.zeros((M, mh, mw), np.float32)
    for i in range(M):
        cy, cx = rng.uniform(0.3, 0.7) * mh, rng.uniform(0.3, 0.7) * mw
        r = rng.uniform(0.2, 0.5) * mh
        out[i] = 1.0 / (1.0 + np.exp((np.hypot(yy - cy, xx - cx) - r) * 0.8))
    return out + rng.uniform(-0.05, 0.05, out.shape).astype(np.float32)


@pytest.mark.parametrize("H,W,mh,mw", [(97, 131, 28, 28), (64, 96, 14, 14), (50, 75, 7, 9), (1, 40, 28, 28)])
def test_paste_masks_small(cuda, oracle_lib, H, W, mh, mw):
    rng = np.random.default_rng(H * W)
    M = 24
    masks = _masks(rng, M, mh, mw)
    boxes, _ = syn.rois(1, M, seed=3, image_hw=(H, W))
    boxes[0] = [-20, -30, H + 10, W + 5]     # larger than the image
    boxes[1] = [5, 5, 5, 20]                 # zero height -> division by zero in the reverse box (inf/NaN)
    boxes[2] = [10.5, 3.25, 11.0, 4.0]       # sub-pixel box
    want = oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W), 0.5)
    got = reframe_box_masks_to_image_masks(torch.from_numpy(masks).to(cuda), torch.from_numpy(boxes).to(cuda), (H, W), 0.5)
    assert got.dtype == torch.uint8 and tuple(got.shape) == (M, H, W)
    assert np.array_equal(got.cpu().numpy(), want)
    e = reframe_box_masks_to_image_masks(torch.zeros((0, mh, mw), device=cuda), torch.zeros((0, 4), device=cuda), (H, W))
    assert tuple(e.shape) == (0, H, W)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_paste_masks_adversarial_boxes(cuda, oracle_lib, seed):
    """memset + a kernel over a conservative bounding rectangle of each box, against the oracle, on boxes that stress
    the rectangle: reversed (negative step), outside the image, degenerate, sub-pixel, huge coordinates, NaN / inf."""
    rng = np.random.default_rng(seed)
    H, W, mh, mw, M = 61, 83, 28, 28, 40
    masks = _masks(rng, M, mh, mw)
    y0 = rng.uniform(-30, H + 10, M); x0 = rng.uniform(-30, W + 10, M)
    boxes = np.stack([y0, x0, y0 + rng.uniform(-20, 60, M), x0 + rng.uniform(-20, 60, M)], 1).astype(np.float32)
    boxes[0] = [40, 60, 10, 5]                 # reversed on both axes
    boxes[1] = [-500, -500, -400, -300]        # far outside
    boxes[2] = [3, 3, 3, 3]                    # a point
    boxes[3] = [1e7, 2e7, 3e7, 4e7]
    boxes[4] = [np.nan, 0, 10, 10]
    boxes[5] = [0, 0, np.inf, 20]
    boxes[6] = [12.25, 7.5, 12.75, 8.0]        # sub-pixel
    boxes[7] = [0, 0, H, W]
    want = oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (H, W), 0.5)
    tm, tb = torch.from_numpy(masks).to(cuda), torch.from_numpy(boxes).to(cuda)
    got = reframe_box_masks_to_image_masks(tm, tb, (H, W), 0.5).cpu().numpy()
    assert np.array_equal(got, want)


def test_paste_masks_full_image(cuda, oracle_lib):
    """100 detections of one 800x1333 image, 28x28 masks (Mask R-CNN inference shapes)."""
    rng = np.random.default_rng(5)
    M = 100
    masks = _masks(rng, M, 28, 28)
    boxes, _ = syn.rois(1, M, seed=8)
    want = oracle_lib.reframe_box_masks_to_image_masks(masks, boxes, (800, 1333), 0.5)
    got = reframe_box_masks_to_image_masks(torch.from_numpy(masks).to(cuda), torch.from_numpy(boxes).to(cuda), (800, 1333))
    assert np.array_equal(got.cpu().numpy(), want)
    assert want.sum() > 0


def test_mask_rcnn_inference(cuda, oracle_lib):
    """mask_rcnn_inference (mask_head.py:71-103): gather of the predicted class channel + sigmoid, bit-exact vs the oracle
    (same Cephes sigmoid), 1e-6 vs the reference-python golden; class-agnostic head; out-of-range classes."""
    import os
    import torch
    from detectron2_tensorflow_b200.modeling import mask_rcnn_inference
    from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList
    rng = np.random.default_rng(31)

    def run(logits, classes):
        M = logits.shape[0]
        idx = torch.stack([torch.zeros(M, dtype=torch.int64), torch.arange(M)], 1).to(cuda)
        inst = SparseBoxList(idx, BoxList(torch.zeros((M, 4), device=cuda)), (1, M))
        inst.data.add_field("pred_classes", torch.from_numpy(classes).to(cuda))
        assert mask_rcnn_inference(torch.from_numpy(logits).to(cuda), inst) is None
        return inst.data.get_field("pred_masks").cpu().numpy()

    for M, hm, C in ((1600, 28, 80), (37, 14, 3), (5, 7, 1)):
        lg = (rng.standard_normal((M, hm, hm, C)) * 4).astype(np.float32)
        cl = rng.integers(0, C, M).astype(np.int64)
        if C > 1:
            cl[0], cl[-1] = -1, C  # out of range: sigmoid(0)
        assert np.array_equal(run(lg, cl), oracle_lib.mask_rcnn_inference(lg, cl))
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_python.npz"))
    assert np.allclose(run(z["mi_logits"], z["mi_classes"]), z["mi_out"], rtol=1e-6, atol=1e-7)
