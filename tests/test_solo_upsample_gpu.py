"""GPU parity of `d2b_solo_upsample` (csrc/solo_upsample.cu) -- the last stage of MaskKernelBranch.inference,
solo_v2.py:599-627: bilinear resize of the kept masks to the image size, threshold, boxes from masks -- against the
CPU oracle and the reference-python golden.  Integer / byte work: masks, packed words and boxes are compared exactly."""
import os
import sys

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200.modeling import solo_upsample_masks

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_golden  # noqa: E402

pytestmark = pytest.mark.gpu


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def pack(masks01):
    """[..., h, w] 0/1 -> int64 words [..., ceil(h*w/64)], bit p of word w = pixel 64*w+p."""
    flat = masks01.reshape(masks01.shape[:-2] + (-1,)).astype(np.uint8)
    pad = (-flat.shape[-1]) % 64
    flat = np.concatenate([flat, np.zeros(flat.shape[:-1] + (pad,), np.uint8)], -1)
    return np.packbits(flat, axis=-1, bitorder="little").view(np.int64)


def blobs(rng, B, D, h, w):
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    m = np.zeros((B, D, h, w), np.float32)
    for b in range(B):
        for d in range(D):
            cy, cx = rng.uniform(0, h), rng.uniform(0, w)
            ry, rx = rng.uniform(0.6, max(0.7, h / 2)), rng.uniform(0.6, max(0.7, w / 2))
            m[b, d] = (((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1).astype(np.float32)
    return m


def check(cuda, oracle_lib, m, HW, ac, thr=0.5):
    B, D, h, w = m.shape
    H, W = HW
    got = solo_upsample_masks(T(pack(m), cuda), (h, w), HW, thr, ac, return_masks=True, return_packed=True)
    for b in range(B):
        wm, wb = oracle_lib.solo_upsample_boxes(m[b], HW, ac, thr)
        assert np.array_equal(got["pred_masks"][b].cpu().numpy(), wm)
        assert np.array_equal(got["boxes"][b].cpu().numpy(), wb)
        bits = np.unpackbits(got["packed_masks"][b].cpu().numpy().view(np.uint8), axis=-1, bitorder="little")
        assert np.array_equal(bits[:, :H * W].reshape(D, H, W), wm)
        assert not bits[:, H * W:].any()
    return got


@pytest.mark.parametrize("hw,HW,ac", [((20, 32), (80, 128), False), ((20, 32), (80, 128), True), ((24, 32), (95, 130), False),
                                      ((24, 32), (95, 130), True), ((25, 37), (101, 149), False), ((40, 64), (33, 50), False),
                                      ((40, 64), (33, 50), True), ((7, 9), (7, 9), False), ((3, 5), (64, 1), True),
                                      ((1, 1), (17, 19), False), ((50, 84), (200, 333), False)])
def test_upsample_masks_and_boxes(cuda, oracle_lib, hw, HW, ac):
    rng = np.random.default_rng(hw[0] * 100 + HW[1] + int(ac))
    B, D = 2, 7
    m = blobs(rng, B, D, *hw)
    m[0, 0] = 0                      # empty mask: zero box (mean = 0 / 1e-5)
    m[0, 1] = 1                      # full mask
    m[1, 0] = 0; m[1, 0, 0, :] = 1   # only row 0: the `yy > 0` rule sends every pixel to the mean
    m[1, 1] = 0; m[1, 1, :, 0] = 1   # only column 0
    m[1, 2] = (rng.random(hw) > 0.5).astype(np.float32)  # salt and pepper: many values exactly at the threshold
    check(cuda, oracle_lib, m, HW, ac)


@pytest.mark.parametrize("thr", [0.3, 0.5, 0.75, 0.0, 1.0, -0.1, 1.5])
def test_thresholds(cuda, oracle_lib, thr):
    rng = np.random.default_rng(3)
    check(cuda, oracle_lib, blobs(rng, 1, 9, 30, 44), (121, 170), False, thr)


def test_reference_python_golden(cuda):
    """MaskKernelBranch.inference of the reference with image_shape != mask size (tests/golden/make_reference_golden.py
    case 15): the image-size masks and the boxes, bit-exact, from the packed masks of the CUDA tail."""
    from detectron2_tensorflow_b200.modeling import SOLOv2Inference
    z = reference_golden.load()
    head = SOLOv2Inference(0.5, 30, "gaussian", 2.0, 0.05, 12)
    tail = head.postprocess(T(z["so_in_logits"], cuda), T(z["so_in_scores"], cuda), T(z["so_in_classes"], cuda),
                            T(z["so_in_strides"], cuda), T(z["so_in_counts"], cuda), return_masks=False)
    Hm, Wm = z["so_in_logits"].shape[2:]
    got = solo_upsample_masks(tail["packed_masks"], (Hm, Wm), tuple(int(v) for v in z["so2_image_shape"]), 0.5, False)
    assert np.array_equal(got["pred_masks"].cpu().numpy(), z["so2_masks"])
    assert np.array_equal(got["boxes"].cpu().numpy(), z["so2_boxes"])


def test_full_size(cuda, oracle_lib):
    """BASELINE config 4 shapes: 100 kept masks at 200x336 -> 800x1333, 2 images."""
    rng = np.random.default_rng(9)
    m = blobs(rng, 2, 100, 200, 336)
    m[1, 50:] = 0  # padding rows of an image with 50 detections
    got = check(cuda, oracle_lib, m, (800, 1333), False)
    assert not got["boxes"][1, 50:].any()
