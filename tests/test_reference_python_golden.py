"""CPU: the oracle against outputs of the REFERENCE'S OWN PYTHON, executed unmodified on a numpy
TF shim in the build container (tests/golden/make_reference_golden.py + tf_numpy_shim.py ->
tests/golden/reference_python.npz).  This pins the oracle's restatement of the reference's composition
(op order, ties, padding, class offsets, level routing, label stitching) to the reference's code.

Exact (np.array_equal) wherever the path contains only +,-,*,/,min,max,compare,floor; 1e-5 relative
where numpy's exp/log stand in for Eigen's (apply_deltas/get_deltas/matrix_nms), per north_star.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_golden  # noqa: E402


@pytest.fixture(scope="module")
def z():
    return reference_golden.load()


def test_pairwise_iou(oracle_lib, z):
    assert np.array_equal(oracle_lib.pairwise_iou(z["iou_b1"], z["iou_b2"]), z["iou_out"])


def test_matcher(oracle_lib, z):
    for c in range(int(z["m_num_cases"])):
        lq, uc, ud = (int(v) for v in z[f"m{c}_cfg"])
        m, l = oracle_lib.matcher(z["m_q"], z[f"m{c}_th"], z[f"m{c}_lab"], bool(lq), z["m_crowd"] if uc else None,
                                  z["m_diff"] if ud else None)
        assert np.array_equal(m, z[f"m{c}_matches"]), c
        assert np.array_equal(l, z[f"m{c}_labels"]), c


def test_box2box_transform(oracle_lib, z):
    w = (10., 10., 5., 5.)
    got = oracle_lib.get_deltas(z["bt_src"], z["bt_tgt"], w)
    assert np.allclose(got, z["bt_get"], rtol=1e-5, atol=1e-6)
    assert np.array_equal(got[:, :2], z["bt_get"][:, :2])  # dy, dx contain no transcendental: exact
    got = oracle_lib.apply_deltas(z["bt_deltas"], z["bt_src"], w)
    assert np.allclose(got, z["bt_apply"], rtol=1e-5, atol=1e-3)


def test_level_assignment(oracle_lib, z):
    assert np.array_equal(oracle_lib.assign_boxes_to_levels(z["rp_boxes"], 2, 5, 224, 4), z["rp_levels"])
    lv = oracle_lib.assign_boxes_to_levels(z["rp_boxes"], 2, 5, 56, 4)
    assert np.array_equal(lv, z["rp_levels56"]) and len(np.unique(lv)) == 4


@pytest.mark.parametrize("ptype,sr,osz", [("ROIAlignV2", 0, 7), ("ROIAlignV2", 2, 7), ("ROIAlign", 0, 14)])
def test_roi_pooler(oracle_lib, z, ptype, sr, osz):
    feats = [z[f"rp_feat{l}"] for l in range(4)]
    got, _ = oracle_lib.roi_pooler(feats, [1 / 4., 1 / 8., 1 / 16., 1 / 32.], z["rp_boxes"], z["rp_idx"][:, 0],
                                   (osz, osz), sr, aligned=(ptype == "ROIAlignV2"), canonical_box_size=56)
    assert np.array_equal(got[z["rp_rows"]], z[f"rp_out_{ptype}_{sr}_{osz}"])


def test_roi_align_and_crop(oracle_lib, z):
    bi = z["rp_idx"][:, 0].astype(np.int32)
    rows = z["rp_rows"]
    got = oracle_lib.roi_align(z["rp_feat1"], z["rp_boxes"], bi, (7, 7), 1 / 8., 0, True)
    assert np.array_equal(got[rows], z["ra_single"])
    got = oracle_lib.crop_and_resize(z["rp_feat0"], z["rp_boxes"] * np.float32(0.25), bi, (5, 6), True, False)
    assert np.array_equal(got[rows], z["cr_nopad"])


def test_find_top_rpn_proposals(oracle_lib, z):
    props = [z[f"rpn_props{l}"] for l in range(3)]
    logits = [z[f"rpn_logits{l}"] for l in range(3)]
    padded = 0
    for c in range(int(z["rpn_num_cases"])):
        pre, post, msl = z[f"rpn{c}_cfg"]
        b, l, v, n = oracle_lib.find_top_rpn_proposals(props, logits, z["rpn_shapes"], 0.7, int(pre), int(post), float(msl))
        assert np.array_equal(v, z[f"rpn{c}_valid"])
        assert np.array_equal(b, z[f"rpn{c}_boxes"])
        assert np.array_equal(l, z[f"rpn{c}_logits"])
        padded += int(v.sum() < v.size)
    assert padded > 0  # at least one case exercises the zero padding / is_valid=False tail


def test_fast_rcnn_inference(oracle_lib, z):
    for c, (agn, boxes) in enumerate(((False, z["fr_pred"]), (True, z["fr_agnostic_boxes"]))):
        b, s, cl, v, _, _ = oracle_lib.fast_rcnn_inference(boxes, z["fr_scores"], z["fr_idx"], tuple(z["fr_dense"]),
                                                           z["fr_shapes"], 0.05, 0.5, 15, agn)
        assert np.array_equal(v, z[f"fr{c}_valid"])
        assert np.array_equal(cl, z[f"fr{c}_classes"])
        assert np.array_equal(s, z[f"fr{c}_scores"])
        assert np.array_equal(b, z[f"fr{c}_boxes"])


def test_matrix_nms(oracle_lib, z):
    shp = tuple(z["mn_shape"])
    m = np.unpackbits(z["mn_masks"])[:int(np.prod(shp))].reshape(shp).astype(np.float32)
    got = oracle_lib.matrix_nms(m, z["mn_classes"], z["mn_scores"], None, "gaussian", 2.0)
    assert np.allclose(got, z["mn_gauss"], rtol=1e-5, atol=1e-7)
    # linear kernel: identical same-class masks give compensate_iou == 1 => the decay column holds 0/0 = NaN
    # next to finite values, and tf.reduce_min over a column containing NaN is order-dependent in TF
    # (Eigen's pmin keeps or drops NaN by operand position).  numpy propagates NaN; the oracle (and the
    # kernel) use IEEE fmin, which drops it.  Columns without NaN must agree; NaN columns are unspecified.
    got = oracle_lib.matrix_nms(m, z["mn_classes"], z["mn_scores"], None, "linear", 2.0)
    want = z["mn_linear"]
    ok = ~np.isnan(want)
    assert ok.sum() >= want.size // 2
    assert np.allclose(got[ok], want[ok], rtol=1e-5, atol=1e-7)


def test_paste_masks(oracle_lib, z):
    got = oracle_lib.reframe_box_masks_to_image_masks(z["pm_masks"], z["pm_boxes"], (60, 80))
    assert np.array_equal(got, z["pm_out"])
    assert 0 < got.sum() < got.size


def test_rpn_ground_truth(oracle_lib, z):
    """RPNOutputs._get_ground_truth (rpn_outputs.py:245-304) == oracle.label_boxes."""
    for c, bthr in enumerate((-1.0, 0.0)):
        _, lab, dl = oracle_lib.label_boxes(z["gt_anchors"], z["gt_boxes"], z["gt_valid"], [0.3, 0.7], [0, -1, 1], True,
                                            gt_crowd=z["gt_crowd"], boundary_threshold=bthr, image_shapes=z["gt_shapes"],
                                            weights=(1., 1., 1., 1.))
        assert np.array_equal(lab, z[f"gt{c}_labels"])
        want = z[f"gt{c}_deltas"]
        assert np.array_equal(dl[..., :2], want[..., :2])
        assert np.allclose(dl, want, rtol=1e-5, atol=1e-6)
        assert (lab == 1).sum() > 0 and (lab == -1).sum() > 0


def test_anchor_generator_host_mirror(z):
    """The product's host-side DefaultAnchorGenerator mirror (plain torch on CPU: host logic, no kernel) against
    the reference's DefaultAnchorGenerator (anchor_generator.py:44-162)."""
    from detectron2_tensorflow_b200.modeling import DefaultAnchorGenerator
    gen = DefaultAnchorGenerator([[32], [64], [128]], [[0.5, 1.0, 2.0]], [int(s) for s in z["ag_strides"]])
    got = gen.grid_anchors([tuple(g) for g in z["ag_grid"]])
    for l in range(3):
        assert np.array_equal(gen.cell_anchors[l].numpy(), z[f"ag_cell{l}"])
        assert np.array_equal(got[l].numpy(), z[f"ag_anchors{l}"])


def test_retinanet_inference(oracle_lib, z):
    """RetinaNetHead.inference (retinanet.py:285-387).  Scores/boxes pass through sigmoid/exp (numpy's in the
    fixture, Eigen-Cephes in the oracle): 1e-5 relative; classes / validity / ordering exact."""
    cls = [z[f"rn_cls{l}"] for l in range(3)]
    reg = [z[f"rn_reg{l}"] for l in range(3)]
    anchors = [z[f"ag_anchors{l}"] for l in range(3)]
    b, s, c, v, n = oracle_lib.retinanet_inference(cls, reg, anchors, 4, 40, 0.05, 0.5, 25)
    assert np.array_equal(v, z["rn_valid"])
    assert np.array_equal(c, z["rn_classes"])
    assert np.allclose(s, z["rn_scores"], rtol=1e-5, atol=1e-7)
    assert np.allclose(b, z["rn_boxes"], rtol=1e-5, atol=1e-3)
    assert 0 < v.sum()


def test_yolo_inference(oracle_lib, z):
    """YOLOV4Outputs.inference (yolov4_outputs.py:331-390): no transcendental on the path => exact."""
    b, s, c, v, n = oracle_lib.yolo_inference(z["yo_boxes_in"], z["yo_probs"], 0.3, 0.5, 40)
    assert np.array_equal(v, z["yo_valid"])
    assert np.array_equal(c, z["yo_classes"])
    assert np.array_equal(s, z["yo_scores"])
    assert np.array_equal(b, z["yo_boxes"])
    assert 0 < v.sum()


def test_point_nms(oracle_lib, z):
    got = oracle_lib.point_nms(z["pn_in"])
    assert np.array_equal(got, z["pn_out"])
    assert 0 < (got != 0).sum() < (z["pn_in"] != 0).sum()


def test_solo_inference_tail(oracle_lib, z):
    """MaskKernelBranch.inference (solo_v2.py:476-612) with image_shape == mask-feature size, from the recorded
    post-conv candidates: masks / classes / validity exact, scores 1e-5 (sigmoid + summation order)."""
    lg, sc, cl, st, cnt = z["so_in_logits"], z["so_in_scores"], z["so_in_classes"], z["so_in_strides"], z["so_in_counts"]
    total = 0
    for b in range(lg.shape[0]):
        c = int(cnt[b])
        m, oc, os_, ov, nv = oracle_lib.solo_postprocess(lg[b, :c], sc[b, :c], cl[b, :c], st[b, :c], 0.5, 30, "gaussian", 2.0,
                                                         0.05, 12)
        assert np.array_equal(ov, z["so_valid"][b])
        assert np.array_equal(oc, z["so_classes"][b])
        assert np.array_equal(m, z["so_masks"][b])
        assert np.allclose(os_, z["so_scores"][b], rtol=1e-5, atol=1e-7)
        total += nv
    assert total > 0


def test_solo_image_masks_and_boxes(oracle_lib, z):
    """The end of MaskKernelBranch.inference (solo_v2.py:599-627) with image_shape != mask-feature size: the reference's
    resize_images (half-pixel branch on the shim) + threshold + boxes from masks, bit-exact."""
    H, W = (int(v) for v in z["so2_image_shape"])
    for b in range(z["so_masks"].shape[0]):
        masks, boxes = oracle_lib.solo_upsample_boxes(z["so_masks"][b], (H, W), False, 0.5)
        assert np.array_equal(masks, z["so2_masks"][b])
        assert np.array_equal(boxes, z["so2_boxes"][b])
    assert z["so2_masks"].any() and not z["so2_masks"].all()


def test_solo_candidate_selection(oracle_lib, z):
    """solo_v2.py:481-497 from the raw arguments of MaskKernelBranch.inference: the oracle's selection equals the
    candidates the golden generator recorded (scores, classes, strides, gathered kernels, counts)."""
    B = z["so_raw_probs_0"].shape[0]
    for b in range(B):
        sc = np.concatenate([z[f"so_raw_probs_{l}"][b].reshape(-1, 3) for l in range(2)], 0)
        kn = np.concatenate([z[f"so_raw_kernels_{l}"][b].reshape(-1, 8) for l in range(2)], 0)
        s, c, k, st = oracle_lib.solo_select(sc, kn, (6, 4), (8, 16), 0.3)
        n = int(z["so_in_counts"][b])
        assert len(s) == n
        assert np.array_equal(s, z["so_in_scores"][b, :n]) and np.array_equal(c, z["so_in_classes"][b, :n])
        assert np.array_equal(k, z["so_in_kernels"][b, :n]) and np.array_equal(st, z["so_in_strides"][b, :n])
        # and the dynamic conv of those candidates reproduces the recorded logits (numpy einsum in the generator)
        lg, absum = oracle_lib.solo_dynamic_conv(z["so_in_mask_features"][b], k)
        assert np.all(np.abs(lg - z["so_in_logits"][b, :n].reshape(n, -1)) <= 1e-5 * absum + 1e-30)


def test_detector_postprocess(oracle_lib, z):
    """detector_postprocess (postprocessing.py:9-59), "fixed" and "conventional": from_dense (row-major valid rows),
    boxes scaled by float32(float64(output_shape) / image_shape) for "fixed", paste, to_dense -- masks bit-exact."""
    valid, shapes = z["dp_valid"], z["dp_shapes"]
    idx = np.argwhere(valid)
    for fmt, oshape in (("fixed", (90, 120)), ("conventional", (60, 80))):
        boxes = z["dp_boxes"][valid]
        if fmt == "fixed":
            sc = (np.array(oshape, np.float64)[None] / shapes.astype(np.float64))[idx[:, 0]].astype(np.float32)
            boxes = np.stack([sc[:, 0] * boxes[:, 0], sc[:, 1] * boxes[:, 1], sc[:, 0] * boxes[:, 2], sc[:, 1] * boxes[:, 3]], 1)
        pasted = oracle_lib.reframe_box_masks_to_image_masks(z["dp_masks"][valid], boxes, oshape, 0.5)
        dense = np.zeros(valid.shape + tuple(oshape), np.uint8)
        dense[valid] = pasted
        assert np.array_equal(dense, z[f"dp_{fmt}_masks"])
        assert np.array_equal(z[f"dp_{fmt}_valid"], valid)
        assert np.array_equal(z[f"dp_{fmt}_boxes"], z["dp_boxes"] * valid[..., None])  # boxes stay unscaled


def test_pairwise_iou_variants(oracle_lib, z):
    """pairwise_iou(iou_type=...) (box_list_ops.py:295-371): iou / giou (with the reference's convex_heights *
    intersect_widths) / diou exact; ciou 1e-5 (atan), same NaN pattern (zero-height boxes)."""
    for ty in ("iou", "giou", "diou"):
        assert np.array_equal(oracle_lib.pairwise_iou(z["pi_a"], z["pi_b"], ty), z[f"pi_{ty}"])
    got, want = oracle_lib.pairwise_iou(z["pi_a"], z["pi_b"], "ciou"), z["pi_ciou"]
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.allclose(got, want, rtol=1e-5, atol=1e-6, equal_nan=True)


def test_mask_rcnn_inference(oracle_lib, z):
    """mask_rcnn_inference (mask_head.py:71-103): class channel of the NHWC logits -> sigmoid (shim sigmoid is numpy's:
    1e-6 relative)."""
    got = oracle_lib.mask_rcnn_inference(z["mi_logits"], z["mi_classes"])
    assert np.allclose(got, z["mi_out"], rtol=1e-6, atol=1e-7)
