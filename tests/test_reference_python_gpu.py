"""GPU: the CUDA path (through the Python mirrors -> C-ABI) against outputs of the REFERENCE'S OWN PYTHON
(tests/golden/reference_python.npz, made by tests/golden/make_reference_golden.py on the numpy TF shim).
Same tolerances as tests/test_reference_python_golden.py: exact except where exp/log/sigmoid are involved."""
import os
import sys

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200.layers import ROIAlign, crop_and_resize, matrix_nms
from detectron2_tensorflow_b200.modeling import (Box2BoxTransform, Matcher, ROIPooler, RetinaNetInference,
                                                 assign_boxes_to_levels, fast_rcnn_inference, find_top_rpn_proposals,
                                                 label_boxes, DefaultAnchorGenerator)
from detectron2_tensorflow_b200.structures import (BoxList, ImageList, SparseBoxList, pairwise_iou,
                                                   reframe_box_masks_to_image_masks)

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_golden  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def z():
    return reference_golden.load()


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def test_pairwise_iou_and_matcher(cuda, z):
    assert np.array_equal(pairwise_iou(T(z["iou_b1"], cuda), T(z["iou_b2"], cuda)).cpu().numpy(), z["iou_out"])
    for c in range(int(z["m_num_cases"])):
        lq, uc, ud = (int(v) for v in z[f"m{c}_cfg"])
        m = Matcher([float(v) for v in z[f"m{c}_th"]], [int(v) for v in z[f"m{c}_lab"]], allow_low_quality_matches=bool(lq))
        mt, ml = m(T(z["m_q"], cuda), T(z["m_crowd"], cuda) if uc else None, T(z["m_diff"], cuda) if ud else None)
        assert np.array_equal(mt.cpu().numpy(), z[f"m{c}_matches"]), c
        assert np.array_equal(ml.cpu().numpy(), z[f"m{c}_labels"]), c


def test_box2box_transform(cuda, z):
    bt = Box2BoxTransform((10., 10., 5., 5.))
    got = bt.get_deltas(T(z["bt_src"], cuda), T(z["bt_tgt"], cuda)).cpu().numpy()
    assert np.array_equal(got[:, :2], z["bt_get"][:, :2])
    assert np.allclose(got, z["bt_get"], rtol=1e-5, atol=1e-6)
    got = bt.apply_deltas(T(z["bt_deltas"], cuda), T(z["bt_src"], cuda)).cpu().numpy()
    assert np.allclose(got, z["bt_apply"], rtol=1e-5, atol=1e-3)


@pytest.mark.parametrize("ptype,sr,osz", [("ROIAlignV2", 0, 7), ("ROIAlignV2", 2, 7), ("ROIAlign", 0, 14)])
def test_roi_pooler(cuda, z, ptype, sr, osz):
    feats = [T(z[f"rp_feat{l}"], cuda) for l in range(4)]
    inst = SparseBoxList(T(z["rp_idx"], cuda), BoxList(T(z["rp_boxes"], cuda)), (2, 60))
    pooler = ROIPooler((osz, osz), [1 / 4., 1 / 8., 1 / 16., 1 / 32.], sr, ptype, canonical_box_size=56)
    got = pooler(feats, inst).cpu().numpy()[z["rp_rows"]]
    want = z[f"rp_out_{ptype}_{sr}_{osz}"]
    if sr == 0:
        assert np.array_equal(got, want)
    else:  # avg-pool summation order is unspecified in TF (SURVEY.md A.4): north_star's 1e-5 relative
        assert np.allclose(got, want, rtol=1e-5, atol=1e-6)
    lv = assign_boxes_to_levels(BoxList(T(z["rp_boxes"], cuda)), 2, 5, 224, 4).cpu().numpy()
    assert np.array_equal(lv, z["rp_levels"])


def test_roi_align_and_crop(cuda, z):
    bi = T(z["rp_idx"][:, 0].astype(np.int32), cuda)
    got = ROIAlign((7, 7), 1 / 8., 0, aligned=True)(T(z["rp_feat1"], cuda), T(z["rp_boxes"], cuda), bi)
    assert np.array_equal(got.cpu().numpy()[z["rp_rows"]], z["ra_single"])
    got = crop_and_resize(T(z["rp_feat0"], cuda), T(z["rp_boxes"] * np.float32(0.25), cuda), bi, [5, 6], aligned=True,
                          pad_border=False)
    assert np.array_equal(got.cpu().numpy()[z["rp_rows"]], z["cr_nopad"])


def test_find_top_rpn_proposals(cuda, z):
    props = [T(z[f"rpn_props{l}"], cuda) for l in range(3)]
    logits = [T(z[f"rpn_logits{l}"], cuda) for l in range(3)]
    images = ImageList(None, T(z["rpn_shapes"], cuda))
    for c in range(int(z["rpn_num_cases"])):
        pre, post, msl = z[f"rpn{c}_cfg"]
        res = find_top_rpn_proposals(props, logits, images, 0.7, int(pre), int(post), float(msl))
        assert np.array_equal(res.get_field("is_valid").cpu().numpy(), z[f"rpn{c}_valid"])
        assert np.array_equal(res.boxes.cpu().numpy(), z[f"rpn{c}_boxes"])
        assert np.array_equal(res.get_field("objectness_logits").cpu().numpy(), z[f"rpn{c}_logits"])


def test_fast_rcnn_inference(cuda, z):
    N, R = (int(v) for v in z["fr_dense"])
    for c, (agn, boxes) in enumerate(((False, z["fr_pred"]), (True, z["fr_agnostic_boxes"]))):
        proposals = SparseBoxList(T(z["fr_idx"], cuda), BoxList(T(z["fr_pred"][:, :4].copy(), cuda)), (N, R))
        proposals.set_tracking("image_shape", T(z["fr_shapes"], cuda))
        res, _ = fast_rcnn_inference(T(boxes, cuda), T(z["fr_scores"], cuda), proposals, 0.05, 0.5, 15, agn)
        assert np.array_equal(res.get_field("is_valid").cpu().numpy(), z[f"fr{c}_valid"])
        assert np.array_equal(res.get_field("pred_classes").cpu().numpy(), z[f"fr{c}_classes"])
        assert np.array_equal(res.get_field("scores").cpu().numpy(), z[f"fr{c}_scores"])
        assert np.array_equal(res.boxes.cpu().numpy(), z[f"fr{c}_boxes"])


def test_matrix_nms_and_paste(cuda, z):
    shp = tuple(z["mn_shape"])
    m = np.unpackbits(z["mn_masks"])[:int(np.prod(shp))].reshape(shp).astype(np.float32)
    got = matrix_nms(T(m, cuda), T(z["mn_classes"], cuda), T(z["mn_scores"], cuda), kernel="gaussian", sigma=2.0)
    assert np.allclose(got.cpu().numpy(), z["mn_gauss"], rtol=1e-5, atol=1e-7)
    got = matrix_nms(T(m, cuda), T(z["mn_classes"], cuda), T(z["mn_scores"], cuda), kernel="linear").cpu().numpy()
    ok = ~np.isnan(z["mn_linear"])  # NaN columns: tf.reduce_min over NaN is unspecified (see the CPU test)
    assert np.allclose(got[ok], z["mn_linear"][ok], rtol=1e-5, atol=1e-7)
    got = reframe_box_masks_to_image_masks(T(z["pm_masks"], cuda), T(z["pm_boxes"], cuda), (60, 80))
    assert np.array_equal(got.cpu().numpy(), z["pm_out"])


def test_rpn_ground_truth(cuda, z):
    m = Matcher([0.3, 0.7], [0, -1, 1], allow_low_quality_matches=True)
    for c, bthr in enumerate((-1, 0)):
        _, lab, dl = label_boxes(T(z["gt_anchors"], cuda), T(z["gt_boxes"], cuda), T(z["gt_valid"], cuda), m,
                                 gt_crowd=T(z["gt_crowd"], cuda), boundary_threshold=bthr,
                                 image_shapes=T(z["gt_shapes"], cuda), box2box_transform=Box2BoxTransform((1., 1., 1., 1.)))
        assert np.array_equal(lab.cpu().numpy(), z[f"gt{c}_labels"])
        assert np.allclose(dl.cpu().numpy(), z[f"gt{c}_deltas"], rtol=1e-5, atol=1e-6)


def test_retinanet_inference_with_synthesised_anchors(cuda, z):
    """In-kernel anchor synthesis (8f #2) + RetinaNet post-processing vs RetinaNetHead.inference."""
    gen = DefaultAnchorGenerator([[32], [64], [128]], [[0.5, 1.0, 2.0]], [int(s) for s in z["ag_strides"]], device=cuda)
    desc = gen.grid_descriptors([tuple(int(v) for v in g) for g in z["ag_grid"]])
    tables = [T(z[f"ag_anchors{l}"], cuda) for l in range(3)]
    head = RetinaNetInference(num_classes=4, topk_candidates=40, score_threshold=0.05, nms_threshold=0.5,
                              max_detections_per_image=25)
    for anchors in (tables, desc):
        res = head.inference([T(z[f"rn_cls{l}"], cuda) for l in range(3)], [T(z[f"rn_reg{l}"], cuda) for l in range(3)], anchors)
        assert np.array_equal(res.get_field("is_valid").cpu().numpy(), z["rn_valid"])
        assert np.array_equal(res.get_field("pred_classes").cpu().numpy(), z["rn_classes"])
        assert np.allclose(res.get_field("scores").cpu().numpy(), z["rn_scores"], rtol=1e-5, atol=1e-7)
        assert np.allclose(res.boxes.cpu().numpy(), z["rn_boxes"], rtol=1e-5, atol=1e-3)


def test_yolo_and_point_nms(cuda, z):
    from detectron2_tensorflow_b200.modeling import YOLOv4Inference, point_nms
    res = YOLOv4Inference(0.3, 0.5, 40).inference(T(z["yo_boxes_in"], cuda), T(z["yo_probs"], cuda))
    assert np.array_equal(res.get_field("is_valid").cpu().numpy(), z["yo_valid"])
    assert np.array_equal(res.get_field("pred_classes").cpu().numpy(), z["yo_classes"])
    assert np.array_equal(res.get_field("scores").cpu().numpy(), z["yo_scores"])
    assert np.array_equal(res.boxes.cpu().numpy(), z["yo_boxes"])
    assert np.array_equal(point_nms(T(z["pn_in"], cuda)).cpu().numpy(), z["pn_out"])


def test_solo_inference_tail(cuda, z):
    from detectron2_tensorflow_b200.modeling import SOLOv2Inference
    head = SOLOv2Inference(0.5, 30, "gaussian", 2.0, 0.05, 12)
    got = head.postprocess(T(z["so_in_logits"], cuda), T(z["so_in_scores"], cuda), T(z["so_in_classes"], cuda),
                           T(z["so_in_strides"], cuda), T(z["so_in_counts"], cuda))
    assert np.array_equal(got["is_valid"].cpu().numpy(), z["so_valid"])
    assert np.array_equal(got["pred_classes"].cpu().numpy(), z["so_classes"])
    assert np.array_equal(got["pred_masks"].cpu().numpy(), z["so_masks"])
    assert np.allclose(got["scores"].cpu().numpy(), z["so_scores"], rtol=1e-5, atol=1e-7)


def test_detector_postprocess(cuda, z):
    """The reference's detector_postprocess (postprocessing.py:9-59) on the dense results of an R-CNN, both mask
    formats: the mirror (from_dense -> scaled boxes -> d2b_paste_masks -> to_dense) is bit-exact."""
    from detectron2_tensorflow_b200.modeling import detector_postprocess
    for fmt, oshape in (("fixed", (90, 120)), ("conventional", (60, 80))):
        bl = BoxList(T(z["dp_boxes"], cuda))
        bl.add_field("pred_masks", T(z["dp_masks"], cuda))
        bl.add_field("is_valid", T(z["dp_valid"], cuda))
        bl.set_tracking("image_shape", T(z["dp_shapes"], cuda))
        res = detector_postprocess(bl, oshape, fmt, image_shapes=T(z["dp_shapes"], cuda))
        assert np.array_equal(res.get_field("pred_masks").cpu().numpy(), z[f"dp_{fmt}_masks"])
        assert np.array_equal(res.boxes.cpu().numpy(), z[f"dp_{fmt}_boxes"])
        assert np.array_equal(res.get_field("is_valid").cpu().numpy(), z[f"dp_{fmt}_valid"])
    with pytest.raises(ValueError):
        detector_postprocess(bl, (60, 80), "bitmap")
