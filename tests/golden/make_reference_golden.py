"""Runs the REFERENCE'S OWN PYTHON for the post-backbone path on the numpy TF shim and freezes its
outputs as tests/golden/reference_python.npz (run in the BUILD container only; /root/reference does
not exist on the GPU box, nothing at test time reads it).

    python tests/golden/make_reference_golden.py

The reference modules are imported unmodified from /root/reference/lib (under the package name
``reflib``; its ``__init__`` files are replaced by empty stub packages because they import the
backbones, data pipeline, ...).  ``tensorflow`` resolves to tests/golden/tf_numpy_shim.py -- see its
docstring for what that does and does not pin.  The FPN maps of case 4 and the SOLOv2 logits of case 14 are
regenerated at load time instead of stored, and case 4's pooled outputs are kept for a sample of rows
(reference_golden.py), so that the file stays under 1 MB.
"""
import importlib
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
REF = "/root/reference/lib"

import reference_golden as golden  # noqa: E402
import tf_numpy_shim as shim  # noqa: E402

t = shim.t


def load_reference():
    tf = shim.install()

    def pkg(name, rel):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF, rel)] if rel is not None else [REF]
        sys.modules[name] = m
        return m
    pkg("reflib", None)
    for sub in ("layers", "structures", "utils", "modeling", "modeling/proposal_generator", "modeling/roi_heads",
                "modeling/single_stage_heads", "data"):
        m = pkg("reflib." + sub.replace("/", "."), sub)
        parent, _, leaf = ("reflib." + sub.replace("/", ".")).rpartition(".")
        setattr(sys.modules[parent], leaf, m)
    imp = importlib.import_module
    tf_utils = imp("reflib.utils.tf_utils")
    tf_utils.set_training_phase(False)
    L = sys.modules["reflib.layers"]
    L.Layer = imp("reflib.layers.base").Layer
    fn = imp("reflib.layers.functional")
    L.crop_and_resize, L.flatten = fn.crop_and_resize, fn.flatten
    L.ROIAlign = imp("reflib.layers.roi_align").ROIAlign
    nms = imp("reflib.layers.nms")
    L.batch_nms, L.matrix_nms = nms.batch_nms, nms.matrix_nms
    # training-only / conv-layer names pulled in by import lines, never called on this path
    for nm in ("smooth_l1_loss", "Linear", "Conv2D", "sigmoid_focal_loss", "iou_loss", "dice_loss", "DeformConv2D",
               "ModulatedDeformConv2D", "GroupNorm", "Upsample", "ConvTranspose2D", "get_norm"):
        setattr(L, nm, None)
    L.resize_images = fn.resize_images
    L.Sequential = imp("reflib.layers.base").Sequential
    L.ShapeSpec = imp("reflib.layers.shape_spec").ShapeSpec
    S = sys.modules["reflib.structures"]
    S.box_list = imp("reflib.structures.box_list")
    S.box_list_ops = imp("reflib.structures.box_list_ops")
    S.mask_ops = imp("reflib.structures.mask_ops")
    mods = dict(tf=tf, box_list=S.box_list, box_list_ops=S.box_list_ops, mask_ops=S.mask_ops, nms=nms, functional=fn,
                roi_align=imp("reflib.layers.roi_align"), matcher=imp("reflib.modeling.matcher"),
                box_regression=imp("reflib.modeling.box_regression"), poolers=imp("reflib.modeling.poolers"),
                rpn_outputs=imp("reflib.modeling.proposal_generator.rpn_outputs"),
                fast_rcnn=imp("reflib.modeling.roi_heads.fast_rcnn"),
                anchor_generator=imp("reflib.modeling.anchor_generator"),
                retinanet=imp("reflib.modeling.single_stage_heads.retinanet"),
                yolo=imp("reflib.modeling.single_stage_heads.yolov4_outputs"),
                solo=imp("reflib.modeling.single_stage_heads.solo_v2"),
                postprocessing=imp("reflib.modeling.postprocessing"),
                mask_head=imp("reflib.modeling.roi_heads.mask_head"))
    return types.SimpleNamespace(**mods)


def rand_boxes(rng, n, H=800, W=1333, smin=8, smax=400):
    cy, cx = rng.uniform(0, H, n), rng.uniform(0, W, n)
    h, w = rng.uniform(smin, smax, n), rng.uniform(smin, smax, n)
    return np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], 1).astype(np.float32)


def main(out_path=None):
    R = load_reference()
    from detectron2_tensorflow_b200.utils import synthetic as syn
    rng = np.random.default_rng(500)
    out = {}
    BoxList, SparseBoxList = R.box_list.BoxList, R.box_list.SparseBoxList

    # ---- 1. pairwise_iou (box_list_ops.py:295-334)
    b1, b2 = rand_boxes(rng, 17), rand_boxes(rng, 400)
    b2[:17] = b1
    b1[3] = 0
    out["iou_b1"], out["iou_b2"] = b1, b2
    out["iou_out"] = np.asarray(R.box_list_ops.pairwise_iou(BoxList(t(b1)), BoxList(t(b2))))

    # ---- 2. Matcher (matcher.py:57-174)
    M, N = 9, 600
    q = rng.random((M, N)).astype(np.float32)
    q[:, ::4] = np.round(q[:, ::4] * 8) / 8
    q[2] = 0
    crowd = (rng.random((3, N)) * (rng.random((3, N)) < 0.02)).astype(np.float32)
    diff = (rng.random((2, N)) * (rng.random((2, N)) < 0.05)).astype(np.float32)
    out["m_q"], out["m_crowd"], out["m_diff"] = q, crowd, diff
    cases = [([0.3, 0.7], [0, -1, 1], True, True, False), ([0.3, 0.7], [0, -1, 1], False, True, True),
             ([0.5], [0, 1], False, False, False), ([0.5], [0, 1], True, True, True)]
    for ci, (th, lab, lq, uc, ud) in enumerate(cases):
        m = R.matcher.Matcher(list(th), list(lab), allow_low_quality_matches=lq)
        mt, ml = m(t(q), t(crowd) if uc else None, t(diff) if ud else None)
        out[f"m{ci}_matches"], out[f"m{ci}_labels"] = np.asarray(mt), np.asarray(ml)
        out[f"m{ci}_cfg"] = np.array([lq, uc, ud], np.int32)
        out[f"m{ci}_th"], out[f"m{ci}_lab"] = np.array(th, np.float32), np.array(lab, np.int32)
    out["m_num_cases"] = np.int32(len(cases))

    # ---- 3. Box2BoxTransform (box_regression.py:38-123); exp/log are numpy's => tolerance in the test
    src, tgt = rand_boxes(rng, 300), rand_boxes(rng, 300)
    deltas = (rng.standard_normal((300, 8)) * 0.5).astype(np.float32)
    deltas[::9, 2] = 30.0
    bt = R.box_regression.Box2BoxTransform(weights=(10., 10., 5., 5.))
    out["bt_src"], out["bt_tgt"], out["bt_deltas"] = src, tgt, deltas
    out["bt_get"] = np.asarray(bt.get_deltas(t(src), t(tgt)))
    out["bt_apply"] = np.asarray(bt.apply_deltas(t(deltas), t(src)))

    # ---- 4. assign_boxes_to_levels + ROIAlign + ROIPooler (poolers.py, roi_align.py, functional.py)
    Nimg, C = 2, 8
    feat_state = golden.pack_state(rng)  # stored instead of the maps: golden.rp_feats(feat_state) draws them again
    feats = [rng.standard_normal((Nimg, h, w, C)).astype(np.float32) for h, w in golden.FEAT_HW]
    boxes, idx = syn.rois(Nimg, 60, seed=501, image_hw=(200, 333))
    boxes[:4] += 40
    out["rp_boxes"], out["rp_idx"], out["rp_feat_state"] = boxes, idx, feat_state
    out["rp_levels"] = np.asarray(R.poolers.assign_boxes_to_levels(BoxList(t(boxes)), 2, 5, 224, 4))
    out["rp_levels56"] = np.asarray(R.poolers.assign_boxes_to_levels(BoxList(t(boxes)), 2, 5, 56, 4))
    rows = out["rp_rows"] = golden.roi_rows(out["rp_levels56"])
    sparse = SparseBoxList(t(idx), BoxList(t(boxes)), [Nimg, 60])
    for ptype, sr, osz in (("ROIAlignV2", 0, 7), ("ROIAlignV2", 2, 7), ("ROIAlign", 0, 14)):
        pooler = R.poolers.ROIPooler((osz, osz), [1 / 4., 1 / 8., 1 / 16., 1 / 32.], sr, ptype,
                                     canonical_box_size=56)  # small canonical size: all 4 levels populated
        out[f"rp_out_{ptype}_{sr}_{osz}"] = np.asarray(pooler([t(f) for f in feats], sparse))[rows]
    bi = idx[:, 0].astype(np.int32)
    ra = R.roi_align.ROIAlign((7, 7), 1 / 8., 0, aligned=True)
    out["ra_single"] = np.asarray(ra(t(feats[1]), t(boxes), t(bi)))[rows]
    out["cr_nopad"] = np.asarray(R.functional.crop_and_resize(t(feats[0]), t(boxes * 0.25), t(bi), [5, 6], aligned=True,
                                                              pad_border=False))[rows]

    # ---- 5. find_top_rpn_proposals (rpn_outputs.py:29-132)
    Nimg = 2
    hwa = [600, 150, 40]
    props = [np.stack([rand_boxes(rng, n, 240, 320, 4, 150) for _ in range(Nimg)]) + rng.normal(0, 30, (Nimg, n, 4)).astype(np.float32)
             for n in hwa]
    props = [p.astype(np.float32) for p in props]
    logits = [np.round(rng.standard_normal((Nimg, n)) * 2 * 16).astype(np.float32) / 16 for n in hwa]  # ties
    shapes = np.array([[240, 320], [200, 300]], np.int32)
    images = types.SimpleNamespace(image_shapes=t(shapes))
    for ci, (pre, post, msl) in enumerate(((100, 60, 0.0), (1000, 50, 12.0), (30, 120, 20.0))):
        res = R.rpn_outputs.find_top_rpn_proposals([t(p) for p in props], [t(l) for l in logits], images, 0.7, pre,
                                                   post, msl)
        out[f"rpn{ci}_boxes"] = np.asarray(res.boxes)
        out[f"rpn{ci}_logits"] = np.asarray(res.get_field("objectness_logits"))
        out[f"rpn{ci}_valid"] = np.asarray(res.get_field("is_valid"))
        out[f"rpn{ci}_cfg"] = np.array([pre, post, msl], np.float32)
    for l in range(3):
        out[f"rpn_props{l}"], out[f"rpn_logits{l}"] = props[l], logits[l]
    out["rpn_shapes"] = shapes
    out["rpn_num_cases"] = np.int32(3)

    # ---- 6. fast_rcnn_inference (fast_rcnn.py:28-187)
    Nimg, Rr, K = 2, 40, 5
    prop, pidx = syn.rois(Nimg, Rr, seed=502, image_hw=(240, 320))
    keep = np.ones(Nimg * Rr, bool)
    keep[[5, 41, 42, 79]] = False  # ragged: different number of ROIs per image
    prop, pidx = prop[keep], pidx[keep]
    d = (rng.standard_normal((prop.shape[0], K * 4)) * 0.3).astype(np.float32)
    import oracle
    pred = oracle.apply_deltas(d, prop, (10., 10., 5., 5.))
    lg = rng.standard_normal((prop.shape[0], K + 1)) * 2
    e = np.exp(lg - lg.max(1, keepdims=True))
    sc = (e / e.sum(1, keepdims=True)).astype(np.float32)
    proposals = SparseBoxList(t(pidx), BoxList(t(prop)), [Nimg, Rr])
    proposals.set_tracking('image_shape', t(shapes))
    out.update(fr_pred=pred, fr_scores=sc, fr_idx=pidx, fr_shapes=shapes, fr_dense=np.array([Nimg, Rr], np.int64))
    for ci, (agn, boxes_in) in enumerate(((False, pred), (True, pred[:, :4].copy()))):
        res, kept = R.fast_rcnn.fast_rcnn_inference(t(boxes_in), t(sc), proposals, 0.05, 0.5, 15, agn)
        out[f"fr{ci}_boxes"], out[f"fr{ci}_scores"] = np.asarray(res.boxes), np.asarray(res.get_field("scores"))
        out[f"fr{ci}_classes"], out[f"fr{ci}_valid"] = (np.asarray(res.get_field("pred_classes")),
                                                        np.asarray(res.get_field("is_valid")))
    out["fr_agnostic_boxes"] = pred[:, :4].copy()

    # ---- 7. matrix_nms / batch_nms (layers/nms.py)
    m, c, s2 = syn.solo_masks(30, hw=(20, 32), num_classes=3, seed=503)
    out.update(mn_masks=np.packbits(m.astype(np.uint8), axis=None), mn_shape=np.array(m.shape), mn_classes=c, mn_scores=s2)
    out["mn_gauss"] = np.asarray(R.nms.matrix_nms(t(m), t(c), t(s2), kernel="gaussian", sigma=2.0))
    out["mn_linear"] = np.asarray(R.nms.matrix_nms(t(m), t(c), t(s2), kernel="linear"))

    # ---- 8. reframe_box_masks_to_image_masks (mask_ops.py:7-56)
    bm = rng.random((6, 14, 14)).astype(np.float32)
    bb = rand_boxes(rng, 6, 60, 80, 8, 50)
    bb[0] = [-5, -5, 20, 30]
    out["pm_masks"], out["pm_boxes"] = bm, bb
    out["pm_out"] = np.asarray(R.mask_ops.reframe_box_masks_to_image_masks(t(bm), t(bb), [60, 80]))

    # ---- 9. RPNOutputs._get_ground_truth (rpn_outputs.py:245-304): pairwise_iou + Matcher + get_deltas
    anchors = [a[::5] for a in syn.rpn_anchors(padded_hw=(96, 128))]
    Nimg, G = 2, 12
    allanch = np.concatenate(anchors, 0)
    gt = np.stack([rand_boxes(rng, G, 96, 128, 8, 90) for _ in range(Nimg)])
    gt[:, 0] = allanch[[7, 300]]
    valid = rng.random((Nimg, G)) < 0.8
    crowd = rng.random((Nimg, G)) < 0.2
    gtb = BoxList(t(gt))
    gtb.add_field("is_valid", t(valid))
    gtb.add_field("gt_is_crowd", t(crowd.astype(np.int64)))
    imgs = types.SimpleNamespace(image_shapes=t(np.array([[96, 128], [90, 120]], np.int32)), num_images=Nimg)
    mt = R.matcher.Matcher([0.3, 0.7], [0, -1, 1], allow_low_quality_matches=True)
    for ci, bthr in enumerate((-1, 0)):
        ro = R.rpn_outputs.RPNOutputs(R.box_regression.Box2BoxTransform(weights=(1., 1., 1., 1.)), mt, 256, 0.5, imgs,
                                      [None] * len(anchors), [None] * len(anchors), [BoxList(t(a)) for a in anchors],
                                      boundary_threshold=bthr, gt_boxes=gtb)
        lab, dl = ro._get_ground_truth()
        out[f"gt{ci}_labels"], out[f"gt{ci}_deltas"] = np.asarray(lab), np.asarray(dl)
    out.update(gt_anchors=allanch, gt_boxes=gt, gt_valid=valid, gt_crowd=crowd, gt_shapes=np.array([[96, 128], [90, 120]], np.int32))

    # ---- 10. DefaultAnchorGenerator (anchor_generator.py:31-162)
    cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(ANCHOR_GENERATOR=types.SimpleNamespace(
        SIZES=[[32], [64], [128]], ASPECT_RATIOS=[[0.5, 1.0, 2.0]])))
    gen = R.anchor_generator.DefaultAnchorGenerator(cfg, [types.SimpleNamespace(stride=s_) for s_ in (4, 8, 16)])
    fmaps = [t(np.zeros((1, h, w, 1), np.float32)) for h, w in ((12, 20), (6, 10), (3, 5))]
    ag = gen(fmaps)
    for l, a in enumerate(ag):
        out[f"ag_anchors{l}"] = np.asarray(a.boxes)
        out[f"ag_cell{l}"] = np.asarray(gen.cell_anchors[l])
    out["ag_grid"] = np.array([[12, 20], [6, 10], [3, 5]], np.int32)
    out["ag_strides"] = np.array([4, 8, 16], np.int32)

    # ---- 11. RetinaNetHead.inference (retinanet.py:285-387); sigmoid/exp are numpy's => tolerance on values
    K, A = 4, 3
    head = types.SimpleNamespace(topk_candidates=40, score_threshold=0.05, num_classes=K, max_detections_per_image=25,
                                 nms_threshold=0.5, box2box_transform=R.box_regression.Box2BoxTransform(weights=(1., 1., 1., 1.)))
    Nimg = 2
    cls = [(rng.standard_normal((Nimg, h, w, A * K)) * 1.5 - 2.0).astype(np.float32) for h, w in ((12, 20), (6, 10), (3, 5))]
    reg = [(rng.standard_normal((Nimg, h, w, A * 4)) * 0.3).astype(np.float32) for h, w in ((12, 20), (6, 10), (3, 5))]
    res = R.retinanet.RetinaNetHead.inference(head, [t(c_) for c_ in cls], [t(r_) for r_ in reg], ag)
    for l in range(3):
        out[f"rn_cls{l}"], out[f"rn_reg{l}"] = cls[l].reshape(Nimg, -1, K), reg[l].reshape(Nimg, -1, 4)
    out["rn_boxes"], out["rn_scores"] = np.asarray(res.boxes), np.asarray(res.get_field("scores"))
    out["rn_classes"], out["rn_valid"] = np.asarray(res.get_field("pred_classes")), np.asarray(res.get_field("is_valid"))

    # ---- 12. YOLOv4Outputs.inference (yolov4_outputs.py:331-390)
    Nimg, nb, K = 2, 300, 6
    yb = np.stack([rand_boxes(rng, nb, 240, 320, 8, 120) for _ in range(Nimg)])
    yb[:, 100:200] = yb[:, :100] + rng.normal(0, 3, (Nimg, 100, 4)).astype(np.float32)  # near duplicates
    yp = (rng.random((Nimg, nb, K)) ** 4).astype(np.float32)
    yp[:, ::7] = np.round(yp[:, ::7] * 4) / 4  # ties across classes (first argmax) and across boxes
    yself = types.SimpleNamespace(score_threshold=0.3, nms_threshold=0.5, post_nms_topk=40,
                                  _get_predictions=lambda: (t(yb), None, t(yp)))
    res = R.yolo.YOLOV4Outputs.inference(yself)
    out.update(yo_boxes_in=yb, yo_probs=yp, yo_boxes=np.asarray(res.boxes), yo_scores=np.asarray(res.get_field("scores")),
               yo_classes=np.asarray(res.get_field("pred_classes")), yo_valid=np.asarray(res.get_field("is_valid")))

    # ---- 13. point_nms (solo_v2.py:29-40)
    pn = np.round(rng.standard_normal((2, 9, 11, 8)) * 2).astype(np.float32) / 2  # plateaus and negatives
    out["pn_in"], out["pn_out"] = pn, np.asarray(R.solo.point_nms(t(pn)))

    # ---- 14. MaskKernelBranch.inference (solo_v2.py:476-612) with image_shape == mask-feature size (resize = identity).
    # The op under test starts after the dynamic conv, so the generator repeats the candidate selection (:481-497)
    # and the 1x1 conv (:499-511, golden.so_logits at load time) to record the op's inputs; everything after is the
    # reference's code.
    Nimg, K, E, Hm, Wm = 2, 3, 8, 24, 32
    grids, sstr = [6, 4], [8, 16]
    shead = types.SimpleNamespace(score_threshold=0.3, num_grids=grids, strides=sstr, mask_kernel_size=1,
                                  mask_feature_out_dims=E, mask_threshold=0.5, pre_nms_topk=30, nms_kernel="gaussian",
                                  nms_sigma=2.0, update_score_threshold=0.05, max_detections_per_image=12)
    probs = [rng.random((Nimg, g_, g_, K)).astype(np.float32) ** 2 for g_ in grids]
    kerns = [(rng.standard_normal((Nimg, g_, g_, E)) * 0.8).astype(np.float32) for g_ in grids]
    yy_, xx_ = np.mgrid[0:Hm, 0:Wm].astype(np.float32)
    mfeat = np.stack([np.stack([np.sin(yy_ * rng.uniform(0.1, 0.5) + xx_ * rng.uniform(0.1, 0.5) + rng.uniform(0, 6))
                                for _ in range(E)], -1) for _ in range(Nimg)]).astype(np.float32)
    res = R.solo.MaskKernelBranch.inference(shead, [t(p_) for p_ in probs], [t(k_) for k_ in kerns], t(mfeat), [Hm, Wm])
    out.update(so_masks=np.asarray(res.get_field("pred_masks")), so_classes=np.asarray(res.get_field("pred_classes")),
               so_scores=np.asarray(res.get_field("scores")), so_valid=np.asarray(res.get_field("is_valid")))
    flat_p = np.concatenate([p_.reshape(Nimg, -1, K) for p_ in probs], 1)
    flat_k = np.concatenate([k_.reshape(Nimg, -1, E) for k_ in kerns], 1)
    cell_stride = np.concatenate([np.full(g_ * g_, s_, np.float32) for g_, s_ in zip(grids, sstr)])
    ncap = int(max((flat_p[i] > 0.3).sum() for i in range(Nimg)))
    so_sc, so_cl, so_st = np.zeros((Nimg, ncap), np.float32), np.zeros((Nimg, ncap), np.int64), np.ones((Nimg, ncap), np.float32)
    so_cnt = np.zeros(Nimg, np.int32)
    so_kern = np.zeros((Nimg, ncap, E), np.float32)  # the gathered pred_kernels (:486): input of the fused dynamic conv
    for i in range(Nimg):
        keep = np.argwhere(flat_p[i] > 0.3)
        c_ = keep.shape[0]
        so_cnt[i] = c_
        so_sc[i, :c_] = flat_p[i][keep[:, 0], keep[:, 1]]
        so_cl[i, :c_] = keep[:, 1]
        so_st[i, :c_] = cell_stride[keep[:, 0]]
        so_kern[i, :c_] = flat_k[i][keep[:, 0]]
    for li, (p_, k_) in enumerate(zip(probs, kerns)):  # the raw arguments of MaskKernelBranch.inference
        out[f"so_raw_probs_{li}"], out[f"so_raw_kernels_{li}"] = p_, k_
    out.update(so_in_scores=so_sc, so_in_classes=so_cl, so_in_strides=so_st, so_in_counts=so_cnt,
               so_in_mask_features=mfeat, so_in_kernels=so_kern)

    # ---- 15. the same inference with image_shape != mask-feature size: resize_images (functional.py:9-36 takes the
    # tf.compat.v2.image.resize branch on the shim -> half-pixel centres) + threshold + boxes from masks (:599-627)
    Hi, Wi = 95, 130
    res2 = R.solo.MaskKernelBranch.inference(shead, [t(p_) for p_ in probs], [t(k_) for k_ in kerns], t(mfeat), [Hi, Wi])
    out.update(so2_masks=np.asarray(res2.get_field("pred_masks")).astype(np.uint8), so2_boxes=np.asarray(res2.boxes),
               so2_image_shape=np.array([Hi, Wi], np.int32))

    # ---- 16. detector_postprocess (postprocessing.py:9-59): dense results -> from_dense -> (scaled) boxes -> paste
    dp_boxes = np.stack([rand_boxes(rng, 5, 60, 80, 8, 40) for _ in range(2)])
    dp_masks = rng.random((2, 5, 14, 14)).astype(np.float32)
    dp_valid = np.array([[1, 1, 0, 1, 1], [1, 0, 0, 1, 0]], bool)
    dp_shapes = np.array([[60, 80], [50, 70]], np.int32)
    out.update(dp_boxes=dp_boxes, dp_masks=dp_masks, dp_valid=dp_valid, dp_shapes=dp_shapes)
    for fmt, oshape in (("fixed", [90, 120]), ("conventional", [60, 80])):
        bl = R.box_list.BoxList(t(dp_boxes))
        bl.add_field("pred_masks", t(dp_masks))
        bl.add_field("is_valid", t(dp_valid))
        bl.set_tracking("image_shape", t(dp_shapes))
        res = R.postprocessing.detector_postprocess(bl, oshape, fmt, image_shapes=t(dp_shapes))
        out[f"dp_{fmt}_masks"] = np.asarray(res.get_field("pred_masks"))
        out[f"dp_{fmt}_boxes"] = np.asarray(res.boxes)
        out[f"dp_{fmt}_valid"] = np.asarray(res.get_field("is_valid"))

    # ---- 17. pairwise_iou with iou_type giou / diou / ciou (box_list_ops.py:335-371)
    ia, ib = rand_boxes(rng, 40, 200, 300, 4, 150), rand_boxes(rng, 25, 200, 300, 4, 150)
    ib[:5] = ia[:5]                      # identical boxes
    ib[5] = [10, 10, 10, 40]             # zero height
    ia[6] = [300, 300, 320, 330]         # disjoint from everything
    out["pi_a"], out["pi_b"] = ia, ib
    for ty in ("iou", "giou", "diou", "ciou"):
        out[f"pi_{ty}"] = np.asarray(R.box_list_ops.pairwise_iou(R.box_list.BoxList(t(ia)), R.box_list.BoxList(t(ib)), ty))

    # ---- 18. mask_rcnn_inference (mask_head.py:71-103): NHWC logits -> class channel -> sigmoid
    ml = (rng.standard_normal((7, 6, 6, 5)) * 3).astype(np.float32)
    mc = rng.integers(0, 5, 7).astype(np.int64)
    inst = R.box_list.SparseBoxList(t(np.stack([np.zeros(7, np.int64), np.arange(7)], 1)),
                                    R.box_list.BoxList(t(rand_boxes(rng, 7, 60, 80, 8, 40))), [1, 7])
    inst.data.add_field("pred_classes", t(mc))
    R.mask_head.mask_rcnn_inference(t(ml), inst)
    out.update(mi_logits=ml, mi_classes=mc, mi_out=np.asarray(inst.data.get_field("pred_masks")))

    out_path = out_path or os.path.join(HERE, "reference_python.npz")
    np.savez_compressed(out_path, **out)
    print(os.path.basename(out_path) + ":", len(out), "arrays,", os.path.getsize(out_path) // 1024, "KiB")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
