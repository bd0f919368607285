"""Drop-in for `point_nms` of lib/modeling/single_stage_heads/solo_v2.py (:29-40)."""
import torch

from ... import _native as nv
from ...structures.mask_ops import rle_call

__all__ = ["point_nms", "solo_mask_encode", "solo_dynamic_masks", "solo_upsample_masks", "SOLOv2Inference"]


def point_nms(inputs, kernel_size=2, scope=None):
    """NHWC category scores: a value survives iff it equals the max of its 2x2 (self, up, left, up-left) window."""
    assert kernel_size == 2
    host = not inputs.is_cuda
    dev = nv.device_of(inputs)
    x = nv.to_device(inputs, dev, torch.float32)
    assert x.dim() == 4
    out = torch.empty_like(x)
    p = nv.PointNmsParams()
    p.scores, p.out = x.data_ptr(), out.data_ptr()
    p.num_images, p.height, p.width, p.channels = x.shape
    nv.call("point_nms", p, dev)
    return nv.to_host(out) if host else out


def solo_mask_encode(mask_logits, mask_threshold=0.5, counts=None):
    """The mask stage of SOLOv2Head.inference (solo_v2.py:513-517, 530-533) in one streaming pass.

    mask_logits [n, H, W] (or [B, n, H, W]): the dynamic-conv output BEFORE the sigmoid.
    Returns (packed_masks int64 [.., n, ceil(H*W/64)], sum_masks fp32 [.., n], score_sums fp32 [.., n]) where
    packed bit p of word w is `sigmoid(logit) > mask_threshold` of pixel 64*w+p, sum_masks = reduce_sum(pred_masks)
    and score_sums = reduce_sum(pred_mask_scores * pred_masks); mask_scoring (:531-533) = score_sums / sum_masks.
    Feed `packed_masks` to `layers.matrix_nms(None, ..., packed_masks=..., mask_hw=H*W)`.
    """
    host = not mask_logits.is_cuda
    dev = nv.device_of(mask_logits)
    x = nv.to_device(mask_logits, dev, torch.float32)
    batched = x.dim() == 4
    if not batched:
        x = x[None]
    B, n, H, W = x.shape
    hw = H * W
    Wd = (hw + 63) // 64
    packed = torch.empty((B, n, Wd), dtype=torch.int64, device=dev)
    sums = torch.empty((B, n), dtype=torch.float32, device=dev)
    ssum = torch.empty((B, n), dtype=torch.float32, device=dev)
    cnt = None if counts is None else nv.to_device(counts, dev, torch.int32)
    p = nv.SoloMaskEncodeParams()
    p.mask_logits, p.counts = x.data_ptr(), nv.ptr(cnt)
    p.batch, p.n, p.hw = B, n, hw
    p.mask_threshold = float(mask_threshold)
    p.packed_masks, p.sum_masks, p.score_sums = packed.data_ptr(), sums.data_ptr(), ssum.data_ptr()
    nv.call("solo_mask_encode", p, dev)
    outs = (packed, sums, ssum)
    if not batched:
        outs = tuple(o[0] for o in outs)
    return tuple(nv.to_host(o) for o in outs) if host else outs


def solo_dynamic_masks(mask_features, mask_kernels, mask_threshold=0.5, counts=None, return_logits=False):
    """Dynamic mask generation + mask stage of SOLOv2Head.inference (solo_v2.py:499-517, 530-533) in ONE kernel.

    mask_features [B, H, W, E] (NHWC, the mask branch output); mask_kernels [B, n, E] (the `pred_kernels` rows of the
    candidates that passed the score threshold, :486).  The 1x1 conv is a per-image GEMM on the tcgen05 tensor cores
    (3 x tf32 = fp32-accurate); its epilogue thresholds the sigmoid and emits bit-packed masks, so the [B, n, H, W]
    logits are never written unless `return_logits` asks for them.
    Returns (packed_masks int64 [B, n, ceil(HW/64)], sum_masks [B, n], score_sums [B, n][, logits [B, n, H, W]]).
    """
    host = not mask_features.is_cuda
    dev = nv.device_of(mask_features)
    f = nv.to_device(mask_features, dev, torch.float32)
    k = nv.to_device(mask_kernels, dev, torch.float32)
    assert f.dim() == 4 and k.dim() == 3 and k.shape[0] == f.shape[0] and k.shape[2] == f.shape[3]
    B, H, W, E = f.shape
    n = k.shape[1]
    hw = H * W
    Wd = (hw + 63) // 64
    packed = torch.empty((B, n, Wd), dtype=torch.int64, device=dev)
    sums = torch.empty((B, n), dtype=torch.float32, device=dev)
    ssum = torch.empty((B, n), dtype=torch.float32, device=dev)
    logits = torch.zeros((B, n, H, W), dtype=torch.float32, device=dev) if return_logits else None
    cnt = None if counts is None else nv.to_device(counts, dev, torch.int32)
    p = nv.SoloDynamicMasksParams()
    p.mask_features, p.mask_kernels, p.counts = f.data_ptr(), k.data_ptr(), nv.ptr(cnt)
    p.batch, p.n, p.channels, p.hw = B, n, E, hw
    p.mask_threshold = float(mask_threshold)
    p.packed_masks, p.sum_masks, p.score_sums = packed.data_ptr(), sums.data_ptr(), ssum.data_ptr()
    p.mask_logits = nv.ptr(logits)
    nv.call("solo_dynamic_masks", p, dev)
    outs = (packed, sums, ssum) + ((logits,) if return_logits else ())
    return tuple(nv.to_host(o) for o in outs) if host else outs


def solo_upsample_masks(packed_masks, mask_hw, image_shape, mask_threshold=0.5, align_corners=False, return_masks=True,
                        return_packed=False, return_rle=False, rle_capacity=None):
    """The last stage of `MaskKernelBranch.inference` (solo_v2.py:599-627): bilinear `resize_images` of the kept masks
    to `image_shape`, threshold, boxes from masks -- from the bit-packed masks of `SOLOv2Inference.postprocess`.

    packed_masks int64 [B, D, ceil(h*w/64)], mask_hw = (h, w), image_shape = (H, W).
    align_corners=False is what `resize_images` does when `tf.compat.v2.image.resize` exists (functional.py:21-24: the
    align_corners kwarg is dropped, half-pixel centres); True is the TF 1.13 fall-back (:26-35).
    Returns dict(pred_masks uint8 [B, D, H, W] or None, packed_masks int64 [B, D, ceil(H*W/64)] or None,
    boxes fp32 [B, D, 4] as (ymin, xmin, ymax, xmax)).
    return_rle=True adds rle = (chars uint8 [capacity], offsets int64 [B*D + 1]) on the device: the COCO run-length
    strings of the B*D image masks, encoded on the GPU (see `structures.mask_ops.reframe_box_masks_to_rle` for
    rle_capacity and `rle_to_coco`); return_masks=False then skips the [B, D, H, W] planes altogether."""
    host = not packed_masks.is_cuda
    dev = nv.device_of(packed_masks)
    pk = nv.to_device(packed_masks, dev, torch.int64)
    assert pk.dim() == 3
    B, D, Wd = pk.shape
    h, w = int(mask_hw[0]), int(mask_hw[1])
    H, W = int(image_shape[0]), int(image_shape[1])
    assert Wd == (h * w + 63) // 64
    masks = torch.empty((B, D, H, W), dtype=torch.uint8, device=dev) if return_masks else None
    packed = torch.empty((B, D, (H * W + 63) // 64), dtype=torch.int64, device=dev) if return_packed else None
    boxes = torch.empty((B, D, 4), dtype=torch.float32, device=dev)
    p = nv.SoloUpsampleParams()
    p.packed_masks = pk.data_ptr()
    p.batch, p.num_dets, p.mask_h, p.mask_w, p.image_h, p.image_w = B, D, h, w, H, W
    p.align_corners = 1 if align_corners else 0
    p.mask_threshold = float(mask_threshold)
    p.out_masks, p.out_packed_masks, p.out_boxes = nv.ptr(masks), nv.ptr(packed), boxes.data_ptr()
    if not return_rle:
        nv.call("solo_upsample", p, dev)
        out = dict(pred_masks=masks, packed_masks=packed, boxes=boxes)
        if host:
            out = {k: (None if v is None else nv.to_host(v)) for k, v in out.items()}
        return out
    spare_boxes = torch.empty_like(boxes) if rle_capacity is None else None

    def run(chars, cap, offsets, again):
        if again:  # the exactly sized call after the sizing call: the planes and boxes are already written
            p.out_masks = p.out_packed_masks = None
            p.out_boxes = spare_boxes.data_ptr()
        p.out_rle, p.rle_capacity, p.out_rle_offsets = chars, cap, offsets
        nv.call("solo_upsample", p, dev)
    out = dict(pred_masks=masks, packed_masks=packed, boxes=boxes, rle=rle_call(run, B * D, dev, rle_capacity))
    if host:
        out = {k: (v if v is None or k == "rle" else nv.to_host(v)) for k, v in out.items()}
    return out


class SOLOv2Inference(object):
    """The tail of `SOLOv2Head.inference` after the dynamic convolution (solo_v2.py:507-558), batched: mask stage,
    `sum_masks > strides` filter, mask scoring, top-k, Matrix-NMS on bit-packed masks, score filter, pad / clip.
    Attributes mirror the ones `SOLOv2Head.__init__` reads from cfg (:140-149)."""

    def __init__(self, mask_threshold=0.5, pre_nms_topk=500, nms_kernel="gaussian", nms_sigma=2.0,
                 update_score_threshold=0.05, max_detections_per_image=100, score_threshold=0.1,
                 num_grids=(40, 36, 24, 16, 12), strides=(8, 8, 16, 32, 32), max_candidates=2048, align_corners=False):
        if nms_kernel not in ("gaussian", "linear"):
            raise NotImplementedError(f"NMS kernel {nms_kernel} not implemented yet.")
        self.score_threshold = score_threshold
        self.num_grids = tuple(num_grids)
        self.strides = tuple(strides)
        self.max_candidates = int(max_candidates)  # static row count of the candidate list (the reference's is dynamic)
        self.align_corners = align_corners         # which TF resize `resize_images` resolved to (functional.py:21-35)
        self.mask_threshold = mask_threshold
        self.pre_nms_topk = pre_nms_topk
        self.nms_kernel = nms_kernel
        self.nms_sigma = nms_sigma
        self.update_score_threshold = update_score_threshold
        self.max_detections_per_image = max_detections_per_image

    def postprocess(self, mask_logits, scores, classes, strides, counts=None, return_masks=True, mask_features=None,
                    mask_kernels=None):
        """mask_logits [B, n, H, W]: conv output of each image's candidates (those with score > score_threshold, in
        `tf.where` order; rows >= counts[b] are padding); scores / classes / strides [B, n].
        With mask_logits=None the masks come from the fused dynamic conv instead (`solo_dynamic_masks`):
        mask_features [B, H, W, E] and mask_kernels [B, n, E].
        Returns dict(pred_masks fp32 0/1 [B, D, H, W] (or None), packed_masks int64 [B, D, ceil(HW/64)],
        pred_classes int64 [B, D], scores [B, D], is_valid [B, D], num [B])."""
        src = mask_logits if mask_logits is not None else mask_features
        host = not src.is_cuda
        dev = nv.device_of(src)
        feat = kern = x = None
        if mask_logits is not None:
            x = nv.to_device(mask_logits, dev, torch.float32)
            assert x.dim() == 4
            B, n, H, W = x.shape
        else:
            feat = nv.to_device(mask_features, dev, torch.float32)
            kern = nv.to_device(mask_kernels, dev, torch.float32)
            assert feat.dim() == 4 and kern.dim() == 3 and kern.shape[0] == feat.shape[0] and kern.shape[2] == feat.shape[3]
            B, H, W, _ = feat.shape
            n = kern.shape[1]
        hw = H * W
        D = int(self.max_detections_per_image)
        sc = nv.to_device(scores, dev, torch.float32).reshape(B, n)
        cl = nv.to_device(classes, dev, torch.int64).reshape(B, n)
        stv = nv.to_device(strides, dev, torch.float32).reshape(B, n)
        cnt = None if counts is None else nv.to_device(counts, dev, torch.int32)
        Wd = (hw + 63) // 64
        masks = torch.empty((B, D, H, W), dtype=torch.float32, device=dev) if return_masks else None
        packed = torch.empty((B, D, Wd), dtype=torch.int64, device=dev)
        oc = torch.empty((B, D), dtype=torch.int64, device=dev)
        os_ = torch.empty((B, D), dtype=torch.float32, device=dev)
        ov = torch.empty((B, D), dtype=torch.bool, device=dev)
        num = torch.empty(B, dtype=torch.int32, device=dev)
        p = nv.SoloPostprocessParams()
        p.mask_logits, p.scores, p.classes, p.strides = nv.ptr(x), sc.data_ptr(), cl.data_ptr(), stv.data_ptr()
        p.mask_features, p.mask_kernels = nv.ptr(feat), nv.ptr(kern)
        p.channels = 0 if feat is None else int(feat.shape[3])
        p.counts = nv.ptr(cnt)
        p.batch, p.n, p.hw = B, n, hw
        p.mask_threshold, p.pre_nms_topk = float(self.mask_threshold), int(self.pre_nms_topk)
        p.kernel = nv.MNMS_GAUSSIAN if self.nms_kernel == "gaussian" else nv.MNMS_LINEAR
        p.sigma, p.update_score_threshold, p.max_detections = float(self.nms_sigma), float(self.update_score_threshold), D
        p.out_masks, p.out_packed_masks = nv.ptr(masks), packed.data_ptr()
        p.out_classes, p.out_scores, p.out_valid, p.out_num = oc.data_ptr(), os_.data_ptr(), ov.data_ptr(), num.data_ptr()
        nv.call("solo_postprocess", p, dev)
        out = dict(pred_masks=masks, packed_masks=packed, pred_classes=oc, scores=os_, is_valid=ov, num=num)
        if host:
            out = {k: (None if v is None else nv.to_host(v)) for k, v in out.items()}
        return out

    def select_candidates(self, pred_scores, pred_kernels):
        """solo_v2.py:481-497 batched: pred_scores [B, G, K], pred_kernels [B, G, E] (levels concatenated) ->
        dict(scores, classes, strides [B, n], kernels [B, n, E], counts [B], total [B]) with n = max_candidates, rows
        in `tf.where` order; total > counts means the static cap dropped candidates."""
        dev = nv.device_of(pred_scores)
        sc = nv.to_device(pred_scores, dev, torch.float32)
        kn = nv.to_device(pred_kernels, dev, torch.float32)
        B, G, K = sc.shape
        E = kn.shape[2]
        assert kn.shape[:2] == (B, G) and G == sum(g * g for g in self.num_grids)
        cell = torch.cat([torch.full((g * g,), float(s_), dtype=torch.float32) for g, s_ in zip(self.num_grids, self.strides)])
        cell = cell.to(dev)
        n = self.max_candidates
        o_sc = torch.empty((B, n), dtype=torch.float32, device=dev)
        o_cl = torch.empty((B, n), dtype=torch.int64, device=dev)
        o_st = torch.empty((B, n), dtype=torch.float32, device=dev)
        o_kn = torch.empty((B, n, E), dtype=torch.float32, device=dev)
        cnt = torch.empty(B, dtype=torch.int32, device=dev)
        tot = torch.empty(B, dtype=torch.int32, device=dev)
        p = nv.SoloSelectParams()
        p.scores, p.kernels, p.cell_strides = sc.data_ptr(), kn.data_ptr(), cell.data_ptr()
        p.batch, p.num_cells, p.num_classes, p.channels = B, G, K, E
        p.score_threshold, p.max_candidates = float(self.score_threshold), n
        p.out_scores, p.out_classes, p.out_strides, p.out_kernels = o_sc.data_ptr(), o_cl.data_ptr(), o_st.data_ptr(), o_kn.data_ptr()
        p.out_counts, p.out_total = cnt.data_ptr(), tot.data_ptr()
        nv.call("solo_select", p, dev)
        return dict(scores=o_sc, classes=o_cl, strides=o_st, kernels=o_kn, counts=cnt, total=tot)

    def inference(self, pred_probs, pred_kernels, pred_mask_features, image_shape):
        """Drop-in for `MaskKernelBranch.inference(pred_probs, pred_kernels, pred_mask_features, image_shape)`
        (solo_v2.py:476-627): per-level lists of [B, g, g, K] probabilities and [B, g, g, E] kernels, mask features
        [B, H, W, E], image_shape (H_img, W_img).  Candidate selection -> dynamic conv + mask stage (tensor cores) ->
        filter / mask scoring / top-k / Matrix-NMS / score filter / pad -> image-size masks + boxes from masks.
        Returns dict(pred_classes int64 [B, D], pred_masks uint8 [B, D, H_img, W_img], scores [B, D], is_valid [B, D],
        boxes fp32 [B, D, 4], num [B], num_candidates [B])."""
        host = not pred_mask_features.is_cuda
        dev = nv.device_of(pred_mask_features)
        feat = nv.to_device(pred_mask_features, dev, torch.float32)
        B = feat.shape[0]
        sc = torch.cat([nv.to_device(p_, dev, torch.float32).reshape(B, -1, p_.shape[-1]) for p_ in pred_probs], 1)
        kn = torch.cat([nv.to_device(k_, dev, torch.float32).reshape(B, -1, k_.shape[-1]) for k_ in pred_kernels], 1)
        cand = self.select_candidates(sc.contiguous(), kn.contiguous())
        tail = self.postprocess(None, cand["scores"], cand["classes"], cand["strides"], cand["counts"], return_masks=False,
                                mask_features=feat, mask_kernels=cand["kernels"])
        up = solo_upsample_masks(tail["packed_masks"], feat.shape[1:3], image_shape, self.mask_threshold, self.align_corners)
        out = dict(pred_classes=tail["pred_classes"], pred_masks=up["pred_masks"], scores=tail["scores"],
                   is_valid=tail["is_valid"], boxes=up["boxes"], num=tail["num"], num_candidates=cand["total"])
        if host:
            out = {k: nv.to_host(v) for k, v in out.items()}
        return out
