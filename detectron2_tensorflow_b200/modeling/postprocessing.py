"""Drop-in for `detector_postprocess` of lib/modeling/postprocessing.py (:9-59): the last step of
`GeneralizedRCNN.inference` (rcnn.py:124-133) -- paste the ROI-head masks into image-size masks.  Beyond the
reference: `detector_postprocess_rle` (a whole batch's masks as COCO run-length strings, each image at its own output
size, in one sync-free call) and `coco_results` (the COCO results list of the batch)."""
import numpy as np
import torch

from .. import _native as nv
from ..structures.box_list import SparseBoxList
from ..structures.mask_ops import _output_shapes, _paste_params, reframe_box_masks_to_image_masks, rle_call


def _scale_boxes(boxes, scales):
    """boxes [..., 4] yxyx times fp32 (sy, sx) scales [..., 2], one fp32 multiply per coordinate (:36-43)."""
    return torch.stack([scales[..., 0] * boxes[..., 0], scales[..., 1] * boxes[..., 1],
                        scales[..., 0] * boxes[..., 2], scales[..., 1] * boxes[..., 3]], -1)


def detector_postprocess(results, output_shape, mask_format, image_shapes=None, mask_threshold=0.5, scope=None):
    """Image-size masks for the detections of an R-CNN (arguments and return structure of the reference function).

    results: dense BoxList [N, R] with `pred_masks` [N, R, mh, mw], `is_valid` and the `image_shape` tracking.
    mask_format "conventional": masks are pasted at the boxes as they are; "fixed": at the boxes scaled by
    output_shape / image_shape (:36-43 -- only the pasting boxes are scaled, `results.boxes` stay, as in the reference;
    the int / int division there is TF's true division, i.e. float64, cast to fp32 by `box_list_ops.scale`);
    "raw": `pred_masks > mask_threshold` (the reference's branch reads an undefined name, :51; this is its intent).
    Returns the dense BoxList with `pred_masks` uint8 [N, R, H, W]."""
    if not results.has_field("pred_masks"):
        return results
    if mask_format in ("conventional", "fixed"):
        results = SparseBoxList.from_dense(results)
        box_masks = results.data.get_field("pred_masks")
        if mask_format == "fixed":
            assert image_shapes is not None, "Detection results should carry the true input shape."
            image_shapes = results.get_tracking('image_shape')
            out = torch.as_tensor([float(output_shape[0]), float(output_shape[1])], dtype=torch.float64,
                                  device=image_shapes.device)
            scales = (out[None] / image_shapes.to(torch.float64))[results.indices[:, 0]].to(torch.float32)
            boxes = _scale_boxes(results.data.boxes, scales)
        else:
            boxes = results.data.boxes
        pred_masks = reframe_box_masks_to_image_masks(box_masks, boxes, output_shape, mask_threshold)
        results.data.set_field("pred_masks", pred_masks)
        results = results.to_dense()
    elif mask_format == "raw":
        pred_masks = results.get_field("pred_masks")
        results.set_field("pred_masks", (pred_masks > mask_threshold).to(torch.uint8))
    else:
        raise ValueError(f"mask format '{mask_format}' is not recognized.")
    return results


def detector_postprocess_rle(results, output_shapes, mask_threshold=0.5, mask_format="fixed", capacity=None):
    """The masks `detector_postprocess` pastes, for a whole batch at once and each image at its own output size, as
    COCO run-length strings encoded on the GPU (d2b_paste_masks in its batched mode); no image plane is written.

    results: dense BoxList [N, R] with `pred_masks` [N, R, mh, mw], `is_valid` and the `image_shape` tracking.
    output_shapes: [N, 2] (h, w) of each image's masks -- a host sequence / array / tensor (checked here), or a CUDA
    int32 tensor, which is how a CUDA graph is given sizes it can replay with.
    mask_format "fixed": boxes scaled by output_shapes[n] / image_shape[n] as `detector_postprocess` does it;
    "conventional": the boxes as they are.
    capacity: None sizes the strings exactly (one host sync); an int issues no sync and can be captured in a CUDA graph
    (the contract of `reframe_box_masks_to_rle`).

    Returns ((chars uint8 [capacity], offsets int64 [N * R + 1]), boxes fp32 [N, R, 4]): slot m = n * R + r is
    chars[offsets[m]:offsets[m + 1]], byte-identical to pycocotools.mask.encode of the mask `detector_postprocess`
    pastes for it at output_shapes[n]; a slot that is not valid has an empty string.  `boxes` are the boxes the masks
    were pasted at (the scaled ones in "fixed")."""
    if mask_format not in ("fixed", "conventional"):
        raise ValueError(f"mask format '{mask_format}' has no pasted masks to encode.")
    pm = results.get_field("pred_masks")
    N, R, mh, mw = pm.shape
    shapes = _output_shapes(output_shapes, N)
    dev = nv.device_of(pm, results.boxes, shapes)
    shapes = nv.to_device(shapes, dev)
    m = nv.to_device(pm, dev, torch.float32).reshape(N * R, mh, mw)
    b = nv.to_device(results.boxes, dev, torch.float32).reshape(N, R, 4)
    valid = nv.to_device(results.get_field("is_valid"), dev, torch.uint8).reshape(N * R)
    p = _paste_params(m, b, 0, 0, mask_threshold)
    p.num_images, p.dets_per_image = N, R
    p.output_shapes, p.valid = shapes.data_ptr(), valid.data_ptr()
    pasted = b
    if mask_format == "fixed":  # the kernel scales the boxes itself; `pasted` is what it pastes at, for the caller
        image_shapes = nv.to_device(results.get_tracking("image_shape"), dev, torch.int32).reshape(N, 2)
        p.input_shapes = image_shapes.data_ptr()
        scales = (shapes.to(torch.float64) / image_shapes.to(torch.float64)).to(torch.float32)
        pasted = _scale_boxes(b, scales[:, None, :])

    def run(chars, cap, offsets, again):
        p.out_rle, p.rle_capacity, p.out_rle_offsets = chars, cap, offsets
        nv.call("paste_masks", p, dev)
    return rle_call(run, N * R, dev, capacity), pasted


def coco_results(results, rle, boxes, output_shapes, image_ids, category_ids):
    """The COCO results list of a batch: one dict per detection,
    {"image_id", "category_id", "bbox": [x, y, w, h], "score", "segmentation": {"size": [h_n, w_n], "counts"}},
    image by image in slot order.

    results: the dense BoxList [N, R] given to `detector_postprocess_rle` (`scores`, `pred_classes`); rle and boxes: its
    return values; output_shapes: the same [N, 2] sizes; image_ids: the N dataset image ids; category_ids: the dataset
    category id of each contiguous class id (a sequence or a dict).  The slots with a string are the detections; `bbox`
    is the box their mask was pasted at.  One device-to-host copy brings the small tensors and the strings over."""
    chars, offsets = rle
    N, R = boxes.shape[0], boxes.shape[1]
    M = N * R
    parts = [offsets.reshape(-1), results.get_field("pred_classes").to(torch.int64).reshape(-1),
             boxes.to(torch.float32).reshape(-1), results.get_field("scores").to(torch.float32).reshape(-1)]
    packed = torch.cat([t.to(offsets.device).contiguous().view(torch.uint8) for t in parts] + [chars.reshape(-1)])
    buf = nv.to_host(packed).numpy()
    at = 0

    def take(dtype, n):
        nonlocal at
        a = np.frombuffer(buf, dtype, n, at)
        at += a.nbytes
        return a
    off, cls, bx, sc = take(np.int64, M + 1), take(np.int64, M), take(np.float32, 4 * M).reshape(M, 4), take(np.float32, M)
    data = buf[at:].tobytes()
    if int(off[-1]) > len(data):
        raise ValueError(f"the RLE strings need {int(off[-1])} bytes but the buffer holds {len(data)}: "
                         f"call again with capacity >= {int(off[-1])}")
    sizes = np.asarray(output_shapes.cpu() if isinstance(output_shapes, torch.Tensor) else output_shapes,
                       np.int64).reshape(N, 2)
    out = []
    for i in np.flatnonzero(off[1:] > off[:-1]).tolist():
        n = i // R
        y0, x0, y1, x1 = bx[i]
        out.append({"image_id": image_ids[n], "category_id": category_ids[int(cls[i])],
                    "bbox": [float(x0), float(y0), float(x1 - x0), float(y1 - y0)], "score": float(sc[i]),
                    "segmentation": {"size": [int(sizes[n, 0]), int(sizes[n, 1])], "counts": data[off[i]:off[i + 1]]}})
    return out
