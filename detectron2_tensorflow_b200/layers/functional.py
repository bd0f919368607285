"""Drop-in for the hot part of lib/layers/functional.py: `crop_and_resize` (:100-166)."""
import torch

from .. import _native as nv


def _roi_align_call(features, scales, boxes, batch_idx, bidx_stride, output_size, sampling_ratio, aligned,
                    pad_border, min_level=0, canonical_box_size=224, canonical_level=4, out_dtype=None,
                    want_levels=False):
    """Shared launcher of d2b_roi_align_multilevel.  `features`: list of NHWC tensors."""
    dev = nv.device_of(*features, boxes)
    host_out = not (isinstance(features[0], torch.Tensor) and features[0].is_cuda)
    fdt = features[0].dtype if isinstance(features[0], torch.Tensor) else torch.float32
    if fdt not in (torch.float32, torch.bfloat16):
        fdt = torch.float32
    feats = [nv.to_device(f, dev, fdt) for f in features]
    for f in feats:
        if f.dim() != 4:
            raise ValueError("feature maps must be NHWC rank-4 tensors")
    N, _, _, Cc = feats[0].shape
    boxes = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    M = boxes.shape[0]
    if not isinstance(batch_idx, torch.Tensor):
        batch_idx = torch.as_tensor(batch_idx)
    if batch_idx.dtype not in (torch.int32, torch.int64):
        batch_idx = batch_idx.to(torch.int32)  # functional.py:165 casts box_ind to int32
    if batch_idx.device != dev:
        batch_idx = batch_idx.to(dev, non_blocking=True)
    # a strided view (SparseBoxList.indices[:, 0]) is consumed in place via batch_idx_stride
    if batch_idx.dim() == 1 and batch_idx.stride(0) != 1 and batch_idx.numel() > 0:
        bidx_stride = batch_idx.stride(0)
        bptr = batch_idx.data_ptr()
    else:
        batch_idx = batch_idx.contiguous()
        bptr = batch_idx.data_ptr()
    oh, ow = int(output_size[0]), int(output_size[1])
    odt = fdt if out_dtype is None else out_dtype
    out = torch.empty((M, oh, ow, Cc), dtype=odt, device=dev)
    L = len(feats)
    counts = torch.empty(L, dtype=torch.int32, device=dev) if want_levels else None  # zeroed by the C entry
    levels = torch.empty(M, dtype=torch.int64, device=dev) if want_levels else None
    p = nv.RoiAlignParams()
    for l, f in enumerate(feats):
        if f.shape[0] != N or f.shape[3] != Cc:
            raise ValueError("all levels must share batch size and channel count")
        p.features[l] = f.data_ptr()
        p.height[l], p.width[l] = f.shape[1], f.shape[2]
        p.scale[l] = float(scales[l])
    p.num_levels, p.num_images, p.channels = L, N, Cc
    p.feature_dtype = nv.DTYPE_F32 if fdt == torch.float32 else nv.DTYPE_BF16
    p.boxes = boxes.data_ptr()
    p.batch_idx = bptr
    p.batch_idx_is_int64 = 1 if batch_idx.dtype == torch.int64 else 0
    p.batch_idx_stride = int(bidx_stride)
    p.num_rois = M
    p.output_h, p.output_w = oh, ow
    p.sampling_ratio = int(sampling_ratio)
    p.aligned = int(bool(aligned))
    p.pad_border = int(bool(pad_border))
    p.min_level = int(min_level)
    p.canonical_box_size = int(canonical_box_size)
    p.canonical_level = int(canonical_level)
    p.out = out.data_ptr()
    p.out_dtype = nv.DTYPE_F32 if odt == torch.float32 else nv.DTYPE_BF16
    p.level_counts = nv.ptr(counts)
    p.level_assignments = nv.ptr(levels)
    nv.call("roi_align_multilevel", p, dev)
    if host_out:
        out = nv.to_host(out)
    if want_levels:
        return out, counts, levels
    return out


def crop_and_resize(image, boxes, box_ind, crop_size, aligned=True, method='bilinear', pad_border=True):
    """
    Aligned version of tf.image.crop_and_resize (lib/layers/functional.py:100-166).

    Args:
        image: [n, h, w, c]
        boxes: [n, 4], ymin, xmin, ymax, xmax
        box_ind: [n]
        crop_size [2]:
    Returns:
        n,size,size,C
    """
    if method != 'bilinear':
        raise ValueError("only method='bilinear' is on the hot path")
    if not (isinstance(image, torch.Tensor) and image.dtype == torch.float32):
        return _roi_align_call([image], [1.0], boxes, box_ind, 1, crop_size, 0, aligned, pad_border)
    host = not image.is_cuda
    dev = nv.device_of(image, boxes)
    img = nv.to_device(image, dev, torch.float32)
    if img.dim() != 4:
        raise ValueError("image must be an NHWC rank-4 tensor")
    b = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    bi = nv.to_device(box_ind, dev, torch.int32)  # functional.py:165 casts box_ind to int32
    out = torch.empty((b.shape[0], int(crop_size[0]), int(crop_size[1]), img.shape[3]), dtype=torch.float32, device=dev)
    p = nv.CropAndResizeParams()
    p.image = img.data_ptr()
    p.num_images, p.height, p.width, p.channels = img.shape
    p.boxes, p.box_ind, p.num_boxes = b.data_ptr(), bi.data_ptr(), b.shape[0]
    p.crop_h, p.crop_w = int(crop_size[0]), int(crop_size[1])
    p.aligned, p.pad_border = int(bool(aligned)), int(bool(pad_border))
    p.out = out.data_ptr()
    nv.call("crop_and_resize_aligned", p, dev)
    return nv.to_host(out) if host else out


def _roi_align_backward_call(grad_out, feature_shapes, scales, boxes, batch_idx, sampling_ratio, aligned,
                             pad_border=True, min_level=0, canonical_box_size=224, canonical_level=4,
                             grad_features=None, deterministic=False):
    """Launcher of d2b_roi_align_backward: gradient of `_roi_align_call` w.r.t. every level's NHWC map.

    `feature_shapes`: list of (N, H, W, C).  `grad_features` (optional list of fp32 tensors) is accumulated
    into; when None, zero-initialised tensors are created.  `deterministic`: sum without floating-point atomics,
    in the CPU kernel's order (bit-identical to it and from run to run); the default is the faster atomic scatter."""
    dev = nv.device_of(grad_out, boxes)
    host = not grad_out.is_cuda
    g = nv.to_device(grad_out, dev, torch.float32)
    M, oh, ow, Cc = g.shape
    boxes = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    assert boxes.shape[0] == M
    if not isinstance(batch_idx, torch.Tensor):
        batch_idx = torch.as_tensor(batch_idx)
    if batch_idx.dtype not in (torch.int32, torch.int64):
        batch_idx = batch_idx.to(torch.int32)
    batch_idx = batch_idx.to(dev).contiguous()
    if grad_features is None:
        grad_features = [torch.zeros(tuple(s), dtype=torch.float32, device=dev) for s in feature_shapes]
    p = nv.RoiAlignBackwardParams()
    f = p.fwd
    for l, gf in enumerate(grad_features):
        assert gf.is_cuda and gf.is_contiguous() and gf.dtype == torch.float32 and gf.shape[3] == Cc
        f.height[l], f.width[l] = gf.shape[1], gf.shape[2]
        f.scale[l] = float(scales[l])
        p.grad_features[l] = gf.data_ptr()
    f.num_levels, f.num_images, f.channels = len(grad_features), grad_features[0].shape[0], Cc
    f.feature_dtype = f.out_dtype = nv.DTYPE_F32
    f.boxes, f.batch_idx = boxes.data_ptr(), batch_idx.data_ptr()
    f.batch_idx_is_int64 = 1 if batch_idx.dtype == torch.int64 else 0
    f.batch_idx_stride = 1
    f.num_rois = M
    f.output_h, f.output_w = oh, ow
    f.sampling_ratio = int(sampling_ratio)
    f.aligned, f.pad_border = int(bool(aligned)), int(bool(pad_border))
    f.min_level = int(min_level)
    f.canonical_box_size, f.canonical_level = int(canonical_box_size), int(canonical_level)
    p.grad_out = g.data_ptr()
    p.deterministic = int(bool(deterministic))
    nv.call("roi_align_backward", p, dev)
    if host:
        return [nv.to_host(t) for t in grad_features]
    return grad_features
