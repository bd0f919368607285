"""Drop-in for lib/structures/mask_ops.py: `reframe_box_masks_to_image_masks` (:7-56), plus the COCO run-length
encoding of the pasted masks on the GPU (`reframe_box_masks_to_rle`, `rle_to_coco`)."""
import torch

from .. import _native as nv


def reframe_box_masks_to_image_masks(box_masks, boxes, image_shape, mask_threshold=0.5, scope=None):
    """Transforms the box masks back to full image masks.

    Args:
        box_masks: [M, mh, mw] fp32 mask probabilities.
        boxes: [M, 4] absolute boxes (ymin, xmin, ymax, xmax) in the output image.
        image_shape: (height, width) of the output masks.
    Returns:
        uint8 [M, height, width] (1 where the pasted probability exceeds `mask_threshold`).
    """
    host = not box_masks.is_cuda
    dev = nv.device_of(box_masks, boxes)
    m = nv.to_device(box_masks, dev, torch.float32)
    b = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    assert m.dim() == 3 and m.shape[0] == b.shape[0]
    H, W = int(image_shape[0]), int(image_shape[1])
    out = torch.empty((m.shape[0], H, W), dtype=torch.uint8, device=dev)
    p = _paste_params(m, b, H, W, mask_threshold)
    p.out = out.data_ptr()
    nv.call("paste_masks", p, dev)
    return nv.to_host(out) if host else out


def _paste_params(m, b, H, W, mask_threshold):
    p = nv.PasteMasksParams()
    p.box_masks, p.boxes, p.num_masks = m.data_ptr(), b.data_ptr(), m.shape[0]
    p.mask_h, p.mask_w, p.image_h, p.image_w = m.shape[1], m.shape[2], H, W
    p.mask_threshold = float(mask_threshold)
    return p


def rle_call(run, num_masks, device, capacity):
    """Runs `run(out_rle, rle_capacity, out_rle_offsets, again)` (one op call with RLE requested) and returns
    (chars uint8 [capacity], offsets int64 [num_masks + 1]).  capacity=None: a sizing call with capacity 0, one host
    sync on offsets[-1], then a call with exactly that capacity (again=True).  An int capacity issues one call and no
    sync."""
    offsets = torch.empty(num_masks + 1, dtype=torch.int64, device=device)
    again = capacity is None
    if again:
        run(None, 0, offsets.data_ptr(), False)
        capacity = int(offsets[-1])
    capacity = int(capacity)
    chars = torch.empty(capacity, dtype=torch.uint8, device=device)
    run(chars.data_ptr() if capacity else None, capacity, offsets.data_ptr(), again)
    return chars, offsets


def reframe_box_masks_to_rle(box_masks, boxes, image_shape, mask_threshold=0.5, capacity=None):
    """The masks of `reframe_box_masks_to_image_masks` as COCO run-length strings, encoded on the GPU next to the
    paste; the [M, H, W] planes are never written.  String i is chars[offsets[i]:offsets[i+1]] and equals
    pycocotools.mask.encode(np.asfortranarray(mask_i))["counts"].

    capacity=None sizes the output exactly (one host sync).  With an int capacity there is no sync (the call can be
    captured in a CUDA graph): offsets are always complete, and only the strings with offsets[i+1] <= capacity are
    written -- `rle_to_coco` raises with the size needed when they did not all fit.
    Returns device tensors (chars uint8 [capacity], offsets int64 [M + 1])."""
    dev = nv.device_of(box_masks, boxes)
    m = nv.to_device(box_masks, dev, torch.float32)
    b = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    assert m.dim() == 3 and m.shape[0] == b.shape[0]
    H, W = int(image_shape[0]), int(image_shape[1])
    p = _paste_params(m, b, H, W, mask_threshold)

    def run(chars, cap, offsets, again):
        p.out_rle, p.rle_capacity, p.out_rle_offsets = chars, cap, offsets
        nv.call("paste_masks", p, dev)
    return rle_call(run, m.shape[0], dev, capacity)


def rle_to_coco(chars, offsets, image_shape):
    """(chars, offsets) of `reframe_box_masks_to_rle` / `solo_upsample_masks(return_rle=True)` -> host list of
    {"size": [H, W], "counts": bytes}, the per-mask object pycocotools.mask.encode returns."""
    off = offsets.cpu().tolist()
    need = int(off[-1])
    if need > chars.numel():
        raise ValueError(f"the RLE strings need {need} bytes but the buffer holds {chars.numel()}: "
                         f"call again with capacity >= {need}")
    data = chars[:need].cpu().numpy().tobytes()
    size = [int(image_shape[0]), int(image_shape[1])]
    return [{"size": size, "counts": data[off[i]:off[i + 1]]} for i in range(len(off) - 1)]
