"""COCO run-length encoding as pycocotools defines it (common/maskApi.c rleEncode + rleToString), restated in numpy.
The reference the GPU encoder of d2b_paste_masks / d2b_solo_upsample (csrc/mask_rle.cuh) is compared against.

  rleEncode:   walk the mask column-major (j = x*H + y); the counts alternate starting with a run of ZEROS, so a mask
               whose pixel 0 is set starts with count 0; the last run ends at H*W.
  rleToString: x = cnts[i]; if (i > 2) x -= cnts[i-2]; then 5-bit groups, least significant first:
               c = x & 0x1f; x >>= 5 (arithmetic); more = (c & 0x10) ? x != -1 : x != 0; if (more) c |= 0x20;
               emit c + 48.  No terminator.

encode(mask) equals pycocotools.mask.encode(np.asfortranarray(mask))["counts"] for a uint8 {0,1} mask [H, W]."""
import numpy as np


def counts(mask):
    """rleEncode of one mask [H, W] -> int64 run lengths."""
    flat = np.asarray(mask).astype(bool).T.reshape(-1)  # column-major
    change = np.flatnonzero(flat[1:] != flat[:-1]) + 1
    lead = [0, 0] if flat[0] else [0]                   # a set pixel 0 opens with an empty run of zeros
    return np.diff(np.concatenate([lead, change, [flat.size]])).astype(np.int64)


def to_string(cnts):
    """rleToString of one list of counts -> bytes."""
    cnts = np.asarray(cnts, np.int64)
    x = cnts.copy()
    x[3:] -= cnts[1:-2]                                 # i > 2, not i >= 2
    groups, n = [], np.zeros(x.size, np.int64)
    alive = np.ones(x.size, bool)
    while alive.any():
        c = x & 0x1f
        x = x >> 5
        more = np.where(c & 0x10, x != -1, x != 0)
        groups.append(c | (more.astype(np.int64) << 5))
        n += alive                                      # groups value i emits
        alive &= more
    g = np.stack(groups, 1)
    return (g[np.arange(g.shape[1])[None, :] < n[:, None]] + 48).astype(np.uint8).tobytes()


def encode(masks):
    """uint8 {0,1} masks [M, H, W] -> list of M COCO RLE strings (bytes)."""
    return [to_string(counts(m)) for m in np.asarray(masks)]
