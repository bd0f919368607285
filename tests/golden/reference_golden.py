"""Loader of reference_python.npz (the outputs of the reference's own Python on the numpy TF shim, written by
make_reference_golden.py).  To keep the file small, two seeded inputs are not stored but regenerated here, bit for
bit as the generator drew them:

- rp_feat0..3, the FPN maps of the ROIPooler case, from the state of the generator's random stream just before it
  drew them (rp_feat_state);
- so_in_logits, the dynamic 1x1 conv of the recorded SOLOv2 candidates, with the generator's own numpy einsum.

The pooled ROI outputs of that case (rp_out_*, ra_single, cr_nopad) are stored for the rows rp_rows only."""
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_python.npz")
FEAT_HW = ((50, 84), (25, 42), (13, 21), (7, 11))
FEAT_C = 8
ROWS_PER_LEVEL = 4
_M64 = (1 << 64) - 1


def roi_rows(levels):
    """The rows of the pooled ROI outputs that the file keeps: the first four ROIs (shifted by the generator) and a
    fixed seeded sample of ROWS_PER_LEVEL ROIs of each pyramid level (`levels`: the level of every ROI)."""
    rng = np.random.default_rng(0)
    picks = [np.arange(4)] + [rng.choice(np.flatnonzero(levels == l), ROWS_PER_LEVEL, replace=False)
                              for l in np.unique(levels)]
    return np.unique(np.concatenate(picks))


def pack_state(rng):
    """The PCG64 state of `rng` as six uint64 words."""
    s = rng.bit_generator.state
    return np.array([s["state"]["state"] >> 64, s["state"]["state"] & _M64, s["state"]["inc"] >> 64,
                     s["state"]["inc"] & _M64, s["has_uint32"], s["uinteger"]], np.uint64)


def rp_feats(state):
    """The four FPN maps [2, H, W, 8] drawn from the packed generator state."""
    v = [int(x) for x in state]
    rng = np.random.Generator(np.random.PCG64())
    rng.bit_generator.state = {"bit_generator": "PCG64", "state": {"state": v[0] << 64 | v[1], "inc": v[2] << 64 | v[3]},
                               "has_uint32": v[4], "uinteger": v[5]}
    return [rng.standard_normal((2, h, w, FEAT_C)).astype(np.float32) for h, w in FEAT_HW]


def so_logits(mask_features, kernels, counts):
    """solo_v2.py:499-511 on the recorded candidates: [B, n, H, W] logits, zero beyond counts[b]."""
    B, H, W, _ = mask_features.shape
    out = np.zeros((B, kernels.shape[1], H, W), np.float32)
    for b in range(B):
        c = int(counts[b])
        out[b, :c] = np.einsum("nhwc,co->nhwo", mask_features[b:b + 1], kernels[b, :c].T.copy())[0].transpose(2, 0, 1)
    return out


def load():
    """The stored arrays plus the regenerated rp_feat0..3 and so_in_logits."""
    z = dict(np.load(PATH))
    for l, f in enumerate(rp_feats(z["rp_feat_state"])):
        z[f"rp_feat{l}"] = f
    z["so_in_logits"] = so_logits(z["so_in_mask_features"], z["so_in_kernels"], z["so_in_counts"])
    return z
