"""Drop-in for lib/modeling/poolers.py (`assign_boxes_to_levels` :11-49, `ROIPooler` :52-180).

The reference runs assign -> per-level where/gather -> pad -> crop_and_resize ->
[avg_pool] -> concat -> invert_permutation -> gather.  Here `ROIPooler.call` is ONE
kernel launch (d2b_roi_align_multilevel): the level is computed in-kernel and each
ROI is written straight to its final row.
"""
import math

import torch

from .. import _native as nv
from ..layers import Layer, ROIAlign
from ..layers.functional import _roi_align_call, _roi_align_backward_call

__all__ = ["ROIPooler", "assign_boxes_to_levels"]


def assign_boxes_to_levels(boxlist, min_level, max_level, canonical_box_size, canonical_level):
    """
    Map each box in `boxlist` to a feature map level index (offset from `min_level`), int64 [M].
    Eqn.(1) of the FPN paper in the reference's fp32 op order (poolers.py:37-49).
    """
    boxes = boxlist.boxes if hasattr(boxlist, "boxes") else boxlist
    host = not boxes.is_cuda
    dev = nv.device_of(boxes)
    b = nv.to_device(boxes, dev, torch.float32).reshape(-1, 4)
    M = b.shape[0]
    L = max_level - min_level + 1
    # the level computation lives in the ROIAlign kernel's prologue; run it on a 1x1x4 dummy map
    dummy = [torch.zeros((1, 1, 1, 4), dtype=torch.float32, device=dev) for _ in range(L)]
    bidx = torch.zeros(M, dtype=torch.int32, device=dev)
    _, _, levels = _roi_align_call(dummy, [2.0 ** -(min_level + l) for l in range(L)], b, bidx, 1, (1, 1), 0, True,
                                   True, min_level=min_level, canonical_box_size=canonical_box_size,
                                   canonical_level=canonical_level, want_levels=True)
    return nv.to_host(levels) if host else levels


class ROIPooler(Layer):
    """Pools ROI features from one map or from an FPN pyramid (poolers.py:52-180): every box is routed to the
    level `assign_boxes_to_levels` picks and sampled there with ROIAlign -- here in a single kernel launch."""

    _ALIGNED = {"ROIAlign": False, "ROIAlignV2": True}

    def __init__(self, output_size, scales, sampling_ratio, pooler_type, canonical_box_size=224, canonical_level=4):
        super().__init__()
        size = (output_size, output_size) if isinstance(output_size, int) else tuple(output_size)
        if len(size) != 2 or not all(isinstance(v, int) for v in size):
            raise AssertionError("output_size must be an int or a pair of ints")
        if pooler_type not in self._ALIGNED:
            raise ValueError("Unknown pooler type: {}".format(pooler_type))  # same error as poolers.py:118-119
        self.output_size = size
        self.aligned = self._ALIGNED[pooler_type]
        self.scales = list(scales)
        self.sampling_ratio = sampling_ratio
        # API parity only (callers inspect it); `call` never loops over per-level poolers
        self.level_poolers = [ROIAlign(size, spatial_scale=s, sampling_ratio=sampling_ratio, aligned=self.aligned)
                              for s in self.scales]
        # scales are 1/stride with power-of-two strides: level = -log2(scale)  (poolers.py:121-129)
        lo, hi = -math.log2(self.scales[0]), -math.log2(self.scales[-1])
        if not (math.isclose(lo, round(lo)) and math.isclose(hi, round(hi))):
            raise AssertionError("scales must be powers of two")
        self.min_level, self.max_level = int(round(lo)), int(round(hi))
        if not (0 < self.min_level <= self.max_level):
            raise AssertionError("levels must be positive and ascending")
        if not (self.min_level <= canonical_level <= self.max_level) or canonical_box_size <= 0:
            raise AssertionError("canonical level / box size out of range")
        self.canonical_level = canonical_level
        self.canonical_box_size = canonical_box_size
        self.last_level_counts = None  # per-level ROI counts of the last call ('roi_align/num_roi_level_k', :173)
        self.record_level_counts = True  # False: skip that summary statistic (one memset + an atomic per ROI)

    def call(self, x, instances):
        """
        Args:
            x (list[Tensor]): NHWC feature maps with scales matching those used to construct this module.
            instances (SparseBoxList): `.data.boxes` [M,4], `.indices` [M,2] int64 (column 0 = image)
        Returns:
            Tensor (M, output_h, output_w, C) in input ROI order.
        """
        num_level_assignments = len(self.level_poolers)

        assert len(x) == num_level_assignments, (
            "unequal value, num_level_assignments={}, but x is list of {} "
            "Tensors".format(num_level_assignments, len(x)))

        batch_idx = instances.indices[:, 0]
        if num_level_assignments == 1:
            return _roi_align_call(x, self.scales, instances.data.boxes, batch_idx, 1, self.output_size,
                                   self.sampling_ratio, self.aligned, True)
        if not self.record_level_counts:
            return _roi_align_call(
                x, self.scales, instances.data.boxes, batch_idx, 1, self.output_size, self.sampling_ratio,
                self.aligned, True, min_level=self.min_level, canonical_box_size=self.canonical_box_size,
                canonical_level=self.canonical_level)
        out, counts, _ = _roi_align_call(
            x, self.scales, instances.data.boxes, batch_idx, 1, self.output_size, self.sampling_ratio,
            self.aligned, True, min_level=self.min_level, canonical_box_size=self.canonical_box_size,
            canonical_level=self.canonical_level, want_levels=True)
        self.last_level_counts = counts
        return out

    def backward(self, grad_output, x_shapes, instances, grad_x=None, deterministic=False):
        """Gradient of `call` w.r.t. the feature maps `x` (list of (N,H,W,C) shapes) -> list of NHWC tensors.
        Each ROI's gradient goes to the level `assign_boxes_to_levels` gave it.  Default: one kernel of atomic
        scatters (fastest; the last bits depend on scheduling).  deterministic=True: no floating-point atomics, the
        CPU kernel's summation order -- bit-identical to it and from run to run."""
        assert len(x_shapes) == len(self.level_poolers)
        return _roi_align_backward_call(grad_output, x_shapes, self.scales, instances.data.boxes,
                                        instances.indices[:, 0].contiguous(), self.sampling_ratio, self.aligned,
                                        min_level=self.min_level, canonical_box_size=self.canonical_box_size,
                                        canonical_level=self.canonical_level, grad_features=grad_x,
                                        deterministic=deterministic)
