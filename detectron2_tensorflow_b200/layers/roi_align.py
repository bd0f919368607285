"""Drop-in for lib/layers/roi_align.py (`ROIAlign`, :9-75): same constructor arguments, `call` signature and
printable form; one C-ABI launch instead of pad -> crop_and_resize -> avg_pool."""
from .base import Layer
from .functional import _roi_align_backward_call, _roi_align_call


class ROIAlign(Layer):
    """Single-map ROIAlign.

    output_size     (h, w) of the pooled map
    spatial_scale   factor applied to the boxes (1 / feature stride)
    sampling_ratio  samples per bin axis; 0 means one bilinear sample per bin (roi_align.py:52-66)
    aligned         half-pixel aligned sampling (functional.py:138-152); False reproduces the legacy "ROIAlign"
    """

    def __init__(self, output_size, spatial_scale, sampling_ratio, aligned=True):
        super().__init__()
        if not isinstance(sampling_ratio, int):
            raise AssertionError(sampling_ratio)
        self.output_size, self.spatial_scale = output_size, spatial_scale
        self.sampling_ratio, self.aligned = sampling_ratio, aligned

    def call(self, inputs, boxes, box_inds):
        """inputs: NHWC feature map; boxes: [B, 4] (y1, x1, y2, x2) in image pixels; box_inds: [B] image of each box.
        Returns [B, output_h, output_w, C]."""
        return _roi_align_call([inputs], [self.spatial_scale], boxes, box_inds, 1, self.output_size,
                               self.sampling_ratio, self.aligned, True)

    def backward(self, grad_output, input_shape, boxes, box_inds, grad_input=None, deterministic=False):
        """Gradient of `call` w.r.t. `inputs` (what TF autodiff runs in training; boxes get none,
        functional.py:120).  grad_output [B, oh, ow, C] -> [N, H, W, C]; accumulates into `grad_input` if given.
        deterministic=True sums without atomics in the CPU kernel's order: bit-identical to it and reproducible."""
        grads = _roi_align_backward_call(grad_output, [input_shape], [self.spatial_scale], boxes, box_inds,
                                         self.sampling_ratio, self.aligned,
                                         grad_features=None if grad_input is None else [grad_input],
                                         deterministic=deterministic)
        return grads[0]

    def __repr__(self):
        fields = ("output_size", "spatial_scale", "sampling_ratio", "aligned")
        return f"{type(self).__name__}(" + ", ".join(f"{k}={getattr(self, k)}" for k in fields) + ")"
