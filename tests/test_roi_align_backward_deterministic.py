"""CPU: the workspace contract of the deterministic ROIAlign backward (no device needed; nothing is launched)."""
import ctypes as C

from detectron2_tensorflow_b200 import _native as nv


def params(deterministic, M=1000, N=2, L=4, oh=7, ow=7, sr=0):
    p = nv.RoiAlignBackwardParams()
    f = p.fwd
    f.num_levels, f.num_images, f.channels = L, N, 256
    for l in range(L):
        f.height[l], f.width[l], f.scale[l] = 200 >> l, 336 >> l, 1.0 / (4 << l)
        p.grad_features[l] = 0x1000 * (l + 1)  # never dereferenced: the size check comes first
    f.feature_dtype = f.out_dtype = nv.DTYPE_F32
    f.boxes, f.batch_idx, f.batch_idx_stride = 0x100, 0x200, 1
    f.num_rois, f.output_h, f.output_w, f.sampling_ratio = M, oh, ow, sr
    f.aligned, f.pad_border, f.min_level, f.canonical_box_size, f.canonical_level = 1, 1, 2, 224, 4
    p.grad_out = 0x300
    p.deterministic = deterministic
    return p


def test_workspace_is_zero_in_the_default_mode():
    L = nv._bind("roi_align_backward")
    assert L.d2b_roi_align_backward_workspace_bytes(C.byref(params(0))) == 0
    assert L.d2b_roi_align_backward_workspace_bytes(C.byref(params(1, M=0))) == 0


def test_workspace_grows_with_rois_and_taps():
    L = nv._bind("roi_align_backward")
    ws = lambda **kw: L.d2b_roi_align_backward_workspace_bytes(C.byref(params(1, **kw)))
    base = ws()
    assert base >= 1000 * (4 + 16 + 4 + 14 * 8)
    assert ws(M=2000) > base and ws(sr=2) > base and ws(oh=14, ow=14) > base


def test_too_small_workspace_is_refused_before_any_launch():
    L = nv._bind("roi_align_backward")
    p = params(1)
    need = L.d2b_roi_align_backward_workspace_bytes(C.byref(p))
    before = nv.kernel_launch_count()
    assert L.d2b_roi_align_backward(C.byref(p), None, 0, None) == -2  # D2B_EWORKSPACE
    assert L.d2b_roi_align_backward(C.byref(p), C.c_void_p(0x10000), need - 1, None) == -2
    assert b"workspace" in L.d2b_last_error()
    assert nv.kernel_launch_count() == before
