"""CPU: libd2b200.so builds for sm_100a, loads, and exports every symbol include/d2b200.h declares.
No compute is launched (there is no GPU here); argument validation paths that return before any CUDA
call are exercised through the C-ABI."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from detectron2_tensorflow_b200 import build, _native
    build.build()
    return _native.lib()


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "d2b200.h")).read()
    return sorted(set(re.findall(r"D2B_API\s+[\w\s\*]+?\b(d2b_\w+)\s*\(", src)))


def test_header_symbols_exported(lib):
    from detectron2_tensorflow_b200 import _native
    syms = _declared_symbols()
    assert len(syms) == 4 + 2 * len(_native.OPS) + 5  # + the five d2b_peer_* arena calls
    assert sorted(_native.EXPORTS) == syms
    for s in syms:
        assert hasattr(lib, s), s
    assert lib.d2b_version() >= 100
    assert lib.d2b_status_string(0) == b"ok"
    assert b"invalid" in lib.d2b_status_string(-1)


def test_struct_layout_matches_header(lib, tmp_path):
    """sizeof of every ctypes params struct equals the C compiler's sizeof of the header struct."""
    from detectron2_tensorflow_b200 import _native
    names = {"roi_align_multilevel": "d2b_roi_align_params", "apply_deltas": "d2b_apply_deltas_params",
             "segmented_topk": "d2b_segmented_topk_params", "batched_nms": "d2b_batched_nms_params",
             "rpn_proposals": "d2b_rpn_proposals_params", "fast_rcnn_postprocess": "d2b_fast_rcnn_params",
             "retinanet_postprocess": "d2b_retinanet_params", "matrix_nms": "d2b_matrix_nms_params",
             "paste_masks": "d2b_paste_masks_params", "crop_and_resize_aligned": "d2b_crop_and_resize_params",
             "decode_clip_filter": "d2b_decode_clip_filter_params", "get_deltas": "d2b_get_deltas_params",
             "pairwise_iou": "d2b_pairwise_iou_params", "label_boxes": "d2b_label_boxes_params",
             "matcher": "d2b_matcher_params", "subsample_labels": "d2b_subsample_labels_params", "roi_align_backward": "d2b_roi_align_backward_params",
             "yolo_postprocess": "d2b_yolo_params", "point_nms": "d2b_point_nms_params",
             "solo_mask_encode": "d2b_solo_mask_encode_params", "solo_postprocess": "d2b_solo_postprocess_params",
             "solo_dynamic_masks": "d2b_solo_dynamic_masks_params",
             "solo_upsample": "d2b_solo_upsample_params", "solo_select": "d2b_solo_select_params",
             "mask_rcnn_inference": "d2b_mask_rcnn_inference_params", "peer_copy": "d2b_peer_copy_params"}
    assert set(names) == set(_native.OPS)
    prog = '#include <stdio.h>\n#include "d2b200.h"\nint main(){' + "".join(
        f'printf("{op} %zu\\n", sizeof({st}));' for op, st in names.items()) + "return 0;}"
    src = tmp_path / "sz.c"
    src.write_text(prog)
    exe = tmp_path / "sz"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    sizes = dict(zip(out[0::2], map(int, out[1::2])))
    for op, st in _native.OPS.items():
        assert C.sizeof(st) == sizes[op], op


def test_argument_validation_without_gpu(lib):
    """EINVAL paths return before touching CUDA (reference: ValueError / assert / NotImplementedError)."""
    from detectron2_tensorflow_b200 import _native as nv
    p = nv.RoiAlignParams()
    p.num_levels = 0
    nv._bind("roi_align_multilevel")
    assert lib.d2b_roi_align_multilevel(C.byref(p), None, 0, None) == -1
    assert b"num_levels" in lib.d2b_last_error()
    p.num_levels, p.num_images, p.channels, p.output_h, p.output_w = 1, 1, 6, 7, 7
    assert lib.d2b_roi_align_multilevel(C.byref(p), None, 0, None) == -1  # channels % 4
    m = nv.MatrixNmsParams()
    m.kernel = 5
    nv._bind("matrix_nms")
    assert lib.d2b_matrix_nms(C.byref(m), None, 0, None) == -1
    assert b"not implemented" in lib.d2b_last_error()
    r = nv.RpnProposalsParams()
    r.num_levels, r.pre_nms_topk, r.post_nms_topk = 1, 0, 10
    nv._bind("rpn_proposals")
    assert lib.d2b_rpn_proposals(C.byref(r), None, 0, None) == -1
    lb = nv.LabelBoxesParams()
    lb.num_thresholds, lb.max_gt = 2, 8
    lb.thresholds[0], lb.thresholds[1] = 0.7, 0.3  # matcher.py:49 assert low <= high
    nv._bind("label_boxes")
    assert lib.d2b_label_boxes(C.byref(lb), None, 0, None) == -1
    assert b"ascending" in lib.d2b_last_error()
    lb.thresholds[0], lb.thresholds[1] = 0.3, 0.7
    lb.labels[0], lb.labels[1], lb.labels[2] = 0, 2, 1  # matcher.py:50 labels in {-1,0,1}
    assert lib.d2b_label_boxes(C.byref(lb), None, 0, None) == -1
    bw = nv.RoiAlignBackwardParams()
    bw.fwd.num_levels, bw.fwd.num_images, bw.fwd.channels, bw.fwd.output_h, bw.fwd.output_w = 1, 1, 8, 7, 7
    bw.fwd.feature_dtype = nv.DTYPE_BF16
    nv._bind("roi_align_backward")
    assert lib.d2b_roi_align_backward(C.byref(bw), None, 0, None) == -1
    assert b"fp32 only" in lib.d2b_last_error()
    # SOLOv2 ops
    dm = nv.SoloDynamicMasksParams()
    dm.batch, dm.n, dm.channels, dm.hw = 1, 4, 6, 64  # channels % 4 (16-byte TMA rows)
    nv._bind("solo_dynamic_masks")
    assert lib.d2b_solo_dynamic_masks(C.byref(dm), None, 0, None) == -1
    assert b"multiple of 4" in lib.d2b_last_error()
    dm.channels, dm.hw = 8, 1 << 24  # mask sums must stay exact in fp32
    assert lib.d2b_solo_dynamic_masks(C.byref(dm), None, 0, None) == -1
    dm.hw = 64
    assert lib.d2b_solo_dynamic_masks_workspace_bytes(C.byref(dm)) >= 2 * 4 * 8 * 4
    up = nv.SoloUpsampleParams()
    up.batch, up.num_dets, up.mask_h, up.mask_w, up.image_h, up.image_w = 1, 1, 0, 8, 16, 16
    nv._bind("solo_upsample")
    assert lib.d2b_solo_upsample(C.byref(up), None, 0, None) == -1
    up.mask_h, up.mask_w, up.image_h, up.image_w = 4000, 4000, 8, 8  # a 500x shrink does not fit a CTA's shared memory
    assert lib.d2b_solo_upsample(C.byref(up), None, 0, None) == -1
    assert b"shared memory" in lib.d2b_last_error()
    se = nv.SoloSelectParams()
    se.batch, se.num_cells, se.num_classes, se.channels, se.max_candidates = 1, 4, 2, 8, 0
    nv._bind("solo_select")
    assert lib.d2b_solo_select(C.byref(se), None, 0, None) == -1
    assert b"max_candidates" in lib.d2b_last_error()
    # workspace queries are pure host arithmetic
    t = nv.SegmentedTopkParams()
    t.num_groups, t.rows_per_group, t.k = 2, 4, 1000
    t.row_len[0], t.row_len[1] = 5000, 800
    nv._bind("segmented_topk")
    assert lib.d2b_segmented_topk_workspace_bytes(C.byref(t)) > 8 * 1024 * 8


def test_no_cpu_fallback_in_product():
    """The product package must not import the oracle or fall back to CPU compute."""
    pkg = os.path.join(ROOT, "detectron2_tensorflow_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                s = open(os.path.join(dp, f)).read()
                assert "import oracle" not in s and "from oracle" not in s and "liboracle" not in s, f
    import torch
    if not torch.cuda.is_available():
        from detectron2_tensorflow_b200 import _native as nv
        from detectron2_tensorflow_b200.layers import ROIAlign
        with pytest.raises(nv.D2BError):
            ROIAlign((7, 7), 0.25, 0)(torch.zeros(1, 8, 8, 4), torch.zeros(1, 4), torch.zeros(1, dtype=torch.int32))


def test_product_env_switches():
    """The environment variables the product reads.  A run-time switch that selects a slower variant lets a user step
    off the measured path; variants that lost their A/B are deleted, not left behind a switch.  D2B_RPN_GENERIC runs
    the generic proposal chain (the only one for k > 4096) on inputs the specialised chain would take, so that tests
    compare the two; D2B_LIB, NVCC and D2B_EXTRA_NVCC choose the library and the build."""
    pkg = os.path.join(ROOT, "detectron2_tensorflow_b200")
    read = re.compile(r"""(?:getenv|os\.environ\.get|os\.environ)\s*[(\[]\s*["']([A-Za-z0-9_]+)["']""")
    names = set()
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cc")):
                names.update(read.findall(open(os.path.join(dp, f)).read()))
    assert names == {"D2B_RPN_GENERIC", "D2B_LIB", "NVCC", "D2B_EXTRA_NVCC"}
