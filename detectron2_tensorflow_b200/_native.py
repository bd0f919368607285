"""ctypes binding of libd2b200.so (the C-ABI declared in include/d2b200.h).

There is NO fallback: if the shared library is missing or an entry point fails,
the operators raise.  torch is used only for device memory and streams.
"""
import ctypes as C
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("D2B_LIB") or os.path.join(_PKG, "lib", "libd2b200.so")  # D2B_LIB: A/B builds (tools/)

MAX_LEVELS = 8
DTYPE_F32, DTYPE_BF16 = 0, 1
TOPK_IDENTITY, TOPK_SIGMOID = 0, 1
MNMS_GAUSSIAN, MNMS_LINEAR = 0, 1
IOU_TYPES = {"iou": 0, "giou": 1, "diou": 2, "ciou": 3}

_vp = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f32 = C.c_float


class RoiAlignParams(C.Structure):
    _fields_ = [
        ("features", _vp * MAX_LEVELS), ("height", _i32 * MAX_LEVELS), ("width", _i32 * MAX_LEVELS),
        ("scale", _f32 * MAX_LEVELS), ("num_levels", _i32), ("num_images", _i32), ("channels", _i32),
        ("feature_dtype", _i32), ("boxes", _vp), ("batch_idx", _vp), ("batch_idx_is_int64", _i32),
        ("batch_idx_stride", _i64), ("num_rois", _i64), ("output_h", _i32), ("output_w", _i32),
        ("sampling_ratio", _i32), ("aligned", _i32), ("pad_border", _i32), ("min_level", _i32),
        ("canonical_box_size", _i32), ("canonical_level", _i32), ("out", _vp), ("out_dtype", _i32),
        ("level_counts", _vp), ("level_assignments", _vp),
    ]


class ApplyDeltasParams(C.Structure):
    _fields_ = [("deltas", _vp), ("boxes", _vp), ("n", _i64), ("k", _i32), ("weights", _f32 * 4),
                ("scale_clamp", _f32), ("out", _vp)]


class SegmentedTopkParams(C.Structure):
    _fields_ = [("scores", _vp * MAX_LEVELS), ("row_len", _i64 * MAX_LEVELS), ("k_limit", _i32 * MAX_LEVELS),
                ("num_groups", _i32), ("rows_per_group", _i32), ("k", _i32), ("transform", _i32),
                ("out_values", _vp), ("out_indices", _vp), ("out_counts", _vp)]


class BatchedNmsParams(C.Structure):
    _fields_ = [("boxes", _vp), ("scores", _vp), ("counts", _vp), ("num_segments", _i32), ("n", _i32),
                ("max_output_size", _i32), ("iou_threshold", _f32), ("keep", _vp), ("num_keep", _vp)]


class RpnProposalsParams(C.Structure):
    _fields_ = [("logits", _vp * MAX_LEVELS), ("proposals", _vp * MAX_LEVELS), ("deltas", _vp * MAX_LEVELS),
                ("anchors", _vp * MAX_LEVELS), ("hwa", _i64 * MAX_LEVELS), ("num_levels", _i32),
                ("num_images", _i32), ("image_shapes", _vp), ("nms_thresh", _f32), ("pre_nms_topk", _i32),
                ("post_nms_topk", _i32), ("min_box_side_len", _f32), ("weights", _f32 * 4),
                ("scale_clamp", _f32), ("out_boxes", _vp), ("out_logits", _vp), ("out_valid", _vp),
                ("out_num_valid", _vp), ("out_nms_boxes_in", _vp),
                ("cell_anchors", _vp * MAX_LEVELS), ("num_cell_anchors", _i32 * MAX_LEVELS),
                ("grid_w", _i32 * MAX_LEVELS), ("stride", _i32 * MAX_LEVELS)]


class FastRcnnParams(C.Structure):
    _fields_ = [("boxes", _vp), ("scores", _vp), ("indices", _vp), ("num_preds", _i64), ("num_images", _i32),
                ("rmax", _i32), ("num_bbox_reg_classes", _i32), ("num_classes", _i32), ("image_shapes", _vp),
                ("score_thresh", _f32), ("nms_thresh", _f32), ("topk_per_image", _i32),
                ("nms_cls_agnostic", _i32), ("out_boxes", _vp), ("out_scores", _vp), ("out_classes", _vp),
                ("out_valid", _vp), ("out_roi_index", _vp), ("out_num", _vp), ("out_nms_boxes_in", _vp),
                ("deltas", _vp), ("proposal_boxes", _vp), ("weights", _f32 * 4), ("scale_clamp", _f32)]


class RetinanetParams(C.Structure):
    _fields_ = [("box_cls", _vp * MAX_LEVELS), ("box_delta", _vp * MAX_LEVELS), ("anchors", _vp * MAX_LEVELS),
                ("hwa", _i64 * MAX_LEVELS), ("num_levels", _i32), ("num_images", _i32), ("num_classes", _i32),
                ("topk_candidates", _i32), ("score_thresh", _f32), ("nms_thresh", _f32),
                ("max_detections", _i32), ("weights", _f32 * 4), ("scale_clamp", _f32), ("out_boxes", _vp),
                ("out_scores", _vp), ("out_classes", _vp), ("out_valid", _vp), ("out_num", _vp),
                ("out_nms_boxes_in", _vp),
                ("cell_anchors", _vp * MAX_LEVELS), ("num_cell_anchors", _i32 * MAX_LEVELS),
                ("grid_w", _i32 * MAX_LEVELS), ("stride", _i32 * MAX_LEVELS)]


class MatrixNmsParams(C.Structure):
    _fields_ = [("masks", _vp), ("classes", _vp), ("scores", _vp), ("sum_masks", _vp), ("counts", _vp),
                ("batch", _i32), ("n", _i32), ("hw", _i64), ("kernel", _i32), ("sigma", _f32), ("out", _vp),
                ("packed_masks", _vp)]


class PasteMasksParams(C.Structure):
    _fields_ = [("box_masks", _vp), ("boxes", _vp), ("num_masks", _i64), ("mask_h", _i32), ("mask_w", _i32),
                ("image_h", _i32), ("image_w", _i32), ("mask_threshold", _f32), ("out", _vp),
                ("out_rle", _vp), ("rle_capacity", _i64), ("out_rle_offsets", _vp),
                ("num_images", _i32), ("dets_per_image", _i32), ("output_shapes", _vp), ("input_shapes", _vp),
                ("valid", _vp)]


class CropAndResizeParams(C.Structure):
    _fields_ = [("image", _vp), ("num_images", _i32), ("height", _i32), ("width", _i32), ("channels", _i32),
                ("boxes", _vp), ("box_ind", _vp), ("num_boxes", _i64), ("crop_h", _i32), ("crop_w", _i32),
                ("aligned", _i32), ("pad_border", _i32), ("out", _vp)]


class DecodeClipFilterParams(C.Structure):
    _fields_ = [("deltas", _vp), ("anchors", _vp), ("num_images", _i32), ("n", _i64), ("image_shapes", _vp),
                ("weights", _f32 * 4), ("scale_clamp", _f32), ("min_box_side_len", _f32), ("out_boxes", _vp),
                ("out_keep", _vp)]


class GetDeltasParams(C.Structure):
    _fields_ = [("src_boxes", _vp), ("target_boxes", _vp), ("n", _i64), ("weights", _f32 * 4), ("out", _vp)]


class PairwiseIouParams(C.Structure):
    _fields_ = [("boxes1", _vp), ("boxes2", _vp), ("n1", _i64), ("n2", _i64), ("out", _vp), ("iou_type", _i32)]


MATCH_MAX_THRESHOLDS = 4
MATCH_MAX_GT = 1024


class LabelBoxesParams(C.Structure):
    _fields_ = [("pred_boxes", _vp), ("pred_shared", _i32), ("pred_counts", _vp), ("num_images", _i32),
                ("num_preds", _i32), ("gt_boxes", _vp), ("gt_valid", _vp), ("gt_crowd", _vp), ("gt_difficult", _vp),
                ("max_gt", _i32), ("thresholds", _f32 * MATCH_MAX_THRESHOLDS), ("num_thresholds", _i32),
                ("labels", _i32 * (MATCH_MAX_THRESHOLDS + 1)), ("allow_low_quality_matches", _i32),
                ("boundary_threshold", _f32), ("image_shapes", _vp), ("compute_deltas", _i32), ("weights", _f32 * 4),
                ("out_matches", _vp), ("out_labels", _vp), ("out_deltas", _vp)]


class MatcherParams(C.Structure):
    _fields_ = [("match_quality_matrix", _vp), ("crowd_matrix", _vp), ("difficult_matrix", _vp), ("num_gt", _i32),
                ("num_crowd", _i32), ("num_difficult", _i32), ("use_crowd", _i32), ("use_difficult", _i32),
                ("num_preds", _i64), ("thresholds", _f32 * MATCH_MAX_THRESHOLDS), ("num_thresholds", _i32),
                ("labels", _i32 * (MATCH_MAX_THRESHOLDS + 1)), ("allow_low_quality_matches", _i32),
                ("out_matches", _vp), ("out_labels", _vp)]


class SubsampleLabelsParams(C.Structure):
    _fields_ = [("labels", _vp), ("num_images", _i32), ("num_labels", _i64), ("num_samples", _i32),
                ("max_positives", _i32), ("bg_label", _i64), ("seed", C.c_uint64), ("out_pos_idx", _vp),
                ("out_neg_idx", _vp), ("out_num_pos", _vp), ("out_num_neg", _vp), ("out_labels", _vp)]


class YoloParams(C.Structure):
    _fields_ = [("boxes", _vp), ("probs", _vp), ("num_images", _i32), ("num_boxes", _i32), ("num_classes", _i32),
                ("score_thresh", _f32), ("nms_thresh", _f32), ("post_nms_topk", _i32), ("out_boxes", _vp),
                ("out_scores", _vp), ("out_classes", _vp), ("out_valid", _vp), ("out_num", _vp),
                ("out_nms_boxes_in", _vp)]


class PointNmsParams(C.Structure):
    _fields_ = [("scores", _vp), ("num_images", _i32), ("height", _i32), ("width", _i32), ("channels", _i32),
                ("out", _vp)]


class SoloMaskEncodeParams(C.Structure):
    _fields_ = [("mask_logits", _vp), ("counts", _vp), ("batch", _i32), ("n", _i32), ("hw", _i64),
                ("mask_threshold", _f32), ("packed_masks", _vp), ("sum_masks", _vp), ("score_sums", _vp)]


class SoloPostprocessParams(C.Structure):
    _fields_ = [("mask_logits", _vp), ("scores", _vp), ("classes", _vp), ("strides", _vp), ("counts", _vp),
                ("batch", _i32), ("n", _i32), ("hw", _i64), ("mask_threshold", _f32), ("pre_nms_topk", _i32),
                ("kernel", _i32), ("sigma", _f32), ("update_score_threshold", _f32), ("max_detections", _i32),
                ("out_masks", _vp), ("out_packed_masks", _vp), ("out_classes", _vp), ("out_scores", _vp),
                ("out_valid", _vp), ("out_num", _vp), ("mask_features", _vp), ("mask_kernels", _vp), ("channels", _i32)]


class SoloDynamicMasksParams(C.Structure):
    _fields_ = [("mask_features", _vp), ("mask_kernels", _vp), ("counts", _vp), ("batch", _i32), ("n", _i32),
                ("channels", _i32), ("hw", _i64), ("mask_threshold", _f32), ("packed_masks", _vp), ("sum_masks", _vp),
                ("score_sums", _vp), ("mask_logits", _vp)]


class MaskRcnnInferenceParams(C.Structure):
    _fields_ = [("mask_logits", _vp), ("pred_classes", _vp), ("num_masks", _i64), ("mask_h", _i32), ("mask_w", _i32),
                ("num_classes", _i32), ("out", _vp)]


class SoloSelectParams(C.Structure):
    _fields_ = [("scores", _vp), ("kernels", _vp), ("cell_strides", _vp), ("batch", _i32), ("num_cells", _i32),
                ("num_classes", _i32), ("channels", _i32), ("score_threshold", _f32), ("max_candidates", _i32),
                ("out_scores", _vp), ("out_classes", _vp), ("out_strides", _vp), ("out_kernels", _vp),
                ("out_counts", _vp), ("out_total", _vp)]


class SoloUpsampleParams(C.Structure):
    _fields_ = [("packed_masks", _vp), ("batch", _i32), ("num_dets", _i32), ("mask_h", _i32), ("mask_w", _i32),
                ("image_h", _i32), ("image_w", _i32), ("align_corners", _i32), ("mask_threshold", _f32),
                ("out_masks", _vp), ("out_packed_masks", _vp), ("out_boxes", _vp),
                ("out_rle", _vp), ("rle_capacity", _i64), ("out_rle_offsets", _vp),
                ("output_shapes", _vp), ("mask_shapes", _vp), ("valid", _vp)]


class RoiAlignBackwardParams(C.Structure):
    _fields_ = [("fwd", RoiAlignParams), ("grad_out", _vp), ("grad_features", _vp * MAX_LEVELS),
                ("deterministic", _i32)]


# op name -> params struct; every op exports d2b_<op> and d2b_<op>_workspace_bytes
PEER_HANDLE_BYTES, PEER_MAX_SEGMENTS, PEER_MAX_FLAGS = 64, 112, 16


class CopySegment(C.Structure):
    _fields_ = [("src", _vp), ("dst", _vp), ("bytes", C.c_uint64)]


class PeerCopyParams(C.Structure):
    _fields_ = [("segments", C.POINTER(CopySegment)), ("num_segments", _i32), ("wait_flags", C.POINTER(_vp)),
                ("num_wait", _i32), ("wait_lag", _i32), ("signal_flags", C.POINTER(_vp)), ("num_signal", _i32),
                ("epoch_counter", _vp), ("ticket", _vp), ("error_flag", _vp), ("timeout_ms", C.c_uint32)]


OPS = {
    "roi_align_multilevel": RoiAlignParams,
    "apply_deltas": ApplyDeltasParams,
    "segmented_topk": SegmentedTopkParams,
    "batched_nms": BatchedNmsParams,
    "rpn_proposals": RpnProposalsParams,
    "fast_rcnn_postprocess": FastRcnnParams,
    "retinanet_postprocess": RetinanetParams,
    "matrix_nms": MatrixNmsParams,
    "paste_masks": PasteMasksParams,
    "crop_and_resize_aligned": CropAndResizeParams,
    "decode_clip_filter": DecodeClipFilterParams,
    "get_deltas": GetDeltasParams,
    "pairwise_iou": PairwiseIouParams,
    "label_boxes": LabelBoxesParams,
    "matcher": MatcherParams,
    "subsample_labels": SubsampleLabelsParams,
    "roi_align_backward": RoiAlignBackwardParams,
    "yolo_postprocess": YoloParams,
    "point_nms": PointNmsParams,
    "solo_mask_encode": SoloMaskEncodeParams,
    "solo_postprocess": SoloPostprocessParams,
    "solo_dynamic_masks": SoloDynamicMasksParams,
    "solo_upsample": SoloUpsampleParams,
    "solo_select": SoloSelectParams,
    "mask_rcnn_inference": MaskRcnnInferenceParams,
    "peer_copy": PeerCopyParams,
}
EXPORTS = ["d2b_version", "d2b_status_string", "d2b_last_error", "d2b_kernel_launch_count"] + \
          [f"d2b_{op}{sfx}" for op in OPS for sfx in ("", "_workspace_bytes")] + \
          ["d2b_peer_alloc", "d2b_peer_free", "d2b_peer_export", "d2b_peer_open", "d2b_peer_close"]


class D2BError(RuntimeError):
    pass


_lib = None
launch_count = 0  # C-ABI op calls issued by this process (bench.py reports it)


def lib():
    """Load libd2b200.so; raises if it has not been built (no CPU fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise D2BError(f"{LIB_PATH} not found: build it with `python -m detectron2_tensorflow_b200.build` "
                           "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.d2b_version.restype = C.c_int
        L.d2b_status_string.restype = C.c_char_p
        L.d2b_status_string.argtypes = [C.c_int]
        L.d2b_last_error.restype = C.c_char_p
        L.d2b_kernel_launch_count.restype = C.c_uint64
        _lib = L
    return _lib


_bound = set()


def _bind(op):
    L = lib()
    if op not in _bound:
        st = OPS[op]
        f = getattr(L, f"d2b_{op}")
        f.restype = C.c_int
        f.argtypes = [C.POINTER(st), _vp, C.c_size_t, _vp]
        w = getattr(L, f"d2b_{op}_workspace_bytes")
        w.restype = C.c_size_t
        w.argtypes = [C.POINTER(st)]
        _bound.add(op)
    return L


def kernel_launch_count():
    """CUDA kernels launched by libd2b200 in this process."""
    return int(lib().d2b_kernel_launch_count())


def to_host(t):
    """Device->host through the caching pinned-host allocator (one async copy + stream sync)."""
    if not t.is_cuda:
        return t
    out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    out.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return out


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return t.data_ptr()


_ws_cache = {}


def _workspace(nbytes, device):
    """Scratch buffer owned by the host layer (the C library never allocates).

    Eager calls: a grow-only buffer per (device, CUDA stream) -- two torch Stream objects with the same handle ARE
    the same CUDA stream, so sharing is ordered.  During CUDA-graph capture the buffer is a fresh allocation from
    the capturing graph's private memory pool instead: the graph then owns every workspace its kernels were baked
    with (the pool lives as long as the graph), a later, larger eager call can never free it, and two graphs
    replayed concurrently never share scratch memory."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def call(op, params, device):
    """Run d2b_<op> on torch's current stream of `device`."""
    global launch_count
    L = _bind(op)
    with torch.cuda.device(device):
        nbytes = getattr(L, f"d2b_{op}_workspace_bytes")(C.byref(params))
        ws = _workspace(nbytes, device) if nbytes else None
        stream = torch.cuda.current_stream(device).cuda_stream
        rc = getattr(L, f"d2b_{op}")(C.byref(params), ws.data_ptr() if ws is not None else None,
                                     nbytes, C.c_void_p(stream))
    launch_count += 1
    if rc != 0:
        msg = f"d2b_{op}: {L.d2b_status_string(rc).decode()}: {L.d2b_last_error().decode()}"
        if rc == -1:
            raise ValueError(msg)
        raise D2BError(msg)


def to_device(t, device, dtype=None):
    """Host->device staging used by every operator: accepts torch tensors (any device) or array-likes."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    if t.device != device:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


def default_device():
    if not torch.cuda.is_available():
        raise D2BError("no CUDA device: libd2b200 has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def device_of(*tensors):
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    return default_device()


# ---------------------------------------------------------------- peer-memory arenas (CUDA IPC; sharding.PeerGatherPlan)
def _peer_check(rc, what):
    if rc != 0:
        L = lib()
        raise D2BError(f"{what}: {L.d2b_status_string(rc).decode()}: {L.d2b_last_error().decode()}")


def peer_alloc(nbytes, device):
    """A zero-filled cudaMalloc arena on `device` that other processes of the node can map; returns its address."""
    L = lib()
    L.d2b_peer_alloc.argtypes = [C.c_size_t, C.POINTER(_vp)]
    out = _vp()
    with torch.cuda.device(device):
        _peer_check(L.d2b_peer_alloc(int(nbytes), C.byref(out)), "d2b_peer_alloc")
    return int(out.value)


def peer_free(address, device):
    L = lib()
    L.d2b_peer_free.argtypes = [_vp]
    with torch.cuda.device(device):
        _peer_check(L.d2b_peer_free(_vp(address)), "d2b_peer_free")


def peer_export(address, device):
    """The CUDA IPC handle (bytes) of an arena of this process."""
    L = lib()
    L.d2b_peer_export.argtypes = [_vp, C.c_char_p]
    buf = C.create_string_buffer(PEER_HANDLE_BYTES)
    with torch.cuda.device(device):
        _peer_check(L.d2b_peer_export(_vp(address), buf), "d2b_peer_export")
    return bytes(buf.raw)


def peer_open(handle, device):
    """Map another process's arena into this one (peer access over NVLink); returns the local address."""
    L = lib()
    L.d2b_peer_open.argtypes = [C.c_char_p, C.POINTER(_vp)]
    out = _vp()
    with torch.cuda.device(device):
        _peer_check(L.d2b_peer_open(bytes(handle), C.byref(out)), "d2b_peer_open")
    return int(out.value)


def peer_close(address, device):
    L = lib()
    L.d2b_peer_close.argtypes = [_vp]
    with torch.cuda.device(device):
        _peer_check(L.d2b_peer_close(_vp(address)), "d2b_peer_close")


def peer_copy(segments, device, epoch_counter, ticket, error_flag, wait_flags=(), wait_lag=0, signal_flags=(),
              timeout_ms=2000):
    """d2b_peer_copy on torch's current stream: [wait on flags] -> copy `segments` [(src, dst, nbytes) addresses]
    -> [raise flags].  All addresses are plain ints (this GPU's memory or mapped peer memory)."""
    segs = (CopySegment * max(len(segments), 1))()
    for i, (src, dst, n) in enumerate(segments):
        segs[i].src, segs[i].dst, segs[i].bytes = int(src), int(dst), int(n)
    wf = (_vp * max(len(wait_flags), 1))(*[int(a) for a in wait_flags])
    sf = (_vp * max(len(signal_flags), 1))(*[int(a) for a in signal_flags])
    p = PeerCopyParams(segments=segs, num_segments=len(segments), wait_flags=wf, num_wait=len(wait_flags),
                       wait_lag=int(wait_lag), signal_flags=sf, num_signal=len(signal_flags),
                       epoch_counter=int(epoch_counter), ticket=int(ticket), error_flag=int(error_flag),
                       timeout_ms=int(timeout_ms))
    call("peer_copy", p, device)
