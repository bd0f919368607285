/*
 * d2b200.h -- C-ABI of libd2b200.so: B200 (sm_100a) kernels for the detection
 * post-backbone hot path of SimeonZhang/detectron2_tensorflow.
 *
 * The reference has no FFI boundary of its own (it is pure Python over stock
 * TensorFlow ops).  Each entry point below replaces the TF-op chain behind one
 * reference Python operator; the cited file:line is that operator.  A TF
 * custom-op shim (csrc/tf_ops) or the ctypes host layer
 * (detectron2_tensorflow_b200/_native.py) binds exactly these symbols.
 *
 * Conventions (SURVEY.md section 8b):
 *  - all pointers are DEVICE pointers unless marked "host"; the caller owns all
 *    memory (inputs, outputs, workspace); the library never allocates, frees or
 *    keeps a pointer after the call returns; no global mutable state.
 *  - every op has  size_t d2b_<op>_workspace_bytes(const params*)  and
 *    int d2b_<op>(const params*, void* workspace, size_t workspace_bytes, d2b_stream_t).
 *    All work is enqueued on the caller's stream; nothing synchronises the host.
 *  - outputs are fixed-size and zero-padded like the reference's
 *    pad_or_clip_tensor (lib/utils/shape_utils.py:80-99) with explicit counts.
 *  - return 0 on success, a negative D2B_E* code otherwise; never throws/exits.
 *  - boxes are [ymin, xmin, ymax, xmax] fp32 absolute pixels
 *    (lib/structures/box_list.py:46-49); features are NHWC
 *    (lib/layers/roi_align.py:48); deltas are (dy,dx,dh,dw)
 *    (lib/modeling/box_regression.py:101-106); image shapes are (h, w) int32.
 */
#ifndef D2B200_H_
#define D2B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define D2B_API __attribute__((visibility("default")))
#else
#define D2B_API
#endif

typedef void* d2b_stream_t; /* a cudaStream_t */

enum {
  D2B_OK = 0,
  D2B_EINVAL = -1,     /* shape / attribute violation (reference: ValueError / assert) */
  D2B_EWORKSPACE = -2, /* workspace NULL or smaller than *_workspace_bytes() */
  D2B_ECUDA = -3,      /* a CUDA runtime call or launch failed */
  D2B_EUNSUPPORTED = -4
};

#define D2B_MAX_LEVELS 8
#define D2B_DTYPE_F32 0
#define D2B_DTYPE_BF16 1

D2B_API int d2b_version(void);
D2B_API const char* d2b_status_string(int status);
/* thread-local detail of the last non-zero status returned on this thread */
D2B_API const char* d2b_last_error(void);
/* number of CUDA kernels this library has launched in the process (monotonic; bench bookkeeping) */
D2B_API uint64_t d2b_kernel_launch_count(void);

/* ------------------------------------------------------------------------
 * Multi-level ROIAlign == ROIPooler.call          lib/modeling/poolers.py:134-180
 *   level assignment                               lib/modeling/poolers.py:11-49
 *   ROIAlign.call                                  lib/layers/roi_align.py:45-66
 *   crop_and_resize (aligned / pad_border)         lib/layers/functional.py:100-166
 * One launch: level computed in-kernel, every ROI written to its final row
 * (no per-level gather, no SYMMETRIC pad copy, no inverse-permutation pass).
 * With num_levels == 1 it is ROIAlign.call / crop_and_resize on one map.
 * ---------------------------------------------------------------------- */
typedef struct {
  const void* features[D2B_MAX_LEVELS]; /* level l: [num_images, height[l], width[l], channels] */
  int32_t height[D2B_MAX_LEVELS];
  int32_t width[D2B_MAX_LEVELS];
  float scale[D2B_MAX_LEVELS]; /* spatial_scale of level l (1/stride) */
  int32_t num_levels;          /* 1..D2B_MAX_LEVELS */
  int32_t num_images;
  int32_t channels;
  int32_t feature_dtype; /* D2B_DTYPE_F32 | D2B_DTYPE_BF16 */
  const float* boxes;    /* [num_rois, 4] */
  const void* batch_idx; /* image of each ROI; element i at batch_idx[i*batch_idx_stride] */
  int32_t batch_idx_is_int64; /* 1: int64 (SparseBoxList.indices[:,0]); 0: int32 (box_ind) */
  int64_t batch_idx_stride;   /* in elements (2 when pointing at SparseBoxList.indices) */
  int64_t num_rois;
  int32_t output_h, output_w;
  int32_t sampling_ratio;     /* 0 => one sample per bin (reference default) */
  int32_t aligned;            /* 1: "ROIAlignV2"; 0: "ROIAlign" */
  int32_t pad_border;         /* functional.crop_and_resize pad_border (ROIAlign: always 1) */
  int32_t min_level;          /* -log2(scale[0]); used only when num_levels > 1 */
  int32_t canonical_box_size; /* 224 */
  int32_t canonical_level;    /* 4 */
  void* out;                  /* [num_rois, output_h, output_w, channels] */
  int32_t out_dtype;          /* D2B_DTYPE_F32 (or BF16 when feature_dtype is BF16) */
  int32_t* level_counts;      /* optional [num_levels]: 'roi_align/num_roi_level_k' (poolers.py:173) */
  int64_t* level_assignments; /* optional [num_rois]: assign_boxes_to_levels output */
} d2b_roi_align_params;

D2B_API size_t d2b_roi_align_multilevel_workspace_bytes(const d2b_roi_align_params* p);
D2B_API int d2b_roi_align_multilevel(const d2b_roi_align_params* p, void* workspace,
                                     size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Box2BoxTransform.apply_deltas               lib/modeling/box_regression.py:76-123
 * deltas [n, k*4], boxes [n, 4] -> out [n, k*4]
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* deltas;
  const float* boxes;
  int64_t n;
  int32_t k;
  float weights[4]; /* (wy, wx, wh, ww) */
  float scale_clamp;
  float* out;
} d2b_apply_deltas_params;
D2B_API size_t d2b_apply_deltas_workspace_bytes(const d2b_apply_deltas_params* p);
D2B_API int d2b_apply_deltas(const d2b_apply_deltas_params* p, void* workspace,
                             size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Segmented top-k == tf.nn.top_k per (image, level) row
 *   lib/modeling/proposal_generator/rpn_outputs.py:70,106
 *   lib/modeling/single_stage_heads/retinanet.py:321-326 (transform = sigmoid)
 * Rows are described per group (level): group g holds rows_per_group rows of
 * row_len[g] contiguous fp32 each.  Row r = image * num_groups + g.
 * Output per row: the k_r = min(k, row_len[g]) largest in (value desc, index asc)
 * order, zero/-1 padded to k.  NaN ranks lowest.
 * ---------------------------------------------------------------------- */
#define D2B_TOPK_IDENTITY 0
#define D2B_TOPK_SIGMOID 1
typedef struct {
  const float* scores[D2B_MAX_LEVELS]; /* group g: [rows_per_group, row_len[g]] */
  int64_t row_len[D2B_MAX_LEVELS];
  int32_t k_limit[D2B_MAX_LEVELS];     /* per-group cap on k (0 => k); RetinaNet: #anchors (retinanet.py:325) */
  int32_t num_groups;
  int32_t rows_per_group;
  int32_t k;
  int32_t transform;   /* D2B_TOPK_* applied to every score before ranking */
  float* out_values;   /* [rows, k]  transformed values */
  int32_t* out_indices; /* [rows, k]  index within the row, -1 padding */
  int32_t* out_counts;  /* [rows] */
} d2b_segmented_topk_params;
D2B_API size_t d2b_segmented_topk_workspace_bytes(const d2b_segmented_topk_params* p);
D2B_API int d2b_segmented_topk(const d2b_segmented_topk_params* p, void* workspace,
                               size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Batched hard NMS == tf.image.non_max_suppression per segment
 *   lib/layers/nms.py:6-26 (batch_nms), rpn_outputs.py:90, fast_rcnn.py:145,
 *   retinanet.py:353.  IoU in the TF CPU kernel's op order (division form,
 *   strict '>'), candidates ordered (score desc, index asc), scores of -inf/NaN
 *   never selected, stop at max_output_size.
 * boxes [S, n, 4], scores [S, n], optional counts [S] (valid prefix per segment).
 * keep [S, max_output_size] (indices into the segment, selection order, -1 pad).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* boxes;
  const float* scores;
  const int32_t* counts; /* optional */
  int32_t num_segments;
  int32_t n;
  int32_t max_output_size;
  float iou_threshold;
  int32_t* keep;
  int32_t* num_keep; /* [S] */
} d2b_batched_nms_params;
D2B_API size_t d2b_batched_nms_workspace_bytes(const d2b_batched_nms_params* p);
D2B_API int d2b_batched_nms(const d2b_batched_nms_params* p, void* workspace,
                            size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * RPN proposal stage == RPNOutputs.predict_proposals + find_top_rpn_proposals
 *   lib/modeling/proposal_generator/rpn_outputs.py:403-426, 29-132
 * Either `proposals` (already decoded, the reference signature) or
 * `deltas`+`anchors` (decode fused; only the top-k winners are decoded, which
 * is value-identical because decoding is elementwise).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* logits[D2B_MAX_LEVELS];    /* [N, hwa[l]] */
  const float* proposals[D2B_MAX_LEVELS]; /* [N, hwa[l], 4] or NULL */
  const float* deltas[D2B_MAX_LEVELS];    /* [N, hwa[l], 4] or NULL */
  const float* anchors[D2B_MAX_LEVELS];   /* [hwa[l], 4]    or NULL */
  int64_t hwa[D2B_MAX_LEVELS];
  int32_t num_levels;
  int32_t num_images;
  const int32_t* image_shapes; /* [N, 2] (h, w) */
  float nms_thresh;
  int32_t pre_nms_topk;
  int32_t post_nms_topk;
  float min_box_side_len;
  float weights[4]; /* RPN.BBOX_REG_WEIGHTS */
  float scale_clamp;
  float* out_boxes;      /* [N, post, 4] */
  float* out_logits;     /* [N, post] */
  uint8_t* out_valid;    /* [N, post] */
  int32_t* out_num_valid; /* optional [N] */
  int64_t* out_nms_boxes_in; /* optional [1]: total boxes that entered NMS (metric bookkeeping) */
  /* In-kernel anchor synthesis == DefaultAnchorGenerator.grid_anchors (lib/modeling/anchor_generator.py:92-109),
   * used for level l when anchors[l] == NULL:
   *   anchor(y, x, a) = cell_anchors[l][a] + (y*stride, x*stride, y*stride, x*stride),  index = (y*grid_w + x)*A + a */
  const float* cell_anchors[D2B_MAX_LEVELS]; /* [num_cell_anchors[l], 4] or NULL */
  int32_t num_cell_anchors[D2B_MAX_LEVELS];
  int32_t grid_w[D2B_MAX_LEVELS];
  int32_t stride[D2B_MAX_LEVELS];
} d2b_rpn_proposals_params;
D2B_API size_t d2b_rpn_proposals_workspace_bytes(const d2b_rpn_proposals_params* p);
D2B_API int d2b_rpn_proposals(const d2b_rpn_proposals_params* p, void* workspace,
                              size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * fast_rcnn_inference                      lib/modeling/roi_heads/fast_rcnn.py:28-187
 * boxes [M, Kb*4] (Kb = K or 1), scores [M, K+1] (last column = background),
 * indices [M, 2] int64 (image, slot) with dense shape [N, Rmax].
 * Fused decode (FastRCNNOutputs.inference, fast_rcnn.py:359-369, 381-395): with boxes == NULL the predicted boxes are
 * Box2BoxTransform.apply_deltas(deltas [M, Kb*4], proposal_boxes [M, 4]) (box_regression.py:76-123) evaluated where a
 * box is needed -- value-identical to d2b_apply_deltas followed by this call, without the [M, Kb*4] round trip.
 * Index rows may come in any order.  A row with n outside [0, N) or slot outside [0, Rmax) is dropped.  The result
 * is undefined when two rows name the same (image, slot).  As SparseBoxList.to_dense, a slot that no row fills is a
 * row of zeros: with score_thresh < 0 each of its K classes is a candidate with score 0, a zero box and
 * out_roi_index = the slot; with score_thresh >= 0 it never is.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* boxes;
  const float* scores;
  const int64_t* indices;
  int64_t num_preds; /* M */
  int32_t num_images, rmax;
  int32_t num_bbox_reg_classes; /* Kb */
  int32_t num_classes;          /* K */
  const int32_t* image_shapes;  /* [N, 2] */
  float score_thresh, nms_thresh;
  int32_t topk_per_image;
  int32_t nms_cls_agnostic;
  float* out_boxes;       /* [N, topk, 4] */
  float* out_scores;      /* [N, topk] */
  int64_t* out_classes;   /* [N, topk] */
  uint8_t* out_valid;     /* [N, topk] */
  int32_t* out_roi_index; /* optional [N, topk]: slot of the source ROI, -1 pad (kept_indices) */
  int32_t* out_num;       /* optional [N] */
  int64_t* out_nms_boxes_in; /* optional [1] */
  const float* deltas;         /* used when boxes == NULL: [M, Kb*4] (dy, dx, dh, dw) */
  const float* proposal_boxes; /* [M, 4] */
  float weights[4];            /* (wy, wx, wh, ww) */
  float scale_clamp;
} d2b_fast_rcnn_params;
D2B_API size_t d2b_fast_rcnn_postprocess_workspace_bytes(const d2b_fast_rcnn_params* p);
D2B_API int d2b_fast_rcnn_postprocess(const d2b_fast_rcnn_params* p, void* workspace,
                                      size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * RetinaNetHead.inference        lib/modeling/single_stage_heads/retinanet.py:285-387
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* box_cls[D2B_MAX_LEVELS];   /* [N, hwa[l], K] logits */
  const float* box_delta[D2B_MAX_LEVELS]; /* [N, hwa[l], 4] */
  const float* anchors[D2B_MAX_LEVELS];   /* [hwa[l], 4] or NULL (then cell_anchors below) */
  int64_t hwa[D2B_MAX_LEVELS];
  int32_t num_levels, num_images, num_classes;
  int32_t topk_candidates;
  float score_thresh, nms_thresh;
  int32_t max_detections;
  float weights[4];
  float scale_clamp;
  float* out_boxes;     /* [N, max_det, 4] */
  float* out_scores;    /* [N, max_det] */
  int32_t* out_classes; /* [N, max_det] */
  uint8_t* out_valid;   /* [N, max_det] */
  int32_t* out_num;     /* optional [N] */
  int64_t* out_nms_boxes_in; /* optional [1] */
  /* In-kernel anchor synthesis == DefaultAnchorGenerator.grid_anchors (lib/modeling/anchor_generator.py:92-109),
   * used for level l when anchors[l] == NULL:
   *   anchor(y, x, a) = cell_anchors[l][a] + (y*stride, x*stride, y*stride, x*stride),  index = (y*grid_w + x)*A + a */
  const float* cell_anchors[D2B_MAX_LEVELS]; /* [num_cell_anchors[l], 4] or NULL */
  int32_t num_cell_anchors[D2B_MAX_LEVELS];
  int32_t grid_w[D2B_MAX_LEVELS];
  int32_t stride[D2B_MAX_LEVELS];
} d2b_retinanet_params;
D2B_API size_t d2b_retinanet_postprocess_workspace_bytes(const d2b_retinanet_params* p);
D2B_API int d2b_retinanet_postprocess(const d2b_retinanet_params* p, void* workspace,
                                      size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * matrix_nms (SOLOv2)                                   lib/layers/nms.py:29-83
 * masks [B, n, hw] fp32 in {0,1} (B independent images per call; the reference
 * is called once per image inside tf.map_fn, solo_v2.py:587), classes [B, n]
 * int64, scores [B, n] sorted descending, sum_masks [B, n] or NULL.
 * ---------------------------------------------------------------------- */
#define D2B_MNMS_GAUSSIAN 0
#define D2B_MNMS_LINEAR 1
typedef struct {
  const float* masks;
  const int64_t* classes;
  const float* scores;
  const float* sum_masks; /* optional */
  const int32_t* counts;  /* optional [B]: valid prefix length per image (<= n) */
  int32_t batch, n;
  int64_t hw;
  int32_t kernel;
  float sigma;
  float* out; /* [B, n] */
  /* optional [B, n, ceil(hw/64)] bit-packed masks (bit p of word w = pixel 64*w + p), e.g. from
   * d2b_solo_mask_encode: when non-NULL `masks` is ignored and the 4 B/pixel read disappears */
  const uint64_t* packed_masks;
} d2b_matrix_nms_params;
D2B_API size_t d2b_matrix_nms_workspace_bytes(const d2b_matrix_nms_params* p);
D2B_API int d2b_matrix_nms(const d2b_matrix_nms_params* p, void* workspace, size_t workspace_bytes,
                           d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Mask paste-back == reframe_box_masks_to_image_masks   lib/structures/mask_ops.py:7-56
 * (the crop_and_resize-to-full-image + threshold inside detector_postprocess,
 * lib/modeling/postprocessing.py:9-59).  box_masks [M, mh, mw] fp32, boxes [M, 4]
 * absolute yxyx in output-image pixels -> out [M, image_h, image_w] uint8 {0,1}.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* box_masks;
  const float* boxes;
  int64_t num_masks;
  int32_t mask_h, mask_w;
  int32_t image_h, image_w;
  float mask_threshold;
  uint8_t* out; /* [M, image_h, image_w]; optional when out_rle_offsets is set */
  /* Optional COCO run-length encoding of every mask, equal to
   * pycocotools.mask.encode(np.asfortranarray(mask))["counts"] (column-major runs starting with zeros, deltas of
   * counts 3.. against the count two before, 5-bit groups + 48; no terminator; COCO size [image_h, image_w]).
   * out_rle_offsets[0] = 0 and out_rle_offsets[i+1] = out_rle_offsets[i] + length of string i, always complete.
   * String i is written to out_rle + out_rle_offsets[i] iff out_rle_offsets[i+1] <= rle_capacity; nothing is written
   * at or past rle_capacity, so a call with rle_capacity 0 is the sizing query.  The planes are never staged. */
  uint8_t* out_rle;         /* optional [rle_capacity] bytes: the strings of all masks, back to back */
  int64_t rle_capacity;     /* bytes available at out_rle (0 allowed) */
  int64_t* out_rle_offsets; /* optional [num_masks + 1]; non-NULL requests RLE */
  /* Batched mode (num_images > 0): the num_masks = num_images * dets_per_image masks are the dense [N, R] detection
   * slots of detector_postprocess, image-major (mask m belongs to image m / R), and each image's masks are pasted and
   * encoded at that image's own output size.  Only RLE is produced: `out` must be NULL and out_rle_offsets non-NULL;
   * image_h / image_w are ignored.  The capacity contract is the one above.  With input_shapes set the boxes are
   * scaled as detector_postprocess "fixed" does it (per axis scale = (float)((double)out / (double)in), then one fp32
   * multiply per coordinate); NULL takes them as they are ("conventional").  A slot that is not valid, and every slot
   * of an image whose output size has h < 1, w < 1 or h * w >= 2^31 - 65536, encodes as an empty string
   * (offsets[m + 1] == offsets[m]); no pasted mask does, since an all-zero mask is one count.
   * Left 0 / NULL, the op is the single-size one above. */
  int32_t num_images;           /* N; 0 = single-size mode */
  int32_t dets_per_image;       /* R */
  const int32_t* output_shapes; /* [N, 2] (h, w) device: the size of image n's masks and of its RLE `size` */
  const int32_t* input_shapes;  /* optional [N, 2] (h, w) device: the image_shape the boxes refer to */
  const uint8_t* valid;         /* optional [N, R] device: 0 = no detection in this slot */
} d2b_paste_masks_params;
D2B_API size_t d2b_paste_masks_workspace_bytes(const d2b_paste_masks_params* p);
D2B_API int d2b_paste_masks(const d2b_paste_masks_params* p, void* workspace, size_t workspace_bytes,
                            d2b_stream_t stream);

/* ========================================================================
 * SURVEY.md section 8(b) single-stage entry points (thin: same kernels as above)
 * ====================================================================== */

/* ------------------------------------------------------------------------
 * crop_and_resize (single map)                    lib/layers/functional.py:100-166
 * image [N,H,W,C] fp32 NHWC, boxes [M,4] in image pixels, box_ind [M] int32
 * -> out [M, crop_h, crop_w, C].  aligned / pad_border as in the reference.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* image;
  int32_t num_images, height, width, channels;
  const float* boxes;
  const int32_t* box_ind;
  int64_t num_boxes;
  int32_t crop_h, crop_w;
  int32_t aligned, pad_border;
  float* out;
} d2b_crop_and_resize_params;
D2B_API size_t d2b_crop_and_resize_aligned_workspace_bytes(const d2b_crop_and_resize_params* p);
D2B_API int d2b_crop_and_resize_aligned(const d2b_crop_and_resize_params* p, void* workspace,
                                        size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * decode + clip + small-box filter of one RPN level, all images
 *   RPNOutputs.predict_proposals            rpn_outputs.py:403-426
 *   clip_to_window / prune_small_boxes      box_list_ops.py:112-147, 502-517 (rpn_outputs.py:77-86)
 * deltas [N, n, 4], anchors [n, 4] (shared by the images), image_shapes [N,2]
 * -> out_boxes [N, n, 4] (clipped), out_keep [N, n] uint8 (1 = survives the
 *    min_box_side_len filter; all 1 when min_box_side_len <= 0).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* deltas;
  const float* anchors;
  int32_t num_images;
  int64_t n;
  const int32_t* image_shapes;
  float weights[4];
  float scale_clamp;
  float min_box_side_len;
  float* out_boxes;
  uint8_t* out_keep;
} d2b_decode_clip_filter_params;
D2B_API size_t d2b_decode_clip_filter_workspace_bytes(const d2b_decode_clip_filter_params* p);
D2B_API int d2b_decode_clip_filter(const d2b_decode_clip_filter_params* p, void* workspace,
                                   size_t workspace_bytes, d2b_stream_t stream);

/* ========================================================================
 * SURVEY.md section 8(f) "next" row #3: training-side neighbours of the path
 * ====================================================================== */

/* ------------------------------------------------------------------------
 * Box2BoxTransform.get_deltas                 lib/modeling/box_regression.py:38-74
 * src_boxes [n,4], target_boxes [n,4] -> out [n,4] (dy,dx,dh,dw)
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* src_boxes;
  const float* target_boxes;
  int64_t n;
  float weights[4];
  float* out;
} d2b_get_deltas_params;
D2B_API size_t d2b_get_deltas_workspace_bytes(const d2b_get_deltas_params* p);
D2B_API int d2b_get_deltas(const d2b_get_deltas_params* p, void* workspace, size_t workspace_bytes,
                           d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * pairwise_iou                              lib/structures/box_list_ops.py:295-371
 * boxes1 [n1,4], boxes2 [n2,4] -> out [n1, n2].  iou_type: D2B_IOU (:295-334, the matching path),
 * D2B_GIOU / D2B_DIOU / D2B_CIOU (:335-371, the YOLOv4 losses; GIoU keeps the reference's
 * convex_heights * intersect_widths product; CIoU goes through atan: 1e-5 relative, the others are exact).
 * ---------------------------------------------------------------------- */
#define D2B_IOU 0
#define D2B_GIOU 1
#define D2B_DIOU 2
#define D2B_CIOU 3
typedef struct {
  const float* boxes1;
  const float* boxes2;
  int64_t n1, n2;
  float* out;
  int32_t iou_type;
} d2b_pairwise_iou_params;
D2B_API size_t d2b_pairwise_iou_workspace_bytes(const d2b_pairwise_iou_params* p);
D2B_API int d2b_pairwise_iou(const d2b_pairwise_iou_params* p, void* workspace, size_t workspace_bytes,
                             d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Label assignment == pairwise_iou + Matcher fused (the [G, P] matrices are never written)
 *   Matcher.__call__ / get_low_quality_matches_    lib/modeling/matcher.py:57-174
 *   RPNOutputs._get_ground_truth                   rpn_outputs.py:245-304
 *   ROIHeads.label_and_sample_proposals            roi_heads.py:100-165 (up to subsample_labels,
 *                                                  whose tf.random_shuffle has no defined parity)
 * Per image: valid GT list = gt_valid & ~gt_crowd & ~gt_difficult (order kept, boolean_mask),
 * crowd list = gt_crowd, difficult list = gt_difficult.  out_matches indexes the VALID list.
 * Rows >= pred_counts[i]: matches 0, labels -1, deltas 0.
 * ---------------------------------------------------------------------- */
#define D2B_MATCH_MAX_THRESHOLDS 4
#define D2B_MATCH_MAX_GT 1024
typedef struct {
  const float* pred_boxes;     /* [N, P, 4], or [P, 4] when pred_shared (anchors) */
  int32_t pred_shared;
  const int32_t* pred_counts;  /* optional [N]: valid prefix (proposals' is_valid) */
  int32_t num_images;
  int32_t num_preds;           /* P */
  const float* gt_boxes;       /* [N, G, 4] */
  const uint8_t* gt_valid;     /* [N, G] */
  const uint8_t* gt_crowd;     /* optional [N, G] */
  const uint8_t* gt_difficult; /* optional [N, G] */
  int32_t max_gt;              /* G <= D2B_MATCH_MAX_GT */
  float thresholds[D2B_MATCH_MAX_THRESHOLDS]; /* ascending, without the -inf/+inf ends */
  int32_t num_thresholds;
  int32_t labels[D2B_MATCH_MAX_THRESHOLDS + 1]; /* in {-1,0,1} */
  int32_t allow_low_quality_matches;
  float boundary_threshold;    /* < 0: off (rpn_outputs.py:268) */
  const int32_t* image_shapes; /* [N,2], needed when boundary_threshold >= 0 */
  int32_t compute_deltas;      /* 1: out_deltas = get_deltas(pred, matched gt) where label > 0, else 0 */
  float weights[4];
  int64_t* out_matches;        /* [N, P] */
  int64_t* out_labels;         /* [N, P] */
  float* out_deltas;           /* [N, P, 4] or NULL */
} d2b_label_boxes_params;
D2B_API size_t d2b_label_boxes_workspace_bytes(const d2b_label_boxes_params* p);
D2B_API int d2b_label_boxes(const d2b_label_boxes_params* p, void* workspace, size_t workspace_bytes,
                            d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * subsample_labels                                   lib/modeling/sampling.py:6-45
 * (callers: RPNOutputs.losses resample, rpn_outputs.py:315-332; ROIHeads.label_and_sample_proposals,
 * roi_heads.py:181-187).  labels [N, P] int64 with -1 = ignore, bg_label = negative, anything else = positive.
 * Per image: num_pos = min(#positives, max_positives), num_neg = min(#negatives,
 * num_samples - num_pos); the sampled subsets are uniform random subsets in random order, as
 * tf.random_shuffle(x)[:n] gives.  TF's shuffle has no defined bit pattern: the generator here is counter-based
 * (splitmix64 of seed / image / element, see csrc/sampling.cu) and deterministic per seed.
 * ---------------------------------------------------------------------- */
typedef struct {
  const int64_t* labels;  /* [N, P] */
  int32_t num_images;
  int64_t num_labels;     /* P */
  int32_t num_samples;
  int32_t max_positives;  /* int(num_samples * positive_fraction), evaluated by the caller in Python's double
                             arithmetic exactly as sampling.py:37 does (a float product could round across an integer) */
  int64_t bg_label;
  uint64_t seed;
  int64_t* out_pos_idx;   /* optional [N, num_samples], -1 padded */
  int64_t* out_neg_idx;   /* optional [N, num_samples], -1 padded */
  int32_t* out_num_pos;   /* optional [N] */
  int32_t* out_num_neg;   /* optional [N] */
  int64_t* out_labels;    /* optional [N, P]: labels of the sampled elements, -1 elsewhere (the RPN "resample") */
} d2b_subsample_labels_params;
D2B_API size_t d2b_subsample_labels_workspace_bytes(const d2b_subsample_labels_params* p);
D2B_API int d2b_subsample_labels(const d2b_subsample_labels_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Matcher.__call__ on materialised matrices          lib/modeling/matcher.py:57-150
 * match_quality_matrix [num_gt, num_preds]; optional crowd / difficult matrices
 * (use_crowd / use_difficult = "the argument was not None"; zero rows allowed).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* match_quality_matrix;
  const float* crowd_matrix;
  const float* difficult_matrix;
  int32_t num_gt, num_crowd, num_difficult;
  int32_t use_crowd, use_difficult;
  int64_t num_preds;
  float thresholds[D2B_MATCH_MAX_THRESHOLDS];
  int32_t num_thresholds;
  int32_t labels[D2B_MATCH_MAX_THRESHOLDS + 1];
  int32_t allow_low_quality_matches;
  int64_t* out_matches; /* [num_preds] */
  int64_t* out_labels;  /* [num_preds] */
} d2b_matcher_params;
D2B_API size_t d2b_matcher_workspace_bytes(const d2b_matcher_params* p);
D2B_API int d2b_matcher(const d2b_matcher_params* p, void* workspace, size_t workspace_bytes, d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * ROIPooler / ROIAlign backward: gradient w.r.t. the feature maps (what TF
 * autodiff runs in training for poolers.py:134-180: AvgPoolGrad ->
 * CropAndResizeGradImage -> MirrorPadGrad -> per-level scatter).  Boxes get no
 * gradient (functional.py:120 stop_gradient).  grad_features are ACCUMULATED
 * into (zero them first unless summing with another consumer's gradient).
 * `fwd` describes the forward call; its features/out/level_* fields are ignored.
 *
 * deterministic == 0: one kernel, vector fp32 reductions (red.global.add.v4.f32).
 *   The order of the additions depends on scheduling => fp32 tolerance against
 *   the CPU kernel, and two calls may differ in the last bits.  No workspace.
 * deterministic != 0: no floating-point atomics; BIT-IDENTICAL to the CPU kernel
 *   (TF CropAndResizeGradImage + MirrorPadGrad) and to itself from run to run.
 *   Per level and image, a zeroed padded gradient receives, ROI by ROI in input
 *   order, crop row by crop row, column by column, each sample's TL, TR, BL, BR
 *   products; then every padded pixel is added onto clamp(p - pad) in raster
 *   order.  Only pixels of 8x8 tiles that some ROI reaches are written, so a
 *   -0.0 in grad_features elsewhere stays -0.0 (the CPU kernel adds +0.0).
 *   Needs d2b_roi_align_backward_workspace_bytes() of scratch (per-ROI level,
 *   footprint and sample taps, and the ROI lists of each level and image).
 * ---------------------------------------------------------------------- */
typedef struct {
  d2b_roi_align_params fwd;
  const float* grad_out;                 /* [num_rois, output_h, output_w, channels] fp32 */
  float* grad_features[D2B_MAX_LEVELS];  /* level l: [num_images, height[l], width[l], channels] fp32 */
  int32_t deterministic;                 /* 0: atomic scatter (fastest); 1: bit-exact, reproducible order */
} d2b_roi_align_backward_params;
D2B_API size_t d2b_roi_align_backward_workspace_bytes(const d2b_roi_align_backward_params* p);
D2B_API int d2b_roi_align_backward(const d2b_roi_align_backward_params* p, void* workspace,
                                   size_t workspace_bytes, d2b_stream_t stream);

/* ========================================================================
 * SURVEY.md section 8(f) "next" row #4: YOLOv4 post-processing and SOLOv2's point NMS
 * ====================================================================== */

/* ------------------------------------------------------------------------
 * YOLOv4Outputs.inference    lib/modeling/single_stage_heads/yolov4_outputs.py:331-390
 * boxes [N, n, 4], probs [N, n, K] -> per image: max/argmax over classes, score
 * threshold, ONE class-agnostic NMS capped at post_nms_topk, zero-padded outputs.
 * The class is the FIRST maximal one (+0 and -0 compare equal) and the score is its probability.  NaN: TF's
 * reduce_max propagates it, so a box with a NaN probability in any class is never kept, whatever score_thresh.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* boxes;
  const float* probs;
  int32_t num_images;
  int32_t num_boxes;   /* n */
  int32_t num_classes; /* K */
  float score_thresh, nms_thresh;
  int32_t post_nms_topk;
  float* out_boxes;     /* [N, post, 4] */
  float* out_scores;    /* [N, post] */
  int64_t* out_classes; /* [N, post] */
  uint8_t* out_valid;   /* [N, post] */
  int32_t* out_num;     /* optional [N] */
  int64_t* out_nms_boxes_in; /* optional [1] */
} d2b_yolo_params;
D2B_API size_t d2b_yolo_postprocess_workspace_bytes(const d2b_yolo_params* p);
D2B_API int d2b_yolo_postprocess(const d2b_yolo_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * point_nms (kernel_size 2)        lib/modeling/single_stage_heads/solo_v2.py:29-40
 * scores [N, H, W, C] NHWC -> out (same shape): x survives iff it equals the max of its
 * 2x2 window (itself, up, left, up-left; zeros outside the map), else 0.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* scores;
  int32_t num_images, height, width, channels;
  float* out;
} d2b_point_nms_params;
D2B_API size_t d2b_point_nms_workspace_bytes(const d2b_point_nms_params* p);
D2B_API int d2b_point_nms(const d2b_point_nms_params* p, void* workspace, size_t workspace_bytes,
                          d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * SOLOv2 mask stage        lib/modeling/single_stage_heads/solo_v2.py:513-517, 530-533
 *   pred_mask_scores = sigmoid(mask_logits); pred_masks = cast(scores > mask_threshold)
 *   sum_masks = reduce_sum(pred_masks); score_sums = reduce_sum(scores * pred_masks)
 * One streaming read of the logits [B, n, hw]; the masks leave as bit-packed words for
 * d2b_matrix_nms(packed_masks=...), so the fp32 0/1 masks are never materialised.
 * sum_masks is exact; score_sums is an fp32 sum in unspecified order (like tf.reduce_sum).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* mask_logits;
  const int32_t* counts; /* optional [B]: valid prefix per image */
  int32_t batch, n;
  int64_t hw;
  float mask_threshold;
  uint64_t* packed_masks; /* [B, n, ceil(hw/64)] */
  float* sum_masks;       /* [B, n] */
  float* score_sums;      /* [B, n] */
} d2b_solo_mask_encode_params;
D2B_API size_t d2b_solo_mask_encode_workspace_bytes(const d2b_solo_mask_encode_params* p);
D2B_API int d2b_solo_mask_encode(const d2b_solo_mask_encode_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * SOLOv2 dynamic mask generation fused with the mask stage
 *                          lib/modeling/single_stage_heads/solo_v2.py:499-517, 530-533
 *   pred_mask_logits = conv2d(pred_mask_features [1,H,W,E], pred_kernels as [1,1,E,n])   (a GEMM per image)
 *   then exactly d2b_solo_mask_encode: sigmoid -> > mask_threshold -> bit-pack, sum_masks, score_sums.
 * tcgen05 (tf32 x 3 = fp32-accurate) tensor-core kernel whose epilogue emits the packed masks, so the
 * [B, n, hw] fp32 logits are never written (pass mask_logits != NULL only to inspect them).
 * Floating point: a logit differs from the sequential fp32 sum by <= 2e-6 * sum_k |kernel_k * feature_k|
 * (tests/test_solo_dynconv_gpu.py); mask bits can differ only where the logit is that close to logit(threshold).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* mask_features; /* [B, hw, E] NHWC, 16-byte aligned */
  const float* mask_kernels;  /* [B, n, E]: pred_kernels rows gathered by keep_inds (:486) */
  const int32_t* counts;      /* optional [B]: valid prefix per image */
  int32_t batch, n, channels; /* channels = E, a multiple of 4 */
  int64_t hw;
  float mask_threshold;
  uint64_t* packed_masks; /* [B, n, ceil(hw/64)] */
  float* sum_masks;       /* [B, n] */
  float* score_sums;      /* [B, n] */
  float* mask_logits;     /* optional [B, n, hw] */
} d2b_solo_dynamic_masks_params;
D2B_API size_t d2b_solo_dynamic_masks_workspace_bytes(const d2b_solo_dynamic_masks_params* p);
D2B_API int d2b_solo_dynamic_masks(const d2b_solo_dynamic_masks_params* p, void* workspace, size_t workspace_bytes,
                                   d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * SOLOv2Head.inference tail after the dynamic conv          solo_v2.py:507-558
 * Per image b (B images per call, the reference's tf.map_fn at :587): the first counts[b] of the n rows are
 * the candidates that passed the score threshold, in tf.where order.
 *   mask stage (d2b_solo_mask_encode) -> keep sum_masks > strides -> scores *= mask scoring ->
 *   top_k(min(pre_nms_topk, #kept)) -> Matrix-NMS on the packed masks -> keep > update_score_threshold ->
 *   pad / clip to max_detections.
 * Outputs are zero padded.  out_masks (fp32 0/1, the reference's pred_masks before the resize) and
 * out_packed_masks (bit-packed, 1/32 of the bytes) are both optional.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* mask_logits; /* [B, n, hw] */
  const float* scores;      /* [B, n] */
  const int64_t* classes;   /* [B, n] */
  const float* strides;     /* [B, n] */
  const int32_t* counts;    /* optional [B] */
  int32_t batch, n;
  int64_t hw;
  float mask_threshold;
  int32_t pre_nms_topk;
  int32_t kernel; /* D2B_MNMS_* */
  float sigma;
  float update_score_threshold;
  int32_t max_detections;
  float* out_masks;           /* optional [B, max_det, hw] */
  uint64_t* out_packed_masks; /* optional [B, max_det, ceil(hw/64)] */
  int64_t* out_classes;       /* [B, max_det] */
  float* out_scores;          /* [B, max_det] */
  uint8_t* out_valid;         /* [B, max_det] */
  int32_t* out_num;           /* optional [B] */
  /* When mask_logits is NULL the masks come from the dynamic conv (d2b_solo_dynamic_masks) instead: */
  const float* mask_features; /* [B, hw, E] */
  const float* mask_kernels;  /* [B, n, E] */
  int32_t channels;
} d2b_solo_postprocess_params;
D2B_API size_t d2b_solo_postprocess_workspace_bytes(const d2b_solo_postprocess_params* p);
D2B_API int d2b_solo_postprocess(const d2b_solo_postprocess_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * mask_rcnn_inference                  lib/modeling/roi_heads/mask_head.py:71-103
 *   pred_mask_logits [M, Hm, Wm, C] NHWC -> (transpose, gather_nd by pred_classes, sigmoid) -> [M, Hm, Wm]
 * The soft masks `detector_postprocess` pastes (d2b_paste_masks).  C == 1 is the class-agnostic head (the reference
 * indexes channel 1 of 1 there, :98, which TF's GPU gather_nd turns into zeros; channel 0 is used here).  A class
 * outside [0, C) gives sigmoid(0) = 0.5 like TF's GPU gather_nd.
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* mask_logits;
  const int64_t* pred_classes; /* [M] */
  int64_t num_masks;
  int32_t mask_h, mask_w, num_classes;
  float* out; /* [M, Hm, Wm] */
} d2b_mask_rcnn_inference_params;
D2B_API size_t d2b_mask_rcnn_inference_workspace_bytes(const d2b_mask_rcnn_inference_params* p);
D2B_API int d2b_mask_rcnn_inference(const d2b_mask_rcnn_inference_params* p, void* workspace, size_t workspace_bytes,
                                    d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * SOLOv2 candidate selection          lib/modeling/single_stage_heads/solo_v2.py:481-497
 *   keep_inds = tf.where(pred_scores > score_threshold)   (row-major over [cells, classes])
 *   scores = gather_nd(pred_scores, keep_inds); classes = keep_inds[:, 1];
 *   kernels = gather(pred_kernels, keep_inds[:, 0]); strides = gather(cell strides, keep_inds[:, 0])
 * Ordered compaction per image into fixed [B, max_candidates] rows (zero padded) + counts -- the inputs of
 * d2b_solo_postprocess.  The reference has no cap: out_total[b] is the number that passed the threshold, so
 * out_total[b] > max_candidates tells the caller that candidates were dropped (in tf.where order, from the end).
 * ---------------------------------------------------------------------- */
typedef struct {
  const float* scores;       /* [B, G, K] pred_probs of all levels concatenated (:639-655) */
  const float* kernels;      /* [B, G, E] pred_kernels of all levels concatenated; may be NULL if out_kernels is */
  const float* cell_strides; /* [G] stride of the level each cell belongs to (:489-496) */
  int32_t batch, num_cells, num_classes, channels;
  float score_threshold;
  int32_t max_candidates;
  float* out_scores;    /* [B, max_candidates] */
  int64_t* out_classes; /* [B, max_candidates] */
  float* out_strides;   /* [B, max_candidates] */
  float* out_kernels;   /* optional [B, max_candidates, E] */
  int32_t* out_counts;  /* [B] = min(total, max_candidates) */
  int32_t* out_total;   /* optional [B] */
} d2b_solo_select_params;
D2B_API size_t d2b_solo_select_workspace_bytes(const d2b_solo_select_params* p);
D2B_API int d2b_solo_select(const d2b_solo_select_params* p, void* workspace, size_t workspace_bytes,
                            d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * SOLOv2: image-size masks and boxes from the kept masks
 *                          lib/modeling/single_stage_heads/solo_v2.py:599-627
 *   pred_masks = resize_images(pred_masks [N, D, h, w], image_shape) (bilinear)   (:599-601)
 *   pred_masks = cast(pred_masks > mask_threshold)                                (:602)
 *   boxes from masks: mean / where / reduce_min / reduce_max                      (:606-625)
 * resize_images (lib/layers/functional.py:9-36) resolves to tf.compat.v2.image.resize when TensorFlow has it
 * (half-pixel centres; the align_corners kwarg is filtered out) and to tf.image.resize_images(align_corners=True)
 * otherwise: `align_corners` selects the convention.  Input: the bit-packed masks d2b_solo_postprocess emits
 * (rows past the valid count are zero and give empty masks and zero boxes, like the reference's padding).
 * ---------------------------------------------------------------------- */
typedef struct {
  const uint64_t* packed_masks; /* [B, D, ceil(mask_h*mask_w/64)] */
  int32_t batch, num_dets;
  int32_t mask_h, mask_w;
  int32_t image_h, image_w;
  int32_t align_corners; /* 0 = half-pixel centres (tf.compat.v2.image.resize), 1 = align_corners=True (TF 1.13) */
  float mask_threshold;
  uint8_t* out_masks;         /* optional [B, D, image_h, image_w] {0,1} */
  uint64_t* out_packed_masks; /* optional [B, D, ceil(image_h*image_w/64)] */
  float* out_boxes;           /* [B, D, 4] (ymin, xmin, ymax, xmax) */
  /* optional COCO RLE of the B*D image masks (rows past the valid count encode as [image_h * image_w]);
   * same format and contract as d2b_paste_masks_params.out_rle */
  uint8_t* out_rle;         /* optional [rle_capacity] bytes */
  int64_t rle_capacity;     /* bytes available at out_rle (0 allowed) */
  int64_t* out_rle_offsets; /* optional [B*D + 1]; non-NULL requests RLE */
} d2b_solo_upsample_params;
D2B_API size_t d2b_solo_upsample_workspace_bytes(const d2b_solo_upsample_params* p);
D2B_API int d2b_solo_upsample(const d2b_solo_upsample_params* p, void* workspace, size_t workspace_bytes,
                              d2b_stream_t stream);

/* ------------------------------------------------------------------------
 * Final gather of the fixed-size padded per-image outputs to rank 0 (SURVEY.md 8(e); the reference's
 * tf.map_fn stages keep every image independent: rpn_outputs.py:123, fast_rcnn.py:171), done over NVLink
 * PEER MEMORY instead of a library collective: every rank maps one cudaMalloc'd arena of every other rank
 * (CUDA IPC), the sender's pack kernel stores its block straight into rank 0's receive slot and then raises
 * a flag there; rank 0's unpack kernel waits for the flags, scatters the slots into the full-batch tensors
 * and acknowledges into the senders' arenas (so that a sender never overwrites a slot that is still being
 * read).  One launch per rank per step, no host round trip; both launches can be captured in CUDA graphs
 * (the epoch lives in device memory and is advanced by the kernel).
 *
 *   d2b_peer_alloc/free      an arena that can be exported (plain cudaMalloc, zero-filled)
 *   d2b_peer_export/open/close   CUDA IPC handle (D2B_PEER_HANDLE_BYTES opaque bytes) of an arena / its
 *                            mapping in another process of the same node (peer access is enabled lazily)
 *   d2b_peer_copy            the kernel: [wait] -> copy segments -> [signal]
 *
 * d2b_peer_copy: epoch = *epoch_counter + 1.  If num_wait > 0, waits until every wait_flags[i] >=
 * epoch - wait_lag (flags live in THIS GPU's memory; a wait that exceeds timeout_ms sets *error_flag = 1
 * and the kernel goes on, so a lost peer can never hang the GPU; once *error_flag is set later calls do not wait at all).  Then copies every segment (src / dst are
 * device pointers of this GPU or mapped peer memory; any alignment), makes the copies visible system-wide,
 * stores `epoch` into every signal_flags[i] (peer or local memory) and writes *epoch_counter = epoch.
 * `segments`, `wait_flags` pointer values and `signal_flags` are read on the HOST at call time (they travel
 * as kernel parameters); at most D2B_PEER_MAX_SEGMENTS segments and D2B_PEER_MAX_FLAGS flags per call.
 * ---------------------------------------------------------------------- */
#define D2B_PEER_HANDLE_BYTES 64
#define D2B_PEER_MAX_SEGMENTS 112
#define D2B_PEER_MAX_FLAGS 16
typedef struct {
  const void* src;
  void* dst;
  uint64_t bytes;
} d2b_copy_segment;
typedef struct {
  const d2b_copy_segment* segments; /* HOST array */
  int32_t num_segments;
  const uint64_t* const* wait_flags; /* HOST array of device pointers (this GPU's memory) */
  int32_t num_wait;
  int32_t wait_lag;                  /* 0: wait for this epoch (receiver); 1: for the previous one (sender's ack) */
  uint64_t* const* signal_flags;     /* HOST array of device pointers (local or peer memory) */
  int32_t num_signal;
  uint64_t* epoch_counter;           /* device, this GPU; starts at 0 */
  uint32_t* ticket;                  /* device, this GPU; zero; scratch of the kernel */
  int32_t* error_flag;               /* device, this GPU; set to 1 when a wait timed out */
  uint32_t timeout_ms;               /* 0 = 2000 */
} d2b_peer_copy_params;
D2B_API int d2b_peer_alloc(size_t bytes, void** ptr);
D2B_API int d2b_peer_free(void* ptr);
D2B_API int d2b_peer_export(void* ptr, unsigned char handle[D2B_PEER_HANDLE_BYTES]);
D2B_API int d2b_peer_open(const unsigned char handle[D2B_PEER_HANDLE_BYTES], void** ptr);
D2B_API int d2b_peer_close(void* ptr);
D2B_API size_t d2b_peer_copy_workspace_bytes(const d2b_peer_copy_params* p);
D2B_API int d2b_peer_copy(const d2b_peer_copy_params* p, void* workspace, size_t workspace_bytes,
                          d2b_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* D2B200_H_ */
