// pipelines.cu -- the three fused post-processing stages, each a fixed chain of
// launches over ALL (image, level) segments with no host synchronisation:
//   d2b_rpn_proposals          rpn_outputs.py:403-426 + 29-132
//   d2b_fast_rcnn_postprocess  fast_rcnn.py:28-187
//   d2b_retinanet_postprocess  retinanet.py:285-387
// The reference runs them as tf.map_fn over images with a CPU NMS per segment.
#include <stdlib.h>

#include "nms.cuh"
#include "rpn.cuh"

namespace d2b {
namespace {

constexpr int kRpnThreads = 1024;

// one CTA per (image, level) row: gather/decode the sorted top-k winners, clip, prune (ordered)
__global__ void __launch_bounds__(kRpnThreads) rpn_decode_kernel(RpnArgs a, const u64* keys, const int32_t* k_r,
                                                                  float4* seg_boxes, float* seg_scores,
                                                                  int32_t* seg_count, u64* nms_in_total) {
  __shared__ int s_warp[kRpnThreads / 32];
  const int row = blockIdx.x;
  const int n = row / a.L, l = row - n * a.L;
  const int kr = k_r[row];
  const float h = (float)a.shapes[2 * n], w = (float)a.shapes[2 * n + 1];
  const size_t rbase = (size_t)n * a.hwa[l];
  int base = 0;
  for (int j0 = 0; j0 < kr; j0 += kRpnThreads) {
    const int j = j0 + threadIdx.x;
    bool ok = false;
    float4 box = make_float4(0, 0, 0, 0);
    float score = 0.0f;
    if (j < kr) {
      const unsigned idx = key_index(keys[(size_t)row * a.P + j]);
      score = __ldg(a.logits[l] + rbase + idx);
      if (a.proposals[l]) box = __ldg(a.proposals[l] + rbase + idx);
      else box = d2b_decode(__ldg(a.deltas[l] + rbase + idx), a.anchors[l].at(idx), a.w[0], a.w[1], a.w[2], a.w[3], a.clampv);
      box = d2b_clip(box, h, w);  // rpn_outputs.py:77-80
      ok = true;
      if (a.min_len > 0.0f) {     // prune_small_boxes, :83-87
        const float bh = box.z - box.x, bw = box.w - box.y;
        ok = (bw >= a.min_len) && (bh >= a.min_len);
      }
    }
    const int slot = block_compact<kRpnThreads>(ok, base, s_warp);
    if (slot >= 0) {
      seg_boxes[(size_t)row * a.k + slot] = box;
      seg_scores[(size_t)row * a.k + slot] = score;
    }
  }
  if (threadIdx.x == 0) {
    seg_count[row] = base;
    if (nms_in_total) atomicAdd(nms_in_total, (u64)base);
  }
}

constexpr int kMergeThreadsLocal = kMergeThreads;
__global__ void __launch_bounds__(kMergeThreads) rpn_merge_rank_kernel(
    RpnArgs a, const float4* seg_boxes, const float* seg_scores, const int32_t* keep, const int32_t* num_keep,
    uint32_t* gkeys, int use_smem, float4* out_boxes, float* out_logits, uint8_t* out_valid, int32_t* out_num) {
  extern __shared__ uint32_t s_keys[];
  rpn_merge_rank_body(a, blockIdx.x, seg_boxes, seg_scores, keep, num_keep, gkeys, s_keys, use_smem, out_boxes,
                      out_logits, out_valid, out_num);
}

struct RpnPlan {
  TopkDesc td;
  RpnArgs a;
  int rows;
  size_t bytes;
  // offsets
  size_t o_topk, o_keys, o_kr, o_boxes, o_scores, o_count, o_keep, o_nkeep, o_nms, o_keys2, o_done;
  bool fused_select;  // k small enough for the cluster-fused select / sort / decode kernel (rpn_fused.cu)
  bool fused_sweep;   // ... and the NMS is the bitmask formulation: column sweep fused with the per-image merge
  bool lazy_merge;    // ... and the capped walk in merge order fits shared memory: masks + sweep only for the images
                      // it does not finish
};

int rpn_plan(const d2b_rpn_proposals_params* p, RpnPlan& pl) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_levels >= 1 && p->num_levels <= D2B_MAX_LEVELS, "num_levels=%d out of range", p->num_levels);
  D2B_REQUIRE(p->num_images >= 0, "num_images must be >= 0");
  D2B_REQUIRE(p->pre_nms_topk >= 1 && p->pre_nms_topk <= kTopkMaxK, "pre_nms_topk=%d out of [1,%d]", p->pre_nms_topk, kTopkMaxK);
  D2B_REQUIRE(p->post_nms_topk >= 1 && p->post_nms_topk <= kTopkMaxK, "post_nms_topk=%d out of [1,%d]", p->post_nms_topk, kTopkMaxK);
  // as tf.image.non_max_suppression; checked here, before the first launch (the walk writes outputs)
  D2B_REQUIRE(p->nms_thresh >= 0.0f && p->nms_thresh <= 1.0f, "nms_thresh must be in [0, 1]");
  RpnArgs& a = pl.a;
  TopkDesc& td = pl.td;
  long long maxlen = 0;
  for (int l = 0; l < D2B_MAX_LEVELS; ++l) {
    const bool in = l < p->num_levels;
    a.logits[l] = in ? p->logits[l] : nullptr;
    a.proposals[l] = in ? reinterpret_cast<const float4*>(p->proposals[l]) : nullptr;
    a.deltas[l] = in ? reinterpret_cast<const float4*>(p->deltas[l]) : nullptr;
    a.anchors[l].table = in ? reinterpret_cast<const float4*>(p->anchors[l]) : nullptr;
    a.anchors[l].cell = in ? reinterpret_cast<const float4*>(p->cell_anchors[l]) : nullptr;
    a.anchors[l].A = in && p->num_cell_anchors[l] > 0 ? p->num_cell_anchors[l] : 1;
    a.anchors[l].gw = in && p->grid_w[l] > 0 ? p->grid_w[l] : 1;
    a.anchors[l].stride = in ? p->stride[l] : 0;
    a.hwa[l] = in ? p->hwa[l] : 0;
    td.scores[l] = a.logits[l];
    td.row_len[l] = a.hwa[l];
    td.k_limit[l] = 0;
    if (in) {
      D2B_REQUIRE(p->hwa[l] >= 0, "hwa[%d] negative", l);
      if (p->num_images > 0 && p->hwa[l] > 0) {
        D2B_REQUIRE(p->logits[l] != nullptr, "logits[%d] is NULL", l);
        D2B_REQUIRE(p->proposals[l] != nullptr ||
                        (p->deltas[l] != nullptr &&
                         (p->anchors[l] != nullptr ||
                          (p->cell_anchors[l] != nullptr && p->num_cell_anchors[l] > 0 && p->grid_w[l] > 0 &&
                           p->hwa[l] % p->num_cell_anchors[l] == 0))),
                    "level %d: need proposals, or deltas + anchors, or deltas + cell_anchors/grid_w/stride", l);
      }
      if (p->hwa[l] > maxlen) maxlen = p->hwa[l];
    }
  }
  a.L = p->num_levels; a.N = p->num_images; a.shapes = p->image_shapes; a.min_len = p->min_box_side_len;
  for (int i = 0; i < 4; ++i) a.w[i] = p->weights[i];
  a.clampv = p->scale_clamp;
  // k = min(pre, longest row): no row can yield more (rpn_outputs.py:67-68)
  a.k = (int)(p->pre_nms_topk < maxlen ? p->pre_nms_topk : (maxlen > 0 ? maxlen : 1));
  a.P = topk_padded_k(a.k);
  a.post = p->post_nms_topk;
  a.P2 = pad_pow2((long long)a.L * (a.post < a.k ? a.post : a.k));
  td.G = a.L; td.rows_per_group = a.N; td.k = a.k; td.transform = D2B_TOPK_IDENTITY;
  pl.rows = a.L * a.N;
  const size_t rows = pl.rows, N = a.N;
  size_t o = 0;
  pl.o_topk = o; o += topk_workspace_bytes(td);
  pl.o_keys = o; o += ws_slice(rows * a.P * sizeof(u64));
  pl.o_kr = o; o += ws_slice(rows * sizeof(int32_t));
  pl.o_boxes = o; o += ws_slice(rows * a.k * sizeof(float4));
  pl.o_scores = o; o += ws_slice(rows * a.k * sizeof(float));
  pl.o_count = o; o += ws_slice(rows * sizeof(int32_t));
  pl.o_keep = o; o += ws_slice(rows * a.post * sizeof(int32_t));
  pl.o_nkeep = o; o += ws_slice(rows * sizeof(int32_t));
  pl.o_nms = o; o += nms_sorted_workspace_bytes(pl.rows, a.k, a.post);
  pl.o_keys2 = o; o += ws_slice(N * a.P2 * sizeof(uint32_t));
  pl.o_done = o; o += ws_slice(N * sizeof(int32_t));  // the last slice: per-image "finished by the walk" flags
  pl.bytes = o;
  // D2B_RPN_GENERIC=1 forces the generic multi-launch chain (tests exercise both paths on the same inputs)
  const char* force_generic = getenv("D2B_RPN_GENERIC");
  pl.fused_select = a.k <= kRpnFusedMaxK && !(force_generic && force_generic[0] == '1');
  pl.fused_sweep = pl.fused_select && nms_uses_bitmask(a.k, a.post) &&
                   ((size_t)a.L * 4 + 2) * (a.post < a.k ? a.post : a.k) + 16 <= 200 * 1024;
  pl.lazy_merge = pl.fused_sweep && a.N >= kRpnLazyMinImages && rpn_lazy_merge_smem(a) <= kRpnLazyMaxSmem;
  return D2B_OK;
}

// =====================================================================================
// detection tail shared by Fast R-CNN and RetinaNet:
//   sorted candidate keys -> class-offset boxes -> NMS -> padded outputs
// =====================================================================================
// The predicted box (pred row i, regression class k) of the Fast R-CNN head: read from `boxes`, or -- fused decode --
// Box2BoxTransform.apply_deltas of (deltas[i, k], proposals[i]) evaluated on the spot (same d2b_decode as
// d2b_apply_deltas: identical bits).
struct FrcnnBoxes {
  const float4* boxes;   // [M, Kb] or NULL
  const float4* deltas;  // [M, Kb]
  const float4* props;   // [M]
  float wy, wx, wh, ww, clampv;
  __device__ __forceinline__ float4 get(long long i, int k, int Kb) const {
    if (boxes) return __ldg(boxes + i * Kb + k);
    return d2b_decode(__ldg(deltas + i * Kb + k), __ldg(props + i), wy, wx, wh, ww, clampv);
  }
};

struct FrcnnFetch {
  FrcnnBoxes boxes;       // [M, Kb]
  const float* scores;    // [M, K+1]
  const int32_t* slot_map;  // [N, Rmax] -> pred row
  const int32_t* shapes;
  int Rmax, Kb, K;
  __device__ __forceinline__ void get(int n, unsigned ci, float4& box, float& score, int& cls, int& roi) const {
    cls = (int)(ci / (unsigned)Rmax);
    roi = (int)(ci - (unsigned)cls * (unsigned)Rmax);
    const int i = slot_map[(size_t)n * Rmax + roi];
    if (i < 0) {  // a slot no index row fills: the zero row of SparseBoxList.to_dense (score_thresh < 0 only)
      box = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      score = 0.0f;
      return;
    }
    const float h = (float)shapes[2 * n], w = (float)shapes[2 * n + 1];
    box = d2b_clip(boxes.get(i, Kb == 1 ? 0 : cls, Kb), h, w);
    score = __ldg(scores + (size_t)i * (K + 1) + cls);
  }
};

struct RetinaFetch {
  const float4* cand_boxes;  // [N, stride]
  const float* cand_scores;
  const int32_t* cand_cls;
  int stride;
  __device__ __forceinline__ void get(int n, unsigned ci, float4& box, float& score, int& cls, int& roi) const {
    const size_t o = (size_t)n * stride + ci;
    box = cand_boxes[o];
    score = cand_scores[o];
    cls = cand_cls[o];
    roi = (int)ci;
  }
};

template <typename F>
__global__ void det_gather_kernel(F f, const u64* keys, const int32_t* count, const float* max_coord, int P,
                                  int stride, int agnostic, float4* nms_boxes, u64* nms_in_total) {
  const int n = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int cnt = min(count[n], stride);
  if (j == 0 && nms_in_total) atomicAdd(nms_in_total, (u64)cnt);
  if (j >= cnt) return;
  float4 box; float score; int cls, roi;
  f.get(n, key_index(keys[(size_t)n * P + j]), box, score, cls, roi);
  if (!agnostic) {  // fast_rcnn.py:141-143 / retinanet.py:349-351: fp32 class offset on every coordinate
    const float mc1 = max_coord[n] + 1.0f;
    const float off = (float)cls * mc1;
    box.x = box.x + off; box.y = box.y + off; box.z = box.z + off; box.w = box.w + off;
  }
  nms_boxes[(size_t)n * stride + j] = box;
}

template <typename F, typename TCls>
__global__ void det_emit_kernel(F f, const u64* keys, int P, const int32_t* keep, const int32_t* num_keep, int topk,
                                float4* out_boxes, float* out_scores, TCls* out_classes, uint8_t* out_valid,
                                int32_t* out_roi, int32_t* out_num) {
  const int n = blockIdx.y;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= topk) return;
  const int nk = num_keep[n];
  if (q == 0 && out_num) out_num[n] = nk;
  float4 box = make_float4(0, 0, 0, 0);
  float score = 0.0f;
  int cls = 0, roi = -1;
  uint8_t valid = 0;
  if (q < nk) {
    const int j = keep[(size_t)n * topk + q];
    f.get(n, key_index(keys[(size_t)n * P + j]), box, score, cls, roi);
    valid = 1;
  }
  const size_t o = (size_t)n * topk + q;
  out_boxes[o] = box;
  out_scores[o] = score;
  out_classes[o] = (TCls)cls;
  out_valid[o] = valid;
  if (out_roi) out_roi[o] = roi;
}

// Gather + capped lazy NMS + emit in ONE launch (one CTA per image): the tail of Fast R-CNN / RetinaNet / YOLOv4
// post-processing when the cap is much smaller than the candidate list (top-100 of thousands).  Candidates are
// visited 64 at a time in (score desc, index asc) order; only the visited blocks are fetched (box gather through
// the head's Fetch functor + fp32 class offset), tested against the kept list and among themselves (exact TF IoU
// rule), and resolved by one warp with the same fixpoint as the bitmask sweep; the loop stops at the cap.  Replaces
// det_gather (all candidates) + nms_lazy + det_emit.
constexpr int kTailThreads = 256;
template <typename F, typename TCls>
__global__ void __launch_bounds__(kTailThreads) det_tail_kernel(F f, const u64* keys, const int32_t* count,
                                                                const float* max_coord, const unsigned* maxkey, int P,
                                                                int stride, int agnostic, int max_out, float thr,
                                                                float4* out_boxes, float* out_scores, TCls* out_classes,
                                                                uint8_t* out_valid, int32_t* out_roi, int32_t* out_num,
                                                                u64* nms_in_total) {
  grid_dep_sync();
  extern __shared__ __align__(16) unsigned char s_tail[];
  float4* s_kept = reinterpret_cast<float4*>(s_tail);          // [max_out] offset boxes of the kept candidates
  int32_t* s_keptj = reinterpret_cast<int32_t*>(s_kept + max_out);  // [max_out] their positions in the sorted list
  __shared__ float4 s_blk[64];
  __shared__ u64 s_diag[64];
  __shared__ unsigned s_dead[2];
  __shared__ int s_kept_n;
  const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const int cnt = min(count[n], stride);
  if (tid == 0) {
    s_kept_n = 0;
    if (nms_in_total) atomicAdd(nms_in_total, (u64)cnt);
  }
  float off1 = 0.0f;  // fast_rcnn.py:141-143 / retinanet.py:349-351: fp32 class offset on every coordinate
  if (!agnostic) off1 = (max_coord ? max_coord[n] : key_to_float(maxkey[n])) + 1.0f;
  __syncthreads();
  const int r = tid & 63, q = tid >> 6;  // candidate r of the block, quarter q of the kept list / columns
  for (int b0 = 0; b0 < cnt; b0 += 64) {
    const int kept = s_kept_n;
    if (kept >= max_out) break;
    const int rows = min(64, cnt - b0);
    if (tid < 64) {
      float4 box = make_float4(0, 0, 0, 0);
      if (tid < rows) {
        float score; int cls, roi;
        f.get(n, key_index(keys[(size_t)n * P + b0 + tid]), box, score, cls, roi);
        if (!agnostic) {
          const float off = (float)cls * off1;
          box.x = box.x + off; box.y = box.y + off; box.z = box.z + off; box.w = box.w + off;
        }
      }
      s_blk[tid] = box;
      s_diag[tid] = 0;
    }
    if (tid < 2) s_dead[tid] = 0;
    __syncthreads();
    const float4 bi = s_blk[r];
    bool dead = false;
    if (r < rows)
      for (int j = q; j < kept; j += kTailThreads / 64)
        if (d2b_iou(bi, s_kept[j]) > thr) { dead = true; break; }
    if (dead) atomicOr(&s_dead[r >> 5], 1u << (r & 31));
    u64 bits = 0;  // bit c of row r: box r suppresses box c (c > r); quarter q covers 16 columns
    if (r < rows)
      for (int c = max(q * 16, r + 1); c < min(q * 16 + 16, rows); ++c)
        if (d2b_iou(bi, s_blk[c]) > thr) bits |= 1ull << c;
    if (bits) atomicOr(&s_diag[r], bits);
    __syncthreads();
    if (tid < 32) {  // warp 0: greedy resolve of the 64 candidates (nms.cuh)
      u64 rem = ((u64)s_dead[1] << 32) | (u64)s_dead[0];
      if (rows < 64) rem |= ~0ull << rows;
      const u64 K = nms_tile_resolve(s_diag[lane], s_diag[lane + 32], rem, max_out - kept);
      const int c = __popcll(K);
      const u64 bitA = 1ull << lane, bitB = 1ull << (lane + 32);
      if (K & bitA) { const int s = kept + __popcll(K & (bitA - 1ull)); s_kept[s] = s_blk[lane]; s_keptj[s] = b0 + lane; }
      if (K & bitB) { const int s = kept + __popcll(K & (bitB - 1ull)); s_kept[s] = s_blk[lane + 32]; s_keptj[s] = b0 + lane + 32; }
      if (lane == 0) s_kept_n = kept + c;
    }
    __syncthreads();
  }
  const int nk = s_kept_n;
  if (tid == 0 && out_num) out_num[n] = nk;
  for (int qo = tid; qo < max_out; qo += kTailThreads) {
    float4 box = make_float4(0, 0, 0, 0);
    float score = 0.0f;
    int cls = 0, roi = -1;
    uint8_t valid = 0;
    if (qo < nk) {
      f.get(n, key_index(keys[(size_t)n * P + s_keptj[qo]]), box, score, cls, roi);
      valid = 1;
    }
    const size_t o = (size_t)n * max_out + qo;
    out_boxes[o] = box;
    out_scores[o] = score;
    out_classes[o] = (TCls)cls;
    out_valid[o] = valid;
    if (out_roi) out_roi[o] = roi;
  }
}

template <typename F, typename TCls>
int det_tail(F f, const u64* keys, const int32_t* count, const float* max_coord, const unsigned* maxkey, int P, int stride,
             int agnostic, int N, int max_out, float thr, float4* out_boxes, float* out_scores, TCls* out_classes,
             uint8_t* out_valid, int32_t* out_roi, int32_t* out_num, u64* nms_in_total, cudaStream_t st) {
  D2B_REQUIRE(thr >= 0.0f && thr <= 1.0f, "iou_threshold must be in [0, 1]");  // as tf.image.non_max_suppression
  const size_t smem = (size_t)max_out * (sizeof(float4) + sizeof(int32_t));
  if (smem > 40 * 1024)
    D2B_CUDA(cudaFuncSetAttribute(det_tail_kernel<F, TCls>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  D2B_CUDA(launch_pdl(det_tail_kernel<F, TCls>, dim3(N), dim3(kTailThreads), smem, st, 0, f, keys, count, max_coord, maxkey,
                      P, stride, agnostic, max_out, thr, out_boxes, out_scores, out_classes, out_valid, out_roi, out_num,
                      nms_in_total));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

// ------------------------------------------------------------------ YOLOv4 front (yolov4_outputs.py:352-360)
struct YoloFetch {
  const float4* boxes;      // [N, n]
  const float* cand_score;  // [N, n] max over classes
  const int32_t* cand_cls;  // [N, n] first argmax
  int n;
  __device__ __forceinline__ void get(int img, unsigned ci, float4& box, float& score, int& cls, int& roi) const {
    const size_t o = (size_t)img * n + ci;
    box = __ldg(boxes + o);
    score = cand_score[o];
    cls = cand_cls[o];
    roi = (int)ci;
  }
};

// One warp per box, lanes stride the K class probabilities (coalesced); the (value, ~class) composite makes the
// warp maximum pick the FIRST maximal class like tf.argmax (+0 and -0 are equal).  NaN ranks above every number:
// TF's Max reduction propagates NaN, so a row holding one has score_max NaN and fails `> thresh` (:352-355).
// Boxes above the threshold append a (score, index) key to their image's candidate list; the segment sort
// restores (score desc, index asc).
__global__ void yolo_prep_kernel(const float* probs, int n, int K, float thresh, int P, u64* keys, int32_t* count,
                                 float* cand_score, int32_t* cand_cls) {
  const int img = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  const float* pr = probs + ((size_t)img * n + i) * K;
  u64 best = 0ull;
  for (int k = lane; k < K; k += 32) {
    const float v = __ldg(pr + k);
    const u64 c = ((u64)(v != v ? 0xffffffffu : float_to_key(v)) << 32) | (u64)(0xffffffffu - (unsigned)k);
    best = c > best ? c : best;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const u64 o = __shfl_xor_sync(0xffffffffu, best, d);
    best = o > best ? o : best;
  }
  if (lane == 0) {
    const int cls = (int)(0xffffffffu - (unsigned)best);
    const float s = __ldg(pr + cls);
    const size_t o = (size_t)img * n + i;
    cand_score[o] = s;
    cand_cls[o] = cls;
    if (s > thresh) {
      const int slot = atomicAdd(count + img, 1);
      keys[(size_t)img * P + slot] = make_key(s, (unsigned)i);
    }
  }
}

// ------------------------------------------------------------------ Fast R-CNN front
// one thread per (prediction row, class): threshold -> candidate key; also the dense slot map
// and max_coord over ALL clipped boxes of the image (fast_rcnn.py:109-116,141).
__global__ void frcnn_prep_kernel(const FrcnnBoxes boxes, const float* scores, const long long* indices, long long M,
                                  int N, int Rmax, int Kb, int K, const int32_t* shapes, float thresh, int P,
                                  u64* keys, int32_t* count, int32_t* slot_map, int* max_coord_bits) {
  grid_dep_sync();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  long long n = -1, r = 0, i = 0;
  int k = 0;
  if (t < M * K) {
    i = t / K;
    k = (int)(t - i * K);
    n = indices[2 * i];
    r = indices[2 * i + 1];
    if (n < 0 || n >= N || r < 0 || r >= Rmax) n = -1;
  }
  int mbits = 0;  // clipped coordinates are >= 0, so their int bit patterns order like the floats
  bool cand = false;
  float s = 0.0f;
  if (n >= 0) {
    if (k == 0) slot_map[n * Rmax + r] = (int32_t)i;
    if (k < Kb) {
      const float h = (float)shapes[2 * n], w = (float)shapes[2 * n + 1];
      const float4 b = d2b_clip(boxes.get(i, k, Kb), h, w);
      mbits = __float_as_int(fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w)));
    }
    s = __ldg(scores + i * (K + 1) + k);
    cand = s > thresh;
  }
  // Block-aggregated atomics when the whole CTA belongs to one image (the common, image-major case): one
  // atomicMax and one atomicAdd per CTA instead of one per warp -- the 16 per-image counters would otherwise
  // serialise ~40k same-address atomics at L2.
  __shared__ long long s_n[8];
  __shared__ int s_max[8], s_cnt[8], s_base;
  const int warp = threadIdx.x >> 5;
  const long long n0 = __shfl_sync(0xffffffffu, n, 0);
  const bool wuni = __all_sync(0xffffffffu, n == n0) && n0 >= 0;
  const int wm = __reduce_max_sync(0xffffffffu, mbits);
  const unsigned cm = __ballot_sync(0xffffffffu, cand);
  if (lane == 0) {
    s_n[warp] = wuni ? n0 : -2;
    s_max[warp] = wm;
    s_cnt[warp] = __popc(cm);
  }
  __syncthreads();
  bool buni = true;
#pragma unroll
  for (int w = 0; w < 8; ++w) buni = buni && (s_n[w] == s_n[0]);
  buni = buni && s_n[0] >= 0;
  if (buni) {
    if (threadIdx.x == 0) {
      int bm = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < 8; ++w) { bm = max(bm, s_max[w]); tot += s_cnt[w]; }
      if (bm > 0) atomicMax(max_coord_bits + s_n[0], bm);
      s_base = tot ? atomicAdd(count + s_n[0], tot) : 0;
    }
    __syncthreads();
    if (cand) {
      int before = 0;
#pragma unroll
      for (int w = 0; w < 8; ++w) before += (w < warp) ? s_cnt[w] : 0;
      const int slot = s_base + before + __popc(cm & ((1u << lane) - 1u));
      if (slot < P) keys[(size_t)n0 * P + slot] = make_key(s, (unsigned)(k * Rmax + (int)r));
    }
  } else if (wuni) {
    int base = 0;
    if (lane == 0) {
      if (wm > 0) atomicMax(max_coord_bits + n0, wm);
      if (cm) base = atomicAdd(count + n0, __popc(cm));
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (cand) {
      const int slot = base + __popc(cm & ((1u << lane) - 1u));
      if (slot < P) keys[(size_t)n0 * P + slot] = make_key(s, (unsigned)(k * Rmax + (int)r));
    }
  } else if (n >= 0) {
    if (mbits > 0) atomicMax(max_coord_bits + n, mbits);
    if (cand) {
      const int slot = atomicAdd(count + n, 1);
      if (slot < P) keys[(size_t)n * P + slot] = make_key(s, (unsigned)(k * Rmax + (int)r));
    }
  }
}

// score_thresh < 0 only, after frcnn_prep_kernel: a slot that no index row fills (slot_map still -1) is a row of
// zeros in SparseBoxList.to_dense (box_list.py:204-246), so each of its K classes scores 0 > thresh with a zero box
// and is a candidate like any other (fast_rcnn.py:119-136).  One thread per (image, slot).
__global__ void frcnn_absent_kernel(const int32_t* slot_map, int N, int Rmax, int K, int P, u64* keys, int32_t* count) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)N * Rmax || slot_map[t] >= 0) return;
  const int n = (int)(t / Rmax), r = (int)(t - (long long)n * Rmax);
  const int base = atomicAdd(count + n, K);
  for (int k = 0; k < K && base + k < P; ++k) keys[(size_t)n * P + base + k] = make_key(0.0f, (unsigned)(k * Rmax + r));
}

// ------------------------------------------------------------------ RetinaNet front
struct RetinaArgs {
  const float4* deltas[D2B_MAX_LEVELS];
  AnchorSrc anchors[D2B_MAX_LEVELS];
  long long hwa[D2B_MAX_LEVELS];
  int L, N, K;
  float thresh;
  float w[4];
  float clampv;
  int k, P, stride, P3;
};
constexpr int kRetThreads = 256;

// Per level keep p > thresh (ordered), decode, append to the image's candidate list.  A level's top-k row is sorted by score, so `p > thresh` (retinanet.py:329-331)
// keeps a PREFIX of it: one binary search per (image, level) gives the kept counts, their scan the offsets of the
// level runs in the image's candidate list, and then every kept candidate is decoded independently
// (grid = chunks x levels x images; a single CTA per image walking the levels in turn took 40 us).
__global__ void retina_offsets_kernel(RetinaArgs a, const u64* keys, const int32_t* k_r, int32_t* lvl_off, int32_t* count,
                                      unsigned* maxkey) {
  const int n = blockIdx.x, lane = threadIdx.x;
  int kept = 0;
  if (lane < a.L) {
    const int row = n * a.L + lane;
    const u64* kk = keys + (size_t)row * a.P;
    int lo = 0, hi = k_r[row];
    while (lo < hi) {  // first j whose score does not pass the threshold
      const int mid = (lo + hi) >> 1;
      if (key_to_float((uint32_t)(kk[mid] >> 32)) > a.thresh) lo = mid + 1; else hi = mid;
    }
    kept = lo;
  }
  int inc = kept;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane < a.L) lvl_off[n * (D2B_MAX_LEVELS + 1) + lane] = inc - kept;
  if (lane == a.L - 1) {
    lvl_off[n * (D2B_MAX_LEVELS + 1) + a.L] = inc;
    count[n] = inc;
    maxkey[n] = float_to_key(__int_as_float(0xff800000));  // -inf: reduce_max of an empty list
  }
}
__global__ void __launch_bounds__(kRetThreads) retina_decode_par_kernel(RetinaArgs a, const u64* keys, const int32_t* lvl_off,
                                                                        float4* cand_boxes, float* cand_scores,
                                                                        int32_t* cand_cls, u64* keys3, unsigned* maxkey) {
  const int n = blockIdx.z, l = blockIdx.y;
  const int off = lvl_off[n * (D2B_MAX_LEVELS + 1) + l];
  const int kept = lvl_off[n * (D2B_MAX_LEVELS + 1) + l + 1] - off;
  const int j = blockIdx.x * kRetThreads + threadIdx.x;
  float mx = __int_as_float(0xff800000);
  if (j < kept) {
    const int row = n * a.L + l;
    const u64 c = keys[(size_t)row * a.P + j];
    const float p = key_to_float((uint32_t)(c >> 32));
    const unsigned idx = key_index(c);
    const unsigned anc = idx / (unsigned)a.K;          // :333
    const int cls = (int)(idx - anc * (unsigned)a.K);  // :334
    const float4 box = d2b_decode(__ldg(a.deltas[l] + (size_t)n * a.hwa[l] + anc), a.anchors[l].at(anc), a.w[0], a.w[1],
                                  a.w[2], a.w[3], a.clampv);
    const int slot = off + j;
    const size_t o = (size_t)n * a.stride + slot;
    cand_boxes[o] = box;
    cand_scores[o] = p;
    cand_cls[o] = cls;
    keys3[(size_t)n * a.P3 + slot] = make_key(p, (unsigned)slot);
    mx = fmaxf(fmaxf(box.x, box.y), fmaxf(box.z, box.w));
  }
  const unsigned any = __ballot_sync(0xffffffffu, j < kept);
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && any) atomicMax(maxkey + n, float_to_key(mx));  // block max (retinanet.py:349)
}
__global__ void retina_maxcoord_kernel(const unsigned* maxkey, int N, float* max_coord) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) max_coord[n] = key_to_float(maxkey[n]);
}

// The candidate list of an image is the concatenation of L runs that are already sorted (each level's top-k is
// emitted score desc / index asc and the threshold keeps a prefix), and the composite keys (score key << 32 | ~slot)
// are unique: the rank of a key in the sorted list is its position in its own run plus, per other run, the number of
// keys greater than it (binary search).  One CTA per image, keys staged in shared memory; replaces the 8192-key
// bitonic sort (73 -> ~10 us at 32 images x 5 x 1000 candidates).  Slots past the count are zeroed like the sort did.
__global__ void __launch_bounds__(1024) retina_merge_rank_kernel(const u64* keys3, const int32_t* lvl_off, int L, int P3,
                                                                 u64* out) {
  extern __shared__ __align__(16) unsigned char s_merge_raw[];
  u64* s_keys = reinterpret_cast<u64*>(s_merge_raw);
  __shared__ int s_off[D2B_MAX_LEVELS + 1];
  const int n = blockIdx.x;
  if (threadIdx.x <= L) s_off[threadIdx.x] = lvl_off[n * (D2B_MAX_LEVELS + 1) + threadIdx.x];
  __syncthreads();
  const int cnt = s_off[L];
  const u64* src = keys3 + (size_t)n * P3;
  u64* dst = out + (size_t)n * P3;
  for (int i = threadIdx.x; i < cnt; i += 1024) s_keys[i] = src[i];
  for (int i = cnt + threadIdx.x; i < P3; i += 1024) dst[i] = 0ull;
  __syncthreads();
  for (int i = threadIdx.x; i < cnt; i += 1024) {
    const u64 key = s_keys[i];
    int rank = 0;
    for (int l = 0; l < L; ++l) {
      const int b = s_off[l], e = s_off[l + 1];
      if (i >= b && i < e) {
        rank += i - b;
      } else {  // keys of run l greater than mine (runs are descending)
        int lo = b, hi = e;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (s_keys[mid] > key) lo = mid + 1; else hi = mid;
        }
        rank += lo - b;
      }
    }
    dst[rank] = key;
  }
}

}  // namespace
}  // namespace d2b

using namespace d2b;

// =====================================================================================
extern "C" size_t d2b_rpn_proposals_workspace_bytes(const d2b_rpn_proposals_params* p) {
  RpnPlan pl;
  if (rpn_plan(p, pl) != D2B_OK) return 0;
  return pl.bytes;
}

extern "C" int d2b_rpn_proposals(const d2b_rpn_proposals_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream) {
  RpnPlan pl;
  int rc = rpn_plan(p, pl);
  if (rc != D2B_OK) return rc;
  if (p->num_images == 0) return D2B_OK;
  D2B_REQUIRE(p->image_shapes && p->out_boxes && p->out_logits && p->out_valid, "rpn_proposals: NULL pointer");
  if (workspace == nullptr || workspace_bytes < pl.bytes) {
    set_last_error("rpn_proposals needs %zu workspace bytes", pl.bytes);
    return D2B_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  const RpnArgs& a = pl.a;
  u64* keys = reinterpret_cast<u64*>(ws + pl.o_keys);
  int32_t* kr = reinterpret_cast<int32_t*>(ws + pl.o_kr);
  float4* seg_boxes = reinterpret_cast<float4*>(ws + pl.o_boxes);
  float* seg_scores = reinterpret_cast<float*>(ws + pl.o_scores);
  int32_t* seg_count = reinterpret_cast<int32_t*>(ws + pl.o_count);
  int32_t* keep = reinterpret_cast<int32_t*>(ws + pl.o_keep);
  int32_t* nkeep = reinterpret_cast<int32_t*>(ws + pl.o_nkeep);
  uint32_t* keys2 = reinterpret_cast<uint32_t*>(ws + pl.o_keys2);
  u64* nms_in = reinterpret_cast<u64*>(p->out_nms_boxes_in);
  if (nms_in) D2B_CUDA(cudaMemsetAsync(nms_in, 0, sizeof(u64), st));

  if (pl.fused_select) {
    // ONE cluster launch: top-k select, sort, decode, clip, prune of every (image, level) row (:67-87)
    rc = rpn_select_fused(a, seg_boxes, seg_scores, seg_count, nms_in, st);
    if (rc != D2B_OK) return rc;
  }
  if (pl.fused_sweep) {
    int32_t* done = nullptr;
    if (pl.lazy_merge) {
      // NMS (:90-94) and merge (:101-114) as one capped walk per image in merge order; the images it does not finish
      // within kRpnLazyMaxBlocks blocks are left to the launches below, which skip the finished ones
      done = reinterpret_cast<int32_t*>(ws + pl.o_done);
      rc = rpn_lazy_merge_fused(a, seg_count, seg_boxes, seg_scores, p->nms_thresh,
                                reinterpret_cast<float4*>(p->out_boxes), p->out_logits, p->out_valid,
                                p->out_num_valid, done, st);
      if (rc != D2B_OK) return rc;
    }
    // suppression masks (:90-94), then ONE launch sweeps every segment and merges each image's levels (:101-114)
    rc = nms_sorted(reinterpret_cast<const float*>(seg_boxes), seg_count, pl.rows, a.k, a.post, p->nms_thresh, keep,
                    nkeep, ws + pl.o_nms, st, /*sweep=*/false, done, a.L);
    if (rc != D2B_OK) return rc;
    return rpn_sweep_merge_fused(a, seg_count, reinterpret_cast<const u64*>(ws + pl.o_nms), seg_boxes, seg_scores,
                                 reinterpret_cast<float4*>(p->out_boxes), p->out_logits, p->out_valid,
                                 p->out_num_valid, done, st);
  }
  if (!pl.fused_select) {
    rc = topk_run(pl.td, keys, nullptr, nullptr, kr, ws + pl.o_topk, st);  // rpn_outputs.py:70
    if (rc != D2B_OK) return rc;
    rpn_decode_kernel<<<pl.rows, kRpnThreads, 0, st>>>(a, keys, kr, seg_boxes, seg_scores, seg_count, nms_in);
    D2B_LAUNCH_CHECK();
  }
  rc = nms_sorted(reinterpret_cast<const float*>(seg_boxes), seg_count, pl.rows, a.k, a.post, p->nms_thresh, keep,
                  nkeep, ws + pl.o_nms, st);  // :90-94
  if (rc != D2B_OK) return rc;
  const size_t merge_smem = (size_t)a.P2 * sizeof(uint32_t);
  const int merge_in_smem = merge_smem <= 160 * 1024;
  if (merge_in_smem) D2B_CUDA(allow_dynamic_smem(rpn_merge_rank_kernel, merge_smem));
  rpn_merge_rank_kernel<<<a.N, kMergeThreads, merge_in_smem ? merge_smem : 0, st>>>(
      a, seg_boxes, seg_scores, keep, nkeep, keys2, merge_in_smem, reinterpret_cast<float4*>(p->out_boxes),
      p->out_logits, p->out_valid, p->out_num_valid);  // :101-114
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

// =====================================================================================
namespace {
struct FrcnnPlan {
  int P, stride;
  size_t bytes, o_keys, o_count, o_slot, o_max, o_nmsb, o_keep, o_nkeep, o_nms;
};
int frcnn_plan(const d2b_fast_rcnn_params* p, FrcnnPlan& pl) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_images >= 0 && p->rmax >= 0 && p->num_preds >= 0, "fast_rcnn: negative sizes");
  D2B_REQUIRE(p->num_classes >= 1, "fast_rcnn: num_classes must be >= 1");
  D2B_REQUIRE(p->num_bbox_reg_classes == 1 || p->num_bbox_reg_classes == p->num_classes,
              "fast_rcnn: boxes must be [M,4] or [M,K*4] (Kb=%d, K=%d)", p->num_bbox_reg_classes, p->num_classes);
  D2B_REQUIRE(p->topk_per_image >= 1, "fast_rcnn: topk_per_image must be >= 1");
  // as tf.image.non_max_suppression; checked here, before the first launch, like the NMS sizes below
  D2B_REQUIRE(p->nms_thresh >= 0.0f && p->nms_thresh <= 1.0f, "nms_thresh must be in [0, 1]");
  const long long cmax = (long long)p->rmax * p->num_classes;
  D2B_REQUIRE(cmax < (1ll << 30), "fast_rcnn: Rmax*K too large");
  pl.stride = (int)(cmax > 0 ? cmax : 1);
  pl.P = pad_pow2(pl.stride);
  const int rc = nms_check_sizes(pl.stride, p->topk_per_image);
  if (rc != D2B_OK) return rc;
  const size_t N = p->num_images;
  size_t o = 0;
  pl.o_keys = o; o += ws_slice(N * pl.P * sizeof(u64));
  pl.o_count = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_slot = o; o += ws_slice(N * (size_t)(p->rmax > 0 ? p->rmax : 1) * sizeof(int32_t));
  pl.o_max = o; o += ws_slice(N * sizeof(float));
  pl.o_nmsb = o; o += ws_slice(N * pl.stride * sizeof(float4));
  pl.o_keep = o; o += ws_slice(N * p->topk_per_image * sizeof(int32_t));
  pl.o_nkeep = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_nms = o; o += nms_sorted_workspace_bytes(p->num_images, pl.stride, p->topk_per_image);
  pl.bytes = o;
  return D2B_OK;
}
}  // namespace

extern "C" size_t d2b_fast_rcnn_postprocess_workspace_bytes(const d2b_fast_rcnn_params* p) {
  FrcnnPlan pl;
  if (frcnn_plan(p, pl) != D2B_OK) return 0;
  return pl.bytes;
}

extern "C" int d2b_fast_rcnn_postprocess(const d2b_fast_rcnn_params* p, void* workspace, size_t workspace_bytes,
                                         d2b_stream_t stream) {
  FrcnnPlan pl;
  int rc = frcnn_plan(p, pl);
  if (rc != D2B_OK) return rc;
  if (p->num_images == 0) return D2B_OK;
  D2B_REQUIRE(p->image_shapes && p->out_boxes && p->out_scores && p->out_classes && p->out_valid,
              "fast_rcnn: NULL pointer");
  D2B_REQUIRE(p->num_preds == 0 || (p->scores && p->indices), "fast_rcnn: NULL input");
  D2B_REQUIRE(p->num_preds == 0 || p->boxes || (p->deltas && p->proposal_boxes),
              "fast_rcnn: either boxes or (deltas, proposal_boxes) must be given");
  const FrcnnBoxes fb{reinterpret_cast<const float4*>(p->boxes), reinterpret_cast<const float4*>(p->deltas),
                      reinterpret_cast<const float4*>(p->proposal_boxes), p->weights[0], p->weights[1], p->weights[2],
                      p->weights[3], p->scale_clamp};
  if (workspace == nullptr || workspace_bytes < pl.bytes) {
    set_last_error("fast_rcnn_postprocess needs %zu workspace bytes", pl.bytes);
    return D2B_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  const int N = p->num_images, T = p->topk_per_image;
  u64* keys = reinterpret_cast<u64*>(ws + pl.o_keys);
  int32_t* count = reinterpret_cast<int32_t*>(ws + pl.o_count);
  int32_t* slot_map = reinterpret_cast<int32_t*>(ws + pl.o_slot);
  float* max_coord = reinterpret_cast<float*>(ws + pl.o_max);
  float4* nms_boxes = reinterpret_cast<float4*>(ws + pl.o_nmsb);
  int32_t* keep = reinterpret_cast<int32_t*>(ws + pl.o_keep);
  int32_t* nkeep = reinterpret_cast<int32_t*>(ws + pl.o_nkeep);
  u64* nms_in = reinterpret_cast<u64*>(p->out_nms_boxes_in);
  if (nms_in) D2B_CUDA(cudaMemsetAsync(nms_in, 0, sizeof(u64), st));
  D2B_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t) * N, st));
  D2B_CUDA(cudaMemsetAsync(max_coord, 0, sizeof(float) * N, st));  // clipped coords are >= 0; padding rows are 0
  // a negative threshold passes the zero scores of the slots no index row fills: mark every slot absent first
  const bool absent_cands = p->score_thresh < 0.0f && p->rmax > 0;
  if (absent_cands) D2B_CUDA(cudaMemsetAsync(slot_map, 0xff, sizeof(int32_t) * N * (size_t)p->rmax, st));
  const long long MK = p->num_preds * p->num_classes;
  if (MK > 0) {
    D2B_CUDA(launch_pdl(frcnn_prep_kernel, dim3((unsigned)((MK + 255) / 256)), dim3(256), 0, st, 0,
        fb, p->scores, reinterpret_cast<const long long*>(p->indices),
        p->num_preds, N, p->rmax, p->num_bbox_reg_classes, p->num_classes, p->image_shapes, p->score_thresh, pl.P,
        keys, count, slot_map, reinterpret_cast<int*>(max_coord)));
    D2B_LAUNCH_CHECK();
  }
  if (absent_cands) {
    const long long NR = (long long)N * p->rmax;
    frcnn_absent_kernel<<<(unsigned)((NR + 255) / 256), 256, 0, st>>>(slot_map, N, p->rmax, p->num_classes, pl.P, keys,
                                                                      count);
    D2B_LAUNCH_CHECK();
  }
  rc = sort_segments_desc(keys, N, pl.P, count, st);
  if (rc != D2B_OK) return rc;
  FrcnnFetch f{fb, p->scores, slot_map, p->image_shapes, p->rmax,
               p->num_bbox_reg_classes, p->num_classes};
  if (nms_lazy_applies(pl.stride, T))  // cap << candidates: gather + NMS + emit in one launch
    return det_tail<FrcnnFetch, int64_t>(f, keys, count, max_coord, nullptr, pl.P, pl.stride, p->nms_cls_agnostic ? 1 : 0, N,
                                         T, p->nms_thresh, reinterpret_cast<float4*>(p->out_boxes), p->out_scores,
                                         p->out_classes, p->out_valid, p->out_roi_index, p->out_num, nms_in, st);
  det_gather_kernel<FrcnnFetch><<<dim3((pl.stride + 255) / 256, N), 256, 0, st>>>(
      f, keys, count, max_coord, pl.P, pl.stride, p->nms_cls_agnostic ? 1 : 0, nms_boxes, nms_in);
  D2B_LAUNCH_CHECK();
  rc = nms_sorted(reinterpret_cast<const float*>(nms_boxes), count, N, pl.stride, T, p->nms_thresh, keep, nkeep,
                  ws + pl.o_nms, st);  // fast_rcnn.py:145-146
  if (rc != D2B_OK) return rc;
  det_emit_kernel<FrcnnFetch, int64_t><<<dim3((T + 127) / 128, N), 128, 0, st>>>(
      f, keys, pl.P, keep, nkeep, T, reinterpret_cast<float4*>(p->out_boxes), p->out_scores, p->out_classes,
      p->out_valid, p->out_roi_index, p->out_num);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

// =====================================================================================
namespace {
struct RetinaPlan {
  TopkDesc td;
  RetinaArgs a;
  int rows;
  size_t bytes, o_topk, o_keys, o_kr, o_cb, o_cs, o_cc, o_keys3, o_keys3b, o_lvl, o_maxkey, o_count, o_max, o_nmsb, o_keep, o_nkeep, o_nms;
};
int retina_plan(const d2b_retinanet_params* p, RetinaPlan& pl) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_levels >= 1 && p->num_levels <= D2B_MAX_LEVELS, "num_levels=%d out of range", p->num_levels);
  D2B_REQUIRE(p->num_images >= 0 && p->num_classes >= 1, "retinanet: bad sizes");
  D2B_REQUIRE(p->topk_candidates >= 1 && p->topk_candidates <= kTopkMaxK, "topk_candidates=%d out of [1,%d]",
              p->topk_candidates, kTopkMaxK);
  D2B_REQUIRE(p->max_detections >= 1, "max_detections must be >= 1");
  // as tf.image.non_max_suppression; checked here, before the first launch, like the NMS sizes below
  D2B_REQUIRE(p->nms_thresh >= 0.0f && p->nms_thresh <= 1.0f, "nms_thresh must be in [0, 1]");
  RetinaArgs& a = pl.a;
  TopkDesc& td = pl.td;
  long long maxhwa = 0;
  for (int l = 0; l < D2B_MAX_LEVELS; ++l) {
    const bool in = l < p->num_levels;
    a.deltas[l] = in ? reinterpret_cast<const float4*>(p->box_delta[l]) : nullptr;
    a.anchors[l].table = in ? reinterpret_cast<const float4*>(p->anchors[l]) : nullptr;
    a.anchors[l].cell = in ? reinterpret_cast<const float4*>(p->cell_anchors[l]) : nullptr;
    a.anchors[l].A = in && p->num_cell_anchors[l] > 0 ? p->num_cell_anchors[l] : 1;
    a.anchors[l].gw = in && p->grid_w[l] > 0 ? p->grid_w[l] : 1;
    a.anchors[l].stride = in ? p->stride[l] : 0;
    a.hwa[l] = in ? p->hwa[l] : 0;
    td.scores[l] = in ? p->box_cls[l] : nullptr;
    td.row_len[l] = in ? p->hwa[l] * p->num_classes : 0;
    td.k_limit[l] = in ? (int)(p->hwa[l] < p->topk_candidates ? p->hwa[l] : p->topk_candidates) : 0;
    if (in) {
      D2B_REQUIRE(p->hwa[l] >= 0 && p->hwa[l] * p->num_classes < (1ll << 32) - 1, "hwa[%d] out of range", l);
      if (p->num_images > 0 && p->hwa[l] > 0)
        D2B_REQUIRE(p->box_cls[l] && p->box_delta[l] &&
                        (p->anchors[l] || (p->cell_anchors[l] && p->num_cell_anchors[l] > 0 && p->grid_w[l] > 0)),
                    "level %d: NULL input", l);
      if (p->hwa[l] > maxhwa) maxhwa = p->hwa[l];
      if (td.k_limit[l] == 0 && p->hwa[l] == 0) td.row_len[l] = 0;
    }
  }
  a.L = p->num_levels; a.N = p->num_images; a.K = p->num_classes; a.thresh = p->score_thresh;
  for (int i = 0; i < 4; ++i) a.w[i] = p->weights[i];
  a.clampv = p->scale_clamp;
  a.k = (int)(p->topk_candidates < maxhwa ? p->topk_candidates : (maxhwa > 0 ? maxhwa : 1));
  a.P = topk_padded_k(a.k);
  a.stride = a.L * a.k;
  a.P3 = pad_pow2(a.stride);
  const int rc = nms_check_sizes(a.stride, p->max_detections);
  if (rc != D2B_OK) return rc;
  td.G = a.L; td.rows_per_group = a.N; td.k = a.k; td.transform = D2B_TOPK_SIGMOID;
  pl.rows = a.L * a.N;
  const size_t rows = pl.rows, N = a.N;
  size_t o = 0;
  pl.o_topk = o; o += topk_workspace_bytes(td);
  pl.o_keys = o; o += ws_slice(rows * a.P * sizeof(u64));
  pl.o_kr = o; o += ws_slice(rows * sizeof(int32_t));
  pl.o_cb = o; o += ws_slice(N * a.stride * sizeof(float4));
  pl.o_cs = o; o += ws_slice(N * a.stride * sizeof(float));
  pl.o_cc = o; o += ws_slice(N * a.stride * sizeof(int32_t));
  pl.o_keys3 = o; o += ws_slice(N * a.P3 * sizeof(u64));
  pl.o_keys3b = o; o += ws_slice(N * a.P3 * sizeof(u64));
  pl.o_lvl = o; o += ws_slice(N * (D2B_MAX_LEVELS + 1) * sizeof(int32_t));
  pl.o_maxkey = o; o += ws_slice(N * sizeof(unsigned));
  pl.o_count = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_max = o; o += ws_slice(N * sizeof(float));
  pl.o_nmsb = o; o += ws_slice(N * a.stride * sizeof(float4));
  pl.o_keep = o; o += ws_slice(N * p->max_detections * sizeof(int32_t));
  pl.o_nkeep = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_nms = o; o += nms_sorted_workspace_bytes(a.N, a.stride, p->max_detections);
  pl.bytes = o;
  return D2B_OK;
}
}  // namespace

extern "C" size_t d2b_retinanet_postprocess_workspace_bytes(const d2b_retinanet_params* p) {
  RetinaPlan pl;
  if (retina_plan(p, pl) != D2B_OK) return 0;
  return pl.bytes;
}

extern "C" int d2b_retinanet_postprocess(const d2b_retinanet_params* p, void* workspace, size_t workspace_bytes,
                                         d2b_stream_t stream) {
  RetinaPlan pl;
  int rc = retina_plan(p, pl);
  if (rc != D2B_OK) return rc;
  if (p->num_images == 0) return D2B_OK;
  D2B_REQUIRE(p->out_boxes && p->out_scores && p->out_classes && p->out_valid, "retinanet: NULL output");
  if (workspace == nullptr || workspace_bytes < pl.bytes) {
    set_last_error("retinanet_postprocess needs %zu workspace bytes", pl.bytes);
    return D2B_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  const RetinaArgs& a = pl.a;
  const int N = a.N, T = p->max_detections;
  u64* keys = reinterpret_cast<u64*>(ws + pl.o_keys);
  int32_t* kr = reinterpret_cast<int32_t*>(ws + pl.o_kr);
  float4* cb = reinterpret_cast<float4*>(ws + pl.o_cb);
  float* cs = reinterpret_cast<float*>(ws + pl.o_cs);
  int32_t* cc = reinterpret_cast<int32_t*>(ws + pl.o_cc);
  u64* keys3 = reinterpret_cast<u64*>(ws + pl.o_keys3);
  int32_t* count = reinterpret_cast<int32_t*>(ws + pl.o_count);
  float* max_coord = reinterpret_cast<float*>(ws + pl.o_max);
  float4* nms_boxes = reinterpret_cast<float4*>(ws + pl.o_nmsb);
  int32_t* keep = reinterpret_cast<int32_t*>(ws + pl.o_keep);
  int32_t* nkeep = reinterpret_cast<int32_t*>(ws + pl.o_nkeep);
  u64* nms_in = reinterpret_cast<u64*>(p->out_nms_boxes_in);
  if (nms_in) D2B_CUDA(cudaMemsetAsync(nms_in, 0, sizeof(u64), st));

  rc = topk_run(pl.td, keys, nullptr, nullptr, kr, ws + pl.o_topk, st);  // retinanet.py:321-326
  if (rc != D2B_OK) return rc;
  int32_t* lvl_off = reinterpret_cast<int32_t*>(ws + pl.o_lvl);
  unsigned* maxkey = reinterpret_cast<unsigned*>(ws + pl.o_maxkey);
  retina_offsets_kernel<<<N, 32, 0, st>>>(a, keys, kr, lvl_off, count, maxkey);
  D2B_LAUNCH_CHECK();
  retina_decode_par_kernel<<<dim3((a.k + kRetThreads - 1) / kRetThreads, a.L, N), kRetThreads, 0, st>>>(
      a, keys, lvl_off, cb, cs, cc, keys3, maxkey);
  D2B_LAUNCH_CHECK();
  const size_t merge_smem = (size_t)a.stride * sizeof(u64);
  if (merge_smem <= 96 * 1024) {  // the per-level runs are sorted already: merge by rank instead of sorting
    D2B_CUDA(allow_dynamic_smem(retina_merge_rank_kernel, merge_smem));
    u64* keys3b = reinterpret_cast<u64*>(ws + pl.o_keys3b);
    retina_merge_rank_kernel<<<N, 1024, merge_smem, st>>>(keys3, lvl_off, a.L, a.P3, keys3b);
    D2B_LAUNCH_CHECK();
    keys3 = keys3b;
  } else {
    rc = sort_segments_desc(keys3, N, a.P3, count, st);
    if (rc != D2B_OK) return rc;
  }
  RetinaFetch f{cb, cs, cc, a.stride};
  if (nms_lazy_applies(a.stride, T))
    return det_tail<RetinaFetch, int32_t>(f, keys3, count, nullptr, maxkey, a.P3, a.stride, 0, N, T, p->nms_thresh,
                                          reinterpret_cast<float4*>(p->out_boxes), p->out_scores, p->out_classes,
                                          p->out_valid, nullptr, p->out_num, nms_in, st);
  retina_maxcoord_kernel<<<(N + 255) / 256, 256, 0, st>>>(maxkey, N, max_coord);
  D2B_LAUNCH_CHECK();
  det_gather_kernel<RetinaFetch><<<dim3((a.stride + 255) / 256, N), 256, 0, st>>>(f, keys3, count, max_coord, a.P3,
                                                                                    a.stride, 0, nms_boxes, nms_in);
  D2B_LAUNCH_CHECK();
  rc = nms_sorted(reinterpret_cast<const float*>(nms_boxes), count, N, a.stride, T, p->nms_thresh, keep, nkeep,
                  ws + pl.o_nms, st);  // :353-355
  if (rc != D2B_OK) return rc;
  det_emit_kernel<RetinaFetch, int32_t><<<dim3((T + 127) / 128, N), 128, 0, st>>>(
      f, keys3, a.P3, keep, nkeep, T, reinterpret_cast<float4*>(p->out_boxes), p->out_scores, p->out_classes,
      p->out_valid, nullptr, p->out_num);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

// =====================================================================================
namespace {
struct YoloPlan {
  int P;
  size_t bytes, o_keys, o_count, o_score, o_cls, o_nmsb, o_keep, o_nkeep, o_nms;
};
int yolo_plan(const d2b_yolo_params* p, YoloPlan& pl) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_images >= 0 && p->num_boxes >= 0, "yolo: negative sizes");
  D2B_REQUIRE(p->num_images <= 65535, "yolo: too many images");
  D2B_REQUIRE(p->num_classes >= 1, "yolo: num_classes must be >= 1");
  D2B_REQUIRE(p->post_nms_topk >= 1, "yolo: post_nms_topk must be >= 1");
  // as tf.image.non_max_suppression; checked here, before the first launch, like the NMS sizes below
  D2B_REQUIRE(p->nms_thresh >= 0.0f && p->nms_thresh <= 1.0f, "nms_thresh must be in [0, 1]");
  D2B_REQUIRE(p->num_boxes < (1 << 30), "yolo: num_boxes too large");
  const size_t N = p->num_images, n = p->num_boxes > 0 ? p->num_boxes : 1;
  pl.P = pad_pow2((long long)n);
  const int rc = nms_check_sizes((int)n, p->post_nms_topk);
  if (rc != D2B_OK) return rc;
  size_t o = 0;
  pl.o_keys = o; o += ws_slice(N * pl.P * sizeof(u64));
  pl.o_count = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_score = o; o += ws_slice(N * n * sizeof(float));
  pl.o_cls = o; o += ws_slice(N * n * sizeof(int32_t));
  pl.o_nmsb = o; o += ws_slice(N * n * sizeof(float4));
  pl.o_keep = o; o += ws_slice(N * p->post_nms_topk * sizeof(int32_t));
  pl.o_nkeep = o; o += ws_slice(N * sizeof(int32_t));
  pl.o_nms = o; o += nms_sorted_workspace_bytes(p->num_images, (int)n, p->post_nms_topk);
  pl.bytes = o;
  return D2B_OK;
}
}  // namespace

extern "C" size_t d2b_yolo_postprocess_workspace_bytes(const d2b_yolo_params* p) {
  YoloPlan pl;
  if (yolo_plan(p, pl) != D2B_OK) return 0;
  return pl.bytes;
}

extern "C" int d2b_yolo_postprocess(const d2b_yolo_params* p, void* workspace, size_t workspace_bytes,
                                    d2b_stream_t stream) {
  YoloPlan pl;
  int rc = yolo_plan(p, pl);
  if (rc != D2B_OK) return rc;
  if (p->num_images == 0) return D2B_OK;
  D2B_REQUIRE(p->out_boxes && p->out_scores && p->out_classes && p->out_valid, "yolo: NULL output");
  D2B_REQUIRE(p->num_boxes == 0 || (p->boxes && p->probs), "yolo: NULL input");
  if (workspace == nullptr || workspace_bytes < pl.bytes) {
    set_last_error("yolo_postprocess needs %zu workspace bytes", pl.bytes);
    return D2B_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  const int N = p->num_images, T = p->post_nms_topk, n = p->num_boxes;
  const int stride = n > 0 ? n : 1;
  u64* keys = reinterpret_cast<u64*>(ws + pl.o_keys);
  int32_t* count = reinterpret_cast<int32_t*>(ws + pl.o_count);
  float* cscore = reinterpret_cast<float*>(ws + pl.o_score);
  int32_t* ccls = reinterpret_cast<int32_t*>(ws + pl.o_cls);
  float4* nms_boxes = reinterpret_cast<float4*>(ws + pl.o_nmsb);
  int32_t* keep = reinterpret_cast<int32_t*>(ws + pl.o_keep);
  int32_t* nkeep = reinterpret_cast<int32_t*>(ws + pl.o_nkeep);
  u64* nms_in = reinterpret_cast<u64*>(p->out_nms_boxes_in);
  if (nms_in) D2B_CUDA(cudaMemsetAsync(nms_in, 0, sizeof(u64), st));
  D2B_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t) * N, st));
  if (n > 0) {
    yolo_prep_kernel<<<dim3((n + 7) / 8, N), 256, 0, st>>>(p->probs, n, p->num_classes, p->score_thresh, pl.P, keys,
                                                           count, cscore, ccls);
    D2B_LAUNCH_CHECK();
  }
  rc = sort_segments_desc(keys, N, pl.P, count, st);
  if (rc != D2B_OK) return rc;
  YoloFetch f{reinterpret_cast<const float4*>(p->boxes), cscore, ccls, stride};
  if (nms_lazy_applies(stride, T))
    return det_tail<YoloFetch, int64_t>(f, keys, count, nullptr, nullptr, pl.P, stride, 1, N, T, p->nms_thresh,
                                        reinterpret_cast<float4*>(p->out_boxes), p->out_scores, p->out_classes,
                                        p->out_valid, nullptr, p->out_num, nms_in, st);
  det_gather_kernel<YoloFetch><<<dim3((stride + 255) / 256, N), 256, 0, st>>>(f, keys, count, nullptr, pl.P, stride,
                                                                               1, nms_boxes, nms_in);
  D2B_LAUNCH_CHECK();
  rc = nms_sorted(reinterpret_cast<const float*>(nms_boxes), count, N, stride, T, p->nms_thresh, keep, nkeep,
                  ws + pl.o_nms, st);  // yolov4_outputs.py:362-364 (class-agnostic)
  if (rc != D2B_OK) return rc;
  det_emit_kernel<YoloFetch, int64_t><<<dim3((T + 127) / 128, N), 128, 0, st>>>(
      f, keys, pl.P, keep, nkeep, T, reinterpret_cast<float4*>(p->out_boxes), p->out_scores, p->out_classes,
      p->out_valid, nullptr, p->out_num);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}
