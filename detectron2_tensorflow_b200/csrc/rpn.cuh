// rpn.cuh -- structures and device helpers shared by the proposal-stage translation units
// (pipelines.cu: the generic launch chain; rpn_fused.cu: the cluster-fused select / sort / decode kernel).
#pragma once
#include "kernels.cuh"

namespace d2b {

typedef unsigned long long u64;

__device__ __forceinline__ u64 make_key(float score, unsigned idx) {
  return ((u64)float_to_key(score) << 32) | (u64)(0xffffffffu - idx);
}
__device__ __forceinline__ unsigned key_index(u64 k) { return 0xffffffffu - (unsigned)k; }

inline int pad_pow2(long long n) {
  int P = 1;
  while (P < n) P <<= 1;
  return P;
}

// Ordered block compaction helper: returns this thread's output slot (or -1) and adds the
// block total to `base` (shared), preserving thread order.  All threads must call it.
template <int THREADS>
__device__ __forceinline__ int block_compact(bool flag, int& base_reg, int* s_warp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned m = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_warp[warp] = __popc(m);
  __syncthreads();
  int before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w) {
    const int c = s_warp[w];
    if (w < warp) before += c;
    total += c;
  }
  const int slot = flag ? base_reg + before + __popc(m & ((1u << lane) - 1u)) : -1;
  base_reg += total;
  __syncthreads();
  return slot;
}

// Anchor of flat index idx: read from the materialised table, or synthesised as
// DefaultAnchorGenerator.grid_anchors does (anchor_generator.py:92-109): cell anchor + integer grid shift.
struct AnchorSrc {
  const float4* table;  // [hwa, 4] or NULL
  const float4* cell;   // [A, 4]
  int A, gw, stride;
  __device__ __forceinline__ float4 at(unsigned idx) const {
    if (table) return __ldg(table + idx);
    const unsigned a = idx % (unsigned)A, cellidx = idx / (unsigned)A;
    const unsigned gx = cellidx % (unsigned)gw, gy = cellidx / (unsigned)gw;
    const float sy = (float)(gy * (unsigned)stride), sx = (float)(gx * (unsigned)stride);
    const float4 c = __ldg(cell + a);
    return make_float4(sy + c.x, sx + c.y, sy + c.z, sx + c.w);
  }
};

struct RpnArgs {
  const float* logits[D2B_MAX_LEVELS];
  const float4* proposals[D2B_MAX_LEVELS];
  const float4* deltas[D2B_MAX_LEVELS];
  AnchorSrc anchors[D2B_MAX_LEVELS];
  long long hwa[D2B_MAX_LEVELS];
  int L, N;
  const int32_t* shapes;
  float min_len;
  float w[4];
  float clampv;
  int k, P, post, P2;
};

// Shared-memory layout of rpn_lazy_merge_kernel (rpn_fused.cu), from sizes the host knows: a level holds at most
// kcap = min(k, row length) candidates and keeps at most min(post, kcap) of them.  Scalars only: the kernel keeps
// the per-level offsets in shared memory (an array here would put the struct in local memory).
struct LazyLayout {
  int R;  // merge-order entries: min(kRpnLazyMaxBlocks * 64, all candidates)
  size_t o_cbox, o_keys, o_order, o_ids, bytes;
};


// One CTA per image: the final per-image top-k (rpn_outputs.py:101-114) as a rank computation.
// Each level's NMS survivors are already ordered (score desc, index asc), so the position of a
// survivor in the sorted concatenation is its own position plus, per other level, the number of
// survivors that precede it -- a binary search over that level's keys.  Ties across levels go to the
// lower concat index, i.e. the earlier level (TF top_k rule).  No sort, no intermediate buffers.
constexpr int kMergeThreads = 1024;
// Body shared by rpn_merge_rank_kernel (pipelines.cu) and the fused sweep + merge kernel (rpn_fused.cu): all
// kMergeThreads threads of the CTA call it for image n; s_keys = dynamic shared memory (P2 keys) when use_smem.
__device__ __forceinline__ void rpn_merge_rank_body(
    const RpnArgs& a, int n, const float4* seg_boxes, const float* seg_scores, const int32_t* keep,
    const int32_t* num_keep, uint32_t* gkeys, uint32_t* s_keys, int use_smem, float4* out_boxes, float* out_logits,
    uint8_t* out_valid, int32_t* out_num) {
  __shared__ int s_off[D2B_MAX_LEVELS + 1];
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l < a.L; ++l) { s_off[l] = acc; acc += __ldcg(num_keep + n * a.L + l); }
    s_off[a.L] = acc;
  }
  __syncthreads();
  D2B_PROF(threadIdx.x == 0, 20);
  const int total = s_off[a.L];
  const int kk = min(total, a.post);  // :105
  uint32_t* gk = use_smem ? s_keys : gkeys + (size_t)n * a.P2;
  constexpr int kPer = 8;  // survivors per thread per sweep: their dependent gathers are issued together
  for (int base = 0; base < total; base += kPer * kMergeThreads) {
    int lv[kPer], pos[kPer];
    float sc[kPer];
    float4 bx[kPer];
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int ci = base + u * kMergeThreads + threadIdx.x;
      lv[u] = 0; pos[u] = 0;
      if (ci < total) {
        int l = 0;
        while (l + 1 < a.L && ci >= s_off[l + 1]) ++l;
        lv[u] = l;
        pos[u] = __ldcg(keep + (size_t)(n * a.L + l) * a.post + (ci - s_off[l]));
      }
    }
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int ci = base + u * kMergeThreads + threadIdx.x;
      if (ci < total) {
        const size_t o = (size_t)(n * a.L + lv[u]) * a.k + pos[u];
        sc[u] = seg_scores[o];
        bx[u] = seg_boxes[o];
      }
    }
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int ci = base + u * kMergeThreads + threadIdx.x;
      if (ci < total) gk[ci] = float_to_key(sc[u]);
    }
    __syncthreads();  // (total <= kPer * kMergeThreads in practice: one sweep; keys of this sweep visible)
    D2B_PROF(threadIdx.x == 0, 21);
    if (base + kPer * kMergeThreads < total) continue;  // multi-sweep: ranks are computed in the second loop
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int ci = base + u * kMergeThreads + threadIdx.x;
      if (ci >= total || total > kPer * kMergeThreads) continue;
      const int l = lv[u];
      const uint32_t key = gk[ci];
      int rank = ci - s_off[l];
      for (int l2 = 0; l2 < a.L; ++l2) {
        if (l2 == l) continue;
        const uint32_t* kl = gk + s_off[l2];
        int lo = 0, hi = s_off[l2 + 1] - s_off[l2];
        while (lo < hi) {  // first position whose element does NOT precede (key, ci)
          const int mid = (lo + hi) >> 1;
          const uint32_t ke = kl[mid];
          const bool before = (l2 < l) ? (ke >= key) : (ke > key);
          if (before) lo = mid + 1; else hi = mid;
        }
        rank += lo;
      }
      if (rank < a.post) {
        const size_t o = (size_t)n * a.post + rank;
        out_boxes[o] = bx[u];
        out_logits[o] = sc[u];
        out_valid[o] = 1;
      }
    }
  }
  D2B_PROF(threadIdx.x == 0, 22);
  if (total > kPer * kMergeThreads) {
    // rare: more survivors than one sweep holds (L * min(post, k) > 8192): straightforward second pass
    __syncthreads();
    for (int ci = threadIdx.x; ci < total; ci += kMergeThreads) {
      int l = 0;
      while (l + 1 < a.L && ci >= s_off[l + 1]) ++l;
      const uint32_t key = gk[ci];
      int rank = ci - s_off[l];
      for (int l2 = 0; l2 < a.L; ++l2) {
        if (l2 == l) continue;
        const uint32_t* kl = gk + s_off[l2];
        int lo = 0, hi = s_off[l2 + 1] - s_off[l2];
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          const uint32_t ke = kl[mid];
          const bool before = (l2 < l) ? (ke >= key) : (ke > key);
          if (before) lo = mid + 1; else hi = mid;
        }
        rank += lo;
      }
      if (rank < a.post) {
        const int row = n * a.L + l;
        const int p2 = __ldcg(keep + (size_t)row * a.post + (ci - s_off[l]));
        const size_t o = (size_t)n * a.post + rank;
        out_boxes[o] = seg_boxes[(size_t)row * a.k + p2];
        out_logits[o] = seg_scores[(size_t)row * a.k + p2];
        out_valid[o] = 1;
      }
    }
  }
  for (int j = kk + threadIdx.x; j < a.post; j += kMergeThreads) {  // zero padding :111-114
    const size_t o = (size_t)n * a.post + j;
    out_boxes[o] = make_float4(0, 0, 0, 0);
    out_logits[o] = 0.0f;
    out_valid[o] = 0;
  }
  if (threadIdx.x == 0 && out_num) out_num[n] = kk;
}


// ---------------------------------------------------------------- fused proposal stage (rpn_fused.cu)
// k <= kRpnFusedMaxK: ONE cluster launch (8 CTAs per row) does top-k select + sort + decode + clip + prune for every
// (image, level) row: seg_boxes / seg_scores [rows, a.k], seg_count [rows] ...
constexpr int kRpnFusedMaxK = 4096;
int rpn_select_fused(const RpnArgs& a, float4* seg_boxes, float* seg_scores, int32_t* seg_count,
                     unsigned long long* nms_in_total, cudaStream_t st);
// ... and ONE cluster launch (one cluster per image, one CTA per level) sweeps every segment's suppression mask and
// merges each image's levels (top `post`, zero padded).  skip (device [N], optional): images with skip[n] != 0 are
// left alone (their clusters return before the first cluster barrier).
int rpn_sweep_merge_fused(const RpnArgs& a, const int32_t* seg_count, const unsigned long long* mask,
                          const float4* seg_boxes, const float* seg_scores, float4* out_boxes, float* out_logits,
                          uint8_t* out_valid, int32_t* out_num, const int32_t* skip, cudaStream_t st);

// Capped walk in merge order (rpn_fused.cu): one CTA per image visits the image's candidates 64 at a time in the order
// of the final merge (score desc, level asc, position asc), tests each only against the kept boxes of its own level,
// and stops at `post` kept.  Same result as per-level NMS + merge: a box's fate depends only on the higher-ranked
// boxes of its level, and a level's survivors past the image's first `post` are never output.
// An image that finishes within kRpnLazyMaxBlocks blocks writes its outputs and done[n] = 1; one that does not writes
// done[n] = 0 and nothing else, and the mask + sweep-merge launches (which skip the finished images) produce it.
// 64 blocks = 4,096 candidates; the bench's inputs need 16 per image, the clustered ones 21-22 (tools/rpn_lazy_visits.py).
constexpr int kRpnLazyMaxBlocks = 64;
// Dynamic shared memory of the walk (keys, merge order, per-level kept boxes); the walk runs when it is at most
// kRpnLazyMaxSmem bytes, else the image goes straight to masks + sweep-merge.
constexpr size_t kRpnLazyMaxSmem = 200 * 1024;
// The walk keeps one SM busy per image for about 140 us (B200, bench inputs; DESIGN.md section 6 breaks it down), longer
// than masks + sweep-merge take for one image on the whole machine (about 40 us), so it only pays when other work
// fills the other SMs: batches of at least kRpnLazyMinImages images (bench.py's 4-image blocks, 4 graphs in flight:
// 0.505 -> 0.451 ms per step).  Smaller batches (a single image: 0.139 -> 0.255 ms for configs[0] with the walk) keep
// masks + sweep-merge.
constexpr int kRpnLazyMinImages = 4;
size_t rpn_lazy_merge_smem(const RpnArgs& a);
int rpn_lazy_merge_fused(const RpnArgs& a, const int32_t* seg_count, const float4* seg_boxes, const float* seg_scores,
                         float thr, float4* out_boxes, float* out_logits, uint8_t* out_valid, int32_t* out_num,
                         int32_t* done, cudaStream_t st);

}  // namespace d2b
