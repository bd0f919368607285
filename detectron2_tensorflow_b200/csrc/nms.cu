// nms.cu -- batched hard NMS over score-sorted segments (tf.image.non_max_suppression
// semantics: IoU in the TF CPU kernel's division form, strict '>', greedy in
// (score desc, index asc) order, stop at max_output_size).
//
// Two exact formulations, chosen per call:
//  A. bitmask (RPN-sized segments, large cap): all (segment, 64-row block) CTAs
//     compute the upper-triangular IoU>thr matrix as 64-bit words in parallel
//     (phase 1, spread over every SM); one CTA per segment then sweeps 64 rows at
//     a time: the diagonal 64x64 tile is resolved serially from shared memory,
//     the surviving rows are OR-ed by all warps into a shared "removed" word set,
//     and the sweep stops at the cap (phase 2).
//  B. capped lazy sweep (huge candidate lists, small cap: Fast R-CNN / RetinaNet):
//     one CTA per segment keeps the selected boxes in shared memory and, per
//     64-candidate block, tests candidates against the kept list, resolves the
//     diagonal tile with ballots, and exits once `cap` boxes are kept.  Only
//     O(n * kept) IoUs are ever evaluated and no n^2 mask exists.
// Both are latency/dependency-bound rather than HBM-bound (SURVEY.md 8d).
#include "nms.cuh"

namespace d2b {
namespace {

typedef unsigned long long u64;

// ------------------------------------------------------------------ A: bitmask
constexpr int kMaskThreads = 256;

// Canonical box (min/max of the stored corners) + area, as the TF kernel derives them per pair.
// Degenerate boxes (area <= 0) can neither suppress nor be suppressed (IoU := 0): they are replaced
// by an empty sentinel whose intersection with anything is exactly 0.
struct CBox { float ymin, xmin, ymax, xmax, area; };
__device__ __forceinline__ CBox canon(const float4 b, bool live) {
  CBox c;
  c.ymin = fminf(b.x, b.z); c.xmin = fminf(b.y, b.w);
  c.ymax = fmaxf(b.x, b.z); c.xmax = fmaxf(b.y, b.w);
  c.area = (c.ymax - c.ymin) * (c.xmax - c.xmin);
  if (!live || !(c.area > 0.0f)) {
    const float inf = __int_as_float(0x7f800000);
    c.ymin = inf; c.xmin = inf; c.ymax = -inf; c.xmax = -inf; c.area = 0.0f;
  }
  return c;
}

// inter / (area_a + area_b - inter) > thr, decided without the division whenever the comparison is
// not within 1e-6 relative of the threshold (the division result differs from the real quotient by
// at most 2^-24 relative, so outside that band the outcome is certain); exact division otherwise.
__device__ __forceinline__ bool iou_gt(float inter, float area_a, float area_b, float thr) {
  float u = area_a + area_b;
  u = u - inter;
  const float q = thr * u;
  if (u > 1e-30f && q > 1e-30f && u < 1e30f) {
    if (inter > q * 1.000001f) return true;
    if (inter < q * 0.999999f) return false;
  }
  return inter / u > thr;
}

// Pair filter.  IoU > thr implies ih >= thr*max(h_i,h_j) (the intersection cannot be taller than either box and
// inter >= thr*max(area)), and ih <= (h_i+h_j)/2 - |cy_i-cy_j|, hence
//     |cy_i - cy_j| <= (1-thr)*(h_i+h_j)/2 ,   likewise in x,
// i.e. the boxes SHRUNK about their centres to the fraction (1-thr) of their extent must overlap.  Each box carries
// that shrunk interval [c - r, c + r] with r = (1-0.999*thr)*extent/2 * 1.001 + 1e-6*(|lo|+|hi|): slack three orders
// of magnitude above the fp32 rounding of c, r and c +- r, so the filter never rejects a pair the exact rule
// accepts.  The test is four compares on one 16-byte shared load (no arithmetic) and rejects all but a fraction
// of a percent of pairs, so the exact (divergent) IoU evaluation is rare.  Degenerate boxes get an empty interval
// (lo = +inf, hi = -inf: never pass, IoU := 0).
struct FBox { float ylo, xlo, yhi, xhi; };
__device__ __forceinline__ FBox filter_box(const CBox c, float kf) {
  FBox f;
  if (c.area > 0.0f) {
    const float cy = 0.5f * (c.ymin + c.ymax);
    const float cx = 0.5f * (c.xmin + c.xmax);
    const float ry = 0.5f * (1.0f - kf) * (c.ymax - c.ymin) * 1.001f + 1e-6f * (fabsf(c.ymin) + fabsf(c.ymax));
    const float rx = 0.5f * (1.0f - kf) * (c.xmax - c.xmin) * 1.001f + 1e-6f * (fabsf(c.xmin) + fabsf(c.xmax));
    f.ylo = cy - ry; f.yhi = cy + ry;
    f.xlo = cx - rx; f.xhi = cx + rx;
  } else {
    const float inf = __int_as_float(0x7f800000);
    f.ylo = inf; f.xlo = inf; f.yhi = -inf; f.xhi = -inf;
  }
  return f;
}

// grid (ceil(W/2), S, csplit).  mask word (i, w) of a segment (column-word major, nms_mask_index), bit c: box (w*64+c)
// is suppressed by box i (only j > i).
// csplit > 1 (few segments: the latency regime) deals the column blocks of a row block to csplit CTAs.
// skip (optional): segment s is left alone when skip[s / skip_group] != 0 (its CTAs return at entry).
// A CTA handles the 64-row blocks x and nb-1-x of its segment, so every CTA walks nb+1 column blocks (the upper
// triangle is balanced).  8 independent warps per CTA: warp = (column group q, row half); it owns 32 rows of the
// 64-row block and walks column blocks rb+q, rb+q+4, ...  The 64 column boxes of a block are staged in a
// warp-private shared-memory slice (filter record, canonical box, area), so only __syncwarp is needed.
#ifndef D2B_MASK_MINB
#define D2B_MASK_MINB 4  // 64 registers; 1 (98 registers), 5 (48) and 6 (40) measured the same or slower
#endif
__global__ void __launch_bounds__(kMaskThreads, D2B_MASK_MINB) nms_mask_kernel(const float4* boxes, const int32_t* counts, int n,
                                                                 int W, float thr, u64* mask, const int32_t* skip,
                                                                 int skip_group) {
  grid_dep_sync();
  if (skip && skip[blockIdx.y / skip_group]) return;
  __shared__ float4 s_flt[kMaskThreads / 32][64];  // (ylo, xlo, yhi, xhi) of the shrunk box
  __shared__ float4 s_box[kMaskThreads / 32][64];
  __shared__ float s_area[kMaskThreads / 32][64];
  const int seg = blockIdx.y;
  const int cnt = counts ? min(counts[seg], n) : n;
  const int nb = (cnt + 63) >> 6;
  if ((int)blockIdx.x * 2 >= nb) return;
  const float kf = thr * 0.999f;
  const float4* b = boxes + (size_t)seg * n;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = warp >> 1, r = (warp & 1) * 32 + lane;
  for (int side = 0; side < 2; ++side) {
    const int rb = side == 0 ? (int)blockIdx.x : nb - 1 - (int)blockIdx.x;
    if (side == 1 && rb <= (int)blockIdx.x) break;  // odd nb: the middle block is done once
    const int i = rb * 64 + r;
    const bool live = i < cnt;
    const CBox bi = canon(live ? b[i] : make_float4(0, 0, 0, 0), live);
    const FBox fi = filter_box(bi, kf);
    u64* mseg = mask + (size_t)seg * W * 64 * W;  // word (i, cb) at nms_mask_index: lanes = consecutive rows, coalesced
    const int cstep = (kMaskThreads / 64) * (int)gridDim.z;
    int cb = rb + q + (kMaskThreads / 64) * (int)blockIdx.z;
    float4 nxt[2];  // the column boxes of the next visit are loaded one visit ahead
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = cb * 64 + h * 32 + lane;
      nxt[h] = (cb < nb && j < cnt) ? __ldg(b + j) : make_float4(0, 0, 0, 0);
    }
    for (; cb < nb; cb += cstep) {
      const int j0 = cb * 64;
      float4 cur[2] = {nxt[0], nxt[1]};
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = (cb + cstep) * 64 + h * 32 + lane;
        nxt[h] = (cb + cstep < nb && j < cnt) ? __ldg(b + j) : make_float4(0, 0, 0, 0);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = j0 + h * 32 + lane;
        const CBox c = canon(cur[h], j < cnt);
        const FBox f = filter_box(c, kf);
        s_flt[warp][h * 32 + lane] = make_float4(f.ylo, f.xlo, f.yhi, f.xhi);
        s_box[warp][h * 32 + lane] = make_float4(c.ymin, c.xmin, c.ymax, c.xmax);
        s_area[warp][h * 32 + lane] = c.area;
      }
      __syncwarp();
      // (1) branch-free filter over the 64 columns -> candidate bits (fully unrolled: immediates only)
      unsigned clo = 0, chi = 0;
#pragma unroll
      for (int c = 0; c < 64; ++c) {
        const float4 fj = s_flt[warp][c];
        // four predicate-accumulating compares and ONE predicated OR-immediate per column, spelled in PTX: from the C++
        // forms ptxas emits short-circuit predication or select chains (8-9 instructions per pair instead of 6)
        if (c < 32) {
          asm("{\n\t.reg .pred p;\n\tsetp.le.f32 p, %1, %2;\n\tsetp.le.and.f32 p, %3, %4, p;\n\t"
              "setp.le.and.f32 p, %5, %6, p;\n\tsetp.le.and.f32 p, %7, %8, p;\n\t@p or.b32 %0, %0, %9;\n\t}"
              : "+r"(clo)
              : "f"(fj.x), "f"(fi.yhi), "f"(fi.ylo), "f"(fj.z), "f"(fj.y), "f"(fi.xhi), "f"(fi.xlo), "f"(fj.w),
                "r"(1u << (c & 31)));
        } else {
          asm("{\n\t.reg .pred p;\n\tsetp.le.f32 p, %1, %2;\n\tsetp.le.and.f32 p, %3, %4, p;\n\t"
              "setp.le.and.f32 p, %5, %6, p;\n\tsetp.le.and.f32 p, %7, %8, p;\n\t@p or.b32 %0, %0, %9;\n\t}"
              : "+r"(chi)
              : "f"(fj.x), "f"(fi.yhi), "f"(fi.ylo), "f"(fj.z), "f"(fj.y), "f"(fi.xhi), "f"(fi.xlo), "f"(fj.w),
                "r"(1u << (c & 31)));
        }
      }
      u64 cand = ((u64)chi << 32) | clo;
      if (cb == rb) cand &= (r == 63) ? 0ull : (~0ull << (r + 1));  // only j > i
      // (2) exact rule on the rare candidates
      u64 bits = 0;
      while (cand) {
        const int c = __ffsll((long long)cand) - 1;
        cand &= cand - 1;
        const float4 bj = s_box[warp][c];
        const float ih = fmaxf(fminf(bi.ymax, bj.z) - fmaxf(bi.ymin, bj.x), 0.0f);
        const float iw = fmaxf(fminf(bi.xmax, bj.w) - fmaxf(bi.xmin, bj.y), 0.0f);
        const float inter = ih * iw;
        if (iou_gt(inter, s_area[warp][c], bi.area, thr)) bits |= 1ull << c;
      }
      D2B_BOUND(cb, W);
      D2B_BOUND(i, live ? (long long)W * 64 : (long long)i + 1);
      if (live) mseg[nms_mask_index(i, cb, W)] = bits;
      __syncwarp();
    }
  }
}

// Column-owner sweep (nms.cuh) for W <= kColSweepMaxW; one CTA per segment.
__global__ void __launch_bounds__(kColSweepThreads) nms_sweep_cols_kernel(const int32_t* counts, int n, int W,
                                                                           int max_out, const u64* mask,
                                                                           int32_t* keep, int32_t* num_keep) {
  const int seg = blockIdx.x;
  const int cnt = counts ? min(counts[seg], n) : n;
  const int kept = nms_sweep_columns(cnt, W, max_out, mask + (size_t)seg * W * 64 * W, keep + (size_t)seg * max_out);
  if (threadIdx.x == 0) num_keep[seg] = kept;
}

// Long segments (W > kSweepClusterMinW, i.e. more than 8,192 boxes): one CLUSTER of kSweepCluster CTAs per segment.
constexpr int kSweepCluster = 8;
#ifndef D2B_SWEEP_CLUSTER_MINW
#define D2B_SWEEP_CLUSTER_MINW 128  // A/B: one uncapped segment of 16,384 boxes 0.585 -> 0.493 ms; at 32 (n > 2,048) 4,096 boxes get slower
#endif
constexpr int kSweepClusterMinW = D2B_SWEEP_CLUSTER_MINW;
__global__ void __launch_bounds__(kColSweepThreads) nms_sweep_cols_cluster_kernel(const int32_t* counts, int n, int W,
                                                                                   int max_out, const u64* mask,
                                                                                   int32_t* keep, int32_t* num_keep) {
  const int seg = blockIdx.x / kSweepCluster;
  const int cnt = counts ? min(counts[seg], n) : n;
  const int kept = nms_sweep_columns<false, false, kSweepCluster>(cnt, W, max_out, mask + (size_t)seg * W * 64 * W,
                                                                  keep + (size_t)seg * max_out);
  if (threadIdx.x == 0 && blockIdx.x % kSweepCluster == 0) num_keep[seg] = kept;
}

// ------------------------------------------------------------------ A': small segments, everything in one launch
// n <= kSmallMaxN (512) boxes per segment with UNSORTED scores (the stand-alone batch_nms entry): one CTA per segment
// orders the candidates (score desc, index asc; composite keys, bitonic sort in shared memory), gathers the boxes,
// builds the suppression mask in shared memory (same filter + exact rule as nms_mask_kernel), sweeps it with the
// column-owner warps and maps the kept positions back to input indices.  Replaces 7 launches (memset, prep, sort,
// gather, mask, sweep, unmap): at these sizes the chain is pure launch latency.
constexpr int kSmallMaxN = 512;  // beyond this the n^2 / 2 pair tests on ONE SM cost more than the launches saved
__global__ void __launch_bounds__(kColSweepThreads) nms_small_kernel(const float4* boxes, const float* scores,
                                                                      const int32_t* counts, int n, int P, int W,
                                                                      int max_out, float thr, int32_t* keep,
                                                                      int32_t* num_keep) {
  extern __shared__ __align__(16) unsigned char s_small[];
  u64* s_keys = reinterpret_cast<u64*>(s_small);                       // [P]
  float4* s_box = reinterpret_cast<float4*>(s_keys + P);               // [n] canonical (ymin, xmin, ymax, xmax)
  float4* s_flt = s_box + n;                                           // [n] shrunk interval
  float* s_area = reinterpret_cast<float*>(s_flt + n);                 // [n]
  u64* s_mask = reinterpret_cast<u64*>(s_area + ((n + 1) & ~1));       // [n][W]
  __shared__ int s_live;
  const int seg = blockIdx.x, tid = threadIdx.x;
  const int cnt = counts ? min(counts[seg], n) : n;
  if (tid == 0) s_live = 0;
  __syncthreads();
  int mine = 0;
  for (int i = tid; i < P; i += kColSweepThreads) {
    u64 key = 0;
    if (i < cnt) {
      const float s = scores[(size_t)seg * n + i];
      if (s > __int_as_float(0xff800000)) {  // candidates = { i : score > -inf }
        key = ((u64)float_to_key(s) << 32) | (u64)(0xffffffffu - (unsigned)i);
        ++mine;
      }
    }
    s_keys[i] = key;
  }
  if (mine) atomicAdd(&s_live, mine);
  __syncthreads();
  const int live = s_live;
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int p = tid; p < P / 2; p += kColSweepThreads) {
        const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
        const bool desc = ((i & k) == 0);
        const u64 a = s_keys[i], b = s_keys[i | j];
        if (desc ? (a < b) : (a > b)) { s_keys[i] = b; s_keys[i | j] = a; }
      }
      __syncthreads();
    }
  const float kf = thr * 0.999f;
  for (int j = tid; j < live; j += kColSweepThreads) {
    const unsigned idx = 0xffffffffu - (unsigned)s_keys[j];
    const CBox c = canon(boxes[(size_t)seg * n + idx], true);
    const FBox f = filter_box(c, kf);
    s_box[j] = make_float4(c.ymin, c.xmin, c.ymax, c.xmax);
    s_flt[j] = make_float4(f.ylo, f.xlo, f.yhi, f.xhi);
    s_area[j] = c.area;
  }
  __syncthreads();
  // mask words (row i, word w >= i / 64).  A warp works on 32 consecutive rows against the SAME column word, so the
  // column records are broadcast shared-memory loads (rows across lanes against different words would hit one bank)
  const int nb = (live + 63) >> 6;
  for (int w = 0; w < nb; ++w) {
    const int c1 = min(64, live - w * 64);
    const int row_end = min(live, (w + 1) * 64);  // rows of later blocks have no bits in word w
    for (int i = tid; i < row_end; i += kColSweepThreads) {
      const float4 fi = s_flt[i], bi = s_box[i];
      const float ai = s_area[i];
      u64 bits = 0;
      const int cbeg = (w == (i >> 6)) ? (i & 63) + 1 : 0;
#pragma unroll 8
      for (int c = 0; c < 64; ++c) {
        if (c >= cbeg && c < c1) {
          const int j = w * 64 + c;
          const float4 fj = s_flt[j];
          if ((fj.x <= fi.z) && (fi.x <= fj.z) && (fj.y <= fi.w) && (fi.y <= fj.w)) {
            const float4 bj = s_box[j];
            const float ih = fmaxf(fminf(bi.z, bj.z) - fmaxf(bi.x, bj.x), 0.0f);
            const float iw = fmaxf(fminf(bi.w, bj.w) - fmaxf(bi.y, bj.y), 0.0f);
            if (iou_gt(ih * iw, s_area[j], ai, thr)) bits |= 1ull << c;
          }
        }
      }
      s_mask[(size_t)i * W + w] = bits;
    }
  }
  __syncthreads();
  int32_t* kp = keep + (size_t)seg * max_out;
  const int kept = nms_sweep_columns<false, true>(live, W, max_out, s_mask, kp);
  __syncthreads();
  for (int q = tid; q < kept; q += kColSweepThreads) kp[q] = (int32_t)(0xffffffffu - (unsigned)s_keys[kp[q]]);
  if (tid == 0) num_keep[seg] = kept;
}

size_t nms_small_smem(int n, int P) {
  const size_t W = (n + 63) / 64;
  return (size_t)P * 8 + (size_t)n * 32 + (size_t)((n + 1) & ~1) * 4 + (size_t)n * W * 8;
}

// ------------------------------------------------------------------ B: capped lazy sweep
constexpr int kLazyThreads = 256;

__global__ void __launch_bounds__(kLazyThreads) nms_lazy_kernel(const float4* boxes, const int32_t* counts, int n,
                                                                 int max_out, float thr, int32_t* keep,
                                                                 int32_t* num_keep) {
  extern __shared__ float4 s_kept[];  // [max_out]
  __shared__ float4 s_blk[64];
  __shared__ u64 s_diag[64];
  __shared__ unsigned s_dead[2];
  __shared__ int s_kept_n;
  const int seg = blockIdx.x, tid = threadIdx.x;
  const int cnt = counts ? min(counts[seg], n) : n;
  const float4* b = boxes + (size_t)seg * n;
  int32_t* kp = keep + (size_t)seg * max_out;
  if (tid == 0) s_kept_n = 0;
  __syncthreads();
  const int r = tid & 63, q = tid >> 6;  // candidate r of the block, quarter q of the kept list / columns
  for (int b0 = 0; b0 < cnt; b0 += 64) {
    const int kept = s_kept_n;
    if (kept >= max_out) break;
    const int rows = min(64, cnt - b0);
    if (tid < 64) s_blk[tid] = tid < rows ? b[b0 + tid] : make_float4(0, 0, 0, 0);
    if (tid < 2) s_dead[tid] = 0;
    if (tid < 64) s_diag[tid] = 0;
    __syncthreads();
    const float4 bi = s_blk[r];
    // (1) candidate r vs kept list (strided by quarter)
    bool dead = false;
    if (r < rows)
      for (int j = q; j < kept; j += kLazyThreads / 64)
        if (d2b_iou(bi, s_kept[j]) > thr) { dead = true; break; }
    if (dead) atomicOr(&s_dead[r >> 5], 1u << (r & 31));
    // (2) diagonal tile: bit c of row r set if box r suppresses box c (c > r); quarter q covers 16 columns
    u64 bits = 0;
    if (r < rows)
      for (int c = max(q * 16, r + 1); c < min(q * 16 + 16, rows); ++c)
        if (d2b_iou(bi, s_blk[c]) > thr) bits |= 1ull << c;
    if (bits) atomicOr(&s_diag[r], bits);
    __syncthreads();
    // (3) serial resolve by one thread
    if (tid == 0) {
      u64 rem = ((u64)s_dead[1] << 32) | (u64)s_dead[0];
      int k = kept;
      for (int t = 0; t < rows && k < max_out; ++t) {
        if (!((rem >> t) & 1ull)) {
          D2B_BOUND(k, max_out);
          s_kept[k] = s_blk[t];
          kp[k] = b0 + t;
          ++k;
          rem |= s_diag[t];
        }
      }
      s_kept_n = k;
    }
    __syncthreads();
  }
  const int kept = s_kept_n;
  for (int j = kept + tid; j < max_out; j += kLazyThreads) kp[j] = -1;
  if (tid == 0) num_keep[seg] = kept;
}

constexpr int kLazyMaxOut = 8192;      // 128 KB of kept boxes in shared memory
constexpr int kBitmaskMaxN = 65536;    // 32 removed-words per lane

bool use_lazy(int n, int max_out) {
  if (max_out > kLazyMaxOut) return false;
  if (n > kBitmaskMaxN) return true;
  return (long long)max_out * 8 <= n;  // cap much smaller than the candidate list
}

}  // namespace

int nms_check_sizes(int n, int max_out) {
  D2B_REQUIRE(use_lazy(n, max_out) || n <= kBitmaskMaxN,
              "nms: n=%d with max_output_size=%d is not supported (n <= %d or cap <= %d)", n, max_out, kBitmaskMaxN,
              kLazyMaxOut);
  return D2B_OK;
}

size_t nms_sorted_workspace_bytes(int S, int n, int max_out) {
  if (S <= 0 || n <= 0 || use_lazy(n, max_out) || n > kBitmaskMaxN) return 0;
  const size_t W = (n + 63) / 64;
  return ws_slice((size_t)S * W * 64 * W * sizeof(u64));
}

bool nms_lazy_applies(int n, int max_out) { return n > 0 && max_out > 0 && use_lazy(n, max_out); }

bool nms_small_applies(int n) { return n >= 1 && n <= kSmallMaxN; }

int nms_small(const float* boxes, const float* scores, const int32_t* counts, int S, int n, int max_out, float thr,
              int32_t* keep, int32_t* num_keep, cudaStream_t st) {
  D2B_REQUIRE(thr >= 0.0f && thr <= 1.0f, "iou_threshold must be in [0, 1]");  // as tf.image.non_max_suppression
  int P = 2;  // >= 2 keeps the float4 arrays behind the keys 16-byte aligned
  while (P < n) P <<= 1;
  const int W = (n + 63) / 64;
  const size_t smem = nms_small_smem(n, P);
  D2B_CUDA(allow_dynamic_smem(nms_small_kernel, smem));
  nms_small_kernel<<<S, kColSweepThreads, smem, st>>>(reinterpret_cast<const float4*>(boxes), scores, counts, n, P, W,
                                                      max_out, thr, keep, num_keep);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

bool nms_uses_bitmask(int n, int max_out) { return n > 0 && max_out > 0 && !use_lazy(n, max_out); }

int nms_sorted(const float* boxes, const int32_t* counts, int S, int n, int max_out, float thr, int32_t* keep,
               int32_t* num_keep, void* ws, cudaStream_t st, bool sweep, const int32_t* skip, int skip_group) {
  if (S <= 0) return D2B_OK;
  D2B_REQUIRE(max_out >= 0 && n >= 0, "nms: negative sizes");
  D2B_REQUIRE(thr >= 0.0f && thr <= 1.0f, "iou_threshold must be in [0, 1]");  // as tf.image.non_max_suppression
  if (max_out == 0) {
    D2B_CUDA(cudaMemsetAsync(num_keep, 0, sizeof(int32_t) * S, st));
    return D2B_OK;
  }
  if (n == 0) {
    D2B_CUDA(cudaMemsetAsync(num_keep, 0, sizeof(int32_t) * S, st));
    D2B_CUDA(cudaMemsetAsync(keep, 0xff, sizeof(int32_t) * (size_t)S * max_out, st));
    return D2B_OK;
  }
  D2B_REQUIRE(skip == nullptr || (!sweep && skip_group >= 1), "nms: skip flags apply to mask-only calls");
  const float4* b4 = reinterpret_cast<const float4*>(boxes);
  if (use_lazy(n, max_out)) {
    const size_t smem = (size_t)max_out * sizeof(float4);
    D2B_CUDA(allow_dynamic_smem(nms_lazy_kernel, smem));
    nms_lazy_kernel<<<S, kLazyThreads, smem, st>>>(b4, counts, n, max_out, thr, keep, num_keep);
    D2B_LAUNCH_CHECK();
    return D2B_OK;
  }
  const int rc = nms_check_sizes(n, max_out);
  if (rc != D2B_OK) return rc;
  const int W = (n + 63) / 64;
  u64* mask = static_cast<u64*>(ws);
  // few segments: spread a row block's column blocks over up to 4 CTAs so that the grid still fills the SMs
  int csplit = 1;
  while (csplit < 4 && (long long)((W + 1) / 2) * S * csplit * 2 <= 2 * 148 && csplit * 8 < W) csplit *= 2;
  D2B_CUDA(launch_pdl(nms_mask_kernel, dim3((W + 1) / 2, S, csplit), dim3(kMaskThreads), 0, st, 0, b4, counts, n, W, thr,
                      mask, skip, skip_group));
  D2B_LAUNCH_CHECK();
  if (!sweep) return D2B_OK;  // the caller runs its own sweep over the mask (fused with the proposal merge)
  D2B_REQUIRE(W <= kColSweepMaxW, "nms: n=%d too large for the bitmask sweep", n);
  if (W > kSweepClusterMinW) {
    LaunchCfg L(dim3((unsigned)S * kSweepCluster), dim3(kColSweepThreads), 0, st, kSweepCluster);
    L.cfg.numAttrs = 1;  // the cluster dimension only (no programmatic launch for this kernel)
    D2B_CUDA(cudaLaunchKernelEx(&L.cfg, nms_sweep_cols_cluster_kernel, counts, n, W, max_out,
                                static_cast<const u64*>(mask), keep, num_keep));
  } else {
    nms_sweep_cols_kernel<<<S, kColSweepThreads, 0, st>>>(counts, n, W, max_out, mask, keep, num_keep);
  }
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

}  // namespace d2b
