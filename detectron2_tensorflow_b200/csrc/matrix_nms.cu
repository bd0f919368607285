// matrix_nms.cu -- SOLOv2 Matrix-NMS (lib/layers/nms.py:29-83) on bit-packed masks.
//
// The reference flattens n<=500 binary fp32 masks [n, H*W] and runs an SGEMM
// masks @ masks^T (33.6 GFLOP/img at 200x336).  Because the masks are {0,1}, every
// inner product is an exact integer < 2^24, so AND + POPC on bit-packed masks gives
// bit-identical fp32 results:
//   1. pack: ONE streaming read of the fp32 masks (the 134 MB/img that bounds the
//      op) -> u64 words (4.2 MB/img, L2 resident) + exact mask sums.
//   2. pair kernel: one warp per (i<j, same class) pair, AND+POPC over the words.
//   3. column max, decay (shared expf) and column min exactly in the reference's
//      fp32 op order.
// HBM-bound on step 1; no tensor cores (a binary GEMM would be bound by the same read).
#include "kernels.cuh"

namespace d2b {
namespace {

typedef unsigned long long u64;

struct MnmsArgs {
  const float* masks;
  const long long* classes;
  const float* scores;
  const float* sum_in;
  const int32_t* counts;
  int B, n;
  long long hw;
  int Wd;
  int kernel;
  float nsigma;
  u64* packed;      // [B, n, Wd]
  unsigned* isum;   // [B, n] exact popcount
  unsigned* wlo;    // [B, n] ~first / last non-zero word of a packed mask (0 / 0 when the mask is empty; the first
  unsigned* whi;    //        word is kept inverted so that one memset(0) initialises everything and both ends grow by
                    //        atomicMax): a pair's AND + POPC only runs over the intersection of the two ranges
  float* iou;       // [B, n, n]
  float* cmax;      // [B, n]
  float* out;
};

__device__ __forceinline__ int rows_of(const MnmsArgs& a, int b) { return a.counts ? min(a.counts[b], a.n) : a.n; }

// Scalar fallback (hw % 4 != 0): grid (ceil(Wd/8), n, B); 256 threads: warp w packs word (blockIdx.x*8 + w)
__global__ void __launch_bounds__(256) mnms_pack_kernel(MnmsArgs a) {
  const int b = blockIdx.z, i = blockIdx.y;
  if (i >= rows_of(a, b)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int word = blockIdx.x * 8 + warp;
  if (word >= a.Wd) return;
  const float* m = a.masks + ((size_t)b * a.n + i) * a.hw;
  const long long p0 = (long long)word * 64 + lane, p1 = p0 + 32;
  const float v0 = p0 < a.hw ? __ldg(m + p0) : 0.0f;
  const float v1 = p1 < a.hw ? __ldg(m + p1) : 0.0f;
  const unsigned lo = __ballot_sync(0xffffffffu, v0 != 0.0f);
  const unsigned hi = __ballot_sync(0xffffffffu, v1 != 0.0f);
  if (lane == 0) {
    a.packed[((size_t)b * a.n + i) * a.Wd + word] = ((u64)hi << 32) | lo;
    const unsigned c = __popc(lo) + __popc(hi);
    if (c) {
      atomicAdd(a.isum + (size_t)b * a.n + i, c);
      atomicMax(a.wlo + (size_t)b * a.n + i, ~(unsigned)word);
      atomicMax(a.whi + (size_t)b * a.n + i, (unsigned)word);
    }
  }
}

// packed input (d2b_solo_mask_encode): only the exact mask sums are missing; one warp per mask row
__global__ void __launch_bounds__(256) mnms_popc_kernel(MnmsArgs a) {
  grid_dep_sync();
  const int b = blockIdx.y;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= rows_of(a, b)) return;
  const int lane = threadIdx.x & 31;
  const u64* pi = a.packed + ((size_t)b * a.n + i) * a.Wd;
  unsigned c = 0, lo = 0xffffffffu, hi = 0u;
  for (int w = lane; w < a.Wd; w += 32) {
    const u64 v = pi[w];
    c += __popcll(v);
    if (v) { lo = min(lo, (unsigned)w); hi = max(hi, (unsigned)w); }
  }
  for (int o = 16; o > 0; o >>= 1) {
    c += __shfl_xor_sync(0xffffffffu, c, o);
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if (lane == 0) {
    a.isum[(size_t)b * a.n + i] = c;
    a.wlo[(size_t)b * a.n + i] = ~lo;
    a.whi[(size_t)b * a.n + i] = hi;
  }
}

// Vector path (hw % 4 == 0): the one streaming read of the fp32 masks.  A warp packs 2 words per step
// (lane = one float4 = 4 pixels; 16 lanes = 64 pixels = one word) and keeps kPackSteps independent
// 16-byte loads in flight per lane.  grid (ceil(Wd / 128), n, B), 256 threads = 128 words per CTA.
constexpr int kPackSteps = 8;
#ifndef D2B_PACK_MINB
#define D2B_PACK_MINB 1
#endif
__global__ void __launch_bounds__(256, D2B_PACK_MINB) mnms_pack4_kernel(MnmsArgs a) {
  grid_dep_sync();
  const int b = blockIdx.z, i = blockIdx.y;
  if (i >= rows_of(a, b)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float4* m = reinterpret_cast<const float4*>(a.masks + ((size_t)b * a.n + i) * a.hw);
  const long long nvec = a.hw >> 2;
  const int w_first = blockIdx.x * (8 * kPackSteps * 2) + warp * (kPackSteps * 2);
  float4 v[kPackSteps];
#pragma unroll
  for (int s = 0; s < kPackSteps; ++s) {
    const long long q = (long long)(w_first + 2 * s) * 16 + lane;  // float4 index
    v[s] = q < nvec ? __ldcs(m + q) : make_float4(0, 0, 0, 0);
  }
  unsigned total = 0;
#pragma unroll
  for (int s = 0; s < kPackSteps; ++s) {
    const unsigned nib = (v[s].x != 0.0f ? 1u : 0u) | (v[s].y != 0.0f ? 2u : 0u) | (v[s].z != 0.0f ? 4u : 0u) |
                         (v[s].w != 0.0f ? 8u : 0u);
    u64 w = (u64)nib << (4 * (lane & 15));
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) w |= __shfl_xor_sync(0xffffffffu, w, o);
    const int word = w_first + 2 * s + (lane >> 4);
    if ((lane & 15) == 0 && word < a.Wd) {
      a.packed[((size_t)b * a.n + i) * a.Wd + word] = w;
      total += __popcll(w);
    }
  }
  total += __shfl_xor_sync(0xffffffffu, total, 16);
  if (lane == 0 && total) {  // the word range at the granularity of a warp's 16 words (a superset is enough)
    atomicAdd(a.isum + (size_t)b * a.n + i, total);
    atomicMax(a.wlo + (size_t)b * a.n + i, ~(unsigned)w_first);
    atomicMax(a.whi + (size_t)b * a.n + i, (unsigned)min(w_first + 2 * kPackSteps - 1, a.Wd - 1));
  }
}

__device__ __forceinline__ float sum_of(const MnmsArgs& a, int b, int i) {
  return a.sum_in ? a.sum_in[(size_t)b * a.n + i] : (float)a.isum[(size_t)b * a.n + i];
}

// One CTA per row i: each warp takes one of the few columns j > i of the same class and does the AND+POPC
// reduction over the packed words.  Only those entries of the decayed-IoU matrix are ever written: every other
// entry is a known constant (0, or NaN when both masks are empty) that mnms_decay_kernel synthesises instead of
// reading 1 MB per image of zeros.  grid (n, B), 256 threads.
__global__ void __launch_bounds__(256) mnms_iou_kernel(MnmsArgs a, int stage) {
  grid_dep_sync();
  __shared__ int s_match[256];  // columns j > i of row i's class, compacted (the serial class scan was the latency:
  __shared__ int s_nmatch;      // ~60 dependent global loads per warp for ~3 matching columns)
  extern __shared__ u64 s_pi[];  // row i's packed mask: read from L2 once per row instead of once per pair
  const int b = blockIdx.y, i = blockIdx.x;
  const int nb = rows_of(a, b);
  if (i >= nb) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_nmatch = 0;
  const float si = sum_of(a, b, i);
  const long long ci = a.classes[(size_t)b * a.n + i];
  float* row = a.iou + ((size_t)b * a.n + i) * a.n;
  const u64* pi = a.packed + ((size_t)b * a.n + i) * a.Wd;
  __syncthreads();
  for (int j0 = i + 1; j0 < nb; j0 += 256) {  // all same-class columns in rounds of up to 256 matches
    const int j = j0 + threadIdx.x;
    if (j < nb && a.classes[(size_t)b * a.n + j] == ci) {
      const int s = atomicAdd(&s_nmatch, 1);
      if (s < 256) s_match[s] = j;
    }
  }
  __syncthreads();
  const int nmatch = s_nmatch;
  if (nmatch == 0) return;
  const unsigned lo_i = ~a.wlo[(size_t)b * a.n + i], hi_i = a.whi[(size_t)b * a.n + i];  // non-zero words of row i
  if (stage && nmatch > 0 && nmatch <= 256) {
    for (int w = (int)lo_i + threadIdx.x; w <= (int)hi_i && lo_i != 0xffffffffu; w += 256) {
      D2B_BOUND(w, a.Wd);
      s_pi[w] = pi[w];
    }
    __syncthreads();  // (block-uniform condition)
  }
  if (nmatch > 256) {  // (more than 256 same-class columns: the plain scan)
    for (int j = i + 1 + warp; j < nb; j += 8) {
      if (a.classes[(size_t)b * a.n + j] != ci) continue;  // warp-uniform
      const u64* pj = a.packed + ((size_t)b * a.n + j) * a.Wd;
      unsigned c = 0;
      const unsigned lo = max(lo_i, ~a.wlo[(size_t)b * a.n + j]), hi = min(hi_i, a.whi[(size_t)b * a.n + j]);
      if (lo != 0xffffffffu)
        for (int w = (int)lo + lane; w <= (int)hi; w += 32) c += __popcll(pi[w] & pj[w]);
      for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
      if (lane == 0) {
        const float inter = (float)c;
        float u = sum_of(a, b, j) + si;  // nms.py:51-52
        u = u - inter;
        const float v = inter / u;  // :54
        row[j] = v;
        if (v == v) atomicMax(reinterpret_cast<int*>(a.cmax) + (size_t)b * a.n + j, __float_as_int(v));
      }
    }
    return;
  }
  for (int m = warp; m < nmatch; m += 8) {
    const int j = s_match[m];
    const u64* pj = a.packed + ((size_t)b * a.n + j) * a.Wd;
    unsigned c = 0;
    // only the words where BOTH masks can be non-zero (an object covers a band of rows: ~10 % of the words)
    const unsigned lo = max(lo_i, ~a.wlo[(size_t)b * a.n + j]), hi = min(hi_i, a.whi[(size_t)b * a.n + j]);
    const int w_end = lo == 0xffffffffu ? 0 : (int)hi + 1;
    for (int w0 = lo == 0xffffffffu ? 0 : (int)lo; w0 < w_end; w0 += 32 * 8) {  // 8 independent loads in flight per lane
      u64 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int w = w0 + u * 32 + lane;
        v[u] = w < w_end ? __ldg(pj + w) : 0ull;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int w = w0 + u * 32 + lane;
        D2B_BOUND(w < w_end ? w : 0, a.Wd);
        if (w < w_end) c += __popcll((stage ? s_pi[w] : pi[w]) & v[u]);
      }
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) {
      const float inter = (float)c;
      float u = sum_of(a, b, j) + si;  // nms.py:51-52
      u = u - inter;
      const float v = inter / u;  // :54
      row[j] = v;
      // column maximum (compensate_iou, :67) on the fly: IoUs are >= +0, so the int order of the bits is the float
      // order; every entry this kernel does not compute is 0 (or NaN, see cmax_of)
      if (v == v) atomicMax(reinterpret_cast<int*>(a.cmax) + (size_t)b * a.n + j, __float_as_int(v));
    }
  }
}

// compensate_iou = reduce_max(iou, axis=0) (:67) without a pass over the matrix.  With `(v > m) ? v : m` semantics
// (NaNs skipped unless row 0's entry is NaN) column i of the decayed-IoU matrix has: NaN entries exactly where both
// masks are empty (0 / 0), zeros elsewhere outside the same-class upper triangle, and the pair IoUs inside it.  Hence
// max = NaN when mask i and mask 0 are both empty, else max(0, pair IoUs) = what mnms_iou_kernel accumulated.
__device__ __forceinline__ float cmax_of(const MnmsArgs& a, int b, int i) {
  const float u = sum_of(a, b, i) + sum_of(a, b, 0);
  return (u == 0.0f) ? __int_as_float(0x7fc00000) : a.cmax[(size_t)b * a.n + i];
}

// decay + reduce_min(axis=0) + score update (:72-82), `(d < m) ? d : m` semantics (NaN never enters the minimum, so
// the order of the reduction is free).  CTA = 32 columns: lane = column (coalesced 128-byte rows of the matrix),
// the 32 warps split the rows (4 loads in flight each), partial minima meet in shared memory.
constexpr int kDecayWarps = 32;
constexpr int kDecayStageMax = 4096;  // rows whose per-row values fit the shared-memory table (20 bytes each)

__device__ __forceinline__ float decay_of(const MnmsArgs& a, float v, float ci) {
  if (a.kernel == D2B_MNMS_GAUSSIAN) {
    float x = v * v; float y = ci * ci; x = x - y; x = a.nsigma * x;
    return d2b_expf(x);
  }
  float x = 1.0f - v; float y = 1.0f - ci;
  return x / y;
}

// STAGED: the per-row values (class, mask sum, column maximum and d0 = decay(0, cmax): what EVERY non-pair entry of the
// row contributes, whatever the column) are computed once per CTA into shared memory, so the loop over the rows is a
// shared-memory read and a compare per entry and only the few stored pair entries run the exp / division again.
template <bool STAGED>
__global__ void __launch_bounds__(kDecayWarps * 32) mnms_decay_kernel(MnmsArgs a) {
  grid_dep_sync();
  __shared__ float s_min[kDecayWarps][32];
  extern __shared__ __align__(16) unsigned char s_rows[];
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + lane;
  const int nb = rows_of(a, b);
  const float* io = a.iou + (size_t)b * a.n * a.n;
  long long* s_cls = reinterpret_cast<long long*>(s_rows);
  float* s_sum = reinterpret_cast<float*>(s_cls + (STAGED ? a.n : 0));
  float* s_ci = s_sum + (STAGED ? a.n : 0);
  float* s_d0 = s_ci + (STAGED ? a.n : 0);
  if (STAGED) {
    for (int i = threadIdx.x; i < nb; i += kDecayWarps * 32) {
      const float ci = cmax_of(a, b, i);
      s_cls[i] = a.classes[(size_t)b * a.n + i];
      s_sum[i] = sum_of(a, b, i);
      s_ci[i] = ci;
      s_d0[i] = decay_of(a, 0.0f, ci);
    }
    __syncthreads();
  }
  float m = __int_as_float(0x7f800000);
  if (j < nb) {
    const long long cj = a.classes[(size_t)b * a.n + j];
    const float sj = sum_of(a, b, j);
    if (STAGED) {
      for (int i = warp; i < nb; i += kDecayWarps) {
        float d;
        // same-class upper triangle: the pair IoU mnms_iou_kernel stored.  Elsewhere (x - x) resp. (x * 0) of the
        // reference: zero unless the union is empty (0 / 0), which propagates NaN exactly like the TF graph (and a
        // NaN never enters the minimum).
        if (i < j && s_cls[i] == cj) d = decay_of(a, io[(size_t)i * a.n + j], s_ci[i]);
        else if (s_sum[i] + sj == 0.0f) continue;
        else d = s_d0[i];
        m = (d < m) ? d : m;
      }
    } else {
      for (int i0 = warp; i0 < nb; i0 += 4 * kDecayWarps) {  // 4 independent rows in flight per warp
        float v[4], ci[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * kDecayWarps;
          v[u] = 0.0f;
          ci[u] = 0.0f;
          if (i < nb) {  // (warp-uniform: the per-row values are broadcast loads)
            ci[u] = cmax_of(a, b, i);
            if (i < j && a.classes[(size_t)b * a.n + i] == cj) v[u] = io[(size_t)i * a.n + j];
            else v[u] = (sum_of(a, b, i) + sj == 0.0f) ? __int_as_float(0x7fc00000) : 0.0f;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (i0 + u * kDecayWarps >= nb) break;
          const float d = decay_of(a, v[u], ci[u]);
          m = (d < m) ? d : m;
        }
      }
    }
  }
  s_min[warp][lane] = m;
  __syncthreads();
  if (warp == 0 && j < a.n) {
    if (j >= nb) {
      a.out[(size_t)b * a.n + j] = 0.0f;
      return;
    }
#pragma unroll
    for (int w = 1; w < kDecayWarps; ++w) {
      const float v = s_min[w][lane];
      m = (v < m) ? v : m;
    }
    a.out[(size_t)b * a.n + j] = a.scores[(size_t)b * a.n + j] * m;
  }
}

size_t mnms_bytes(const d2b_matrix_nms_params* p, size_t* o_packed, size_t* o_isum, size_t* o_iou, size_t* o_cmax) {
  const size_t B = p->batch, n = p->n, Wd = (size_t)((p->hw + 63) / 64);
  size_t o = 0;
  *o_packed = o; o += p->packed_masks ? 0 : ws_slice(B * n * Wd * sizeof(u64));
  *o_isum = o; o += 3 * ws_slice(B * n * sizeof(unsigned));  // isum, wlo, whi
  *o_cmax = o; o += ws_slice(B * n * sizeof(float));          // (adjacent: one memset zeroes all four)
  *o_iou = o; o += ws_slice(B * n * n * sizeof(float));
  return o;
}

}  // namespace
}  // namespace d2b

using namespace d2b;

extern "C" size_t d2b_matrix_nms_workspace_bytes(const d2b_matrix_nms_params* p) {
  if (!p || p->batch <= 0 || p->n <= 0 || p->hw <= 0) return 0;
  size_t a, b, c, d;
  return mnms_bytes(p, &a, &b, &c, &d);
}

extern "C" int d2b_matrix_nms(const d2b_matrix_nms_params* p, void* workspace, size_t workspace_bytes,
                              d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->kernel == D2B_MNMS_GAUSSIAN || p->kernel == D2B_MNMS_LINEAR,
              "NMS kernel %d not implemented yet.", p->kernel);  // nms.py:76-77 NotImplementedError
  D2B_REQUIRE(p->batch >= 0 && p->n >= 0 && p->hw >= 0, "matrix_nms: negative sizes");
  if (p->batch == 0 || p->n == 0) return D2B_OK;
  D2B_REQUIRE(p->n <= 65535, "matrix_nms: n=%d too large", p->n);
  D2B_REQUIRE(p->hw > 0 && p->hw < (1ll << 31) * 32, "matrix_nms: bad mask size");
  D2B_REQUIRE((p->masks || p->packed_masks) && p->classes && p->scores && p->out, "matrix_nms: NULL pointer");
  size_t o_packed, o_isum, o_iou, o_cmax;
  const size_t need = mnms_bytes(p, &o_packed, &o_isum, &o_iou, &o_cmax);
  if (workspace == nullptr || workspace_bytes < need) {
    set_last_error("matrix_nms needs %zu workspace bytes", need);
    return D2B_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  MnmsArgs a;
  a.masks = p->masks; a.classes = reinterpret_cast<const long long*>(p->classes); a.scores = p->scores;
  a.sum_in = p->sum_masks; a.counts = p->counts; a.B = p->batch; a.n = p->n; a.hw = p->hw;
  a.Wd = (int)((p->hw + 63) / 64); a.kernel = p->kernel;
  a.nsigma = (float)(-1.0 * (double)p->sigma);
  a.packed = p->packed_masks ? const_cast<u64*>(reinterpret_cast<const u64*>(p->packed_masks))
                             : reinterpret_cast<u64*>(ws + o_packed);
  a.isum = reinterpret_cast<unsigned*>(ws + o_isum);
  a.wlo = reinterpret_cast<unsigned*>(ws + o_isum + ws_slice(sizeof(unsigned) * (size_t)a.B * a.n));
  a.whi = reinterpret_cast<unsigned*>(ws + o_isum + 2 * ws_slice(sizeof(unsigned) * (size_t)a.B * a.n));
  a.iou = reinterpret_cast<float*>(ws + o_iou);
  a.cmax = reinterpret_cast<float*>(ws + o_cmax);
  a.out = p->out;
  // column maxima start at +0; the pack kernels accumulate sums / word ranges with atomics (mnms_popc_kernel writes
  // them whole)
  if (p->packed_masks) D2B_CUDA(cudaMemsetAsync(a.cmax, 0, sizeof(float) * (size_t)a.B * a.n, st));
  else D2B_CUDA(cudaMemsetAsync(a.isum, 0, (o_cmax - o_isum) + sizeof(float) * (size_t)a.B * a.n, st));
  if (p->packed_masks) {  // (also with sum_masks given: the word ranges are needed)
    D2B_CUDA(launch_pdl(mnms_popc_kernel, dim3((a.n + 7) / 8, a.B), dim3(256), 0, st, 0, a));
  } else if (a.hw % 4 == 0 && (reinterpret_cast<uintptr_t>(a.masks) & 15) == 0)
    D2B_CUDA(launch_pdl(mnms_pack4_kernel, dim3((a.Wd + 8 * kPackSteps * 2 - 1) / (8 * kPackSteps * 2), a.n, a.B), dim3(256), 0, st, 0, a));
  else
    mnms_pack_kernel<<<dim3((a.Wd + 7) / 8, a.n, a.B), 256, 0, st>>>(a);
  D2B_LAUNCH_CHECK();
  size_t iou_smem = (size_t)a.Wd * sizeof(u64);
  const int stage = iou_smem <= 160 * 1024;  // (larger masks: the row is re-read from L2 per pair)
  if (!stage) iou_smem = 0;
  if (iou_smem > 0) D2B_CUDA(allow_dynamic_smem(mnms_iou_kernel, iou_smem));
  D2B_CUDA(launch_pdl(mnms_iou_kernel, dim3(a.n, a.B), dim3(256), iou_smem, st, 0, a, stage));
  D2B_LAUNCH_CHECK();
  if (a.n <= kDecayStageMax) {
    const size_t dsm = (size_t)a.n * (sizeof(long long) + 3 * sizeof(float));
    if (dsm > 32 * 1024)
      D2B_CUDA(cudaFuncSetAttribute(mnms_decay_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
    D2B_CUDA(launch_pdl(mnms_decay_kernel<true>, dim3((a.n + 31) / 32, a.B), dim3(kDecayWarps * 32), dsm, st, 0, a));
  } else {
    D2B_CUDA(launch_pdl(mnms_decay_kernel<false>, dim3((a.n + 31) / 32, a.B), dim3(kDecayWarps * 32), 0, st, 0, a));
  }
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}
