// roi_align.cu -- multi-level ROIAlign (ROIPooler.call) as ONE gather kernel.
//
// Replaces, per reference call of ROIPooler.call (lib/modeling/poolers.py:134-180):
//   assign_boxes_to_levels (poolers.py:11-49)  -> computed in the CTA prologue
//   tf.where/gather per level (:166-169)       -> gone: every ROI knows its level
//   tf.pad SYMMETRIC (functional.py:125)       -> gone: border rule = index clamp
//   tf.image.crop_and_resize (functional.py:164) + avg_pool (roi_align.py:59-65)
//                                              -> fused gather + register accumulate
//   concat + invert_permutation + gather (:175-178) -> gone: ROI i writes row i
//
// Layout: one CTA per ROI.  The prologue computes, once per ROI and in exactly
// the reference's fp32 operation order, the sample coordinates of every crop
// row and column (top/bottom index, lerp weight, validity) into shared memory.
// Main loop: one warp per output bin, lanes own contiguous 16-byte channel
// groups (NHWC => 512 B coalesced per warp request), the 4 corner vectors of
// each sample are loaded with ld.global.nc and the result is written with a
// streaming store so the output stream does not evict feature maps from L2.
// HBM-bound gather: no contraction, so no tensor cores.
#include <cuda_bf16.h>

#include <climits>

#include "common.cuh"

namespace d2b {
namespace {

constexpr int kMaxSamples = 128;  // max crop rows / cols per ROI (output * sampling_ratio)
#ifndef D2B_RA_THREADS
#define D2B_RA_THREADS 224  // 7 warps: 49 (98) bins = 7 (14) per warp, balanced; same-box A/B vs 256: box pooler 0.2827 -> 0.2785 ms, mask pooler 0.1004 -> 0.0984 ms
#endif
constexpr int kThreads = D2B_RA_THREADS;
#ifndef D2B_RA_BINS
#define D2B_RA_BINS 98  // same-box A/B on the 14x14 mask pooler (196 bins): 56 -> 0.107 ms, 98 / 112 / 196 -> 0.100 ms
#endif
#ifndef D2B_RA_MINB
#define D2B_RA_MINB 1
#endif
constexpr int kBinsPerCta = D2B_RA_BINS;  // bins per CTA (8 warps); larger outputs are split over blockIdx.y

struct Level {
  const void* ptr;
  int H, W;
  float scale;
};

struct RoiAlignArgs {
  Level lv[D2B_MAX_LEVELS];
  int L, N, C;
  const float* boxes;
  const void* bidx;
  int bidx64;
  long long bidx_stride;
  long long M;
  int oh, ow, sr, aligned, pad;
  int min_level, max_level;
  float canon_size, canon_level;
  void* out;
  int* level_counts;
  int64_t* level_out;
};

struct Tap {   // one crop row (or column) of one ROI
  int i0, i1;  // ELEMENT offsets of the two (clamped, un-padded) neighbours inside one image's map
  float w;     // lerp weight toward i1
  int valid;   // 0 => extrapolation (zeros)
};

// assign_boxes_to_levels, poolers.py:37-49 (one rounding per op)
__device__ __forceinline__ int level_of(float y1, float x1, float y2, float x2, int min_level,
                                        int max_level, float canon_size, float canon_level) {
  const float eps = 2.220446049250313e-16f;
  const float ln2 = 0.6931471805599453f;
  float hh = y2 - y1;
  float ww = x2 - x1;
  float area = hh * ww;
  float s = sqrtf(area);
  float t = s / canon_size;
  t = t + eps;
  float v = d2b_logf(t);
  v = v / ln2;
  v = canon_level + v;
  v = floorf(v);
  int lvl;
  if (v != v) lvl = min_level;
  else if (v <= (float)min_level) lvl = min_level;
  else if (v >= (float)max_level) lvl = max_level;
  else lvl = (int)v;
  return lvl - min_level;
}

// functional.py:128-160 + TF CropAndResize coordinate rule: position (in padded pixels) of sample `s` of `cs`
// along an axis of (padded) extent P; lo/hi are the scaled (+pad) box edges.
__device__ __forceinline__ float sample_coord(float lo, float hi, int s, int cs, int P, int aligned) {
  float n1, n2;
  if (aligned) {
    float sp = (hi - lo) / (float)cs;
    float im = (float)(P - 1);
    float a = sp / 2.0f;
    a = lo + a;
    a = a - 0.5f;
    n1 = a / im;
    float nl = sp * (float)(cs - 1);
    nl = nl / im;
    n2 = n1 + nl;
  } else {
    n1 = lo / (float)P;
    n2 = hi / (float)P;
  }
  float in;
  if (cs > 1) {
    const float step = (n2 - n1) * (float)(P - 1) / (float)(cs - 1);
    in = n1 * (float)(P - 1) + (float)s * step;
  } else {
    in = 0.5f * (n1 + n2) * (float)(P - 1);
  }
  return in;
}

__device__ __forceinline__ Tap make_tap(float lo, float hi, int s, int cs, int P, int pad,
                                        int dim, int aligned, int stride) {
  const float in = sample_coord(lo, hi, s, cs, P, aligned);
  Tap t;
  t.valid = (in >= 0.0f && in <= (float)(P - 1)) ? 1 : 0;
  const float f = floorf(in);
  const int i0 = (int)f, i1 = (int)ceilf(in);
  t.w = in - f;
  // padded index p holds un-padded pixel clamp(p - pad, 0, dim-1)  (SYMMETRIC pad of 1)
  t.i0 = min(max(i0 - pad, 0), dim - 1) * stride;
  t.i1 = min(max(i1 - pad, 0), dim - 1) * stride;
  return t;
}

// CTA prologue shared by the forward and backward kernels: every participating thread derives the ROI frame
// redundantly (level, image, and the sample taps of every crop row / column) into shared memory.
__device__ __forceinline__ void build_roi_frame(const RoiAlignArgs& a, long long roi, int ch, int cw, Tap* ty, Tap* tx,
                                                int* s_level, int* s_img, bool publish_level) {
  const int tid = threadIdx.x;
  if (tid < ch + cw || tid == kThreads - 1) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(a.boxes) + roi);
    int lvl = 0;
    if (a.L > 1) lvl = level_of(b.x, b.y, b.z, b.w, a.min_level, a.max_level, a.canon_size, a.canon_level);
    const Level L = a.lv[lvl];
    const float padf = a.pad ? 1.0f : 0.0f;
    for (int t = tid; t < ch + cw; t += kThreads) {  // (one trip unless the crop has more samples than the CTA threads)
      if (t < ch) {
        const float lo = b.x * L.scale + padf, hi = b.z * L.scale + padf;
        ty[t] = make_tap(lo, hi, t, ch, L.H + 2 * a.pad, a.pad, L.H, a.aligned, L.W * a.C);
      } else {
        const float lo = b.y * L.scale + padf, hi = b.w * L.scale + padf;
        tx[t - ch] = make_tap(lo, hi, t - ch, cw, L.W + 2 * a.pad, a.pad, L.W, a.aligned, a.C);
      }
    }
    if (tid == kThreads - 1) {
      long long img = a.bidx64 ? reinterpret_cast<const long long*>(a.bidx)[roi * a.bidx_stride]
                               : (long long)reinterpret_cast<const int*>(a.bidx)[roi * a.bidx_stride];
      *s_level = lvl;
      *s_img = (img >= 0 && img < a.N) ? (int)img : -1;
      if (publish_level) {
        if (a.level_counts) atomicAdd(a.level_counts + lvl, 1);
        if (a.level_out) a.level_out[roi] = lvl;
      }
    }
  }
  __syncthreads();
}

template <typename T>
struct Vec;  // 16-byte channel group
template <>
struct Vec<float> {
  static constexpr int kElems = 4;
  float v[4];
  __device__ __forceinline__ static Vec load(const float* p) {
    const float4 r = __ldg(reinterpret_cast<const float4*>(p));
    Vec o; o.v[0] = r.x; o.v[1] = r.y; o.v[2] = r.z; o.v[3] = r.w;
    return o;
  }
};
template <>
struct Vec<__nv_bfloat16> {
  static constexpr int kElems = 8;
  float v[8];
  __device__ __forceinline__ static Vec load(const __nv_bfloat16* p) {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    Vec o;
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      o.v[2 * i] = __uint_as_float(w[i] << 16);
      o.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
    return o;
  }
};

template <int E>
__device__ __forceinline__ void store_out(float* p, const float (&v)[E]) {
#pragma unroll
  for (int i = 0; i < E; i += 4) __stcs(reinterpret_cast<float4*>(p + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
}
template <int E>
__device__ __forceinline__ void store_out(__nv_bfloat16* p, const float (&v)[E]) {
  static_assert(E == 8, "bf16 output groups are 8 wide");
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  __stcs(reinterpret_cast<uint4*>(p), make_uint4(w[0], w[1], w[2], w[3]));
}

// TIn: feature element type; TOut: output element type; GROUPS: 16-byte groups
// each lane owns per bin (0 => runtime loop for any channel count).  S1: 1 / 2 = unrolled fast path for that
// many samples per bin axis, 0 = generic loop.
template <typename TIn, typename TOut, int GROUPS, int S1>
__global__ void __launch_bounds__(kThreads, D2B_RA_MINB) roi_align_kernel(const RoiAlignArgs a) {
  grid_dep_sync();
  constexpr int E = Vec<TIn>::kElems;
  __shared__ Tap ty[kMaxSamples];
  __shared__ Tap tx[kMaxSamples];
  __shared__ int s_level;
  __shared__ int s_img;

  const long long roi = blockIdx.x;
  const int s1 = a.sr > 0 ? a.sr : 1;
  const int ch = a.oh * s1, cw = a.ow * s1;
  const int tid = threadIdx.x;

  build_roi_frame(a, roi, ch, cw, ty, tx, &s_level, &s_img, blockIdx.y == 0);

  const int lvl = s_level;
  const int img = s_img;
  const Level L = a.lv[lvl];
  const int C = a.C;
  const int lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  const TIn* base = reinterpret_cast<const TIn*>(L.ptr) + (size_t)(img < 0 ? 0 : img) * L.H * L.W * C;
  TOut* obase = reinterpret_cast<TOut*>(a.out) + (size_t)roi * a.oh * a.ow * C;
  const float cnt = (float)(s1 * s1);
  const int groups_total = C / E;  // 16-byte groups per pixel
  const int bin_begin = blockIdx.y * kBinsPerCta;
  const int bin_end = min(bin_begin + kBinsPerCta, a.oh * a.ow);

  if constexpr (S1 > 0 && GROUPS > 0) {
    // sampling_ratio 0/1 (the reference default; S1 == 1) and 2 (the keypoint head, defaults.py:513; S1 == 2):
    // fully unrolled channel groups and samples, corner addresses formed once per sample from the precomputed
    // element offsets, 8 x 16-byte corner loads in flight per lane.  S1 == 2 accumulates the 4 samples in the
    // reference's row-major order and divides by 4 (roi_align.py:59-65 avg_pool).
    for (int bin = bin_begin + warp; bin < bin_end; bin += kWarps) {
      const int oy = bin / a.ow, ox = bin - oy * a.ow;
      TOut* o = obase + (size_t)bin * C + lane * E;
      constexpr int G = GROUPS > 0 ? GROUPS : 1;
      float acc[G][E];
#pragma unroll
      for (int j = 0; j < G; ++j)
#pragma unroll
        for (int e = 0; e < E; ++e) acc[j][e] = 0.0f;
#pragma unroll
      for (int dy = 0; dy < S1; ++dy) {
        const Tap y = ty[oy * S1 + dy];
#pragma unroll
        for (int dx = 0; dx < S1; ++dx) {
          const Tap x = tx[ox * S1 + dx];
          if (y.valid && x.valid && img >= 0) {  // warp-uniform
            const TIn* p00 = base + (y.i0 + x.i0) + lane * E;
            const TIn* p01 = base + (y.i0 + x.i1) + lane * E;
            const TIn* p10 = base + (y.i1 + x.i0) + lane * E;
            const TIn* p11 = base + (y.i1 + x.i1) + lane * E;
            Vec<TIn> tl[G], tr[G], bl[G], br[G];
#pragma unroll
            for (int j = 0; j < GROUPS; ++j) {
              tl[j] = Vec<TIn>::load(p00 + j * 32 * E);
              tr[j] = Vec<TIn>::load(p01 + j * 32 * E);
              bl[j] = Vec<TIn>::load(p10 + j * 32 * E);
              br[j] = Vec<TIn>::load(p11 + j * 32 * E);
            }
#pragma unroll
            for (int j = 0; j < GROUPS; ++j) {
#pragma unroll
              for (int e = 0; e < E; ++e) {
                float t = tr[j].v[e] - tl[j].v[e]; t = t * x.w; t = tl[j].v[e] + t;
                float bb = br[j].v[e] - bl[j].v[e]; bb = bb * x.w; bb = bl[j].v[e] + bb;
                float r = bb - t; r = r * y.w; r = t + r;
                acc[j][e] = (S1 == 1) ? r : acc[j][e] + r;
              }
            }
          }  // an extrapolated sample contributes 0 (acc + 0.0f == acc)
        }
      }
#pragma unroll
      for (int j = 0; j < GROUPS; ++j) {
        if (S1 > 1) {
#pragma unroll
          for (int e = 0; e < E; ++e) acc[j][e] = acc[j][e] / cnt;
        }
        store_out<E>(o + j * 32 * E, acc[j]);
      }
    }
  } else {
  for (int bin = bin_begin + warp; bin < bin_end; bin += kWarps) {
    const int oy = bin / a.ow, ox = bin - oy * a.ow;
    TOut* o = obase + (size_t)bin * C;
    auto do_group = [&](int g) {
      const int c = g * E;
      float acc[E];
#pragma unroll
      for (int e = 0; e < E; ++e) acc[e] = 0.0f;
      for (int dy = 0; dy < s1; ++dy) {
        const Tap y = ty[oy * s1 + dy];
        for (int dx = 0; dx < s1; ++dx) {
          const Tap x = tx[ox * s1 + dx];
          float val[E];
          if (y.valid && x.valid && img >= 0) {
            const TIn* r0 = base + y.i0 + c;
            const TIn* r1 = base + y.i1 + c;
            const Vec<TIn> tl = Vec<TIn>::load(r0 + x.i0);
            const Vec<TIn> tr = Vec<TIn>::load(r0 + x.i1);
            const Vec<TIn> bl = Vec<TIn>::load(r1 + x.i0);
            const Vec<TIn> br = Vec<TIn>::load(r1 + x.i1);
#pragma unroll
            for (int e = 0; e < E; ++e) {
              float t = tr.v[e] - tl.v[e]; t = t * x.w; t = tl.v[e] + t;
              float bb = br.v[e] - bl.v[e]; bb = bb * x.w; bb = bl.v[e] + bb;
              float r = bb - t; r = r * y.w; r = t + r;
              val[e] = r;
            }
          } else {
#pragma unroll
            for (int e = 0; e < E; ++e) val[e] = 0.0f;
          }
          if (s1 == 1) {
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = val[e];
          } else {
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = acc[e] + val[e];
          }
        }
      }
      if (s1 > 1) {
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = acc[e] / cnt;
      }
      store_out<E>(o + c, acc);
    };
    if (GROUPS > 0) {
#pragma unroll
      for (int j = 0; j < GROUPS; ++j) do_group(lane + 32 * j);
    } else {
      for (int g = lane; g < groups_total; g += 32) do_group(g);
    }
  }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward: gradient w.r.t. the feature maps (AvgPoolGrad -> CropAndResizeGradImage ->
// MirrorPadGrad -> per-level scatter in the reference's TF graph).  Same CTA-per-ROI frame and
// tap tables as the forward kernel; one warp per crop sample, lanes own 16-byte channel groups,
// the four corner contributions go out as vector reductions (RED.E.ADD.F32x4: one L2 atomic
// transaction per 16 B instead of four).  The SYMMETRIC pad fold is the same index clamp the
// forward uses, so border rows accumulate straight onto the edge pixel.
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

struct RoiAlignGradArgs {
  RoiAlignArgs f;
  const float* grad_out;
  float* grad[D2B_MAX_LEVELS];
};

__global__ void __launch_bounds__(kThreads) roi_align_backward_kernel(const RoiAlignGradArgs ga) {
  const RoiAlignArgs& a = ga.f;
  __shared__ Tap ty[kMaxSamples];
  __shared__ Tap tx[kMaxSamples];
  __shared__ int s_level;
  __shared__ int s_img;
  const long long roi = blockIdx.x;
  const int s1 = a.sr > 0 ? a.sr : 1;
  const int ch = a.oh * s1, cw = a.ow * s1;
  const int tid = threadIdx.x;
  build_roi_frame(a, roi, ch, cw, ty, tx, &s_level, &s_img, false);
  const int img = s_img;
  if (img < 0) return;  // TF skips boxes whose box_ind is out of range
  const int lvl = s_level;
  const Level L = a.lv[lvl];
  const int C = a.C;
  const int lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  float* base = ga.grad[lvl] + (size_t)img * L.H * L.W * C;
  const float* gbase = ga.grad_out + (size_t)roi * a.oh * a.ow * C;
  const float cnt = (float)(s1 * s1);
  const int groups_total = C / 4;
  const int bin_begin = blockIdx.y * kBinsPerCta;
  const int bin_end = min(bin_begin + kBinsPerCta, a.oh * a.ow);
  const int samples = s1 * s1;
  // work item = (bin, sub-sample); a warp walks items, lanes walk channel groups
  for (int item = bin_begin * samples + warp; item < bin_end * samples; item += kWarps) {
    const int bin = item / samples, sub = item - bin * samples;
    const int oy = bin / a.ow, ox = bin - oy * a.ow;
    const int dy = sub / s1, dx = sub - dy * s1;
    const Tap y = ty[oy * s1 + dy];
    const Tap x = tx[ox * s1 + dx];
    if (!(y.valid && x.valid)) continue;
    const float omy = 1.0f - y.w, omx = 1.0f - x.w;
    const float* g = gbase + (size_t)bin * C;
    for (int grp = lane; grp < groups_total; grp += 32) {
      float4 gv = __ldcs(reinterpret_cast<const float4*>(g) + grp);
      if (s1 > 1) { gv.x = gv.x / cnt; gv.y = gv.y / cnt; gv.z = gv.z / cnt; gv.w = gv.w / cnt; }
      const int c = grp * 4;
      const float4 dt = make_float4(omy * gv.x, omy * gv.y, omy * gv.z, omy * gv.w);
      const float4 db = make_float4(y.w * gv.x, y.w * gv.y, y.w * gv.z, y.w * gv.w);
      red_add_v4(base + y.i0 + x.i0 + c, omx * dt.x, omx * dt.y, omx * dt.z, omx * dt.w);
      red_add_v4(base + y.i0 + x.i1 + c, x.w * dt.x, x.w * dt.y, x.w * dt.z, x.w * dt.w);
      red_add_v4(base + y.i1 + x.i0 + c, omx * db.x, omx * db.y, omx * db.z, omx * db.w);
      red_add_v4(base + y.i1 + x.i1 + c, x.w * db.x, x.w * db.y, x.w * db.z, x.w * db.w);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Deterministic backward: the CPU kernel's summation order, bit for bit, without floating-point atomics.
// Per level and image, a zeroed padded gradient receives, ROI by ROI in input order, crop row y by crop row, column
// x by column, the TL, TR, BL, BR products of each sample; then each padded pixel is added onto clamp(p - pad) in
// raster order.  Every padded accumulator is owned by one thread, which pulls its contributions in that order:
//   roi_align_grad_bin_kernel        thread per ROI: (level, image) key, padded footprint, sample taps
//   roi_align_grad_partition_kernel  CTA per (level, image): its ROI indices in input order (ballot compaction)
//   roi_align_grad_accum_kernel      CTA per (level, image, 8x8 destination tile, 128 channels): warp per padded
//                                    row, lane per 16-byte channel group; walks the key's ROI list, then folds
constexpr int kGradTile = 8;                   // destination tile edge (un-padded pixels)
constexpr int kGradRows = kGradTile + 2;       // + the border row / column of each side that folds onto an edge tile
constexpr int kGradThreads = 32 * kGradRows;   // warp w owns padded row w of the tile
constexpr int kGradChannels = 32 * 4;          // channels per accumulate CTA (one float4 per lane)
constexpr int kBinThreads = 256;
constexpr int kPartThreads = 1024;

struct GTap {  // one crop row / column of one ROI, padded coordinates
  int p;       // floor of the sample position; -1 => outside [0, P-1] (the sample contributes nothing)
  float w;     // position - p; the ceil neighbour is p + (w != 0)
};

struct GradDetArgs {
  RoiAlignGradArgs g;
  int* key;      // [M] level * N + image, -1 => no contribution
  int4* rect;    // [M] padded footprint: rows y0..y1, columns x0..x1 (inclusive)
  int* list;     // [M] ROI indices grouped by key, input order inside a key
  int2* range;   // [L * N] [begin, end) of each key in `list`
  GTap* taps;    // [M, ch + cw]
  long long tile_start[D2B_MAX_LEVELS + 1];  // first accumulate CTA of each level
  int tiles_x[D2B_MAX_LEVELS], tiles_y[D2B_MAX_LEVELS];
};

__global__ void __launch_bounds__(kBinThreads) roi_align_grad_bin_kernel(const GradDetArgs d) {
  const RoiAlignArgs& a = d.g.f;
  const long long roi = (long long)blockIdx.x * kBinThreads + threadIdx.x;
  if (roi >= a.M) return;
  const int s1 = a.sr > 0 ? a.sr : 1;
  const int ch = a.oh * s1, cw = a.ow * s1;
  const float4 b = __ldg(reinterpret_cast<const float4*>(a.boxes) + roi);
  int lvl = 0;
  if (a.L > 1) lvl = level_of(b.x, b.y, b.z, b.w, a.min_level, a.max_level, a.canon_size, a.canon_level);
  D2B_BOUND(lvl, a.L);
  const Level L = a.lv[lvl];
  const float padf = a.pad ? 1.0f : 0.0f;
  GTap* tap = d.taps + (size_t)roi * (ch + cw);
  int lo[2] = {INT_MAX, INT_MAX}, hi[2] = {-1, -1};
  for (int t = 0; t < ch + cw; ++t) {
    const int ax = t < ch ? 0 : 1;
    const float e0 = ax ? b.y : b.x, e1 = ax ? b.w : b.z;
    const float elo = e0 * L.scale + padf, ehi = e1 * L.scale + padf;
    const int cs = ax ? cw : ch, P = (ax ? L.W : L.H) + 2 * a.pad;
    const float in = sample_coord(elo, ehi, ax ? t - ch : t, cs, P, a.aligned);
    GTap g{-1, 0.0f};
    if (in >= 0.0f && in <= (float)(P - 1)) {
      const float f = floorf(in);
      g.p = (int)f;
      g.w = in - f;
      lo[ax] = min(lo[ax], g.p);
      hi[ax] = max(hi[ax], g.p + (g.w != 0.0f ? 1 : 0));
    }
    tap[t] = g;
  }
  const long long img = a.bidx64 ? reinterpret_cast<const long long*>(a.bidx)[roi * a.bidx_stride]
                                 : (long long)reinterpret_cast<const int*>(a.bidx)[roi * a.bidx_stride];
  const bool live = img >= 0 && img < a.N && hi[0] >= 0 && hi[1] >= 0;  // TF skips out-of-range box_ind
  d.key[roi] = live ? lvl * a.N + (int)img : -1;
  d.rect[roi] = make_int4(lo[0], hi[0], lo[1], hi[1]);
}

__global__ void __launch_bounds__(kPartThreads) roi_align_grad_partition_kernel(const GradDetArgs d) {
  __shared__ int s_warp[kPartThreads / 32];
  const int key = blockIdx.x;
  const int M = (int)d.g.f.M;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int begin = 0;  // ROIs of smaller keys
  for (int b0 = 0; b0 < M; b0 += kPartThreads) {
    const int i = b0 + tid;
    int k = -1;
    if (i < M) k = d.key[i];
    begin += __syncthreads_count(k >= 0 && k < key);
  }
  int pos = begin;
  for (int b0 = 0; b0 < M; b0 += kPartThreads) {
    const int i = b0 + tid;
    const bool hit = i < M && d.key[i] == key;
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < kPartThreads / 32; ++w) {
      const int c = s_warp[w];
      before += w < warp ? c : 0;
      total += c;
    }
    if (hit) {
      const int o = pos + before + __popc(m & ((1u << lane) - 1u));
      D2B_BOUND(o, M);
      d.list[o] = i;
    }
    pos += total;
    __syncthreads();
  }
  if (tid == 0) d.range[key] = make_int2(begin, pos);
}

__device__ __forceinline__ float4 f4_scale(float s, float4 v) { return make_float4(s * v.x, s * v.y, s * v.z, s * v.w); }
__device__ __forceinline__ void f4_acc(float4& a, float4 v) {
  a.x = a.x + v.x; a.y = a.y + v.y; a.z = a.z + v.z; a.w = a.w + v.w;
}

__global__ void __launch_bounds__(kGradThreads) roi_align_grad_accum_kernel(const GradDetArgs d) {
  const RoiAlignArgs& a = d.g.f;
  long long t = blockIdx.x;
  int lvl = 0;
  while (lvl + 1 < a.L && t >= d.tile_start[lvl + 1]) ++lvl;
  t -= d.tile_start[lvl];
  const int tx_n = d.tiles_x[lvl], per_img = tx_n * d.tiles_y[lvl];
  const int img = (int)(t / per_img);
  const int tr = (int)(t - (long long)img * per_img);
  const int ty = tr / tx_n, tx = tr - ty * tx_n;
  D2B_BOUND(img, a.N);
  const int2 rg = d.range[lvl * a.N + img];
  if (rg.x == rg.y) return;  // no ROI on this level and image
  const Level L = a.lv[lvl];
  const int pad = a.pad, C = a.C;
  // padded rows [py0, py1) and columns [px0, px1) whose fold lands in this tile
  const int sy0 = ty * kGradTile, sy1 = min(sy0 + kGradTile, L.H);
  const int sx0 = tx * kGradTile, sx1 = min(sx0 + kGradTile, L.W);
  const int py0 = sy0 == 0 ? 0 : sy0 + pad, py1 = sy1 == L.H ? L.H + 2 * pad : sy1 + pad;
  const int px0 = sx0 == 0 ? 0 : sx0 + pad, px1 = sx1 == L.W ? L.W + 2 * pad : sx1 + pad;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int py = py0 + warp;
  const bool row_live = py < py1;
  const int c = (blockIdx.y * 32 + lane) * 4;  // this lane's channel group
  const bool grp_live = c < C;
  const int s1 = a.sr > 0 ? a.sr : 1;
  const int ch = a.oh * s1, cw = a.ow * s1;
  const float cnt = (float)(s1 * s1);

  float4 acc[kGradRows];
#pragma unroll
  for (int j = 0; j < kGradRows; ++j) acc[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  int touched = 0;
  if (row_live) {
    for (int b0 = rg.x; b0 < rg.y; b0 += 32) {
      const int i = b0 + lane;
      int roi = -1;
      bool hit = false;
      if (i < rg.y) {
        D2B_BOUND(i, a.M);
        roi = d.list[i];
        D2B_BOUND(roi, a.M);
        const int4 r = d.rect[roi];
        hit = r.x <= py && py <= r.y && r.z < px1 && r.w >= px0;
      }
      unsigned m = __ballot_sync(0xffffffffu, hit);
      while (m) {  // ROIs of this chunk, in input order
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const int r = __shfl_sync(0xffffffffu, roi, src);
        touched = 1;
        const GTap* tap_y = d.taps + (size_t)r * (ch + cw);
        const GTap* tap_x = tap_y + ch;
        const float* gro = d.g.grad_out + (size_t)r * a.oh * a.ow * C + c;
        for (int y = 0; y < ch; ++y) {
          const GTap ty_ = tap_y[y];
          if (ty_.p < 0) continue;
          const int top = ty_.p, bot = ty_.p + (ty_.w != 0.0f ? 1 : 0);
          if (top != py && bot != py) continue;
          const float ly = ty_.w, omy = 1.0f - ly;
          for (int x = 0; x < cw; ++x) {
            const GTap tx_ = tap_x[x];
            if (tx_.p < 0) continue;
            const int left = tx_.p, right = tx_.p + (tx_.w != 0.0f ? 1 : 0);
            if (right < px0 || left >= px1) continue;
            if (!grp_live) continue;
            const float lx = tx_.w, omx = 1.0f - lx;
            const size_t bin = (size_t)(y / s1) * a.ow + x / s1;
            D2B_BOUND(bin, (size_t)a.oh * a.ow);
            float4 gv = __ldg(reinterpret_cast<const float4*>(gro + bin * C));
            if (s1 > 1) { gv.x = gv.x / cnt; gv.y = gv.y / cnt; gv.z = gv.z / cnt; gv.w = gv.w / cnt; }
            const float4 dtop = f4_scale(omy, gv), dbot = f4_scale(ly, gv);
            const int jl = left - px0, jr = right - px0;
#pragma unroll
            for (int j = 0; j < kGradRows; ++j) {
              if (j != jl && j != jr) continue;  // warp-uniform
              if (top == py) {
                if (j == jl) f4_acc(acc[j], f4_scale(omx, dtop));
                if (j == jr) f4_acc(acc[j], f4_scale(lx, dtop));
              }
              if (bot == py) {
                if (j == jl) f4_acc(acc[j], f4_scale(omx, dbot));
                if (j == jr) f4_acc(acc[j], f4_scale(lx, dbot));
              }
            }
          }
        }
      }
    }
  }
  // Fold (MirrorPadGrad): padded rows reach their un-padded row in ascending order -- one barrier-separated phase
  // per rank inside the fold group (rank 2 only when H == 1); columns in ascending order inside a thread.  Only
  // tiles some ROI reaches are written.
  if (!__syncthreads_or(touched)) return;
  const int sy = min(max(py - pad, 0), L.H - 1);
  const int rank = py - (sy == 0 ? 0 : sy + pad);
  float* grow = d.g.grad[lvl] + ((size_t)img * L.H + sy) * L.W * C + c;
  for (int ph = 0; ph < 3; ++ph) {
    if (row_live && grp_live && rank == ph) {
#pragma unroll
      for (int j = 0; j < kGradRows; ++j) {
        if (px0 + j >= px1) break;
        const int sx = min(max(px0 + j - pad, 0), L.W - 1);
        D2B_BOUND((size_t)sy * L.W + sx, (size_t)L.H * L.W);
        float4* q = reinterpret_cast<float4*>(grow + (size_t)sx * C);
        float4 v = *q;
        f4_acc(v, acc[j]);
        *q = v;
      }
    }
    __syncthreads();
  }
}

template <typename TIn, typename TOut>
int launch(const RoiAlignArgs& a, cudaStream_t st) {
  constexpr int E = Vec<TIn>::kElems;
  const dim3 grid((unsigned)a.M, (unsigned)((a.oh * a.ow + kBinsPerCta - 1) / kBinsPerCta)), block(kThreads);
  const int g = a.C / E;
  const int s1 = a.sr > 0 ? a.sr : 1;
  cudaError_t rc;
  if (g == 32 && s1 == 1) rc = launch_pdl(roi_align_kernel<TIn, TOut, 1, 1>, grid, block, 0, st, 0, a);
  else if (g == 64 && s1 == 1) rc = launch_pdl(roi_align_kernel<TIn, TOut, 2, 1>, grid, block, 0, st, 0, a);
  else if (g == 32 && s1 == 2) rc = launch_pdl(roi_align_kernel<TIn, TOut, 1, 2>, grid, block, 0, st, 0, a);
  else if (g == 64 && s1 == 2) rc = launch_pdl(roi_align_kernel<TIn, TOut, 2, 2>, grid, block, 0, st, 0, a);
  else if (g == 32) rc = launch_pdl(roi_align_kernel<TIn, TOut, 1, 0>, grid, block, 0, st, 0, a);
  else if (g == 64) rc = launch_pdl(roi_align_kernel<TIn, TOut, 2, 0>, grid, block, 0, st, 0, a);
  else rc = launch_pdl(roi_align_kernel<TIn, TOut, 0, 0>, grid, block, 0, st, 0, a);
  D2B_CUDA(rc);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

}  // namespace
}  // namespace d2b

using namespace d2b;

extern "C" size_t d2b_roi_align_multilevel_workspace_bytes(const d2b_roi_align_params*) { return 0; }

// validates the forward description and fills the kernel argument block; `backward` relaxes the pointer checks
static int fill_args(const d2b_roi_align_params* p, RoiAlignArgs& a, bool backward) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  // poolers.py:148-150 asserts len(x) == len(scales); unknown pooler types raise ValueError (:118)
  D2B_REQUIRE(p->num_levels >= 1 && p->num_levels <= D2B_MAX_LEVELS, "num_levels=%d out of [1,%d]",
              p->num_levels, D2B_MAX_LEVELS);
  D2B_REQUIRE(p->num_rois >= 0 && p->num_rois < (1ll << 31), "num_rois=%lld out of range", (long long)p->num_rois);
  D2B_REQUIRE(p->output_h > 0 && p->output_w > 0, "output size must be positive");
  D2B_REQUIRE(p->sampling_ratio >= 0, "sampling_ratio must be >= 0");
  const int s1 = p->sampling_ratio > 0 ? p->sampling_ratio : 1;
  D2B_REQUIRE(p->output_h * s1 <= kMaxSamples && p->output_w * s1 <= kMaxSamples,
              "output_size*sampling_ratio too large (max %d per axis)", kMaxSamples);
  if (backward) {
    D2B_REQUIRE(p->feature_dtype == D2B_DTYPE_F32 && p->out_dtype == D2B_DTYPE_F32, "backward is fp32 only");
  }
  D2B_REQUIRE(p->feature_dtype == D2B_DTYPE_F32 || p->feature_dtype == D2B_DTYPE_BF16, "bad feature_dtype");
  D2B_REQUIRE(p->out_dtype == D2B_DTYPE_F32 || (p->out_dtype == D2B_DTYPE_BF16 && p->feature_dtype == D2B_DTYPE_BF16),
              "bad out_dtype");
  const int E = p->feature_dtype == D2B_DTYPE_F32 ? 4 : 8;
  D2B_REQUIRE(p->channels > 0 && p->channels % E == 0, "channels=%d must be a multiple of %d", p->channels, E);
  D2B_REQUIRE(p->num_images > 0, "num_images must be positive");
  a.M = 0;
  if (p->num_rois == 0) return D2B_OK;
  D2B_REQUIRE(p->boxes && p->batch_idx && (backward || p->out), "boxes/batch_idx/out must be non-NULL");

  for (int l = 0; l < p->num_levels; ++l) {
    D2B_REQUIRE((backward || p->features[l] != nullptr) && p->height[l] > 0 && p->width[l] > 0, "level %d: bad feature map", l);
    D2B_REQUIRE((long long)p->height[l] * p->width[l] * p->channels < (1ll << 31), "level %d: H*W*C must fit in int32", l);
    a.lv[l].ptr = p->features[l];
    a.lv[l].H = p->height[l];
    a.lv[l].W = p->width[l];
    a.lv[l].scale = p->scale[l];
  }
  for (int l = p->num_levels; l < D2B_MAX_LEVELS; ++l) a.lv[l] = a.lv[0];
  a.L = p->num_levels; a.N = p->num_images; a.C = p->channels;
  a.boxes = p->boxes; a.bidx = p->batch_idx; a.bidx64 = p->batch_idx_is_int64;
  a.bidx_stride = p->batch_idx_stride > 0 ? p->batch_idx_stride : 1;
  a.M = p->num_rois;
  a.oh = p->output_h; a.ow = p->output_w; a.sr = p->sampling_ratio; a.aligned = p->aligned ? 1 : 0;
  a.pad = p->pad_border ? 1 : 0;
  a.min_level = p->min_level; a.max_level = p->min_level + p->num_levels - 1;
  a.canon_size = (float)p->canonical_box_size; a.canon_level = (float)p->canonical_level;
  a.out = p->out; a.level_counts = p->level_counts; a.level_out = p->level_assignments;
  if (p->num_levels > 1) {
    D2B_REQUIRE(p->min_level > 0 && p->canonical_box_size > 0, "min_level and canonical_box_size must be positive");
  }

  return D2B_OK;
}

extern "C" int d2b_roi_align_multilevel(const d2b_roi_align_params* p, void* /*workspace*/,
                                        size_t /*workspace_bytes*/, d2b_stream_t stream) {
  RoiAlignArgs a;
  const int rc = fill_args(p, a, false);
  if (rc != D2B_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p->level_counts) D2B_CUDA(cudaMemsetAsync(p->level_counts, 0, sizeof(int32_t) * p->num_levels, st));
  if (a.M == 0) return D2B_OK;
  if (p->feature_dtype == D2B_DTYPE_F32) return launch<float, float>(a, st);
  if (p->out_dtype == D2B_DTYPE_F32) return launch<__nv_bfloat16, float>(a, st);
  return launch<__nv_bfloat16, __nv_bfloat16>(a, st);
}

static size_t ws_align(size_t n) { return (n + 255) & ~(size_t)255; }

// deterministic mode: key, rect, list, range and tap arrays, each 256-byte aligned; 0 when there is nothing to do
extern "C" size_t d2b_roi_align_backward_workspace_bytes(const d2b_roi_align_backward_params* p) {
  if (p == nullptr || !p->deterministic) return 0;
  const d2b_roi_align_params& f = p->fwd;
  if (f.num_rois <= 0 || f.num_levels < 1 || f.num_levels > D2B_MAX_LEVELS || f.num_images <= 0 ||
      f.output_h <= 0 || f.output_w <= 0 || f.sampling_ratio < 0)
    return 0;
  const size_t M = (size_t)f.num_rois;
  const size_t s1 = f.sampling_ratio > 0 ? (size_t)f.sampling_ratio : 1;
  const size_t taps = s1 * ((size_t)f.output_h + (size_t)f.output_w);
  return ws_align(M * sizeof(int)) + ws_align(M * sizeof(int4)) + ws_align(M * sizeof(int)) +
         ws_align((size_t)f.num_levels * f.num_images * sizeof(int2)) + ws_align(M * taps * sizeof(GTap));
}

static int launch_backward_deterministic(const RoiAlignGradArgs& g, void* workspace, cudaStream_t st) {
  const RoiAlignArgs& a = g.f;
  GradDetArgs d;
  d.g = g;
  const size_t M = (size_t)a.M;
  char* w = static_cast<char*>(workspace);
  d.key = reinterpret_cast<int*>(w); w += ws_align(M * sizeof(int));
  d.rect = reinterpret_cast<int4*>(w); w += ws_align(M * sizeof(int4));
  d.list = reinterpret_cast<int*>(w); w += ws_align(M * sizeof(int));
  d.range = reinterpret_cast<int2*>(w); w += ws_align((size_t)a.L * a.N * sizeof(int2));
  d.taps = reinterpret_cast<GTap*>(w);
  long long tiles = 0;
  for (int l = 0; l < D2B_MAX_LEVELS; ++l) {
    d.tile_start[l] = tiles;
    d.tiles_y[l] = d.tiles_x[l] = 1;
    if (l < a.L) {
      d.tiles_y[l] = (a.lv[l].H + kGradTile - 1) / kGradTile;
      d.tiles_x[l] = (a.lv[l].W + kGradTile - 1) / kGradTile;
      tiles += (long long)a.N * d.tiles_y[l] * d.tiles_x[l];
    }
  }
  d.tile_start[D2B_MAX_LEVELS] = tiles;
  D2B_REQUIRE(tiles < (1ll << 31), "too many destination tiles (%lld)", tiles);
  roi_align_grad_bin_kernel<<<(unsigned)((M + kBinThreads - 1) / kBinThreads), kBinThreads, 0, st>>>(d);
  D2B_LAUNCH_CHECK();
  roi_align_grad_partition_kernel<<<(unsigned)(a.L * a.N), kPartThreads, 0, st>>>(d);
  D2B_LAUNCH_CHECK();
  const dim3 grid((unsigned)tiles, (unsigned)((a.C + kGradChannels - 1) / kGradChannels));
  roi_align_grad_accum_kernel<<<grid, kGradThreads, 0, st>>>(d);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

extern "C" int d2b_roi_align_backward(const d2b_roi_align_backward_params* p, void* workspace, size_t workspace_bytes,
                                      d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  RoiAlignGradArgs g;
  const int rc = fill_args(&p->fwd, g.f, true);
  if (rc != D2B_OK) return rc;
  if (g.f.M == 0) return D2B_OK;
  D2B_REQUIRE(p->grad_out != nullptr, "grad_out is NULL");
  for (int l = 0; l < D2B_MAX_LEVELS; ++l) {
    g.grad[l] = p->grad_features[l < p->fwd.num_levels ? l : 0];
    D2B_REQUIRE(g.grad[l] != nullptr, "grad_features[%d] is NULL", l);
  }
  g.grad_out = p->grad_out;
  g.f.level_counts = nullptr;
  g.f.level_out = nullptr;
  if (p->deterministic) {
    const size_t need = d2b_roi_align_backward_workspace_bytes(p);
    if (workspace == nullptr || workspace_bytes < need) {
      set_last_error("deterministic roi_align_backward needs %zu workspace bytes", need);
      return D2B_EWORKSPACE;
    }
    return launch_backward_deterministic(g, workspace, static_cast<cudaStream_t>(stream));
  }
  const dim3 grid((unsigned)g.f.M, (unsigned)((g.f.oh * g.f.ow + kBinsPerCta - 1) / kBinsPerCta));
  roi_align_backward_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(g);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

extern "C" size_t d2b_crop_and_resize_aligned_workspace_bytes(const d2b_crop_and_resize_params*) { return 0; }

// functional.py:100-166 on one map: the multi-level kernel with one level of scale 1
extern "C" int d2b_crop_and_resize_aligned(const d2b_crop_and_resize_params* p, void* ws, size_t ws_bytes,
                                           d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  d2b_roi_align_params r = {};
  r.features[0] = p->image;
  r.height[0] = p->height; r.width[0] = p->width; r.scale[0] = 1.0f;
  r.num_levels = 1; r.num_images = p->num_images; r.channels = p->channels;
  r.feature_dtype = D2B_DTYPE_F32; r.out_dtype = D2B_DTYPE_F32;
  r.boxes = p->boxes; r.batch_idx = p->box_ind; r.batch_idx_is_int64 = 0; r.batch_idx_stride = 1;
  r.num_rois = p->num_boxes;
  r.output_h = p->crop_h; r.output_w = p->crop_w;
  r.sampling_ratio = 0; r.aligned = p->aligned; r.pad_border = p->pad_border;
  r.min_level = 0; r.canonical_box_size = 224; r.canonical_level = 4;
  r.out = p->out;
  return d2b_roi_align_multilevel(&r, ws, ws_bytes, stream);
}
