// solo_upsample.cu -- what MaskKernelBranch.inference does after the per-image tail (solo_v2.py:599-627):
//   resize_images(pred_masks, image_shape) (bilinear)  ->  > mask_threshold  ->  boxes from masks.
// The reference materialises [N, D, H, W] fp32 twice (resize output, thresholded masks) plus the yy / xx products
// (427 MB per image each at D=100, 800x1333).  Here the kept masks arrive BIT-PACKED from d2b_solo_postprocess; one
// kernel re-samples them, thresholds, writes uint8 (or packed) image masks and reduces the box statistics on the fly.
//   * flat 16-pixel runs per thread (16-byte stores); the few source rows a CTA needs are expanded to fp32 0/1 in
//     shared memory together with each row's [first, last] set column and the per-output-column taps;
//   * a run whose source window is empty in both rows is written as zeros without sampling (most of an image);
//   * box statistics are exact integers (count, sum y, sum x, min / max over pixels with y > 0 / x > 0), reduced per
//     warp and accumulated with 64-bit atomics; a finalise kernel applies the reference's mean / where rule.
// TF ResizeBilinear arithmetic in the reference's op order (no FMA), both coordinate conventions the reference can
// end up with (functional.py:21-35): half-pixel centres (tf.compat.v2.image.resize) and align_corners=True.
// With out_rle_offsets the same per-pixel rule (resize_tap / up_lerp) feeds the COCO run-length encoder of
// mask_rle.cuh (solo_rle_kernel) over the rectangle the taps of the set source pixels can reach.
#include <limits.h>
#include <math.h>

#include "kernels.cuh"
#include "mask_rle.cuh"

namespace d2b {
namespace {
typedef unsigned long long u64;

constexpr int kUpThreads = 256;
constexpr int kRun = 16;  // output pixels per thread per step

struct Tap {
  unsigned short lo, hi;
  float lerp;
};
struct Stats {  // per (image, detection); zero-initialised except the min fields (0x7fffffff)
  u64 count, sum_y, sum_x;
  int min_y, max_y, min_x, max_x;
};
struct UpArgs {
  const u64* packed;
  int B, D, h, w, H, W, Wd_in, Wd_out;
  int align_corners;
  float scale_y, scale_x, thr;
  int iters;     // runs per thread: a CTA covers iters * 256 * 16 flat output pixels
  int rows_cap;  // source rows staged per CTA
  uint8_t* out_masks;
  u64* out_packed;
  Stats* stats;
};

__device__ __forceinline__ void resize_tap(int i, int in_size, float scale, int align_corners, int& lo, int& hi, float& lerp) {
  float src;
  if (align_corners) {
    src = (float)i * scale;
  } else {
    src = (float)i + 0.5f;
    src = src * scale;
    src = src - 0.5f;
  }
  const float f = floorf(src);
  lo = max((int)f, 0);
  hi = min((int)ceilf(src), in_size - 1);
  lerp = src - f;
}

// bilinear value of one output pixel from its four source pixels (the reference's op order)
__device__ __forceinline__ float up_lerp(float tl, float tr, float bl, float br, float lx, float ly) {
  float top = tr - tl; top = top * lx; top = tl + top;
  float bot = br - bl; bot = bot * lx; bot = bl + bot;
  float v = bot - top; v = v * ly; v = top + v;
  return v;
}

__global__ void up_init_stats(Stats* s, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Stats z;
  z.count = z.sum_y = z.sum_x = 0ull;
  z.min_y = z.min_x = 0x7fffffff;
  z.max_y = z.max_x = -1;
  s[i] = z;
}

__global__ void __launch_bounds__(kUpThreads) solo_upsample_kernel(const UpArgs a) {
  extern __shared__ __align__(16) unsigned char up_smem[];
  float* rows = reinterpret_cast<float*>(up_smem);                                 // [rows_cap][w]
  int2* span = reinterpret_cast<int2*>(rows + (((size_t)a.rows_cap * a.w + 1) & ~(size_t)1));  // [rows_cap] first / last set column
  Tap* xt = reinterpret_cast<Tap*>(span + a.rows_cap);                             // [W]

  const int b = blockIdx.z, d = blockIdx.y;
  const long long hw_out = (long long)a.H * a.W;
  const long long chunk = (long long)a.iters * kUpThreads * kRun;
  const long long p_begin = (long long)blockIdx.x * chunk;
  const long long p_end = min(p_begin + chunk, hw_out);
  const int y_first = (int)(p_begin / a.W), y_last = (int)((p_end - 1) / a.W);
  int r0, r1, tmp;
  float tf;
  resize_tap(y_first, a.h, a.scale_y, a.align_corners, r0, tmp, tf);
  resize_tap(y_last, a.h, a.scale_y, a.align_corners, tmp, r1, tf);
  const int n_rows = r1 - r0 + 1;  // <= rows_cap by construction (host)
  const u64* src = a.packed + ((size_t)b * a.D + d) * a.Wd_in;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint8_t* om = a.out_masks ? a.out_masks + ((size_t)b * a.D + d) * hw_out : nullptr;
  u64* op = a.out_packed ? a.out_packed + ((size_t)b * a.D + d) * a.Wd_out : nullptr;
  const bool vec16 = om && ((reinterpret_cast<uintptr_t>(om) & 15) == 0);  // flat runs start at multiples of 16
  // every shortcut below assumes "all four corners 0 -> off, all four corners 1 -> on", i.e. 0 <= thr < 1
  const bool shortcuts = a.thr >= 0.0f && a.thr < 1.0f;
  if (shortcuts) {
    // ---- cheap rejection first: OR of the words that hold source rows r0..r1 (edge words may carry neighbouring
    // rows' bits: conservative).  Most chunks of an image see no mask at all and leave as zeros right here.
    const long long w_first = ((long long)r0 * a.w) >> 6, w_last = (((long long)(r1 + 1) * a.w - 1) >> 6);
    u64 acc = 0;
    for (long long q = w_first + tid; q <= w_last; q += kUpThreads) acc |= __ldg(src + q);
    if (!__syncthreads_or(acc != 0ull)) {
      const int len = (int)(p_end - p_begin);
      if (om) {
        if (vec16) {  // p_begin is a multiple of 16: whole 16-byte stores, then the (image-end) tail
          uint4* dst = reinterpret_cast<uint4*>(om + p_begin);
          for (int v = tid; v < (len >> 4); v += kUpThreads) dst[v] = make_uint4(0, 0, 0, 0);
          for (int q = (len & ~15) + tid; q < len; q += kUpThreads) om[p_begin + q] = 0;
        } else {
          for (int q = tid; q < len; q += kUpThreads) om[p_begin + q] = 0;
        }
      }
      if (op) {
        u64* dst = op + (p_begin >> 6);  // p_begin is a multiple of 64
        for (int v = tid; v < ((len + 63) >> 6); v += kUpThreads) dst[v] = 0ull;
      }
      return;
    }
  }

  // ---- stage the source rows: bits -> fp32 0/1, and each row's span of set columns
  for (int r = warp; r < n_rows; r += kUpThreads / 32) {
    const long long bit0 = (long long)(r0 + r) * a.w;
    int first = 0x7fffffff, last = -1;
    for (int x = lane; x < a.w; x += 32) {
      const long long q = bit0 + x;
      const unsigned on = (unsigned)((__ldg(src + (q >> 6)) >> (q & 63)) & 1ull);
      rows[(size_t)r * a.w + x] = on ? 1.0f : 0.0f;
      if (on) { first = min(first, x); last = max(last, x); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
      last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if (lane == 0) span[r] = make_int2(first, last);
  }
  __syncthreads();
  for (int x = tid; x < a.W; x += kUpThreads) {
    int lo, hi;
    float l;
    resize_tap(x, a.w, a.scale_x, a.align_corners, lo, hi, l);
    Tap t;
    t.lo = (unsigned short)lo; t.hi = (unsigned short)hi; t.lerp = l;
    xt[x] = t;
  }
  __syncthreads();

  // per-thread statistics fit 32 bits (<= iters * 16 pixels per thread, coordinates < 65536); widened at the reduction
  unsigned cnt32 = 0, sum_y32 = 0, sum_x32 = 0;
  int min_y = 0x7fffffff, max_y = -1, min_x = 0x7fffffff, max_x = -1;
  // A warp owns 512 consecutive flat pixels per step; in sub-step j lane l samples pixel base + 32 j + l, so the tap
  // table and the source rows are read without bank conflicts (neighbouring pixels share or neighbour their taps) and
  // the 32 decisions leave as one ballot = 32 packed mask bits.  Lane j keeps ballot j; a shuffle then hands every
  // lane the 16 bits of ITS 16-pixel run for the 16-byte uint8 store.
  const int chunk_len = (int)(p_end - p_begin);
  for (int it = 0; it < a.iters; ++it) {
    const int off = (it * (kUpThreads / 32) + warp) * (32 * kRun);  // offset of the warp's 512 pixels in the chunk
    if (off >= chunk_len) break;  // warp-uniform
    const long long base = p_begin + off;
    const int span_len = min(32 * kRun, chunk_len - off);
    const int ya = (int)(base / a.W), xa = (int)(base - (long long)ya * a.W);
    const int yb = (int)((base + span_len - 1) / a.W);
    unsigned mine = 0;
    // The span is cut by output row (1-2 rows for W >= 512): everything that depends on the row -- its two source
    // rows, their lerp weight and set-column spans -- is warp-uniform inside the sub-step loop.
    for (int y = ya; y <= yb; ++y) {
      const int f0 = y == ya ? 0 : (y - ya) * a.W - xa;                 // flat range of this row inside the span
      const int f1 = min(span_len, (y - ya + 1) * a.W - xa);
      int ylo, yhi;
      float yl;
      resize_tap(y, a.h, a.scale_y, a.align_corners, ylo, yhi, yl);
      const int2 s0 = span[ylo - r0], s1 = span[yhi - r0];
      const int xbase = xa - (y - ya) * a.W;                             // x = xbase + f
      {  // row-level rejection over the columns this row's part can touch
        const int c0 = xt[xbase + f0].lo, c1 = xt[xbase + f1 - 1].hi;
        if (shortcuts && (s0.y < c0 || s0.x > c1) && (s1.y < c0 || s1.x > c1)) continue;
      }
      const float* q0 = rows + (ylo - r0) * a.w;
      const float* q1 = rows + (yhi - r0) * a.w;
      unsigned row_cnt = 0;
      for (int j = f0 >> 5; j <= (f1 - 1) >> 5; ++j) {
        const int f = lane + 32 * j;
        bool on = false;
        if (f >= f0 && f < f1) {
          const int x = xbase + f;
          const Tap t = xt[x];
          const int lo = t.lo, hi = t.hi;
          // (tried: a warp-uniform all-zeros / all-ones test of the 32 pixels' source window on row-aligned bit words,
          //  so that only mask edges are sampled: its ~45 instructions per sub-step cost more than they save -- object
          //  masks 0.81 -> 1.23 ms, noise 4.2 -> 7.6 ms)
          const bool empty = shortcuts && (s0.y < lo || s0.x > hi) && (s1.y < lo || s1.x > hi);
          if (!empty) {
            on = up_lerp(q0[lo], q0[hi], q1[lo], q1[hi], t.lerp, yl) > a.thr;
            if (on) {
              row_cnt += 1; sum_x32 += (unsigned)x;
              if (x > 0) { min_x = min(min_x, x); max_x = max(max_x, x); }
            }
          }
        }
        const unsigned word = __ballot_sync(0xffffffffu, on);  // pixels base + 32 j .. + 31 (this row's part)
        if (lane == j) mine |= word;
      }
      cnt32 += row_cnt;
      sum_y32 += row_cnt * (unsigned)y;
      if (row_cnt && y > 0) { min_y = min(min_y, y); max_y = max(max_y, y); }
    }
    if (op) {  // lanes 0..15 hold the 16 ballots: two neighbours make one 64-bit word
      const unsigned hi32 = __shfl_down_sync(0xffffffffu, mine, 1);
      const long long pw = base + 64ll * (lane >> 1);
      if (lane < kRun && (lane & 1) == 0 && pw < p_end) op[pw >> 6] = (u64)mine | ((u64)hi32 << 32);
    }
    if (om) {
      const unsigned src_word = __shfl_sync(0xffffffffu, mine, lane >> 1);
      const unsigned bits = (src_word >> (16 * (lane & 1))) & 0xffffu;
      const long long pr = base + (long long)lane * kRun;  // this lane's 16-pixel run
      if (pr < p_end) {
        const int n = (int)min((long long)kRun, p_end - pr);
        if (vec16 && n == kRun) {
          uint4 v4;
          unsigned* wv = reinterpret_cast<unsigned*>(&v4);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const unsigned nib = (bits >> (4 * q)) & 15u;
            wv[q] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
          }
          *reinterpret_cast<uint4*>(om + pr) = v4;
        } else {
          for (int q = 0; q < n; ++q) om[pr + q] = (uint8_t)((bits >> q) & 1u);
        }
      }
    }
  }
  // ---- box statistics: warp reduce, then one set of atomics per warp
  u64 cnt = cnt32, sum_y = sum_y32, sum_x = sum_x32;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    sum_y += __shfl_xor_sync(0xffffffffu, sum_y, o);
    sum_x += __shfl_xor_sync(0xffffffffu, sum_x, o);
    min_y = min(min_y, __shfl_xor_sync(0xffffffffu, min_y, o));
    max_y = max(max_y, __shfl_xor_sync(0xffffffffu, max_y, o));
    min_x = min(min_x, __shfl_xor_sync(0xffffffffu, min_x, o));
    max_x = max(max_x, __shfl_xor_sync(0xffffffffu, max_x, o));
  }
  if (lane == 0 && cnt) {
    Stats* s = a.stats + (size_t)b * a.D + d;
    atomicAdd(&s->count, cnt);
    atomicAdd(&s->sum_y, sum_y);
    atomicAdd(&s->sum_x, sum_x);
    if (max_y >= 0) { atomicMin(&s->min_y, min_y); atomicMax(&s->max_y, max_y); }
    if (max_x >= 0) { atomicMin(&s->min_x, min_x); atomicMax(&s->max_x, max_x); }
  }
}

// solo_v2.py:606-625: mean = sum / (count + 1e-5); where(yy > 0, yy, mean); min / max over all pixels
__global__ void up_boxes_kernel(const Stats* stats, int n, float* boxes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Stats s = stats[i];
  const float den = (float)s.count + 1e-5f;
  const float ymean = (float)s.sum_y / den, xmean = (float)s.sum_x / den;
  const float ymin = s.max_y >= 0 ? (float)s.min_y : INFINITY, ymax = s.max_y >= 0 ? (float)s.max_y : -INFINITY;
  const float xmin = s.max_x >= 0 ? (float)s.min_x : INFINITY, xmax = s.max_x >= 0 ? (float)s.max_x : -INFINITY;
  boxes[i * 4 + 0] = fminf(ymin, ymean);
  boxes[i * 4 + 1] = fminf(xmin, xmean);
  boxes[i * 4 + 2] = fmaxf(ymax, ymean);
  boxes[i * 4 + 3] = fmaxf(xmax, xmean);
}

struct SoloPixel {
  const u64* src;  // packed source mask
  int h, w, align_corners;
  float scale_y, scale_x, thr;
  int y0, y1;
  __device__ __forceinline__ float bit(int y, int x) const {
    const long long q = (long long)y * w + x;
    return ((src[q >> 6] >> (q & 63)) & 1ull) ? 1.0f : 0.0f;
  }
  __device__ __forceinline__ bool operator()(int y, int x) const {
    if (y < y0 || y > y1) return false;
    int ylo, yhi, xlo, xhi;
    float ly, lx;
    resize_tap(y, h, scale_y, align_corners, ylo, yhi, ly);
    resize_tap(x, w, scale_x, align_corners, xlo, xhi, lx);
    return up_lerp(bit(ylo, xlo), bit(ylo, xhi), bit(yhi, xlo), bit(yhi, xhi), lx, ly) > thr;
  }
};

// CTA-wide min of lo and max of hi (every thread calls it)
__device__ __forceinline__ void block_min_max(int& lo, int& hi, int* s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if (threadIdx.x == 0) { s[0] = INT_MAX; s[1] = INT_MIN; }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { atomicMin(&s[0], lo); atomicMax(&s[1], hi); }
  __syncthreads();
  lo = s[0]; hi = s[1];
  __syncthreads();
}

// One CTA per (image, detection): count pass (kWrite = false) or write pass of the COCO RLE of its image mask.
// For 0 <= thr < 1 a pixel whose four source pixels are 0 is off, so only output rows / columns whose taps reach the
// set source rows / columns are walked; an empty source mask (padding rows) walks nothing and encodes [H*W].
template <bool kWrite>
__global__ void __launch_bounds__(kRleThreads) solo_rle_kernel(const UpArgs a, RleOut o, int stage_src) {
  extern __shared__ u64 s_src[];
  __shared__ RleShared sh;
  __shared__ int s_mm[2];
  const long long m = (long long)blockIdx.y * a.D + blockIdx.x;
  long long beg = 0, end = 0;
  if (kWrite) {
    beg = o.offsets[m]; end = o.offsets[m + 1];
    if (end > o.capacity) return;  // block-uniform: this string does not fit
  }
  SoloPixel px;
  px.src = a.packed + m * a.Wd_in;
  if (stage_src) {
    for (int i = threadIdx.x; i < a.Wd_in; i += kRleThreads) s_src[i] = __ldg(px.src + i);
    __syncthreads();
    px.src = s_src;
  }
  px.h = a.h; px.w = a.w; px.align_corners = a.align_corners;
  px.scale_y = a.scale_y; px.scale_x = a.scale_x; px.thr = a.thr;
  int y0 = 0, y1 = a.H - 1, x0 = 0, x1 = a.W - 1;
  if (a.thr >= 0.0f && a.thr < 1.0f) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int r0 = INT_MAX, r1 = INT_MIN, c0 = INT_MAX, c1 = INT_MIN;  // set source rows / columns
    for (int r = warp; r < a.h; r += kRleWarps) {
      for (int x = lane; x < a.w; x += 32) {
        if (px.bit(r, x) != 0.0f) {
          r0 = min(r0, r); r1 = max(r1, r);
          c0 = min(c0, x); c1 = max(c1, x);
        }
      }
    }
    block_min_max(r0, r1, s_mm);
    block_min_max(c0, c1, s_mm);
    y0 = INT_MAX; y1 = INT_MIN; x0 = INT_MAX; x1 = INT_MIN;
    if (r1 >= 0) {
      for (int y = threadIdx.x; y < a.H; y += kRleThreads) {
        int lo, hi;
        float l;
        resize_tap(y, a.h, a.scale_y, a.align_corners, lo, hi, l);
        if (hi >= r0 && lo <= r1) { y0 = min(y0, y); y1 = max(y1, y); }
      }
      for (int x = threadIdx.x; x < a.W; x += kRleThreads) {
        int lo, hi;
        float l;
        resize_tap(x, a.w, a.scale_x, a.align_corners, lo, hi, l);
        if (hi >= c0 && lo <= c1) { x0 = min(x0, x); x1 = max(x1, x); }
      }
    }
    block_min_max(y0, y1, s_mm);
    block_min_max(x0, x1, s_mm);
  }
  px.y0 = y0; px.y1 = y1;
  rle_encode_mask<kWrite>(px, rle_walk_of(a.H, a.W, y0, y1, x0, x1), sh, o.offsets + m + 1, o.chars + beg, end - beg);
}

struct UpPlan {
  int iters, rows_cap;
  size_t smem;
  float scale_y, scale_x;
};
int up_plan(const d2b_solo_upsample_params* p, UpPlan& pl) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->batch >= 0 && p->num_dets >= 0, "solo_upsample: negative sizes");
  D2B_REQUIRE(p->batch <= 65535 && p->num_dets <= 65535, "solo_upsample: batch / num_dets too large");
  D2B_REQUIRE(p->mask_h >= 1 && p->mask_w >= 1 && p->image_h >= 1 && p->image_w >= 1, "solo_upsample: empty mask / image");
  D2B_REQUIRE(p->mask_w <= 65535 && p->mask_h <= 65535 && (long long)p->image_h * p->image_w < (1ll << 31),
              "solo_upsample: sizes out of range");
  const int ac = p->align_corners != 0;
  pl.scale_y = (ac && p->image_h > 1) ? (float)(p->mask_h - 1) / (float)(p->image_h - 1) : (float)p->mask_h / (float)p->image_h;
  pl.scale_x = (ac && p->image_w > 1) ? (float)(p->mask_w - 1) / (float)(p->image_w - 1) : (float)p->mask_w / (float)p->image_w;
  for (int iters = 8; iters >= 1; iters >>= 1) {
    const long long chunk = (long long)iters * kUpThreads * kRun;
    const long long out_rows = chunk / p->image_w + 2;
    long long rows = (long long)ceil((double)out_rows * (double)pl.scale_y) + 3;
    if (rows > p->mask_h) rows = p->mask_h;
    const size_t smem = (((size_t)rows * p->mask_w + 1) & ~(size_t)1) * 4 + (size_t)rows * 8 + (size_t)p->image_w * sizeof(Tap) + 16;
    if (smem <= 96 * 1024 || iters == 1) {
      pl.iters = iters;
      pl.rows_cap = (int)rows;
      pl.smem = smem;
      D2B_REQUIRE(smem <= 200 * 1024, "solo_upsample: a %d x %d -> %d x %d resize needs %zu bytes of shared memory per CTA",
                  p->mask_h, p->mask_w, p->image_h, p->image_w, smem);
      return D2B_OK;
    }
  }
  return D2B_EINVAL;
}
}  // namespace
}  // namespace d2b

using namespace d2b;

extern "C" size_t d2b_solo_upsample_workspace_bytes(const d2b_solo_upsample_params* p) {
  UpPlan pl;
  if (up_plan(p, pl) != D2B_OK) return 0;
  return ws_slice(sizeof(Stats) * (size_t)p->batch * (p->num_dets > 0 ? p->num_dets : 1));
}

extern "C" int d2b_solo_upsample(const d2b_solo_upsample_params* p, void* workspace, size_t workspace_bytes,
                                 d2b_stream_t stream) {
  UpPlan pl;
  int rc = up_plan(p, pl);
  if (rc != D2B_OK) return rc;
  const int n = p->batch * p->num_dets;
  const bool rle = p->out_rle_offsets != nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rle) {
    rc = rle_check("solo_upsample", p->out_rle, p->rle_capacity);
    if (rc != D2B_OK) return rc;
  }
  if (n == 0) {
    if (rle) D2B_CUDA(cudaMemsetAsync(p->out_rle_offsets, 0, sizeof(int64_t), st));
    return D2B_OK;
  }
  D2B_REQUIRE(p->packed_masks && p->out_boxes, "solo_upsample: NULL pointer");
  const size_t need = ws_slice(sizeof(Stats) * (size_t)n);
  if (workspace == nullptr || workspace_bytes < need) {
    set_last_error("solo_upsample needs %zu workspace bytes", need);
    return D2B_EWORKSPACE;
  }
  UpArgs a;
  a.packed = reinterpret_cast<const u64*>(p->packed_masks);
  a.B = p->batch; a.D = p->num_dets; a.h = p->mask_h; a.w = p->mask_w; a.H = p->image_h; a.W = p->image_w;
  a.Wd_in = (int)(((long long)p->mask_h * p->mask_w + 63) / 64);
  a.Wd_out = (int)(((long long)p->image_h * p->image_w + 63) / 64);
  a.align_corners = p->align_corners != 0;
  a.scale_y = pl.scale_y; a.scale_x = pl.scale_x; a.thr = p->mask_threshold;
  a.iters = pl.iters; a.rows_cap = pl.rows_cap;
  a.out_masks = p->out_masks;
  a.out_packed = reinterpret_cast<u64*>(p->out_packed_masks);
  a.stats = static_cast<Stats*>(workspace);
  up_init_stats<<<(n + 255) / 256, 256, 0, st>>>(a.stats, n);
  D2B_LAUNCH_CHECK();
  if (pl.smem > 48 * 1024) {
    static size_t set_to = 0;  // grow-only opt-in (any device: the attribute is per function per device, re-setting is cheap)
    if (pl.smem > set_to) set_to = pl.smem;
    D2B_CUDA(cudaFuncSetAttribute(solo_upsample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)set_to));
  }
  const long long chunk = (long long)pl.iters * kUpThreads * kRun;
  const long long hw_out = (long long)p->image_h * p->image_w;
  const dim3 grid((unsigned)((hw_out + chunk - 1) / chunk), (unsigned)p->num_dets, (unsigned)p->batch);
  solo_upsample_kernel<<<grid, kUpThreads, pl.smem, st>>>(a);
  D2B_LAUNCH_CHECK();
  up_boxes_kernel<<<(n + 255) / 256, 256, 0, st>>>(a.stats, n, p->out_boxes);
  D2B_LAUNCH_CHECK();
  if (rle) {
    RleOut o;
    o.chars = p->out_rle; o.offsets = p->out_rle_offsets; o.capacity = p->rle_capacity;
    const size_t src_bytes = sizeof(u64) * (size_t)a.Wd_in;
    const int stage = src_bytes <= 64 * 1024;  // 200 x 336 source masks: 8.4 KB
    const size_t smem = stage ? src_bytes : 0;
    D2B_CUDA(allow_dynamic_smem(solo_rle_kernel<false>, smem));
    D2B_CUDA(allow_dynamic_smem(solo_rle_kernel<true>, smem));
    const dim3 g((unsigned)p->num_dets, (unsigned)p->batch);
    solo_rle_kernel<false><<<g, kRleThreads, smem, st>>>(a, o, stage);
    D2B_LAUNCH_CHECK();
    rle_offsets_kernel<<<1, kRleThreads, 0, st>>>(o.offsets, n);
    D2B_LAUNCH_CHECK();
    solo_rle_kernel<true><<<g, kRleThreads, smem, st>>>(a, o, stage);
    D2B_LAUNCH_CHECK();
  }
  return D2B_OK;
}
