// mask_rle.cuh -- COCO run-length encoding of image masks that a producer kernel defines pixel by pixel, without the
// image plane ever existing in memory.  Shared by d2b_paste_masks (paste_masks.cu) and d2b_solo_upsample
// (solo_upsample.cu); each supplies a Pixel functor `bool operator()(int y, int x)` that applies its exact per-pixel
// rule, and a rectangle outside which every pixel is 0.
//
// Format (pycocotools maskApi.c rleEncode + rleToString, restated in numpy in tests/coco_rle.py):
//   * the mask is walked column-major (j = x*H + y); cnts[] alternate starting with a run of ZEROS (cnts[0] may be 0)
//     and the last run ends at H*W;
//   * count i is written as x = cnts[i], minus cnts[i-2] when i > 2 (not i >= 2), in 5-bit groups, least significant
//     first: c = x & 31, x >>= 5 (arithmetic), more = (c & 16) ? x != -1 : x != 0, c |= 32 if more, emit c + 48.
//
// Walk: a CTA per mask visits the 32-row words (rows 32k .. 32k+31 of one column) that meet the rectangle, in
// column-major order, 256 words per chunk.  Warp q of the CTA evaluates words 32q .. 32q+31 of the chunk one ballot at
// a time (lane = row), so thread t ends up holding word t.  Transitions of a word are
//   bits ^ (bits << 1 | last bit of the preceding pixel)
// where the preceding pixel is the previous word's last one when the two are contiguous in column-major order and 0
// otherwise; a word whose last pixel is set and whose successor is not contiguous adds a fall just past its end.  A
// block scan of the per-word counts places the transition positions of the chunk in order in shared memory.  The
// byte length of run g depends only on t[g-3] .. t[g] (the transitions), so every run of the chunk is sized in
// parallel; the last three transitions, the transition count and the previous word's last bit carry to the next
// chunk, so a mask may have any number of runs.  The count pass stores each mask's byte length; an in-place scan
// turns the lengths into offsets; the write pass re-evaluates the pixels and writes the bytes of every string that
// fits the caller's capacity.
#pragma once
#include "common.cuh"

namespace d2b {
namespace {

constexpr int kRleThreads = 256;
constexpr int kRleWarps = kRleThreads / 32;
constexpr int kRleMaxTrans = kRleThreads * 33;  // per chunk: 32 inside a word + one fall after it

struct RleShared {
  int pos[kRleMaxTrans];  // transition positions of the current chunk, ascending
  unsigned char last[kRleThreads];
  int iscan[kRleWarps];
  long long lscan[kRleWarps];
};

struct RleOut {
  uint8_t* chars;
  int64_t* offsets;  // [num_masks + 1]
  long long capacity;
};

// The words of one mask that meet rows y0..y1 and columns x0..x1.
struct RleWalk {
  int H, W;
  int x0, ncols;  // columns x0 .. x0 + ncols - 1
  int k0, nk;     // words k0 .. k0 + nk - 1 of each column (rows 32 k0 ..)
  bool wrap;      // the last visited word of a column is contiguous with the first of the next column
};
__device__ __forceinline__ RleWalk rle_walk_of(int H, int W, int y0, int y1, int x0, int x1) {
  RleWalk wk;
  wk.H = H; wk.W = W;
  if (y0 > y1 || x0 > x1) {
    wk.x0 = wk.ncols = wk.k0 = wk.nk = 0;
    wk.wrap = false;
    return wk;
  }
  wk.x0 = x0; wk.ncols = x1 - x0 + 1;
  wk.k0 = y0 >> 5; wk.nk = (y1 >> 5) - wk.k0 + 1;
  wk.wrap = wk.k0 == 0 && wk.k0 + wk.nk == ((H + 31) >> 5);
  return wk;
}

__device__ __forceinline__ int rle_len(long long x) {
  int n = 0;
  bool more;
  do {
    const int c = (int)(x & 0x1f);
    x >>= 5;
    more = (c & 0x10) ? x != -1 : x != 0;
    ++n;
  } while (more);
  return n;
}

__device__ __forceinline__ void rle_put(long long x, uint8_t* dst, long long at, long long limit) {
  bool more;
  do {
    int c = (int)(x & 0x1f);
    x >>= 5;
    more = (c & 0x10) ? x != -1 : x != 0;
    if (more) c |= 0x20;
    D2B_BOUND(at, limit);
    dst[at++] = (uint8_t)(c + 48);
  } while (more);
}

// Exclusive prefix of v over the CTA; `total` = the sum.  Every thread must call it.
template <typename T>
__device__ __forceinline__ T rle_block_scan(T v, T* s, T& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s[warp] = inc;
  __syncthreads();
  T before = 0;
  total = 0;
#pragma unroll
  for (int q = 0; q < kRleWarps; ++q) {
    const T wv = s[q];
    if (q < warp) before += wv;
    total += wv;
  }
  __syncthreads();
  return before + inc - v;
}

// Count pass (kWrite = false): *len_out = byte length of the mask's string.
// Write pass (kWrite = true): the string to dst[0 .. limit).  Every thread of the CTA calls it.
template <bool kWrite, class Pixel>
__device__ void rle_encode_mask(const Pixel& px, const RleWalk& wk, RleShared& sh, int64_t* len_out, uint8_t* dst,
                                long long limit) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long HW = (long long)wk.H * wk.W;
  const int NW = wk.ncols * wk.nk;  // <= W * ceil(H / 32) < 2^31
  long long G = 0;             // transitions before the chunk
  int c1 = 0, c2 = 0, c3 = 0;  // t[G-1], t[G-2], t[G-3]
  unsigned prev_last = 0;      // last pixel of the word before the chunk
  long long bytes = 0;         // write pass: bytes before the chunk; count pass: this thread's bytes
  for (int wb = 0; wb < NW; wb += kRleThreads) {
    unsigned mine = 0;
    {
      const int w0 = wb + warp * 32;
      int c = w0 / wk.nk, kk = w0 - c * wk.nk;  // column and word of word w0 + j, stepped below
      for (int j = 0; j < 32 && w0 + j < NW; ++j) {  // warp-uniform bound
        const int y = 32 * (wk.k0 + kk) + lane;
        const bool on = y < wk.H && px(y, wk.x0 + c);
        const unsigned b = __ballot_sync(0xffffffffu, on);
        if (lane == j) mine = b;
        if (++kk == wk.nk) { kk = 0; ++c; }
      }
    }
    const int w = wb + tid;
    const bool valid = w < NW;
    int s = 0, len = 0, k = 0;
    unsigned last = 0;
    if (valid) {
      const int c = w / wk.nk;
      k = w - c * wk.nk;
      const int r = 32 * (wk.k0 + k);
      len = min(32, wk.H - r);
      s = (wk.x0 + c) * wk.H + r;
      last = (mine >> (len - 1)) & 1u;
    }
    sh.last[tid] = (unsigned char)last;
    __syncthreads();
    unsigned T = 0;
    int ext = 0;
    if (valid) {
      const bool from_prev = w > 0 && (k != 0 || wk.wrap);
      const unsigned pb = from_prev ? (tid ? (unsigned)sh.last[tid - 1] : prev_last) : 0u;
      const unsigned lm = len == 32 ? 0xffffffffu : ((1u << len) - 1u);
      T = (mine ^ ((mine << 1) | pb)) & lm;
      const bool to_next = w + 1 < NW && (k != wk.nk - 1 || wk.wrap);
      ext = (last && !to_next && (long long)s + len < HW) ? 1 : 0;
    }
    int K;
    int q = rle_block_scan<int>(__popc(T) + ext, sh.iscan, K);
    for (unsigned t = T; t; t &= t - 1) {
      D2B_BOUND(q, kRleMaxTrans);
      sh.pos[q++] = s + __ffs(t) - 1;
    }
    if (ext) {
      D2B_BOUND(q, kRleMaxTrans);
      sh.pos[q] = s + len;
    }
    prev_last = sh.last[kRleThreads - 1];  // only read again when this chunk was full
    __syncthreads();
    auto at = [&](int i) -> int { return i >= 0 ? sh.pos[i] : (i == -1 ? c1 : (i == -2 ? c2 : c3)); };
    for (int r0 = 0; r0 < K; r0 += kRleThreads) {  // K is CTA-uniform
      const int i = r0 + tid;
      long long x = 0;
      int n = 0;
      if (i < K) {
        const long long g = G + i;  // run g ends at transition g
        x = (long long)sh.pos[i] - (g >= 1 ? at(i - 1) : 0);
        if (g > 2) x -= (long long)at(i - 2) - at(i - 3);
        n = rle_len(x);
      }
      if (kWrite) {
        int tot;
        const int o = rle_block_scan<int>(n, sh.iscan, tot);
        if (i < K) rle_put(x, dst, bytes + o, limit);
        bytes += tot;
      } else {
        bytes += n;
      }
    }
    const int n1 = at(K - 1), n2 = at(K - 2), n3 = at(K - 3);
    c1 = n1; c2 = n2; c3 = n3;
    G += K;
    __syncthreads();  // pos / last are refilled by the next chunk
  }
  // the last run ends at H*W
  long long x = HW - (G >= 1 ? c1 : 0);
  if (G > 2) x -= (long long)c2 - c3;
  if (kWrite) {
    if (tid == 0) rle_put(x, dst, bytes, limit);
  } else {
    if (tid == 0) bytes += rle_len(x);
    long long total;
    rle_block_scan<long long>(bytes, sh.lscan, total);
    if (tid == 0) *len_out = total;
  }
}

// offsets[1..n] hold the byte lengths; make them running totals and set offsets[0] = 0.  One CTA.
__global__ void __launch_bounds__(kRleThreads) rle_offsets_kernel(int64_t* offsets, long long n) {
  __shared__ long long s[kRleWarps];
  long long carry = 0;
  for (long long b = 0; b < n; b += kRleThreads) {
    const long long i = b + threadIdx.x;
    const long long v = i < n ? offsets[i + 1] : 0;
    long long total;
    const long long ex = rle_block_scan<long long>(v, s, total);
    if (i < n) offsets[i + 1] = carry + ex + v;
    carry += total;
  }
  if (threadIdx.x == 0) offsets[0] = 0;
}

// Host side: validates the optional RLE output fields of a params struct.
inline int rle_check(const char* op, const uint8_t* chars, int64_t capacity) {
  D2B_REQUIRE(capacity >= 0, "%s: rle_capacity=%lld is negative", op, (long long)capacity);
  D2B_REQUIRE(capacity == 0 || chars != nullptr, "%s: rle_capacity=%lld with out_rle NULL", op, (long long)capacity);
  return D2B_OK;
}

}  // namespace
}  // namespace d2b
