// solo_dynconv.cu -- SOLOv2 mask generation fused with the mask stage (SURVEY.md 8f "next" #4):
//   solo_v2.py:499-517, 530-533   mask_logits = conv2d(mask_features, pred_kernels 1x1)  ->  sigmoid  ->  > thr
//                                 -> sum_masks, sum(scores * masks)
// The 1x1 "dynamic convolution" is a GEMM per image:  logits[n, HW] = kernels[n, E] . features[HW, E]^T.  It is the
// one contraction on the path, so it runs on the 5th-generation tensor cores:
//   * tcgen05.mma kind::tf32, M=128 (mask kernels) x N=256 (pixels) x K=8, accumulators in TMEM (2 x 256 columns,
//     double buffered), operands staged by TMA (cp.async.bulk.tensor, 128-byte swizzle) through an mbarrier ring;
//     with more than 128 mask kernels two CTAs of a cluster form a cta_group::2 pair (M=256): each CTA owns one
//     128-row block of D in its own TMEM and stages / converts only HALF of the feature tile, the leader CTA issues
//     the MMAs for both and tcgen05.commit multicasts the completion to the barriers of both CTAs;
//   * fp32 accuracy from three tf32 products per k-step (3xTF32: a = a_hi + a_lo, D += a_lo.b_hi + a_hi.b_hi +
//     a_hi.b_lo; the dropped a_lo.b_lo is O(2^-22)): the kernels are split once by a tiny prologue kernel (both halves
//     rounded to tf32); for the feature tile the raw fp32 tile IS the hi half (the tensor core ignores the low 13
//     mantissa bits) and four converter warps write lo = x - trunc_tf32(x) beside it between the TMA and the MMA
//     (elementwise, so the swizzled layout is preserved), published to the async proxy with fence.proxy.async;
//   * epilogue warps read the accumulators with tcgen05.ld (thread = one mask row, 16 consecutive pixels per load),
//     take the threshold decision on the logit (exact sigmoid only inside the guard band around logit(thr), the rule
//     of solo_encode_kernel) and emit BIT-PACKED masks, exact mask sums and the score sums (2-MUFU sigmoid: the sums
//     are tolerance-based like every fp32 reduction here) -- the 4 B/pixel logits (134 MB per image at
//     500 x 200 x 336) never exist.
// Persistent: one CTA (pair) per SM (pair) walks the (image, pixel tile, row block) tiles round-robin.
// Non-finite features / kernels give unspecified bits (inf - inf in the lo half).
// Warp roles: 0 = TMA producer, 1 = MMA issuer (+ TMEM owner), 2-5 = converters, 6-13 = epilogue.
#include <cuda.h>
#include <math.h>

#include "kernels.cuh"

namespace d2b {
namespace {
typedef unsigned long long u64;

constexpr int kBM = 128;   // mask kernels per tile (UMMA M, = TMEM lanes)
constexpr int kBN = 256;   // pixels per tile (UMMA N, = TMEM columns of one accumulator)
constexpr int kUmmaK = 8;  // tf32 MMA depth
constexpr int kThreads = 448;
constexpr int kCvtThreads = 128, kEpiThreads = 256;  // 2 epilogue warps per TMEM lane quarter (half the columns each)
constexpr uint32_t kTmemCols = 512;

// One pipeline stage holds a K block of BK fp32 = one swizzle row (BK = 32: 128-byte swizzle, BK = 16: 64-byte
// swizzle); the ring fills 192 KB: 2 x 96 KB / 4 x 48 KB for one CTA, 3 x 64 KB / 6 x 32 KB for a pair (which stages
// only half of the feature tile per CTA).
template <int BK, int CTAS>
struct Cfg {
  static_assert(BK == 32 || BK == 16, "one swizzle row per K block");
  static_assert(CTAS == 1 || CTAS == 2, "one CTA or a cta_group::2 pair");
  static constexpr uint32_t kRowBytes = BK * 4;
  static constexpr int kBRows = kBN / CTAS;  // feature rows (pixels) staged and converted by one CTA
  static constexpr uint32_t kABytes = kBM * kRowBytes;
  static constexpr uint32_t kBBytes = kBRows * kRowBytes;
  static constexpr uint32_t kStageBytes = 2 * kABytes + 2 * kBBytes;  // A_hi, A_lo, B (raw = hi), B_lo
  static constexpr uint32_t kTxBytes = 2 * kABytes + kBBytes;        // what the TMA writes per stage
  static constexpr int kStages = (192 * 1024) / kStageBytes;          // 2 / 4 (one CTA), 3 / 6 (pair)
  static constexpr size_t kSmemBytes = 1024 + (size_t)kStages * kStageBytes + 256;
  // UMMA shared-memory descriptor, K-major: 8-row groups (SBO) 8 * row bytes apart, LBO unused (1), version 1,
  // layout type 2 = SWIZZLE_128B / 4 = SWIZZLE_64B
  static constexpr uint64_t kDescHi = (1ull << 16) | ((uint64_t)(8 * kRowBytes >> 4) << 32) | (1ull << 46) |
                                      ((uint64_t)(BK == 32 ? 2 : 4) << 61);
  // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, N >> 3, M >> 4
  // (M = 256 for the pair: each CTA owns 128 rows of D and stages half of B)
  static constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kBN >> 3) << 17) |
                                     ((uint32_t)((kBM * CTAS) >> 4) << 24);
};

struct DynArgs {
  const int32_t* counts;
  int B, n, E, RB, PT, KB;
  long long hw;
  int Wd;
  float thr, lo, hi;
  u64* packed;
  float* sum_masks;
  float* score_sums;
  float* logits;  // optional
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
               : "memory");
}
// Bounded wait: a protocol bug traps (the launch fails with an error) instead of hanging the device.
template <bool CLUSTER = false>  // CLUSTER: the arrivals come from the peer CTA too (acquire at cluster scope)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  long long t0 = 0;
  for (unsigned spin = 0;; ++spin) {
    if constexpr (CLUSTER)
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(ok)
          : "r"(bar), "r"(parity)
          : "memory");
    else
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(ok)
          : "r"(bar), "r"(parity)
          : "memory");
    if (ok) return;
    if ((spin & 1023u) == 1023u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 20000000000ll) __trap();  // ~10 s: a kernel that takes 1 ms is deadlocked by then
    }
  }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
template <int BK>
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | Cfg<BK, 1>::kDescHi;
}
template <int CTAS>
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CTAS == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// tcgen05.commit: the mbarrier (same offset in every CTA of the pair) is signalled when the MMAs issued so far are done
template <int CTAS>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  if constexpr (CTAS == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
  else
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3)
                 : "memory");
}
// arrive on the barrier at the same offset in the LEADER CTA (rank 0) of the pair
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, 0;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
// sigmoid for the score sums of the fused path: 2 MUFU ops, ~2 ulp (the logits themselves carry ~1e-6 of rounding)
__device__ __forceinline__ float fast_sigmoid(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.44269504088896341f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}
__device__ __noinline__ bool exact_sigmoid_above(float x, float thr) { return d2b_sigmoidf(x) > thr; }
__device__ __forceinline__ void split4(const float4 v, float4& h, float4& l) {
  h.x = tf32_rn(v.x); h.y = tf32_rn(v.y); h.z = tf32_rn(v.z); h.w = tf32_rn(v.w);
  l.x = tf32_rn(v.x - h.x); l.y = tf32_rn(v.y - h.y); l.z = tf32_rn(v.z - h.z); l.w = tf32_rn(v.w - h.w);
}

// kernels [B*n*E] -> hi / lo halves (both exactly representable in tf32)
__global__ void dyn_split_kernel(const float4* x, float4* hi, float4* lo, long long total4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  float4 h, l;
  split4(__ldg(x + i), h, l);
  hi[i] = h;
  lo[i] = l;
}

// Every role walks the same tile sequence.  Tiles are numbered (image, pixel tile, row block) with the row block
// fastest and dealt round-robin to the CTAs, so the RB row blocks of one pixel tile run at the same time on
// neighbouring SMs: the feature tile comes from DRAM once and from L2 for the others (measured: DRAM reads
// 4.45 GB -> see profiles/), and a CTA keeps its row block for long runs (row sums stay in registers).
template <int CTAS>
struct TileIter {
  long long t, total;
  int b, rb, pt, units, rank;
  const DynArgs& a;
  __device__ TileIter(const DynArgs& a_, int rank_) : rank(rank_), a(a_) {
    units = (a.RB + CTAS - 1) / CTAS;  // row-block groups: one row block per CTA of the pair
    total = (long long)a.B * units * a.PT;
    t = (long long)(blockIdx.x / CTAS) - (long long)(gridDim.x / CTAS);
  }
  __device__ bool next() {
    for (;;) {
      t += gridDim.x / CTAS;
      if (t >= total) return false;
      const int u = (int)(t % units);
      const long long r = t / units;
      pt = (int)(r % a.PT);
      b = (int)(r / a.PT);
      rb = u * CTAS + rank;
      const int cnt = a.counts ? min(a.counts[b], a.n) : a.n;
      // groups past the valid prefix have no work (their words are pre-zeroed); the test is on the group's FIRST row
      // block so that both CTAs of a pair take the same decision
      if (u * CTAS * kBM < cnt) return true;
    }
  }
};

template <int BK, int CTAS>
__global__ void __launch_bounds__(kThreads, 1)
solo_dynconv_kernel(const __grid_constant__ CUtensorMap tm_ahi, const __grid_constant__ CUtensorMap tm_alo,
                    const __grid_constant__ CUtensorMap tm_feat, const DynArgs a) {
  using C = Cfg<BK, CTAS>;
  constexpr int kBK = BK, kStages = C::kStages;
  constexpr uint32_t kABytes = C::kABytes, kBBytes = C::kBBytes, kStageBytes = C::kStageBytes, kTxBytes = C::kTxBytes;
  uint32_t rank = 0;  // CTA rank in the pair; rank 0 (the leader) issues the MMAs and owns the cross-CTA barriers
  if constexpr (CTAS == 2) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // swizzle-128B tiles need 1024-byte alignment
  const uint32_t bars = base + kStages * kStageBytes;
  // barrier slots (8 B each): full_raw[s], full_cvt[s], empty[s], tmem_full[2], tmem_empty[2], then the TMEM address
  auto full_raw = [&](int s) { return bars + 8u * s; };
  auto full_cvt = [&](int s) { return bars + 8u * (kStages + s); };
  auto empty = [&](int s) { return bars + 8u * (2 * kStages + s); };
  auto tmem_full = [&](int s) { return bars + 8u * (3 * kStages + s); };
  auto tmem_empty = [&](int s) { return bars + 8u * (3 * kStages + 2 + s); };
  const uint32_t tmem_slot = bars + 8u * (3 * kStages + 4);
  auto sA_hi = [&](int s) { return base + s * kStageBytes; };
  auto sA_lo = [&](int s) { return base + s * kStageBytes + kABytes; };
  auto sB_hi = [&](int s) { return base + s * kStageBytes + 2 * kABytes; };
  auto sB_lo = [&](int s) { return base + s * kStageBytes + 2 * kABytes + kBBytes; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_raw(s), 1);
      mbar_init(full_cvt(s), kCvtThreads * CTAS);
      mbar_init(empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tmem_full(s), 1);
      mbar_init(tmem_empty(s), kEpiThreads * CTAS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: the whole 512 columns (one CTA per SM by shared-memory footprint)
    if constexpr (CTAS == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {  // the same warp of both CTAs, same destination offset
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync_all();  // the peer's barriers are initialised before anyone signals them
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0) {
      TileIter<CTAS> it(a, rank);
      int s = 0;
      uint32_t ph = 0;
      while (it.next()) {
        for (int kb = 0; kb < a.KB; ++kb) {
          mbar_wait(empty(s), ph ^ 1u);
          mbar_expect_tx(full_raw(s), kTxBytes);
          tma_load_3d(sA_hi(s), &tm_ahi, full_raw(s), kb * kBK, it.rb * kBM, it.b);
          tma_load_3d(sA_lo(s), &tm_alo, full_raw(s), kb * kBK, it.rb * kBM, it.b);
          tma_load_3d(sB_hi(s), &tm_feat, full_raw(s), kb * kBK, it.pt * kBN + (int)rank * C::kBRows, it.b);
          if (++s == kStages) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer (one thread)
    if (lane == 0 && rank == 0) {
      TileIter<CTAS> it(a, rank);
      int s = 0;
      uint32_t ph = 0;
      uint32_t n_tile = 0;
      while (it.next()) {
        const uint32_t as = n_tile & 1u, aph = (n_tile >> 1) & 1u;
        ++n_tile;
        mbar_wait<CTAS == 2>(tmem_empty(as), aph ^ 1u);  // the epilogue (of both CTAs) has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + as * kBN;
        for (int kb = 0; kb < a.KB; ++kb) {
          mbar_wait(full_raw(s), ph);
          mbar_wait<CTAS == 2>(full_cvt(s), ph);  // converters of both CTAs (each waited for its own TMA)
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k) {
            const uint32_t ko = k * kUmmaK * 4;  // bytes along K inside the swizzle row
            const uint64_t ahi = umma_desc<BK>(sA_hi(s) + ko), alo = umma_desc<BK>(sA_lo(s) + ko);
            const uint64_t bhi = umma_desc<BK>(sB_hi(s) + ko), blo = umma_desc<BK>(sB_lo(s) + ko);
            umma_tf32<CTAS>(d, alo, bhi, C::kIdesc, (kb | k) != 0);  // consecutive MMAs share one operand tile
            umma_tf32<CTAS>(d, ahi, bhi, C::kIdesc, 1u);
            umma_tf32<CTAS>(d, ahi, blo, C::kIdesc, 1u);
          }
          umma_commit<CTAS>(empty(s));  // implies tcgen05.fence::before_thread_sync
          if (++s == kStages) { s = 0; ph ^= 1u; }
        }
        umma_commit<CTAS>(tmem_full(as));
      }
    }
  } else if (warp < 6) {
    // ===================================================== converters: feature tile -> tf32 hi (in place) + lo
    const int tid = threadIdx.x - 64;
    TileIter<CTAS> it(a, rank);
    int s = 0;
    uint32_t ph = 0;
    while (it.next()) {
      for (int kb = 0; kb < a.KB; ++kb) {
        mbar_wait(full_raw(s), ph);
        const uint32_t src = sB_hi(s), dst = sB_lo(s);
#pragma unroll 4
        for (int i = tid; i < (int)(kBBytes / 16); i += kCvtThreads) {
          float4 v, l;
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(src + 16u * i));
          // The tensor core reads only the upper 19 bits of a tf32 operand, so the raw tile already IS the hi half
          // (x truncated to tf32); the converter adds lo = x - trunc(x), exact in fp32 with <= 13 significant bits
          // (the MMA keeps its upper 11: < 2^-20 |x| lost, in the direction of x, i.e. a scale of the dot product by
          // 1 - O(2^-21), plus zero-mean noise far below the fp32 rounding of the sum).  No write-back of hi: one
          // LDS + one STS per 16 bytes, which matters because this kernel is bound by shared-memory bandwidth.
          l.x = v.x - tf32_trunc(v.x); l.y = v.y - tf32_trunc(v.y); l.z = v.z - tf32_trunc(v.z); l.w = v.w - tf32_trunc(v.w);
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 16u * i), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the tensor core
        if constexpr (CTAS == 1) mbar_arrive(full_cvt(s));
        else mbar_arrive_leader(full_cvt(s));
        if (++s == kStages) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===================================================== epilogue: TMEM -> threshold -> packed bits + sums
    const int q = warp & 3;  // a warp may only touch TMEM lanes 32*(warp % 4) .. +31
    const int half = (warp - 6) >> 2;  // which 128 of the tile's 256 columns
    const int row_in_tile = q * 32 + lane;
    TileIter<CTAS> it(a, rank);
    uint32_t n_tile = 0;
    int cur_b = -1, cur_rb = -1;
    unsigned acc_cnt = 0;
    float acc_score = 0.0f;
    auto flush = [&]() {
      if (cur_b >= 0) {
        const int row = cur_rb * kBM + row_in_tile;
        D2B_BOUND(acc_cnt || acc_score != 0.0f ? row : 0, a.n);  // only live rows accumulate
        D2B_BOUND(cur_b, a.B);
        if (acc_cnt) atomicAdd(a.sum_masks + (size_t)cur_b * a.n + row, (float)acc_cnt);  // integer valued < 2^24: exact
        if (acc_score != 0.0f) atomicAdd(a.score_sums + (size_t)cur_b * a.n + row, acc_score);
      }
      acc_cnt = 0;
      acc_score = 0.0f;
    };
    while (it.next()) {
      const uint32_t as = n_tile & 1u, aph = (n_tile >> 1) & 1u;
      ++n_tile;
      if (it.b != cur_b || it.rb != cur_rb) {
        flush();
        cur_b = it.b;
        cur_rb = it.rb;
      }
      const int cnt = a.counts ? min(a.counts[it.b], a.n) : a.n;
      const int row = it.rb * kBM + row_in_tile;
      const bool live = row < cnt;
      mbar_wait(tmem_full(as), aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * kBN;
      const long long p0 = (long long)it.pt * kBN;
      u64 word = 0;
      D2B_BOUND(it.b, a.B);
      D2B_BOUND(live ? row : 0, a.n);
      u64* dstw = a.packed + ((size_t)it.b * a.n + (live ? row : 0)) * a.Wd;
      float* lg = a.logits ? a.logits + ((size_t)it.b * a.n + (live ? row : 0)) * a.hw : nullptr;
#pragma unroll 1  // a rolled loop: the unrolled form is 160 KB of straight-line code and lives in instruction-cache misses
      for (int c = half * (kBN / 32); c < (half + 1) * (kBN / 32); ++c) {
        uint32_t r[16];
        __syncwarp();  // .sync.aligned: the whole warp issues the load together
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr + c * 16)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        uint32_t bits = 0, band = 0;
        const long long pc = p0 + c * 16;
        if (live) {
          if (lg) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (pc + j < a.hw) lg[pc + j] = __uint_as_float(r[j]);
          }
          // sigmoid(x) > thr is decided on x outside the guard band around logit(thr); branch-free so that the 16
          // elements' MUFU chains overlap.  The (rare) elements inside the band take the exact sigmoid below.
          float s0 = 0.0f, s1 = 0.0f;
          const long long left = a.hw - pc;  // pixels of this chunk inside the map
          if (left >= 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float x = __uint_as_float(r[j]);
              const float sg = fast_sigmoid(x);
              if (x > a.hi) {
                bits |= 1u << j;
                if (j & 1) s1 = s1 + sg;
                else s0 = s0 + sg;
              } else if (x >= a.lo) {
                band |= 1u << j;
              }
            }
          } else {  // the last tile of the map: TMA zero-filled the rows past hw, they must not set bits
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float x = __uint_as_float(r[j]);
              if (j < left) {
                if (x > a.hi) {
                  bits |= 1u << j;
                  s0 = s0 + fast_sigmoid(x);
                } else if (x >= a.lo) {
                  band |= 1u << j;
                }
              }
            }
          }
          acc_score = acc_score + (s0 + s1);
          if (band) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if ((band >> j) & 1u) {
                const float x = __uint_as_float(r[j]);
                if (exact_sigmoid_above(x, a.thr)) {
                  bits |= 1u << j;
                  acc_score = acc_score + fast_sigmoid(x);
                }
              }
          }
        }
        acc_cnt += __popc(bits);
        word |= (u64)bits << (16 * (c & 3));
        if ((c & 3) == 3) {
          const int wi = it.pt * (kBN / 64) + (c >> 2);
          if (live && wi < a.Wd) dstw[wi] = word;
          word = 0;
        }
      }
      // the accumulator has been consumed: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      if constexpr (CTAS == 1) mbar_arrive(tmem_empty(as));
      else mbar_arrive_leader(tmem_empty(as));
    }
    flush();
  }

  // ------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync_all();  // no CTA of the pair leaves while the other can still signal it
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CTAS == 1)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
        qr != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}
// [batch, rows, E] fp32, E contiguous -> 3-D map with a (bk x box_rows x 1) box, swizzle = row bytes, zero OOB fill
int make_map(CUtensorMap* m, const void* ptr, int E, long long rows, int batch, int box_rows, int bk) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled is not available from the driver");
    return D2B_ECUDA;
  }
  const cuuint64_t dims[3] = {(cuuint64_t)E, (cuuint64_t)rows, (cuuint64_t)batch};
  const cuuint64_t strides[2] = {(cuuint64_t)E * 4, (cuuint64_t)rows * E * 4};
  const cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, bk == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (E=%d rows=%lld batch=%d)", (int)r, E, rows, batch);
    return D2B_ECUDA;
  }
  return D2B_OK;
}

// Variants measured at 16 x 500 x 200x336, E=256 (the two slower ones were removed):
//   pair, BK=32 (128-byte swizzle, 3 stages of 64 KB)  1.19 ms   <- used when n > 128
//   one CTA, BK=16 (64-byte swizzle, 4 stages of 48 KB) 1.23 ms   <- used when n <= 128 (a pair would idle one SM)
//   one CTA, BK=32 (2 stages of 96 KB)                  1.29 ms
//   pair, BK=16 (6 stages of 32 KB)                     1.74 ms
template <int BK, int CTAS>
int launch_dyn(const CUtensorMap& tm_ahi, const CUtensorMap& tm_alo, const CUtensorMap& tm_feat, const DynArgs& a, int sms,
               int dev, cudaStream_t st) {
  using C = Cfg<BK, CTAS>;
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    D2B_CUDA(cudaFuncSetAttribute(solo_dynconv_kernel<BK, CTAS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)C::kSmemBytes));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const long long units = (a.RB + CTAS - 1) / CTAS;
  const long long tiles = (long long)a.B * units * a.PT;
  long long grid = tiles * CTAS < sms ? tiles * CTAS : sms;
  grid -= grid % CTAS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CTAS == 2 ? 1 : 0;
  D2B_CUDA(cudaLaunchKernelEx(&cfg, solo_dynconv_kernel<BK, CTAS>, tm_ahi, tm_alo, tm_feat, a));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

int dyn_check(const d2b_solo_dynamic_masks_params* p) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->batch >= 0 && p->n >= 0 && p->hw >= 0 && p->channels >= 0, "solo_dynamic_masks: negative sizes");
  D2B_REQUIRE(p->n <= 65535 && p->batch <= 65535, "solo_dynamic_masks: n / batch too large");
  D2B_REQUIRE(p->hw < (1ll << 24), "solo_dynamic_masks: hw=%lld >= 2^24 (mask sums must stay exact in fp32)", (long long)p->hw);
  D2B_REQUIRE(p->channels % 4 == 0 && p->channels >= 4 && p->channels <= 4096,
              "solo_dynamic_masks: channels=%d must be a multiple of 4 in [4, 4096] (16-byte TMA rows)", p->channels);
  return D2B_OK;
}
}  // namespace

size_t solo_dynamic_masks_ws(int batch, int n, int channels) {
  return 2 * ws_slice((size_t)batch * (n > 0 ? n : 1) * channels * 4);
}
}  // namespace d2b

using namespace d2b;

extern "C" size_t d2b_solo_dynamic_masks_workspace_bytes(const d2b_solo_dynamic_masks_params* p) {
  if (dyn_check(p) != D2B_OK) return 0;
  return solo_dynamic_masks_ws(p->batch, p->n, p->channels);
}

extern "C" int d2b_solo_dynamic_masks(const d2b_solo_dynamic_masks_params* p, void* workspace, size_t workspace_bytes,
                                      d2b_stream_t stream) {
  int rc = dyn_check(p);
  if (rc != D2B_OK) return rc;
  if (p->batch == 0 || p->n == 0) return D2B_OK;
  D2B_REQUIRE(p->packed_masks && p->sum_masks && p->score_sums, "solo_dynamic_masks: NULL output");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t rows = (size_t)p->batch * p->n;
  D2B_CUDA(cudaMemsetAsync(p->sum_masks, 0, sizeof(float) * rows, st));
  D2B_CUDA(cudaMemsetAsync(p->score_sums, 0, sizeof(float) * rows, st));
  if (p->hw == 0) return D2B_OK;
  D2B_REQUIRE(p->mask_features && p->mask_kernels, "solo_dynamic_masks: NULL input");
  D2B_REQUIRE((reinterpret_cast<uintptr_t>(p->mask_features) & 15) == 0 && (reinterpret_cast<uintptr_t>(p->mask_kernels) & 15) == 0,
              "solo_dynamic_masks: inputs must be 16-byte aligned");
  const size_t need = solo_dynamic_masks_ws(p->batch, p->n, p->channels);
  if (workspace == nullptr || workspace_bytes < need) {
    set_last_error("solo_dynamic_masks needs %zu workspace bytes", need);
    return D2B_EWORKSPACE;
  }
  const int E = p->channels;
  Workspace ws(workspace);
  float* a_hi = ws.take<float>(rows * E);
  float* a_lo = ws.take<float>(rows * E);

  DynArgs a;
  a.counts = p->counts; a.B = p->batch; a.n = p->n; a.E = E; a.hw = p->hw;
  a.RB = (p->n + kBM - 1) / kBM;
  a.PT = (int)((p->hw + kBN - 1) / kBN);
  // a cta_group::2 pair works on two row blocks at once; with a single row block (n <= 128) it would idle one SM
  const int ctas = p->n > kBM ? 2 : 1;
  const int bk = ctas == 2 ? 32 : 16;
  a.KB = (E + bk - 1) / bk;
  a.Wd = (int)((p->hw + 63) / 64);
  a.thr = p->mask_threshold;
  const double t = (double)p->mask_threshold;  // same guard band as solo_encode_kernel
  if (t > 1e-3 && t < 1.0 - 1e-3) {
    const double x0 = log(t / (1.0 - t));
    const double d = 1e-3 * (fabs(x0) > 1.0 ? fabs(x0) : 1.0);
    a.lo = (float)(x0 - d);
    a.hi = (float)(x0 + d);
  } else {
    a.lo = -INFINITY;
    a.hi = INFINITY;
  }
  a.packed = reinterpret_cast<u64*>(p->packed_masks);
  a.sum_masks = p->sum_masks;
  a.score_sums = p->score_sums;
  a.logits = p->mask_logits;

  // rows past the valid prefix / row blocks without work keep defined (empty) masks
  if (p->counts) D2B_CUDA(cudaMemsetAsync(p->packed_masks, 0, sizeof(u64) * rows * a.Wd, st));

  CUtensorMap tm_ahi, tm_alo, tm_feat;
  if ((rc = make_map(&tm_ahi, a_hi, E, p->n, p->batch, kBM, bk)) != D2B_OK) return rc;
  if ((rc = make_map(&tm_alo, a_lo, E, p->n, p->batch, kBM, bk)) != D2B_OK) return rc;
  if ((rc = make_map(&tm_feat, p->mask_features, E, p->hw, p->batch, kBN / ctas, bk)) != D2B_OK) return rc;

  const long long total4 = (long long)rows * E / 4;
  dyn_split_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(p->mask_kernels),
                                                                     reinterpret_cast<float4*>(a_hi),
                                                                     reinterpret_cast<float4*>(a_lo), total4);
  D2B_LAUNCH_CHECK();

  static int sm_count[64] = {0};
  int dev = 0;
  D2B_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && sm_count[dev] == 0) {
    int v = 0;
    D2B_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    sm_count[dev] = v > 0 ? v : 148;
  }
  const int sms = (dev >= 0 && dev < 64) ? sm_count[dev] : 148;
  if (ctas == 2) return launch_dyn<32, 2>(tm_ahi, tm_alo, tm_feat, a, sms, dev, st);
  return launch_dyn<16, 1>(tm_ahi, tm_alo, tm_feat, a, sms, dev, st);
}
