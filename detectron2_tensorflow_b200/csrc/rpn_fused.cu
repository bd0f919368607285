// rpn_fused.cu -- the front of the RPN proposal stage as ONE thread-block-cluster launch:
//   tf.nn.top_k per (image, level) row (rpn_outputs.py:67-70)  ->  order (score desc, index asc)
//   -> gather + Box2BoxTransform.apply_deltas (:403-426, only the winners) -> clip_to_window (:77-80)
//   -> prune_small_boxes (:83-87), ordered.
// One cluster of kSelCluster CTAs owns one row (a row of P2 logits is 806 KB: each CTA streams 1/8 of it).
//   select   radix-select over the order-preserving 32-bit value keys, 8 bits per pass: every CTA histograms its
//            chunk into warp-private shared-memory bins, the 8 per-CTA histograms are summed by every CTA through
//            distributed shared memory (2 KB per peer), and a block scan finds the digit that holds the k-th
//            largest key.  The cluster barrier replaces the kernel boundary of a multi-launch radix select; the
//            row is read from HBM once and from L2 afterwards.  A pass whose boundary bucket is taken whole ends
//            the selection early.
//   ties     if the k-th value is tied, the lower indices win (TF TopKV2): chunks are contiguous index ranges in
//            rank order, so per-CTA tie counts give each CTA a quota, and only the one CTA with a partial quota
//            walks its chunk in index order.
//   collect  winners go to a CTA-local list (shared-memory atomics), one remote atomic per CTA reserves a range
//            of the leader's list, and the local list is copied there through DSMEM.
//   leader   bitonic sort of the <= 4096 composite keys (value key << 32 | ~index: unique, so a plain descending
//            sort realises the tie rule), then decode / clip / ordered prune into the NMS input buffers.
// Replaces 11 launches (memset, init, 6 histogram passes, collect, sort, decode) of the generic chain in
// pipelines.cu / topk.cu, which remains for k > kRpnFusedMaxK.
#include <cooperative_groups.h>

#include "nms.cuh"
#include "rpn.cuh"

namespace cg = cooperative_groups;

namespace d2b {
namespace {

constexpr int kSelThreads = 512;
constexpr int kSelCluster = 8;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kHistCopies = 8;   // two warps share one copy of the 256 bins
constexpr int kHistStride = 260;  // 256 bins + [256] = "raw list overflowed" flag; two buffers (pass parity)
constexpr int kCandCap = 256;     // boundary buckets up to this size are resolved by ranking their elements

struct SelCtl {
  unsigned digit, need, bucket, overflow;  // result of one pass (identical in every CTA of the cluster)
  unsigned raw_cnt;                // fast path: entries of the raw list (top byte >= boundary byte of pass 0)
  unsigned local_cnt;              // entries of this CTA's final list
  unsigned my_cand;                // fast path: candidates of this CTA written so far
  unsigned tie_cnt;                // elements equal to the k-th value in this CTA's chunk
  unsigned cand_cnt[kSelCluster];  // candidates (boundary-bucket elements) per CTA
  unsigned cnt[kSelCluster];       // winners per CTA (written by the owners through DSMEM)
  unsigned sel_cnt[kSelCluster];   // candidates selected per CTA (computed redundantly by every CTA)
  unsigned ties[kSelCluster];      // tie counts of every CTA (written remotely)
  unsigned wcnt[kSelThreads / 32];  // fast path: entries of each warp's raw sublist
};

// Radix digits: 11 + 8 + 8 + 5 bits of the 32-bit value key.  Pass 0 takes 11 bits (sign + exponent + 2 mantissa
// bits = a quarter binade per bin: 8 bits would lump two binades into one bucket) with a two-level exchange: the
// peers' 256 coarse sums are scanned first, then the 8 fine bins of the coarse boundary bin.
__constant__ int c_sel_shift[4] = {21, 13, 5, 0};
__constant__ int c_sel_bits[4] = {11, 8, 8, 5};
constexpr int kFineBins = 2048;
// Dynamic shared memory: [hist 2*260][fine 2048][whist kHistCopies*256][scan 32+64][ctl 256 B][cand 256 u64][raw P u64][tmp P u64]
constexpr size_t kSelOffFine = 2 * kHistStride * 4;
constexpr size_t kSelOffWhist = kSelOffFine + kFineBins * 4;
constexpr size_t kSelOffScan = kSelOffWhist + kHistCopies * 256 * 4;
constexpr size_t kSelOffCtl = kSelOffScan + (32 + 64) * 4;
constexpr size_t kSelOffCand = kSelOffCtl + 256;
constexpr size_t kSelOffRaw = kSelOffCand + kCandCap * 8;
static_assert(kSelOffCtl % 8 == 0 && kSelOffCand % 8 == 0 && kSelOffRaw % 16 == 0, "shared-memory layout alignment");

__device__ __forceinline__ unsigned key_of(float v) { return float_to_key(v); }

__device__ __forceinline__ float4 ldg_nc_v4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// Calls f(value, index, valid) for the elements of [beg, end) of row x with warp-uniform control flow.  16-byte loads
// when aligned; the kV loads of a trip are issued together (volatile loads + a compiler barrier: without it the
// compiler sinks each load next to its conditional use and the trip pays kV dependent L2 round trips).
template <typename F>
__device__ __forceinline__ void scan_chunk(const float* __restrict__ x, long long beg, long long end, F f) {
  if (end <= beg) return;
  const bool vec = ((reinterpret_cast<uintptr_t>(x + beg) & 15) == 0);
  if (vec) {
    const long long nvec = (end - beg) >> 2;
    const float4* xv = reinterpret_cast<const float4*>(x + beg);
    constexpr int kV = 4;
    for (long long v0 = 0; v0 < nvec; v0 += (long long)kV * kSelThreads) {  // block-uniform trip count
      float4 q[kV];
#pragma unroll
      for (int u = 0; u < kV; ++u) {
        const long long vi = v0 + (long long)u * kSelThreads + threadIdx.x;
        q[u] = ldg_nc_v4(xv + (vi < nvec ? vi : 0));  // clamped: always a valid address
      }
      asm volatile("" ::: "memory");
#pragma unroll
      for (int u = 0; u < kV; ++u) {
        const long long vi = v0 + (long long)u * kSelThreads + threadIdx.x;
        const bool ok = vi < nvec;
        const long long i = beg + 4 * vi;
        f(q[u].x, i, ok); f(q[u].y, i + 1, ok); f(q[u].z, i + 2, ok); f(q[u].w, i + 3, ok);
      }
    }
    const long long t0 = beg + 4 * nvec;
    for (long long i0 = t0; i0 < end; i0 += kSelThreads) {  // < 4 leftover elements: one uniform trip
      const long long i = i0 + threadIdx.x;
      const bool ok = i < end;
      f(ok ? __ldg(x + i) : 0.0f, i, ok);
    }
  } else {
    constexpr int kS = 8;
    for (long long i0 = beg; i0 < end; i0 += (long long)kS * kSelThreads) {
      float q[kS];
#pragma unroll
      for (int u = 0; u < kS; ++u) {
        const long long i = i0 + (long long)u * kSelThreads + threadIdx.x;
        q[u] = __ldg(x + (i < end ? i : beg));
      }
      asm volatile("" ::: "memory");
#pragma unroll
      for (int u = 0; u < kS; ++u) {
        const long long i = i0 + (long long)u * kSelThreads + threadIdx.x;
        f(q[u], i, i < end);
      }
    }
  }
}

// Exclusive scan of `v` over the block in thread order; `total` gets the block sum.  s_w: kSelWarps ints.
__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned* s_w, unsigned& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  unsigned before = 0;
  total = 0;
#pragma unroll
  for (int w = 0; w < kSelWarps; ++w) {
    const unsigned c = s_w[w];
    if (w < warp) before += c;
    total += c;
  }
  __syncthreads();
  return before + inc - v;
}

#ifndef D2B_SEL_MINB
#define D2B_SEL_MINB 2  // A/B: 1 (104 registers) 0.197 ms at 16 images, 2 (64) 0.160, 4 (32, spills) 0.150 alone but the pipelined step 0.512 -> 0.575 ms
#endif
__global__ void __launch_bounds__(kSelThreads, D2B_SEL_MINB) rpn_select_kernel(RpnArgs a, float4* seg_boxes, float* seg_scores,
                                                                  int32_t* seg_count, u64* nms_in_total) {
  grid_dep_sync();
  extern __shared__ __align__(16) unsigned char s_raw_bytes[];
  unsigned* hist = reinterpret_cast<unsigned*>(s_raw_bytes);                         // [2][kHistStride], peers read it
  unsigned* fine = reinterpret_cast<unsigned*>(s_raw_bytes + kSelOffFine);           // [2048] pass 0 (peers read 8 bins)
  unsigned* whist = reinterpret_cast<unsigned*>(s_raw_bytes + kSelOffWhist);         // [kHistCopies][256] / 2nd fine copy
  unsigned* s_scan = reinterpret_cast<unsigned*>(s_raw_bytes + kSelOffScan);         // [32]
  unsigned* s_f = s_scan + 32;                                                       // [8 peers][8 fine bins]
  SelCtl* ctl = reinterpret_cast<SelCtl*>(s_raw_bytes + kSelOffCtl);
  u64* s_cand = reinterpret_cast<u64*>(s_raw_bytes + kSelOffCand);                   // [kCandCap] all CTAs' candidates
  u64* s_raw = reinterpret_cast<u64*>(s_raw_bytes + kSelOffRaw);                     // [P] raw list, later all sorted runs
  u64* s_tmp = s_raw + a.P;                                                          // [P] this CTA's final list / run

  cg::cluster_group cluster = cg::this_cluster();
  const unsigned rank = cluster.block_rank();
  const int cid = blockIdx.x / kSelCluster;  // level-major: the long P2 rows are scheduled first
  const int l = cid / a.N, n = cid - l * a.N;
  const int row = n * a.L + l;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long len = a.hwa[l];
  const float* x = a.logits[l] + (size_t)n * len;
  const unsigned kr = (unsigned)(len < (long long)a.k ? len : (long long)a.k);
  const unsigned P = (unsigned)a.P;
  const bool prof = (blockIdx.x == 0 && tid == 0);
  D2B_PROF(prof, 0);

  if (tid < (int)(sizeof(SelCtl) / 4)) reinterpret_cast<unsigned*>(ctl)[tid] = 0u;
  if (kr == 0) {  // uniform over the cluster: nobody touches a peer
    if (rank == 0 && tid == 0) seg_count[row] = 0;
    return;
  }
  __syncthreads();
  // contiguous chunk of the row, multiple of 4 elements so that 16-byte loads stay aligned
  long long per = (len + kSelCluster - 1) / kSelCluster;
  per = (per + 3) & ~3ll;
  const long long beg = per * rank < len ? per * rank : len;
  const long long end = beg + per < len ? beg + per : len;

  // One radix pass over the cluster: this CTA's warp-private counts -> hist[pass & 1] -> cluster barrier -> every
  // CTA sums the 8 histograms through DSMEM (thread t owns bin 255 - t) and scans from the top bin down.
  // hist is double-buffered by pass parity: a CTA overwrites buffer b two barriers after its peers read it.
  unsigned prefix = 0;  // resolved high bits of the k-th largest key
  unsigned k_rem = kr;  // winners still to be found inside the prefix bucket
  unsigned bucket = 0, any_overflow = 0;
  auto exchange = [&](int pass, unsigned my_overflow) {
    unsigned* hb = hist + (pass & 1) * kHistStride;
    const int nbits = c_sel_bits[pass];
    if (pass == 0) {
      // fine (2048 bins) = copy of the even warps + copy of the odd warps; coarse bin = 8 fine bins
      for (int i = tid; i < kFineBins; i += kSelThreads) fine[i] += whist[i];
      __syncthreads();
      if (tid < 256) {
        unsigned v = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) v += fine[tid * 8 + j];
        hb[tid] = v;
      }
    } else if (tid < 256) {
      unsigned v = 0;
#pragma unroll
      for (int c = 0; c < kHistCopies; ++c) v += whist[c * 256 + tid];
      hb[tid] = v;
    }
    if (tid == 256) hb[256] = my_overflow;
    cluster.sync();  // the 8 per-CTA histograms are visible cluster-wide
    D2B_PROF(prof, 64 + pass * 8 + 3);
    unsigned tot = 0, ovf = 0;
    if (tid < 256) {
#pragma unroll
      for (unsigned r = 0; r < kSelCluster; ++r) tot += cluster.map_shared_rank(hb, r)[255 - tid];
    } else if (tid < 256 + kSelCluster) {
      ovf = cluster.map_shared_rank(hb, tid - 256)[256];
    }
    if (ovf) ctl->overflow = 1u;
    unsigned total;
    const unsigned excl = block_excl_scan(tot, s_scan, total);
    if (tid < 256 && excl < k_rem && k_rem <= excl + tot) {
      ctl->digit = 255u - (unsigned)tid;
      ctl->need = k_rem - excl;
      ctl->bucket = tot;
    }
    __syncthreads();
    unsigned digit = ctl->digit;
    if (pass == 0) {
      // second level: the 8 fine bins of the coarse boundary bin, per peer
      if (tid < 64) s_f[tid] = cluster.map_shared_rank(fine, tid >> 3)[digit * 8 + (tid & 7)];
      __syncthreads();
      if (tid == 0) {
        unsigned need = ctl->need, above = 0;
        for (int j = 7; j >= 0; --j) {
          unsigned t = 0;
          for (int r = 0; r < kSelCluster; ++r) t += s_f[r * 8 + j];
          if (above + t >= need) {
            ctl->digit = digit * 8 + (unsigned)j;
            ctl->need = need - above;
            ctl->bucket = t;
            for (int r = 0; r < kSelCluster; ++r) ctl->cand_cnt[r] = s_f[r * 8 + j];
            break;
          }
          above += t;
        }
      }
      __syncthreads();
      digit = ctl->digit;
    } else if (tid < kSelCluster) {
      ctl->cand_cnt[tid] = cluster.map_shared_rank(hb, tid)[digit];  // per-CTA boundary counts
    }
    prefix = (prefix << nbits) | digit;
    k_rem = ctl->need;
    bucket = ctl->bucket;
    any_overflow = ctl->overflow;
    __syncthreads();  // ctl fields are rewritten by the next pass
    D2B_PROF(prof, 1 + pass);
  };
  auto zero_whist = [&]() {
    for (int i = tid; i < kHistCopies * 256; i += kSelThreads) whist[i] = 0;
    __syncthreads();
  };
  auto append_to = [&](u64* list, unsigned* counter, u64 c, bool take) -> bool {  // warp-uniform call; false = overflow
    const unsigned m = __ballot_sync(0xffffffffu, take);
    bool fits = true;
    if (m) {
      unsigned base = 0;
      if (lane == 0) base = atomicAdd(counter, (unsigned)__popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (take) {
        const unsigned slot = base + __popc(m & ((1u << lane) - 1u));
        if (slot < P) list[slot] = c; else fits = false;
      }
    }
    return fits;
  };
  unsigned* my = whist + (warp >> 1) * 256;

  bool all = (kr == (unsigned)len);  // the whole row is taken (e.g. P6: 819 anchors < k)
  if (all) cluster.sync();  // no radix pass follows: peers must be running (and initialised) before the first DSMEM store
  bool have_lists = false;           // s_tmp / ctl->cnt[] hold the final per-CTA lists
  bool ties = false;                 // k-th value tied: only `k_rem` of the elements equal to `prefix` are taken
  bool resolved = all;
  unsigned cut = 0;                  // generic collect: take key > cut (plus the tie quota)
  int next_pass = 0;

  if (!all) {
    // ---------------------------------------------------------------- pass 0: top byte (the one HBM read of the row)
    for (int i = tid; i < kFineBins; i += kSelThreads) { fine[i] = 0; whist[i] = 0; }
    __syncthreads();
    unsigned* f0 = (warp & 1) ? whist : fine;
    scan_chunk(x, beg, end, [&](float v, long long, bool ok) {
      D2B_BOUND(key_of(v) >> 21, kFineBins);
      if (ok) atomicAdd(f0 + (key_of(v) >> 21), 1u);
    });
    __syncthreads();
    D2B_PROF(prof, 64 + 1);
    exchange(0, 0u);
    next_pass = 1;
    if (bucket == k_rem) {  // boundary bucket taken whole: every key >= prefix << 21 wins
      const unsigned thr = prefix << 21;
      if (thr == 0u) all = true; else cut = thr - 1u;
      resolved = true;
    }
  }
  if (!resolved) {
    // ---------------------------------------------------------------- pass 1 (L2 read): next 8 bits of the boundary
    // bucket, and every element whose 11-bit digit is >= the boundary digit goes to the raw list (composite keys).
    const unsigned d0 = prefix;
    zero_whist();
    // raw list = 16 per-warp sublists of P/16 entries, filled with a warp-uniform register count (a single shared
    // counter serialises ~400 same-address shared-memory atomics per CTA: measured 11 us for this scan)
    const unsigned cap_w = P / kSelWarps;
    u64* wlist = s_raw + (size_t)warp * cap_w;
    unsigned wcnt = 0;
    // `top >= d0` is decided on the raw float (v >= smallest value of bin d0; extra NaNs taken when d0 <= 3 are dropped
    // by the classification below), one compare per element; the order-preserving key is only computed for the ~2 % that are taken.
    const float thr_f = key_to_float(d0 << 21);
    const bool take_all = !(thr_f == thr_f);  // d0 <= 3: the bin of NaN (key 0) / -inf; its lower edge is no float
    auto take_one = [&](float v, long long i, unsigned& slot) {
      const unsigned key = key_of(v);
      if (slot < cap_w) wlist[slot] = ((u64)key << 32) | (u64)(0xffffffffu - (unsigned)i);
      ++slot;
      if ((key >> 21) == d0) atomicAdd(my + ((key >> 13) & 255u), 1u);
    };
    if (end > beg && (reinterpret_cast<uintptr_t>(x + beg) & 15) == 0) {
      const long long nvec = (end - beg) >> 2;
      const float4* xv = reinterpret_cast<const float4*>(x + beg);
      constexpr int kV = 4;
      for (long long v0 = 0; v0 < nvec; v0 += (long long)kV * kSelThreads) {  // block-uniform trip count
        float4 q[kV];
#pragma unroll
        for (int u = 0; u < kV; ++u) {
          const long long vi = v0 + (long long)u * kSelThreads + tid;
          q[u] = ldg_nc_v4(xv + (vi < nvec ? vi : 0));
        }
        asm volatile("" ::: "memory");
        unsigned mask = 0;  // bit 4u+c: component c of vector u is taken
#pragma unroll
        for (int u = 0; u < kV; ++u) {
          const long long vi = v0 + (long long)u * kSelThreads + tid;
          if (vi < nvec) {
            mask |= ((take_all || q[u].x >= thr_f) ? 1u : 0u) << (4 * u);
            mask |= ((take_all || q[u].y >= thr_f) ? 2u : 0u) << (4 * u);
            mask |= ((take_all || q[u].z >= thr_f) ? 4u : 0u) << (4 * u);
            mask |= ((take_all || q[u].w >= thr_f) ? 8u : 0u) << (4 * u);
          }
        }
        // slots: warp-exclusive scan of the per-thread counts, once per trip
        const unsigned c = __popc(mask);
        unsigned inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += t;
        }
        unsigned slot = wcnt + inc - c;
        wcnt += __shfl_sync(0xffffffffu, inc, 31);
        if (mask) {
#pragma unroll
          for (int u = 0; u < kV; ++u) {
            const long long i = beg + 4 * (v0 + (long long)u * kSelThreads + tid);
            if (mask & (1u << (4 * u))) take_one(q[u].x, i, slot);
            if (mask & (2u << (4 * u))) take_one(q[u].y, i + 1, slot);
            if (mask & (4u << (4 * u))) take_one(q[u].z, i + 2, slot);
            if (mask & (8u << (4 * u))) take_one(q[u].w, i + 3, slot);
          }
        }
      }
      const long long t0 = beg + 4 * nvec;  // < 4 leftover elements
      {
        const long long i = t0 + tid;
        const bool ok = i < end;
        const float v = ok ? __ldg(x + i) : 0.0f;
        const bool take = ok && (take_all || v >= thr_f);
        const unsigned m = __ballot_sync(0xffffffffu, take);
        unsigned slot = wcnt + __popc(m & ((1u << lane) - 1u));
        wcnt += __popc(m);
        if (take) take_one(v, i, slot);
      }
    } else {
      scan_chunk(x, beg, end, [&](float v, long long i, bool ok) {
        const bool take = ok && (take_all || v >= thr_f);
        const unsigned m = __ballot_sync(0xffffffffu, take);
        if (m) {
          unsigned slot = wcnt + __popc(m & ((1u << lane) - 1u));
          wcnt += __popc(m);
          if (take) take_one(v, i, slot);
        }
      });
    }
    if (lane == 0) ctl->wcnt[warp] = wcnt;
    const unsigned my_overflow = __syncthreads_or(wcnt > cap_w ? 1 : 0) ? 1u : 0u;
    D2B_PROF(prof, 64 + 8 + 1);
    exchange(1, my_overflow);
    next_pass = 2;
    const bool whole = (bucket == k_rem);
    if (!any_overflow && (whole || bucket <= (unsigned)kCandCap)) {
      // ---- fast finish: winners = raw entries above the 19-bit boundary; the boundary bucket's elements
      // (candidates) are sent to every CTA and ranked there (composites are unique: ties fall to the lower index)
      unsigned cbase = 0;
      for (unsigned r = 0; r < rank; ++r) cbase += ctl->cand_cnt[r];
      unsigned wmax = 0;
#pragma unroll
      for (int q = 0; q < kSelWarps; ++q) wmax = max(wmax, ctl->wcnt[q]);
      const unsigned my_n = wcnt;
      for (unsigned i0 = 0; i0 < wmax; i0 += 32) {  // block-uniform trip count; warp q walks its own sublist
        const unsigned i = i0 + lane;
        const bool live = i < my_n;
        const u64 c = live ? wlist[i] : 0ull;
        const unsigned t19 = (unsigned)(c >> 45);
        const bool win = live && (t19 > prefix || (whole && t19 == prefix));
        const bool cand = live && !whole && t19 == prefix;
        append_to(s_tmp, &ctl->local_cnt, c, win);
        if (cand) {
          const unsigned j = cbase + atomicAdd(&ctl->my_cand, 1u);
          D2B_BOUND(j, kCandCap);
#pragma unroll
          for (unsigned r = 0; r < kSelCluster; ++r) cluster.map_shared_rank(s_cand, r)[j] = c;
        }
      }
      __syncthreads();
      if (tid < kSelCluster) cluster.map_shared_rank(ctl, tid)->cnt[rank] = ctl->local_cnt;
      cluster.sync();  // every CTA holds all candidates and every CTA's winner count
      if (!whole) {
        const unsigned T = bucket;
        if (tid < (int)T) {
          const u64 mine = s_cand[tid];
          unsigned r = 0;
          for (unsigned j = 0; j < T; ++j) r += (s_cand[j] > mine) ? 1u : 0u;
          if (r < k_rem) {  // selected: one of the k_rem largest candidates
            unsigned q = 0, b = 0;
            while (q + 1 < kSelCluster && tid >= (int)(b + ctl->cand_cnt[q])) { b += ctl->cand_cnt[q]; ++q; }
            atomicAdd(&ctl->sel_cnt[q], 1u);
            D2B_BOUND(ctl->local_cnt, P);
            if (q == rank) s_tmp[atomicAdd(&ctl->local_cnt, 1u)] = mine;
          }
        }
        __syncthreads();
        if (tid < kSelCluster) ctl->cnt[tid] += ctl->sel_cnt[tid];
        __syncthreads();
      }
      have_lists = true;
    } else if (whole) {
      const unsigned thr = prefix << 13;
      cut = thr - 1u;
      if (thr == 0u) all = true;
      resolved = true;
    }
  }
  if (!have_lists) {
    // ------------------------------------------------------------------ generic path (huge boundary buckets, i.e.
    // massively tied values, or a raw list that overflowed): remaining radix passes over the row, then a collect
    // scan; exact ties are split by index order through per-CTA quotas.
    if (!resolved) {
      for (int pass = next_pass; pass < 4; ++pass) {
        const int shift = c_sel_shift[pass];
        const int hs = shift + c_sel_bits[pass];
        const unsigned dmask = (1u << c_sel_bits[pass]) - 1u;
        zero_whist();
        scan_chunk(x, beg, end, [&](float v, long long, bool ok) {
          const unsigned key = key_of(v);
          if (ok && (key >> hs) == prefix) atomicAdd(my + ((key >> shift) & dmask), 1u);
        });
        __syncthreads();
        exchange(pass, 0u);
        if (bucket == k_rem) {  // boundary bucket taken whole: every key >= prefix << shift wins
          const unsigned thr = prefix << shift;
          if (thr == 0u) all = true; else cut = thr - 1u;
          resolved = true;
          break;
        }
      }
      if (!resolved) {  // all 32 value bits fixed and the bucket holds more than k_rem equal keys
        ties = true;
        cut = prefix;
      }
    }
    if (tid == 0) ctl->local_cnt = 0;
    __syncthreads();
    unsigned my_ties = 0;
    scan_chunk(x, beg, end, [&](float v, long long i, bool ok) {
      const unsigned key = key_of(v);
      const bool take = ok && (all || key > cut);
      if (ties) my_ties += (ok && key == cut) ? 1u : 0u;
      append_to(s_tmp, &ctl->local_cnt, ((u64)key << 32) | (u64)(0xffffffffu - (unsigned)i), take);
    });
    if (ties) {  // block-uniform (identical in the whole cluster)
      // per-CTA tie counts -> every CTA's table; chunks are contiguous index ranges in rank order
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) my_ties += __shfl_xor_sync(0xffffffffu, my_ties, o);
      if (lane == 0 && my_ties) atomicAdd(&ctl->tie_cnt, my_ties);
      __syncthreads();
      if (tid < kSelCluster) cluster.map_shared_rank(ctl, tid)->ties[rank] = ctl->tie_cnt;
      cluster.sync();
      unsigned before = 0;
      for (unsigned r = 0; r < rank; ++r) before += ctl->ties[r];
      const unsigned mine = ctl->ties[rank];
      const unsigned quota = before >= k_rem ? 0u : (k_rem - before < mine ? k_rem - before : mine);
      if (quota == mine) {  // all of this chunk's ties (possibly none)
        if (mine)
          scan_chunk(x, beg, end, [&](float v, long long i, bool ok) {
            const unsigned key = key_of(v);
            append_to(s_tmp, &ctl->local_cnt, ((u64)key << 32) | (u64)(0xffffffffu - (unsigned)i), ok && key == cut);
          });
      } else if (quota > 0) {
        // the one CTA with a partial quota: its `quota` lowest-index ties, found by walking the chunk in index
        // order (thread t owns 4 consecutive elements per trip; an ordered block scan gives every tie its ordinal)
        unsigned running = 0;
        for (long long i0 = beg; i0 < end && running < quota; i0 += 4ll * kSelThreads) {
          const long long i = i0 + 4ll * tid;
          unsigned keyv[4];
          unsigned cnt = 0;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const bool ok = i + c < end;
            keyv[c] = ok ? key_of(__ldg(x + i + c)) : 0u;
            if (!ok || keyv[c] != cut) keyv[c] = cut + 1u;  // marks "not a tie" (cut + 1 != cut even on wrap-around)
            else ++cnt;
          }
          unsigned total;
          unsigned ord = running + block_excl_scan(cnt, s_scan, total);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            if (keyv[c] == cut) {
              if (ord < quota) {
                const unsigned slot = atomicAdd(&ctl->local_cnt, 1u);
                if (slot < P) s_tmp[slot] = ((u64)cut << 32) | (u64)(0xffffffffu - (unsigned)(i + c));
              }
              ++ord;
            }
          }
          running += total;
        }
      }
    }
    __syncthreads();
    if (tid < kSelCluster) cluster.map_shared_rank(ctl, tid)->cnt[rank] = ctl->local_cnt;
    cluster.sync();  // every CTA knows every CTA's winner count
  }
  D2B_PROF(prof, 5);

  // ------------------------------------------------------------------ merge: every CTA sorts its own winners, the
  // sorted runs are broadcast to all CTAs, and every CTA ranks, decodes and writes ITS winners (rank = position in
  // its own run + per other run the number of larger keys: composites are unique).
  const unsigned c_mine = min(ctl->cnt[rank], P);
  unsigned base_mine = 0;
  for (unsigned r = 0; r < rank; ++r) base_mine += ctl->cnt[r];
  const float h = (float)a.shapes[2 * n], w = (float)a.shapes[2 * n + 1];
  const size_t rbase = (size_t)n * len;
  for (unsigned i = tid; i < c_mine; i += kSelThreads) {  // the gathers of the decode below: start them now
    const unsigned idx = key_index(s_tmp[i]);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.logits[l] + rbase + idx));
    if (a.proposals[l]) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.proposals[l] + rbase + idx));
    else {
      asm volatile("prefetch.global.L2 [%0];" ::"l"(a.deltas[l] + rbase + idx));
      if (a.anchors[l].table) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.anchors[l].table + idx));
    }
  }
  if (c_mine <= (unsigned)kSelThreads) {
    // small list (the usual ~k/8 winners): rank by counting, one element per thread, then permute in place
    // (every key is unique; two keys per broadcast 16-byte shared load)
    u64 mine = 0;
    unsigned r = 0;
    if (tid < (int)c_mine) {
      mine = s_tmp[tid];
      const unsigned even = c_mine & ~1u;
      for (unsigned j = 0; j < even; j += 2) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(s_tmp + j);
        r += (v.x > mine ? 1u : 0u) + (v.y > mine ? 1u : 0u);
      }
      if (even < c_mine) r += s_tmp[even] > mine ? 1u : 0u;
    }
    __syncthreads();
    D2B_BOUND(r, tid < (int)c_mine ? c_mine : r + 1);
    if (tid < (int)c_mine) s_tmp[r] = mine;
    __syncthreads();
  } else {
    int Pe = 1;
    while (Pe < (int)c_mine) Pe <<= 1;
    for (int i = (int)c_mine + tid; i < Pe; i += kSelThreads) s_tmp[i] = 0ull;
    __syncthreads();
    for (int k = 2; k <= Pe; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int p = tid; p < Pe / 2; p += kSelThreads) {
          const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
          const bool desc = ((i & k) == 0);
          const u64 va = s_tmp[i], vb = s_tmp[i | j];
          if (desc ? (va < vb) : (va > vb)) { s_tmp[i] = vb; s_tmp[i | j] = va; }
        }
        __syncthreads();
      }
  }
  D2B_PROF(prof, 6);
  for (unsigned i = tid; i < c_mine; i += kSelThreads) {
    const u64 c = s_tmp[i];
    D2B_BOUND(base_mine + i, kr);  // the per-CTA counts add up to exactly kr winners
    if (base_mine + i < P) {
#pragma unroll
      for (unsigned r = 0; r < kSelCluster; ++r) cluster.map_shared_rank(s_raw, r)[base_mine + i] = c;
    }
  }
  cluster.sync();  // all runs are in every CTA's s_raw; nobody touches a peer's shared memory after this point
  D2B_PROF(prof, 7);
  for (unsigned i = tid; i < c_mine; i += kSelThreads) {
    const u64 key = s_tmp[i];
    unsigned pos = i;
    unsigned b = 0;
#pragma unroll
    for (unsigned r = 0; r < kSelCluster; ++r) {
      const unsigned c = ctl->cnt[r];
      if (r != rank) {
        unsigned lo = 0, hi = min(c, P - min(b, P));
        const u64* run = s_raw + b;
        while (lo < hi) {  // keys of run r greater than mine (runs are descending)
          const unsigned mid = (lo + hi) >> 1;
          if (run[mid] > key) lo = mid + 1; else hi = mid;
        }
        pos += lo;
      }
      b += c;
    }
    D2B_BOUND(pos, kr);
    if (pos < kr) {
      const unsigned idx = key_index(key);
      D2B_BOUND(idx, len);
      const float score = __ldg(a.logits[l] + rbase + idx);
      float4 box;
      if (a.proposals[l]) box = __ldg(a.proposals[l] + rbase + idx);
      else box = d2b_decode(__ldg(a.deltas[l] + rbase + idx), a.anchors[l].at(idx), a.w[0], a.w[1], a.w[2], a.w[3], a.clampv);
      box = d2b_clip(box, h, w);  // rpn_outputs.py:77-80
      seg_boxes[(size_t)row * a.k + pos] = box;
      seg_scores[(size_t)row * a.k + pos] = score;
    }
  }
  if (!(a.min_len > 0.0f)) {
    if (rank == 0 && tid == 0) {
      seg_count[row] = (int32_t)kr;
      if (nms_in_total) atomicAdd(nms_in_total, (u64)kr);
    }
    D2B_PROF(prof, 8);
    return;
  }
  // prune_small_boxes (rpn_outputs.py:83-87): ordered compaction of the row, in place, by the leader.  A trip reads
  // positions [j0, j0 + 512) before anything is written, and writes land at or below the positions read so far.
  cluster.sync();
  if (rank != 0) return;
  int* s_warp = reinterpret_cast<int*>(s_scan);
  int base = 0;
  for (int j0 = 0; j0 < (int)kr; j0 += kSelThreads) {
    const int j = j0 + tid;
    bool ok = false;
    float4 box = make_float4(0, 0, 0, 0);
    float score = 0.0f;
    if (j < (int)kr) {
      box = __ldcg(seg_boxes + (size_t)row * a.k + j);
      score = __ldcg(seg_scores + (size_t)row * a.k + j);
      const float bh = box.z - box.x, bw = box.w - box.y;
      ok = (bw >= a.min_len) && (bh >= a.min_len);
    }
    const int slot = block_compact<kSelThreads>(ok, base, s_warp);
    if (slot >= 0) {
      seg_boxes[(size_t)row * a.k + slot] = box;
      seg_scores[(size_t)row * a.k + slot] = score;
    }
  }
  if (tid == 0) {
    seg_count[row] = base;
    if (nms_in_total) atomicAdd(nms_in_total, (u64)base);
  }
}

// One CTA per (image, level) segment, one CLUSTER per image (cluster size = number of levels <= 8): every CTA sweeps
// its segment's suppression mask (nms.cuh), then the image's levels are merged into its top `post` proposals
// (rpn_outputs.py:101-114) by all CTAs of the cluster: each publishes the score keys of its survivors (already in
// (score desc, index asc) order) in shared memory, copies the other levels' lists through DSMEM, and ranks ITS OWN
// survivors -- rank = position in its own list + per other level the number of survivors that precede it (binary
// search; ties across levels go to the earlier level = lower concat index, TF top_k rule) -- and writes them
// straight to their output slots.  No sort, no intermediate buffers, no last-block hand-off.
__global__ void __launch_bounds__(kColSweepThreads) rpn_sweep_merge_kernel(
    RpnArgs a, const int32_t* seg_count, int W, int cap, const u64* mask, const float4* seg_boxes,
    const float* seg_scores, float4* out_boxes, float* out_logits, uint8_t* out_valid, int32_t* out_num,
    const int32_t* skip) {
  grid_dep_sync();
  if (skip && skip[blockIdx.x / a.L]) return;  // the whole cluster (= image), before its first barrier
  extern __shared__ uint32_t s_keys[];  // [L][cap] score keys of every level's survivors, then [cap] u16 positions
  __shared__ int s_cnt;
  __shared__ int s_off[D2B_MAX_LEVELS + 1];
  cg::cluster_group cluster = cg::this_cluster();
  const int seg = blockIdx.x;
  const int n = seg / a.L, l = seg - n * a.L;
  const int tid = threadIdx.x;
  const int cnt = min(seg_count[seg], a.k);
  uint32_t* mine = s_keys + (size_t)l * cap;
  uint16_t* s_pos = reinterpret_cast<uint16_t*>(s_keys + (size_t)a.L * cap);
  const float* sc = seg_scores + (size_t)seg * a.k;
  D2B_PROF(blockIdx.x == 0 && tid == 0, 16);
  // the sweep leaves the survivors' positions and score keys in shared memory (selection order = score order)
  const int kept = nms_sweep_columns<true>(cnt, W, cap, mask + (size_t)seg * W * 64 * W, nullptr, sc, mine, s_pos);
  D2B_PROF(blockIdx.x == 0 && tid == 0, 17);
  if (tid == 0) s_cnt = kept;
  cluster.sync();
  if (tid < a.L) s_off[tid + 1] = *cluster.map_shared_rank(&s_cnt, tid);
  if (tid == 0) s_off[0] = 0;
  __syncthreads();
  if (tid == 0) {
    for (int i = 0; i < a.L; ++i) s_off[i + 1] += s_off[i];
  }
  __syncthreads();
  for (int l2 = 0; l2 < a.L; ++l2) {  // copy the other levels' key lists (DSMEM reads, coalesced)
    if (l2 == l) continue;
    const int c2 = s_off[l2 + 1] - s_off[l2];
    const uint32_t* src = cluster.map_shared_rank(s_keys + (size_t)l2 * cap, l2);
    uint32_t* dst = s_keys + (size_t)l2 * cap;
    for (int j = tid; j < c2; j += kColSweepThreads) dst[j] = src[j];
  }
  cluster.sync();  // copies done: from here on every CTA works on its own shared memory only
  D2B_PROF(blockIdx.x == 0 && tid == 0, 20);
  const int total = s_off[a.L];
  const int kk = min(total, a.post);  // :105
  for (int j = tid; j < kept; j += kColSweepThreads) {
    const uint32_t key = mine[j];
    int rank = j;
    for (int l2 = 0; l2 < a.L; ++l2) {
      if (l2 == l) continue;
      const uint32_t* kl = s_keys + (size_t)l2 * cap;
      int lo = 0, hi = s_off[l2 + 1] - s_off[l2];
      while (lo < hi) {  // first position whose element does NOT precede (key, level l)
        const int mid = (lo + hi) >> 1;
        const uint32_t ke = kl[mid];
        const bool before = (l2 < l) ? (ke >= key) : (ke > key);
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    D2B_BOUND(rank, total);
    if (rank < a.post) {
      const int p = s_pos[j];
      D2B_BOUND(p, cnt);
      const size_t o = (size_t)n * a.post + rank;
      out_boxes[o] = seg_boxes[(size_t)seg * a.k + p];
      out_logits[o] = sc[p];
      out_valid[o] = 1;
    }
  }
  for (int j = kk + l * kColSweepThreads + tid; j < a.post; j += a.L * kColSweepThreads) {  // zero padding :111-114
    const size_t o = (size_t)n * a.post + j;
    out_boxes[o] = make_float4(0, 0, 0, 0);
    out_logits[o] = 0.0f;
    out_valid[o] = 0;
  }
  if (l == 0 && tid == 0 && out_num) out_num[n] = kk;
  D2B_PROF(blockIdx.x == 0 && tid == 0, 18);
}

size_t select_smem_bytes(int P) { return kSelOffRaw + 2 * (size_t)P * sizeof(u64); }

// ------------------------------------------------------------------ capped walk in merge order (rpn.cuh)
constexpr int kLazyThreads = 1024;  // 16 threads per candidate of a 64-candidate block
constexpr int kLazyChunk = 1024;    // merge ranks are computed for this many positions of every level at a time

// Candidates (kcap) and kept boxes (vcap) level l can hold.
__host__ __device__ __forceinline__ void lazy_level(const RpnArgs& a, int l, int& kcap, int& vcap) {
  kcap = (int)(a.hwa[l] < (long long)a.k ? a.hwa[l] : (long long)a.k);
  vcap = a.post < kcap ? a.post : kcap;
}

__host__ __device__ __forceinline__ LazyLayout lazy_layout(const RpnArgs& a) {
  int KT = 0, VT = 0;
  for (int l = 0; l < a.L; ++l) {
    int kc, vc;
    lazy_level(a, l, kc, vc);
    KT += kc;
    VT += vc;
  }
  LazyLayout g;
  g.R = KT < kRpnLazyMaxBlocks * 64 ? KT : kRpnLazyMaxBlocks * 64;
  const int ids = a.post < KT ? a.post : KT;
  // [kept canonical boxes VT float4][chunk canonical boxes kLazyChunk float4][keys KT u32][order R u32][ids u32]
  g.o_cbox = (size_t)VT * 16;
  g.o_keys = g.o_cbox + (size_t)kLazyChunk * 16;
  g.o_order = g.o_keys + (size_t)KT * 4;
  g.o_ids = g.o_order + (size_t)g.R * 4;
  g.bytes = g.o_ids + (size_t)ids * 4;
  return g;
}

// One CTA per image.  The merge order is built in chunks: ranks (exactly as rpn_sweep_merge_kernel ranks survivors:
// own position + per other level a binary search, ties to the lower level) of the positions [plo, plo + kLazyChunk)
// of every level; since a rank is never below the position, the order is then complete up to plo + kLazyChunk.  A
// block of 64 candidates in that order is tested against the kept boxes of each candidate's own level (16 threads per
// candidate; a pre-test that the kept box covers a (1 - thr) shrunk span of the candidate in y and x -- implied by
// IoU > thr, with slack for rounding -- then the exact TF rule d2b_iou > thr), the same-level pairs of the diagonal tile
// are tested exactly, and warp 0 resolves the tile (nms_tile_resolve) and appends the kept boxes to their level lists.
// Coordinates carry no level offset: the reference runs NMS per level on the raw boxes.
__global__ void __launch_bounds__(kLazyThreads) rpn_lazy_merge_kernel(
    RpnArgs a, const int32_t* seg_count, const float4* seg_boxes, const float* seg_scores, float thr,
    float4* out_boxes, float* out_logits, uint8_t* out_valid, int32_t* out_num, int32_t* done) {
  grid_dep_sync();
  extern __shared__ __align__(16) unsigned char s_lz[];
  __shared__ float4 s_can[64];  // canonical (ymin, xmin, ymax, xmax) of the block's candidates
  __shared__ float4 s_flt[64];  // (ylo, yhi, xlo, xhi): a suppressing box must reach ylo and xlo, start by yhi and xhi
  __shared__ int s_lvl[64];     // level, -1 past the end
  __shared__ uint32_t s_id[64];  // level << 16 | position
  __shared__ u64 s_diag[64];
  __shared__ unsigned s_dead[2];
  __shared__ int s_cnt[D2B_MAX_LEVELS], s_kc[D2B_MAX_LEVELS], s_koff[D2B_MAX_LEVELS + 1], s_voff[D2B_MAX_LEVELS + 1];
  __shared__ int s_nk, s_total;
  const LazyLayout g = lazy_layout(a);
  const int R = g.R;
  float4* s_kept = reinterpret_cast<float4*>(s_lz);                   // [voff[L]] per-level kept canonical boxes
  float4* s_cbox = reinterpret_cast<float4*>(s_lz + g.o_cbox);        // [kLazyChunk] candidates of the current chunk
  uint32_t* s_keys = reinterpret_cast<uint32_t*>(s_lz + g.o_keys);    // [koff[L]] score keys, per level
  uint32_t* s_order = reinterpret_cast<uint32_t*>(s_lz + g.o_order);  // [R] merge order: level << 16 | position
  uint32_t* s_ids = reinterpret_cast<uint32_t*>(s_lz + g.o_ids);      // [min(post, koff[L])] kept, in output order
  const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, L = a.L;
  const size_t rbase = (size_t)n * L;
  D2B_PROF(n == 0 && tid == 0, 128);  // phase stamps of image 0 (tools/phase_probe.py): 128-131, 132 + block, 200
  if (tid == 0) {
    s_koff[0] = 0; s_voff[0] = 0;
    for (int l = 0; l < L; ++l) {
      int kc, vc;
      lazy_level(a, l, kc, vc);
      s_cnt[l] = min(seg_count[rbase + l], kc);
      s_kc[l] = 0;
      s_koff[l + 1] = s_koff[l] + kc;
      s_voff[l + 1] = s_voff[l] + vc;
    }
    s_nk = 0;
  }
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int l = 0; l < L; ++l) t += s_cnt[l];
    s_total = t;
  }
  for (int l = 0; l < L; ++l) {  // the loads of a trip are issued together
    const int c = s_cnt[l];
    const float* sc = seg_scores + (rbase + l) * a.k;
    for (int p0 = 0; p0 < c; p0 += 4 * kLazyThreads) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int p = p0 + u * kLazyThreads + tid;
        v[u] = p < c ? __ldg(sc + p) : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int p = p0 + u * kLazyThreads + tid;
        if (p < c) {
          D2B_BOUND(s_koff[l] + p, s_koff[L]);
          s_keys[s_koff[l] + p] = float_to_key(v[u]);
        }
      }
    }
  }
  __syncthreads();
  const bool prof = (n == 0 && tid == 0);
  D2B_PROF(prof, 129);
  const int total = s_total;
  const float kf = thr * 0.999f;
  int plo = 0, base = 0, ready = 0;  // order complete on [0, ready); s_cbox holds the candidates of [base, ready)
  bool finished = false;
  for (int b0 = 0;; b0 += 64) {
    const int nk = s_nk;
    if (nk >= a.post || b0 >= total) { finished = true; break; }
    if (b0 >= R) break;  // visit budget spent: this image goes to masks + sweep-merge
    if (b0 >= ready) {
      const int phi = plo + kLazyChunk;
      for (int l = 0; l < L; ++l) {
        const uint32_t* kl = s_keys + s_koff[l];
        for (int p = plo + tid; p < min(phi, s_cnt[l]); p += kLazyThreads) {
          const uint32_t key = kl[p];
          int rank = p;
          for (int l2 = 0; l2 < L && rank < R; ++l2) {
            if (l2 == l) continue;
            const uint32_t* k2 = s_keys + s_koff[l2];
            int lo = 0, hi = s_cnt[l2];
            while (lo < hi) {  // first position whose element does NOT precede (key, level l)
              const int mid = (lo + hi) >> 1;
              const uint32_t ke = k2[mid];
              const bool before = (l2 < l) ? (ke >= key) : (ke > key);
              if (before) lo = mid + 1; else hi = mid;
            }
            rank += lo;
          }
          if (rank < R) s_order[rank] = ((uint32_t)l << 16) | (uint32_t)p;
        }
      }
      __syncthreads();
      D2B_PROF(prof && plo == 0, 130);
      base = ready;
      ready = min(min(phi, total), R);
      plo = phi;
      for (int q = base + tid; q < ready; q += kLazyThreads) {
        const uint32_t id = s_order[q];
        const int l = (int)(id >> 16), p = (int)(id & 0xffffu);
        D2B_BOUND(l, L);
        D2B_BOUND(p, s_cnt[l]);
        D2B_BOUND(q - base, kLazyChunk);
        const float4 b = __ldg(seg_boxes + (rbase + l) * a.k + p);
        s_cbox[q - base] = make_float4(fminf(b.x, b.z), fminf(b.y, b.w), fmaxf(b.x, b.z), fmaxf(b.y, b.w));
      }
      __syncthreads();
      D2B_PROF(prof && base == 0, 131);
    }
    const int rows = min(64, ready - b0);
    if (tid < 64) {
      int lv = -1;
      uint32_t id = 0;
      float4 c = make_float4(0, 0, 0, 0), f = c;
      if (tid < rows) {
        D2B_BOUND(b0 + tid, R);
        id = s_order[b0 + tid];
        lv = (int)(id >> 16);
        c = s_cbox[b0 + tid - base];
        const float h = c.z - c.x, w = c.w - c.y;
        const float ey = 1e-6f * (fabsf(c.x) + fabsf(c.z)), ex = 1e-6f * (fabsf(c.y) + fabsf(c.w));
        f = make_float4(c.x + kf * h - ey, c.z - kf * h + ey, c.y + kf * w - ex, c.w - kf * w + ex);
      }
      s_can[tid] = c; s_flt[tid] = f; s_lvl[tid] = lv; s_id[tid] = id;
    }
    if (tid < 2) s_dead[tid] = 0;
    __syncthreads();
    // candidate r against the kept boxes of its level; the two candidates of a warp stop together once both are dead
    const int r = tid >> 4, sub = tid & 15;
    const int lv = s_lvl[r];
    const float4 cr = s_can[r], fr = s_flt[r];
    const int kc = lv >= 0 ? s_kc[lv] : 0;
    const float4* kl = s_kept + (lv >= 0 ? s_voff[lv] : 0);
    const int kmax = max(kc, __shfl_xor_sync(0xffffffffu, kc, 16));
    const unsigned half = (lane < 16) ? 0x0000ffffu : 0xffff0000u;
    bool dead = false;
    for (int j0 = 0; j0 < kmax; j0 += 16) {
      const int j = j0 + sub;
      bool hit = false;
      if (j < kc && !dead) {
        const float4 kb = kl[j];
        if (kb.z >= fr.x && kb.x <= fr.y && kb.w >= fr.z && kb.y <= fr.w) hit = d2b_iou(cr, kb) > thr;
      }
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      dead = dead || (m & half) != 0;
      if (__all_sync(0xffffffffu, dead)) break;
    }
    if (dead && sub == 0) atomicOr(&s_dead[r >> 5], 1u << (r & 31));
    // diagonal tile: bit c of row r = candidate r suppresses candidate c (c > r, same level)
    u64 bits = 0;
    if (lv >= 0)
      for (int c = r + 1 + sub; c < rows; c += 16)
        if (s_lvl[c] == lv && d2b_iou(cr, s_can[c]) > thr) bits |= 1ull << c;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) bits |= __shfl_xor_sync(0xffffffffu, bits, o);
    if (sub == 0) s_diag[r] = bits;
    __syncthreads();
    if (tid < 32) {
      u64 rem = ((u64)s_dead[1] << 32) | (u64)s_dead[0];
      if (rows < 64) rem |= ~0ull << rows;
      const u64 K = nms_tile_resolve(s_diag[lane], s_diag[lane + 32], rem, a.post - nk);
      const u64 bitA = 1ull << lane, bitB = 1ull << (lane + 32);
      const int lA = s_lvl[lane], lB = s_lvl[lane + 32];
      u64 sameA = 0, sameB = 0;
      int mine = 0;  // lane l < L: boxes of level l kept in this block
      for (int l = 0; l < L; ++l) {
        const u64 m = ((u64)__ballot_sync(0xffffffffu, lB == l) << 32) | __ballot_sync(0xffffffffu, lA == l);
        if (lA == l) sameA = m;
        if (lB == l) sameB = m;
        if (lane == l) mine = __popcll(K & m);
      }
      if (K & bitA) {
        const int slot = s_kc[lA] + __popcll(K & sameA & (bitA - 1ull)), o = nk + __popcll(K & (bitA - 1ull));
        D2B_BOUND(slot, s_voff[lA + 1] - s_voff[lA]);
        D2B_BOUND(o, a.post);
        s_kept[s_voff[lA] + slot] = s_can[lane];
        s_ids[o] = s_id[lane];
      }
      if (K & bitB) {
        const int slot = s_kc[lB] + __popcll(K & sameB & (bitB - 1ull)), o = nk + __popcll(K & (bitB - 1ull));
        D2B_BOUND(slot, s_voff[lB + 1] - s_voff[lB]);
        D2B_BOUND(o, a.post);
        s_kept[s_voff[lB] + slot] = s_can[lane + 32];
        s_ids[o] = s_id[lane + 32];
      }
      __syncwarp();
      if (lane < L) s_kc[lane] += mine;
      if (lane == 0) s_nk = nk + __popcll(K);
    }
    __syncthreads();
    D2B_PROF(prof, 132 + (b0 >> 6));
  }
  if (!finished) {
    if (tid == 0) done[n] = 0;
    return;
  }
  // outputs as rpn_sweep_merge_kernel writes them: the kept boxes in merge order, then zero padding (:101-114)
  const int nk = s_nk;
  for (int o = tid; o < a.post; o += kLazyThreads) {
    float4 box = make_float4(0, 0, 0, 0);
    float logit = 0.0f;
    uint8_t valid = 0;
    if (o < nk) {
      const uint32_t id = s_ids[o];
      const size_t src = (rbase + (id >> 16)) * a.k + (id & 0xffffu);
      box = seg_boxes[src];
      logit = seg_scores[src];
      valid = 1;
    }
    const size_t dst = (size_t)n * a.post + o;
    out_boxes[dst] = box;
    out_logits[dst] = logit;
    out_valid[dst] = valid;
  }
  if (tid == 0) {
    if (out_num) out_num[n] = nk;
    done[n] = 1;
  }
  D2B_PROF(prof, 200);
}

}  // namespace

size_t rpn_lazy_merge_smem(const RpnArgs& a) { return lazy_layout(a).bytes; }

int rpn_lazy_merge_fused(const RpnArgs& a, const int32_t* seg_count, const float4* seg_boxes, const float* seg_scores,
                         float thr, float4* out_boxes, float* out_logits, uint8_t* out_valid, int32_t* out_num,
                         int32_t* done, cudaStream_t st) {
  D2B_REQUIRE(a.k <= kRpnFusedMaxK && a.L <= D2B_MAX_LEVELS, "lazy merge: k=%d, L=%d out of range", a.k, a.L);
  const size_t smem = rpn_lazy_merge_smem(a);
  D2B_REQUIRE(smem <= kRpnLazyMaxSmem, "lazy merge: %zu bytes of shared memory > %zu", smem, kRpnLazyMaxSmem);
  if (a.N == 0) return D2B_OK;
  D2B_CUDA(allow_dynamic_smem(rpn_lazy_merge_kernel, smem));
  D2B_CUDA(launch_pdl(rpn_lazy_merge_kernel, dim3((unsigned)a.N), dim3(kLazyThreads), smem, st, 0, a, seg_count,
                      seg_boxes, seg_scores, thr, out_boxes, out_logits, out_valid, out_num, done));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

int rpn_select_fused(const RpnArgs& a, float4* seg_boxes, float* seg_scores, int32_t* seg_count,
                     unsigned long long* nms_in_total, cudaStream_t st) {
  static_assert(sizeof(SelCtl) <= 256, "control block must fit its slot");
  D2B_REQUIRE(a.k <= kRpnFusedMaxK, "fused proposal stage: k=%d > %d", a.k, kRpnFusedMaxK);
  const int rows = a.L * a.N;
  if (rows == 0) return D2B_OK;
  const size_t smem = select_smem_bytes(a.P);
  if (smem > 48 * 1024)
    D2B_CUDA(cudaFuncSetAttribute(rpn_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  D2B_CUDA(launch_pdl(rpn_select_kernel, dim3((unsigned)rows * kSelCluster, 1, 1), dim3(kSelThreads, 1, 1), smem, st,
                      kSelCluster, a, seg_boxes, seg_scores, seg_count, reinterpret_cast<u64*>(nms_in_total)));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

int rpn_sweep_merge_fused(const RpnArgs& a, const int32_t* seg_count, const unsigned long long* mask,
                          const float4* seg_boxes, const float* seg_scores, float4* out_boxes, float* out_logits,
                          uint8_t* out_valid, int32_t* out_num, const int32_t* skip, cudaStream_t st) {
  const int rows = a.L * a.N;
  if (rows == 0) return D2B_OK;
  const int W = (a.k + 63) / 64;
  D2B_REQUIRE(W <= kColSweepMaxW, "fused sweep: k=%d too large", a.k);
  const int cap = a.post < a.k ? a.post : a.k;  // survivors per segment
  const size_t smem = (size_t)a.L * cap * sizeof(uint32_t) + align_up((size_t)cap * sizeof(uint16_t), 16);
  D2B_REQUIRE(smem <= 200 * 1024, "fused sweep: %d levels x %d survivors do not fit shared memory", a.L, cap);
  D2B_CUDA(allow_dynamic_smem(rpn_sweep_merge_kernel, smem));
  // one cluster per image (L <= D2B_MAX_LEVELS = 8: portable size)
  D2B_CUDA(launch_pdl(rpn_sweep_merge_kernel, dim3((unsigned)rows, 1, 1), dim3(kColSweepThreads, 1, 1), smem, st,
                      (unsigned)a.L, a, seg_count, W, cap, reinterpret_cast<const u64*>(mask), seg_boxes, seg_scores,
                      out_boxes, out_logits, out_valid, out_num, skip));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

}  // namespace d2b

#ifdef D2B_PROFILE
// Debug builds only (-DD2B_PROFILE): copies the 256 phase timestamps of this translation unit to `out`.
extern "C" __attribute__((visibility("default"))) int d2b_debug_read_profile(unsigned long long* out) {
  return cudaMemcpyFromSymbol(out, d2b::g_d2b_prof, sizeof(unsigned long long) * 256) == cudaSuccess ? 0 : -2;
}
#endif
