// nms.cuh -- device pieces of the bitmask NMS shared by nms.cu and rpn_fused.cu.
#pragma once
#include <cooperative_groups.h>

#include "kernels.cuh"

namespace d2b {

__device__ __forceinline__ unsigned long long warp_or64(unsigned long long v) {
  const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v);
  const unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
  return ((unsigned long long)hi << 32) | lo;
}

// Greedy resolve of one 64-candidate tile by a full warp, as a fixpoint (same result as the serial scan).  Lane l
// holds the suppression rows of candidates l and l + 32 (dA, dB: bit c set = the row's candidate suppresses candidate
// c, c > row); `rem` marks candidates already removed (suppressed from outside the tile, or absent).  Returns the
// kept candidates, of which at most `left` (the first ones) remain when the cap is reached inside the tile.
// Shared by the bitmask sweep (nms_sweep_columns), det_tail_kernel and rpn_lazy_merge_kernel.
__device__ __forceinline__ unsigned long long nms_tile_resolve(unsigned long long dA, unsigned long long dB,
                                                               unsigned long long rem, int left) {
  typedef unsigned long long u64;
  const int lane = threadIdx.x & 31;
  const u64 bitA = 1ull << lane, bitB = 1ull << (lane + 32);
  u64 U = ~rem, K = 0;
  while (U) {  // warp-uniform
    const u64 blocked = warp_or64(((U & bitA) ? dA : 0ull) | ((U & bitB) ? dB : 0ull));
    const u64 nk = U & ~blocked;  // never empty: the first undecided candidate cannot be blocked
    K |= nk;
    U &= ~nk;
    if (!U) break;  // (the usual sparse tile: nothing undecided is blocked, one round)
    U &= ~warp_or64(((nk & bitA) ? dA : 0ull) | ((nk & bitB) ? dB : 0ull));
  }
  int c = __popcll(K);
  while (c > left) {  // cap reached inside this tile: keep only the first `left`
    K &= ~(1ull << (63 - __clzll((long long)K)));
    --c;
  }
  return K;
}

// Greedy sweep over the suppression bitmask of ONE segment by a CTA of kColSweepThreads threads (32 warps).
// mask word (row i, column word w), bit c: box i suppresses box 64w+c (only c > i is set / read).  In global memory
// the mask is stored COLUMN-WORD MAJOR -- word (i, w) at w * (64 W) + i -- so that the 64 rows of a block's column
// word are 512 contiguous bytes: the sweep's loads (lane = row) and nms_mask_kernel's stores (lane = row) are
// coalesced; row-major they were 32 separate sectors per warp access.  Warp q OWNS the column words
// q, q+32, ...: for word b it ORs, block by block, the rows of the KEPT boxes of every earlier 64-row block into a
// per-lane accumulator (lane = rows l and l+32 of the block; the loads do not depend on the kept bits, so they are
// issued several blocks ahead of the flag they wait for), then resolves the diagonal 64x64 tile with a
// warp-parallel fixpoint and publishes the kept bits of block b in shared memory.  The serial chain per block is
// flag -> select -> REDUX -> fixpoint (a few hundred cycles, all shared memory / registers); every global load is
// off that chain.  Same result as the serial greedy scan: a box is kept iff no earlier kept box suppresses it.
// Blocks after the cap (max_out kept) publish an empty set at once.  Returns the number of kept boxes (uniform
// over the CTA, after a __syncthreads()).
constexpr int kColSweepThreads = 1024;
// position of mask word (row, column word) of a segment whose mask has W column words (64 W rows)
__host__ __device__ __forceinline__ size_t nms_mask_index(int row, int word, int W) {
  return (size_t)word * ((size_t)W * 64) + (size_t)row;
}
constexpr int kColSweepMaxW = 1024;  // n <= 65536 (a warp owns words q, q + 32, ...: up to 32 of them)

// SMEM_OUT: instead of the global keep list, the kept boxes' positions and the order-preserving keys of their scores
// (sc = the segment's scores in candidate order) go to shared memory (s_pos / s_key, max_out entries each).
// MASK_SMEM: the mask lives in shared memory, row-major [row][W] (plain loads instead of ld.global.cg).
// CL > 1: the segment is swept by a CLUSTER of CL CTAs (launch with cluster dimension CL; every CTA calls this with the
// same arguments): warp (rank * 32 + warp) owns the column words congruent to it modulo 32 CL, so the mask streams
// into CL SMs instead of one (a 65,536-box segment is 268 MB of upper triangle), and the owner of a block publishes
// its kept bits into the shared memory of EVERY CTA of the cluster (st.shared::cluster + a cluster-scope fence before
// the flag); the polling stays local.  The return value is valid in every CTA; rank 0 writes the -1 padding.
template <bool SMEM_OUT = false, bool MASK_SMEM = false, int CL = 1>
__device__ __forceinline__ int nms_sweep_columns(int cnt, int W, int max_out, const unsigned long long* __restrict__ m,
                                                 int32_t* __restrict__ kp, const float* __restrict__ sc = nullptr,
                                                 uint32_t* s_key = nullptr, uint16_t* s_pos = nullptr) {
  typedef unsigned long long u64;
  auto ldm = [&](int row, int word) -> u64 {
    return MASK_SMEM ? m[(size_t)row * W + word] : __ldcg(m + nms_mask_index(row, word, W));
  };
  __shared__ volatile u64 s_keep[kColSweepMaxW];
  __shared__ volatile int s_flag[kColSweepMaxW];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = (cnt + 63) >> 6;
  if (tid < kColSweepMaxW) { s_keep[tid] = 0; s_flag[tid] = 0; }
  namespace cg = cooperative_groups;
  int crank = 0;
  if constexpr (CL > 1) {
    crank = (int)cg::this_cluster().block_rank();
    cg::this_cluster().sync();  // nobody publishes into a peer that has not cleared its flags yet
  } else {
    __syncthreads();
  }
  const u64 bitA = 1ull << lane, bitB = 1ull << (lane + 32);
  constexpr int kAhead = 4;  // blocks whose rows are loaded before their flag is awaited
  for (int word = crank * 32 + warp; word < nb; word += 32 * CL) {
    u64 acc = 0;
    int kept_before = 0;
    bool capped = false;
    // the diagonal tile of this block (independent of everything before it): in flight during the wait below
    const int rows = min(64, cnt - word * 64);
    u64 dA = 0, dB = 0;
    if (lane < rows) dA = ldm(word * 64 + lane, word);
    if (lane + 32 < rows) dB = ldm(word * 64 + 32 + lane, word);
    float scA = 0.0f, scB = 0.0f;
    if (SMEM_OUT) {
      if (lane < rows) scA = __ldg(sc + word * 64 + lane);
      if (lane + 32 < rows) scB = __ldg(sc + word * 64 + 32 + lane);
    }
    u64 pa[kAhead], pb[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      pa[u] = 0; pb[u] = 0;
      if (u < word) {
        pa[u] = ldm(u * 64 + lane, word);
        pb[u] = ldm(u * 64 + 32 + lane, word);
      }
    }
    for (int b0 = 0; b0 < word && !capped; b0 += kAhead) {
#pragma unroll
      for (int u = 0; u < kAhead; ++u) {
        const int b = b0 + u;
        if (b < word && !capped) {  // warp-uniform
          const u64 va = pa[u], vb = pb[u];
          const int nx = b + kAhead;  // refill this slot for the block kAhead further on
          if (nx < word) {
            D2B_BOUND(nx * 64 + 32 + lane, (long long)W * 64);
            pa[u] = ldm(nx * 64 + lane, word);
            pb[u] = ldm(nx * 64 + 32 + lane, word);
          }
          // only the owner of the next block polls back to back; warps further from their turn sleep in between, so
          // that the polling does not take issue slots and shared-memory bandwidth from the warp on the critical path
          while (s_flag[b] == 0) {
            const int dist = word - b;
            if (dist > 1) __nanosleep(dist > 8 ? 400 : 50 * dist);
          }
          if constexpr (CL > 1) asm volatile("fence.acq_rel.cluster;" ::: "memory");  // the flag came from a peer CTA
          const u64 K = s_keep[b];
          acc |= ((K & bitA) ? va : 0ull) | ((K & bitB) ? vb : 0ull);
          kept_before += __popcll(K);
          capped = kept_before >= max_out;
        }
      }
    }
    u64 K = 0;
    if (!capped) {
      u64 rem = warp_or64(acc);
      if (rows < 64) rem |= ~0ull << rows;
      K = nms_tile_resolve(dA, dB, rem, max_out - kept_before);
      D2B_BOUND(word, W);
      if (K & bitA) {
        const int slot = kept_before + __popcll(K & (bitA - 1ull));
        D2B_BOUND(slot, max_out);
        if (SMEM_OUT) { s_key[slot] = float_to_key(scA); s_pos[slot] = (uint16_t)(word * 64 + lane); }
        else kp[slot] = word * 64 + lane;
      }
      if (K & bitB) {
        const int slot = kept_before + __popcll(K & (bitB - 1ull));
        D2B_BOUND(slot, max_out);
        if (SMEM_OUT) { s_key[slot] = float_to_key(scB); s_pos[slot] = (uint16_t)(word * 64 + 32 + lane); }
        else kp[slot] = word * 64 + 32 + lane;
      }
    }
    __syncwarp();
    if constexpr (CL > 1) {
      if (lane < CL) {  // lane p publishes into CTA p of the cluster (its own included)
        volatile u64* rk = cg::this_cluster().map_shared_rank(const_cast<u64*>(&s_keep[word]), lane);
        volatile int* rf = cg::this_cluster().map_shared_rank(const_cast<int*>(&s_flag[word]), lane);
        *rk = K;
        asm volatile("fence.acq_rel.cluster;" ::: "memory");
        *rf = 1;
      }
    } else if (lane == 0) {
      s_keep[word] = K;
      __threadfence_block();
      s_flag[word] = 1;
      D2B_PROF(blockIdx.x == 0 && word < 32, 32 + word);
    }
  }
  if constexpr (CL > 1) cg::this_cluster().sync();  // (also: no CTA exits while a peer may still store into it)
  else __syncthreads();
  int kept = 0;
  for (int b = 0; b < nb; ++b) kept += __popcll(s_keep[b]);
  kept = min(kept, max_out);
  if (!SMEM_OUT && crank == 0)
    for (int j = kept + tid; j < max_out; j += kColSweepThreads) kp[j] = -1;
  return kept;
}

}  // namespace d2b
