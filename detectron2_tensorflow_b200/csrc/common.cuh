// common.cuh -- shared helpers for the sm_100a kernels of libd2b200.
// The library is compiled with -fmad=false: every written fp32 operation is one
// IEEE rounding, so kernels reproduce the reference's op order bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "d2b200.h"

namespace d2b {

void set_last_error(const char* fmt, ...);
void count_launch();  // every kernel launch of the library bumps d2b_kernel_launch_count()

#define D2B_REQUIRE(cond, ...)              \
  do {                                      \
    if (!(cond)) {                          \
      ::d2b::set_last_error(__VA_ARGS__);   \
      return D2B_EINVAL;                    \
    }                                       \
  } while (0)

#define D2B_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      ::d2b::set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                            __FILE__, __LINE__);                                         \
      return D2B_ECUDA;                                                                  \
    }                                                                                    \
  } while (0)

#define D2B_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    ::d2b::count_launch();                                                               \
    cudaError_t _e = cudaGetLastError();                                                 \
    if (_e != cudaSuccess) {                                                             \
      ::d2b::set_last_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),  \
                            __FILE__, __LINE__);                                         \
      return D2B_ECUDA;                                                                  \
    }                                                                                    \
  } while (0)

// -DD2B_DEBUG_BOUNDS (D2B_EXTRA_NVCC=-DD2B_DEBUG_BOUNDS python -m detectron2_tensorflow_b200.build --force): device-side
// asserts on computed indices of the scan / select / NMS / dynamic-conv kernels.  A violated bound traps the kernel
// (cudaErrorAssert) and every later call of the process fails; the parity suite is run once under this build and the
// log is committed under profiles/.  Compiled out of the product build.
#ifdef D2B_DEBUG_BOUNDS
#include <assert.h>
#define D2B_BOUND(i, n) assert((unsigned long long)(i) < (unsigned long long)(n))
#else
#define D2B_BOUND(i, n) ((void)0)
#endif

// -DD2B_PROFILE: phase timestamps (%globaltimer, ns) of selected CTAs in a device array read back by
// d2b_debug_read_profile() (tools/phase_probe.py).  Compiled out of the product build.
#ifdef D2B_PROFILE
static __device__ unsigned long long g_d2b_prof[256];  // one copy per translation unit (no -rdc)
__device__ __forceinline__ void d2b_prof_stamp(int slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  g_d2b_prof[slot] = t;
}
#define D2B_PROF(cond, slot) do { if (cond) ::d2b::d2b_prof_stamp(slot); } while (0)
#else
#define D2B_PROF(cond, slot) do { } while (0)
#endif

// ---------------------------------------------------------------- programmatic dependent launch
// The latency chains (proposal stage -> pooler -> detection tail) are sequences of short kernels; with the
// programmatic-stream-serialization attribute the NEXT kernel's CTAs are scheduled while the current one drains,
// and `grid_dep_sync()` at the top of every such kernel blocks until the predecessor has completed and its writes
// are visible.  Rules: (1) a kernel launched through launch_pdl() calls grid_dep_sync() before it touches global
// memory -- every thread, unconditionally; (2) kernels launched the ordinary way are unaffected.  MEASURED (B200,
// profiles/r02aj_step_probe_*.jsonl): eager chains gain (Fast R-CNN post 87 -> 68 us at 2 images), but the step the
// bench replays is a captured multi-stream graph and there the programmatic edges cost time (2 image blocks: 0.209 ->
// 0.257 ms; 4 blocks of 16 images: 0.648 -> 0.701 ms).  Hence: the attribute is set on EAGER launches only -- never
// while the stream is being captured.  The RetinaNet top-k chain does not use it at all: there it measured slower
// even eagerly (0.572 -> 0.645 ms at N = 32: the early CTAs of the dependents take slots from the HBM-bound scan);
// Matrix-NMS gains a little (0.418 -> 0.4135 ms).
bool pdl_enabled(cudaStream_t st);
__device__ __forceinline__ void grid_dep_sync() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
struct LaunchCfg {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  LaunchCfg(dim3 grid, dim3 block, size_t smem, cudaStream_t st, unsigned cluster_x = 0) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 0;
    if (cluster_x) {
      attr[cfg.numAttrs].id = cudaLaunchAttributeClusterDimension;
      attr[cfg.numAttrs].val.clusterDim.x = cluster_x;
      attr[cfg.numAttrs].val.clusterDim.y = 1;
      attr[cfg.numAttrs].val.clusterDim.z = 1;
      ++cfg.numAttrs;
    }
    if (pdl_enabled(st)) {
      attr[cfg.numAttrs].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[cfg.numAttrs].val.programmaticStreamSerializationAllowed = 1;
      ++cfg.numAttrs;
    }
  }
};
// launch_pdl(kernel, grid, block, smem, stream, cluster_x, args...): the kernel MUST call grid_dep_sync() first.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     unsigned cluster_x, Args&&... args) {
  LaunchCfg L(grid, block, smem, st, cluster_x);
  return cudaLaunchKernelEx(&L.cfg, kernel, static_cast<KArgs>(args)...);
}

// Raises `kernel`'s dynamic shared-memory limit to `smem` bytes when it is below that.  For a kernel with static
// shared memory the default limit is 48 KB MINUS the static size, so a fixed "smem > 48 KB" test misses the sizes just
// below 48 KB.  The limit is per kernel and per device, and is only ever raised.
template <typename... KArgs>
static inline cudaError_t allow_dynamic_smem(void (*kernel)(KArgs...), size_t smem) {
  cudaFuncAttributes fa;
  const cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
  if (e != cudaSuccess || smem <= (size_t)fa.maxDynamicSharedSizeBytes) return e;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over the caller's workspace (256-byte aligned slices).
struct Workspace {
  char* base;
  size_t off;
  explicit Workspace(void* p) : base(static_cast<char*>(p)), off(0) {}
  template <typename T>
  T* take(size_t count) {
    T* r = reinterpret_cast<T*>(base + off);
    off += align_up(count * sizeof(T), 256);
    return r;
  }
};
static inline size_t ws_slice(size_t bytes) { return align_up(bytes, 256); }

// ---------------------------------------------------------------- math
// Cephes single-precision exp/log in the form Eigen's packet math evaluates them
// (TF's CPU backend), separate multiply and add.  Same operation sequence as the
// test oracle's restatement; results are bit-identical by construction.
__device__ __forceinline__ float d2b_expf(float x0) {
  float x = x0;
  if (x != x) return x;
  x = fminf(x, 88.3762626647950f);
  x = fmaxf(x, -88.3762626647949f);
  float fx = x * 1.44269504088896341f;
  fx = fx + 0.5f;
  fx = floorf(fx);
  float tmp = fx * 0.693359375f;
  float z = fx * -2.12194440e-4f;
  x = x - tmp;
  x = x - z;
  z = x * x;
  float y = 1.9875691500E-4f;
  y = y * x; y = y + 1.3981999507E-3f;
  y = y * x; y = y + 8.3334519073E-3f;
  y = y * x; y = y + 4.1665795894E-2f;
  y = y * x; y = y + 1.6666665459E-1f;
  y = y * x; y = y + 5.0000001201E-1f;
  y = y * z; y = y + x;
  y = y + 1.0f;
  int n = (int)fx;
  float p2n = __int_as_float((n + 0x7f) << 23);
  y = y * p2n;
  return fmaxf(y, x0);
}

__device__ __forceinline__ float d2b_logf(float x0) {
  if (x0 != x0) return x0;
  if (x0 < 0.0f) return __int_as_float(0x7fc00000);
  if (x0 == 0.0f) return __int_as_float(0xff800000);
  if (x0 == __int_as_float(0x7f800000)) return x0;
  float x = fmaxf(x0, __int_as_float(0x00800000));
  uint32_t ux = __float_as_uint(x);
  int emm0 = (int)(ux >> 23);
  ux = (ux & ~0x7f800000u) | 0x3f000000u;
  x = __uint_as_float(ux);
  emm0 -= 0x7f;
  float e = (float)emm0;
  e = e + 1.0f;
  if (x < 0.707106781186547524f) {
    float t = x;
    x = x - 1.0f;
    e = e - 1.0f;
    x = x + t;
  } else {
    x = x - 1.0f;
  }
  float x2 = x * x;
  float x3 = x2 * x;
  float y, y1, y2;
  y = 7.0376836292E-2f * x;   y = y + -1.1514610310E-1f;
  y1 = -1.2420140846E-1f * x; y1 = y1 + 1.4249322787E-1f;
  y2 = 2.0000714765E-1f * x;  y2 = y2 + -2.4999993993E-1f;
  y = y * x;   y = y + 1.1676998740E-1f;
  y1 = y1 * x; y1 = y1 + -1.6668057665E-1f;
  y2 = y2 * x; y2 = y2 + 3.3333331174E-1f;
  y = y * x3; y = y + y1;
  y = y * x3; y = y + y2;
  y = y * x3;
  y1 = e * -2.12194440e-4f;
  float tmp = x2 * 0.5f;
  y = y + y1;
  x = x - tmp;
  y2 = e * 0.693359375f;
  x = x + y;
  x = x + y2;
  return x;
}

__device__ __forceinline__ float d2b_sigmoidf(float x) {
  float e = d2b_expf(-x);
  float d = 1.0f + e;
  return __frcp_rn(d);  // correctly rounded reciprocal == IEEE 1.0f / d
}

// Order-preserving fp32 -> u32 key: larger float <=> larger key; -0 == +0;
// NaN maps to 0 (ranks below -inf).
__device__ __forceinline__ uint32_t float_to_key(float x) {
  if (x != x) return 0u;
  if (x == 0.0f) x = 0.0f;  // canonical +0
  uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  if (k == 0u) return __int_as_float(0x7fc00000);
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

// TF NonMaxSuppression CPU kernel IoU (division form).
__device__ __forceinline__ float d2b_iou(const float4 a, const float4 b) {
  // float4 = (y1, x1, y2, x2) as stored
  const float ymin_i = fminf(a.x, a.z), xmin_i = fminf(a.y, a.w);
  const float ymax_i = fmaxf(a.x, a.z), xmax_i = fmaxf(a.y, a.w);
  const float ymin_j = fminf(b.x, b.z), xmin_j = fminf(b.y, b.w);
  const float ymax_j = fmaxf(b.x, b.z), xmax_j = fmaxf(b.y, b.w);
  const float area_i = (ymax_i - ymin_i) * (xmax_i - xmin_i);
  const float area_j = (ymax_j - ymin_j) * (xmax_j - xmin_j);
  if (area_i <= 0.0f || area_j <= 0.0f) return 0.0f;
  const float iymin = fmaxf(ymin_i, ymin_j), ixmin = fmaxf(xmin_i, xmin_j);
  const float iymax = fminf(ymax_i, ymax_j), ixmax = fminf(xmax_i, xmax_j);
  const float ih = fmaxf(iymax - iymin, 0.0f), iw = fmaxf(ixmax - ixmin, 0.0f);
  const float inter = ih * iw;
  float u = area_i + area_j;
  u = u - inter;
  return inter / u;
}

// Box2BoxTransform.apply_deltas on one (delta, box) pair.
__device__ __forceinline__ float4 d2b_decode(const float4 d, const float4 b, float wy, float wx,
                                             float wh, float ww, float clampv) {
  const float heights = b.z - b.x;
  const float widths = b.w - b.y;
  float cy = 0.5f * heights; cy = b.x + cy;
  float cx = 0.5f * widths;  cx = b.y + cx;
  float dy = d.x / wy, dx = d.y / wx, dh = d.z / wh, dw = d.w / ww;
  dh = fminf(dh, clampv);
  dw = fminf(dw, clampv);
  float pcy = dy * heights; pcy = pcy + cy;
  float pcx = dx * widths;  pcx = pcx + cx;
  float ph = d2b_expf(dh) * heights;
  float pw = d2b_expf(dw) * widths;
  float hh = 0.5f * ph, hw = 0.5f * pw;
  return make_float4(pcy - hh, pcx - hw, pcy + hh, pcx + hw);
}

__device__ __forceinline__ float4 d2b_clip(float4 b, float h, float w) {
  b.x = fmaxf(fminf(b.x, h), 0.0f);
  b.y = fmaxf(fminf(b.y, w), 0.0f);
  b.z = fmaxf(fminf(b.z, h), 0.0f);
  b.w = fmaxf(fminf(b.w, w), 0.0f);
  return b;
}

}  // namespace d2b
