// boxes.cu -- Box2BoxTransform.apply_deltas and the stand-alone batched NMS entry.
#include "kernels.cuh"

namespace d2b {
namespace {

typedef unsigned long long u64;

// box_regression.py:95-123; one thread per (box, class-slot)
__global__ void apply_deltas_kernel(const float4* deltas, const float4* boxes, long long n, int k, float wy,
                                    float wx, float wh, float ww, float clampv, float4* out) {
  grid_dep_sync();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * k) return;
  const long long i = t / k;
  out[t] = d2b_decode(__ldg(deltas + t), __ldg(boxes + i), wy, wx, wh, ww, clampv);
}

// candidates = { i : score > -inf } ordered (score desc, index asc); dead slots key 0
__global__ void nms_prep_kernel(const float* scores, const int32_t* counts, int n, int P, u64* keys,
                                int32_t* live) {
  const int seg = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int cnt = counts ? min(counts[seg], n) : n;
  bool ok = false;
  if (i < P) {
    u64 key = 0;
    if (i < cnt) {
      const float s = scores[(size_t)seg * n + i];
      if (s > __int_as_float(0xff800000)) {
        key = ((u64)float_to_key(s) << 32) | (u64)(0xffffffffu - (unsigned)i);
        ok = true;
      }
    }
    keys[(size_t)seg * P + i] = key;
  }
  const unsigned m = __ballot_sync(0xffffffffu, ok);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(live + seg, __popc(m));
}

__global__ void nms_gather_kernel(const float4* boxes, const u64* keys, const int32_t* live, int n, int P,
                                  float4* sorted) {
  const int seg = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= live[seg]) return;
  const unsigned idx = 0xffffffffu - (unsigned)keys[(size_t)seg * P + j];
  sorted[(size_t)seg * n + j] = boxes[(size_t)seg * n + idx];
}

__global__ void nms_unmap_kernel(const u64* keys, int P, int max_out, const int32_t* num_keep, int32_t* keep) {
  const int seg = blockIdx.y;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= max_out) return;
  int32_t v = -1;
  if (q < num_keep[seg]) {
    const int j = keep[(size_t)seg * max_out + q];
    v = (int32_t)(0xffffffffu - (unsigned)keys[(size_t)seg * P + j]);
  }
  keep[(size_t)seg * max_out + q] = v;
}

}  // namespace
}  // namespace d2b

using namespace d2b;

extern "C" size_t d2b_apply_deltas_workspace_bytes(const d2b_apply_deltas_params*) { return 0; }

extern "C" int d2b_apply_deltas(const d2b_apply_deltas_params* p, void*, size_t, d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->n >= 0 && p->k >= 1, "apply_deltas: bad sizes n=%lld k=%d", (long long)p->n, p->k);
  if (p->n == 0) return D2B_OK;
  D2B_REQUIRE(p->deltas && p->boxes && p->out, "apply_deltas: NULL pointer");
  const long long total = p->n * p->k;
  D2B_REQUIRE(total < (1ll << 31) * 256, "apply_deltas: too many boxes");
  D2B_CUDA(launch_pdl(apply_deltas_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), 0,
      reinterpret_cast<const float4*>(p->deltas), reinterpret_cast<const float4*>(p->boxes), p->n, p->k,
      p->weights[0], p->weights[1], p->weights[2], p->weights[3], p->scale_clamp,
      reinterpret_cast<float4*>(p->out)));
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

static int nms_pad(int n) {
  int P = 1;
  while (P < n) P <<= 1;
  return P;
}

extern "C" size_t d2b_batched_nms_workspace_bytes(const d2b_batched_nms_params* p) {
  if (!p || p->num_segments <= 0 || p->n <= 0) return 0;
  const size_t S = p->num_segments, n = p->n, P = nms_pad(p->n);
  return ws_slice(S * P * sizeof(unsigned long long)) + ws_slice(S * sizeof(int32_t)) +
         ws_slice(S * n * sizeof(float4)) + nms_sorted_workspace_bytes(p->num_segments, p->n, p->max_output_size);
}

extern "C" int d2b_batched_nms(const d2b_batched_nms_params* p, void* workspace, size_t workspace_bytes,
                               d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_segments >= 0 && p->n >= 0 && p->max_output_size >= 0, "batched_nms: negative sizes");
  if (p->num_segments == 0) return D2B_OK;
  D2B_REQUIRE(p->keep && p->num_keep, "batched_nms: keep/num_keep must be non-NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int S = p->num_segments, n = p->n, mo = p->max_output_size;
  if (n == 0 || mo == 0) return nms_sorted(nullptr, nullptr, S, n, mo, p->iou_threshold, p->keep, p->num_keep, nullptr, st);
  D2B_REQUIRE(p->boxes && p->scores, "batched_nms: boxes/scores must be non-NULL");
  const int size_rc = nms_check_sizes(n, mo);  // before the ordering launches below
  if (size_rc != D2B_OK) return size_rc;
  if (nms_small_applies(n))  // the latency regime: the whole chain in one launch, no workspace
    return nms_small(p->boxes, p->scores, p->counts, S, n, mo, p->iou_threshold, p->keep, p->num_keep, st);
  if (workspace == nullptr || workspace_bytes < d2b_batched_nms_workspace_bytes(p)) {
    set_last_error("batched_nms needs %zu workspace bytes", d2b_batched_nms_workspace_bytes(p));
    return D2B_EWORKSPACE;
  }
  const int P = nms_pad(n);
  Workspace w(workspace);
  unsigned long long* keys = w.take<unsigned long long>((size_t)S * P);
  int32_t* live = w.take<int32_t>(S);
  float4* sorted = w.take<float4>((size_t)S * n);
  void* nms_ws = w.base + w.off;
  D2B_CUDA(cudaMemsetAsync(live, 0, sizeof(int32_t) * S, st));
  nms_prep_kernel<<<dim3((P + 255) / 256, S), 256, 0, st>>>(p->scores, p->counts, n, P, keys, live);
  D2B_LAUNCH_CHECK();
  int rc = sort_segments_desc(keys, S, P, nullptr, st);
  if (rc != D2B_OK) return rc;
  nms_gather_kernel<<<dim3((n + 255) / 256, S), 256, 0, st>>>(reinterpret_cast<const float4*>(p->boxes), keys, live,
                                                                n, P, sorted);
  D2B_LAUNCH_CHECK();
  rc = nms_sorted(reinterpret_cast<const float*>(sorted), live, S, n, mo, p->iou_threshold, p->keep, p->num_keep,
                  nms_ws, st);
  if (rc != D2B_OK) return rc;
  nms_unmap_kernel<<<dim3((mo + 255) / 256, S), 256, 0, st>>>(keys, P, mo, p->num_keep, p->keep);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}
