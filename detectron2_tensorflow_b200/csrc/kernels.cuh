// kernels.cuh -- internal (non-ABI) interfaces shared by the pipeline translation units.
#pragma once
#include "common.cuh"

namespace d2b {

// ---------------------------------------------------------------- segmented top-k (topk.cu)
// Row r = image * G + g;  row pointer = scores[g] + image * row_len[g].
struct TopkDesc {
  const float* scores[D2B_MAX_LEVELS];
  long long row_len[D2B_MAX_LEVELS];
  int k_limit[D2B_MAX_LEVELS];  // 0 => no extra cap
  int G;
  int rows_per_group;
  int k;
  int transform;  // D2B_TOPK_*
};
constexpr int kTopkMaxK = 16384;
size_t topk_workspace_bytes(const TopkDesc& d);
// Writes, per row, the k_r winners sorted (value desc, index asc):
//   out_keys [rows, P] u64 composites (key32<<32 | ~index), zero padded, P = topk_padded_k(k)
//   optional out_values/out_indices [rows, k] (-1 / 0 padded), out_counts [rows] (always written)
int topk_run(const TopkDesc& d, unsigned long long* out_keys, float* out_values, int32_t* out_indices,
             int32_t* out_counts, void* ws, cudaStream_t st);
int topk_padded_k(int k);

// ---------------------------------------------------------------- segment sort (sort.cu)
// Sort each of S segments of P (power of two) u64 keys in DESCENDING order in place.
// seg_len (optional, device [S]): only the first seg_len[s] entries are live; the rest are
// overwritten with 0 before sorting (0 sorts last).
// skip (optional, device [S]): segments with skip[s] != 0 are left untouched.
int sort_segments_desc(unsigned long long* keys, int S, int P, const int32_t* seg_len, cudaStream_t st,
                       const int32_t* skip = nullptr);

// ---------------------------------------------------------------- NMS (nms.cu)
// Boxes of every segment are already in candidate order (score desc, index asc).
// boxes [S, n, 4]; counts [S] (device, live prefix per segment; NULL => n).
// keep [S, max_out] positions into the segment (selection order, -1 padded), num_keep [S].
size_t nms_sorted_workspace_bytes(int S, int n, int max_out);
// sweep = false (bitmask formulation only, see nms_uses_bitmask): only the suppression mask is built in `ws`
// ([S][64 W][W] u64, W = ceil(n / 64)); the caller sweeps it itself (rpn_fused.cu fuses the sweep with the merge).
// skip (device, optional, mask-only calls): no mask is built for segment s when skip[s / skip_group] != 0.
int nms_sorted(const float* boxes, const int32_t* counts, int S, int n, int max_out, float thr, int32_t* keep,
               int32_t* num_keep, void* ws, cudaStream_t st, bool sweep = true, const int32_t* skip = nullptr,
               int skip_group = 1);
bool nms_uses_bitmask(int n, int max_out);
bool nms_lazy_applies(int n, int max_out);  // the capped lazy sweep would be chosen (cap << n)
// D2B_OK when nms_sorted accepts (n, max_out), else D2B_EINVAL with the last error set; callers that launch work of
// their own before nms_sorted check it first, so that a rejected call launches nothing.
int nms_check_sizes(int n, int max_out);
// Small segments with UNSORTED scores (n <= 512): order, mask, sweep and index un-mapping in ONE launch, one CTA per
// segment; keep holds input indices (selection order, -1 padded).  No workspace.
bool nms_small_applies(int n);
int nms_small(const float* boxes, const float* scores, const int32_t* counts, int S, int n, int max_out, float thr,
              int32_t* keep, int32_t* num_keep, cudaStream_t st);

// ---------------------------------------------------------------- SOLOv2 dynamic conv (solo_dynconv.cu)
size_t solo_dynamic_masks_ws(int batch, int n, int channels);

}  // namespace d2b
