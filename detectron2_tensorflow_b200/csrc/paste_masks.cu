// paste_masks.cu -- mask paste-back (SURVEY.md 8f "next" #1):
//   reframe_box_masks_to_image_masks   lib/structures/mask_ops.py:7-56
//   (called by detector_postprocess    lib/modeling/postprocessing.py:9-59)
// The reference crops every box mask to the FULL image with tf.image.crop_and_resize on inverted boxes,
// materialising [M, H, W, 1] fp32 (430 MB per 100 detections at 800x1344), then thresholds to uint8.
// Here the bilinear sample and the threshold are fused and only the uint8 plane is written: the op is
// bound by that write (1 B/pixel).  Pixels outside the box are zeros by the extrapolation rule, so the
// planes are zero-filled by a memset, and paste_boxes_kernel then visits only a conservative bounding
// rectangle of each box -- the index range the inverse of the affine crop_and_resize map gives, widened
// by 2 -- and applies the exact per-pixel rule there, storing the ones.  A one-pass kernel that computed
// every pixel wrote 2.3-2.5 TB/s on a B200 against 7.3 TB/s for the memset.
// With out_rle_offsets the same rule (paste_row / paste_on) feeds the COCO run-length encoder of mask_rle.cuh over
// the same rectangles, and the planes are written only when `out` is given too.  The batched mode (num_images > 0)
// encodes the dense [N, R] detection slots of a whole batch, each image at its own output size, in the same three
// launches.
#include "kernels.cuh"
#include "mask_rle.cuh"

namespace d2b {
namespace {

constexpr int kPasteThreads = 256;
constexpr int kMaxMaskSmem = 16384;  // floats

struct PasteArgs {
  const float* masks;  // [M, mh, mw]
  const float* boxes;  // [M, 4] absolute yxyx in output-image pixels
  int mh, mw, H, W;
  float thr;
  uint8_t* out;  // [M, H, W]
  int smem_mask;
};

struct Axis {  // tf.image.crop_and_resize coordinate rule along one axis
  float n1, step, mid;
  int crop, dim;
  __device__ __forceinline__ float at(int i) const { return crop > 1 ? n1 * (float)(dim - 1) + (float)i * step : mid; }
};
__device__ __forceinline__ Axis make_axis(float lo, float hi, int crop, int dim) {
  Axis a;
  a.crop = crop; a.dim = dim;
  // reverse box: ([0,1] - min) / (max - min)   mask_ops.py:44-49
  const float n1 = (0.0f - lo) / (hi - lo);
  const float n2 = (1.0f - lo) / (hi - lo);
  a.n1 = n1;
  a.step = crop > 1 ? (n2 - n1) * (float)(dim - 1) / (float)(crop - 1) : 0.0f;
  a.mid = 0.5f * (n1 + n2) * (float)(dim - 1);
  return a;
}

#ifndef D2B_PASTE_RECT_CTAS
#define D2B_PASTE_RECT_CTAS 8  // A/B at 1,600 masks: 32 -> 0.515 ms, 16 -> 0.452, 8 -> 0.431, 4 -> 0.441, 2 -> 0.476
#endif
constexpr int kRectCtas = D2B_PASTE_RECT_CTAS;  // CTAs per mask: rows y0 + blockIdx.x, + kRectCtas, ...

// index range [lo, hi] of the output axis (n samples) whose input coordinate can fall inside [0, max_in]
__device__ __forceinline__ void axis_range(const Axis& ax, int n, float max_in, int& lo, int& hi) {
  lo = 0; hi = n - 1;
  if (ax.crop <= 1) return;
  const float c = ax.n1 * (float)(ax.dim - 1), st = ax.step;
  if (!(st > 0.0f) && !(st < 0.0f)) return;                  // 0 or NaN: every index has the same / no coordinate
  if (!(fabsf(c) < 1e30f) || !(fabsf(st) < 1e30f)) return;   // inf / NaN: leave it to the exact per-pixel rule
  float a = (0.0f - c) / st, b = (max_in - c) / st;
  if (a > b) { const float t = a; a = b; b = t; }
  a = fminf(fmaxf(a, -4.0f), (float)n + 4.0f);
  b = fminf(fmaxf(b, -4.0f), (float)n + 4.0f);
  lo = max(0, (int)floorf(a) - 2);
  hi = min(n - 1, (int)ceilf(b) + 2);
}

// Mask m's sampling axes and the rectangle [y0, y1] x [x0, x1] outside which every pasted pixel is 0.
struct PasteBox {
  Axis ay, ax;
  float ymax_in, xmax_in;
  int y0, y1, x0, x1;
};
// Box bx (yxyx in output-image pixels) of an H x W output image.
__device__ __forceinline__ PasteBox paste_box_at(const float4 bx, int H, int W, int mh, int mw) {
  PasteBox g;
  // to_normalized_coordinates: scale by 1/height, 1/width (box_list_ops.py:829-839)
  const float ys = 1.0f / (float)H, xs = 1.0f / (float)W;
  g.ay = make_axis(ys * bx.x, ys * bx.z, H, mh);
  g.ax = make_axis(xs * bx.y, xs * bx.w, W, mw);
  g.ymax_in = (float)(mh - 1); g.xmax_in = (float)(mw - 1);
  axis_range(g.ay, H, g.ymax_in, g.y0, g.y1);
  axis_range(g.ax, W, g.xmax_in, g.x0, g.x1);
  return g;
}
__device__ __forceinline__ PasteBox paste_box(const PasteArgs& a, long long m) {
  return paste_box_at(__ldg(reinterpret_cast<const float4*>(a.boxes) + m), a.H, a.W, a.mh, a.mw);
}

// The per-pixel rule, split at the row so the plane kernel hoists the row part out of its column loop.
struct PasteRow {
  int top, bot;
  float ly;
};
// false: row y samples outside the box mask (extrapolation value 0)
__device__ __forceinline__ bool paste_row(const PasteBox& g, int y, PasteRow& r) {
  const float in_y = g.ay.at(y);
  if (!(in_y >= 0.0f && in_y <= g.ymax_in)) return false;
  const float fy = floorf(in_y);
  r.top = (int)fy; r.bot = (int)ceilf(in_y);
  r.ly = in_y - fy;
  return true;
}
__device__ __forceinline__ bool paste_on(const float* mk, int mw, float thr, const PasteBox& g, const PasteRow& r, int x) {
  const float in_x = g.ax.at(x);
  if (!(in_x >= 0.0f && in_x <= g.xmax_in)) return false;
  const float f = floorf(in_x);
  const int left = (int)f, right = (int)ceilf(in_x);
  const float lx = in_x - f;
  const float tl = mk[r.top * mw + left], tr = mk[r.top * mw + right];
  const float bl = mk[r.bot * mw + left], br = mk[r.bot * mw + right];
  float t = tr - tl; t = t * lx; t = tl + t;
  float bb = br - bl; bb = bb * lx; bb = bl + bb;
  float v = bb - t; v = v * r.ly; v = t + v;
  return v > thr;
}

__device__ __forceinline__ const float* stage_mask(const PasteArgs& a, long long m, float* s_mask, int nthreads) {
  const float* mk = a.masks + (size_t)m * a.mh * a.mw;
  if (!a.smem_mask) return mk;
  for (int i = threadIdx.x; i < a.mh * a.mw; i += nthreads) s_mask[i] = __ldg(mk + i);
  __syncthreads();
  return s_mask;
}

__global__ void __launch_bounds__(kPasteThreads) paste_boxes_kernel(PasteArgs a) {
  extern __shared__ float s_mask[];
  const long long m = blockIdx.y;
  const PasteBox g = paste_box(a, m);
  if (g.y0 + (int)blockIdx.x > g.y1 || g.x0 > g.x1) return;  // block-uniform
  const float* mk = stage_mask(a, m, s_mask, kPasteThreads);
  uint8_t* o = a.out + (size_t)m * ((size_t)a.H * a.W);
  for (int y = g.y0 + (int)blockIdx.x; y <= g.y1; y += kRectCtas) {
    PasteRow r;
    if (!paste_row(g, y, r)) continue;
    for (int x = g.x0 + (int)threadIdx.x; x <= g.x1; x += kPasteThreads)
      if (paste_on(mk, a.mw, a.thr, g, r, x)) o[(size_t)y * a.W + x] = 1;
  }
}

struct PastePixel {
  const float* mk;
  int mw, y0, y1;
  float thr;
  PasteBox g;
  __device__ __forceinline__ bool operator()(int y, int x) const {  // x is inside [g.x0, g.x1]
    PasteRow r;
    return y >= y0 && y <= y1 && paste_row(g, y, r) && paste_on(mk, mw, thr, g, r, x);
  }
};

// Per-image geometry of the batched mode (d2b_paste_masks_params.num_images > 0): mask m is slot m % R of image m / R.
struct PasteBatch {
  const int32_t* out_shapes;  // [N, 2] (h, w)
  const int32_t* in_shapes;   // [N, 2] (h, w) or NULL: boxes as they are
  const uint8_t* valid;       // [N * R] or NULL
  int R;
};

constexpr long long kMaxPlane = (1ll << 31) - 65536;  // H * W below this keeps every column-major position an int

// Mask m's output size and pasting box in the batched mode; false: the slot encodes as an empty string.
__device__ __forceinline__ bool batch_slot(const PasteArgs& a, const PasteBatch& bt, long long m, int& H, int& W,
                                           float4& bx) {
  const long long n = m / bt.R;
  H = __ldg(bt.out_shapes + 2 * n);
  W = __ldg(bt.out_shapes + 2 * n + 1);
  if (!(H >= 1 && W >= 1 && (long long)H * W < kMaxPlane)) return false;
  if (bt.valid && !__ldg(bt.valid + m)) return false;
  bx = __ldg(reinterpret_cast<const float4*>(a.boxes) + m);
  if (bt.in_shapes) {  // postprocessing.py:36-43: scales = float32(float64(out) / float64(image_shape)), then boxes * scales
    const float sy = __double2float_rn(__ddiv_rn((double)H, (double)__ldg(bt.in_shapes + 2 * n)));
    const float sx = __double2float_rn(__ddiv_rn((double)W, (double)__ldg(bt.in_shapes + 2 * n + 1)));
    bx.x = __fmul_rn(sy, bx.x); bx.y = __fmul_rn(sx, bx.y);
    bx.z = __fmul_rn(sy, bx.z); bx.w = __fmul_rn(sx, bx.w);
  }
  return true;
}

// One CTA per mask: count pass (kWrite = false) or write pass over the rectangle of paste_boxes_kernel.  kBatched takes
// the output size, the box scale and the validity from the mask's image (PasteBatch) instead of from PasteArgs.
template <bool kWrite, bool kBatched>
__global__ void __launch_bounds__(kRleThreads) paste_rle_kernel(PasteArgs a, RleOut o, PasteBatch bt) {
  extern __shared__ float s_mask[];
  __shared__ RleShared sh;
  const long long m = blockIdx.x;
  int H = a.H, W = a.W;
  float4 bx;
  if (kBatched && !batch_slot(a, bt, m, H, W, bx)) {  // block-uniform: an empty string
    if (!kWrite && threadIdx.x == 0) o.offsets[m + 1] = 0;
    return;
  }
  long long beg = 0, end = 0;
  if (kWrite) {
    beg = o.offsets[m]; end = o.offsets[m + 1];
    if (end > o.capacity) return;  // block-uniform: this string does not fit
  }
  const PasteBox g = kBatched ? paste_box_at(bx, H, W, a.mh, a.mw) : paste_box(a, m);
  PastePixel px;
  px.mk = stage_mask(a, m, s_mask, kRleThreads);
  px.mw = a.mw; px.y0 = g.y0; px.y1 = g.y1; px.thr = a.thr; px.g = g;
  rle_encode_mask<kWrite>(px, rle_walk_of(H, W, g.y0, g.y1, g.x0, g.x1), sh, o.offsets + m + 1, o.chars + beg,
                          end - beg);
}

template <bool kBatched>
int paste_rle(const PasteArgs& a, const RleOut& o, const PasteBatch& bt, long long num_masks, size_t smem,
              cudaStream_t st) {
  D2B_CUDA(allow_dynamic_smem(paste_rle_kernel<false, kBatched>, smem));
  D2B_CUDA(allow_dynamic_smem(paste_rle_kernel<true, kBatched>, smem));
  paste_rle_kernel<false, kBatched><<<(unsigned)num_masks, kRleThreads, smem, st>>>(a, o, bt);
  D2B_LAUNCH_CHECK();
  rle_offsets_kernel<<<1, kRleThreads, 0, st>>>(o.offsets, num_masks);
  D2B_LAUNCH_CHECK();
  paste_rle_kernel<true, kBatched><<<(unsigned)num_masks, kRleThreads, smem, st>>>(a, o, bt);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}

}  // namespace
}  // namespace d2b

using namespace d2b;

// The RLE byte lengths are staged in out_rle_offsets itself: no workspace either way.
extern "C" size_t d2b_paste_masks_workspace_bytes(const d2b_paste_masks_params*) { return 0; }

extern "C" int d2b_paste_masks(const d2b_paste_masks_params* p, void*, size_t, d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_masks >= 0 && p->num_masks <= 65535ll * 16, "paste_masks: num_masks=%lld out of range",
              (long long)p->num_masks);
  const bool batched = p->num_images > 0;
  if (batched) {  // every image's size lives in device memory: the kernels check it per mask
    D2B_REQUIRE(p->dets_per_image >= 0 && (long long)p->num_images * p->dets_per_image == p->num_masks,
                "paste_masks: num_masks=%lld is not num_images=%d x dets_per_image=%d", (long long)p->num_masks,
                (int)p->num_images, (int)p->dets_per_image);
    D2B_REQUIRE(p->out == nullptr && p->out_rle_offsets != nullptr,
                "paste_masks: the batched mode (num_images > 0) writes RLE only: out must be NULL, out_rle_offsets set");
    D2B_REQUIRE(p->output_shapes != nullptr, "paste_masks: num_images > 0 with output_shapes NULL");
    D2B_REQUIRE(p->mask_h >= 1 && p->mask_w >= 1, "paste_masks: bad sizes");
  } else {
    D2B_REQUIRE(p->num_images == 0 && p->dets_per_image == 0 && !p->output_shapes && !p->input_shapes && !p->valid,
                "paste_masks: num_images=%d: the batched fields need num_images > 0", (int)p->num_images);
    D2B_REQUIRE(p->mask_h >= 1 && p->mask_w >= 1 && p->image_h >= 1 && p->image_w >= 1, "paste_masks: bad sizes");
    D2B_REQUIRE((long long)p->image_h * p->image_w < kMaxPlane, "paste_masks: image too large");
  }
  const bool rle = p->out_rle_offsets != nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rle) {
    const int rc = rle_check("paste_masks", p->out_rle, p->rle_capacity);
    if (rc != D2B_OK) return rc;
  }
  if (p->num_masks == 0) {  // mask_ops.py:25-28: zeros [0, H, W]
    if (rle) D2B_CUDA(cudaMemsetAsync(p->out_rle_offsets, 0, sizeof(int64_t), st));
    return D2B_OK;
  }
  D2B_REQUIRE(p->box_masks && p->boxes && (p->out || rle), "paste_masks: NULL pointer");
  PasteArgs a;
  a.masks = p->box_masks; a.boxes = p->boxes; a.mh = p->mask_h; a.mw = p->mask_w;
  a.H = p->image_h; a.W = p->image_w; a.thr = p->mask_threshold;
  const long long plane = (long long)a.H * a.W;
  a.smem_mask = (a.mh * a.mw <= kMaxMaskSmem);
  const size_t smem = a.smem_mask ? sizeof(float) * a.mh * a.mw : 0;
  if (p->out) {
    D2B_CUDA(cudaMemsetAsync(p->out, 0, (size_t)p->num_masks * (size_t)plane, st));
    if (smem > 48 * 1024)
      D2B_CUDA(cudaFuncSetAttribute(paste_boxes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (long long m0 = 0; m0 < p->num_masks; m0 += 65535) {  // grid.y limit
      const long long cnt = p->num_masks - m0 < 65535 ? p->num_masks - m0 : 65535;
      PasteArgs c = a;
      c.masks = p->box_masks + (size_t)m0 * a.mh * a.mw;
      c.boxes = p->boxes + 4 * m0;
      c.out = p->out + (size_t)m0 * plane;
      paste_boxes_kernel<<<dim3(kRectCtas, (unsigned)cnt), kPasteThreads, smem, st>>>(c);
      D2B_LAUNCH_CHECK();
    }
  }
  if (rle) {
    RleOut o;
    o.chars = p->out_rle; o.offsets = p->out_rle_offsets; o.capacity = p->rle_capacity;
    a.out = nullptr;
    PasteBatch bt;
    bt.out_shapes = p->output_shapes; bt.in_shapes = p->input_shapes; bt.valid = p->valid; bt.R = p->dets_per_image;
    return batched ? paste_rle<true>(a, o, bt, p->num_masks, smem, st)
                   : paste_rle<false>(a, o, bt, p->num_masks, smem, st);
  }
  return D2B_OK;
}

// ------------------------------------------------------------------ mask_rcnn_inference (mask_head.py:71-103)
//   pred_mask_logits [M, Hm, Wm, C] (NHWC) -> transpose to NCHW -> gather_nd([m, pred_classes[m]]) -> sigmoid
// The reference transposes the whole tensor (C = 80: 400 MB at 1,600 masks of 28x28) to pick one channel per mask;
// here a thread reads exactly the element it needs (one 32-byte sector per pixel) and applies the bit-exact sigmoid.
namespace d2b {
namespace {
__global__ void mask_select_kernel(const float* logits, const long long* classes, long long total, int hw, int C,
                                   float* out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const long long m = t / hw;
  long long c = C == 1 ? 0 : classes[m];
  float v = 0.0f;  // tf.gather_nd on the GPU returns 0 for an out-of-range index
  if (c >= 0 && c < C) v = __ldg(logits + t * C + c);
  out[t] = d2b_sigmoidf(v);
}
}  // namespace
}  // namespace d2b

extern "C" size_t d2b_mask_rcnn_inference_workspace_bytes(const d2b_mask_rcnn_inference_params*) { return 0; }
extern "C" int d2b_mask_rcnn_inference(const d2b_mask_rcnn_inference_params* p, void*, size_t, d2b_stream_t stream) {
  D2B_REQUIRE(p != nullptr, "params is NULL");
  D2B_REQUIRE(p->num_masks >= 0 && p->mask_h >= 0 && p->mask_w >= 0 && p->num_classes >= 1, "mask_rcnn_inference: bad sizes");
  const long long total = (long long)p->num_masks * p->mask_h * p->mask_w;
  if (total == 0) return D2B_OK;
  D2B_REQUIRE(p->mask_logits && p->out && (p->num_classes == 1 || p->pred_classes), "mask_rcnn_inference: NULL pointer");
  D2B_REQUIRE(total < (1ll << 31) * 256, "mask_rcnn_inference: too many elements");
  d2b::mask_select_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p->mask_logits, reinterpret_cast<const long long*>(p->pred_classes), total, p->mask_h * p->mask_w, p->num_classes, p->out);
  D2B_LAUNCH_CHECK();
  return D2B_OK;
}
