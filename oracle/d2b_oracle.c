/*
 * d2b_oracle.c -- CPU ORACLE for the detection post-backbone hot path.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, bench.py's
 * cpu_baseline / --impl reference legs and __graft_entry__.smoke() may load it.
 * The product (detectron2_tensorflow_b200/) never imports, links or calls it.
 *
 * It restates, in plain C, the algorithm of the reference
 * (SimeonZhang/detectron2_tensorflow, paths relative to the reference root) and
 * of the stock TensorFlow 1.x CPU kernels the reference calls
 * (tensorflow>=1.13.1, requirements.txt:42 -- un-vendored, absent from the
 * reference tree; their published semantics are restated here, see SURVEY.md
 * Appendix A).  Every function cites the reference file:line it follows.
 *
 * PARITY STATUS: pinned on the reference's own Python for the COMPOSITION, "parity unpinned" for the
 * arithmetic inside the stock TF kernels.  The reference has no tests/golden vectors and TensorFlow is not
 * installable here, but its post-backbone modules are plain Python over ~90 TF ops: they are executed
 * UNMODIFIED on a numpy stand-in for that API slice (tests/golden/tf_numpy_shim.py) and their outputs are
 * committed as tests/golden/reference_python.npz (generator: tests/golden/make_reference_golden.py;
 * checked by tests/test_reference_python_golden.py).  That pins operation order, tie rules, padding, class
 * offsets, level routing and label stitching of ROIPooler / ROIAlign / crop_and_resize, find_top_rpn_proposals,
 * fast_rcnn_inference, RetinaNet / YOLOv4 / SOLOv2 inference, pairwise_iou, Matcher, _get_ground_truth,
 * mask paste-back, point_nms and the anchor generator.  The kernels of CropAndResize, NonMaxSuppression,
 * TopKV2 and AvgPool are restated there a second time, in numpy, independently of this file -- not run
 * from TensorFlow itself.  Further pins: (a) the reference's own TF-free numpy NMS
 * (lib/structures/np_box_list_ops.py:146-216), (b) torchvision.ops.roi_align/nms (+ autograd for the
 * backward) and torch.topk as independent implementations; vectors under tests/golden/.
 *
 * The oracle deliberately keeps the reference's DATA MOVEMENT (SYMMETRIC pad
 * copy, per-level gather, concat + inverse-permutation gather, decode of all
 * anchors before top-k) because it doubles as the timed CPU baseline.
 *
 * Arithmetic policy: fp32, one rounding per written operation, no FMA
 * contraction (compile with -ffp-contract=off).  exp/log follow the Cephes
 * single-precision algorithms that Eigen's packet math (TF's CPU backend)
 * uses, with separate multiply and add (TF 1.x wheels are AVX-only, no FMA).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------ threads */
static int g_threads = 0; /* 0 = OpenMP default */
ORC_API void orc_set_num_threads(int n) { g_threads = n; }
ORC_API int orc_get_max_threads(void) {
#ifdef _OPENMP
  return g_threads > 0 ? g_threads : omp_get_max_threads();
#else
  return 1;
#endif
}
#ifdef _OPENMP
#define ORC_NT (g_threads > 0 ? g_threads : omp_get_max_threads())
#else
#define ORC_NT 1
#endif

/* ------------------------------------------------------------------ math */
static inline float bits2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f2bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

/* Cephes expf as vectorised by Eigen (pexp<Packet4f>): clamp, n = floor(x*log2e+0.5),
 * two-step Cody-Waite reduction, degree-5 polynomial, scale by 2^n, max with x. */
ORC_API float orc_expf(float x0) {
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
  int32_t n = (int32_t)fx;
  float p2n = bits2f((uint32_t)(n + 0x7f) << 23);
  y = y * p2n;
  return fmaxf(y, x0);
}

/* Cephes logf as vectorised by Eigen (plog<Packet4f>). */
ORC_API float orc_logf(float x0) {
  if (x0 != x0) return x0;
  if (x0 < 0.0f) return bits2f(0x7fc00000u);
  if (x0 == 0.0f) return -INFINITY;
  if (isinf(x0)) return x0;
  float x = fmaxf(x0, bits2f(0x00800000u)); /* cut off denormals */
  uint32_t ux = f2bits(x);
  int32_t emm0 = (int32_t)(ux >> 23);
  ux = (ux & ~0x7f800000u) | 0x3f000000u; /* mantissa in [0.5,1) */
  x = bits2f(ux);
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
  y = 7.0376836292E-2f * x;  y = y + -1.1514610310E-1f;
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

/* tf.nn.sigmoid restated as 1/(1+exp(-x)) on the shared expf (SURVEY A.12). */
ORC_API float orc_sigmoidf(float x) {
  float e = orc_expf(-x);
  float d = 1.0f + e;
  return 1.0f / d;
}

/* ------------------------------------------------------------------ A.5 levels */
/* lib/modeling/poolers.py:37-49, area from lib/structures/box_list_ops.py:31-44 */
ORC_API void orc_assign_boxes_to_levels(const float* boxes, int64_t M, int min_level,
                                        int max_level, int canonical_box_size,
                                        int canonical_level, int64_t* out) {
  const float eps = (float)2.220446049250313e-16; /* sys.float_info.epsilon -> f32 */
  const float ln2 = (float)0.6931471805599453;    /* math.log(2) -> f32 */
  for (int64_t i = 0; i < M; ++i) {
    const float* b = boxes + 4 * i;
    float hh = b[2] - b[0];
    float ww = b[3] - b[1];
    float area = hh * ww;
    float s = sqrtf(area);
    float t = s / (float)canonical_box_size;
    t = t + eps;
    float v = orc_logf(t);
    v = v / ln2;
    v = (float)canonical_level + v;
    v = floorf(v);
    int64_t lvl;
    if (v != v) lvl = min_level;          /* NaN: defined as lowest level */
    else if (v <= (float)min_level) lvl = min_level;
    else if (v >= (float)max_level) lvl = max_level;
    else lvl = (int64_t)v;
    out[i] = lvl - min_level;
  }
}

/* ------------------------------------------------------------------ A.1 pad */
/* tf.pad(image, [[0,0],[1,1],[1,1],[0,0]], mode='SYMMETRIC')  lib/layers/functional.py:125 */
ORC_API void orc_symmetric_pad1(const float* img, int N, int H, int W, int C, float* out) {
  const int Hp = H + 2, Wp = W + 2;
#pragma omp parallel for collapse(2) num_threads(ORC_NT) schedule(static)
  for (int n = 0; n < N; ++n)
    for (int y = 0; y < Hp; ++y) {
      int sy = y - 1; if (sy < 0) sy = 0; if (sy > H - 1) sy = H - 1;
      const float* src = img + ((size_t)n * H + sy) * (size_t)W * C;
      float* dst = out + ((size_t)n * Hp + y) * (size_t)Wp * C;
      memcpy(dst, src, sizeof(float) * C);
      memcpy(dst + C, src, sizeof(float) * (size_t)W * C);
      memcpy(dst + (size_t)(W + 1) * C, src + (size_t)(W - 1) * C, sizeof(float) * C);
    }
}

/* ------------------------------------------------------------------ A.3 TF CropAndResize */
/* tf.image.crop_and_resize (bilinear, extrapolation_value=0), TF CPU kernel semantics,
 * called from lib/layers/functional.py:164-165.  Sharded over boxes like TF's Shard(). */
ORC_API void orc_tf_crop_and_resize(const float* image, int N, int H, int W, int C,
                                    const float* nboxes, const int32_t* box_ind, int64_t M,
                                    int ch, int cw, float* out) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 8)
  for (int64_t b = 0; b < M; ++b) {
    const float y1 = nboxes[4 * b + 0], x1 = nboxes[4 * b + 1];
    const float y2 = nboxes[4 * b + 2], x2 = nboxes[4 * b + 3];
    const int32_t bi = box_ind[b];
    float* ob = out + (size_t)b * ch * cw * C;
    if (bi < 0 || bi >= N) continue; /* TF skips the box (output left as allocated: zero here) */
    const float hs = (ch > 1) ? (y2 - y1) * (float)(H - 1) / (float)(ch - 1) : 0.0f;
    const float ws = (cw > 1) ? (x2 - x1) * (float)(W - 1) / (float)(cw - 1) : 0.0f;
    for (int y = 0; y < ch; ++y) {
      const float in_y = (ch > 1) ? y1 * (float)(H - 1) + (float)y * hs
                                  : 0.5f * (y1 + y2) * (float)(H - 1);
      float* orow = ob + (size_t)y * cw * C;
      if (!(in_y >= 0.0f && in_y <= (float)(H - 1))) { /* in_y<0 || in_y>H-1 (NaN -> garbage in TF; zero here) */
        memset(orow, 0, sizeof(float) * (size_t)cw * C);
        continue;
      }
      const int top = (int)floorf(in_y), bot = (int)ceilf(in_y);
      const float ly = in_y - (float)top;
      for (int x = 0; x < cw; ++x) {
        const float in_x = (cw > 1) ? x1 * (float)(W - 1) + (float)x * ws
                                    : 0.5f * (x1 + x2) * (float)(W - 1);
        float* o = orow + (size_t)x * C;
        if (!(in_x >= 0.0f && in_x <= (float)(W - 1))) {
          memset(o, 0, sizeof(float) * C);
          continue;
        }
        const int left = (int)floorf(in_x), right = (int)ceilf(in_x);
        const float lx = in_x - (float)left;
        const float* TL = image + (((size_t)bi * H + top) * W + left) * C;
        const float* TR = image + (((size_t)bi * H + top) * W + right) * C;
        const float* BL = image + (((size_t)bi * H + bot) * W + left) * C;
        const float* BR = image + (((size_t)bi * H + bot) * W + right) * C;
        for (int c = 0; c < C; ++c) {
          float t = TR[c] - TL[c]; t = t * lx; t = TL[c] + t;
          float bb = BR[c] - BL[c]; bb = bb * lx; bb = BL[c] + bb;
          float r = bb - t; r = r * ly; r = t + r;
          o[c] = r;
        }
      }
    }
  }
}

/* ------------------------------------------------------------------ A.2 crop_and_resize */
/* lib/layers/functional.py:100-166 */
ORC_API int orc_crop_and_resize(const float* image, int N, int H, int W, int C,
                                const float* boxes, const int32_t* box_ind, int64_t M,
                                int ch, int cw, int aligned, int pad_border, float* out) {
  const float* img = image;
  float* padded = NULL;
  int Hp = H, Wp = W;
  float shift = 0.0f;
  if (pad_border) { /* :123-126 */
    Hp = H + 2; Wp = W + 2;
    padded = (float*)malloc(sizeof(float) * (size_t)N * Hp * Wp * C);
    if (!padded) return -1;
    orc_symmetric_pad1(image, N, H, W, C, padded);
    img = padded;
    shift = 1.0f;
  }
  float* nb = (float*)malloc(sizeof(float) * 4 * (size_t)(M > 0 ? M : 1));
  for (int64_t i = 0; i < M; ++i) { /* transform_fpcoor_for_tf :128-160 */
    const float ymin = boxes[4 * i + 0] + shift, xmin = boxes[4 * i + 1] + shift;
    const float ymax = boxes[4 * i + 2] + shift, xmax = boxes[4 * i + 3] + shift;
    if (aligned) {
      float sph = (ymax - ymin) / (float)ch;
      float spw = (xmax - xmin) / (float)cw;
      float imh = (float)(Hp - 1), imw = (float)(Wp - 1);
      float ny = sph / 2.0f; ny = ymin + ny; ny = ny - 0.5f; ny = ny / imh;
      float nx = spw / 2.0f; nx = xmin + nx; nx = nx - 0.5f; nx = nx / imw;
      float nh = sph * (float)(ch - 1); nh = nh / imh;
      float nw = spw * (float)(cw - 1); nw = nw / imw;
      nb[4 * i + 0] = ny; nb[4 * i + 1] = nx;
      nb[4 * i + 2] = ny + nh; nb[4 * i + 3] = nx + nw;
    } else {
      nb[4 * i + 0] = ymin / (float)Hp; nb[4 * i + 1] = xmin / (float)Wp;
      nb[4 * i + 2] = ymax / (float)Hp; nb[4 * i + 3] = xmax / (float)Wp;
    }
  }
  memset(out, 0, sizeof(float) * (size_t)M * ch * cw * C);
  orc_tf_crop_and_resize(img, N, Hp, Wp, C, nb, box_ind, M, ch, cw, out);
  free(nb);
  free(padded);
  return 0;
}

/* ------------------------------------------------------------------ A.4 ROIAlign */
/* lib/layers/roi_align.py:45-66 (crop at output*sr, then slim.avg_pool2d k=s=sr 'SAME') */
ORC_API int orc_roi_align(const float* image, int N, int H, int W, int C, const float* boxes,
                          const int32_t* box_ind, int64_t M, int oh, int ow,
                          float spatial_scale, int sampling_ratio, int aligned, float* out) {
  int ch = oh, cw = ow;
  if (sampling_ratio > 0) { ch = oh * sampling_ratio; cw = ow * sampling_ratio; }
  float* sb = (float*)malloc(sizeof(float) * 4 * (size_t)(M > 0 ? M : 1));
  for (int64_t i = 0; i < 4 * M; ++i) sb[i] = boxes[i] * spatial_scale; /* :55 */
  int rc;
  if (sampling_ratio <= 0) {
    rc = orc_crop_and_resize(image, N, H, W, C, sb, box_ind, M, ch, cw, aligned, 1, out);
  } else {
    const int sr = sampling_ratio;
    float* big = (float*)malloc(sizeof(float) * (size_t)(M > 0 ? M : 1) * ch * cw * C);
    rc = orc_crop_and_resize(image, N, H, W, C, sb, box_ind, M, ch, cw, aligned, 1, big);
    const float cnt = (float)(sr * sr);
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
    for (int64_t b = 0; b < M; ++b)
      for (int y = 0; y < oh; ++y)
        for (int x = 0; x < ow; ++x) {
          float* o = out + (((size_t)b * oh + y) * ow + x) * C;
          for (int c = 0; c < C; ++c) {
            float acc = 0.0f;
            for (int dy = 0; dy < sr; ++dy)
              for (int dx = 0; dx < sr; ++dx)
                acc = acc + big[(((size_t)b * ch + (y * sr + dy)) * cw + (x * sr + dx)) * C + c];
            o[c] = acc / cnt;
          }
        }
    free(big);
  }
  free(sb);
  return rc;
}

/* ------------------------------------------------------------------ ROIPooler */
/* lib/modeling/poolers.py:134-180: assign levels; per level where/gather -> ROIAlign;
 * concat; invert_permutation; gather.  level_counts mirrors the
 * 'roi_align/num_roi_level_k' summaries (:173). */
ORC_API int orc_roi_pooler(const float* const* feats, const int* Hs, const int* Ws, int L, int N,
                           int C, const float* scales, const float* boxes,
                           const int64_t* batch_idx, int64_t M, int oh, int ow,
                           int sampling_ratio, int aligned, int canonical_box_size,
                           int canonical_level, float* out, int32_t* level_counts) {
  const size_t row = (size_t)oh * ow * C;
  if (L == 1) { /* :152-155 */
    int32_t* bi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M > 0 ? M : 1));
    for (int64_t i = 0; i < M; ++i) bi[i] = (int32_t)batch_idx[i];
    int rc = orc_roi_align(feats[0], N, Hs[0], Ws[0], C, boxes, bi, M, oh, ow, scales[0],
                           sampling_ratio, aligned, out);
    if (level_counts) level_counts[0] = (int32_t)M;
    free(bi);
    return rc;
  }
  /* min/max level from scales (:123-129) */
  const int min_level = (int)lroundf(-log2f(scales[0]));
  const int max_level = (int)lroundf(-log2f(scales[L - 1]));
  int64_t* lv = (int64_t*)malloc(sizeof(int64_t) * (size_t)(M > 0 ? M : 1));
  orc_assign_boxes_to_levels(boxes, M, min_level, max_level, canonical_box_size, canonical_level, lv);
  float* cat = (float*)malloc(sizeof(float) * (size_t)(M > 0 ? M : 1) * row);
  int32_t* out_inds = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M > 0 ? M : 1));
  float* lboxes = (float*)malloc(sizeof(float) * 4 * (size_t)(M > 0 ? M : 1));
  int32_t* lbi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M > 0 ? M : 1));
  int64_t pos = 0;
  int rc = 0;
  for (int l = 0; l < L; ++l) {
    int64_t m = 0;
    for (int64_t i = 0; i < M; ++i)
      if (lv[i] == l) { /* tf.where + gather :167-169 */
        memcpy(lboxes + 4 * m, boxes + 4 * i, 16);
        lbi[m] = (int32_t)batch_idx[i];
        out_inds[pos + m] = (int32_t)i;
        ++m;
      }
    if (level_counts) level_counts[l] = (int32_t)m;
    rc |= orc_roi_align(feats[l], N, Hs[l], Ws[l], C, lboxes, lbi, m, oh, ow, scales[l],
                        sampling_ratio, aligned, cat + (size_t)pos * row);
    pos += m;
  }
  /* invert_permutation + gather :177-178 */
  int32_t* inv = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M > 0 ? M : 1));
  for (int64_t p = 0; p < M; ++p) inv[out_inds[p]] = (int32_t)p;
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < M; ++i)
    memcpy(out + (size_t)i * row, cat + (size_t)inv[i] * row, sizeof(float) * row);
  free(inv); free(lbi); free(lboxes); free(out_inds); free(cat); free(lv);
  return rc;
}

/* ------------------------------------------------------------------ A.6 decode */
/* lib/modeling/box_regression.py:76-123 Box2BoxTransform.apply_deltas
 * deltas [n, k*4] (dy,dx,dh,dw), boxes [n,4] -> out [n, k*4] */
ORC_API void orc_apply_deltas(const float* deltas, const float* boxes, int64_t n, int k,
                              const float* weights, float scale_clamp, float* out) {
  const float wy = weights[0], wx = weights[1], wh = weights[2], ww = weights[3];
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n; ++i) {
    const float* b = boxes + 4 * i;
    const float heights = b[2] - b[0];
    const float widths = b[3] - b[1];
    float cy = 0.5f * heights; cy = b[0] + cy;
    float cx = 0.5f * widths;  cx = b[1] + cx;
    for (int j = 0; j < k; ++j) {
      const float* d = deltas + ((size_t)i * k + j) * 4;
      float dy = d[0] / wy, dx = d[1] / wx, dh = d[2] / wh, dw = d[3] / ww;
      dh = fminf(dh, scale_clamp);
      dw = fminf(dw, scale_clamp);
      float pcy = dy * heights; pcy = pcy + cy;
      float pcx = dx * widths;  pcx = pcx + cx;
      float ph = orc_expf(dh) * heights;
      float pw = orc_expf(dw) * widths;
      float hh = 0.5f * ph, hw = 0.5f * pw;
      float* o = out + ((size_t)i * k + j) * 4;
      o[0] = pcy - hh; o[1] = pcx - hw; o[2] = pcy + hh; o[3] = pcx + hw;
    }
  }
}

/* ------------------------------------------------------------------ A.8 top_k */
/* tf.nn.top_k: k largest, equal values -> lower index first; NaN ranks lowest. */
typedef struct { float v; int32_t i; } orc_vi;
static inline int vi_before(float av, int32_t ai, float bv, int32_t bi) {
  const int an = (av != av), bn = (bv != bv);
  if (an || bn) { if (an != bn) return bn; return ai < bi; }
  if (av > bv) return 1;
  if (av < bv) return 0;
  return ai < bi;
}
static int vi_cmp(const void* pa, const void* pb) {
  const orc_vi* a = (const orc_vi*)pa; const orc_vi* b = (const orc_vi*)pb;
  if (vi_before(a->v, a->i, b->v, b->i)) return -1;
  if (vi_before(b->v, b->i, a->v, a->i)) return 1;
  return 0;
}
/* heap-select: keep the k best in a heap whose root is the worst of them (what
 * TF's TopKV2 CPU kernel does for small k), then sort. */
static void sift_down(orc_vi* h, int64_t n, int64_t p) {
  for (;;) {
    int64_t c = 2 * p + 1;
    if (c >= n) return;
    /* root = worst: child "worse" means the other is before it */
    if (c + 1 < n && vi_before(h[c].v, h[c].i, h[c + 1].v, h[c + 1].i)) c = c + 1;
    if (vi_before(h[p].v, h[p].i, h[c].v, h[c].i)) { orc_vi t = h[p]; h[p] = h[c]; h[c] = t; p = c; }
    else return;
  }
}
ORC_API void orc_top_k(const float* x, int64_t n, int64_t k, float* vals, int32_t* idx) {
  if (k > n) k = n;
  if (k <= 0) return;
  orc_vi* h = (orc_vi*)malloc(sizeof(orc_vi) * (size_t)k);
  for (int64_t i = 0; i < k; ++i) { h[i].v = x[i]; h[i].i = (int32_t)i; }
  for (int64_t p = k / 2 - 1; p >= 0; --p) sift_down(h, k, p);
  for (int64_t i = k; i < n; ++i)
    if (vi_before(x[i], (int32_t)i, h[0].v, h[0].i)) { h[0].v = x[i]; h[0].i = (int32_t)i; sift_down(h, k, 0); }
  qsort(h, (size_t)k, sizeof(orc_vi), vi_cmp);
  for (int64_t i = 0; i < k; ++i) { vals[i] = h[i].v; idx[i] = h[i].i; }
  free(h);
}

/* ------------------------------------------------------------------ A.9 NMS */
/* tf.image.non_max_suppression (V3, CPU kernel), score_threshold = -inf */
static inline float orc_iou(const float* a, const float* b) {
  const float ymin_i = fminf(a[0], a[2]), xmin_i = fminf(a[1], a[3]);
  const float ymax_i = fmaxf(a[0], a[2]), xmax_i = fmaxf(a[1], a[3]);
  const float ymin_j = fminf(b[0], b[2]), xmin_j = fminf(b[1], b[3]);
  const float ymax_j = fmaxf(b[0], b[2]), xmax_j = fmaxf(b[1], b[3]);
  const float area_i = (ymax_i - ymin_i) * (xmax_i - xmin_i);
  const float area_j = (ymax_j - ymin_j) * (xmax_j - xmin_j);
  if (area_i <= 0.0f || area_j <= 0.0f) return 0.0f;
  const float iymin = fmaxf(ymin_i, ymin_j), ixmin = fmaxf(xmin_i, xmin_j);
  const float iymax = fminf(ymax_i, ymax_j), ixmax = fminf(xmax_i, xmax_j);
  const float ih = fmaxf(iymax - iymin, 0.0f), iw = fmaxf(ixmax - ixmin, 0.0f);
  const float inter = ih * iw;
  float u = area_i + area_j; u = u - inter;
  return inter / u;
}
ORC_API float orc_box_iou(const float* a, const float* b) { return orc_iou(a, b); }

ORC_API int32_t orc_nms(const float* boxes, const float* scores, int64_t n, int32_t max_out,
                        float iou_thr, int32_t* keep) {
  orc_vi* c = (orc_vi*)malloc(sizeof(orc_vi) * (size_t)(n > 0 ? n : 1));
  int64_t m = 0;
  for (int64_t i = 0; i < n; ++i)
    if (scores[i] > -INFINITY) { c[m].v = scores[i]; c[m].i = (int32_t)i; ++m; }
  qsort(c, (size_t)m, sizeof(orc_vi), vi_cmp); /* priority queue order: score desc, index asc */
  int32_t ns = 0;
  for (int64_t q = 0; q < m && ns < max_out; ++q) {
    const int32_t i = c[q].i;
    int ok = 1;
    for (int32_t j = ns - 1; j >= 0; --j) /* most recently selected first */
      if (orc_iou(boxes + 4 * (size_t)i, boxes + 4 * (size_t)keep[j]) > iou_thr) { ok = 0; break; }
    if (ok) keep[ns++] = i;
  }
  free(c);
  return ns;
}

/* lib/layers/nms.py:6-26 batch_nms (padded-output variant: keep [B,max_out] filled with -1) */
ORC_API void orc_batch_nms(const float* boxes, const float* scores, int B, int64_t n,
                           int32_t max_out, float iou_thr, int32_t* keep, int32_t* num_keep) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int b = 0; b < B; ++b) {
    int32_t* kb = keep + (size_t)b * max_out;
    int32_t* tmp = (int32_t*)malloc(sizeof(int32_t) * (size_t)(max_out > 0 ? max_out : 1));
    int32_t c = orc_nms(boxes + (size_t)b * n * 4, scores + (size_t)b * n, n, max_out, iou_thr, tmp);
    for (int32_t i = 0; i < max_out; ++i) kb[i] = i < c ? tmp[i] : -1;
    num_keep[b] = c;
    free(tmp);
  }
}

/* ------------------------------------------------------------------ A.7 clip / prune */
/* lib/structures/box_list_ops.py:131-137 */
static inline void clip_box(float* b, float h, float w) {
  b[0] = fmaxf(fminf(b[0], h), 0.0f);
  b[1] = fmaxf(fminf(b[1], w), 0.0f);
  b[2] = fmaxf(fminf(b[2], h), 0.0f);
  b[3] = fmaxf(fminf(b[3], w), 0.0f);
}

/* ------------------------------------------------------------------ A.10 RPN */
/* lib/modeling/proposal_generator/rpn_outputs.py:403-426 predict_proposals: decode ALL anchors */
ORC_API void orc_rpn_predict_proposals(const float* deltas, const float* anchors, int N,
                                       int64_t hwa, const float* weights, float scale_clamp,
                                       float* out) {
  for (int n = 0; n < N; ++n)
    orc_apply_deltas(deltas + (size_t)n * hwa * 4, anchors, hwa, 1, weights, scale_clamp,
                     out + (size_t)n * hwa * 4);
}

/* lib/modeling/proposal_generator/rpn_outputs.py:29-132 find_top_rpn_proposals */
ORC_API void orc_find_top_rpn_proposals(const float* const* proposals, const float* const* logits,
                                        const int64_t* hwa, int L, int N,
                                        const int32_t* image_shapes, float nms_thresh,
                                        int pre_nms_topk, int post_nms_topk,
                                        float min_box_side_len, float* out_boxes,
                                        float* out_logits, uint8_t* out_valid,
                                        int32_t* out_num_valid) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int n = 0; n < N; ++n) {
    const float h = (float)image_shapes[2 * n + 0], w = (float)image_shapes[2 * n + 1];
    const size_t cap = (size_t)L * (size_t)(post_nms_topk > 0 ? post_nms_topk : 1);
    float* cat_boxes = (float*)malloc(sizeof(float) * 4 * cap);
    float* cat_scores = (float*)malloc(sizeof(float) * cap);
    int64_t total = 0;
    for (int l = 0; l < L; ++l) {
      const int64_t len = hwa[l];
      int64_t k = pre_nms_topk < len ? pre_nms_topk : len; /* :67-68 */
      if (k < 0) k = 0;
      float* tv = (float*)malloc(sizeof(float) * (size_t)(k > 0 ? k : 1));
      int32_t* ti = (int32_t*)malloc(sizeof(int32_t) * (size_t)(k > 0 ? k : 1));
      orc_top_k(logits[l] + (size_t)n * len, len, k, tv, ti); /* :70 */
      float* bx = (float*)malloc(sizeof(float) * 4 * (size_t)(k > 0 ? k : 1));
      int64_t m = 0;
      for (int64_t j = 0; j < k; ++j) {
        float b[4];
        memcpy(b, proposals[l] + ((size_t)n * len + ti[j]) * 4, 16); /* gather :71 */
        clip_box(b, h, w);                                           /* :77-80 */
        if (min_box_side_len > 0.0f) {                               /* :83-87 */
          const float bh = b[2] - b[0], bw = b[3] - b[1];
          if (!(bw >= min_box_side_len && bh >= min_box_side_len)) continue;
        }
        memcpy(bx + 4 * m, b, 16);
        tv[m] = tv[j];
        ++m;
      }
      int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(post_nms_topk > 0 ? post_nms_topk : 1));
      const int32_t nk = orc_nms(bx, tv, m, post_nms_topk, nms_thresh, keep); /* :90-94 */
      for (int32_t q = 0; q < nk; ++q) { /* gather + concat :95-102 */
        memcpy(cat_boxes + 4 * (size_t)(total + q), bx + 4 * (size_t)keep[q], 16);
        cat_scores[total + q] = tv[keep[q]];
      }
      total += nk;
      free(keep); free(bx); free(ti); free(tv);
    }
    const int64_t kk = total < post_nms_topk ? total : post_nms_topk; /* :105 */
    float* fv = (float*)malloc(sizeof(float) * (size_t)(kk > 0 ? kk : 1));
    int32_t* fi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(kk > 0 ? kk : 1));
    orc_top_k(cat_scores, total, kk, fv, fi); /* :106 sorted=True */
    float* ob = out_boxes + (size_t)n * post_nms_topk * 4;
    float* ol = out_logits + (size_t)n * post_nms_topk;
    uint8_t* ov = out_valid + (size_t)n * post_nms_topk;
    for (int64_t j = 0; j < post_nms_topk; ++j) { /* pad :111-114 */
      if (j < kk) { memcpy(ob + 4 * j, cat_boxes + 4 * (size_t)fi[j], 16); ol[j] = fv[j]; ov[j] = 1; }
      else { ob[4 * j] = ob[4 * j + 1] = ob[4 * j + 2] = ob[4 * j + 3] = 0.0f; ol[j] = 0.0f; ov[j] = 0; }
    }
    if (out_num_valid) out_num_valid[n] = (int32_t)kk;
    free(fi); free(fv); free(cat_scores); free(cat_boxes);
  }
}

/* ------------------------------------------------------------------ A.11 Fast R-CNN */
/* lib/modeling/roi_heads/fast_rcnn.py:28-187 fast_rcnn_inference
 * boxes [M, Kb*4] (Kb = K class-specific, or 1 class-agnostic regression), scores [M, K+1],
 * indices [M,2] (image, slot) int64, dense shape [N, Rmax]. */
ORC_API void orc_fast_rcnn_inference(const float* boxes, const float* scores,
                                     const int64_t* indices, int64_t M, int N, int Rmax, int Kb,
                                     int K, const int32_t* image_shapes, float score_thresh,
                                     float nms_thresh, int topk_per_image, int nms_cls_agnostic,
                                     float* out_boxes, float* out_scores, int64_t* out_classes,
                                     uint8_t* out_valid, int32_t* out_roi, int32_t* out_num) {
  /* SparseBoxList.to_dense (lib/structures/box_list.py:204-246): zero-filled dense tensors */
  float* dboxes = (float*)calloc((size_t)N * Rmax * Kb * 4 + 1, sizeof(float));
  float* dscores = (float*)calloc((size_t)N * Rmax * K + 1, sizeof(float));
  for (int64_t i = 0; i < M; ++i) {
    const int64_t n = indices[2 * i], r = indices[2 * i + 1];
    if (n < 0 || n >= N || r < 0 || r >= Rmax) continue;
    memcpy(dboxes + ((size_t)n * Rmax + r) * Kb * 4, boxes + (size_t)i * Kb * 4, sizeof(float) * Kb * 4);
    memcpy(dscores + ((size_t)n * Rmax + r) * K, scores + (size_t)i * (K + 1), sizeof(float) * K); /* drop bg :66 */
  }
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int n = 0; n < N; ++n) {
    const float h = (float)image_shapes[2 * n], w = (float)image_shapes[2 * n + 1];
    float* bx = dboxes + (size_t)n * Rmax * Kb * 4;  /* [Rmax, Kb, 4] */
    const float* sc = dscores + (size_t)n * Rmax * K; /* [Rmax, K] */
    float max_coord = -INFINITY;
    for (int64_t i = 0; i < (int64_t)Rmax * Kb; ++i) { /* clip :109-116, reduce_max :141 */
      clip_box(bx + 4 * i, h, w);
      for (int c = 0; c < 4; ++c) max_coord = fmaxf(max_coord, bx[4 * i + c]);
    }
    /* scores > thresh on the transposed [K, R] tensor; tf.where => class-major order :119-128 */
    int64_t cnt = 0;
    for (int k = 0; k < K; ++k)
      for (int r = 0; r < Rmax; ++r)
        if (sc[(size_t)r * K + k] > score_thresh) ++cnt;
    float* fb = (float*)malloc(sizeof(float) * 4 * (size_t)(cnt > 0 ? cnt : 1));
    float* nb = (float*)malloc(sizeof(float) * 4 * (size_t)(cnt > 0 ? cnt : 1));
    float* fs = (float*)malloc(sizeof(float) * (size_t)(cnt > 0 ? cnt : 1));
    int32_t* fc = (int32_t*)malloc(sizeof(int32_t) * (size_t)(cnt > 0 ? cnt : 1));
    int32_t* fr = (int32_t*)malloc(sizeof(int32_t) * (size_t)(cnt > 0 ? cnt : 1));
    int64_t q = 0;
    const float mc1 = max_coord + 1.0f;
    for (int k = 0; k < K; ++k)
      for (int r = 0; r < Rmax; ++r)
        if (sc[(size_t)r * K + k] > score_thresh) {
          const float* b = bx + ((size_t)r * Kb + (Kb == 1 ? 0 : k)) * 4; /* :131-136 */
          memcpy(fb + 4 * q, b, 16);
          fs[q] = sc[(size_t)r * K + k];
          fc[q] = k; fr[q] = r;
          if (nms_cls_agnostic) memcpy(nb + 4 * q, b, 16);
          else { const float off = (float)k * mc1; /* :141-143 */
                 for (int c = 0; c < 4; ++c) nb[4 * q + c] = b[c] + off; }
          ++q;
        }
    int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(topk_per_image > 0 ? topk_per_image : 1));
    const int32_t nk = orc_nms(nb, fs, cnt, topk_per_image, nms_thresh, keep); /* :145-146 */
    for (int j = 0; j < topk_per_image; ++j) { /* gather + pad_or_clip :147-159 */
      float* ob = out_boxes + ((size_t)n * topk_per_image + j) * 4;
      const size_t o = (size_t)n * topk_per_image + j;
      if (j < nk) {
        memcpy(ob, fb + 4 * (size_t)keep[j], 16);
        out_scores[o] = fs[keep[j]]; out_classes[o] = fc[keep[j]]; out_valid[o] = 1;
        if (out_roi) out_roi[o] = fr[keep[j]];
      } else {
        ob[0] = ob[1] = ob[2] = ob[3] = 0.0f;
        out_scores[o] = 0.0f; out_classes[o] = 0; out_valid[o] = 0;
        if (out_roi) out_roi[o] = -1;
      }
    }
    if (out_num) out_num[n] = nk;
    free(keep); free(fr); free(fc); free(fs); free(nb); free(fb);
  }
  free(dscores); free(dboxes);
}

/* ------------------------------------------------------------------ A.12 RetinaNet */
/* lib/modeling/single_stage_heads/retinanet.py:285-387 RetinaNetHead.inference
 * box_cls[l] [N, HWA_l, K], box_delta[l] [N, HWA_l, 4], anchors[l] [HWA_l, 4] */
ORC_API void orc_retinanet_inference(const float* const* box_cls, const float* const* box_delta,
                                     const float* const* anchors, const int64_t* hwa, int L,
                                     int N, int K, int topk_candidates, float score_thresh,
                                     float nms_thresh, int max_det, const float* weights,
                                     float scale_clamp, float* out_boxes, float* out_scores,
                                     int32_t* out_classes, uint8_t* out_valid, int32_t* out_num) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int n = 0; n < N; ++n) {
    const size_t cap = (size_t)L * (size_t)(topk_candidates > 0 ? topk_candidates : 1);
    float* ab = (float*)malloc(sizeof(float) * 4 * cap);
    float* as = (float*)malloc(sizeof(float) * cap);
    int32_t* ac = (int32_t*)malloc(sizeof(int32_t) * cap);
    int64_t total = 0;
    for (int l = 0; l < L; ++l) {
      const int64_t len = hwa[l] * K;
      float* p = (float*)malloc(sizeof(float) * (size_t)(len > 0 ? len : 1));
      const float* x = box_cls[l] + (size_t)n * len;
      for (int64_t i = 0; i < len; ++i) p[i] = orc_sigmoidf(x[i]); /* :321-322 */
      int64_t k = topk_candidates < hwa[l] ? topk_candidates : hwa[l]; /* :325 (min with #anchors) */
      float* tv = (float*)malloc(sizeof(float) * (size_t)(k > 0 ? k : 1));
      int32_t* ti = (int32_t*)malloc(sizeof(int32_t) * (size_t)(k > 0 ? k : 1));
      orc_top_k(p, len, k, tv, ti); /* :326 */
      for (int64_t j = 0; j < k; ++j) {
        if (!(tv[j] > score_thresh)) continue; /* :329-331 */
        const int64_t a = ti[j] / K; const int32_t c = (int32_t)(ti[j] % K); /* :333-334 */
        orc_apply_deltas(box_delta[l] + ((size_t)n * hwa[l] + a) * 4, anchors[l] + (size_t)a * 4, 1, 1,
                         weights, scale_clamp, ab + 4 * (size_t)total); /* :336-339 */
        as[total] = tv[j]; ac[total] = c;
        ++total;
      }
      free(ti); free(tv); free(p);
    }
    float max_coord = -INFINITY; /* :349 */
    for (int64_t i = 0; i < 4 * total; ++i) max_coord = fmaxf(max_coord, ab[i]);
    const float mc1 = max_coord + 1.0f;
    float* nb = (float*)malloc(sizeof(float) * 4 * (size_t)(total > 0 ? total : 1));
    for (int64_t i = 0; i < total; ++i) { /* :350-351 */
      const float off = (float)ac[i] * mc1;
      for (int c = 0; c < 4; ++c) nb[4 * i + c] = ab[4 * i + c] + off;
    }
    int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(max_det > 0 ? max_det : 1));
    const int32_t nk = orc_nms(nb, as, total, max_det, nms_thresh, keep); /* :353-355 */
    for (int j = 0; j < max_det; ++j) { /* :356-367 */
      const size_t o = (size_t)n * max_det + j;
      float* ob = out_boxes + o * 4;
      if (j < nk) { memcpy(ob, ab + 4 * (size_t)keep[j], 16); out_scores[o] = as[keep[j]];
                    out_classes[o] = ac[keep[j]]; out_valid[o] = 1; }
      else { ob[0] = ob[1] = ob[2] = ob[3] = 0.0f; out_scores[o] = 0.0f; out_classes[o] = 0; out_valid[o] = 0; }
    }
    if (out_num) out_num[n] = nk;
    free(keep); free(nb); free(ac); free(as); free(ab);
  }
}

/* ------------------------------------------------------------------ A.13 matrix NMS */
/* lib/layers/nms.py:29-83 matrix_nms.  masks [n, HW] fp32; kernel 0=gaussian 1=linear.
 * The fp32 matmul (:50) is restated as a plain fp32 dot product (exact for 0/1 masks). */
ORC_API int orc_matrix_nms(const float* masks, const int64_t* classes, const float* scores,
                           const float* sum_masks_in, int n, int64_t hw, int kernel, float sigma,
                           float* out) {
  if (kernel != 0 && kernel != 1) return -1; /* NotImplementedError :77 */
  if (n <= 0) return 0;
  float* sum_masks = (float*)malloc(sizeof(float) * n);
  if (sum_masks_in) memcpy(sum_masks, sum_masks_in, sizeof(float) * n);
  else
    for (int i = 0; i < n; ++i) { /* reduce_sum :46 */
      float s = 0.0f;
      for (int64_t p = 0; p < hw; ++p) s = s + masks[(size_t)i * hw + p];
      sum_masks[i] = s;
    }
  float* iou = (float*)calloc((size_t)n * n, sizeof(float));
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int i = 0; i < n; ++i) {
    const float* mi = masks + (size_t)i * hw;
    for (int j = 0; j < n; ++j) {
      const float* mj = masks + (size_t)j * hw;
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      int64_t p = 0;
      for (; p + 8 <= hw; p += 8)
        for (int u = 0; u < 8; ++u) acc[u] += mi[p + u] * mj[p + u];
      float inter = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
      for (; p < hw; ++p) inter += mi[p] * mj[p];
      /* union[i][j] = sum[j] + sum[i] - inter :51-52 */
      float u = sum_masks[j] + sum_masks[i]; u = u - inter;
      float v = inter / u;                       /* :54 */
      if (j <= i) v = v - v;                     /* minus matrix_band_part(-1,0) :55 (NaN stays NaN) */
      const float cls = (classes[i] == classes[j]) ? 1.0f : 0.0f; /* :58-61 */
      iou[(size_t)i * n + j] = v * cls;          /* :64 */
    }
  }
  float* cmax = (float*)malloc(sizeof(float) * n);
  for (int j = 0; j < n; ++j) { /* reduce_max axis 0 :67 */
    float m = iou[j];
    for (int i = 1; i < n; ++i) { const float v = iou[(size_t)i * n + j]; m = (v > m) ? v : m; }
    cmax[j] = m;
  }
  const float nsig = (float)(-1.0 * (double)sigma);
  for (int j = 0; j < n; ++j) { /* decay + reduce_min axis 0 :72-79 */
    float m = INFINITY;
    for (int i = 0; i < n; ++i) {
      const float v = iou[(size_t)i * n + j];
      const float ci = cmax[i]; /* compensate_iou broadcast per ROW after the transpose :68-69 */
      float d;
      if (kernel == 0) { float a = v * v; float b = ci * ci; a = a - b; a = nsig * a; d = orc_expf(a); }
      else { float a = 1.0f - v; float b = 1.0f - ci; d = a / b; }
      m = (d < m) ? d : m;
    }
    out[j] = scores[j] * m; /* :82 */
  }
  free(cmax); free(iou); free(sum_masks);
  return 0;
}

/* ------------------------------------------------------------------ mask paste-back (SURVEY.md 8f "next" #1) */
/* lib/structures/mask_ops.py:7-56 reframe_box_masks_to_image_masks:
 *   boxes -> to_normalized_coordinates (box_list_ops.py:806-839: scale by 1/height, 1/width)
 *   reverse_boxes = ([0,0,1,1] - min_corner) / (max_corner - min_corner)           (:40-52)
 *   tf.image.crop_and_resize(box_masks[..., None], reverse_boxes, range(M), image_shape)  (:53-59)
 *   cast(image_masks > mask_threshold, uint8)                                        (:29-30)
 * box_masks [M, mh, mw] fp32, boxes [M,4] absolute yxyx, out [M, H, W] uint8. */
ORC_API void orc_reframe_box_masks(const float* box_masks, const float* boxes, int64_t M, int mh, int mw,
                                   int H, int W, float thr, uint8_t* out) {
  const float ys = 1.0f / (float)H, xs = 1.0f / (float)W;
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int64_t b = 0; b < M; ++b) {
    const float ymin = ys * boxes[4 * b + 0], xmin = xs * boxes[4 * b + 1];
    const float ymax = ys * boxes[4 * b + 2], xmax = xs * boxes[4 * b + 3];
    float nb[4];
    nb[0] = (0.0f - ymin) / (ymax - ymin);
    nb[1] = (0.0f - xmin) / (xmax - xmin);
    nb[2] = (1.0f - ymin) / (ymax - ymin);
    nb[3] = (1.0f - xmin) / (xmax - xmin);
    float* tmp = (float*)malloc(sizeof(float) * (size_t)H * W);
    memset(tmp, 0, sizeof(float) * (size_t)H * W); /* extrapolation_value = 0 */
    { /* tf.image.crop_and_resize of box b against its own mask (a [1, mh, mw, 1] image), crop = (H, W) */
      const float* image = box_masks + (size_t)b * mh * mw;
      const float y1 = nb[0], x1 = nb[1], y2 = nb[2], x2 = nb[3];
      const float hs = (H > 1) ? (y2 - y1) * (float)(mh - 1) / (float)(H - 1) : 0.0f;
      const float ws = (W > 1) ? (x2 - x1) * (float)(mw - 1) / (float)(W - 1) : 0.0f;
      for (int y = 0; y < H; ++y) {
        const float in_y = (H > 1) ? y1 * (float)(mh - 1) + (float)y * hs : 0.5f * (y1 + y2) * (float)(mh - 1);
        if (!(in_y >= 0.0f && in_y <= (float)(mh - 1))) continue;
        const int top = (int)floorf(in_y), bot = (int)ceilf(in_y);
        const float ly = in_y - (float)top;
        for (int x = 0; x < W; ++x) {
          const float in_x = (W > 1) ? x1 * (float)(mw - 1) + (float)x * ws : 0.5f * (x1 + x2) * (float)(mw - 1);
          if (!(in_x >= 0.0f && in_x <= (float)(mw - 1))) continue;
          const int left = (int)floorf(in_x), right = (int)ceilf(in_x);
          const float lx = in_x - (float)left;
          const float tl = image[top * mw + left], tr = image[top * mw + right];
          const float bl = image[bot * mw + left], br = image[bot * mw + right];
          float t = tr - tl; t = t * lx; t = tl + t;
          float bb = br - bl; bb = bb * lx; bb = bl + bb;
          float r = bb - t; r = r * ly; r = t + r;
          tmp[(size_t)y * W + x] = r;
        }
      }
    }
    uint8_t* o = out + (size_t)b * H * W;
    for (size_t p = 0; p < (size_t)H * W; ++p) o[p] = tmp[p] > thr ? 1 : 0;
    free(tmp);
  }
}

/* ------------------------------------------------------------------ training-side neighbours (SURVEY.md 8f "next" #3) */
/* lib/structures/box_list_ops.py:295-334 pairwise_iou (iou_type='iou'): boxes1 [n1,4] rows, boxes2 [n2,4] columns */
static inline float orc_pair_iou(const float* a, const float* b) {
  const float ih = fmaxf(0.0f, fminf(a[2], b[2]) - fmaxf(a[0], b[0]));
  const float iw = fmaxf(0.0f, fminf(a[3], b[3]) - fmaxf(a[1], b[1]));
  const float inter = ih * iw;
  const float area1 = (a[2] - a[0]) * (a[3] - a[1]);
  const float area2 = (b[2] - b[0]) * (b[3] - b[1]);
  float u = area1 + area2;
  u = u - inter;
  return (u == 0.0f) ? 0.0f : inter / u;
}
ORC_API void orc_pairwise_iou(const float* b1, int64_t n1, const float* b2, int64_t n2, float* out) {
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n1; ++i)
    for (int64_t j = 0; j < n2; ++j) out[i * n2 + j] = orc_pair_iou(b1 + 4 * i, b2 + 4 * j);
}

/* lib/structures/box_list_ops.py:335-371: the iou_type != "iou" branches of pairwise_iou (YOLOv4 losses).
 *   giou (:343-349): convex = convex_heights * intersect_widths  (sic: the reference multiplies by the INTERSECTION
 *        width); giou = iou - where(convex == 0, 0, (convex - unions) / convex)
 *   diou (:351-364): iou - where(diag2 == 0, 0, centre_dist2 / diag2)
 *   ciou (:365-370): v = 4/pi^2 * (atan(w1/h1) - atan(w2/h2))^2; alpha = v / (1 - iou + v); diou - alpha * v
 * fp32, one rounding per written op; tf.atan on the CPU is libm's atanf.  type: 1 giou, 2 diou, 3 ciou. */
static float orc_pair_iou_variant(const float* a, const float* b, int type) {
  const float ih = fmaxf(0.0f, fminf(a[2], b[2]) - fmaxf(a[0], b[0]));
  const float iw = fmaxf(0.0f, fminf(a[3], b[3]) - fmaxf(a[1], b[1]));
  const float inter = ih * iw;
  const float h1 = a[2] - a[0], w1 = a[3] - a[1], h2 = b[2] - b[0], w2 = b[3] - b[1];
  float u = h1 * w1 + h2 * w2;
  u = u - inter;
  const float iou = (u == 0.0f) ? 0.0f : inter / u;
  const float dy = fmaxf(a[2], b[2]) - fminf(a[0], b[0]);
  const float dx = fmaxf(a[3], b[3]) - fminf(a[1], b[1]);
  if (type == 1) {
    const float convex = fmaxf(0.0f, dy) * iw;
    float t = convex - u;
    t = (convex == 0.0f) ? 0.0f : t / convex;
    return iou - t;
  }
  const float diag2 = dy * dy + dx * dx;
  float cx = (a[1] + a[3]) / 2.0f - (b[1] + b[3]) / 2.0f;
  float cy = (a[0] + a[2]) / 2.0f - (b[0] + b[2]) / 2.0f;
  const float cd2 = cx * cx + cy * cy;
  const float diou = iou - ((diag2 == 0.0f) ? 0.0f : cd2 / diag2);
  if (type == 2) return diou;
  float d = atanf(w1 / h1) - atanf(w2 / h2);
  const float v = 0.40528473456935109f * (d * d); /* 4 / pi^2 */
  float den = 1.0f - iou;
  den = den + v;
  const float alpha = v / den;
  return diou - alpha * v;
}
ORC_API void orc_pairwise_iou_variant(const float* b1, int64_t n1, const float* b2, int64_t n2, int type, float* out) {
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n1; ++i)
    for (int64_t j = 0; j < n2; ++j)
      out[i * n2 + j] = type == 0 ? orc_pair_iou(b1 + 4 * i, b2 + 4 * j) : orc_pair_iou_variant(b1 + 4 * i, b2 + 4 * j, type);
}

/* lib/modeling/matcher.py:8-174 Matcher.__call__ on a match-quality matrix q [M, N] (+ optional crowd matrix
 * [Mc, N]).  thresholds has nt entries (without the -inf/+inf ends), labels nt+1 entries. */
ORC_API void orc_matcher(const float* q, int64_t M, int64_t N, const float* crowd, int64_t Mc,
                         const float* difficult, int64_t Md, const float* thresholds, int nt,
                         const int32_t* labels, int allow_low_quality, int64_t* matches,
                         int64_t* match_labels) {
  if (M <= 0) {
    for (int64_t j = 0; j < N; ++j) { matches[j] = 0; match_labels[j] = 0; }
  } else {
    for (int64_t j = 0; j < N; ++j) { /* argmax / reduce_max over axis 0 (first maximum wins) :93-94 */
      int64_t bi = 0; float bv = q[j];
      for (int64_t i = 1; i < M; ++i) { const float v = q[i * N + j]; if (v > bv) { bv = v; bi = i; } }
      matches[j] = bi;
      int64_t lab = 0;
      for (int t = 0; t <= nt; ++t) { /* :97-107 */
        const float low = (t == 0) ? -INFINITY : thresholds[t - 1];
        const float high = (t == nt) ? INFINITY : thresholds[t];
        if (bv >= low && bv < high) lab = labels[t];
      }
      match_labels[j] = lab;
    }
    if (allow_low_quality) { /* get_low_quality_matches_ :152-174: dynamic_stitch overrides with 1 */
      for (int64_t i = 0; i < M; ++i) {
        float mx = q[i * N];
        for (int64_t j = 1; j < N; ++j) { const float v = q[i * N + j]; mx = (v > mx) ? v : mx; }
        for (int64_t j = 0; j < N; ++j) if (q[i * N + j] == mx) match_labels[j] = 1;
      }
    }
  }
  if (crowd) { /* :124-134 */
    for (int64_t j = 0; j < N; ++j) {
      int cb = 0;
      if (Mc > 0) {
        float mx = crowd[j];
        for (int64_t i = 1; i < Mc; ++i) { const float v = crowd[i * N + j]; mx = (v > mx) ? v : mx; }
        cb = mx > 1e-3f;
      }
      if (match_labels[j] == 0 && cb) match_labels[j] = -1;
    }
  }
  if (difficult) { /* :136-148: reduce_max(difficult_matrix) > self.thresholds[1] (first user threshold) */
    for (int64_t j = 0; j < N; ++j) {
      int db = 0;
      if (Md > 0) {
        float mx = difficult[j];
        for (int64_t i = 1; i < Md; ++i) { const float v = difficult[i * N + j]; mx = (v > mx) ? v : mx; }
        db = mx > thresholds[0];
      }
      if (match_labels[j] == 0 && db) match_labels[j] = -1;
    }
  }
}

/* lib/modeling/box_regression.py:38-74 Box2BoxTransform.get_deltas (src -> target), weights (wy,wx,wh,ww) */
ORC_API void orc_get_deltas(const float* src, const float* tgt, int64_t n, const float* w, float* out) {
  for (int64_t i = 0; i < n; ++i) {
    const float* s = src + 4 * i; const float* t = tgt + 4 * i;
    const float sh = s[2] - s[0], sw = s[3] - s[1];
    float scy = 0.5f * sh; scy = s[0] + scy;
    float scx = 0.5f * sw; scx = s[1] + scx;
    const float th = t[2] - t[0], tw = t[3] - t[1];
    float tcy = 0.5f * th; tcy = t[0] + tcy;
    float tcx = 0.5f * tw; tcx = t[1] + tcx;
    float dy = tcy - scy; dy = w[0] * dy; dy = dy / sh;
    float dx = tcx - scx; dx = w[1] * dx; dx = dx / sw;
    float dh = th / sh; dh = orc_logf(dh); dh = w[2] * dh;
    float dw = tw / sw; dw = orc_logf(dw); dw = w[3] * dw;
    out[4 * i + 0] = dy; out[4 * i + 1] = dx; out[4 * i + 2] = dh; out[4 * i + 3] = dw;
  }
}

/* Label assignment of one batch, composition of
 *   RPNOutputs._get_ground_truth            lib/modeling/proposal_generator/rpn_outputs.py:245-304
 *   ROIHeads.label_and_sample_proposals     lib/modeling/roi_heads/roi_heads.py:100-165 (up to the random sampling)
 * per image: boolean_mask GT by (valid & ~crowd [& ~difficult]), crowd list by is_crowd, difficult list by
 * gt_difficult; pairwise_iou x3; Matcher; optional inside_window (box_list_ops.py:150-161); get_deltas of the
 * positives stitched over zeros.  pred [N,P,4] (or [P,4] when pred_shared), pred_counts: valid prefix.
 * Rows beyond the prefix: matches 0, labels -1, deltas 0 (the reference drops them with boolean_mask). */
ORC_API void orc_label_boxes(const float* pred, int pred_shared, const int32_t* pred_counts, int N, int P,
                             const float* gt, const uint8_t* gt_valid, const uint8_t* gt_crowd,
                             const uint8_t* gt_difficult, int G, const float* thresholds, int nt,
                             const int32_t* labels, int allow_low_quality, float boundary_threshold,
                             const int32_t* image_shapes, const float* weights, int64_t* matches,
                             int64_t* out_labels, float* deltas) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int n = 0; n < N; ++n) {
    const float* pb = pred_shared ? pred : pred + (size_t)n * P * 4;
    const int64_t cnt = pred_counts ? (pred_counts[n] < P ? pred_counts[n] : P) : P;
    float* vg = (float*)malloc(sizeof(float) * 4 * (size_t)(G + 1));
    float* cg = (float*)malloc(sizeof(float) * 4 * (size_t)(G + 1));
    float* dg = (float*)malloc(sizeof(float) * 4 * (size_t)(G + 1));
    int64_t nv = 0, nc = 0, nd = 0;
    for (int g = 0; g < G; ++g) {
      const int v = gt_valid[(size_t)n * G + g] != 0;
      const int c = gt_crowd ? gt_crowd[(size_t)n * G + g] != 0 : 0;
      const int d = gt_difficult ? gt_difficult[(size_t)n * G + g] != 0 : 0;
      const float* b = gt + ((size_t)n * G + g) * 4;
      if (v && !c && !d) memcpy(vg + 4 * nv++, b, 16);
      if (c) memcpy(cg + 4 * nc++, b, 16);
      if (d) memcpy(dg + 4 * nd++, b, 16);
    }
    const size_t cc = (size_t)(cnt > 0 ? cnt : 1);
    float* q = (float*)malloc(sizeof(float) * (size_t)(nv + 1) * cc);
    float* qc = gt_crowd ? (float*)malloc(sizeof(float) * (size_t)(nc + 1) * cc) : NULL;
    float* qd = gt_difficult ? (float*)malloc(sizeof(float) * (size_t)(nd + 1) * cc) : NULL;
    for (int64_t i = 0; i < nv; ++i)
      for (int64_t j = 0; j < cnt; ++j) q[i * cnt + j] = orc_pair_iou(vg + 4 * i, pb + 4 * j);
    for (int64_t i = 0; i < nc && qc; ++i)
      for (int64_t j = 0; j < cnt; ++j) qc[i * cnt + j] = orc_pair_iou(cg + 4 * i, pb + 4 * j);
    for (int64_t i = 0; i < nd && qd; ++i)
      for (int64_t j = 0; j < cnt; ++j) qd[i * cnt + j] = orc_pair_iou(dg + 4 * i, pb + 4 * j);
    int64_t* m = matches + (size_t)n * P;
    int64_t* l = out_labels + (size_t)n * P;
    orc_matcher(q, nv, cnt, qc, nc, qd, nd, thresholds, nt, labels, allow_low_quality, m, l);
    if (boundary_threshold >= 0.0f) { /* rpn_outputs.py:268-278 */
      const float wy1 = 0.0f - boundary_threshold, wx1 = 0.0f - boundary_threshold;
      const float wy2 = (float)image_shapes[2 * n] + boundary_threshold;
      const float wx2 = (float)image_shapes[2 * n + 1] + boundary_threshold;
      for (int64_t j = 0; j < cnt; ++j) {
        const float* b = pb + 4 * j;
        const int viol = (b[0] < wy1) || (b[1] < wx1) || (b[2] > wy2) || (b[3] > wx2);
        if (viol) l[j] = -1;
      }
    }
    for (int64_t j = cnt; j < P; ++j) { m[j] = 0; l[j] = -1; }
    if (deltas) { /* rpn_outputs.py:280-292 */
      float* d = deltas + (size_t)n * P * 4;
      memset(d, 0, sizeof(float) * 4 * (size_t)P);
      for (int64_t j = 0; j < cnt; ++j)
        if (l[j] > 0 && nv > 0) orc_get_deltas(pb + 4 * j, vg + 4 * m[j], 1, weights, d + 4 * j);
    }
    free(q); free(qc); free(qd); free(vg); free(cg); free(dg);
  }
}

/* ------------------------------------------------------------------ ROIAlign backward (gradient w.r.t. the feature maps)
 * What TF autodiff runs for lib/layers/roi_align.py:45-66 + functional.py:100-166 in training:
 *   AvgPoolGrad (each sample gets g / sr^2)  ->  CropAndResizeGradImage (TF CPU kernel: per box, per crop pixel,
 *   dtop = (1-ly)*g; TL += (1-lx)*dtop; TR += lx*dtop; dbottom = ly*g; BL += (1-lx)*dbottom; BR += lx*dbottom,
 *   boxes in index order)  ->  MirrorPadGrad SYMMETRIC (border rows/cols folded onto the edge pixel).
 * Boxes receive no gradient (functional.py:120 stop_gradient).  grad_image [N,H,W,C] is ACCUMULATED into. */
ORC_API int orc_roi_align_backward(const float* grad_out, int N, int H, int W, int C, const float* boxes,
                                   const int32_t* box_ind, int64_t M, int oh, int ow, float spatial_scale,
                                   int sampling_ratio, int aligned, float* grad_image) {
  const int sr = sampling_ratio > 0 ? sampling_ratio : 1;
  const int ch = oh * sr, cw = ow * sr;
  const int Hp = H + 2, Wp = W + 2;
  float* gp = (float*)calloc((size_t)N * Hp * Wp * C, sizeof(float));
  if (!gp) return -1;
  const float cnt = (float)(sr * sr);
  for (int64_t b = 0; b < M; ++b) {
    const int32_t bi = box_ind[b];
    if (bi < 0 || bi >= N) continue;
    const float ymin = boxes[4 * b + 0] * spatial_scale + 1.0f, xmin = boxes[4 * b + 1] * spatial_scale + 1.0f;
    const float ymax = boxes[4 * b + 2] * spatial_scale + 1.0f, xmax = boxes[4 * b + 3] * spatial_scale + 1.0f;
    float y1, x1, y2, x2;
    if (aligned) {
      float sph = (ymax - ymin) / (float)ch;
      float spw = (xmax - xmin) / (float)cw;
      float imh = (float)(Hp - 1), imw = (float)(Wp - 1);
      float ny = sph / 2.0f; ny = ymin + ny; ny = ny - 0.5f; ny = ny / imh;
      float nx = spw / 2.0f; nx = xmin + nx; nx = nx - 0.5f; nx = nx / imw;
      float nh = sph * (float)(ch - 1); nh = nh / imh;
      float nw = spw * (float)(cw - 1); nw = nw / imw;
      y1 = ny; x1 = nx; y2 = ny + nh; x2 = nx + nw;
    } else {
      y1 = ymin / (float)Hp; x1 = xmin / (float)Wp; y2 = ymax / (float)Hp; x2 = xmax / (float)Wp;
    }
    const float hs = (ch > 1) ? (y2 - y1) * (float)(Hp - 1) / (float)(ch - 1) : 0.0f;
    const float ws = (cw > 1) ? (x2 - x1) * (float)(Wp - 1) / (float)(cw - 1) : 0.0f;
    for (int y = 0; y < ch; ++y) {
      const float in_y = (ch > 1) ? y1 * (float)(Hp - 1) + (float)y * hs : 0.5f * (y1 + y2) * (float)(Hp - 1);
      if (!(in_y >= 0.0f && in_y <= (float)(Hp - 1))) continue;
      const int top = (int)floorf(in_y), bot = (int)ceilf(in_y);
      const float ly = in_y - (float)top;
      for (int x = 0; x < cw; ++x) {
        const float in_x = (cw > 1) ? x1 * (float)(Wp - 1) + (float)x * ws : 0.5f * (x1 + x2) * (float)(Wp - 1);
        if (!(in_x >= 0.0f && in_x <= (float)(Wp - 1))) continue;
        const int left = (int)floorf(in_x), right = (int)ceilf(in_x);
        const float lx = in_x - (float)left;
        const float* g = grad_out + (((size_t)b * oh + y / sr) * ow + x / sr) * C;
        float* TL = gp + (((size_t)bi * Hp + top) * Wp + left) * C;
        float* TR = gp + (((size_t)bi * Hp + top) * Wp + right) * C;
        float* BL = gp + (((size_t)bi * Hp + bot) * Wp + left) * C;
        float* BR = gp + (((size_t)bi * Hp + bot) * Wp + right) * C;
        const float omy = 1.0f - ly, omx = 1.0f - lx;
        for (int c = 0; c < C; ++c) {
          const float gv = (sr > 1) ? g[c] / cnt : g[c];
          const float dtop = omy * gv;
          TL[c] = TL[c] + omx * dtop;
          TR[c] = TR[c] + lx * dtop;
          const float dbot = ly * gv;
          BL[c] = BL[c] + omx * dbot;
          BR[c] = BR[c] + lx * dbot;
        }
      }
    }
  }
  /* MirrorPadGrad SYMMETRIC, 1 px: padded (py,px) folds onto un-padded clamp(p-1) */
  for (int n = 0; n < N; ++n)
    for (int py = 0; py < Hp; ++py) {
      int sy = py - 1; if (sy < 0) sy = 0; if (sy > H - 1) sy = H - 1;
      for (int px = 0; px < Wp; ++px) {
        int sx = px - 1; if (sx < 0) sx = 0; if (sx > W - 1) sx = W - 1;
        const float* s = gp + (((size_t)n * Hp + py) * Wp + px) * C;
        float* d = grad_image + (((size_t)n * H + sy) * W + sx) * C;
        for (int c = 0; c < C; ++c) d[c] = d[c] + s[c];
      }
    }
  free(gp);
  return 0;
}

/* ROIPooler backward: routes each ROI's gradient to the level assign_boxes_to_levels gave it
 * (gradient of the where/gather/concat/un-permute chain of lib/modeling/poolers.py:160-178). */
ORC_API int orc_roi_pooler_backward(const float* grad_out, float* const* grad_feats, const int* Hs, const int* Ws,
                                    int L, int N, int C, const float* scales, const float* boxes,
                                    const int64_t* batch_idx, int64_t M, int oh, int ow, int sampling_ratio,
                                    int aligned, int canonical_box_size, int canonical_level) {
  const size_t row = (size_t)oh * ow * C;
  int64_t* lv = (int64_t*)calloc((size_t)(M > 0 ? M : 1), sizeof(int64_t));
  if (L > 1) {
    const int min_level = (int)lroundf(-log2f(scales[0]));
    const int max_level = (int)lroundf(-log2f(scales[L - 1]));
    orc_assign_boxes_to_levels(boxes, M, min_level, max_level, canonical_box_size, canonical_level, lv);
  }
  int rc = 0;
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int l = 0; l < L; ++l) {
    float* lb = (float*)malloc(sizeof(float) * 4 * (size_t)(M > 0 ? M : 1));
    int32_t* bi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M > 0 ? M : 1));
    float* g = (float*)malloc(sizeof(float) * row * (size_t)(M > 0 ? M : 1));
    int64_t m = 0;
    for (int64_t i = 0; i < M; ++i)
      if (lv[i] == l) {
        memcpy(lb + 4 * m, boxes + 4 * i, 16);
        bi[m] = (int32_t)batch_idx[i];
        memcpy(g + (size_t)m * row, grad_out + (size_t)i * row, sizeof(float) * row);
        ++m;
      }
    int r = orc_roi_align_backward(g, N, Hs[l], Ws[l], C, lb, bi, m, oh, ow, scales[l], sampling_ratio, aligned,
                                   grad_feats[l]);
    if (r) {
#pragma omp atomic write
      rc = r;
    }
    free(lb); free(bi); free(g);
  }
  free(lv);
  return rc;
}

/* ------------------------------------------------------------------ YOLOv4 post-processing (SURVEY.md 8f "next" #4)
 * lib/modeling/single_stage_heads/yolov4_outputs.py:331-390 YOLOv4Outputs.inference, per image:
 *   score_max = reduce_max(probs, -1); keep = where(score_max > score_threshold)        (:352-355)
 *   classes = argmax(probs[keep], -1) (first maximum), scores = reduce_max(probs[keep]) (:359-360)
 *   ONE class-agnostic tf.image.non_max_suppression(boxes[keep], scores, post_nms_topk) (:362-364)
 *   gather, zero-pad to post_nms_topk with is_valid                                     (:365-375)
 * boxes [N, n, 4], probs [N, n, K]. */
ORC_API void orc_yolo_inference(const float* boxes, const float* probs, int N, int64_t n, int K,
                                float score_thresh, float nms_thresh, int post_nms_topk, float* out_boxes,
                                float* out_scores, int64_t* out_classes, uint8_t* out_valid, int32_t* out_num) {
#pragma omp parallel for num_threads(ORC_NT) schedule(dynamic, 1)
  for (int im = 0; im < N; ++im) {
    const size_t cap = (size_t)(n > 0 ? n : 1);
    float* cb = (float*)malloc(sizeof(float) * 4 * cap);
    float* cs = (float*)malloc(sizeof(float) * cap);
    int64_t* cc = (int64_t*)malloc(sizeof(int64_t) * cap);
    int64_t total = 0;
    for (int64_t i = 0; i < n; ++i) {
      const float* pr = probs + ((size_t)im * n + i) * K;
      /* reduce_max propagates NaN (TF's Max kernel reduces with Eigen::PropagateNaN): a row holding a NaN has
       * score_max NaN and is never kept, whatever the threshold; argmax then only sees NaN-free rows */
      float mx = pr[0]; int64_t am = 0; int has_nan = pr[0] != pr[0];
      for (int k = 1; k < K; ++k) { if (pr[k] != pr[k]) has_nan = 1; else if (pr[k] > mx) { mx = pr[k]; am = k; } }
      if (has_nan || !(mx > score_thresh)) continue;
      memcpy(cb + 4 * total, boxes + ((size_t)im * n + i) * 4, 16);
      cs[total] = mx; cc[total] = am; ++total;
    }
    int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(post_nms_topk > 0 ? post_nms_topk : 1));
    const int32_t nk = orc_nms(cb, cs, total, post_nms_topk, nms_thresh, keep);
    for (int j = 0; j < post_nms_topk; ++j) {
      const size_t o = (size_t)im * post_nms_topk + j;
      float* ob = out_boxes + o * 4;
      if (j < nk) { memcpy(ob, cb + 4 * (size_t)keep[j], 16); out_scores[o] = cs[keep[j]];
                    out_classes[o] = cc[keep[j]]; out_valid[o] = 1; }
      else { ob[0] = ob[1] = ob[2] = ob[3] = 0.0f; out_scores[o] = 0.0f; out_classes[o] = 0; out_valid[o] = 0; }
    }
    if (out_num) out_num[im] = nk;
    free(keep); free(cc); free(cs); free(cb);
  }
}

/* lib/modeling/single_stage_heads/solo_v2.py:29-40 point_nms (kernel_size 2) on NHWC scores:
 * zero-pad 1, max_pool 2x2 stride 1 VALID, keep = (x == pooled[:, :-1, :-1]) => x[y,x] survives iff it equals
 * max(x[y-1..y, x-1..x], with zeros outside). */
ORC_API void orc_point_nms(const float* x, int N, int H, int W, int C, float* out) {
#pragma omp parallel for collapse(2) num_threads(ORC_NT) schedule(static)
  for (int n = 0; n < N; ++n)
    for (int y = 0; y < H; ++y)
      for (int xx = 0; xx < W; ++xx)
        for (int c = 0; c < C; ++c) {
          const size_t o = (((size_t)n * H + y) * W + xx) * C + c;
          const float v = x[o];
          float m = v;
          const float up = (y > 0) ? x[o - (size_t)W * C] : 0.0f;
          const float lf = (xx > 0) ? x[o - C] : 0.0f;
          const float ul = (y > 0 && xx > 0) ? x[o - (size_t)W * C - C] : 0.0f;
          m = fmaxf(m, up); m = fmaxf(m, lf); m = fmaxf(m, ul);
          out[o] = (v == m) ? v * 1.0f : v * 0.0f;
        }
}

/* lib/modeling/single_stage_heads/solo_v2.py:513-517, 530-533 (mask stage of SOLOv2Head.inference):
 *   scores = sigmoid(logits); masks = cast(scores > thr, float32); sum_masks = reduce_sum(masks);
 *   score_sums = reduce_sum(scores * masks)   (TF's summation order is unspecified: the fp32 products are
 *                                              accumulated in double here and rounded once)
 * logits [n, hw] -> masks [n, hw] fp32 0/1, sum_masks [n], score_sums [n]. */
ORC_API void orc_solo_mask_stage(const float* logits, int64_t n, int64_t hw, float thr, float* masks,
                                 float* sum_masks, float* score_sums) {
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n; ++i) {
    float sm = 0.0f;
    double ss = 0.0;
    for (int64_t p = 0; p < hw; ++p) {
      const float s = orc_sigmoidf(logits[i * hw + p]);
      const float m = (s > thr) ? 1.0f : 0.0f;
      masks[i * hw + p] = m;
      sm = sm + m;
      const float prod = s * m;
      if (m != 0.0f) ss += (double)prod;
    }
    sum_masks[i] = sm; score_sums[i] = (float)ss;
  }
}

/* lib/modeling/single_stage_heads/solo_v2.py:499-511 (dynamic mask generation): tf.nn.conv2d of the mask features
 * [1, H, W, E] with the candidates' kernels reshaped to [1, 1, E, n], VALID, stride 1 -- per pixel a dot product over
 * E.  fp32, one multiply and one add per term in channel order (TF's CPU conv is an Eigen contraction whose summation
 * order is blocked and unspecified; GPU parity for this op is a tolerance, stated in the test).  Also returns
 * sum_k |kernel_k * feature_k| per output, the scale the tolerance is relative to.
 * features [hw, E], kernels [n, E] -> logits [n, hw], absum [n, hw] (optional). */
ORC_API void orc_solo_dynamic_conv(const float* features, const float* kernels, int64_t n, int64_t hw, int64_t E,
                                   float* logits, float* absum) {
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n; ++i)
    for (int64_t p = 0; p < hw; ++p) {
      float acc = 0.0f;
      double ab = 0.0;
      for (int64_t k = 0; k < E; ++k) {
        const float prod = kernels[i * E + k] * features[p * E + k];
        acc = acc + prod;
        ab += fabs((double)prod);
      }
      logits[i * hw + p] = acc;
      if (absum) absum[i * hw + p] = (float)ab;
    }
}

/* vectorised orc_sigmoidf (test convenience) */
ORC_API void orc_sigmoid_array(const float* x, int64_t n, float* out) {
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t i = 0; i < n; ++i) out[i] = orc_sigmoidf(x[i]);
}

/* lib/modeling/single_stage_heads/solo_v2.py:507-558: the tail of SOLOv2Head.inference_single_image after the
 * dynamic convolution, for ONE image.  mask_logits [n, hw] (conv output of the candidates that passed the score
 * threshold, in tf.where order), scores / classes / strides [n].
 *   pred_mask_scores = sigmoid(logits); pred_masks = scores > mask_threshold; sum_masks        (:513-517)
 *   keep = sum_masks > strides (boolean_mask keeps order)                                       (:520-526)
 *   pred_scores *= reduce_sum(mask_scores * masks) / sum_masks                                  (:529-533)
 *   top_k(min(pre_nms_topk, #kept), sorted)  + gathers                                          (:536-540)
 *   matrix_nms(masks, classes, scores, sum_masks)                                               (:543-546)
 *   keep = scores > update_score_threshold (order kept); pad_or_clip to max_det                 (:549-556)
 * Outputs zero padded: out_masks [max_det, hw] fp32 0/1, out_classes int64, out_scores, out_valid. Returns #valid. */
ORC_API int orc_solo_postprocess(const float* mask_logits, const float* scores, const int64_t* classes,
                                 const float* strides, int n, int64_t hw, float mask_thr, int pre_nms_topk, int kernel,
                                 float sigma, float update_thr, int max_det, float* out_masks, int64_t* out_classes,
                                 float* out_scores, uint8_t* out_valid) {
  memset(out_masks, 0, sizeof(float) * (size_t)max_det * hw);
  for (int j = 0; j < max_det; ++j) { out_classes[j] = 0; out_scores[j] = 0.0f; out_valid[j] = 0; }
  if (n <= 0) return 0;
  float* masks = (float*)malloc(sizeof(float) * (size_t)n * hw);
  float* sm = (float*)malloc(sizeof(float) * n);
  float* ss = (float*)malloc(sizeof(float) * n);
  orc_solo_mask_stage(mask_logits, n, hw, mask_thr, masks, sm, ss);
  int* kept = (int*)malloc(sizeof(int) * n);
  float* ks = (float*)malloc(sizeof(float) * n);
  int m = 0;
  for (int i = 0; i < n; ++i)
    if (sm[i] > strides[i]) {
      float sc = ss[i] / sm[i];
      ks[m] = scores[i] * sc;
      kept[m++] = i;
    }
  int k = pre_nms_topk < m ? pre_nms_topk : m;
  int nv = 0;
  if (k > 0) {
    float* tv = (float*)malloc(sizeof(float) * k);
    int32_t* ti = (int32_t*)malloc(sizeof(int32_t) * k);
    orc_top_k(ks, m, k, tv, ti);
    float* gm = (float*)malloc(sizeof(float) * (size_t)k * hw);
    float* gs = (float*)malloc(sizeof(float) * k);
    int64_t* gc = (int64_t*)malloc(sizeof(int64_t) * k);
    for (int r = 0; r < k; ++r) {
      const int src = kept[ti[r]];
      memcpy(gm + (size_t)r * hw, masks + (size_t)src * hw, sizeof(float) * hw);
      gs[r] = sm[src]; gc[r] = classes[src];
    }
    float* upd = (float*)malloc(sizeof(float) * k);
    orc_matrix_nms(gm, gc, tv, gs, k, hw, kernel, sigma, upd);
    for (int r = 0; r < k && nv < max_det; ++r)
      if (upd[r] > update_thr) {
        memcpy(out_masks + (size_t)nv * hw, gm + (size_t)r * hw, sizeof(float) * hw);
        out_classes[nv] = gc[r]; out_scores[nv] = upd[r]; out_valid[nv] = 1;
        ++nv;
      }
    free(upd); free(gc); free(gs); free(gm); free(ti); free(tv);
  }
  free(ks); free(kept); free(ss); free(sm); free(masks);
  return nv;
}

/* lib/modeling/single_stage_heads/solo_v2.py:599-627: what MaskKernelBranch.inference does with the kept masks after
 * the per-image tail: resize_images(bilinear) to the image size -> > mask_threshold -> boxes from masks.
 *   resize_images (lib/layers/functional.py:9-36) picks tf.compat.v2.image.resize when it exists (TF >= 1.14; the
 *   align_corners kwarg is then filtered out, :23-24 -> half-pixel centres) and tf.image.resize_images(
 *   align_corners=True) otherwise (:26-35): `align_corners` selects which of the two is restated.
 *   TF ResizeBilinear CPU kernel (un-vendored tensorflow, core/kernels/resize_bilinear_op.cc +
 *   image_resizer_state.h), fp32: scale = (align_corners && out > 1) ? (in-1)/(float)(out-1) : in/(float)out;
 *   src = half_pixel ? (i + 0.5f)*scale - 0.5f : i*scale; lower = max((int)floorf(src), 0);
 *   upper = min((int)ceilf(src), in-1); lerp = src - floorf(src);
 *   top = tl + (tr - tl)*x_lerp; bottom = bl + (br - bl)*x_lerp; value = top + (bottom - top)*y_lerp.
 *   boxes (:606-625): yy = mask*y, xx = mask*x; mean = sum/(count + 1e-5); yy = where(yy > 0, yy, mean);
 *   [ymin, xmin, ymax, xmax] = min / max over ALL pixels (so the mean always takes part, and mask pixels in row /
 *   column 0 count as "mean").  The sums are integer valued; TF's fp32 reduce_sum order is unspecified, here they
 *   are exact (double) and rounded once.
 * masks [D, h, w] fp32 0/1 -> out_masks [D, H, W] uint8 0/1, boxes [D, 4]. */
static void orc_resize_taps(int in_size, int out_size, int align_corners, int* lo, int* hi, float* lerp) {
  const float scale = (align_corners && out_size > 1) ? (float)(in_size - 1) / (float)(out_size - 1)
                                                      : (float)in_size / (float)out_size;
  for (int i = 0; i < out_size; ++i) {
    float src;
    if (align_corners) {
      src = (float)i * scale;
    } else {
      src = (float)i + 0.5f;
      src = src * scale;
      src = src - 0.5f;
    }
    const float f = floorf(src);
    int l = (int)f; if (l < 0) l = 0;
    int u = (int)ceilf(src); if (u > in_size - 1) u = in_size - 1;
    lo[i] = l; hi[i] = u; lerp[i] = src - f;
  }
}
ORC_API void orc_solo_upsample_boxes(const float* masks, int64_t D, int h, int w, int H, int W, int align_corners,
                                     float thr, uint8_t* out_masks, float* boxes) {
  int* ylo = (int*)malloc(sizeof(int) * (size_t)(2 * H + 2 * W + 4));
  int* yhi = ylo + H; int* xlo = yhi + H; int* xhi = xlo + W;
  float* yl = (float*)malloc(sizeof(float) * (size_t)(H + W + 2));
  float* xl = yl + H;
  orc_resize_taps(h, H, align_corners, ylo, yhi, yl);
  orc_resize_taps(w, W, align_corners, xlo, xhi, xl);
#pragma omp parallel for num_threads(ORC_NT) schedule(static)
  for (int64_t d = 0; d < D; ++d) {
    const float* m = masks + (size_t)d * h * w;
    uint8_t* o = out_masks + (size_t)d * H * W;
    double cnt = 0.0, sy = 0.0, sx = 0.0;
    float ymin = INFINITY, xmin = INFINITY, ymax = -INFINITY, xmax = -INFINITY;
    for (int y = 0; y < H; ++y) {
      const float* r0 = m + (size_t)ylo[y] * w;
      const float* r1 = m + (size_t)yhi[y] * w;
      for (int x = 0; x < W; ++x) {
        const float tl = r0[xlo[x]], tr = r0[xhi[x]], bl = r1[xlo[x]], br = r1[xhi[x]];
        float top = tr - tl; top = top * xl[x]; top = tl + top;
        float bot = br - bl; bot = bot * xl[x]; bot = bl + bot;
        float v = bot - top; v = v * yl[y]; v = top + v;
        const int on = v > thr;
        o[(size_t)y * W + x] = (uint8_t)on;
        if (on) {
          cnt += 1.0; sy += (double)y; sx += (double)x;
          if (y > 0) { if ((float)y < ymin) ymin = (float)y; if ((float)y > ymax) ymax = (float)y; }
          if (x > 0) { if ((float)x < xmin) xmin = (float)x; if ((float)x > xmax) xmax = (float)x; }
        }
      }
    }
    const float den = (float)cnt + 1e-5f;
    const float ymean = (float)sy / den, xmean = (float)sx / den;
    boxes[d * 4 + 0] = fminf(ymin, ymean); boxes[d * 4 + 1] = fminf(xmin, xmean);
    boxes[d * 4 + 2] = fmaxf(ymax, ymean); boxes[d * 4 + 3] = fmaxf(xmax, xmean);
  }
  free(ylo); free(yl);
}
