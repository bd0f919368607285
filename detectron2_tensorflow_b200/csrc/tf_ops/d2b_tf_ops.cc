// d2b_tf_ops.cc -- TensorFlow custom-op shim over the C-ABI of libd2b200.so.
//
// NOT LINKED IN THIS REPOSITORY'S BUILD: TensorFlow is not installable in the build image (no wheel, no network).
// What IS checked here: `tests/test_tf_shim_syntax.py` type-checks this file with
// `g++ -std=c++14 -fsyntax-only` against `tests/tf_stub/` -- minimal declarations of the TF C++ API it uses
// (OpKernel, OpKernelContext, REGISTER_OP, InferenceContext, Tensor, errors::*) -- so names, argument types,
// attr getters and the d2b200.h structs are verified; the runtime behaviour of TensorFlow itself is not.
// It is the glue a maintainer of the reference compiles against their own TensorFlow:
//   g++ -std=c++14 -shared -fPIC d2b_tf_ops.cc -o libd2b200_tf.so \
//       $(python -c 'import tensorflow as tf; print(" ".join(tf.sysconfig.get_compile_flags()))') \
//       -I<repo>/include -L<repo>/detectron2_tensorflow_b200/lib -ld2b200 \
//       $(python -c 'import tensorflow as tf; print(" ".join(tf.sysconfig.get_link_flags()))')
// and loads with tf.load_op_library("libd2b200_tf.so") (see INTEGRATION.md).  Every OpKernel only
// validates shapes, allocates outputs and a temp workspace, fetches the CUDA stream and calls ONE
// C function; all logic lives behind include/d2b200.h.
#include "tensorflow/core/framework/op.h"
#include "tensorflow/core/framework/op_kernel.h"
#include "tensorflow/core/framework/shape_inference.h"

#define EIGEN_USE_GPU
#include "tensorflow/core/util/gpu_kernel_helper.h"

#include <cmath>
#include <string>
#include <vector>

#include "d2b200.h"

namespace tf = tensorflow;
using tf::shape_inference::InferenceContext;

namespace {

cudaStream_t StreamOf(tf::OpKernelContext* ctx) { return ctx->eigen_device<Eigen::GpuDevice>().stream(); }

// Allocates the op's scratch as a temp uint8 tensor and runs `fn(workspace, bytes, stream)`.
template <typename Params, typename BytesFn, typename RunFn>
void RunOp(tf::OpKernelContext* ctx, const Params& p, BytesFn bytes_fn, RunFn run_fn) {
  const size_t bytes = bytes_fn(&p);
  tf::Tensor ws;
  OP_REQUIRES_OK(ctx, ctx->allocate_temp(tf::DT_UINT8, tf::TensorShape({static_cast<tf::int64>(bytes ? bytes : 1)}), &ws));
  const int rc = run_fn(&p, ws.flat<tf::uint8>().data(), bytes, StreamOf(ctx));
  OP_REQUIRES(ctx, rc == D2B_OK,
              tf::errors::Internal(d2b_status_string(rc), ": ", d2b_last_error()));
}

}  // namespace

// ------------------------------------------------------------------ D2RoiAlignMultilevel
// Replaces ROIPooler.call (lib/modeling/poolers.py:134-180).
REGISTER_OP("D2RoiAlignMultilevel")
    .Input("features: L * float")  // L NHWC maps
    .Input("boxes: float")         // [M, 4]
    .Input("batch_idx: int64")     // [M]
    .Attr("L: int >= 1")
    .Attr("output_h: int")
    .Attr("output_w: int")
    .Attr("sampling_ratio: int = 0")
    .Attr("aligned: bool = true")
    .Attr("scales: list(float)")
    .Attr("canonical_box_size: int = 224")
    .Attr("canonical_level: int = 4")
    .Output("pooled: float")       // [M, output_h, output_w, C]
    .Output("level_counts: int32")  // [L]
    .SetShapeFn([](InferenceContext* c) {
      int L, oh, ow;
      TF_RETURN_IF_ERROR(c->GetAttr("L", &L));
      TF_RETURN_IF_ERROR(c->GetAttr("output_h", &oh));
      TF_RETURN_IF_ERROR(c->GetAttr("output_w", &ow));
      c->set_output(0, c->MakeShape({c->Dim(c->input(L), 0), oh, ow, c->Dim(c->input(0), 3)}));
      c->set_output(1, c->MakeShape({L}));
      return tf::Status::OK();
    });

class D2RoiAlignMultilevelOp : public tf::OpKernel {
 public:
  explicit D2RoiAlignMultilevelOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("L", &L_));
    OP_REQUIRES_OK(c, c->GetAttr("output_h", &oh_));
    OP_REQUIRES_OK(c, c->GetAttr("output_w", &ow_));
    OP_REQUIRES_OK(c, c->GetAttr("sampling_ratio", &sr_));
    OP_REQUIRES_OK(c, c->GetAttr("aligned", &aligned_));
    OP_REQUIRES_OK(c, c->GetAttr("scales", &scales_));
    OP_REQUIRES_OK(c, c->GetAttr("canonical_box_size", &cbs_));
    OP_REQUIRES_OK(c, c->GetAttr("canonical_level", &cl_));
    OP_REQUIRES(c, static_cast<int>(scales_.size()) == L_ && L_ <= D2B_MAX_LEVELS,
                tf::errors::InvalidArgument("len(scales) must equal L <= ", D2B_MAX_LEVELS));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& boxes = ctx->input(L_);
    const tf::Tensor& bidx = ctx->input(L_ + 1);
    OP_REQUIRES(ctx, boxes.dims() == 2 && boxes.dim_size(1) == 4, tf::errors::InvalidArgument("boxes must be [M,4]"));
    d2b_roi_align_params p = {};
    for (int l = 0; l < L_; ++l) {
      const tf::Tensor& f = ctx->input(l);
      OP_REQUIRES(ctx, f.dims() == 4, tf::errors::InvalidArgument("features must be NHWC"));
      p.features[l] = f.flat<float>().data();
      p.height[l] = f.dim_size(1);
      p.width[l] = f.dim_size(2);
      p.scale[l] = scales_[l];
    }
    p.num_levels = L_;
    p.num_images = ctx->input(0).dim_size(0);
    p.channels = ctx->input(0).dim_size(3);
    p.feature_dtype = D2B_DTYPE_F32;
    p.boxes = boxes.flat<float>().data();
    p.batch_idx = bidx.flat<tf::int64>().data();
    p.batch_idx_is_int64 = 1;
    p.batch_idx_stride = 1;
    p.num_rois = boxes.dim_size(0);
    p.output_h = oh_; p.output_w = ow_; p.sampling_ratio = sr_; p.aligned = aligned_; p.pad_border = 1;
    p.min_level = static_cast<int>(std::lround(-std::log2(scales_[0])));
    p.canonical_box_size = cbs_; p.canonical_level = cl_;
    tf::Tensor* out = nullptr;
    tf::Tensor* counts = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_rois, oh_, ow_, p.channels}), &out));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({L_}), &counts));
    p.out = out->flat<float>().data();
    p.out_dtype = D2B_DTYPE_F32;
    p.level_counts = counts->flat<tf::int32>().data();
    RunOp(ctx, p, d2b_roi_align_multilevel_workspace_bytes, d2b_roi_align_multilevel);
  }

 private:
  int L_, oh_, ow_, sr_, cbs_, cl_;
  bool aligned_;
  std::vector<float> scales_;
};
REGISTER_KERNEL_BUILDER(Name("D2RoiAlignMultilevel").Device(tf::DEVICE_GPU), D2RoiAlignMultilevelOp);

// ------------------------------------------------------------------ D2BatchedNms
// Replaces tf.map_fn(tf.image.non_max_suppression) (lib/layers/nms.py:6-26).
REGISTER_OP("D2BatchedNms")
    .Input("boxes: float")   // [S, n, 4]
    .Input("scores: float")  // [S, n]
    .Attr("max_output_size: int")
    .Attr("iou_threshold: float = 0.5")
    .Output("keep: int32")      // [S, max_output_size], -1 padded
    .Output("num_keep: int32")  // [S]
    .SetShapeFn([](InferenceContext* c) {
      int mo;
      TF_RETURN_IF_ERROR(c->GetAttr("max_output_size", &mo));
      c->set_output(0, c->MakeShape({c->Dim(c->input(0), 0), mo}));
      c->set_output(1, c->MakeShape({c->Dim(c->input(0), 0)}));
      return tf::Status::OK();
    });

class D2BatchedNmsOp : public tf::OpKernel {
 public:
  explicit D2BatchedNmsOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("max_output_size", &mo_));
    OP_REQUIRES_OK(c, c->GetAttr("iou_threshold", &thr_));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& boxes = ctx->input(0);
    const tf::Tensor& scores = ctx->input(1);
    OP_REQUIRES(ctx, boxes.dims() == 3 && scores.dims() == 2, tf::errors::InvalidArgument("ranks must be 3 and 2"));
    d2b_batched_nms_params p = {};
    p.boxes = boxes.flat<float>().data();
    p.scores = scores.flat<float>().data();
    p.num_segments = boxes.dim_size(0);
    p.n = boxes.dim_size(1);
    p.max_output_size = mo_;
    p.iou_threshold = thr_;
    tf::Tensor *keep = nullptr, *num = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_segments, mo_}), &keep));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({p.num_segments}), &num));
    p.keep = keep->flat<tf::int32>().data();
    p.num_keep = num->flat<tf::int32>().data();
    RunOp(ctx, p, d2b_batched_nms_workspace_bytes, d2b_batched_nms);
  }

 private:
  int mo_;
  float thr_;
};
REGISTER_KERNEL_BUILDER(Name("D2BatchedNms").Device(tf::DEVICE_GPU), D2BatchedNmsOp);

// ------------------------------------------------------------------ D2RpnProposals
// Replaces RPNOutputs.predict_proposals + find_top_rpn_proposals (rpn_outputs.py:403-426, 29-132).
REGISTER_OP("D2RpnProposals")
    .Input("logits: L * float")   // L x [N, HWA_l]
    .Input("deltas: L * float")   // L x [N, HWA_l, 4]
    .Input("anchors: L * float")  // L x [HWA_l, 4]
    .Input("image_shapes: int32")  // [N, 2] (h, w)
    .Attr("L: int >= 1")
    .Attr("pre_nms_topk: int")
    .Attr("post_nms_topk: int")
    .Attr("nms_thresh: float = 0.7")
    .Attr("min_box_side_len: float = 0.0")
    .Attr("weights: list(float) = [1.0, 1.0, 1.0, 1.0]")
    .Output("boxes: float")     // [N, post, 4]
    .Output("logits_out: float")  // [N, post]
    .Output("is_valid: bool")   // [N, post]
    .SetShapeFn([](InferenceContext* c) {
      int post;
      TF_RETURN_IF_ERROR(c->GetAttr("post_nms_topk", &post));
      auto n = c->Dim(c->input(0), 0);
      c->set_output(0, c->MakeShape({n, post, 4}));
      c->set_output(1, c->MakeShape({n, post}));
      c->set_output(2, c->MakeShape({n, post}));
      return tf::Status::OK();
    });

class D2RpnProposalsOp : public tf::OpKernel {
 public:
  explicit D2RpnProposalsOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("L", &L_));
    OP_REQUIRES_OK(c, c->GetAttr("pre_nms_topk", &pre_));
    OP_REQUIRES_OK(c, c->GetAttr("post_nms_topk", &post_));
    OP_REQUIRES_OK(c, c->GetAttr("nms_thresh", &thr_));
    OP_REQUIRES_OK(c, c->GetAttr("min_box_side_len", &min_len_));
    OP_REQUIRES_OK(c, c->GetAttr("weights", &w_));
    OP_REQUIRES(c, L_ <= D2B_MAX_LEVELS && w_.size() == 4, tf::errors::InvalidArgument("bad L / weights"));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    d2b_rpn_proposals_params p = {};
    for (int l = 0; l < L_; ++l) {
      p.logits[l] = ctx->input(l).flat<float>().data();
      p.deltas[l] = ctx->input(L_ + l).flat<float>().data();
      p.anchors[l] = ctx->input(2 * L_ + l).flat<float>().data();
      p.hwa[l] = ctx->input(2 * L_ + l).dim_size(0);
    }
    p.num_levels = L_;
    p.num_images = ctx->input(0).dim_size(0);
    p.image_shapes = ctx->input(3 * L_).flat<tf::int32>().data();
    p.nms_thresh = thr_; p.pre_nms_topk = pre_; p.post_nms_topk = post_; p.min_box_side_len = min_len_;
    for (int i = 0; i < 4; ++i) p.weights[i] = w_[i];
    p.scale_clamp = 4.135166556742356f;  // log(1000/16), box_regression.py:10
    tf::Tensor *b = nullptr, *lg = nullptr, *v = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_images, post_, 4}), &b));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({p.num_images, post_}), &lg));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(2, tf::TensorShape({p.num_images, post_}), &v));
    p.out_boxes = b->flat<float>().data();
    p.out_logits = lg->flat<float>().data();
    p.out_valid = reinterpret_cast<uint8_t*>(v->flat<bool>().data());
    RunOp(ctx, p, d2b_rpn_proposals_workspace_bytes, d2b_rpn_proposals);
  }

 private:
  int L_, pre_, post_;
  float thr_, min_len_;
  std::vector<float> w_;
};
REGISTER_KERNEL_BUILDER(Name("D2RpnProposals").Device(tf::DEVICE_GPU), D2RpnProposalsOp);
// image_shapes is read by the kernels, so it is a DEVICE input (no HostMemory): a custom GPU kernel receives
// every input in device memory unless the registration says otherwise.

// ------------------------------------------------------------------ D2MatrixNms
// Replaces matrix_nms (lib/layers/nms.py:29-83).
REGISTER_OP("D2MatrixNms")
    .Input("masks: float")    // [n, H, W]
    .Input("classes: int64")  // [n]
    .Input("scores: float")   // [n]
    .Input("sum_masks: float")  // [n]
    .Attr("kernel: string = 'gaussian'")
    .Attr("sigma: float = 2.0")
    .Output("updated_scores: float")
    .SetShapeFn([](InferenceContext* c) {
      c->set_output(0, c->input(2));
      return tf::Status::OK();
    });

class D2MatrixNmsOp : public tf::OpKernel {
 public:
  explicit D2MatrixNmsOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    std::string k;
    OP_REQUIRES_OK(c, c->GetAttr("kernel", &k));
    OP_REQUIRES_OK(c, c->GetAttr("sigma", &sigma_));
    OP_REQUIRES(c, k == "gaussian" || k == "linear", tf::errors::Unimplemented("NMS kernel ", k, " not implemented yet."));
    kernel_ = k == "gaussian" ? D2B_MNMS_GAUSSIAN : D2B_MNMS_LINEAR;
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& m = ctx->input(0);
    OP_REQUIRES(ctx, m.dims() == 3, tf::errors::InvalidArgument("masks must be [n,H,W]"));
    d2b_matrix_nms_params p = {};
    p.masks = m.flat<float>().data();
    p.classes = reinterpret_cast<const int64_t*>(ctx->input(1).flat<tf::int64>().data());
    p.scores = ctx->input(2).flat<float>().data();
    p.sum_masks = ctx->input(3).flat<float>().data();
    p.batch = 1;
    p.n = m.dim_size(0);
    p.hw = m.dim_size(1) * m.dim_size(2);
    p.kernel = kernel_;
    p.sigma = sigma_;
    tf::Tensor* out = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, ctx->input(2).shape(), &out));
    p.out = out->flat<float>().data();
    RunOp(ctx, p, d2b_matrix_nms_workspace_bytes, d2b_matrix_nms);
  }

 private:
  int kernel_;
  float sigma_;
};
REGISTER_KERNEL_BUILDER(Name("D2MatrixNms").Device(tf::DEVICE_GPU), D2MatrixNmsOp);

// ------------------------------------------------------------------ D2FastRcnnPostprocess
// Replaces fast_rcnn_inference (lib/modeling/roi_heads/fast_rcnn.py:28-187): clip -> score threshold -> fp32
// class-offset NMS -> top-k, zero padded.  `indices` / `rmax` are SparseBoxList.indices and dense_shape[1].
REGISTER_OP("D2FastRcnnPostprocess")
    .Input("boxes: float")         // [M, Kb*4], Kb = num_classes or 1 (class-agnostic regression)
    .Input("scores: float")        // [M, K+1], last column = background
    .Input("indices: int64")       // [M, 2] (image, slot)
    .Input("image_shapes: int32")  // [N, 2] (h, w)
    .Attr("rmax: int")
    .Attr("score_thresh: float = 0.05")
    .Attr("nms_thresh: float = 0.5")
    .Attr("topk_per_image: int = 100")
    .Attr("nms_cls_agnostic: bool = false")
    .Output("pred_boxes: float")     // [N, topk, 4]
    .Output("scores_out: float")     // [N, topk]
    .Output("pred_classes: int64")   // [N, topk]   (fast_rcnn.py:178)
    .Output("is_valid: bool")        // [N, topk]
    .Output("kept_roi_index: int32")  // [N, topk] slot of the source ROI, -1 padded (kept_indices, :150-166)
    .SetShapeFn([](InferenceContext* c) {
      int topk;
      TF_RETURN_IF_ERROR(c->GetAttr("topk_per_image", &topk));
      auto n = c->Dim(c->input(3), 0);
      c->set_output(0, c->MakeShape({n, topk, 4}));
      for (int i = 1; i < 5; ++i) c->set_output(i, c->MakeShape({n, topk}));
      return tf::Status::OK();
    });

class D2FastRcnnPostprocessOp : public tf::OpKernel {
 public:
  explicit D2FastRcnnPostprocessOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("rmax", &rmax_));
    OP_REQUIRES_OK(c, c->GetAttr("score_thresh", &score_thr_));
    OP_REQUIRES_OK(c, c->GetAttr("nms_thresh", &nms_thr_));
    OP_REQUIRES_OK(c, c->GetAttr("topk_per_image", &topk_));
    OP_REQUIRES_OK(c, c->GetAttr("nms_cls_agnostic", &agnostic_));
    OP_REQUIRES(c, rmax_ >= 0 && topk_ >= 1, tf::errors::InvalidArgument("rmax must be >= 0 and topk_per_image >= 1"));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& boxes = ctx->input(0);
    const tf::Tensor& scores = ctx->input(1);
    const tf::Tensor& indices = ctx->input(2);
    const tf::Tensor& shapes = ctx->input(3);
    OP_REQUIRES(ctx, boxes.dims() == 2 && scores.dims() == 2 && scores.dim_size(1) >= 2 &&
                         boxes.dim_size(0) == scores.dim_size(0),
                tf::errors::InvalidArgument("boxes must be [M,Kb*4] and scores [M,K+1]"));
    OP_REQUIRES(ctx, indices.dims() == 2 && indices.dim_size(1) == 2 && indices.dim_size(0) == boxes.dim_size(0),
                tf::errors::InvalidArgument("indices must be [M,2]"));
    OP_REQUIRES(ctx, shapes.dims() == 2 && shapes.dim_size(1) == 2, tf::errors::InvalidArgument("image_shapes must be [N,2]"));
    const int K = static_cast<int>(scores.dim_size(1)) - 1;
    OP_REQUIRES(ctx, boxes.dim_size(1) == 4 || boxes.dim_size(1) == 4 * K,
                tf::errors::InvalidArgument("boxes must have 4 or 4*num_classes columns"));
    d2b_fast_rcnn_params p = {};
    p.boxes = boxes.flat<float>().data();
    p.scores = scores.flat<float>().data();
    p.indices = reinterpret_cast<const int64_t*>(indices.flat<tf::int64>().data());
    p.num_preds = boxes.dim_size(0);
    p.num_images = static_cast<int>(shapes.dim_size(0));
    p.rmax = rmax_;
    p.num_bbox_reg_classes = static_cast<int>(boxes.dim_size(1) / 4);
    p.num_classes = K;
    p.image_shapes = shapes.flat<tf::int32>().data();
    p.score_thresh = score_thr_;
    p.nms_thresh = nms_thr_;
    p.topk_per_image = topk_;
    p.nms_cls_agnostic = agnostic_ ? 1 : 0;
    tf::Tensor *ob = nullptr, *os = nullptr, *oc = nullptr, *ov = nullptr, *oi = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_images, topk_, 4}), &ob));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({p.num_images, topk_}), &os));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(2, tf::TensorShape({p.num_images, topk_}), &oc));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(3, tf::TensorShape({p.num_images, topk_}), &ov));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(4, tf::TensorShape({p.num_images, topk_}), &oi));
    p.out_boxes = ob->flat<float>().data();
    p.out_scores = os->flat<float>().data();
    p.out_classes = reinterpret_cast<int64_t*>(oc->flat<tf::int64>().data());
    p.out_valid = reinterpret_cast<uint8_t*>(ov->flat<bool>().data());
    p.out_roi_index = oi->flat<tf::int32>().data();
    RunOp(ctx, p, d2b_fast_rcnn_postprocess_workspace_bytes, d2b_fast_rcnn_postprocess);
  }

 private:
  int rmax_, topk_;
  float score_thr_, nms_thr_;
  bool agnostic_;
};
REGISTER_KERNEL_BUILDER(Name("D2FastRcnnPostprocess").Device(tf::DEVICE_GPU), D2FastRcnnPostprocessOp);

// ------------------------------------------------------------------ D2RetinanetPostprocess
// Replaces RetinaNetHead.inference (lib/modeling/single_stage_heads/retinanet.py:285-387) for the whole batch:
// sigmoid -> per-level top-k -> threshold -> decode -> class-offset NMS -> top max_detections, zero padded.
REGISTER_OP("D2RetinanetPostprocess")
    .Input("box_cls: L * float")    // L x [N, HWA_l, K] logits
    .Input("box_delta: L * float")  // L x [N, HWA_l, 4]
    .Input("anchors: L * float")    // L x [HWA_l, 4]
    .Attr("L: int >= 1")
    .Attr("topk_candidates: int = 1000")
    .Attr("score_thresh: float = 0.05")
    .Attr("nms_thresh: float = 0.5")
    .Attr("max_detections: int = 100")
    .Attr("weights: list(float) = [1.0, 1.0, 1.0, 1.0]")
    .Output("pred_boxes: float")    // [N, max_detections, 4]
    .Output("scores: float")        // [N, max_detections]
    .Output("pred_classes: int32")  // [N, max_detections]   (retinanet.py:381)
    .Output("is_valid: bool")       // [N, max_detections]
    .SetShapeFn([](InferenceContext* c) {
      int d;
      TF_RETURN_IF_ERROR(c->GetAttr("max_detections", &d));
      auto n = c->Dim(c->input(0), 0);
      c->set_output(0, c->MakeShape({n, d, 4}));
      for (int i = 1; i < 4; ++i) c->set_output(i, c->MakeShape({n, d}));
      return tf::Status::OK();
    });

class D2RetinanetPostprocessOp : public tf::OpKernel {
 public:
  explicit D2RetinanetPostprocessOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("L", &L_));
    OP_REQUIRES_OK(c, c->GetAttr("topk_candidates", &topk_));
    OP_REQUIRES_OK(c, c->GetAttr("score_thresh", &score_thr_));
    OP_REQUIRES_OK(c, c->GetAttr("nms_thresh", &nms_thr_));
    OP_REQUIRES_OK(c, c->GetAttr("max_detections", &det_));
    OP_REQUIRES_OK(c, c->GetAttr("weights", &w_));
    OP_REQUIRES(c, L_ <= D2B_MAX_LEVELS && w_.size() == 4, tf::errors::InvalidArgument("bad L / weights"));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    d2b_retinanet_params p = {};
    const tf::Tensor& cls0 = ctx->input(0);
    OP_REQUIRES(ctx, cls0.dims() == 3, tf::errors::InvalidArgument("box_cls must be [N,HWA,K]"));
    for (int l = 0; l < L_; ++l) {
      const tf::Tensor& cls = ctx->input(l);
      const tf::Tensor& dl = ctx->input(L_ + l);
      const tf::Tensor& an = ctx->input(2 * L_ + l);
      OP_REQUIRES(ctx, cls.dims() == 3 && dl.dims() == 3 && an.dims() == 2 && an.dim_size(1) == 4 &&
                           cls.dim_size(1) == an.dim_size(0) && dl.dim_size(1) == an.dim_size(0) &&
                           dl.dim_size(2) == 4 && cls.dim_size(2) == cls0.dim_size(2),
                  tf::errors::InvalidArgument("level ", l, ": box_cls [N,HWA,K], box_delta [N,HWA,4], anchors [HWA,4]"));
      p.box_cls[l] = cls.flat<float>().data();
      p.box_delta[l] = dl.flat<float>().data();
      p.anchors[l] = an.flat<float>().data();
      p.hwa[l] = an.dim_size(0);
    }
    p.num_levels = L_;
    p.num_images = static_cast<int>(cls0.dim_size(0));
    p.num_classes = static_cast<int>(cls0.dim_size(2));
    p.topk_candidates = topk_;
    p.score_thresh = score_thr_;
    p.nms_thresh = nms_thr_;
    p.max_detections = det_;
    for (int i = 0; i < 4; ++i) p.weights[i] = w_[i];
    p.scale_clamp = 4.135166556742356f;  // log(1000/16), box_regression.py:10
    tf::Tensor *ob = nullptr, *os = nullptr, *oc = nullptr, *ov = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_images, det_, 4}), &ob));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({p.num_images, det_}), &os));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(2, tf::TensorShape({p.num_images, det_}), &oc));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(3, tf::TensorShape({p.num_images, det_}), &ov));
    p.out_boxes = ob->flat<float>().data();
    p.out_scores = os->flat<float>().data();
    p.out_classes = oc->flat<tf::int32>().data();
    p.out_valid = reinterpret_cast<uint8_t*>(ov->flat<bool>().data());
    RunOp(ctx, p, d2b_retinanet_postprocess_workspace_bytes, d2b_retinanet_postprocess);
  }

 private:
  int L_, topk_, det_;
  float score_thr_, nms_thr_;
  std::vector<float> w_;
};
REGISTER_KERNEL_BUILDER(Name("D2RetinanetPostprocess").Device(tf::DEVICE_GPU), D2RetinanetPostprocessOp);

// ------------------------------------------------------------------ D2CropAndResizeAligned
// Replaces crop_and_resize on ONE feature map (lib/layers/functional.py:100-166): SYMMETRIC 1-px pad, the
// aligned half-pixel box transform and tf.image.crop_and_resize, without materialising the padded copy.
REGISTER_OP("D2CropAndResizeAligned")
    .Input("image: float")    // [N, H, W, C]
    .Input("boxes: float")    // [M, 4] in image pixels (y1, x1, y2, x2)
    .Input("box_ind: int32")  // [M]
    .Attr("crop_h: int")
    .Attr("crop_w: int")
    .Attr("aligned: bool = true")
    .Attr("pad_border: bool = true")
    .Output("crops: float")   // [M, crop_h, crop_w, C]
    .SetShapeFn([](InferenceContext* c) {
      int ch, cw;
      TF_RETURN_IF_ERROR(c->GetAttr("crop_h", &ch));
      TF_RETURN_IF_ERROR(c->GetAttr("crop_w", &cw));
      c->set_output(0, c->MakeShape({c->Dim(c->input(1), 0), ch, cw, c->Dim(c->input(0), 3)}));
      return tf::Status::OK();
    });

class D2CropAndResizeAlignedOp : public tf::OpKernel {
 public:
  explicit D2CropAndResizeAlignedOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("crop_h", &ch_));
    OP_REQUIRES_OK(c, c->GetAttr("crop_w", &cw_));
    OP_REQUIRES_OK(c, c->GetAttr("aligned", &aligned_));
    OP_REQUIRES_OK(c, c->GetAttr("pad_border", &pad_));
    OP_REQUIRES(c, ch_ >= 1 && cw_ >= 1, tf::errors::InvalidArgument("crop size must be positive"));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& image = ctx->input(0);
    const tf::Tensor& boxes = ctx->input(1);
    const tf::Tensor& ind = ctx->input(2);
    OP_REQUIRES(ctx, image.dims() == 4, tf::errors::InvalidArgument("image must be NHWC"));
    OP_REQUIRES(ctx, boxes.dims() == 2 && boxes.dim_size(1) == 4 && ind.dims() == 1 && ind.dim_size(0) == boxes.dim_size(0),
                tf::errors::InvalidArgument("boxes must be [M,4] and box_ind [M]"));
    d2b_crop_and_resize_params p = {};
    p.image = image.flat<float>().data();
    p.num_images = static_cast<int>(image.dim_size(0));
    p.height = static_cast<int>(image.dim_size(1));
    p.width = static_cast<int>(image.dim_size(2));
    p.channels = static_cast<int>(image.dim_size(3));
    p.boxes = boxes.flat<float>().data();
    p.box_ind = ind.flat<tf::int32>().data();
    p.num_boxes = boxes.dim_size(0);
    p.crop_h = ch_; p.crop_w = cw_;
    p.aligned = aligned_ ? 1 : 0;
    p.pad_border = pad_ ? 1 : 0;
    tf::Tensor* out = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_boxes, ch_, cw_, p.channels}), &out));
    p.out = out->flat<float>().data();
    RunOp(ctx, p, d2b_crop_and_resize_aligned_workspace_bytes, d2b_crop_and_resize_aligned);
  }

 private:
  int ch_, cw_;
  bool aligned_, pad_;
};
REGISTER_KERNEL_BUILDER(Name("D2CropAndResizeAligned").Device(tf::DEVICE_GPU), D2CropAndResizeAlignedOp);

// ------------------------------------------------------------------ D2RoiAlignMultilevelGrad
// Gradient of D2RoiAlignMultilevel w.r.t. the feature maps (boxes carry none: functional.py:120
// stop_gradient).  Registered from Python with @tf.RegisterGradient (INTEGRATION.md).
REGISTER_OP("D2RoiAlignMultilevelGrad")
    .Input("grad_pooled: float")   // [M, output_h, output_w, C]
    .Input("features: L * float")  // only their shapes are read
    .Input("boxes: float")
    .Input("batch_idx: int64")
    .Attr("L: int >= 1")
    .Attr("sampling_ratio: int = 0")
    .Attr("aligned: bool = true")
    .Attr("scales: list(float)")
    .Attr("canonical_box_size: int = 224")
    .Attr("canonical_level: int = 4")
    .Attr("deterministic: bool = false")  // true: no atomics, bit-identical to the CPU kernel (CropAndResizeGradImage)
    .Output("grad_features: L * float")
    .SetShapeFn([](InferenceContext* c) {
      int L;
      TF_RETURN_IF_ERROR(c->GetAttr("L", &L));
      for (int l = 0; l < L; ++l) c->set_output(l, c->input(1 + l));
      return tf::Status::OK();
    });

class D2RoiAlignMultilevelGradOp : public tf::OpKernel {
 public:
  explicit D2RoiAlignMultilevelGradOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("L", &L_));
    OP_REQUIRES_OK(c, c->GetAttr("sampling_ratio", &sr_));
    OP_REQUIRES_OK(c, c->GetAttr("aligned", &aligned_));
    OP_REQUIRES_OK(c, c->GetAttr("scales", &scales_));
    OP_REQUIRES_OK(c, c->GetAttr("canonical_box_size", &cbs_));
    OP_REQUIRES_OK(c, c->GetAttr("canonical_level", &cl_));
    OP_REQUIRES_OK(c, c->GetAttr("deterministic", &deterministic_));
    OP_REQUIRES(c, static_cast<int>(scales_.size()) == L_ && L_ <= D2B_MAX_LEVELS,
                tf::errors::InvalidArgument("len(scales) must equal L <= ", D2B_MAX_LEVELS));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& g = ctx->input(0);
    const tf::Tensor& boxes = ctx->input(1 + L_);
    const tf::Tensor& bidx = ctx->input(2 + L_);
    OP_REQUIRES(ctx, g.dims() == 4, tf::errors::InvalidArgument("grad_pooled must be [M,oh,ow,C]"));
    d2b_roi_align_backward_params p = {};
    d2b_roi_align_params& f = p.fwd;
    for (int l = 0; l < L_; ++l) {
      const tf::Tensor& x = ctx->input(1 + l);
      tf::Tensor* gx = nullptr;
      OP_REQUIRES_OK(ctx, ctx->allocate_output(l, x.shape(), &gx));
      // the kernel accumulates: start from zero
      cudaMemsetAsync(gx->flat<float>().data(), 0, sizeof(float) * gx->NumElements(), StreamOf(ctx));
      p.grad_features[l] = gx->flat<float>().data();
      f.height[l] = x.dim_size(1);
      f.width[l] = x.dim_size(2);
      f.scale[l] = scales_[l];
    }
    f.num_levels = L_;
    f.num_images = ctx->input(1).dim_size(0);
    f.channels = g.dim_size(3);
    f.feature_dtype = f.out_dtype = D2B_DTYPE_F32;
    f.boxes = boxes.flat<float>().data();
    f.batch_idx = bidx.flat<tf::int64>().data();
    f.batch_idx_is_int64 = 1;
    f.batch_idx_stride = 1;
    f.num_rois = boxes.dim_size(0);
    f.output_h = g.dim_size(1); f.output_w = g.dim_size(2);
    f.sampling_ratio = sr_; f.aligned = aligned_; f.pad_border = 1;
    f.min_level = static_cast<int>(std::lround(-std::log2(scales_[0])));
    f.canonical_box_size = cbs_; f.canonical_level = cl_;
    p.grad_out = g.flat<float>().data();
    p.deterministic = deterministic_ ? 1 : 0;
    RunOp(ctx, p, d2b_roi_align_backward_workspace_bytes, d2b_roi_align_backward);
  }

 private:
  int L_, sr_, cbs_, cl_;
  bool aligned_, deterministic_;
  std::vector<float> scales_;
};
REGISTER_KERNEL_BUILDER(Name("D2RoiAlignMultilevelGrad").Device(tf::DEVICE_GPU), D2RoiAlignMultilevelGradOp);

// ------------------------------------------------------------------ D2LabelBoxes
// Replaces pairwise_iou + Matcher (+ inside_window + get_deltas) of RPNOutputs._get_ground_truth
// (lib/modeling/proposal_generator/rpn_outputs.py:245-304) for the whole batch.
REGISTER_OP("D2LabelBoxes")
    .Input("anchors: float")        // [P, 4] shared by the images
    .Input("gt_boxes: float")       // [N, G, 4]
    .Input("gt_valid: bool")        // [N, G]
    .Input("gt_crowd: bool")        // [N, G]
    .Input("image_shapes: int32")   // [N, 2]
    .Attr("thresholds: list(float)")
    .Attr("labels: list(int)")
    .Attr("allow_low_quality_matches: bool = false")
    .Attr("boundary_threshold: float = -1.0")
    .Attr("weights: list(float) = [1.0, 1.0, 1.0, 1.0]")
    .Output("matches: int64")       // [N, P]
    .Output("match_labels: int64")  // [N, P]  == gt_objectness_logits
    .Output("gt_deltas: float")     // [N, P, 4]
    .SetShapeFn([](InferenceContext* c) {
      auto n = c->Dim(c->input(1), 0), pdim = c->Dim(c->input(0), 0);
      c->set_output(0, c->MakeShape({n, pdim}));
      c->set_output(1, c->MakeShape({n, pdim}));
      c->set_output(2, c->MakeShape({n, pdim, 4}));
      return tf::Status::OK();
    });

class D2LabelBoxesOp : public tf::OpKernel {
 public:
  explicit D2LabelBoxesOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("thresholds", &thr_));
    OP_REQUIRES_OK(c, c->GetAttr("labels", &labels_));
    OP_REQUIRES_OK(c, c->GetAttr("allow_low_quality_matches", &lq_));
    OP_REQUIRES_OK(c, c->GetAttr("boundary_threshold", &boundary_));
    OP_REQUIRES_OK(c, c->GetAttr("weights", &w_));
    OP_REQUIRES(c, thr_.size() >= 1 && thr_.size() <= D2B_MATCH_MAX_THRESHOLDS && labels_.size() == thr_.size() + 1 &&
                       w_.size() == 4,
                tf::errors::InvalidArgument("bad thresholds / labels / weights"));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& anchors = ctx->input(0);
    const tf::Tensor& gt = ctx->input(1);
    OP_REQUIRES(ctx, anchors.dims() == 2 && gt.dims() == 3, tf::errors::InvalidArgument("anchors [P,4], gt_boxes [N,G,4]"));
    d2b_label_boxes_params p = {};
    p.pred_boxes = anchors.flat<float>().data();
    p.pred_shared = 1;
    p.num_images = gt.dim_size(0);
    p.num_preds = anchors.dim_size(0);
    p.gt_boxes = gt.flat<float>().data();
    p.gt_valid = reinterpret_cast<const uint8_t*>(ctx->input(2).flat<bool>().data());
    p.gt_crowd = reinterpret_cast<const uint8_t*>(ctx->input(3).flat<bool>().data());
    p.max_gt = gt.dim_size(1);
    p.num_thresholds = static_cast<int>(thr_.size());
    for (size_t i = 0; i < thr_.size(); ++i) p.thresholds[i] = thr_[i];
    for (size_t i = 0; i < labels_.size(); ++i) p.labels[i] = labels_[i];
    p.allow_low_quality_matches = lq_;
    p.boundary_threshold = boundary_;
    p.image_shapes = ctx->input(4).flat<tf::int32>().data();
    p.compute_deltas = 1;
    for (int i = 0; i < 4; ++i) p.weights[i] = w_[i];
    tf::Tensor *m = nullptr, *l = nullptr, *d = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({p.num_images, p.num_preds}), &m));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({p.num_images, p.num_preds}), &l));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(2, tf::TensorShape({p.num_images, p.num_preds, 4}), &d));
    p.out_matches = reinterpret_cast<int64_t*>(m->flat<tf::int64>().data());
    p.out_labels = reinterpret_cast<int64_t*>(l->flat<tf::int64>().data());
    p.out_deltas = d->flat<float>().data();
    RunOp(ctx, p, d2b_label_boxes_workspace_bytes, d2b_label_boxes);
  }

 private:
  std::vector<float> thr_, w_;
  std::vector<int> labels_;
  bool lq_;
  float boundary_;
};
REGISTER_KERNEL_BUILDER(Name("D2LabelBoxes").Device(tf::DEVICE_GPU), D2LabelBoxesOp);

// ------------------------------------------------------------------ D2SoloDynamicMasks
// Replaces the dynamic mask generation + mask stage of SOLOv2Head.inference_single_image
// (lib/modeling/single_stage_heads/solo_v2.py:499-517, 530-533): tf.nn.conv2d(mask_features, pred_kernels) ->
// sigmoid -> > mask_threshold -> reduce_sum, for one image.  Outputs the bit-packed masks (int64 words, bit p of
// word w = pixel 64*w+p), sum_masks and the score sums; mask_scoring (:531-533) = score_sums / sum_masks and the
// packed words feed D2MatrixNms' packed variant (d2b_matrix_nms_params.packed_masks).
REGISTER_OP("D2SoloDynamicMasks")
    .Input("mask_features: float")  // [H, W, E]   (pred_mask_features of one image)
    .Input("mask_kernels: float")   // [n, E]      (pred_kernels gathered by keep_inds, :486)
    .Attr("mask_threshold: float = 0.5")
    .Output("packed_masks: int64")  // [n, ceil(H*W/64)]
    .Output("sum_masks: float")     // [n]
    .Output("score_sums: float")    // [n]
    .SetShapeFn([](InferenceContext* c) {
      c->set_output(0, c->Matrix(c->Dim(c->input(1), 0), InferenceContext::kUnknownDim));
      c->set_output(1, c->Vector(c->Dim(c->input(1), 0)));
      c->set_output(2, c->Vector(c->Dim(c->input(1), 0)));
      return tf::Status::OK();
    });

class D2SoloDynamicMasksOp : public tf::OpKernel {
 public:
  explicit D2SoloDynamicMasksOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("mask_threshold", &thr_));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& f = ctx->input(0);
    const tf::Tensor& k = ctx->input(1);
    OP_REQUIRES(ctx, f.dims() == 3 && k.dims() == 2 && k.dim_size(1) == f.dim_size(2),
                tf::errors::InvalidArgument("mask_features must be [H,W,E] and mask_kernels [n,E]"));
    d2b_solo_dynamic_masks_params p = {};
    p.mask_features = f.flat<float>().data();
    p.mask_kernels = k.flat<float>().data();
    p.batch = 1;
    p.n = k.dim_size(0);
    p.channels = k.dim_size(1);
    p.hw = f.dim_size(0) * f.dim_size(1);
    p.mask_threshold = thr_;
    tf::Tensor *packed = nullptr, *sums = nullptr, *ssum = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({k.dim_size(0), (p.hw + 63) / 64}), &packed));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({k.dim_size(0)}), &sums));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(2, tf::TensorShape({k.dim_size(0)}), &ssum));
    p.packed_masks = reinterpret_cast<uint64_t*>(packed->flat<tf::int64>().data());
    p.sum_masks = sums->flat<float>().data();
    p.score_sums = ssum->flat<float>().data();
    RunOp(ctx, p, d2b_solo_dynamic_masks_workspace_bytes, d2b_solo_dynamic_masks);
  }

 private:
  float thr_;
};
REGISTER_KERNEL_BUILDER(Name("D2SoloDynamicMasks").Device(tf::DEVICE_GPU), D2SoloDynamicMasksOp);

// ------------------------------------------------------------------ D2SoloUpsample
// Replaces the end of MaskKernelBranch.inference (solo_v2.py:599-627): resize_images(pred_masks, image_shape) ->
// > mask_threshold -> boxes from masks, from the packed masks of the tail.  image_shape is a host-memory input
// because it sizes the output (the reference passes a Python list).
REGISTER_OP("D2SoloUpsample")
    .Input("packed_masks: int64")  // [N, D, ceil(h*w/64)]
    .Input("image_shape: int32")   // [2] (H, W), host memory
    .Attr("mask_h: int")
    .Attr("mask_w: int")
    .Attr("mask_threshold: float = 0.5")
    .Attr("align_corners: bool = false")  // false: tf.compat.v2.image.resize exists (functional.py:21-24)
    .Output("pred_masks: uint8")          // [N, D, H, W]
    .Output("boxes: float")               // [N, D, 4]
    .SetShapeFn([](InferenceContext* c) {
      c->set_output(0, c->MakeShape({c->Dim(c->input(0), 0), c->Dim(c->input(0), 1), InferenceContext::kUnknownDim,
                                     InferenceContext::kUnknownDim}));
      c->set_output(1, c->MakeShape({c->Dim(c->input(0), 0), c->Dim(c->input(0), 1), 4}));
      return tf::Status::OK();
    });

class D2SoloUpsampleOp : public tf::OpKernel {
 public:
  explicit D2SoloUpsampleOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) {
    OP_REQUIRES_OK(c, c->GetAttr("mask_h", &h_));
    OP_REQUIRES_OK(c, c->GetAttr("mask_w", &w_));
    OP_REQUIRES_OK(c, c->GetAttr("mask_threshold", &thr_));
    OP_REQUIRES_OK(c, c->GetAttr("align_corners", &ac_));
  }
  void Compute(tf::OpKernelContext* ctx) override {
    const tf::Tensor& pk = ctx->input(0);
    const tf::Tensor& shp = ctx->input(1);
    OP_REQUIRES(ctx, pk.dims() == 3 && shp.NumElements() == 2, tf::errors::InvalidArgument("packed_masks [N,D,Wd], image_shape [2]"));
    d2b_solo_upsample_params p = {};
    p.packed_masks = reinterpret_cast<const uint64_t*>(pk.flat<tf::int64>().data());
    p.batch = pk.dim_size(0);
    p.num_dets = pk.dim_size(1);
    p.mask_h = h_;
    p.mask_w = w_;
    p.image_h = shp.flat<tf::int32>()(0);
    p.image_w = shp.flat<tf::int32>()(1);
    p.align_corners = ac_ ? 1 : 0;
    p.mask_threshold = thr_;
    tf::Tensor *masks = nullptr, *boxes = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({pk.dim_size(0), pk.dim_size(1), p.image_h, p.image_w}), &masks));
    OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({pk.dim_size(0), pk.dim_size(1), 4}), &boxes));
    p.out_masks = masks->flat<tf::uint8>().data();
    p.out_boxes = boxes->flat<float>().data();
    RunOp(ctx, p, d2b_solo_upsample_workspace_bytes, d2b_solo_upsample);
  }

 private:
  int h_, w_;
  float thr_;
  bool ac_;
};
REGISTER_KERNEL_BUILDER(Name("D2SoloUpsample").Device(tf::DEVICE_GPU).HostMemory("image_shape"), D2SoloUpsampleOp);

// D2SoloSelect / D2SoloPostprocess follow the same pattern over d2b_solo_select / d2b_solo_postprocess (static
// max_candidates / max_detections attrs give the fixed output shapes TF needs).
