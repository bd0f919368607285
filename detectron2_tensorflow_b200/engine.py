"""Post-backbone inference wiring of `GeneralizedRCNN.inference` (lib/modeling/meta_arch/rcnn.py:92-144):

    RPN.call -> find_top_rpn_proposals           (lib/modeling/proposal_generator/rpn.py:143-195)
    StandardROIHeads._forward_box  -> box pooler + fast_rcnn_inference   (roi_heads.py:545-577)
    StandardROIHeads._forward_mask -> mask pooler on the detections      (roi_heads.py:579-605)

with the dense conv/FC layers (RPN head, box head, mask head) outside: their outputs are inputs here.
Only reference-facing operators of this package are called; everything runs on torch's current stream
with no host synchronisation (static instance grids replace the reference's tf.where compaction: every
slot of the zero-padded dense outputs is pooled, `is_valid` tells which rows are live).

`run_host` is the host-buffer entry point (the analogue of `sess.run(fetches, feed_dict)`): inputs are host
tensors, outputs are pinned host tensors.  Images are independent, so the batch is cut into chunks that are
software-pipelined over three CUDA streams: the upload of chunk i+1, the kernels of chunk i and the download
of chunk i-1 overlap (PCIe is full duplex).
"""
import numpy as np
import torch

from .modeling import Box2BoxTransform, ROIPooler, RPNOutputs, fast_rcnn_inference
from .structures import BoxList, ImageList, SparseBoxList

PER_IMAGE_KEYS = ("logits", "deltas", "feats", "shapes")   # tensors (or lists of) with a leading image dim
PER_ROI_KEYS = ("scores", "cls_deltas")                      # [N * rois_per_image, ...], image-major
# the fixed-size padded per-image results a caller may want on rank 0 (SURVEY.md 8e); ROI features stay local
GATHER_KEYS = ("proposal_boxes", "proposal_logits", "proposal_valid", "det_boxes", "det_scores", "det_classes",
               "det_valid")


class GraphedStep(object):
    """A captured step: `replay()` enqueues it on the current stream; `outputs[c]` are the static per-block output
    tensors (flatten_outputs keys) of image block `bounds[c]`; `kernels_per_replay` counts the captured kernels."""

    def __init__(self, graph, outputs, bounds, kernels_per_replay):
        self.graph, self.outputs, self.bounds, self.kernels_per_replay = graph, outputs, bounds, int(kernels_per_replay)

    def replay(self):
        self.graph.replay()
        return self.outputs

    def gathered(self, keys=None):
        """Concatenate the per-block outputs in image order (a copy; for checks and small tensors)."""
        keys = list(self.outputs[0].keys()) if keys is None else keys
        return {k: torch.cat([o[k] for o in self.outputs]) for k in keys}


class StepPipeline(object):
    """`depth` captured steps (each with its own static outputs) replayed round-robin on their own streams, so that
    consecutive, independent batches overlap: the single-CTA latency chains of one step run under the HBM-bound
    pooling of the next.  `run(k)` enqueues k steps forked from / joined to the current stream."""

    def __init__(self, steps, device):
        self.steps = list(steps)
        self.device = device
        self.streams = [torch.cuda.Stream(device) for _ in self.steps]
        self._next = 0

    def run(self, k):
        cur = torch.cuda.current_stream(self.device)
        ev = torch.cuda.Event()
        ev.record(cur)
        for s in self.streams:
            s.wait_event(ev)
        last = None
        for _ in range(k):
            i = self._next
            self._next = (i + 1) % len(self.steps)
            with torch.cuda.stream(self.streams[i]):
                last = self.steps[i].replay()
        for s in self.streams:
            cur.wait_stream(s)
        return last


class MaskRCNNPostBackbone(object):
    def __init__(self, rois_per_image=1000, dets_per_image=100, pre_nms_topk=2000, rpn_nms_thresh=0.7,
                 min_box_side_len=0.0, score_thresh=0.05, nms_thresh=0.5, nms_cls_agnostic=False,
                 scales=(1 / 4., 1 / 8., 1 / 16., 1 / 32.), box_resolution=7, mask_resolution=14, sampling_ratio=0,
                 pooler_type="ROIAlignV2", rpn_weights=(1.0, 1.0, 1.0, 1.0), box_weights=(10.0, 10.0, 5.0, 5.0),
                 mask_on=True):
        self.mask_on = bool(mask_on)  # False: Faster R-CNN (no mask pooler; BASELINE.json configs[0])
        self.R, self.D = int(rois_per_image), int(dets_per_image)
        self.pre, self.rpn_thr, self.min_len = int(pre_nms_topk), float(rpn_nms_thresh), float(min_box_side_len)
        self.score_thr, self.nms_thr, self.agnostic = float(score_thresh), float(nms_thresh), bool(nms_cls_agnostic)
        self.rpn_tf = Box2BoxTransform(rpn_weights)
        self.box_tf = Box2BoxTransform(box_weights)
        self.box_pooler = ROIPooler(box_resolution, list(scales), sampling_ratio, pooler_type)
        self.mask_pooler = ROIPooler(mask_resolution, list(scales), sampling_ratio, pooler_type)
        # the per-level ROI counts are a training-time tf.summary (poolers.py:173); inference does not record them
        self.box_pooler.record_level_counts = self.mask_pooler.record_level_counts = False
        self._grids = {}
        self._streams = {}
        self._host_out = {}
        self._dev_in = {}

    # ------------------------------------------------------------------ helpers
    def _grid(self, n, per, dev):
        key = (n, per, str(dev))
        g = self._grids.get(key)
        if g is None:
            img = np.repeat(np.arange(n, dtype=np.int64), per)
            slot = np.tile(np.arange(per, dtype=np.int64), n)
            g = torch.from_numpy(np.stack([img, slot], 1)).to(dev)
            self._grids[key] = g
        return g

    # ------------------------------------------------------------------ device-resident step
    def __call__(self, x, events=None):
        """x: dict of DEVICE tensors -- logits L x [n,HWA], deltas L x [n,HWA,4], anchors L x [HWA,4],
        feats 4 x [n,H,W,C], shapes [n,2] int32, scores [n*R,K+1], cls_deltas [n*R,K*4].
        Returns dict(proposals BoxList, box_feats, dets BoxList, mask_feats)."""
        def mark(i):
            if events is not None:
                events[i].record()
        mark(0)
        st = self.stage_proposals(x)
        mark(1)
        self.stage_box_pool(x, st)
        mark(2)
        self.stage_detections(x, st)
        mark(3)
        self.stage_mask_pool(x, st)
        mark(4)
        return dict(proposals=st["props"], box_feats=st["box_feats"], dets=st["dets"], mask_feats=st["mask_feats"])

    # the four stages of the step (each runs on torch's current stream; `st` carries the intermediate results)
    def stage_proposals(self, x):
        n, dev = x["shapes"].shape[0], x["shapes"].device
        outs = RPNOutputs(self.rpn_tf, ImageList(None, x["shapes"]), x["logits"], x["deltas"], x["anchors"])
        props = outs.find_top_proposals(self.rpn_thr, self.pre, self.R, self.min_len)
        inst = SparseBoxList(self._grid(n, self.R, dev), BoxList(props.boxes.reshape(-1, 4)), (n, self.R))
        inst.set_tracking("image_shape", x["shapes"])
        return {"props": props, "inst": inst, "box_feats": None, "dets": None, "mask_feats": None}

    def stage_box_pool(self, x, st):
        st["box_feats"] = self.box_pooler(x["feats"], st["inst"])

    def stage_detections(self, x, st):
        # FastRCNNOutputs.inference (fast_rcnn.py:381-395): predict_boxes' decode is fused into the post-processing
        st["dets"], _ = fast_rcnn_inference(None, x["scores"], st["inst"], self.score_thr, self.nms_thr, self.D,
                                            self.agnostic, pred_proposal_deltas=x["cls_deltas"],
                                            box2box_transform=self.box_tf)

    def stage_mask_pool(self, x, st):
        if self.mask_on:
            n, dev = x["shapes"].shape[0], x["shapes"].device
            dinst = SparseBoxList(self._grid(n, self.D, dev), BoxList(st["dets"].boxes.reshape(-1, 4)), (n, self.D))
            st["mask_feats"] = self.mask_pooler(x["feats"], dinst)

    # ------------------------------------------------------------------ CUDA-graphed, chunk-concurrent step
    def capture(self, x, chunks=4, epilogue=None, epilogue_warmup=True):
        """Capture the device-resident step as ONE CUDA graph in which the batch is cut into `chunks` image blocks
        that run on their own streams (forked from / joined to the capturing stream).  Images are independent, so
        the latency-bound proposal / post-processing kernels of one block overlap the HBM-bound ROIAlign of
        another, and replaying the graph removes the per-launch host cost of the ~47 x chunks kernel launches.
        `x` holds the STATIC input tensors: refill them in place between replays.  `epilogue(outs)` (optional) is
        captured at the end of the step, on the capturing stream after the image blocks have joined -- e.g.
        `sharding.GatherPlan.pack`, so that packing the send buffer costs graph nodes instead of eager launches.
        Returns a `GraphedStep`."""
        from . import _native as nv
        from .sharding import image_block
        dev = x["shapes"].device
        n = x["shapes"].shape[0]
        chunks = max(1, min(int(chunks), n))
        bounds = [image_block(n, chunks, c) for c in range(chunks)]
        streams = [torch.cuda.Stream(dev) for _ in range(chunks)]
        R = self.R

        def cut(b, e):
            d = {"anchors": x["anchors"], "shapes": x["shapes"][b:e], "scores": x["scores"][b * R:e * R],
                 "cls_deltas": x["cls_deltas"][b * R:e * R]}
            for k in ("logits", "deltas", "feats"):
                d[k] = [t[b:e] for t in x[k]]
            return d

        def step(with_epilogue=True):
            cur = torch.cuda.current_stream(dev)
            start = torch.cuda.Event()
            start.record(cur)
            outs = []
            for s, (b, e) in zip(streams, bounds):
                s.wait_event(start)
                with torch.cuda.stream(s):
                    outs.append(self.flatten_outputs(self(cut(b, e))))
            for s in streams:
                cur.wait_stream(s)
            if epilogue is not None and with_epilogue:
                epilogue(outs)
            return outs

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):  # warm-up outside the capture: workspaces, grids, smem attributes
            for _ in range(2):
                step(epilogue_warmup)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        l0 = nv.kernel_launch_count()
        with torch.cuda.graph(graph):
            outs = step()
        return GraphedStep(graph, outs, bounds, nv.kernel_launch_count() - l0)

    def pipeline(self, x, chunks=4, depth=2, epilogues=None, epilogue_warmup=True):
        """`depth` independent captures of the step over the same static inputs `x` -> StepPipeline
        (`epilogues[i]`: the capture epilogue of step i)."""
        depth = max(1, int(depth))
        return StepPipeline([self.capture(x, chunks, epilogues[i] if epilogues else None, epilogue_warmup)
                             for i in range(depth)],
                            x["shapes"].device)

    # ------------------------------------------------------------------ host-buffer step
    @staticmethod
    def flatten_outputs(out):
        p, d = out["proposals"], out["dets"]
        flat = {"proposal_boxes": p.boxes, "proposal_logits": p.get_field("objectness_logits"),
                "proposal_valid": p.get_field("is_valid"), "box_feats": out["box_feats"],
                "det_boxes": d.boxes, "det_scores": d.get_field("scores"), "det_classes": d.get_field("pred_classes"),
                "det_valid": d.get_field("is_valid")}
        if out["mask_feats"] is not None:
            flat["mask_feats"] = out["mask_feats"]
        return flat

    def gather_spec(self):
        """{key: (per-image shape, dtype)} of the GATHER_KEYS outputs (for sharding.GatherPlan)."""
        R, D = self.R, self.D
        return {"proposal_boxes": ((R, 4), torch.float32), "proposal_logits": ((R,), torch.float32),
                "proposal_valid": ((R,), torch.bool), "det_boxes": ((D, 4), torch.float32),
                "det_scores": ((D,), torch.float32), "det_classes": ((D,), torch.int64), "det_valid": ((D,), torch.bool)}

    def run_host(self, x, device=None, chunk_images=2):
        """x: dict of HOST tensors (pinned for full PCIe rate).  Returns a dict of pinned host tensors
        (flatten_outputs keys) for the whole batch, byte-identical to the un-chunked device step.  The
        returned buffers are owned by this object and are overwritten by the next `run_host` call.

        Three streams: `up` carries only host->device copies, `run` only kernels, `down` only device->host
        copies, chained per chunk by events; device input buffers are double-buffered by chunk parity."""
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        N = x["shapes"].shape[0]
        R = self.R
        key = str(dev)
        if key not in self._streams:
            self._streams[key] = [torch.cuda.Stream(dev) for _ in range(3)]
        up, run, down = self._streams[key]
        cur = torch.cuda.current_stream(dev)
        for s in (up, run, down):
            s.wait_stream(cur)
        with torch.cuda.stream(up):
            anchors = [a.to(dev, non_blocking=True) for a in x["anchors"]]
        sets = self._device_inputs(x, dev, chunk_images)
        free_ev = [None, None]  # kernels that last read input set p have finished
        host_out = None
        pending = []
        for ci, b in enumerate(range(0, N, chunk_images)):
            e = min(b + chunk_images, N)
            n = e - b
            p = ci % 2
            bufs = sets[p]
            with torch.cuda.stream(up):
                if free_ev[p] is not None:
                    up.wait_event(free_ev[p])
                xd = {"anchors": anchors}
                for k in PER_IMAGE_KEYS:
                    v = x[k]
                    if isinstance(v, (list, tuple)):
                        xd[k] = []
                        for dst, src in zip(bufs[k], v):
                            dst[:n].copy_(src[b:e], non_blocking=True)
                            xd[k].append(dst[:n])
                    else:
                        bufs[k][:n].copy_(v[b:e], non_blocking=True)
                        xd[k] = bufs[k][:n]
                for k in PER_ROI_KEYS:
                    bufs[k][:n * R].copy_(x[k][b * R:e * R], non_blocking=True)
                    xd[k] = bufs[k][:n * R]
                up_done = torch.cuda.Event()
                up_done.record(up)
            with torch.cuda.stream(run):
                run.wait_event(up_done)
                out = self.flatten_outputs(self(xd))
                run_done = torch.cuda.Event()
                run_done.record(run)
                free_ev[p] = run_done
            with torch.cuda.stream(down):
                down.wait_event(run_done)
                if host_out is None:
                    host_out = self._host_buffers(out, N, n)
                for k, t in out.items():
                    per = t.shape[0] // n
                    host_out[k][b * per:e * per].copy_(t, non_blocking=True)
                    t.record_stream(down)  # allocated on `run`, read on `down`
            pending.append(out)
        for s in (up, run, down):
            cur.wait_stream(s)
        cur.synchronize()
        return host_out

    def _device_inputs(self, x, dev, chunk_images):
        """Two sets of device input buffers (double buffering), cached across calls."""
        def shape_sig(v):
            return tuple((tuple(t.shape[1:]), t.dtype) for t in v) if isinstance(v, (list, tuple)) \
                else (tuple(v.shape[1:]), v.dtype)
        sig = (str(dev), chunk_images, self.R) + tuple((k, shape_sig(x[k])) for k in PER_IMAGE_KEYS + PER_ROI_KEYS)
        if self._dev_in.get("sig") != sig:
            def alloc(v, rows):
                if isinstance(v, (list, tuple)):
                    return [torch.empty((rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev) for t in v]
                return torch.empty((rows,) + tuple(v.shape[1:]), dtype=v.dtype, device=dev)
            sets = []
            for _ in range(2):
                d = {k: alloc(x[k], chunk_images) for k in PER_IMAGE_KEYS}
                d.update({k: alloc(x[k], chunk_images * self.R) for k in PER_ROI_KEYS})
                sets.append(d)
            self._dev_in = {"sig": sig, "sets": sets}
        return self._dev_in["sets"]

    def _host_buffers(self, out, N, n_chunk):
        sig = tuple((k, tuple(t.shape[1:]), t.dtype, t.shape[0] // n_chunk) for k, t in out.items()) + (N,)
        if self._host_out.get("sig") != sig:
            bufs = {k: torch.empty((N * (t.shape[0] // n_chunk),) + tuple(t.shape[1:]), dtype=t.dtype, pin_memory=True)
                    for k, t in out.items()}
            self._host_out = {"sig": sig, "bufs": bufs}
        return self._host_out["bufs"]
