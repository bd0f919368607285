#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json on the Mask R-CNN R50-FPN batch-16 config.

One STEP = one pass of the post-backbone hot path over one batch of 16 synthetic 800x1333 images
(BASELINE.json configs[1]; training-time RPN settings 2000 pre / 1000 post):
    RPN proposal stage   (top-k 2000/level -> fused decode+clip -> NMS 0.7 -> per-image top-1000)
    box ROIAlign 7x7     (16,000 ROIs over P2..P5, C=256, fp32)
    Fast R-CNN post      (decode 80 classes -> clip -> score>0.05 -> class-offset NMS 0.5 -> top-100)
    mask ROIAlign 14x14  (the 1,600 detections)
Every rank of an N-GPU run processes its own batch of 16 images (images are independent: weak scaling,
no data-path collective).  `value` = ROIs pooled by all ranks / max-over-ranks step time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMAGES_PER_RANK = 16
ROIS_PER_IMAGE = 1000
DETS_PER_IMAGE = 100
PRE_NMS, POST_NMS, RPN_THR = 2000, 1000, 0.7
NUM_CLASSES = 80
SCORE_THR, NMS_THR = 0.05, 0.5
CHANNELS = 256
METRIC = "ROIAlign ROIs/s + NMS boxes/s (Mask R-CNN R50-FPN batch-16 post-backbone path)"
WORKLOAD = ("configs[1]: Mask R-CNN R50-FPN, 16 synthetic 800x1333 images/GPU: RPN 2000 pre/1000 post NMS 0.7, "
            "box ROIAlign 7x7 on 16000 ROIs, Fast R-CNN per-class NMS, mask ROIAlign 14x14 on 1600 dets")


def workload_config(world=1):
    """The `config` object of BOTH arms (GPU and --impl reference): one workload, described once."""
    n = IMAGES_PER_RANK
    return {"workload": WORKLOAD, "images_per_gpu": n, "rois_per_step_per_gpu": n * (ROIS_PER_IMAGE + DETS_PER_IMAGE),
            "cache": "inputs larger than L2 (1.46 GB features + 0.8 GB outputs per step vs 126 MB L2)",
            "sharding": "images by batch index, no collective"}


def measured_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/roofline_traffic.json; null when absent)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get("roi_align_box_7x7_dram_bytes_per_launch")
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- synthetic inputs (host, numpy)
def make_host_inputs(n_images, seed_offset=0):
    from detectron2_tensorflow_b200.utils import synthetic as syn
    anchors = syn.rpn_anchors()
    logits, deltas = syn.rpn_inputs(n_images, seed=2 + seed_offset, variant="gaussian", anchors=anchors)
    feats = syn.fpn_features(n_images, CHANNELS, seed=0 + seed_offset)
    scores, cls_deltas = syn.fast_rcnn_inputs(n_images, ROIS_PER_IMAGE, NUM_CLASSES, seed=5 + seed_offset)
    cls_deltas = (cls_deltas.reshape(-1, NUM_CLASSES, 4) * 0.5).reshape(-1, NUM_CLASSES * 4).astype(np.float32)
    return dict(anchors=anchors, logits=logits, deltas=deltas, feats=feats, scores=scores, cls_deltas=cls_deltas,
                shapes=syn.image_shapes(n_images))


def algorithmic_bytes_box_pool(n_images):
    """SURVEY.md 8(d): output write + compulsory feature read (each pixel once, never more than gathered) + boxes."""
    from detectron2_tensorflow_b200.utils import synthetic as syn
    M = n_images * ROIS_PER_IMAGE
    feat = sum(n_images * h * w * CHANNELS * 4 for h, w in (syn.level_hw(s) for s in syn.FPN_STRIDES))
    gathered = M * 7 * 7 * 4 * CHANNELS * 4
    return M * 7 * 7 * CHANNELS * 4 + min(feat, gathered) + M * 24


# --------------------------------------------------------------------------- the step through the public API
def make_engine():
    """detectron2_tensorflow_b200.engine.MaskRCNNPostBackbone: the reference-facing operators wired as
    GeneralizedRCNN.inference wires them (rcnn.py:92-144)."""
    from detectron2_tensorflow_b200.engine import MaskRCNNPostBackbone
    return MaskRCNNPostBackbone(rois_per_image=ROIS_PER_IMAGE, dets_per_image=DETS_PER_IMAGE, pre_nms_topk=PRE_NMS,
                                rpn_nms_thresh=RPN_THR, score_thresh=SCORE_THR, nms_thresh=NMS_THR)


def to_torch(host, dev=None, pin=False):
    import torch
    out = {}
    for k, v in host.items():
        def conv(a):
            t = torch.from_numpy(np.ascontiguousarray(a))
            if dev is not None:
                return t.to(dev)
            return t.pin_memory() if pin else t
        out[k] = [conv(a) for a in v] if isinstance(v, list) else conv(v)
    return out


# ROI feature rows written by --dump-outputs: 512 of 16,000 box rows (50 KB each) and 128 of 1,600 mask rows
# (200 KB each) keep the files at about 52 MB in all
DUMP_ROWS = {"box_feats": 512, "mask_feats": 128}


def dump_rows(name, n):
    """The rows of output `name` (of n rows) that --dump-outputs writes: all of them, or the same seeded sample."""
    if name not in DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS[name], replace=False))


def dump_outputs(path, outs):
    """Write what one step returned -- a list of per-image-block output dicts (torch tensors of a graphed step, or
    numpy arrays of the CPU arm), concatenated in image order -- as `path`/<name>.npy: float64 for 8-byte types,
    float32 otherwise.  The pooled ROI features are written as the same seeded sample of rows on every run, taken
    block by block, so that two builds can be compared output for output."""
    import torch
    os.makedirs(path, exist_ok=True)
    for k in outs[0]:
        rows = dump_rows(k, sum(o[k].shape[0] for o in outs))
        parts, b = [], 0
        for o in outs:
            x, n = o[k], o[k].shape[0]
            sel = rows[(rows >= b) & (rows < b + n)] - b
            parts.append(x[torch.from_numpy(sel).to(x.device)].cpu().numpy() if isinstance(x, torch.Tensor) else x[sel])
            b += n
        a = np.concatenate(parts)
        np.save(os.path.join(path, k + ".npy"), a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32))


def oracle_outputs(o):
    """cpu_step's result under the output names of the graphed step (MaskRCNNPostBackbone.flatten_outputs)."""
    (pb, pl, pv), (db, ds, dc, dv) = o["proposals"], o["dets"]
    return {"proposal_boxes": pb, "proposal_logits": pl, "proposal_valid": pv, "box_feats": o["box_feats"],
            "det_boxes": db, "det_scores": ds, "det_classes": dc, "det_valid": dv, "mask_feats": o["mask_feats"]}


def nbytes(obj):
    import torch
    if isinstance(obj, torch.Tensor):
        return obj.numel() * obj.element_size()
    if isinstance(obj, (list, tuple)):
        return sum(nbytes(o) for o in obj)
    if isinstance(obj, dict):
        return sum(nbytes(o) for o in obj.values())
    if hasattr(obj, "data") and isinstance(obj.data, dict):
        return sum(nbytes(o) for o in obj.data.values())
    return 0


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons DURING the timed region (NVML every ~2 ms; nvidia-smi fallback)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip() != ""]
            if i < len(ids) and ids[i].strip().isdigit():
                return int(ids[i])
        return i

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        bits = int(get(self.h))
        for bit, name in self.REASONS.items():
            if bits & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        o = subprocess.check_output(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                     "--format=csv,noheader,nounits"], timeout=5).decode().strip()
        f = [x.strip() for x in o.split(",")]
        self.sm.append(float(f[0]))
        self.max_mhz = float(f[1])
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
            if v == "Active":
                self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# --------------------------------------------------------------------------- CPU arm (oracle = port of the reference's TF CPU path)
def cpu_step(host, n_images, stage_s=None):
    """The same step on the CPU oracle for the first `n_images` images, following the reference's own
    data movement (decode ALL anchors, per-level pad/crop/unpermute).  `stage_s` (list of 4) accumulates
    the wall time of the four stages."""
    import oracle
    sl = slice(0, n_images)
    t = [time.perf_counter()]
    props = [oracle.rpn_predict_proposals(d[sl], a) for d, a in zip(host["deltas"], host["anchors"])]
    pb, pl, pv, pn = oracle.find_top_rpn_proposals(props, [x[sl] for x in host["logits"]], host["shapes"][sl], RPN_THR,
                                                   PRE_NMS, POST_NMS, 0.0)
    t.append(time.perf_counter())
    M = n_images * ROIS_PER_IMAGE
    idx = np.stack([np.repeat(np.arange(n_images), ROIS_PER_IMAGE), np.tile(np.arange(ROIS_PER_IMAGE), n_images)], 1)
    boxes = pb.reshape(-1, 4)
    scales = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]
    feats = [f[sl] for f in host["feats"]]
    box_feats, _ = oracle.roi_pooler(feats, scales, boxes, idx[:, 0], (7, 7), 0)
    t.append(time.perf_counter())
    pred = oracle.apply_deltas(host["cls_deltas"][:M], boxes, (10., 10., 5., 5.))
    db, ds, dc, dv, dr, dn = oracle.fast_rcnn_inference(pred, host["scores"][:M], idx, (n_images, ROIS_PER_IMAGE),
                                                        host["shapes"][sl], SCORE_THR, NMS_THR, DETS_PER_IMAGE, False)
    t.append(time.perf_counter())
    didx = np.repeat(np.arange(n_images), DETS_PER_IMAGE)
    mask_feats, _ = oracle.roi_pooler(feats, scales, db.reshape(-1, 4), didx, (14, 14), 0)
    t.append(time.perf_counter())
    if stage_s is not None:
        for i in range(4):
            stage_s[i] += t[i + 1] - t[i]
    return dict(proposals=(pb, pl, pv), box_feats=box_feats, dets=(db, ds, dc, dv), mask_feats=mask_feats)


def time_cpu(host, n_images, steps, warmup, threads=None):
    """Returns dict: ROIs/s (from the median step), seconds per step (median, mean), threads, per-stage seconds per
    step, NMS boxes entering per step, the outputs of the last step."""
    import oracle
    oracle.build()
    # all the host threads this process may use -- explicitly, because torchrun exports OMP_NUM_THREADS=1
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    oracle.set_num_threads(threads if threads else avail)
    ts = []
    stage = [0.0, 0.0, 0.0, 0.0]
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = cpu_step(host, n_images, stage if i >= warmup else None)
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
    rois = n_images * (ROIS_PER_IMAGE + DETS_PER_IMAGE)
    # boxes entering NMS on this sample: min(pre, HWA) per (image, level) + Fast R-CNN candidates
    nms_in = n_images * sum(min(PRE_NMS, a.shape[0]) for a in host["anchors"]) + \
        int((host["scores"][:n_images * ROIS_PER_IMAGE, :-1] > SCORE_THR).sum())
    med = float(np.median(ts))
    r = {"rois_per_s": rois / med, "sec_median": med, "sec_mean": float(np.mean(ts)), "threads": oracle.max_threads(),
         "stage_sec": [x / steps for x in stage], "nms_in": nms_in, "rois": rois, "outputs": out}
    oracle.set_num_threads(avail)
    return r


def cpu_baseline_dict(host, n_images, steps, warmup, sample, one_thread_images=2):
    """The CPU oracle (port of the reference's TF-CPU path) on `n_images` of the workload with every host thread
    (median of `steps` after `warmup`), plus a 1-thread leg on a smaller sample (BASELINE.md section 3).
    Returns the cpu_baseline object and time_cpu's result for all threads."""
    r = time_cpu(host, n_images, steps, warmup)
    st = r["stage_sec"]
    cb = {"value": r["rois_per_s"], "unit": "ROIs/s", "cores": r["threads"], "kind": "port", "sample": sample,
          "ms_per_step": r["sec_median"] * 1e3, "ms_per_step_mean": r["sec_mean"] * 1e3, "statistic": "median",
          "stages_ms": {"rpn_proposals": st[0] * 1e3, "box_roi_align_7x7": st[1] * 1e3, "fast_rcnn_post": st[2] * 1e3,
                        "mask_roi_align_14x14": st[3] * 1e3},
          "roi_align_rois_per_s": r["rois"] / (st[1] + st[3]),
          "nms_boxes_per_s": r["nms_in"] / (st[0] + st[2]),
          "note": "oracle/ = C restatement of the reference's TF-CPU path (TensorFlow is not installable here), "
                  "OpenMP over all host threads"}
    if one_thread_images:
        k = min(one_thread_images, n_images)
        r1 = time_cpu(host, k, 3, 1, threads=1)
        s1 = r1["stage_sec"]
        cb["one_thread"] = {"value": r1["rois_per_s"], "unit": "ROIs/s", "cores": 1,
                            "sample": f"first {k} of the {IMAGES_PER_RANK} images, median of 3 steps after 1 warm-up",
                            "ms_per_image": r1["sec_median"] * 1e3 / k,
                            "roi_align_rois_per_s": r1["rois"] / (s1[1] + s1[3]),
                            "nms_boxes_per_s": r1["nms_in"] / (s1[0] + s1[2])}
    return cb, r


def run_reference(args):
    """The reference arm: the CPU oracle (port of the reference's TF-CPU path) on the SAME config as the GPU arm --
    all 16 images per step, the same warm-up count, every host thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_img = IMAGES_PER_RANK
    host = make_host_inputs(n_img)
    steps, warmup = args.steps, max(args.warmup, 3)  # ~0.7 s of CPU per step
    cb, r = cpu_baseline_dict(host, n_img, steps, warmup,
                              f"{n_img} of {n_img} images per step, median of {steps} steps after {warmup} warm-ups")
    v, sec = r["rois_per_s"], r["sec_median"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [oracle_outputs(r["outputs"])])
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "ROIs/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "ROIs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    EMIT(json.dumps(line))


# --------------------------------------------------------------------------- GPU arm
def bind_to_gpu_numa_node(local_rank):
    """Pin this rank to the CPUs NVML reports as local to its GPU BEFORE any pinned host buffer is allocated,
    so that the H2D / D2H staging memory of the end-to-end leg lives on the GPU's own NUMA node (8 ranks on a
    two-socket host otherwise push half of their PCIe traffic through the inter-socket link)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(ClockSampler._physical_index(local_rank))
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return {"cpus_before": before, "cpus_after": len(os.sched_getaffinity(0))}
    except Exception as e:  # restricted cpusets, missing NVML: run unbound
        return {"error": type(e).__name__}


def host_path_probe(dev, world, h2d_bytes, d2h_bytes, e2e_step_s):
    """What the host<->device path of this box can carry with all `world` ranks copying at once (256 MiB pinned
    buffers, both directions concurrently, max over ranks), and how close the e2e step comes to it."""
    import torch
    import torch.distributed as dist
    n = 256 << 20
    h_in = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(n, dtype=torch.uint8, device=dev)
    d_out = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def both():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
    both()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        both()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 4
    if world > 1:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t[0])
    duplex = n / dt / 1e9  # GB/s per rank in EACH direction with every rank copying both ways
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
    torch.cuda.synchronize()
    du = (time.perf_counter() - t0) / 4
    if world > 1:
        t = torch.tensor([du], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        du = float(t[0])
    uni = n / du / 1e9  # GB/s per rank, uploads only
    # two lower bounds of the copy time of a step: the ranks share the host-memory / PCIe path (total bytes at the
    # both-directions rate), and the longer direction cannot go faster than a one-directional stream
    floor_s = max((h2d_bytes + d2h_bytes) / (2.0 * duplex * 1e9), max(h2d_bytes, d2h_bytes) / (uni * 1e9))
    frac = floor_s / e2e_step_s
    return {"duplex_GBps_per_rank_each_direction": duplex, "aggregate_GBps_each_direction": duplex * world,
            "h2d_only_GBps_per_rank": uni,
            "copy_floor_ms_per_step": floor_s * 1e3, "e2e_over_copy_floor": e2e_step_s / floor_s,
            "limiter": ("host<->device copies of this box: the e2e step runs at %.0f %% of what %d rank(s) copying in "
                        "both directions at once can move (measured in this run)" % (100.0 * frac, world))}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from detectron2_tensorflow_b200 import _native as nv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # (N=1 stays unbound: the cpu_baseline leg of the same process must see every host core)
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"skipped": "single rank"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nv.lib()

    n = IMAGES_PER_RANK
    host = make_host_inputs(n, seed_offset=0)
    x = to_torch(host, dev=dev)
    hp = make_engine()
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing, (1) eager single stream with per-stage CUDA events: stage breakdown + roofline
    for _ in range(W):
        out = hp(x)
    barrier()
    Ks = max(3, min(K, 30))
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(Ks)]
    barrier()
    for s in range(Ks):
        out = hp(x, evs[s])
    barrier()
    eager_ms = evs[0][0].elapsed_time(evs[-1][4]) / Ks
    stage = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in evs])  # rpn, boxpool, frcnn, maskpool
    st = stage.mean(0)

    # ---- (2) the timed region: the same step captured as ONE CUDA graph (4 image blocks on concurrent streams:
    # images are independent; latency-bound proposal / post-processing kernels overlap the HBM-bound ROIAlign),
    # and `--in-flight` such graphs replayed round-robin on their own streams so that consecutive (independent)
    # steps overlap as well.  Every step does all of its work; K steps are timed as a whole.
    pipe = hp.pipeline(x, chunks=args.chunks, depth=args.in_flight)
    gstep = pipe.steps[0]
    for _ in range(W):
        gstep.replay()
    barrier()
    lat = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    lat[0].record()
    for _ in range(10):
        gstep.replay()  # one graph at a time: the latency of a single step
    lat[1].record()
    barrier()
    step_latency_ms = lat[0].elapsed_time(lat[1]) / 10
    pipe.run(2 * args.in_flight)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    last = pipe.run(K)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    launches = gstep.kernels_per_replay * K
    clocks = sampler.summary()
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    if world > 1:
        t = torch.tensor([dev_ms, wall * 1e3, eager_ms, step_latency_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, eager_ms, step_latency_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    else:
        wall_ms = wall * 1e3
    ms_per_step = dev_ms / K  # CUDA events on the launching stream, max over ranks
    rois_rank = n * (ROIS_PER_IMAGE + DETS_PER_IMAGE)
    value = rois_rank * world / (ms_per_step * 1e-3)

    # NMS bookkeeping: boxes entering NMS (RPN segments + Fast R-CNN candidates), counted by the kernels
    from detectron2_tensorflow_b200.modeling.proposal_generator import rpn_outputs as ro
    r = ro._rpn_call([t_.reshape(n, -1) for t_ in x["logits"]], None, x["deltas"], x["anchors"], x["shapes"], RPN_THR,
                     PRE_NMS, POST_NMS, 0.0, count_nms_in=True)
    rpn_nms_in = int(r.get_tracking("nms_boxes_in").item())
    cand = int((x["scores"][:, :-1] > SCORE_THR).sum().item())

    hbm_peak, peak_src = peaks()
    alg = algorithmic_bytes_box_pool(n)
    ach = alg / (st[1] * 1e-3) / 1e9
    traffic = measured_traffic()
    roofline = {"kernel": "roi_align_kernel<float,float,2> (box pooler 7x7, 16000 ROIs)", "bound": "hbm",
                "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": alg, "peak_source": peak_src, "kernel_ms": float(st[1]),
                "traffic_source": "profiles/roofline_traffic.json (ncu capture of the same launch of the same binary; "
                                  "constant, not re-measured in this run)",
                "note": "frac uses SURVEY 8(d)'s algorithmic bytes (whole pyramid read once), which over-count: 1,000 "
                        "ROIs/image touch about 2/3 of the pyramid.  frac_on_traffic = DRAM bytes actually moved / "
                        "kernel time / peak is the honest distance from the HBM roofline."}
    if traffic:
        roofline["achieved_on_traffic"] = traffic / (st[1] * 1e-3) / 1e9
        roofline["frac_on_traffic"] = roofline["achieved_on_traffic"] / hbm_peak
    line = {
        "metric": METRIC, "value": value, "unit": "ROIs/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(world),
        "wall_ms_per_step": wall_ms / K,
        "execution": {"timed_region": f"one CUDA graph per step ({args.chunks} image blocks on concurrent streams), "
                                      f"{args.in_flight} steps in flight on alternating streams",
                      "steps_in_flight": args.in_flight,
                      "kernels_per_step": gstep.kernels_per_replay,
                      "single_step_latency_ms": step_latency_ms,
                      "value_one_step_at_a_time": rois_rank * world / (step_latency_ms * 1e-3),
                      "eager_single_stream_ms_per_step": eager_ms,
                      "note": "ms_per_step = time of the K timed steps / K (throughput; consecutive steps are "
                              "independent batches and overlap); single_step_latency_ms = one graph replay at a time; "
                              "stages_ms and roofline come from the eager single-stream run (CUDA events between "
                              "stages on the launching stream)"},
        "stages_ms": {"rpn_proposals": st[0], "box_roi_align_7x7": st[1], "fast_rcnn_post": st[2],
                      "mask_roi_align_14x14": st[3]},
        "roi_align": {"rois_per_s": rois_rank * world / ((st[1] + st[3]) * 1e-3), "unit": "ROIs/s"},
        "nms": {"boxes_per_s": (rpn_nms_in + cand) * world / ((st[0] + st[2]) * 1e-3), "unit": "boxes/s",
                "boxes_in_per_step_per_gpu": rpn_nms_in + cand,
                "note": "boxes entering NMS / time of the full proposal + Fast R-CNN post stages"},
        "roofline": roofline,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }

    # ---- strong scaling of the fixed 16-image batch (north_star / SURVEY 8e), gather to rank 0 timed
    pipe.run(2 * args.in_flight)
    barrier()
    if world > 1:
        try:
            line["strong"] = strong_scaling(hp, x, dev, world, rank, K, W, args.chunks, args.strong_in_flight, gstep,
                                            step_latency_ms, ms_per_step, transport="peer")
        except Exception as e:  # noqa: BLE001
            line["strong"] = {"error": repr(e)[:300]}
        barrier()
        try:  # the library-collective route beside it (what the peer-memory kernels replace)
            nccl = strong_scaling(hp, x, dev, world, rank, K, W, args.chunks, args.strong_in_flight, gstep,
                                  step_latency_ms, ms_per_step, transport="nccl")
            line["strong_nccl"] = {k: nccl[k] for k in ("transport", "ms_per_step", "speedup_vs_1gpu", "gather_ms",
                                                        "pipelined_ms_per_step", "pipelined_speedup_vs_1gpu",
                                                        "gathered_identical_to_1gpu")}
        except Exception as e:  # noqa: BLE001
            line["strong_nccl"] = {"error": repr(e)[:300]}
    else:
        line["strong"] = {"global_batch": n, "images_per_rank": [n], "ms_per_step": step_latency_ms,
                          "speedup_vs_1gpu": 1.0, "gather_ms": 0.0, "pipelined_ms_per_step": ms_per_step,
                          "pipelined_speedup_vs_1gpu": 1.0,
                          "note": "1 GPU: the whole batch on one rank, results already on rank 0 (no gather); "
                                  "ms_per_step = one graphed step at a time"}
    if args.no_e2e:
        if rank == 0:
            EMIT(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- end-to-end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region
    hx = to_torch(host, dev=None, pin=True)
    for _ in range(2):
        ho = hp.run_host(hx, dev)
    barrier()
    Ke = max(3, min(K, 10))
    t0 = time.perf_counter()
    for _ in range(Ke):
        ho = hp.run_host(hx, dev)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    h2d = sum(nbytes(hx[k]) for k in ("feats", "logits", "deltas", "anchors", "scores", "cls_deltas", "shapes"))
    d2h = nbytes(ho)
    del ho
    host_path = host_path_probe(dev, world, h2d, d2h, e2e_s / Ke)
    line["e2e"] = {"value": rois_rank * world / (e2e_s / Ke), "unit": "ROIs/s", "ms_per_step": e2e_s / Ke * 1e3,
                   "host_path": host_path, "limiter": host_path["limiter"],
                   "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": Ke,
                   "host_numa_binding": numa,
                   "note": "MaskRCNNPostBackbone.run_host: pinned host tensors in, pinned host tensors out (all "
                           "inputs uploaded and all four outputs downloaded every step), 2-image chunks pipelined "
                           "over three CUDA streams (upload / kernels / download)"}

    # ---- the other BASELINE.json configs (parity-test cases, not bench lines): device-resident timings, N=1 only
    if not args.no_extras:
        del hx, x, pipe, gstep, out
        torch.cuda.empty_cache()
        oc = {}
        if world == 1:
            try:
                oc["configs[0] Faster R-CNN R50-FPN post-backbone ops, 1 image"] = config0_single_image(dev, cpu=not args.no_cpu)
            except Exception as e:  # noqa: BLE001  (informational leg: never fails the bench line)
                oc["configs[0]"] = {"error": repr(e)[:200]}
            try:
                oc.update(other_configs(dev, cpu=not args.no_cpu))
            except Exception as e:  # noqa: BLE001
                oc["configs[2..3]"] = {"error": repr(e)[:200]}
        try:
            oc["configs[4] ROIAlign / NMS sweep 256..65536"] = config4_sweep(dev, world, rank, cpu=not args.no_cpu)
        except Exception as e:  # noqa: BLE001
            oc["configs[4]"] = {"error": repr(e)[:200]}
        line["other_configs"] = oc

    # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload
    if world == 1 and not args.no_cpu:
        cb, _ = cpu_baseline_dict(host, n, 10, 2, f"{n} of {n} images per step, median of 10 steps after 2 warm-ups")
        line["cpu_baseline"] = cb
    if rank == 0:
        EMIT(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def strong_scaling(hp, x, dev, world, rank, K, W, chunks, in_flight, full_step, full_latency_ms, full_pipe_ms,
                   transport="peer"):
    """SURVEY.md 8(e) / north_star: the FIXED batch of 16 images partitioned by image index over the ranks, no
    collective on the path, and the fixed-size padded results (proposals + detections) gathered to rank 0 with one
    grouped send/recv over NVLink inside the timed region.  Every rank holds the same seeded global batch and cuts
    its own block.  Returns the `strong` object of the bench line (rank 0's view; times are max over ranks)."""
    import torch
    import torch.distributed as dist
    from detectron2_tensorflow_b200 import sharding
    from detectron2_tensorflow_b200.engine import GATHER_KEYS
    n = IMAGES_PER_RANK
    R = ROIS_PER_IMAGE
    b, e = sharding.image_block(n, world, rank)
    xl = {"anchors": x["anchors"], "shapes": x["shapes"][b:e].contiguous(), "scores": x["scores"][b * R:e * R].contiguous(),
          "cls_deltas": x["cls_deltas"][b * R:e * R].contiguous()}
    for k in ("logits", "deltas", "feats"):
        xl[k] = [t[b:e].contiguous() for t in x[k]]
    chunks_of = lambda k: max(1, min(chunks, k // 2))
    layout = sharding.block_layout(n, world, chunks_of)
    # one GatherPlan per graphed step: its pack() is captured inside the step's graph, its unpack() is a graph of
    # its own on rank 0, so a step costs two graph launches + one NCCL gather on the host
    spec = hp.gather_spec()
    peer = transport == "peer"
    if peer:
        # NVLink peer memory: the pack kernel captured in the step graph stores the block straight into rank 0's
        # receive slot and raises a flag; rank 0's unpack kernel waits for the flags (sharding.PeerGatherPlan)
        plans = [sharding.PeerGatherPlan(spec, layout, dev, timeout_ms=5000) for _ in range(in_flight)]
    else:
        plans = [sharding.GatherPlan(spec, layout, dev) for _ in range(in_flight)]
    pipe = hp.pipeline(xl, chunks=chunks_of(e - b), depth=in_flight,
                       epilogues=[(lambda outs, p=p: p.pack([{k: o[k] for k in GATHER_KEYS} for o in outs])) for p in plans],
                       epilogue_warmup=not peer)
    g0 = pipe.steps[0]
    assert [(b + lb, b + le) for lb, le in g0.bounds] == layout[rank]
    unpack_graphs = []
    if rank == 0:
        for p in plans:
            if not peer:
                p.unpack()
                torch.cuda.synchronize()
            ug = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ug):
                p.unpack()
            unpack_graphs.append(ug)
    pack_only = None
    if peer:  # the gather alone = this rank's pack kernel (+ rank 0's unpack): its own small graph over g0's outputs
        pack_only = torch.cuda.CUDAGraph()
        with torch.cuda.graph(pack_only):
            plans[0].pack([{k: o[k] for k in GATHER_KEYS} for o in g0.outputs])
    step_plan = {id(st): (plans[i], unpack_graphs[i] if rank == 0 else None) for i, st in enumerate(pipe.steps)}

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def gather(step):
        plan, ug = step_plan[id(step)]
        plan.gather()
        if ug is not None:
            ug.replay()
        return plan.out

    barrier()  # captures take different times on different ranks: start the hand-shaking steps together
    for _ in range(W):
        g0.replay()
        full = gather(g0)
    barrier()
    # byte identity of the gathered results with the 1-GPU run of the whole batch (rank 0's own full-batch graph)
    identical = None
    if rank == 0:
        want = full_step.gathered(GATHER_KEYS)
        identical = all(torch.equal(full[k], want[k]) for k in GATHER_KEYS)
    # (1) latency: one step at a time, gather inside
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    barrier()
    ev[0].record()
    for _ in range(K):
        g0.replay()
        gather(g0)
    ev[1].record()
    barrier()
    lat_ms = ev[0].elapsed_time(ev[1]) / K
    # (2) the gather alone
    barrier()
    ev[2].record()
    for _ in range(K):
        if pack_only is not None:
            pack_only.replay()
        gather(g0)
    ev[3].record()
    barrier()
    gather_ms = ev[2].elapsed_time(ev[3]) / K
    # (3) throughput: `in_flight` graphed steps on alternating streams, each followed by its gather
    cur = torch.cuda.current_stream(dev)

    def run_pipe(k):
        start = torch.cuda.Event()
        start.record(cur)
        for s_ in pipe.streams:
            s_.wait_event(start)
        for i in range(k):
            j = i % len(pipe.steps)
            with torch.cuda.stream(pipe.streams[j]):
                pipe.steps[j].replay()
                gather(pipe.steps[j])
        for s_ in pipe.streams:
            cur.wait_stream(s_)
    run_pipe(2 * in_flight)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    run_pipe(K)
    p1.record()
    barrier()
    pipe_ms = p0.elapsed_time(p1) / K
    t = torch.tensor([lat_ms, gather_ms, pipe_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    lat_ms, gather_ms, pipe_ms = (float(v) for v in t)
    rois = n * (ROIS_PER_IMAGE + DETS_PER_IMAGE)
    if peer:
        for p in plans:
            p.check()  # a timed-out flag wait is an error, not a slow step
    # the gathered results after the pipelined run too
    if rank == 0:
        last = step_plan[id(pipe.steps[(K - 1) % len(pipe.steps)])][0].out
        identical = bool(identical and all(torch.equal(last[k], want[k]) for k in GATHER_KEYS))
    kernels_gather = (1 + (1 if rank == 0 else 0)) if peer else None
    del unpack_graphs, pack_only, pipe
    if peer:
        for p in plans:
            p.close()
    return {"transport": ("NVLink peer memory: 1 pack kernel per rank (remote stores + flag) + 1 unpack kernel on rank 0 "
                          "(csrc/peer.cu)") if peer else "NCCL (one collective per step + packed copies)",
            "gather_kernels_rank0": kernels_gather,
            "global_batch": n, "images_per_rank": [sharding.image_block(n, world, r)[1] - sharding.image_block(n, world, r)[0]
                                                   for r in range(world)],
            "ms_per_step": lat_ms, "rois_per_s": rois / (lat_ms * 1e-3),
            "one_gpu_ms_per_step": full_latency_ms, "speedup_vs_1gpu": full_latency_ms / lat_ms,
            "gather_ms": gather_ms, "gather_bytes_per_rank": int(sum(nbytes(v) for v in g0.gathered(GATHER_KEYS).values())),
            "pipelined_ms_per_step": pipe_ms, "one_gpu_pipelined_ms_per_step": full_pipe_ms,
            "pipelined_speedup_vs_1gpu": full_pipe_ms / pipe_ms, "pipelined_rois_per_s": rois / (pipe_ms * 1e-3),
            "gathered_identical_to_1gpu": identical, "kernels_per_step_per_rank": g0.kernels_per_replay,
            "note": "the fixed 16-image batch split by image index; ms_per_step = graph replay of the rank's block "
                    "(with the pack of proposals + detections captured inside it) + the transport + rank 0's unpack "
                    "graph, one step at a time, max over ranks (CUDA events); one_gpu_* = the same measurement of the "
                    "whole batch on one GPU in this run (no gather needed); pipelined_* = several steps in flight on "
                    "alternating streams"}


def config0_single_image(dev, iters=20, cpu=True):
    """BASELINE.json configs[0]: Faster R-CNN R50-FPN inference post-backbone ops on ONE 800x1333 image (test-time
    RPN settings 1000 pre / 1000 post, 1000 ROIs 7x7, Fast R-CNN per-class NMS; rcnn.py:92-144): the latency regime."""
    import torch
    from detectron2_tensorflow_b200.engine import MaskRCNNPostBackbone
    pre = post = 1000
    host = make_host_inputs(1)
    x = to_torch(host, dev=dev)
    hp = MaskRCNNPostBackbone(rois_per_image=post, dets_per_image=DETS_PER_IMAGE, pre_nms_topk=pre, rpn_nms_thresh=RPN_THR,
                              score_thresh=SCORE_THR, nms_thresh=NMS_THR, mask_on=False)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def med(fn, cold):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            if cold:
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))
    g = hp.capture(x, chunks=1)
    r = {"workload": "1 image: RPN top-k 1000/level + NMS 0.7 -> 1000 proposals, ROIAlign 7x7 on 1000 ROIs, Fast R-CNN "
                     "per-class NMS -> 100 detections",
         "eager_ms_cold_l2": med(lambda: hp(x), True), "eager_ms_warm": med(lambda: hp(x), False),
         "graph_ms_cold_l2": med(g.replay, True), "graph_ms_warm": med(g.replay, False),
         "kernels_per_step": g.kernels_per_replay}
    r["rois_per_s"] = post / (r["graph_ms_cold_l2"] * 1e-3)
    r["images_per_s"] = 1e3 / r["graph_ms_cold_l2"]
    if cpu:
        import oracle
        avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

        def cpu_once():
            props = [oracle.rpn_predict_proposals(d, a) for d, a in zip(host["deltas"], host["anchors"])]
            pb, _, _, _ = oracle.find_top_rpn_proposals(props, host["logits"], host["shapes"], RPN_THR, pre, post, 0.0)
            idx = np.stack([np.zeros(post, np.int64), np.arange(post)], 1)
            boxes = pb.reshape(-1, 4)
            oracle.roi_pooler(host["feats"], [1 / 4., 1 / 8., 1 / 16., 1 / 32.], boxes, idx[:, 0], (7, 7), 0)
            pred = oracle.apply_deltas(host["cls_deltas"][:post], boxes, (10., 10., 5., 5.))
            oracle.fast_rcnn_inference(pred, host["scores"][:post], idx, (1, post), host["shapes"], SCORE_THR, NMS_THR,
                                       DETS_PER_IMAGE, False)
        for thr in (avail, 1):
            oracle.set_num_threads(thr)
            cpu_once()
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                cpu_once()
                ts.append(time.perf_counter() - t0)
            ms = float(np.median(ts)) * 1e3
            r[f"cpu_oracle_{'all' if thr == avail else 'one'}_thread{'s' if thr == avail else ''}"] = {
                "ms": ms, "cores": thr, "rois_per_s": post / (ms * 1e-3), "gpu_over_cpu": ms / r["graph_ms_cold_l2"],
                "sample": "the whole config (1 image), median of 5 after 1 warm-up"}
        oracle.set_num_threads(avail)
    return r


def config4_sweep(dev, world=1, rank=0, iters=10, cpu=True):
    """BASELINE.json configs[4]: ROIAlign / NMS microbenchmark sweep, 256 .. 65536 ROIs / boxes, C=256, FPN P2-P5
    maps of 16 images, L2 flushed between iterations, CPU oracle beside each point.  Under --gpus N the M ROIs /
    the 16 NMS segments are partitioned by image / segment index over the ranks (time = max over ranks)."""
    import torch
    import torch.distributed as dist
    from detectron2_tensorflow_b200 import sharding
    from detectron2_tensorflow_b200.layers import batch_nms
    from detectron2_tensorflow_b200.modeling import ROIPooler
    from detectron2_tensorflow_b200.structures import BoxList, SparseBoxList
    from detectron2_tensorflow_b200.utils import synthetic as syn
    hbm_peak, _ = peaks()
    N, C = 16, CHANNELS
    b0, e0 = sharding.image_block(N, world, rank)
    nl = e0 - b0
    g = torch.Generator(device=dev).manual_seed(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    feats = [torch.randn((nl,) + syn.level_hw(s_) + (C,), device=dev, generator=g) for s_ in syn.FPN_STRIDES]
    scales = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]

    def med(fn, it=iters):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(it):
            flush.zero_()
            if world > 1:
                dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = float(np.median(ts))
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    do_cpu = cpu and world == 1
    if do_cpu:
        import oracle
        oracle.set_num_threads(avail)
        hfeats = [f.cpu().numpy() for f in feats]
    pooler = ROIPooler(7, scales, 0, "ROIAlignV2")
    fbytes_all = sum(N * h * w * C * 4 for h, w in (syn.level_hw(s_) for s_ in syn.FPN_STRIDES))
    roi_pts, nms_pts = [], []
    for M in (256, 1024, 4096, 16384, 65536):
        boxes, idx = syn.rois(N, M // N, seed=1)
        sel = (idx[:, 0] >= b0) & (idx[:, 0] < e0)
        lb, li = boxes[sel], idx[sel].copy()
        li[:, 0] -= b0
        inst = SparseBoxList(torch.from_numpy(li).to(dev), BoxList(torch.from_numpy(lb).to(dev)), (nl, M // N))
        ms = med(lambda: pooler(feats, inst))
        alg = M * 49 * C * 4 + min(fbytes_all, M * 49 * 4 * C * 4) + M * 24
        pt = {"rois": M, "ms": ms, "rois_per_s": M / ms * 1e3, "alg_GBps": alg / ms / 1e6,
              "frac_hbm": alg / ms / 1e6 / hbm_peak / world}
        if do_cpu:
            Mc = min(M, 16384)  # bounded sample of the larger points
            t0 = time.perf_counter()
            oracle.roi_pooler(hfeats, scales, boxes[:Mc], idx[:Mc, 0], (7, 7), 0)
            dt = time.perf_counter() - t0
            pt["cpu_oracle"] = {"rois_per_s": Mc / dt, "cores": avail, "sample": f"first {Mc} ROIs, one pass",
                                "gpu_over_cpu": (M / ms * 1e3) / (Mc / dt)}
        roi_pts.append(pt)
    del feats
    rng = np.random.default_rng(5)
    S = 16  # segments (one per image), partitioned like the images
    for n in (256, 1024, 4096, 16384, 65536):
        cy, cx = rng.uniform(0, 800, (S, n)), rng.uniform(0, 1333, (S, n))
        h, w = rng.uniform(16, 300, (S, n)), rng.uniform(16, 300, (S, n))
        hb = np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], 2).astype(np.float32)
        hs = rng.standard_normal((S, n)).astype(np.float32)
        pt = {"boxes_per_segment": n}
        for label, segs, cap in (("one_segment_uncapped", 1, n), ("sixteen_segments_cap1000", S, min(n, 1000))):
            if segs == 1 and rank != 0:
                continue
            sb, se = (0, 1) if segs == 1 else (b0, e0)
            tb = torch.from_numpy(hb[sb:se]).to(dev)
            tsc = torch.from_numpy(hs[sb:se]).to(dev)
            if segs == 1 and world > 1:  # a single segment does not shard: rank 0 only, no barrier
                for _ in range(3):
                    batch_nms(tb, tsc, cap, axis=1, iou_threshold=0.7)
                torch.cuda.synchronize()
                ts = []
                for _ in range(5):
                    flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    batch_nms(tb, tsc, cap, axis=1, iou_threshold=0.7)
                    b.record()
                    torch.cuda.synchronize()
                    ts.append(a.elapsed_time(b))
                ms = float(np.median(ts))
            elif segs == 1:
                ms = med(lambda: batch_nms(tb, tsc, cap, axis=1, iou_threshold=0.7), 5)
            else:
                ms = med(lambda: batch_nms(tb, tsc, cap, axis=1, iou_threshold=0.7), 5)
            pt[label] = {"ms": ms, "boxes_per_s": segs * n / ms * 1e3, "max_output_size": cap}
            if do_cpu:
                k = 1 if segs == 1 else (S if n <= 4096 else 2)  # bounded sample of the big multi-segment points
                t0 = time.perf_counter()
                oracle.batch_nms(hb[:k], hs[:k], cap, 0.7)
                dt = time.perf_counter() - t0
                pt[label]["cpu_oracle"] = {"boxes_per_s": k * n / dt, "cores": min(avail, k), "sample": f"{k} segment(s), one pass",
                                           "gpu_over_cpu": (segs * n / ms * 1e3) / (k * n / dt)}
        nms_pts.append(pt)
    return {"roi_align_7x7_sweep": roi_pts, "nms_sweep_thr0.7": nms_pts, "n_gpus": world,
            "note": "16 images' P2-P5 maps, C=256, fp32; L2 flushed (256 MB write) before every timed iteration; median; "
                    "under --gpus N the ROIs (with their images) and the 16 NMS segments are split by index over the ranks "
                    "and the time is the max over ranks; `one_segment` cannot shard and runs on rank 0"}


def other_configs(dev, iters=10, cpu=True):
    """configs[2] (RetinaNet post-processing, batch 32) and configs[3] (SOLOv2: Matrix-NMS over 500 candidates at 1/4
    resolution, batch 16, plus the steps either side of it), inputs resident, CUDA events, median of `iters` after 3
    warm-ups; inputs (2 GB each) are larger than L2.  Informational: a failure is recorded, it does not fail the bench."""
    import torch
    from detectron2_tensorflow_b200.layers import matrix_nms
    from detectron2_tensorflow_b200.modeling import (RetinaNetInference, SOLOv2Inference, solo_dynamic_masks,
                                                     solo_upsample_masks)
    from detectron2_tensorflow_b200.utils import synthetic as syn
    out = {}
    g = torch.Generator(device=dev).manual_seed(0)

    def med(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))
    try:
        N, K = 32, 80
        anchors = [torch.from_numpy(a).to(dev) for a in syn.retinanet_anchors()]
        cls = [torch.randn((N, a.shape[0], K), device=dev, generator=g) * 1.5 - 4.6 for a in anchors]
        dl = [torch.randn((N, a.shape[0], 4), device=dev, generator=g) * 0.3 for a in anchors]
        head = RetinaNetInference(num_classes=K)
        ms = med(lambda: head.inference(cls, dl, anchors))
        nsc = sum(c.numel() for c in cls)
        r2 = {"ms": ms, "images_per_s": N / ms * 1e3, "logit_GB": nsc * 4 / 1e9, "single_read_GBps": nsc * 4 / ms / 1e6}
        if cpu:  # the oracle (port of the reference's TF-CPU path) on 2 of the 32 images, all host threads
            import oracle
            hc = [c[:2].cpu().numpy() for c in cls]
            hd = [d[:2].cpu().numpy() for d in dl]
            ha = [a.cpu().numpy() for a in anchors]
            t0 = time.perf_counter()
            oracle.retinanet_inference(hc, hd, ha, K, 1000, 0.05, 0.5, 100)
            dt = time.perf_counter() - t0
            r2["cpu_oracle"] = {"images_per_s": 2 / dt, "cores": oracle.max_threads(), "sample": "2 of the 32 images, one pass",
                                "gpu_over_cpu": (N / ms * 1e3) / (2 / dt)}
        out["configs[2] RetinaNet R50-FPN post-processing, batch 32"] = r2
        del cls, dl, anchors
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["configs[2]"] = {"error": repr(e)[:200]}
    try:
        B, n, H, W, E = 16, 500, 200, 336, 256
        m, c, s = syn.solo_masks(n, hw=(H, W), seed=7)
        masks = torch.from_numpy(m).to(dev)[None].repeat(B, 1, 1, 1).contiguous()
        classes = torch.from_numpy(c).to(dev)[None].repeat(B, 1).contiguous()
        scores = torch.from_numpy(s).to(dev)[None].repeat(B, 1).contiguous()
        ms = med(lambda: matrix_nms(masks, classes, scores))
        by = masks.numel() * 4
        r = {"matrix_nms_fp32_masks_ms": ms, "matrix_nms_images_per_s": B / ms * 1e3, "mask_read_GBps": by / ms / 1e6}
        if cpu:  # the oracle's matrix_nms (lib/layers/nms.py:29-83 restated) on ONE image's 500 masks, all host threads
            import oracle
            t0 = time.perf_counter()
            oracle.matrix_nms(m, c, s, None, "gaussian", 2.0)
            dt = time.perf_counter() - t0
            r["matrix_nms_cpu_oracle"] = {"images_per_s": 1 / dt, "cores": oracle.max_threads(),
                                          "sample": "1 of the 16 images (500 masks), one pass",
                                          "gpu_over_cpu": (B / ms * 1e3) * dt}
        del masks
        torch.cuda.empty_cache()
        feat = torch.randn((B, H, W, E), device=dev, generator=g)
        kern = torch.randn((B, n, E), device=dev, generator=g) / 16
        ms = med(lambda: solo_dynamic_masks(feat, kern))
        r.update(dynamic_conv_plus_mask_stage_ms=ms, tf32_mma_tflops_issued=3 * 2.0 * B * n * H * W * E / ms / 1e9)
        head = SOLOv2Inference(0.5, 500, "gaussian", 2.0, 0.05, 100)
        strides = torch.full((B, n), 8.0, device=dev)
        ms = med(lambda: head.postprocess(None, scores, classes, strides, return_masks=False, mask_features=feat,
                                          mask_kernels=kern))
        r.update(inference_tail_from_features_ms=ms, inference_tail_images_per_s=B / ms * 1e3)
        obj = np.stack([syn.solo_masks(100, hw=(H, W), seed=70 + i)[0] for i in range(B)]).reshape(B, 100, -1).astype(np.uint8)
        obj = np.concatenate([obj, np.zeros((B, 100, (-obj.shape[-1]) % 64), np.uint8)], -1)
        kept = torch.from_numpy(np.packbits(obj, axis=-1, bitorder="little").view(np.int64)).to(dev)
        ms = med(lambda: solo_upsample_masks(kept, (H, W), (800, 1333), 0.5, False))
        r.update(image_masks_and_boxes_ms=ms, image_mask_write_GBps=B * 100 * 800 * 1333 / ms / 1e6)
        # the whole MaskKernelBranch.inference from the head outputs (about 500 cells x classes above the threshold)
        grids = (40, 36, 24, 16, 12)
        probs = [torch.where(torch.rand((B, g_, g_, 80), device=dev, generator=g) < 0.0016,
                             torch.rand((B, g_, g_, 80), device=dev, generator=g) * 0.8 + 0.15, torch.zeros((), device=dev))
                 for g_ in grids]
        kerns = [torch.randn((B, g_, g_, E), device=dev, generator=g) / 16 for g_ in grids]
        full = SOLOv2Inference(0.5, 500, "gaussian", 2.0, 0.05, 100, score_threshold=0.1, num_grids=grids,
                               strides=(8, 8, 16, 32, 32), max_candidates=1024)
        # object-like masks (one blob per candidate, like a trained head): channel 0 is a bias, every other channel a
        # Gaussian bump; a candidate's kernel picks one bump (+8) against the bias (-4) -> a disk of radius ~1.2 sigma
        yy = torch.arange(H, device=dev, dtype=torch.float32)[None, :, None, None]
        xx = torch.arange(W, device=dev, dtype=torch.float32)[None, None, :, None]
        cy = torch.rand((B, 1, 1, E), device=dev, generator=g) * H
        cx = torch.rand((B, 1, 1, E), device=dev, generator=g) * W
        sg = torch.rand((B, 1, 1, E), device=dev, generator=g) * 35 + 5
        sfeat = torch.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * sg * sg)).contiguous()
        sfeat[..., 0] = 1.0
        for k_ in kerns:
            k_.mul_(0.01)
            pick = torch.randint(1, E, k_.shape[:-1] + (1,), device=dev, generator=g)
            k_.scatter_(-1, pick, 8.0)
            k_[..., 0] = -4.0
        ms = med(lambda: full.inference(probs, kerns, sfeat, (800, 1333)))
        res = full.inference(probs, kerns, sfeat, (800, 1333))
        r["full_inference_mask_coverage"] = float(res["pred_masks"].float().mean())
        r.update(full_inference_from_head_outputs_ms=ms, full_inference_images_per_s=B / ms * 1e3,
                 full_inference_candidates_per_image=float(res["num_candidates"].float().mean()),
                 full_inference_detections_per_image=float(res["num"].float().mean()))
        out["configs[3] SOLOv2 R50: 500 candidates at 200x336, batch 16"] = r
    except Exception as e:  # noqa: BLE001
        out["configs[3]"] = {"error": repr(e)[:200]}
    return out


def _protect_stdout():
    """Libraries (NCCL's version banner, torchrun warnings) may write to fd 1; the contract is ONE JSON line on
    stdout.  Point fd 1 at stderr for the duration of the run and hand back a writer for the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w", buffering=1)

    def emit(line):
        os.write(real, (line + "\n").encode())
    return emit


EMIT = print


def main():
    global EMIT
    EMIT = _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="d2b200", choices=["d2b200", "reference"])
    ap.add_argument("--chunks", type=int, default=4, help="image blocks run concurrently inside the graphed step")
    ap.add_argument("--in-flight", type=int, default=4, dest="in_flight",
                    help="graphed steps replayed concurrently on alternating streams (1 = strictly one after another)")
    ap.add_argument("--strong-in-flight", type=int, default=6, dest="strong_in_flight",
                    help="graphed steps in flight in the strong-scaling leg (small per-rank blocks: more steps overlap)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", dest="no_extras",
                    help="skip the device timings of the other BASELINE.json configs (other_configs key)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, about 52 MB; "
                         "a fixed sample of the pooled ROI feature rows); both arms write the same names")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
