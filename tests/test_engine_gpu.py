"""GPU: the post-backbone engine (RPN -> box pooler -> Fast R-CNN post -> mask pooler) against the oracle,
and the pipelined host-buffer path against the device-resident path (byte-identical, any chunking)."""
import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200.engine import MaskRCNNPostBackbone
from detectron2_tensorflow_b200.utils import synthetic as syn

pytestmark = pytest.mark.gpu


def _inputs(N, R, K, C, padded=(160, 224), seed=0):
    rng = np.random.default_rng(seed)
    anchors = syn.rpn_anchors(padded_hw=padded)
    logits = [(rng.standard_normal((N, a.shape[0])) * 2).astype(np.float32) for a in anchors]
    deltas = [(rng.standard_normal((N, a.shape[0], 4)) * 0.3).astype(np.float32) for a in anchors]
    feats = syn.fpn_features(N, C, padded_hw=padded, seed=seed)
    sc = rng.uniform(0, 1, (N * R, K + 1)).astype(np.float32) ** 4
    sc /= sc.sum(1, keepdims=True)
    cd = (rng.standard_normal((N * R, K * 4)) * 0.5).astype(np.float32)
    shapes = np.tile(np.array([[150, 210]], np.int32), (N, 1))
    return dict(anchors=anchors, logits=logits, deltas=deltas, feats=feats, scores=sc, cls_deltas=cd, shapes=shapes)


def _t(host, dev=None):
    conv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)) if dev is not None else \
        (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory())
    return {k: [conv(a) for a in v] if isinstance(v, list) else conv(v) for k, v in host.items()}


def test_engine_matches_oracle_and_host_path(cuda, oracle_lib):
    N, R, D, K, C = 5, 48, 12, 6, 16
    host = _inputs(N, R, K, C)
    eng = MaskRCNNPostBackbone(rois_per_image=R, dets_per_image=D, pre_nms_topk=150)
    out = eng.flatten_outputs(eng(_t(host, cuda)))
    torch.cuda.synchronize()
    # oracle, stage by stage
    pr = [oracle_lib.rpn_predict_proposals(d, a) for d, a in zip(host["deltas"], host["anchors"])]
    pb, pl, pv, _ = oracle_lib.find_top_rpn_proposals(pr, host["logits"], host["shapes"], 0.7, 150, R, 0.0)
    assert np.array_equal(out["proposal_boxes"].cpu().numpy(), pb)
    assert np.array_equal(out["proposal_valid"].cpu().numpy(), pv)
    idx = np.stack([np.repeat(np.arange(N), R), np.tile(np.arange(R), N)], 1).astype(np.int64)
    scales = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]
    bf, _ = oracle_lib.roi_pooler(host["feats"], scales, pb.reshape(-1, 4), idx[:, 0], (7, 7), 0)
    assert np.array_equal(out["box_feats"].cpu().numpy(), bf)
    ob = oracle_lib.apply_deltas(host["cls_deltas"], pb.reshape(-1, 4), (10., 10., 5., 5.))
    db, ds, dc, dv, dr, dn = oracle_lib.fast_rcnn_inference(ob, host["scores"], idx, (N, R), host["shapes"], 0.05, 0.5,
                                                            D, False)
    assert np.array_equal(out["det_boxes"].cpu().numpy(), db) and np.array_equal(out["det_classes"].cpu().numpy(), dc)
    assert np.array_equal(out["det_valid"].cpu().numpy(), dv)
    mf, _ = oracle_lib.roi_pooler(host["feats"], scales, db.reshape(-1, 4), np.repeat(np.arange(N), D), (14, 14), 0)
    assert np.array_equal(out["mask_feats"].cpu().numpy(), mf)
    # host-buffer path, several chunkings (ragged last chunk included): byte-identical
    hx = _t(host)
    for chunk in (1, 2, 3, 5):
        ho = eng.run_host(hx, cuda, chunk_images=chunk)
        for k, v in out.items():
            assert ho[k].is_pinned() and not ho[k].is_cuda
            assert torch.equal(ho[k], v.cpu()), (chunk, k)


@pytest.mark.parametrize("chunks", [1, 2, 3, 5])
def test_graphed_chunked_step_matches_eager(cuda, chunks):
    """`capture()`: the step as one CUDA graph, image blocks on concurrent streams.  Replays must reproduce the
    eager single-stream outputs bit for bit, also after the static inputs are refilled in place."""
    N, R, D, K, C = 5, 48, 12, 6, 16
    eng = MaskRCNNPostBackbone(rois_per_image=R, dets_per_image=D, pre_nms_topk=150)
    x = _t(_inputs(N, R, K, C, seed=1), cuda)
    g = eng.capture(x, chunks=chunks)
    assert g.kernels_per_replay > 0 and len(g.outputs) == min(chunks, N)
    for seed in (1, 2):
        fresh = _t(_inputs(N, R, K, C, seed=seed), cuda)
        for k, v in fresh.items():  # refill the static input tensors in place
            if isinstance(v, list):
                for dst, src in zip(x[k], v):
                    dst.copy_(src)
            else:
                x[k].copy_(v)
        g.replay()
        got = g.gathered()
        want = eng.flatten_outputs(eng(fresh))
        torch.cuda.synchronize()
        for k, v in want.items():
            assert torch.equal(got[k], v), (chunks, seed, k)


def test_step_pipeline_outputs(cuda):
    """StepPipeline: two captured steps in flight produce, each, the eager outputs."""
    N, R, D, K, C = 4, 48, 12, 6, 16
    eng = MaskRCNNPostBackbone(rois_per_image=R, dets_per_image=D, pre_nms_topk=150)
    x = _t(_inputs(N, R, K, C, seed=3), cuda)
    pipe = eng.pipeline(x, chunks=2, depth=2)
    pipe.run(5)
    torch.cuda.synchronize()
    want = eng.flatten_outputs(eng(x))
    for st in pipe.steps:
        got = st.gathered()
        for k, v in want.items():
            assert torch.equal(got[k], v), k
