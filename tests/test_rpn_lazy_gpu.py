"""GPU: the capped walk in merge order of the fused proposal stage (rpn_lazy_merge_kernel, rpn_fused.cu) against
oracle.find_top_rpn_proposals, bit-exact (boxes, logits, valid, num_valid).

Each case also shows which path produced each image.  The walk writes a per-image flag into the last slice of the
stage's workspace: 1 = finished by the walk, 0 = visit budget spent (the mask + sweep-merge launches produce that
image).  The test allocates the workspace (through the canary guard, filled with a byte pattern), so an untouched
flag reads as the pattern, and a torch.profiler trace shows which kernels ran.  The budget cases are built from
groups of identical boxes, so that the position of the post-th kept box, and with it the number of visited blocks,
is known exactly.  The walk runs for batches of at least kRpnLazyMinImages images, so every walk case has 4."""
import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import Box2BoxTransform, RPNOutputs, find_top_rpn_proposals
from detectron2_tensorflow_b200.structures import ImageList
from detectron2_tensorflow_b200.utils import synthetic as syn

from test_canary_gpu import Guard
from test_dispatch_boundaries_gpu import K, Launch, reach, traced
import test_fuzz_gpu as fz

pytestmark = pytest.mark.gpu

MAX_BLOCKS = 64                # kRpnLazyMaxBlocks (rpn.cuh)
MAX_SMEM = 200 * 1024          # kRpnLazyMaxSmem (rpn.cuh)
MIN_IMAGES = 4                 # kRpnLazyMinImages (rpn.cuh)
CHUNK = 1024                   # kLazyChunk (rpn_fused.cu)
UNTOUCHED = int.from_bytes(b"\xa5" * 4, "little", signed=True)  # guard PATTERN: the walk did not run


def lazy_smem(hwa, pre, post):
    """rpn_fused.cu lazy_layout(): bytes of dynamic shared memory of the walk."""
    k = min(pre, max(hwa))
    kcap = [min(k, h) for h in hwa]
    KT, VT = sum(kcap), sum(min(post, c) for c in kcap)
    return 16 * VT + 16 * CHUNK + 4 * KT + 4 * min(MAX_BLOCKS * 64, KT) + 4 * min(post, KT)


class Flags(object):
    """Records the workspaces handed to the library (allocated by the canary guard) and reads the walk's flags."""

    def __init__(self, monkeypatch):
        self.guard = Guard(monkeypatch)
        self.ws = []
        inner = self.guard.workspace

        def workspace(nbytes, device):
            buf = inner(nbytes, device)
            self.ws.append(buf)
            return buf
        monkeypatch.setattr(nv, "_workspace", workspace)
        self.num_valid = None
        call = nv.call

        def call_with_num_valid(op, params, device):  # the Python layer passes no out_num_valid: ask for it here
            if op == "rpn_proposals":
                self.num_valid = torch.full((params.num_images,), -7, dtype=torch.int32, device=device)
                params.out_num_valid = self.num_valid.data_ptr()
            return call(op, params, device)
        monkeypatch.setattr(nv, "call", call_with_num_valid)

    def done(self, N):
        ws = self.ws[-1]
        start = ws.numel() - (-(-4 * N // 256) * 256)  # the last 256-byte slice of the workspace
        return ws[start:start + 4 * N].view(torch.int32).cpu().numpy()


@pytest.fixture
def flags(monkeypatch):
    return Flags(monkeypatch)


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def check(cuda, oracle_lib, flags, props, logits, shapes, pre, post, expect, run=None, thr=0.7):
    """Runs the stage (run() or find_top_rpn_proposals on props), compares with the oracle, and checks the per-image
    path: expect = list of 1 (walk) / 0 (fallback), "any" (the walk ran and flagged every image 0 or 1), or None when
    the walk must not run (shared-memory or batch-size gate)."""
    N = logits[0].shape[0]
    wb, wl, wv, wn = oracle_lib.find_top_rpn_proposals(props, logits, shapes, thr, pre, post, 0.0)
    if run is None:
        tp, tl, ts = [T(p, cuda) for p in props], [T(x, cuda) for x in logits], T(shapes, cuda)
        run = lambda: find_top_rpn_proposals(tp, tl, ImageList(None, ts), thr, pre, post, 0.0)
    res, trace = traced(run)
    assert np.array_equal(res.get_field("is_valid").cpu().numpy(), wv)
    assert np.array_equal(res.boxes.cpu().numpy().view(np.uint32), wb.view(np.uint32))
    assert np.array_equal(res.get_field("objectness_logits").cpu().numpy().view(np.uint32), wl.view(np.uint32))
    assert np.array_equal(flags.num_valid.cpu().numpy(), wn)
    done = flags.done(N)
    hwa = [x.shape[1] for x in logits]
    fits = lazy_smem(hwa, pre, post) <= MAX_SMEM
    masks_and_sweep = [Launch(K("nms_mask_kernel")), Launch(K("rpn_sweep_merge_kernel"))]
    if expect is None:
        assert not fits or N < MIN_IMAGES
        assert (done == UNTOUCHED).all(), done
        reach(trace, [Launch(K("rpn_select_kernel"))] + masks_and_sweep, [K("rpn_lazy_merge_kernel")])
    else:
        assert fits and N >= MIN_IMAGES
        if expect == "any":
            assert set(done.tolist()) <= {0, 1}, done
        else:
            assert done.tolist() == list(expect), done
        reach(trace, [Launch(K("rpn_select_kernel")), Launch(K("rpn_lazy_merge_kernel"), grid_x=N)] + masks_and_sweep)
    flags.guard.check()
    return wv


def anchored(cuda, oracle_lib, flags, logits, deltas, pre, post, expect):
    """Proposals decoded from deltas + anchors in the kernel, as bench.py runs the stage."""
    anchors = syn.rpn_anchors()
    N = logits[0].shape[0]
    shapes = syn.image_shapes(N)
    props = [oracle_lib.rpn_predict_proposals(d, a) for d, a in zip(deltas, anchors)]
    images = ImageList(None, T(shapes, cuda))
    outs = RPNOutputs(Box2BoxTransform((1., 1., 1., 1.)), images, [T(x, cuda) for x in logits],
                      [T(d, cuda) for d in deltas], [T(a, cuda) for a in anchors])
    return check(cuda, oracle_lib, flags, props, logits, shapes, pre, post, expect,
                 run=lambda: outs.find_top_proposals(0.7, pre, post, 0.0))


def test_bench_inputs(cuda, oracle_lib, flags):
    logits, deltas = syn.rpn_inputs(16, seed=2, variant="gaussian", anchors=syn.rpn_anchors())  # bench.py's
    anchored(cuda, oracle_lib, flags, logits, deltas, 2000, 1000, [1] * 16)


@pytest.mark.parametrize("variant", ["clustered", "ties"])
def test_rpn_input_variants(cuda, oracle_lib, flags, variant):
    logits, deltas = syn.rpn_inputs(4, seed=3, variant=variant, anchors=syn.rpn_anchors())
    anchored(cuda, oracle_lib, flags, logits, deltas, 2000, 1000, [1] * 4)


def fuzz(rng, hwa, N=4, H=300, W=400, quant=16):
    props = [np.stack([fz.fuzz_boxes(rng, h, H, W) for _ in range(N)]) for h in hwa]
    logits = [(np.round(rng.standard_normal((N, h)) * quant) / quant).astype(np.float32) for h in hwa]
    shapes = np.array([[H, W]] * N, np.int32)
    return props, logits, shapes


def test_equal_scores_across_levels(cuda, oracle_lib, flags):
    # logits on a grid of 1/2: every score occurs in every level many times, so the merge order rests on the tie rule
    # (lower level first, then position)
    props, logits, shapes = fuzz(np.random.default_rng(11), [1500, 900, 400], quant=2)
    wv = check(cuda, oracle_lib, flags, props, logits, shapes, 1000, 600, [1] * 4)
    assert wv.all()


def test_nan_and_inf_logits(cuda, oracle_lib, flags):
    rng = np.random.default_rng(12)
    props, logits, shapes = fuzz(rng, [1200, 700, 300])
    for x in logits:
        x[rng.random(x.shape) < 0.1] = np.nan
        x[rng.random(x.shape) < 0.1] = -np.inf
        x[rng.random(x.shape) < 0.02] = np.inf
    check(cuda, oracle_lib, flags, props, logits, shapes, 1000, 1000, [1] * 4)


def test_degenerate_and_clipped_boxes(cuda, oracle_lib, flags):
    rng = np.random.default_rng(13)
    props, logits, shapes = fuzz(rng, [1000, 600])
    for p in props:
        sel = rng.random(p.shape[:2]) < 0.3
        p[sel] = p[sel] + np.array([1000, 1000, 1000, 1000], np.float32)  # outside the image: clipped to zero area
        line = rng.random(p.shape[:2]) < 0.1
        p[line, 2] = p[line, 0]  # zero height
        neg = rng.random(p.shape[:2]) < 0.1
        p[neg] = -np.abs(p[neg]) - 5.0  # left of / above the image: clipped to the corner
    check(cuda, oracle_lib, flags, props, logits, shapes, 800, 700, [1] * 4)


def test_fewer_candidates_than_post(cuda, oracle_lib, flags):
    props, logits, shapes = fuzz(np.random.default_rng(14), [300, 120, 40])
    wv = check(cuda, oracle_lib, flags, props, logits, shapes, 2000, 1000, [1] * 4)
    assert not wv.all(axis=1).any()  # zero padding in every image


def test_eight_levels(cuda, oracle_lib, flags):
    props, logits, shapes = fuzz(np.random.default_rng(15), [3000, 1500, 700, 300, 120, 50, 20, 9])
    check(cuda, oracle_lib, flags, props, logits, shapes, 300, 1000, [1] * 4)


# ------------------------------------------------------------------ visit budget
def groups(dups, n_groups, cell=20, side=12, grid=70):
    """One image, two levels: candidate i (global score order) belongs to group i // dups; a group's boxes are identical
    (IoU 1: the first suppresses the rest) and lie alone in one grid cell (no IoU with other groups).  Groups alternate
    between the levels, so each level's NMS sees whole groups.  Kept boxes sit at positions 0, dups, 2 dups, ..."""
    T_ = dups * n_groups
    g = np.arange(T_) // dups
    cy, cx = (g // grid) * cell + 4.0, (g % grid) * cell + 4.0
    boxes = np.stack([cy, cx, cy + side, cx + side], 1).astype(np.float32)
    score = ((T_ - np.arange(T_)) / 64.0).astype(np.float32)  # strictly descending, exact in fp32
    lvl = g % 2
    props = [boxes[lvl == l][None] for l in (0, 1)]
    logits = [score[lvl == l][None] for l in (0, 1)]
    return props, logits


def batch(images):
    L = len(images[0][0])
    hw = [max(im[0][l].shape[1] for im in images) for l in range(L)]
    props, logits = [], []
    for l in range(L):  # pad every image's level to the same length with far-away, lowest-scored boxes
        P = np.full((len(images), hw[l], 4), -100.0, np.float32)
        X = np.full((len(images), hw[l]), -1e30, np.float32)
        for n, (p, x) in enumerate(images):
            P[n, :p[l].shape[1]] = p[l][0]
            X[n, :x[l].shape[1]] = x[l][0]
        props.append(P)
        logits.append(X)
    return props, logits


SHAPES = lambda N: np.array([[1400, 1400]] * N, np.int32)


@pytest.mark.parametrize("post,expect", [(1024, 1), (1025, 0)], ids=["exactly-budget", "budget-plus-one"])
def test_visit_budget(cuda, oracle_lib, flags, post, expect):
    # 4 copies per group: the post-th kept box is candidate 4 (post - 1): 4,092 (block 63, the last of the budget)
    # for post = 1,024, 4,096 (block 64) for post = 1,025
    assert (4 * (post - 1)) // 64 == MAX_BLOCKS - 1 + (1 - expect)
    props, logits = batch([groups(4, 1100)] * 4)
    wv = check(cuda, oracle_lib, flags, props, logits, SHAPES(4), 4096, post, [expect] * 4)
    assert wv.all()


def test_mixed_batch(cuda, oracle_lib, flags):
    # images 0, 2: no duplicates, finished after 1,025 candidates; images 1, 3: 4 copies per group, over the budget
    props, logits = batch([groups(1, 4400), groups(4, 1100)] * 2)
    check(cuda, oracle_lib, flags, props, logits, SHAPES(4), 4096, 1025, [1, 0, 1, 0])


@pytest.mark.parametrize("N", [MIN_IMAGES - 1, MIN_IMAGES])
def test_batch_size_gate(cuda, oracle_lib, flags, N):
    # fewer than kRpnLazyMinImages images: masks + sweep-merge only
    props, logits, shapes = fuzz(np.random.default_rng(16), [2000, 1000, 500, 250, 100], N=N)
    check(cuda, oracle_lib, flags, props, logits, shapes, 2000, 1000, [1] * N if N >= MIN_IMAGES else None)


@pytest.mark.parametrize("post", [3868, 3869])
def test_shared_memory_gate(cuda, oracle_lib, flags, post):
    # two levels of 4,096 candidates: 36 post + 65,536 bytes, 204,784 (walk) and 204,820 (> 200 KB: masks + sweep only)
    hwa = [4096, 4096]
    fits = lazy_smem(hwa, 4096, post) <= MAX_SMEM
    assert fits == (post == 3868)
    props, logits, shapes = fuzz(np.random.default_rng(post), hwa)
    wv = check(cuda, oracle_lib, flags, props, logits, shapes, 4096, post, "any" if fits else None)
    assert wv.any()


@pytest.mark.parametrize("thr", [1.5, -0.1, float("nan")])
def test_rejects_threshold_before_any_launch(cuda, flags, thr):
    # the walk writes outputs, so an invalid threshold must be rejected before the first launch, not by the NMS
    props, logits, shapes = fuzz(np.random.default_rng(17), [600, 300])
    tp, tl, ts = [T(p, cuda) for p in props], [T(x, cuda) for x in logits], T(shapes, cuda)
    before = nv.lib().d2b_kernel_launch_count()
    with pytest.raises(ValueError, match="nms_thresh"):
        find_top_rpn_proposals(tp, tl, ImageList(None, ts), thr, 1000, 1000, 0.0)
    assert nv.lib().d2b_kernel_launch_count() == before, "a rejected call launched kernels"
    flags.guard.check()
