"""Phase timeline of the fused RPN kernels (debug build only: D2B_EXTRA_NVCC=-DD2B_PROFILE python -m
detectron2_tensorflow_b200.build --force).  Prints the %globaltimer deltas (us) recorded by cluster 0 of
rpn_select_kernel (the P2 row of image 0), by segment 0 of rpn_sweep_merge_kernel and, with N >= 4 images (the walk
runs), by image 0 of rpn_lazy_merge_kernel: keys loaded, merge ranks of the first chunk, its boxes gathered, and the
end of every 64-candidate block.

    python tools/phase_probe.py [N]"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import Box2BoxTransform, RPNOutputs
from detectron2_tensorflow_b200.structures import ImageList
from detectron2_tensorflow_b200.utils import synthetic as syn

dev = torch.device("cuda", 0)
N = int(sys.argv[1]) if len(sys.argv) > 1 else 1
anchors = syn.rpn_anchors()
logits, deltas = syn.rpn_inputs(N, seed=2, variant="gaussian", anchors=anchors)
ta = [torch.from_numpy(a).to(dev) for a in anchors]
tl = [torch.from_numpy(x).to(dev) for x in logits]
td = [torch.from_numpy(x).to(dev) for x in deltas]
outs = RPNOutputs(Box2BoxTransform((1., 1., 1., 1.)), ImageList(None, torch.from_numpy(syn.image_shapes(N)).to(dev)), tl, td, ta)
L = nv.lib()
buf = (C.c_uint64 * 256)()
for it in range(3):
    outs.find_top_proposals(0.7, 2000, 1000, 0.0)
    torch.cuda.synchronize()
    assert L.d2b_debug_read_profile(buf) == 0
    t = np.array(buf[:], dtype=np.int64)
    sel = t[0:9]
    names = ["start", "pass0", "pass1", "pass2", "pass3", "lists_final", "run_sorted", "runs_exchanged", "decoded"]
    print(f"N={N} iter {it}: select kernel (cluster 0), us since start:")
    print("   " + "  ".join(f"{n}={(sel[i] - sel[0]) / 1e3:.1f}" for i, n in enumerate(names) if sel[i] >= sel[0]))
    print(f"   sweep kernel (segment 0): sweep={(t[17] - t[16]) / 1e3:.1f} us, merge end={(t[18] - t[16]) / 1e3:.1f} us; "
          f"select start -> sweep start {(t[16] - t[0]) / 1e3:.1f} us")
    print("   pass 0: scanned={:.1f} cluster_sync={:.1f};  pass 1: scanned={:.1f} cluster_sync={:.1f}".format(
        *[(t[i] - sel[0]) / 1e3 for i in (65, 67, 73, 75)]))
    print(f"   merge (since sweep start): lists exchanged={(t[20] - t[16]) / 1e3:.1f} written={(t[18] - t[16]) / 1e3:.1f}")
    blk = t[32:64]
    print("   block publish times (us since sweep start): " + " ".join(f"{(b - t[16]) / 1e3:.1f}" for b in blk))
    if t[128] and t[200] >= t[128]:
        blocks = [(t[132 + b] - t[128]) / 1e3 for b in range(64) if t[132 + b] >= t[128] and t[132 + b] <= t[200]]
        steps = np.diff([(t[131] - t[128]) / 1e3] + blocks)
        print("   walk (image 0), us since start: keys={:.1f} ranks={:.1f} gathered={:.1f} blocks={} end={:.1f}".format(
            *[(t[i] - t[128]) / 1e3 for i in (129, 130, 131)], len(blocks), (t[200] - t[128]) / 1e3))
        print("   per block (us): " + " ".join(f"{x:.2f}" for x in steps))
