import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from detectron2_tensorflow_b200.modeling import solo_upsample_masks
from detectron2_tensorflow_b200.utils import synthetic as syn
dev = torch.device("cuda", 0)
B, H, W = 16, 200, 336
obj = np.stack([syn.solo_masks(100, hw=(H, W), seed=70 + i)[0] for i in range(B)]).reshape(B, 100, -1).astype(np.uint8)
obj = np.concatenate([obj, np.zeros((B, 100, (-obj.shape[-1]) % 64), np.uint8)], -1)
kept = torch.from_numpy(np.packbits(obj, axis=-1, bitorder="little").view(np.int64)).to(dev)
for _ in range(3):
    solo_upsample_masks(kept, (H, W), (800, 1333), 0.5, False)
torch.cuda.synchronize()
