"""CPU: the batched, per-image-size RLE mode of d2b_paste_masks without a GPU: the params struct field by field against
the header, the argument checks that return before any CUDA call, the host-side size checks of
`detector_postprocess_rle`, and the host assemblers `rle_to_coco` (per-mask sizes, empty slots) and `coco_results`."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import coco_results, detector_postprocess_rle
from detectron2_tensorflow_b200.structures import BoxList, rle_to_coco

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from detectron2_tensorflow_b200 import build
    build.build()
    return nv._bind("paste_masks")


def test_paste_params_field_offsets_match_header(tmp_path):
    """offsetof of every field of d2b_paste_masks_params, and its sizeof, equal the ctypes layout."""
    st = nv.PasteMasksParams
    names = [f[0] for f in st._fields_]
    assert names[-5:] == ["num_images", "dets_per_image", "output_shapes", "input_shapes", "valid"]
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "d2b200.h"\nint main(){'
            + "".join(f'printf("{n} %zu\\n", offsetof(d2b_paste_masks_params, {n}));' for n in names)
            + 'printf("sizeof %zu\\n", sizeof(d2b_paste_masks_params));return 0;}')
    src = tmp_path / "off.c"
    src.write_text(prog)
    exe = tmp_path / "off"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    got = dict(zip(out[0::2], map(int, out[1::2])))
    for n in names:
        assert getattr(st, n).offset == got[n], n
    assert C.sizeof(st) == got["sizeof"]


def _batched(**kw):
    p = nv.PasteMasksParams()
    # addresses are never dereferenced: every case returns before any CUDA call
    p.box_masks, p.boxes, p.num_masks, p.mask_h, p.mask_w, p.mask_threshold = 0x1000, 0x2000, 6, 14, 14, 0.5
    p.num_images, p.dets_per_image, p.output_shapes, p.out_rle_offsets = 2, 3, 0x3000, 0x4000
    for k, v in kw.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("case,msg", [
    (dict(out=0x5000), b"RLE only"),
    (dict(out_rle_offsets=None), b"RLE only"),
    (dict(output_shapes=None), b"output_shapes NULL"),
    (dict(dets_per_image=4), b"not num_images"),
    (dict(dets_per_image=-3, num_masks=-6), b"out of range"),
    (dict(mask_h=0), b"bad sizes"),
    (dict(rle_capacity=16), b"out_rle NULL"),
    (dict(num_images=0), b"need num_images > 0"),
    (dict(num_images=-1, dets_per_image=0, output_shapes=None), b"need num_images > 0"),
])
def test_batched_misuse_is_einval_before_cuda(lib, case, msg):
    assert lib.d2b_paste_masks(C.byref(_batched(**case)), None, 0, None) == -1
    assert msg in lib.d2b_last_error()
    assert lib.d2b_paste_masks_workspace_bytes(C.byref(_batched())) == 0


def _results(N, R, mh=4, mw=4):
    bl = BoxList(torch.zeros(N, R, 4))
    bl.add_field("pred_masks", torch.zeros(N, R, mh, mw))
    bl.add_field("is_valid", torch.ones(N, R, dtype=torch.bool))
    bl.set_tracking("image_shape", torch.full((N, 2), 10, dtype=torch.int32))
    return bl


@pytest.mark.parametrize("shapes,msg", [
    ([[10, 10], [0, 5]], r"output_shapes\[1\]"),
    ([[10, -1], [5, 5]], r"output_shapes\[0\]"),
    ([[46341, 46341], [5, 5]], r"output_shapes\[0\]"),
    ([[10, 10]], "2 values for 2 images"),
])
def test_host_output_shapes_checked_before_any_device_work(shapes, msg):
    with pytest.raises(ValueError, match=msg):
        detector_postprocess_rle(_results(2, 3), shapes)
    with pytest.raises(ValueError, match="no pasted masks"):
        detector_postprocess_rle(_results(2, 3), [[4, 4], [4, 4]], mask_format="raw")


def test_rle_to_coco_per_mask_sizes_and_empty_slots():
    chars = torch.frombuffer(bytearray(b"<0<525"), dtype=torch.uint8)
    offsets = torch.tensor([0, 1, 1, 3, 3, 6], dtype=torch.int64)   # slots 1 and 3 are empty
    sizes = np.array([[4, 3], [9, 9], [4, 3], [7, 7], [3, 4]])
    got = rle_to_coco(chars, offsets, sizes=sizes)
    assert got == [{"size": [4, 3], "counts": b"<"}, None, {"size": [4, 3], "counts": b"0<"}, None,
                   {"size": [3, 4], "counts": b"525"}]
    # the sizes of an [N, R] batch: np.repeat(output_shapes, R, 0)
    got = rle_to_coco(chars, offsets[:5], sizes=np.repeat([[4, 3], [2, 6]], 2, 0))
    assert [g and g["size"] for g in got] == [[4, 3], None, [2, 6], None]
    with pytest.raises(AssertionError, match="3 sizes for 5 strings"):
        rle_to_coco(chars, offsets, sizes=sizes[:3])
    with pytest.raises(ValueError, match="need 9 bytes"):
        rle_to_coco(chars, torch.tensor([0, 9]), sizes=[[1, 1]])


def test_coco_results_assembles_valid_slots():
    """Two images x three slots; image 0 slots 0 and 2 and image 1 slot 1 hold detections (non-empty strings)."""
    N, R = 2, 3
    bl = _results(N, R)
    bl.add_field("scores", torch.tensor([[0.9, 0.0, 0.25], [0.0, 0.5, 0.0]]))
    bl.add_field("pred_classes", torch.tensor([[0, 0, 2], [0, 1, 0]]))
    boxes = torch.tensor([[[1.5, 2.0, 11.5, 22.25], [0, 0, 0, 0], [0.1, 0.2, 0.3, 0.7]],
                          [[0, 0, 0, 0], [5.0, 7.0, 6.0, 17.0], [0, 0, 0, 0]]], dtype=torch.float32)
    chars = torch.frombuffer(bytearray(b"<0<525" + b"\xa5" * 4), dtype=torch.uint8)  # spare capacity at the end
    offsets = torch.tensor([0, 1, 1, 3, 3, 6, 6], dtype=torch.int64)
    shapes = [[4, 3], [3, 4]]
    res = coco_results(bl, (chars, offsets), boxes, shapes, ["a", "b"], {0: 1, 1: 3, 2: 90})
    f32 = np.float32
    assert res == [
        {"image_id": "a", "category_id": 1, "bbox": [2.0, 1.5, 20.25, 10.0], "score": float(f32(0.9)),
         "segmentation": {"size": [4, 3], "counts": b"<"}},
        {"image_id": "a", "category_id": 90, "bbox": [float(f32(0.2)), float(f32(0.1)), float(f32(0.7) - f32(0.2)),
                                                       float(f32(0.3) - f32(0.1))],
         "score": 0.25, "segmentation": {"size": [4, 3], "counts": b"0<"}},
        {"image_id": "b", "category_id": 3, "bbox": [7.0, 5.0, 10.0, 1.0], "score": 0.5,
         "segmentation": {"size": [3, 4], "counts": b"525"}},
    ]
    with pytest.raises(ValueError, match="need 6 bytes"):
        coco_results(bl, (chars[:5], offsets), boxes, shapes, ["a", "b"], {0: 1, 1: 3, 2: 90})
