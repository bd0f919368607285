"""CPU: the batched, per-image-size RLE mode of d2b_solo_upsample without a GPU: the params struct field by field
against the header, the argument checks that return before any CUDA call, the workspace query of both modes, and the
host-side size checks of `solo_upsample_rle` and `SOLOv2Inference.inference_rle`."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from detectron2_tensorflow_b200 import _native as nv
from detectron2_tensorflow_b200.modeling import SOLOv2Inference, solo_upsample_rle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from detectron2_tensorflow_b200 import build
    build.build()
    return nv._bind("solo_upsample")


def test_solo_upsample_params_field_offsets_match_header(tmp_path):
    """offsetof of every field of d2b_solo_upsample_params, and its sizeof, equal the ctypes layout."""
    st = nv.SoloUpsampleParams
    names = [f[0] for f in st._fields_]
    assert names[-3:] == ["output_shapes", "mask_shapes", "valid"]
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "d2b200.h"\nint main(){'
            + "".join(f'printf("{n} %zu\\n", offsetof(d2b_solo_upsample_params, {n}));' for n in names)
            + 'printf("sizeof %zu\\n", sizeof(d2b_solo_upsample_params));return 0;}')
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
    p = nv.SoloUpsampleParams()
    # addresses are never dereferenced: every case returns before any CUDA call
    p.packed_masks, p.batch, p.num_dets, p.mask_h, p.mask_w, p.mask_threshold = 0x1000, 2, 3, 20, 34, 0.5
    p.out_boxes, p.out_rle_offsets, p.output_shapes = 0x2000, 0x3000, 0x4000
    for k, v in kw.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("case,msg", [
    (dict(out_masks=0x5000), b"no planes"),
    (dict(out_packed_masks=0x5000), b"no planes"),
    (dict(out_rle_offsets=None), b"needs out_rle_offsets and out_boxes"),
    (dict(out_boxes=None), b"needs out_rle_offsets and out_boxes"),
    (dict(output_shapes=None, mask_shapes=0x6000, image_h=8, image_w=8), b"need output_shapes"),
    (dict(output_shapes=None, valid=0x6000, image_h=8, image_w=8), b"need output_shapes"),
    (dict(batch=-1), b"negative sizes"),
    (dict(num_dets=-2), b"negative sizes"),
    (dict(batch=65536), b"too large"),
    (dict(num_dets=65536), b"too large"),
    (dict(mask_h=0), b"bad mask_h / mask_w"),
    (dict(mask_w=-4), b"bad mask_h / mask_w"),
    (dict(mask_w=65536), b"bad mask_h / mask_w"),
    (dict(rle_capacity=16), b"out_rle NULL"),
    (dict(rle_capacity=-1), b"negative"),
])
def test_batched_misuse_is_einval_before_cuda(lib, case, msg):
    assert lib.d2b_solo_upsample(C.byref(_batched(**case)), None, 0, None) == -1
    assert msg in lib.d2b_last_error()


def test_workspace_query_both_modes(lib):
    """The batched mode reduces its boxes inside each CTA and needs no workspace; the single-size mode keeps one
    statistics record per mask; a misused struct answers 0."""
    assert lib.d2b_solo_upsample_workspace_bytes(C.byref(_batched())) == 0
    assert lib.d2b_solo_upsample_workspace_bytes(C.byref(_batched(num_dets=0))) == 0
    single = _batched(output_shapes=None, image_h=80, image_w=136)
    n = lib.d2b_solo_upsample_workspace_bytes(C.byref(single))
    assert n >= 6 * 40 and n % 256 == 0  # 6 statistics records of 40 bytes, 256-byte aligned
    assert lib.d2b_solo_upsample_workspace_bytes(C.byref(_batched(out_masks=0x5000))) == 0
    assert lib.d2b_solo_upsample_workspace_bytes(C.byref(_batched(output_shapes=None, valid=0x6000))) == 0


@pytest.mark.parametrize("kw,msg", [
    (dict(output_shapes=[[10, 10], [0, 5]]), r"output_shapes\[1\]"),
    (dict(output_shapes=[[10, -1], [5, 5]]), r"output_shapes\[0\]"),
    (dict(output_shapes=[[46341, 46341], [5, 5]]), r"output_shapes\[0\]"),
    (dict(output_shapes=[[10, 10]]), "output_shapes has 2 values for 2 images"),
    (dict(mask_shapes=[[4, 4], [4, 5]]), r"mask_shapes\[1\]"),       # w > mask_w
    (dict(mask_shapes=[[5, 4], [4, 4]]), r"mask_shapes\[0\]"),       # h > mask_h
    (dict(mask_shapes=[[4, 4], [0, 4]]), r"mask_shapes\[1\]"),
    (dict(mask_shapes=[[4, 4], [4, 4], [4, 4]]), "mask_shapes has 6 values for 2 images"),
])
def test_host_shapes_checked_before_any_device_work(kw, msg):
    """Masks are 4 x 4; nothing here reaches a device (the checks raise first)."""
    args = dict(output_shapes=[[10, 10], [5, 5]], mask_shapes=None)
    args.update(kw)
    packed = torch.zeros(2, 3, 1, dtype=torch.int64)
    with pytest.raises(ValueError, match=msg):
        solo_upsample_rle(packed, (4, 4), args["output_shapes"], args["mask_shapes"])
    head = SOLOv2Inference(num_grids=(2,), strides=(8,))
    feats = torch.zeros(2, 4, 4, 8)
    with pytest.raises(ValueError, match=msg):
        head.inference_rle([torch.zeros(2, 2, 2, 3)], [torch.zeros(2, 2, 2, 8)], feats, args["output_shapes"],
                           args["mask_shapes"])
