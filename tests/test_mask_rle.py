"""CPU: the COCO run-length encoding the mask ops emit (pycocotools maskApi.c rleEncode + rleToString): the restatement
in coco_rle.py pinned on known answers and by an independent numpy decoder (rleFrString + rleDecode restated), and
the host-side slicing of `rle_to_coco`."""
import numpy as np
import pytest
import torch

from detectron2_tensorflow_b200.structures import rle_to_coco

import coco_rle


def decode(s, H, W):
    """pycocotools rleFrString + rleDecode: string -> uint8 mask [H, W]."""
    cnts = []
    p = 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = s[p] - 48
            x |= (c & 0x1f) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(cnts) > 2:
            x += cnts[-2]
        cnts.append(x)
    flat = np.zeros(H * W, np.uint8)
    j, v = 0, 0
    for c in cnts:
        flat[j:j + c] = v
        j += c
        v ^= 1
    assert j == H * W
    return flat.reshape(W, H).T


def checker(H, W):
    return (np.indices((H, W)).sum(0) % 2).astype(np.uint8)


KNOWN = [  # mask, counts, string
    (np.zeros((4, 3), np.uint8), [12], b"<"),
    (np.ones((4, 3), np.uint8), [0, 12], b"0<"),
    (np.pad(np.ones((2, 1), np.uint8), ((1, 1), (1, 1))), [5, 2, 5], b"525"),
    (np.array([[1, 0], [0, 0], [0, 1]], np.uint8), [0, 1, 4, 1], b"0140"),
    (checker(4, 4), [1, 1, 1, 2, 1, 1, 2, 1, 1, 2, 1, 1, 1], b"11110O10O10O0"),
    (np.zeros((800, 1333), np.uint8), [1066400], b"P]aP1"),
]


@pytest.mark.parametrize("case", range(len(KNOWN)))
def test_known_answers(case):
    mask, counts, want = KNOWN[case]
    assert coco_rle.encode(mask[None]) == [want]
    flat = mask.T.reshape(-1)  # column-major
    edges = np.flatnonzero(np.diff(np.concatenate([[0], flat])))  # positions where the value changes, from a zero
    assert np.diff(np.concatenate([[0], edges, [flat.size]])).tolist() == counts
    assert coco_rle.counts(mask).tolist() == counts
    assert np.array_equal(decode(want, *mask.shape), mask)


def test_delta_starts_at_the_fourth_count():
    """x -= cnts[i-2] applies for i > 2, not i >= 2: cnts [3, 40, 5] write 5 as itself ('5'), not as 5 - 3 ('2')."""
    m = np.zeros((48, 1), np.uint8)
    m[3:43] = 1
    s = coco_rle.encode(m[None])[0]
    assert s == b"3X15"  # 40 = 8 + 1 * 32: "X" (8 | 0x20) then "1"
    assert np.array_equal(decode(s, 48, 1), m)


def test_round_trip_random_masks():
    rng = np.random.default_rng(0)
    masks, shapes = [], [(1, 1), (1, 37), (37, 1), (31, 33), (64, 64), (97, 5)]
    for H, W in shapes:
        for density in (0.0, 0.02, 0.5, 0.98, 1.0):
            masks.append(((H, W), (rng.random((3, H, W)) < density).astype(np.uint8)))
    yy, xx = np.mgrid[0:120, 0:150]
    blob = ((yy - 60) ** 2 / 900 + (xx - 70) ** 2 / 2500 <= 1).astype(np.uint8)
    masks.append(((120, 150), np.stack([blob, 1 - blob, checker(120, 150)])))
    for (H, W), m in masks:
        for s, mk in zip(coco_rle.encode(m), m):
            assert np.array_equal(decode(s, H, W), mk)


def test_rle_to_coco_slicing_and_overflow():
    chars = torch.frombuffer(bytearray(b"<0<525xyz"), dtype=torch.uint8)
    offsets = torch.tensor([0, 1, 3, 6], dtype=torch.int64)
    got = rle_to_coco(chars, offsets, (4, 3))
    assert got == [{"size": [4, 3], "counts": b"<"}, {"size": [4, 3], "counts": b"0<"},
                   {"size": [4, 3], "counts": b"525"}]
    assert rle_to_coco(chars[:0], torch.zeros(1, dtype=torch.int64), (4, 3)) == []
    with pytest.raises(ValueError, match="need 12 bytes"):
        rle_to_coco(chars, torch.tensor([0, 1, 3, 12], dtype=torch.int64), (4, 3))
