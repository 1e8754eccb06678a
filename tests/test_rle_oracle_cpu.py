"""COCO compressed RLE without a GPU: the oracle (oracle/rle_oracle.py, a restatement of pycocotools' maskApi.c) on
hand-checked strings, round trips and numpy's area / box, the C restatement the timing tool runs against the same
oracle, and the argument refusals of cim_mask_rle (checked before anything touches CUDA)."""
import ctypes as C

import numpy as np
import pytest
import torch

from cim_b200 import _lib, mask_ops, postproc
from oracle import rle_oracle as R

NULL = C.c_void_p(0)
FAKE = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch


def _m(rows):
    return np.array(rows, np.uint8)


def _two_pixels():
    m = np.zeros((31, 5), np.uint8)
    m[30, 1] = m[0, 2] = 1
    return m


def _last_pixel():
    m = np.zeros((1000, 1000), np.uint8)
    m[999, 999] = 1
    return m


# (mask [h][w], counts, string) worked out by hand from maskApi.c
HAND = [
    (_m([[0, 1, 1, 0], [0, 1, 0, 0], [1, 1, 0, 0]]), [2, 5, 5], b"255"),
    (_m([[0, 0, 0], [1, 0, 0], [1, 1, 0], [1, 0, 0]]), [1, 3, 2, 1, 5], b"132N3"),     # negative delta
    (np.ones((2, 3), np.uint8), [0, 6], b"06"),
    (np.zeros((4, 4), np.uint8), [16], b"`0"),                                        # 16 needs the sign continuation
    (_two_pixels(), [61, 2, 92], b"m12l2"),                                           # a run across a column boundary
    (_last_pixel(), [999999, 1], b"oa`n01"),
]


@pytest.mark.parametrize("case", range(len(HAND)))
def test_hand_checked_strings(case):
    mask, counts, string = HAND[case]
    cnts = R.encode(mask)
    assert cnts.tolist() == counts
    assert R.to_string(cnts) == string
    assert R.fr_string(string).tolist() == counts
    assert R.CEncoder(mask.size)(np.asfortranarray(mask)) == string


def numpy_bbox(mask):
    ys, xs = np.nonzero(mask)
    if ys.size == 0:
        return np.zeros(4)
    return np.array([xs.min(), ys.min(), xs.max() - xs.min() + 1, ys.max() - ys.min() + 1], np.float64)


def masks():
    """A few hundred random and structured masks: densities from empty to full, checkerboards, stripes, rectangles,
    single pixels, h or w of 1, h % 32 in {0, 1, 31}."""
    rs = np.random.RandomState(0)
    out = [np.zeros((1, 1), np.uint8), np.ones((1, 1), np.uint8)]
    out += [(np.indices(s).sum(0) % 2).astype(np.uint8) for s in ((33, 64), (1, 17), (31, 1))]
    for t in range(300):
        h, w = rs.choice([1, 2, 31, 32, 33, 64, 65]) if t % 3 == 0 else rs.randint(1, 70), rs.randint(1, 70)
        kind = t % 5
        if kind == 0:
            m = rs.rand(h, w) < rs.rand()
        elif kind == 1:
            m = np.zeros((h, w), bool)
            m[rs.randint(h):rs.randint(h + 1), rs.randint(w):rs.randint(w + 1)] = True
        elif kind == 2:
            m = (np.arange(h)[:, None] // rs.randint(1, 5) + np.arange(w)[None] // rs.randint(1, 5)) % 2 == 0
        elif kind == 3:
            m = np.zeros((h, w), bool)
            m.flat[rs.randint(h * w)] = True
        else:
            m = np.ones((h, w), bool)
            m.flat[rs.randint(h * w, size=rs.randint(0, 4))] = False
        out.append(m.astype(np.uint8))
    return out


def test_round_trip_area_and_bbox():
    enc = R.CEncoder(70 * 70)
    for mask in masks():
        h, w = mask.shape
        cnts = R.encode(mask)
        assert cnts.sum() == h * w and (cnts[1:] > 0).all()
        s = R.to_string(cnts)
        np.testing.assert_array_equal(R.fr_string(s), cnts)
        np.testing.assert_array_equal(R.decode(R.fr_string(s), h, w), mask)
        assert R.area(cnts) == int(mask.sum())
        np.testing.assert_array_equal(R.to_bbox(cnts, h, w), numpy_bbox(mask))
        assert enc(np.asfortranarray(mask)) == s
        d, a, bb = R.encode_mask(mask)
        assert d == {"size": [h, w], "counts": s} and a == mask.sum() and (bb == numpy_bbox(mask)).all()


def test_long_counts_take_up_to_seven_characters():
    for x in (0, 15, 16, 2 ** 20, 2 ** 31 - 1, -(2 ** 31)):
        s = R.to_string(np.array([x], np.int64))
        assert 1 <= len(s) <= 7 and R.fr_string(s)[0] == (x & 0xffffffff)
    assert len(R.to_string(np.array([2 ** 31 - 1]))) == 7


def test_mask_rle_argument_validation():
    L = _lib.lib()

    def call(packed=FAKE, n_img=2, r=10, words=8192, h=512, w=512, kbr=0, mask_hw=NULL, count=FAKE, idx=FAKE, cap=5,
             chars=FAKE, chars_cap=100, off=FAKE, len_=FAKE, area=NULL, bbox=NULL, need=FAKE):
        return L.cim_mask_rle(packed, n_img, r, words, h, w, kbr, mask_hw, count, idx, cap, chars, chars_cap, off,
                              len_, area, bbox, need, NULL)

    for kw in ({"packed": NULL}, {"count": NULL}, {"idx": NULL}, {"off": NULL}, {"len_": NULL}, {"need": NULL},
               {"chars": NULL}, {"n_img": -1}, {"r": -1}, {"cap": -1}, {"words": -1}, {"chars_cap": -1}, {"h": 0},
               {"w": 0}, {"kbr": -1}, {"kbr": 16}, {"kbr": 32, "h": 500}, {"kbr": 2, "w": 40, "words": 640}):
        assert call(**kw) == -1, kw
    assert call(words=8191) == -2                                   # fewer words than ceil(h * w / 32)
    assert call(h=65536, w=32768, words=2 ** 26) == -2              # h * w > 2^31 - 1
    assert call(n_img=65536, cap=65536) == -2
    for kw in ({"packed": C.c_void_p(4098)}, {"off": C.c_void_p(4100)}, {"need": C.c_void_p(4100)},
               {"bbox": C.c_void_p(4104)}, {"len_": C.c_void_p(4097)}, {"mask_hw": C.c_void_p(4098)}):
        assert call(**kw) == -4, kw


def test_no_cpu_path():
    z = torch.zeros(1, 4, 8, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mask_ops.mask_rle(z, torch.zeros(1, dtype=torch.int32), torch.zeros(1, 2, dtype=torch.int32), 16, 16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        postproc.segms_batched(z, (torch.zeros(1, dtype=torch.int32), torch.zeros(1, 2, dtype=torch.int32),
                                   torch.zeros(1, 2, dtype=torch.int32)), 16, 16, 2)
