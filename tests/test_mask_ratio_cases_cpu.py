"""The rounding chain of the mask overlap maps at float16 rounding boundaries, and the generator of the boundary cases
(oracle/mask_cases.py) that tests/test_gpu_mask_limits.py feeds to the kernels.  No GPU.

maps_from_counts is the oracle every overlap test compares with; here it is checked against exact rational
arithmetic, RN16(RN32(i / d)) with fractions.Fraction, on every class of quotient the generator produces -- including
the double-rounding ties, where the correctly rounded RN16(i / d) is a different float16 and the kernels must
reproduce the reference's double rounding instead."""
import numpy as np
import pytest

from oracle import mask_cases as mc
from oracle import mask_oracle

SIZES = [(512, 512), (375, 500)]


def oracle_pair(i, d):
    """uint16 of maps_from_counts for a mask of i pixels inside one of d pixels: iou[0, 1] and asy[1, 0] are i / d."""
    inter = np.array([[d, i], [i, i]], np.int64)
    iou, asy = mask_oracle.maps_from_counts(inter, np.array([d, i], np.int64))
    return int(iou[0, 1].view(np.uint16)), int(asy[1, 0].view(np.uint16))


def all_pairs():
    i, d = [], []
    for k, (h, w) in enumerate(SIZES):
        a, b = mc.boundary_pairs(h * w, seed=k)
        i.append(a)
        d.append(b)
    rng = np.random.default_rng(3)
    dg = rng.integers(1, 1 << 21, 400)                       # generic quotients, 0, 1
    i += [rng.integers(0, dg + 1), np.array([0, 5, 7])]
    d += [dg, np.array([9, 5, 7])]
    return np.concatenate(i), np.concatenate(d)


def test_maps_from_counts_is_rn16_of_rn32_on_every_class():
    i, d = all_pairs()
    cls = mc.classify(i, d)
    for k in ("tie", "near", "double", "subtie", "sub", "gap", "zero", "one"):
        assert cls[k].sum() > 0, k
    q32 = mc.quotient32(i, d)
    n_double = 0
    for a, b, q, dbl in zip(i, d, q32, cls["double"]):
        want = mc.ref_chain_f16(a, b)
        assert float(mc.rn32(mc.Fraction(int(a), int(b)))) == float(q), (a, b)   # float64 -> float32: one rounding
        assert oracle_pair(a, b) == (want, want), (a, b)
        if dbl:                                              # the reference's value is not the correctly rounded one
            assert mc.exact_f16(a, b) != want, (a, b)
            n_double += 1
    assert n_double >= 60
    # 0 / 0 -> NaN in both maps
    iou, asy = mask_oracle.maps_from_counts(np.zeros((2, 2), np.int64), np.zeros(2, np.int64))
    assert np.isnan(iou).all() and np.isnan(asy).all()


def test_double_rounding_and_subnormal_ties_are_what_classify_says():
    # the fp32 quotients of these pairs are exactly float16-subnormal midpoints (k + 1/2) 2^-24
    n_double = 0
    for a, b in ((1, 18631), (2, 41605), (1, 133683), (3, 133683)):
        c = mc.classify(a, b)
        assert c["sub"] and c["subtie"], (a, b)
        q = mc.rn32(mc.Fraction(a, b)) * 2 ** 25
        assert q.denominator == 1 and q.numerator % 2 == 1
        n_double += int(c["double"][0])
        assert bool(c["double"][0]) == (mc.ref_chain_f16(a, b) != mc.exact_f16(a, b))
    assert n_double >= 1
    # s o / (s 2^12): exact normal ties, not double rounding (the fp32 quotient is exact)
    i, d = mc.tie_pairs(1 << 18)
    c = mc.classify(i, d)
    assert c["tie"].all() and not c["double"].any() and not c["near"].any()
    assert all(mc.Fraction(int(a), int(b)).denominator == 4096 for a, b in zip(i, d))


def test_subnormal_tie_search():
    i, d = mc.subnormal_ties(1 << 21)
    assert len(i) >= 381
    pairs = set(zip(i.tolist(), d.tolist()))
    assert {(1, 18631), (2, 41605), (1, 133683), (3, 133683)} <= pairs
    c = mc.classify(i, d)
    assert c["subtie"].all()
    assert (d <= 1 << 21).all() and (mc.quotient32(i, d) < np.float32(2.0 ** -14)).all()


@pytest.mark.parametrize("h,w,n_img", [(512, 512, 3), (375, 500, 2)], ids=["512x512", "375x500"])
def test_generator_produces_every_class(h, w, n_img):
    """The image batches of tests/test_gpu_mask_limits.py::test_rounding_boundaries (mask_cases.boundary_batch): the
    least counts per class and map, and the interval counts against np.bitwise_count over the packed words."""
    total, words, n = h * w, (h * w + 31) // 32, mc.BOUNDARY_N
    tot = {"iou": dict.fromkeys(mc.CLASSES, 0), "asy": dict.fromkeys(mc.CLASSES, 0)}
    for b, (s, e) in enumerate(mc.boundary_batch(total, n_img)):
        assert (s >= 0).all() and (e <= total).all() and (s <= e).all()
        inter, area = mc.interval_counts(s, e)
        for m, c in mc.class_counts(inter, area).items():
            for k, v in c.items():
                tot[m][k] += v
        packed = mc.pack_intervals(s, e, words)
        rows = np.random.default_rng(b).choice(n, 8, replace=False)
        p_inter, p_area = mc.popcount_counts(packed, rows)
        np.testing.assert_array_equal(p_area, area)
        np.testing.assert_array_equal(p_inter, inter[rows])
    for m in ("iou", "asy"):
        for k, lo in mc.MIN_PER_MAP.items():
            assert tot[m][k] >= lo, (m, k, tot[m][k])


def test_pack_helpers():
    s, e = np.array([0, 3, 31, 40, 0]), np.array([1, 35, 33, 104, 0])
    packed = mc.pack_intervals(s, e, 4)
    bits = np.unpackbits(packed.view(np.uint8), axis=1, bitorder="little")
    want = np.zeros((5, 128), np.uint8)
    for k in range(5):
        want[k, s[k]:e[k]] = 1
    np.testing.assert_array_equal(bits, want)
    # tiled order: pixel (y, x) -> q = ((y >> 3) * (W >> 4) + (x >> 4)) * 128 + (y & 7) * 16 + (x & 15)
    rng = np.random.default_rng(0)
    m = rng.random((3, 16, 48)) < 0.5
    got = np.unpackbits(mc.pack_pixels(m, "tiled").view(np.uint8), axis=1, bitorder="little")
    y, x = np.divmod(np.arange(16 * 48), 48)
    q = ((y >> 3) * 3 + (x >> 4)) * 128 + (y & 7) * 16 + (x & 15)
    want = np.zeros_like(got)
    want[:, q] = m.reshape(3, -1)
    np.testing.assert_array_equal(got, want)
    flat = np.unpackbits(mc.pack_pixels(m[:, :, :37], "flat").view(np.uint8), axis=1, bitorder="little")
    np.testing.assert_array_equal(flat[:, :16 * 37], m[:, :, :37].reshape(3, -1))
    assert not flat[:, 16 * 37:].any()
