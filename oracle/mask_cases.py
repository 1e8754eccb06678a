"""oracle/mask_cases.py -- mask sets with known overlap counts at the float16 rounding boundaries of the overlap maps.

TEST INFRASTRUCTURE ONLY (like the rest of oracle/): imported by tests/.  Nothing under cim_b200/ may import it.

The overlap maps are fp16(fp32(i / d)) of integer counts (mask_oracle.maps_from_counts).  The tensor-core epilogue
(mask_overlap_tc.cu, ratio_f16) computes q = i * rcp.approx(d) and falls back to an IEEE division when q lies within
8 fp32 ulps of a float16 rounding midpoint, below 6.2e-5 (float16 subnormals) or is NaN.  classify() sorts quotients
into the classes that decide whether that is right; the constructors build masks whose counts hit those classes.

Masks are bit intervals [start, end) in the PACKED order (bit p & 31 of word p >> 5, whatever the pixel layout): the
counts of two intervals are their overlap, so the reference needs no pass over pixels, and np.bitwise_count over the
packed words recomputes them independently.
"""
from fractions import Fraction

import numpy as np

F16_MIN_NORMAL = 2.0 ** -14
SUB_GUARD = np.float32(6.2e-5)      # ratio_f16's subnormal guard
WINDOW = 8                          # ratio_f16's midpoint window, fp32 ulps
CLASSES = ("tie", "near", "double", "subtie", "sub", "gap", "zero", "one", "nan")
# least number of entries per class and map that a batch of boundary images (one of random intervals, the others of
# boundary_image()) must contain
MIN_PER_MAP = {"tie": 100, "near": 100, "double": 40, "subtie": 40, "sub": 100, "gap": 20, "zero": 1, "one": 1,
               "nan": 1}


# ------------------------------------------------------------------------------------------ exact rounding
def _round_rational(x, prec, emin):
    """x (Fraction >= 0) rounded to `prec` significant bits, ulp at least 2^emin, ties to even."""
    if x == 0:
        return Fraction(0)
    e = x.numerator.bit_length() - x.denominator.bit_length()
    while x < Fraction(2) ** e:
        e -= 1
    while x >= Fraction(2) ** (e + 1):
        e += 1
    ue = max(e - (prec - 1), emin)
    s = x / Fraction(2) ** ue
    q, r = divmod(s.numerator, s.denominator)
    if 2 * r > s.denominator or (2 * r == s.denominator and q & 1):
        q += 1
    return Fraction(q) * Fraction(2) ** ue


def rn32(x):
    return _round_rational(Fraction(x), 24, -149)


def rn16(x):
    return _round_rational(Fraction(x), 11, -24)


def f16_bits(x):
    """uint16 pattern of a Fraction that float16 represents exactly."""
    return int(np.float16(float(x)).view(np.uint16))


def ref_chain_f16(i, d):
    """RN16(RN32(i / d)) with exact rational arithmetic: the reference's rounding chain (int / int -> float64 ->
    float32 -> float16), which for counts below 2^24 equals one float32 rounding followed by one float16 rounding."""
    return f16_bits(rn16(rn32(Fraction(int(i), int(d)))))


def exact_f16(i, d):
    """RN16(i / d): the correctly rounded float16, which the reference does NOT compute at double-rounding ties."""
    return f16_bits(rn16(Fraction(int(i), int(d))))


# ------------------------------------------------------------------------------------------ classes
def quotient32(i, d):
    """float32 quotient the way the reference forms it: int / int in float64, stored to float32."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return (np.asarray(i, np.float64) / np.asarray(d, np.float64)).astype(np.float32)


def _sub_midpoint_ulps(q):
    """distance of subnormal-range quotients q (float32) from the nearest float16 subnormal midpoint (k + 1/2) 2^-24,
    in fp32 ulps of q"""
    t = q.astype(np.float64) * 2.0 ** 25                       # exact; midpoints are the odd integers
    m = 2.0 * np.floor(t / 2.0) + 1.0
    return np.abs(t - m) * 2.0 ** -25 / np.spacing(q).astype(np.float64)


def classify(i, d):
    """Classes of the quotients i / d (integer arrays, broadcast): dict name -> bool array.
      tie     fp32 quotient exactly on a float16 rounding midpoint, normal range
      near    within +-8 fp32 ulps of such a midpoint, not on it
      double  the reference's double rounding differs from RN16(i / d) (always a tie or a subtie)
      subtie  float16-subnormal result within +-8 fp32 ulps of a subnormal midpoint (k + 1/2) 2^-24, on it included
      sub     float16-subnormal result (0 < q < 2^-14)
      gap     2^-14 <= q < 6.2e-5: normal float16, but below ratio_f16's guard
      zero, one, nan   i = 0 < d, i = d > 0, 0 / 0"""
    i, d = np.broadcast_arrays(np.atleast_1d(np.asarray(i, np.int64)), np.atleast_1d(np.asarray(d, np.int64)))
    q = quotient32(i, d)
    fin = d > 0
    normal = fin & (q >= np.float32(F16_MIN_NORMAL))
    low = (q.view(np.uint32) & 0x1FFF).astype(np.int64) - 0x1000
    sub = fin & (q > 0) & (q < np.float32(F16_MIN_NORMAL))
    out = {
        "tie": normal & (low == 0),
        "near": normal & (low != 0) & (np.abs(low) <= WINDOW),
        "sub": sub,
        "gap": normal & (q < SUB_GUARD),
        "zero": fin & (i == 0),
        "one": fin & (i == d),
        "nan": ~fin & (i == 0),
    }
    subtie = np.zeros(q.shape, bool)
    if sub.any():
        subtie[sub] = _sub_midpoint_ulps(q[sub]) <= WINDOW
    out["subtie"] = subtie
    double = np.zeros(q.shape, bool)
    cand = np.nonzero(out["tie"] | subtie)
    if cand[0].size:
        pairs = np.stack([i[cand], d[cand]], 1)
        uniq, inv = np.unique(pairs, axis=0, return_inverse=True)
        dr = np.array([ref_chain_f16(a, b) != exact_f16(a, b) for a, b in uniq], bool)
        double[cand] = dr[inv.reshape(-1)]
    out["double"] = double
    return out


def class_counts(inter, area):
    """Per map, how many entries of fp16 iou (inter / union) and asy (inter / area of the column) fall in each class."""
    inter = np.asarray(inter, np.int64)
    area = np.asarray(area, np.int64)
    union = area[..., :, None] + area[..., None, :] - inter
    res = {}
    for name, den in (("iou", union), ("asy", np.broadcast_to(area[..., None, :], inter.shape))):
        c = classify(inter, den)
        res[name] = {k: int(c[k].sum()) for k in CLASSES}
    return res


# ------------------------------------------------------------------------------------------ (i, d) families
def tie_pairs(max_d, per_s=3, rng=None):
    """Exact normal-range ties without an exact reciprocal: d = s 2^12 with odd s >= 3, i = s o with odd o in
    [2049, 4095], so i / d = o 2^-12 has 12 significant bits (a float16 midpoint) while 1 / d is inexact."""
    rng = rng or np.random.default_rng(0)
    ii, dd = [], []
    for s in range(3, max_d // 4096 + 1, 2):
        for o in rng.choice(np.arange(2049, 4096, 2), per_s, replace=False):
            ii.append(s * int(o))
            dd.append(s * 4096)
    return np.array(ii, np.int64), np.array(dd, np.int64)


def midpoint_pairs(rng, max_d, draws=200_000):
    """(i, d) drawn next to normal float16 midpoints m 2^-e (m odd, 12 bits), d in [max_d / 4, max_d]: about 1.5 %
    land exactly on the midpoint after the fp32 rounding (half of those are double-rounding cases) and ~25 % within
    8 ulps of it.  Returns the pairs and their classify() dict."""
    d = rng.integers(max_d // 4, max_d + 1, draws)
    m = 2 * rng.integers(1024, 2048, draws) + 1
    e = rng.integers(12, 15, draws)
    i = np.rint(m.astype(np.float64) * d / 2.0 ** e).astype(np.int64)
    ok = (i >= 1) & (i < d)
    i, d = i[ok], d[ok]
    return i, d, classify(i, d)


def subnormal_ties(max_d, window=WINDOW):
    """Every (i, d) with d <= max_d whose fp32 quotient is a float16 subnormal within `window` fp32 ulps of a subnormal
    midpoint (k + 1/2) 2^-24: per i, the d nearest to i 2^25 / m for every odd m < 2^11."""
    ii, dd = [], []
    m = np.arange(1, 2048, 2, dtype=np.float64)
    for i in range(1, max_d // 16384 + 1):
        c = np.rint(i * 2.0 ** 25 / m).astype(np.int64)
        c = np.unique(np.concatenate([c + k for k in (-2, -1, 0, 1, 2)]))
        c = c[(c >= 1) & (c <= max_d)]
        q = quotient32(i, c)
        c = c[(q > 0) & (q < np.float32(F16_MIN_NORMAL))]
        q = quotient32(i, c)
        keep = _sub_midpoint_ulps(q) <= window
        ii.append(np.full(int(keep.sum()), i, np.int64))
        dd.append(c[keep])
    return np.concatenate(ii), np.concatenate(dd)


def boundary_pairs(total, seed):
    """The hazard family for masks of `total` pixels: exact ties, drawn ties (incl. double rounding), near misses,
    the 160 subnormal ties closest to their midpoint (every exact one, then those within ~1 fp32 ulp, where an
    approximate quotient can land on the other side), plain subnormals and the [2^-14, 6.2e-5) gap."""
    rng = np.random.default_rng(seed)
    fam = [tie_pairs(total, rng=rng)]
    i, d, c = midpoint_pairs(rng, total)
    for k, want in (("double", 60), ("tie", 100), ("near", 100)):
        sel = np.nonzero(c[k] & ~c["double"] if k != "double" else c[k])[0][:want]
        fam.append((i[sel], d[sel]))
    si, sd = subnormal_ties(total)
    near = np.argsort(_sub_midpoint_ulps(quotient32(si, sd)), kind="stable")[:160]  # the exact ones first
    fam.append((si[near], sd[near]))
    gi = rng.integers(1, 8, 24)                                    # gap: d in (i / 6.2e-5, i 2^14]
    fam.append((gi, np.array([rng.integers(int(a / 6.2e-5) + 1, a * 16384 + 1) for a in gi], np.int64)))
    ui = rng.integers(1, max(2, total // 65536), 24)               # subnormal results
    fam.append((ui, np.array([rng.integers(a * 16384 + 1, total + 1) for a in ui], np.int64)))
    return np.concatenate([f[0] for f in fam]), np.concatenate([f[1] for f in fam])


# ------------------------------------------------------------------------------------------ masks as intervals
def nested_intervals(i, d, total, rng):
    """Two masks per pair: an interval of d pixels at a random place and one of i pixels inside it, alternately at
    its start and its end, so that the smaller mask sorts before the larger one for half of the pairs (by position)
    and after it for the other half.  iou = asy[small, large] = i / d."""
    n = len(i)
    b = rng.integers(0, total - d + 1)
    at_end = (np.arange(n) % 2) == 1
    s_small = np.where(at_end, b + d - i, b)
    starts = np.stack([b, s_small], 1).reshape(-1)
    ends = np.stack([b + d, s_small + i], 1).reshape(-1)
    return starts, ends


def random_intervals(n, total, rng):
    """Intervals of log-uniform length at uniform positions: generic iou / asy values."""
    length = np.minimum(total, np.exp(rng.uniform(0, np.log(total), n)).astype(np.int64) + 1)
    s = rng.integers(0, total - length + 1)
    return s, s + length


def boundary_image(total, n, seed):
    """n interval masks of `total` pixels: two empty masks (0 / 0), then the nested hazard pairs of boundary_pairs(),
    filled up with random intervals, in a random order."""
    rng = np.random.default_rng(seed)
    i, d = boundary_pairs(total, seed)
    s, e = nested_intervals(i, d, total, rng)
    assert len(s) + 2 <= n, "too many hazard pairs for n masks"
    rs, re = random_intervals(n - 2 - len(s), total, rng)
    s, e = np.concatenate([[0, 0], s, rs]), np.concatenate([[0, 0], e, re])
    p = rng.permutation(n)
    return s[p], e[p]


BOUNDARY_N = 1280                   # masks per image of boundary_batch()


def boundary_batch(total, n_img, n=BOUNDARY_N):
    """The images of the GPU boundary test: image 1 random intervals (generic values and the hazards they hit by
    chance), every other image boundary_image() with its index as seed.  List of (starts, ends)."""
    return [random_intervals(n, total, np.random.default_rng(b)) if b == 1 else boundary_image(total, n, b)
            for b in range(n_img)]


def interval_counts(starts, ends):
    """(inter [n, n], area [n]) int64 of interval masks."""
    s, e = np.asarray(starts, np.int64), np.asarray(ends, np.int64)
    inter = np.maximum(0, np.minimum(e[:, None], e[None, :]) - np.maximum(s[:, None], s[None, :]))
    return inter, e - s


def pack_intervals(starts, ends, words):
    """uint32 [n, words]: bit p & 31 of word p >> 5 set for start <= p < end."""
    s, e = np.asarray(starts, np.int64)[:, None], np.asarray(ends, np.int64)[:, None]
    out = np.empty((len(starts), words), np.uint32)
    w0 = 32 * np.arange(words, dtype=np.int64)[None, :]
    for c in range(0, words, 4096):
        w = w0[:, c:c + 4096]
        hi, lo = np.clip(e - w, 0, 32), np.clip(s - w, 0, 32)
        out[:, c:c + 4096] = (((np.uint64(1) << hi.astype(np.uint64)) - np.uint64(1)) &
                              ~((np.uint64(1) << lo.astype(np.uint64)) - np.uint64(1))).astype(np.uint32)
    return out


def popcount_counts(packed, rows=None):
    """Intersection counts of packed masks [n, words] by np.bitwise_count: rows x all columns (rows = all if None),
    and the areas.  Independent of the pixel order."""
    p = np.ascontiguousarray(packed)
    if p.shape[1] % 2 == 0:
        p = p.view(np.uint64)
    area = np.bitwise_count(p).sum(1, dtype=np.int64)
    rows = np.arange(len(p)) if rows is None else np.asarray(rows)
    inter = np.empty((len(rows), len(p)), np.int64)
    for k, r in enumerate(rows):
        inter[k] = np.bitwise_count(p[r] & p).sum(1, dtype=np.int64)
    return inter, area


# ------------------------------------------------------------------------------------------ pixel masks
def pack_pixels(masks, layout):
    """bool/uint8 masks [n, H, W] -> uint32 [n, ceil(H W / 32)] in the flat or the tiled (8 x 16 patch) pixel order
    of cim_mask_pack / cim_mask_pack_tiled, on the CPU."""
    m = np.asarray(masks) != 0
    n, h, w = m.shape
    if layout == "tiled":
        m = m.reshape(n, h // 8, 8, w // 16, 16).transpose(0, 1, 3, 2, 4)
    flat = m.reshape(n, -1)
    words = (h * w + 31) // 32
    bits = np.zeros((n, words * 32), bool)
    bits[:, :h * w] = flat
    return np.packbits(bits, axis=1, bitorder="little").view("<u4").reshape(n, words)
