"""The mask overlap stage (cim_mask_overlap*) where it is fragile: float16 rounding boundaries of the ratio epilogue,
native (non-square, padded) image sizes in both pixel orders and the dispatch between the tensor and the popcount
kernel, counts up to 2^21 in the mxf4 accumulator and the K-block list capacity, the largest n and the unranked tile
order, and the tile geometry / K-block skipping for every n from 64 to 640.

References never run either GPU overlap path: counts come from interval arithmetic, np.bitwise_count over packed words
built on the CPU, mask_oracle.overlap_counts, or (full native-size maps only) a float32 matmul of the 0/1 masks,
and the maps from mask_oracle.maps_from_counts.  Every comparison is exact.  Each test first asserts that its inputs
contain the cases it targets (oracle/mask_cases.py classifies them), so a change to a generator cannot make it pass
vacuously."""
import gc

import numpy as np
import pytest
import torch

from cim_b200 import mask_ops, synth
from oracle import mask_cases as mc
from oracle import mask_oracle
from conftest import assert_f16_bits_equal

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def u16(t):
    return t.cpu().numpy().view(np.uint16)


def cuda_words(packed):
    return torch.from_numpy(np.ascontiguousarray(packed).view(np.int32)).to(DEV)


def f16_equal_dev(a, b):
    """float16 maps bit-identical on the device, any NaN equal to any NaN."""
    a, b = a.view(torch.int16), b.view(torch.int16)
    nan = lambda v: ((v & 0x7C00) == 0x7C00) & ((v & 0x03FF) != 0)
    na = nan(a)
    return bool(torch.equal(na, nan(b))) and bool(torch.equal(torch.where(na, 0, a), torch.where(na, 0, b)))


def check_maps(out, inter, area, what=""):
    """out = mask_overlap(..., return_counts=True) of ONE image against integer reference counts."""
    iou, asy, g_inter, g_area = out[:4]
    np.testing.assert_array_equal(g_area.cpu().numpy(), area, err_msg=f"{what}: area")
    np.testing.assert_array_equal(g_inter.cpu().numpy(), inter, err_msg=f"{what}: inter")
    o_iou, o_asy = mask_oracle.maps_from_counts(inter, area)
    assert_f16_bits_equal(u16(iou), o_iou.view(np.uint16))
    assert_f16_bits_equal(u16(asy), o_asy.view(np.uint16))


def ordered_tiles(n, n_img):
    """Whether the tensor path ranks the tiles (mask_rank_kernel) or decodes them by their distance from the
    diagonal: the rule of cim_mask_overlap_meta (mask_overlap.cu)."""
    nrb, ncb = (n + 127) // 128, (n + 255) // 256
    per_img = sum(ncb - (i >> 1) for i in range(nrb))
    tpad = 1
    while tpad < per_img:
        tpad <<= 1
    return n_img < 32768 and nrb < 256 and ncb < 256 and tpad * 8 <= 48 * 1024


# ----------------------------------------------------------------------------------- rounding boundaries
@pytest.mark.parametrize("h,w,layout,n_img", [(512, 512, "tiled", 3), (375, 500, "flat", 2)],
                         ids=["512x512-tiled", "375x500-flat"])
def test_rounding_boundaries(h, w, layout, n_img):
    """Masks whose quotients sit on and next to float16 rounding midpoints (exact ties, double-rounding ties, near
    misses within ratio_f16's +-8 ulp window, subnormal ties, the [2^-14, 6.2e-5) gap): image 1 random intervals, the
    others nested hazard pairs.  Tensor path and popcount path, both maps in full, against the reference."""
    total, words, n = h * w, (h * w + 31) // 32, mc.BOUNDARY_N
    imgs = mc.boundary_batch(total, n_img)
    refs = [mc.interval_counts(s, e) for s, e in imgs]
    packed = np.stack([mc.pack_intervals(s, e, words) for s, e in imgs])
    if total % 32:                                               # 375 x 500: the last word is partly padding
        assert not (packed[:, :, -1] >> np.uint32(total % 32)).any() and packed[:, :, -1].any()
    tot = {m: dict.fromkeys(mc.CLASSES, 0) for m in ("iou", "asy")}
    for b, (inter, area) in enumerate(refs):
        rows = np.random.default_rng(b).choice(n, 6, replace=False)
        p_inter, p_area = mc.popcount_counts(packed[b], rows)
        np.testing.assert_array_equal(p_area, area)
        np.testing.assert_array_equal(p_inter, inter[rows])
        for m, c in mc.class_counts(inter, area).items():
            for k, v in c.items():
                tot[m][k] += v
    print(f"\n{h}x{w} {layout}: class counts {tot}")
    for m in ("iou", "asy"):
        for k, lo in mc.MIN_PER_MAP.items():
            assert tot[m][k] >= lo, (m, k, tot[m][k])
    dev = cuda_words(packed)
    kb = w // 16 if layout == "tiled" else 0
    for algo in ("tensor", "popc"):
        out = mask_ops.mask_overlap(dev, return_counts=True, algo=algo, kb_per_row=kb)
        for b, (inter, area) in enumerate(refs):
            check_maps([o[b] for o in out], inter, area, f"{algo} image {b}")


# ----------------------------------------------------------------------------------- native image sizes
TENSOR_SIZES = {(375, 500), (333, 500), (500, 375), (427, 640), (480, 640)}
NATIVE = [(375, 500), (333, 500), (500, 375), (427, 640), (480, 640), (281, 500), (612, 612)]


def rasterize_hw(n, h, w, seed):
    """The synthetic proposals of a 512 x 512 image scaled into an h x w canvas, uint8 [n, h, w] on the device;
    mask 0 empty, mask 1 full, mask n - 1 a copy of mask 2."""
    p = synth.proposal_params(n, 512, seed)
    t = lambda a, s: torch.as_tensor(np.maximum(1, np.rint(a * s / 512.0)).astype(np.int64), device=DEV)
    cx, cy, ax, ay = t(p.cx, w), t(p.cy, h), t(p.ax, w), t(p.ay, h)
    xs, ys = torch.arange(w, device=DEV), torch.arange(h, device=DEV)
    out = torch.empty((n, h, w), dtype=torch.uint8, device=DEV)
    for s in range(0, n, 256):
        e = min(n, s + 256)
        dx2 = (xs[None, :] - cx[s:e, None]) ** 2
        dy2 = (ys[None, :] - cy[s:e, None]) ** 2
        a2, b2 = (ax[s:e] ** 2)[:, None, None], (ay[s:e] ** 2)[:, None, None]
        out[s:e] = (dx2[:, None, :] * b2 + dy2[:, :, None] * a2 <= a2 * b2).to(torch.uint8)
    out[0] = 0
    out[1] = 1
    out[n - 1] = out[2]
    return out


@pytest.mark.parametrize("h,w", NATIVE, ids=[f"{h}x{w}" for h, w in NATIVE])
@pytest.mark.parametrize("n", [300, 2000], ids=["n300", "n2000"])
def test_native_image_sizes(h, w, n):
    """VOC / COCO image sizes with algo="auto": the dispatch (tensor path for words % 4 == 0, popcount otherwise;
    tiled order only for H % 8 == W % 16 == 0) and the maps against the reference."""
    words = (h * w + 31) // 32
    assert ((h, w) in TENSOR_SIZES) == (words % 4 == 0)
    masks = rasterize_hw(n, h, w, seed=h + w + n)
    layout = "tiled" if mask_ops.tiled_ok(h, w) else "flat"
    assert layout == ("tiled" if (h, w) == (480, 640) else "flat")
    packed = mask_ops.mask_pack(masks)
    m_cpu = masks.cpu().numpy()
    want_packed = mc.pack_pixels(m_cpu, layout)
    np.testing.assert_array_equal(packed.cpu().numpy().view(np.uint32), want_packed)
    out = mask_ops.mask_overlap(packed, return_counts=True, return_visited=True)
    visited = out[-1]
    assert (visited > 0) == ((h, w) in TENSOR_SIZES), visited
    # counts: float32 matmul of the 0/1 masks (exact: partial sums are integers below 2^24), then sampled rows by
    # np.bitwise_count over the CPU-packed words
    flat = masks.view(n, -1)
    inter = torch.zeros((n, n), dtype=torch.float32, device=DEV)
    for k0 in range(0, h * w, 1 << 15):
        a = flat[:, k0:k0 + (1 << 15)].float()
        inter += a @ a.t()
    inter = inter.cpu().numpy().astype(np.int64)
    rows = np.random.default_rng(n).choice(n, 8, replace=False)
    p_inter, area = mc.popcount_counts(want_packed, rows)
    np.testing.assert_array_equal(inter[rows], p_inter)
    np.testing.assert_array_equal(np.diagonal(inter), area)
    check_maps(out, inter, area, f"{h}x{w} n={n}")


# ----------------------------------------------------------------------------------- 2 Mpixel masks
def big_masks(n, seed, h=2048, w=1024):
    """bool [n, h, w]: full, full minus k pixels (odd counts just below 2^21), one pixel in K-block 0 and one in the
    last K-block (the last bit of the last word, in both pixel orders), half-planes, random rectangles and their
    complements, an empty mask and a duplicate."""
    rng = np.random.default_rng(seed)
    m = np.zeros((n, h, w), bool)
    m[0] = True
    for j, k in enumerate((1, 3, 7, 127)):
        m[1 + j] = True
        idx = rng.choice(h * w, k, replace=False)
        m[1 + j].reshape(-1)[idx] = False
    m[5, 0, 5] = True                                   # K-block 0 (flat: row 0, x < 128; tiled: patch (0, 0))
    m[6, h - 1, w - 1] = True                           # K-block h w / 128 - 1, bit 31 of the last word
    m[7, :h // 2] = True
    m[8, h // 2:] = True
    m[9, :, :w // 2] = True
    m[10, :, w // 3:] = True
    # 11: empty
    k = 12
    while k < n - 1:
        y0, x0 = rng.integers(0, h - 1), rng.integers(0, w - 1)
        y1, x1 = rng.integers(y0 + 1, h + 1), rng.integers(x0 + 1, w + 1)
        m[k, y0:y1, x0:x1] = True
        if k + 1 < n - 1:
            m[k + 1] = ~m[k]
        k += 2
    m[n - 1] = m[3]
    return m


@pytest.mark.parametrize("layout", ["tiled", "flat"])
def test_largest_masks_on_the_tensor_path(layout):
    """2048 x 1024 masks: 65 536 words = 16 384 K-blocks, exactly the tile's K-block list; counts up to 2^21 in the
    fp32 accumulator of the mxf4 MMA."""
    h, w, n, n_img = 2048, 1024, 96, 2
    words = h * w // 32
    packed = np.stack([mc.pack_pixels(big_masks(n, 10 * b + (layout == "flat")), layout) for b in range(n_img)])
    assert packed.shape[-1] == 65536 and packed[0, 5, :4].any() and not packed[0, 5, 4:].any()
    assert packed[0, 6, -1] == np.uint32(1 << 31) and not packed[0, 6, :-1].any()
    refs = [mc.popcount_counts(p) for p in packed]
    for inter, area in refs:
        assert inter.max() == 1 << 21 and {(1 << 21) - k for k in (1, 3, 7, 127)} <= set(area.tolist())
        assert (area == 1).sum() >= 2 and (area == 0).sum() == 1
    dev = cuda_words(packed)
    out = mask_ops.mask_overlap(dev, return_counts=True, algo="tensor", kb_per_row=w // 16 if layout == "tiled" else 0,
                                return_visited=True)
    assert out[-1] > 0
    for b, (inter, area) in enumerate(refs):
        check_maps([o[b] for o in out[:4]], inter, area, f"{layout} image {b}")
    # and the popcount path agrees on everything
    pop = mask_ops.mask_overlap(dev, return_counts=True, algo="popc")
    for a, c in zip(out[:4], pop):
        assert f16_equal_dev(a, c) if a.dtype == torch.float16 else torch.equal(a, c)


def interval_case(words, n, seed):
    """n interval masks over `words` words: full, full minus one pixel at either end, empty, one pixel at the last
    position, random intervals."""
    total = 32 * words
    rng = np.random.default_rng(seed)
    s, e = mc.random_intervals(n, total, rng)
    s[:5], e[:5] = [0, 1, 0, 0, total - 1], [total, total, total - 1, 0, total]
    return s, e


def test_k_block_list_capacity_and_count_range():
    """65 540 words: one K-block more than the tile list holds -> the tensor path refuses, auto runs popcount.
    2^19 - 4 words (counts just below 2^24): popcount is exact.  2^19 words (2^24 pixels): refused."""
    words, n = 65540, 256                                        # n >= 256: auto would take the tensor path if it could
    s, e = interval_case(words, n, 1)
    inter, area = mc.interval_counts(s, e)
    packed = mc.pack_intervals(s, e, words)
    np.testing.assert_array_equal(mc.popcount_counts(packed, np.arange(4))[0], inter[:4])
    dev = cuda_words(packed)
    with pytest.raises(RuntimeError, match="shape"):
        mask_ops.mask_overlap(dev, algo="tensor")
    out = mask_ops.mask_overlap(dev, return_counts=True, return_visited=True)
    assert out[-1] == 0
    check_maps(out, inter, area, "65540 words")
    del dev, out

    words, n = (1 << 19) - 4, 8
    s, e = interval_case(words, n, 2)
    inter, area = mc.interval_counts(s, e)
    assert inter.max() == (1 << 24) - 128
    packed = mc.pack_intervals(s, e, words)
    p_inter, p_area = mc.popcount_counts(packed)
    np.testing.assert_array_equal(p_inter, inter)
    out = mask_ops.mask_overlap(cuda_words(packed), return_counts=True, return_visited=True)
    assert out[-1] == 0
    check_maps(out, inter, area, "2^19 - 4 words")

    big = torch.zeros((n, 1 << 19), dtype=torch.int32, device=DEV)
    for algo in ("auto", "popc", "tensor"):
        with pytest.raises(RuntimeError, match="shape"):
            mask_ops.mask_overlap(big, algo=algo)


# ----------------------------------------------------------------------------------- largest n
def small_masks(n, seed):
    """bool [n, 16, 32]: random rectangles with random holes, a few empty and full masks."""
    rng = np.random.default_rng(seed)
    y0, x0 = rng.integers(0, 15, n), rng.integers(0, 31, n)
    y1, x1 = rng.integers(y0 + 1, 17), rng.integers(x0 + 1, 33)
    ys, xs = np.arange(16)[None, :, None], np.arange(32)[None, None, :]
    m = (ys >= y0[:, None, None]) & (ys < y1[:, None, None]) & (xs >= x0[:, None, None]) & (xs < x1[:, None, None])
    m &= rng.random((n, 16, 32)) < 0.8
    m[::997] = False
    m[5::1009] = True
    return m


@pytest.mark.parametrize("n,n_img", [(16128, 1), (16129, 1), (16129, 2), (16384, 1)])
def test_largest_n_and_the_unranked_tile_order(n, n_img):
    """16 x 32 masks, n up to the API limit 16384: from n = 16129 an image has more than 4096 tiles and the tensor
    kernel decodes tiles by their distance from the diagonal instead of a ranking.  Tensor == popcount on the full
    maps, sampled rows against np.bitwise_count."""
    assert ordered_tiles(n, n_img) == (n <= 16128)
    packed = np.stack([mc.pack_pixels(small_masks(n, 100 * b + n), "tiled") for b in range(n_img)])
    dev = cuda_words(packed)
    t_iou, t_asy = mask_ops.mask_overlap(dev, algo="tensor", kb_per_row=2)
    counts = n == 16384
    pop = mask_ops.mask_overlap(dev, algo="popc", return_counts=counts)
    assert f16_equal_dev(t_iou, pop[0]) and f16_equal_dev(t_asy, pop[1])
    del t_iou, t_asy
    for b in range(n_img):
        rows = np.sort(np.random.default_rng(b).choice(n, 12, replace=False))
        rows[-1] = n - 1
        inter, area = mc.popcount_counts(packed[b], rows)
        o_iou, o_asy = mask_oracle.maps_from_counts(inter, area, row_area=area[rows])
        ridx = torch.as_tensor(rows, device=DEV)
        assert_f16_bits_equal(u16(pop[0][b][ridx]), o_iou.view(np.uint16))
        assert_f16_bits_equal(u16(pop[1][b][ridx]), o_asy.view(np.uint16))
        if counts:
            np.testing.assert_array_equal(pop[2][b][ridx].cpu().numpy(), inter)
            np.testing.assert_array_equal(pop[3][b].cpu().numpy(), area)
    del pop, dev
    gc.collect()
    torch.cuda.empty_cache()
    if n == 16384:
        with pytest.raises(RuntimeError, match="shape"):
            mask_ops.mask_overlap(torch.zeros((n + 1, 16), dtype=torch.int32, device=DEV), algo="popc")


# ----------------------------------------------------------------------------------- tile geometry sweep
def split_pool(n, seed):
    """bool [n, 16, 32] and group [n]: mask 1 empty (group -1), the others random non-empty pixel sets inside the
    top-left 8 x 16 patch (tiled K-block 0, group 0) or the bottom-right one (K-block 3, the last, group 1)."""
    rng = np.random.default_rng(seed)
    grp = rng.integers(0, 2, n)
    grp[1] = -1
    m = np.zeros((n, 16, 32), bool)
    for k in range(n):
        if grp[k] < 0:
            continue
        patch = rng.random((8, 16)) < rng.uniform(0.05, 0.9)
        patch[rng.integers(0, 8), rng.integers(0, 16)] = True
        if grp[k] == 0:
            m[k, :8, :16] = patch
        else:
            m[k, 8:, 16:] = patch
    return m, grp


def predicted_visited(grp):
    """K-blocks the tensor path visits for one image.  This follows the locality sort (mask_sort_kernel, tiled
    order): empty masks and the K-block-0 group have key 0 (stripe 0), the K-block-3 group is in stripe 1, ties
    keep the index order; a tile visits the K-blocks in both its row block's (128 masks) and its column block's
    (256 masks) unions."""
    n = len(grp)
    key = np.where(grp == 1, (1 << 24) | 2, 0)
    g = grp[np.lexsort((np.arange(n), key))]
    def union(lo, hi):
        return {0 if x == 0 else 3 for x in g[lo:hi] if x >= 0}
    nrb, ncb = (n + 127) // 128, (n + 255) // 256
    per_tile = [len(union(128 * ti, 128 * ti + 128) & union(256 * tj, 256 * tj + 256))
                for ti in range(nrb) for tj in range(ti >> 1, ncb)]
    return sum(per_tile), len(per_tile), min(per_tile)


@pytest.mark.parametrize("n_img", [1, 3], ids=["one_image", "three_images"])
def test_tile_geometry_sweep(n_img):
    """Every n from 64 to 640 (partial 128-row / 256-column blocks, the mirror rule, the n % 4 store path, the
    n % 8 / n % 2 unpermute branches), with an all-empty image between two normal ones for n_img = 3: tensor,
    popcount and the reference in full (inter, area, both maps), and the visited K-blocks as the sort predicts."""
    N = 640
    pools = [split_pool(N, 7 + b) for b in range(n_img)]
    if n_img == 3:
        pools[1] = (np.zeros((N, 16, 32), bool), np.full(N, -1))
    packed = cuda_words(np.stack([mc.pack_pixels(m, "tiled") for m, _ in pools]))
    ref_inter, ref_area, ref_iou, ref_asy = [], [], [], []
    for m, _ in pools:
        inter, area = mask_oracle.overlap_counts(m)
        iou, asy = mask_oracle.maps_from_counts(inter, area)
        ref_inter.append(inter)
        ref_area.append(area)
        ref_iou.append(iou)
        ref_asy.append(asy)
    to = lambda a, dt: torch.from_numpy(np.stack(a).astype(dt)).to(DEV)
    R_inter, R_area = to(ref_inter, np.int32), to(ref_area, np.int32)
    R_iou, R_asy = to(ref_iou, np.float16), to(ref_asy, np.float16)
    if n_img == 3:
        assert np.isnan(ref_iou[1]).all() and np.isnan(ref_asy[1]).all()
    skipped = 0
    for n in range(64, N + 1):
        p = packed[:, :n].contiguous()
        t = mask_ops.mask_overlap(p, return_counts=True, algo="tensor", kb_per_row=2, return_visited=True)
        c = mask_ops.mask_overlap(p, return_counts=True, algo="popc")
        want = (R_iou[:, :n, :n], R_asy[:, :n, :n], R_inter[:, :n, :n], R_area[:, :n])
        for k, (a, b, r) in enumerate(zip(t[:4], c, want)):
            if a.dtype == torch.float16:
                ok = f16_equal_dev(a, r) and f16_equal_dev(b, r)
            else:
                ok = torch.equal(a, r) and torch.equal(b, r)
            if not ok:                                   # readable failure: the first differing image on the CPU
                for img in range(n_img):
                    for got in (a, b):
                        if a.dtype == torch.float16:
                            assert_f16_bits_equal(u16(got[img]), u16(r[img]))
                        else:
                            np.testing.assert_array_equal(got[img].cpu().numpy(), r[img].cpu().numpy(),
                                                          err_msg=f"n={n} output {k}")
                raise AssertionError(f"n={n}: output {k} differs")
        pred = [predicted_visited(g[:n]) for _, g in pools]
        assert t[-1] == sum(v for v, _, _ in pred), (n, t[-1], pred)
        full = sum(2 * tiles for v, tiles, _ in pred if v)           # every tile of a normal image visiting both
        if any(lo == 0 and v for v, _, lo in pred):
            assert t[-1] < full, n
            skipped += 1
    assert skipped >= 300                                 # tiles with disjoint unions from n ~ 300 on
