"""Per-image feature-map extents without a GPU: the window plan with extents (cim_debug_roi_window_plan_ex) rebuilt
into a forward and compared with the oracle on each image's cropped map, argument validation of the RoIAlign _ex entry
points and of _lib.feat_hw_arg, and the batch wire format of mask_ops.batch_crops_host decoded on the CPU."""
import ctypes as C

import numpy as np
import pytest
import torch

from cim_b200 import _lib, mask_ops
from oracle import roi_oracle
from test_roi_window_plan import DESC_WORDS, D_ROI, D_WX, D_WY, D_XLO, D_XMAP, D_YLO, D_YMAP, D_YN, rebuild_forward

NULL = C.c_void_p(0)
FAKE = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch
ODD = C.c_void_p(4098)            # a feat_hw pointer that is not 4-byte aligned


def plan_ex(rois, feat_hw, B, H, W, scale, sr=0, aligned=True, cap_per_roi=49):
    K = len(rois)
    rois = np.ascontiguousarray(rois, np.float32)
    hw = np.ascontiguousarray(feat_hw, np.int32)
    desc = np.zeros((K * cap_per_roi, DESC_WORDS), np.int32)
    keys = np.zeros(K * cap_per_roi, np.int32)
    flags = np.zeros(K, np.int32)
    geom = np.zeros(6, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    n = _lib.lib().cim_debug_roi_window_plan_ex(p(rois), p(hw), K, B, H, W, float(scale), sr, int(aligned), p(desc),
                                                p(keys), K * cap_per_roi, p(flags), p(geom))
    assert n >= 0, n
    return desc[:n], keys[:n], flags, geom


def per_image_oracle(feat, rois, hw, scale, sr, aligned):
    """RoIAlign of every roi on its image's cropped map feat[b, :, :H_b, :W_b] alone."""
    out = np.zeros((len(rois), feat.shape[1], 7, 7), np.float64)
    for b in range(feat.shape[0]):
        sel = np.nonzero(rois[:, 0] == b)[0]
        if len(sel):
            r = rois[sel].copy()
            r[:, 0] = 0
            out[sel] = roi_oracle.roi_align_fwd(np.ascontiguousarray(feat[b:b + 1, :, :hw[b, 0], :hw[b, 1]]), r, 7, 7,
                                                scale, sr, aligned)
    return out


def extent_rois(rng, B, hw, scale, K):
    """Random rois per image plus, for every image, boxes on and beyond its bottom / right edge."""
    rows = []
    for k in range(K):
        b = k % B
        sh, sw = hw[b, 0] / scale, hw[b, 1] / scale
        w, h = rng.uniform(0.05, 1.0) * sw, rng.uniform(0.05, 1.0) * sh
        x1, y1 = rng.uniform(0, 1) * max(sw - w, 1), rng.uniform(0, 1) * max(sh - h, 1)
        rows.append([b, x1, y1, x1 + w, y1 + h])
    for b in range(B):
        sh, sw = hw[b, 0] / scale, hw[b, 1] / scale
        rows += [[b, 0, 0, sw, sh],                                       # the whole image, edge to edge
                 [b, sw * 0.5, sh * 0.5, sw, sh],                         # touching the bottom-right corner
                 [b, sw * 0.7, sh * 0.2, sw * 1.4, sh * 0.6],             # beyond the right edge
                 [b, sw * 0.1, sh * 0.8, sw * 0.5, sh * 1.5]]             # beyond the bottom edge
    return np.array(rows, np.float32)


CASES = [
    # canvas H, W, scale, extents
    (64, 64, 1 / 8, [(64, 48), (43, 64), (64, 64)]),          # VGG-16 canvas
    (75, 75, 1 / 16, [(75, 56), (43, 75), (60, 71)]),         # R-50 training scales 688 .. 1200
    (43, 57, 1 / 16, [(43, 57), (31, 40), (17, 29)]),         # odd sizes, H odd
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("aligned,sr", [(True, 0), (False, 0), (True, 2), (False, 2)])
def test_window_plan_with_extents_matches_oracle_on_cropped_maps(case, aligned, sr):
    H, W, scale, ext = case
    B, Cc, K = len(ext), 2, 45
    hw = np.array(ext, np.int32)
    rng = np.random.RandomState(H * 100 + W + 3 * int(aligned) + sr)
    feat = rng.randn(B, Cc, H, W).astype(np.float32)          # the canvas outside the extents holds other data
    garbage, zero = feat.copy(), feat.copy()
    for b, (h, w) in enumerate(ext):
        garbage[b, :, h:, :] = 1e30                                       # large finite values
        garbage[b, :, :, w:] = -1e30
        zero[b, :, h:, :] = 0
        zero[b, :, :, w:] = 0
    rois = extent_rois(rng, B, hw, scale, K)
    desc, keys, flags, geom = plan_ex(rois, hw, B, H, W, scale, sr, aligned)
    ok = flags == 0
    assert ok.sum() >= len(rois) * 0.8
    want = per_image_oracle(feat, rois, hw, scale, sr, aligned)
    # the inputs discriminate: the canvas-wide oracle differs from the per-image one on edge rois
    canvas = roi_oracle.roi_align_fwd(feat, rois, 7, 7, scale, sr, aligned)
    assert np.abs(canvas - want).max() > 1e-3 * np.abs(want).max()
    got, written = rebuild_forward(feat, rois, desc, keys, geom)
    assert (written[ok] == 1).all()
    assert np.abs(got[ok] - want[ok]).max() <= 1e-5 * np.abs(want).max()
    for other in (garbage, zero):
        got_o, _ = rebuild_forward(other, rois, desc, keys, geom)
        assert np.array_equal(got_o[ok], got[ok])
    # no tap of nonzero weight lies outside the roi's image
    Hp, wh, ww, nwy, nwx, G = (int(v) for v in geom)
    f32 = lambda a: a.view(np.float32)
    for d, key in zip(desc, keys):
        b = int(rois[int(d[D_ROI]), 0])
        wy, wx = divmod(int(key), nwx)
        oy, ox = min(wy * G, Hp - wh), min(wx * G, W - ww)
        ny, nx = (int(np.uint32(d[D_YMAP])) >> 28) & 7, (int(np.uint32(d[D_XMAP])) >> 28) & 7
        for s in range(ny):
            wyv = f32(d[D_WY + s * 10 + 1:D_WY + s * 10 + 9])
            rows = oy + int(d[D_YLO + s]) + np.nonzero(wyv)[0]
            assert (rows < hw[b, 0]).all()
        for s in range(nx):
            wxv = f32(d[D_WX + s * 8:D_WX + s * 8 + 8])
            cols = ox + int(d[D_XLO + s]) + np.nonzero(wxv)[0]
            assert (cols < hw[b, 1]).all()


def test_window_plan_ex_null_and_full_extents_equal_the_plain_plan():
    H, W, scale, B = 64, 64, 1 / 8, 2
    rng = np.random.RandomState(5)
    rois = extent_rois(rng, B, np.array([[H, W]] * B), scale, 30)
    rois_c = np.ascontiguousarray(rois, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    cap = len(rois) * 49
    outs = []
    for hw in (None, np.array([[H, W]] * B, np.int32), np.array([[H + 9, W + 100]] * B, np.int32)):
        desc, keys = np.zeros((cap, DESC_WORDS), np.int32), np.zeros(cap, np.int32)
        flags, geom = np.zeros(len(rois), np.int32), np.zeros(6, np.int32)
        n = _lib.lib().cim_debug_roi_window_plan_ex(p(rois_c), NULL if hw is None else p(hw), len(rois), B, H, W, scale,
                                                    0, 1, p(desc), p(keys), cap, p(flags), p(geom))
        outs.append((desc[:n], keys[:n], flags))
    desc, keys, flags, geom = np.zeros((cap, DESC_WORDS), np.int32), np.zeros(cap, np.int32), \
        np.zeros(len(rois), np.int32), np.zeros(6, np.int32)
    n = _lib.lib().cim_debug_roi_window_plan(p(rois_c), len(rois), B, H, W, scale, 0, 1, p(desc), p(keys), cap,
                                             p(flags), p(geom))
    for d, k, f in outs:                        # (values above the canvas are clamped to it, as on the device)
        assert np.array_equal(d, desc[:n]) and np.array_equal(k, keys[:n]) and np.array_equal(f, flags)


def test_window_plan_ex_argument_validation():
    L = _lib.lib()
    rois = np.zeros((1, 5), np.float32)
    buf = np.zeros(49 * DESC_WORDS, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    call = lambda r=p(rois), hw=NULL, B=1, H=64, W=64: L.cim_debug_roi_window_plan_ex(
        r, hw, 1, B, H, W, 0.125, 0, 1, p(buf), p(buf), 49, p(buf), p(buf))
    assert call() >= 0
    assert call(r=NULL) == -1 and call(B=0) == -1 and call(H=0) == -1 and call(W=4) == -1
    assert call(hw=ODD) == -4


def test_roi_align_ex_argument_validation():
    L = _lib.lib()
    big = 1 << 40
    prep = lambda r=FAKE, hw=FAKE, B=2, C_=64, H=32, W=32, K=10, ws=FAKE, ws_bytes=big: L.cim_roi_align_prepare_ex(
        r, hw, B, C_, H, W, K, 7, 7, 0.0625, 0, 1, ws, ws_bytes, NULL)
    for kw in ({"r": NULL}, {"B": 0}, {"C_": 0}, {"H": 0}, {"W": -1}, {"K": -1}):
        assert prep(**kw) == -1, kw
    assert prep(B=4097) == -2 and prep(H=1 << 13, W=1 << 12) == -2
    assert prep(ws=NULL) == -3 and prep(ws_bytes=64) == -3
    assert prep(hw=ODD) == -4 and prep(ws=C.c_void_p(4104)) == -4
    assert prep(K=0) == 0                                                  # nothing to do
    for fn in (L.cim_roi_align_fwd_prepared_ex, L.cim_roi_align_bwd_prepared_ex):
        call = lambda a=FAKE, r=FAKE, hw=FAKE, out=FAKE, B=2, K=10, ws=FAKE, ws_bytes=big: fn(
            a, r, hw, NULL, out, B, 64, 32, 32, K, 7, 7, 0.0625, 0, 1, ws, ws_bytes, NULL)
        for kw in ({"a": NULL}, {"r": NULL}, {"out": NULL}, {"B": 0}, {"K": -1}):
            assert call(**kw) == -1, (fn, kw)
        assert call(B=4097) == -2
        assert call(ws=NULL) == -3 and call(ws_bytes=64) == -3
        assert call(hw=ODD) == -4 and call(a=C.c_void_p(4100)) == -4


def test_feat_hw_arg_validation():
    assert _lib.feat_hw_arg(None, 2, 32, 32, "cpu") is None
    t = _lib.feat_hw_arg([[32, 24], [17, 29]], 2, 32, 32, "cpu")
    assert t.dtype == torch.int32 and t.tolist() == [[32, 24], [17, 29]]
    assert _lib.feat_hw_arg(np.array([[1, 1]], np.int64), 1, 32, 32, "cpu").tolist() == [[1, 1]]
    assert _lib.feat_hw_arg(torch.tensor([[5, 6]], dtype=torch.int16), 1, 32, 32, "cpu").tolist() == [[5, 6]]
    for bad, exc in (([[32, 24]], ValueError),                     # shape
                     ([32, 24, 17, 29], ValueError),
                     ([[32, 24, 1], [17, 29, 1]], ValueError),
                     ([[32.0, 24.0], [17.0, 29.0]], TypeError),    # dtype
                     ([[0, 24], [17, 29]], ValueError),            # 0
                     ([[32, 0], [17, 29]], ValueError),
                     ([[33, 24], [17, 29]], ValueError),           # > H
                     ([[32, 24], [17, 33]], ValueError)):          # > W
        with pytest.raises(exc):
            _lib.feat_hw_arg(bad, 2, 32, 32, "cpu")


# ------------------------------------------------------------------ batch crop wire format
def decode_crops(crops, n, height, width):
    """MaskCrops -> uint8 masks [n, height, width] (what the unpack kernels build on the device)."""
    words = crops.words.numpy().view(np.uint32)
    out = np.zeros((n, height, ((width + 31) // 32) * 32), np.uint8)
    for i in range(n):
        wx0, y0, ww, h = (int(v) for v in crops.meta[i])
        if ww == 0 or h == 0:
            continue
        o = int(crops.off[i])
        blk = words[o:o + ww * h].reshape(h, ww)
        bits = np.unpackbits(blk.view(np.uint8).reshape(h, ww * 4), axis=1, bitorder="little")
        out[i, y0:y0 + h, 32 * wx0:32 * (wx0 + ww)] = bits
    return out[:, :, :width]


def random_masks(rng, n, h, w):
    m = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        if i % 7 == 3:
            continue                                        # an empty proposal
        y0, x0 = rng.randint(0, h), rng.randint(0, w)
        m[i, y0:rng.randint(y0 + 1, h + 1), x0:rng.randint(x0 + 1, w + 1)] = rng.rand() < 2
    m[0, -1, -1] = 1                                        # touches the image's bottom-right corner
    return m


def test_batch_crops_decode_to_the_canvas_padded_masks():
    rng = np.random.RandomState(11)
    R, H, W = 12, 128, 128
    sizes, counts = [(120, 96), (96, 128), (80, 128), (128, 50)], [12, 5, 9, 1]
    masks = [random_masks(rng, n, h, w) for n, (h, w) in zip(counts, sizes)]
    crops = mask_ops.batch_crops_host([mask_ops.pack_crops_host(m) for m in masks], R, H, W)
    assert (crops.height, crops.width) == (H, W) and crops.meta.shape == (len(sizes) * R, 4)
    got = decode_crops(crops, len(sizes) * R, H, W)
    want = np.zeros_like(got)
    for b, m in enumerate(masks):
        want[b * R:b * R + len(m), :m.shape[1], :m.shape[2]] = m
    assert np.array_equal(got, want)
    for b, n in enumerate(counts):                          # padding rows are empty crops
        assert not crops.meta[b * R + n:(b + 1) * R].numpy().any()
    off = crops.off.numpy()
    sizes_w = crops.meta[:, 2].numpy().astype(np.int64) * crops.meta[:, 3].numpy()
    assert (np.diff(off) == sizes_w[:-1]).all() and off[-1] + sizes_w[-1] == crops.words.numel()


def test_batch_crops_reject_what_does_not_fit():
    rng = np.random.RandomState(2)
    ok = mask_ops.pack_crops_host(random_masks(rng, 4, 40, 70))
    mask_ops.batch_crops_host([ok], 4, 40, 70)
    mask_ops.batch_crops_host([ok], 4, 40, 96)              # 70 px = 3 words, 96 px = 3 words
    with pytest.raises(ValueError):
        mask_ops.batch_crops_host([ok], 3, 40, 70)          # more masks than R
    with pytest.raises(ValueError):
        mask_ops.batch_crops_host([ok], 4, 39, 70)          # taller than the canvas
    with pytest.raises(ValueError):
        mask_ops.batch_crops_host([ok], 4, 40, 64)          # wider than the canvas
    m = np.zeros((1, 40, 64), np.uint8)
    m[0, 5, 63] = 1
    c = mask_ops.pack_crops_host(m)
    c.meta[0, 0] = 2                                        # a crop at word 2 of a 2-word (64 px) canvas
    with pytest.raises(ValueError):
        mask_ops.batch_crops_host([mask_ops.MaskCrops(c.words, c.meta, c.off, 40, 64)], 1, 40, 64)
    c.meta[0, 0], c.meta[0, 1] = 1, 39                      # rows 39 .. 39 fit, 40 do not
    mask_ops.batch_crops_host([c], 1, 40, 64)
    c.meta[0, 1] = 40
    with pytest.raises(ValueError):
        mask_ops.batch_crops_host([c], 1, 40, 64)
