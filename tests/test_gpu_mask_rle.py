"""COCO compressed RLE of selected proposal masks on the device (cim_mask_rle through mask_ops.mask_rle and
postproc.segms_batched), byte for byte against oracle/rle_oracle.py (pycocotools' maskApi.c restated), with exact areas
and boxes.  Each test first asserts that its inputs contain the case it is about."""
import numpy as np
import pytest
import torch

from cim_b200 import mask_ops, postproc, synth
from oracle import nms_oracle
from oracle import rle_oracle as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def synth_masks(n_img, n, H, W, seed):
    """Synthetic proposals (synth.proposal_params) cropped to H x W: uint8 [n_img, n, H, W]."""
    size = max(H, W)
    out = np.empty((n_img, n, H, W), np.uint8)
    for b in range(n_img):
        out[b] = synth.rasterize(synth.proposal_params(n, size, seed=seed + b), device=DEV)[:, :H, :W].cpu().numpy()
    return out


def encode(masks, sel_count, sel_idx, layout, mask_hw=None, chars_cap=None):
    H, W = masks.shape[-2:]
    packed = mask_ops.mask_pack(cuda(masks), layout=layout)
    assert packed.cim_kb_per_row == (W // 16 if layout == "tiled" else 0)
    out = mask_ops.mask_rle(packed, cuda(np.asarray(sel_count, np.int32)), cuda(np.asarray(sel_idx, np.int32)), H, W,
                            mask_hw=mask_hw, chars_cap=chars_cap)
    return [t.cpu().numpy() for t in out]


def check(masks, sel_count, sel_idx, out, mask_hw=None):
    """out = mask_rle's buffers for masks [B, R, H, W]; every slot against the oracle.  Returns the number of strings
    compared."""
    chars, off, len_, area, bbox, need = out
    B, Rn, H, W = masks.shape
    cap = sel_idx.shape[1]
    hw = np.tile([H, W], (B, 1)) if mask_hw is None else np.asarray(mask_hw)
    np.testing.assert_array_equal(off.reshape(-1), np.concatenate(([0], np.cumsum(len_.reshape(-1))[:-1])))
    assert need[0] == len_.sum()
    bad, checked = 0, 0
    for b in range(B):
        h, w = hw[b]
        for j in range(cap):
            i = sel_idx[b, j]
            if j >= min(max(sel_count[b], 0), cap) or not 0 <= i < Rn:
                bad += j < min(max(sel_count[b], 0), cap)
                assert len_[b, j] == 0 and area[b, j] == 0 and (bbox[b, j] == 0).all(), (b, j)
                continue
            d, a, bb = R.encode_mask(masks[b, i, :h, :w])
            assert len_[b, j] == len(d["counts"]), (b, j)
            assert area[b, j] == a, (b, j)
            np.testing.assert_array_equal(bbox[b, j], bb.astype(np.int32))
            if off[b, j] + len_[b, j] <= chars.size:
                assert chars[off[b, j]:off[b, j] + len_[b, j]].tobytes() == d["counts"], (b, j)
                checked += 1
    assert need[1] == bad
    return checked


def selection(rs, n_img, n, cap):
    return np.full(n_img, cap, np.int32), rs.randint(0, n, size=(n_img, cap)).astype(np.int32)


@pytest.mark.parametrize("H,W,layout", [(512, 512, "tiled"), (512, 512, "flat"), (480, 640, "tiled"),
                                        (480, 640, "flat"), (375, 500, "flat"), (333, 500, "flat")])
def test_synthetic_proposals(H, W, layout):
    assert (W % 32 != 0) == (W == 500)                   # the flat 500-wide cases have rows that are not word-aligned
    masks = synth_masks(2, 64, H, W, seed=H + W)
    assert masks.any(axis=(2, 3)).mean() > 0.5
    count, idx = selection(np.random.RandomState(H), 2, 64, 40)
    out = encode(masks, count, idx, layout)
    assert out[5][0] <= out[0].size
    assert check(masks, count, idx, out) == 80


@pytest.mark.parametrize("layout", ["tiled", "flat"])
def test_native_sizes_on_a_canvas_ignore_bits_outside(layout):
    H, W = 480, 640
    hw = np.array([[480, 640], [375, 500], [333, 499], [1, 1], [200, 33]], np.int32)
    rs = np.random.RandomState(5)
    masks = synth_masks(5, 32, H, W, seed=11)
    masks |= (rs.rand(5, 32, H, W) < 0.02).astype(np.uint8)  # set bits everywhere, outside the extents too
    assert all(masks[b, :, hw[b, 0]:, :].any() or masks[b, :, :, hw[b, 1]:].any() for b in range(1, 5))
    count, idx = selection(rs, 5, 32, 20)
    out = encode(masks, count, idx, layout, mask_hw=hw, chars_cap=10 ** 7)
    assert check(masks, count, idx, out, mask_hw=hw) == 100


def alternating(h, w):
    return ((np.arange(w)[None] * h + np.arange(h)[:, None] + 1) % 2).astype(np.uint8)


def edge_masks(h, w):
    """Empty, full, first pixel, last pixel, runs across every column boundary, alternating pixels in column-major
    order starting with a one (a checkerboard for odd h: a count per pixel, m = h*w + 1), a random one."""
    m = np.zeros((7, h, w), np.uint8)
    m[1] = 1
    m[2, 0, 0] = 1
    m[3, h - 1, w - 1] = 1
    m[4, h - 1, :] = 1
    m[4, 0, :] = 1                                         # (h-1, x) then (0, x+1): one run across the boundary
    m[5] = alternating(h, w)
    m[6] = np.random.RandomState(h * w).rand(h, w) < 0.5
    return m


@pytest.mark.parametrize("h,w,layout", [(32, 7, "flat"), (33, 5, "flat"), (63, 9, "flat"), (95, 33, "flat"),
                                        (1, 40, "flat"), (40, 1, "flat"), (1, 1, "flat"), (64, 48, "tiled"),
                                        (8, 16, "tiled"), (96, 80, "tiled")])
def test_edge_shapes_and_masks(h, w, layout):
    masks = edge_masks(h, w)[None]
    cnts = [R.encode(m) for m in masks[0]]
    assert cnts[2][0] == 0 and cnts[0].size == 1
    assert cnts[5].size == h * w + 1
    assert h < 3 or (cnts[4][:3].tolist() == [0, 1, h - 2] and (w == 1 or cnts[4][3] == 2))
    n = masks.shape[1]
    out = encode(masks, [n], np.arange(n, dtype=np.int32)[None], layout, chars_cap=10 ** 6)
    assert check(masks, np.array([n]), np.arange(n)[None], out) == n


def test_checkerboard_and_counts_of_two_to_the_twenty():
    h, w = 2048, 1024
    masks = np.zeros((1, 3, h, w), np.uint8)
    masks[0, 0] = alternating(h, w)                       # m = h*w + 1
    masks[0, 1, h - 1, w - 1] = 1                          # a count of h*w - 1
    masks[0, 2, 100:2000, 600:] = 1
    cnts = [R.encode(m) for m in masks[0]]
    assert cnts[0].size == h * w + 1 and cnts[1][0] >= 2 ** 20 and cnts[2].max() >= 2 ** 20
    count, idx = np.array([3], np.int32), np.array([[0, 1, 2]], np.int32)
    for layout in ("flat", "tiled"):
        out = encode(masks, count, idx, layout, chars_cap=0)
        need = int(out[5][0])
        assert need > h * w and out[0].size == 0
        out = encode(masks, count, idx, layout, chars_cap=need)
        assert check(masks, count, idx, out) == 3


def test_selections_empty_truncated_repeated_and_invalid():
    masks = synth_masks(4, 16, 64, 96, seed=3)
    count = np.array([0, 9, 3, 5], np.int32)               # image 0 selects nothing, image 1 more than cap = 6
    idx = np.array([[1, 2, 3, 4, 5, 6], [7, 7, 0, 15, 2, 7], [3, 16, -1, 0, 0, 0], [-5, 1, 1, 99, 2, 0]], np.int32)
    assert count[1] > idx.shape[1] and (idx[1, :6] == 7).sum() == 3
    out = encode(masks, count, idx, "flat")
    assert out[5][1] == 4                                  # 16, -1, -5 and 99 are outside [0, 16)
    assert (out[2][0] == 0).all() and (out[2][2, 1:] == 0).all()
    assert check(masks, count, idx, out) == 6 + 1 + 3
    dets = (cuda(count), cuda(np.zeros_like(idx)), cuda(idx))
    with pytest.raises(ValueError, match="outside"):
        postproc.segms_batched(mask_ops.mask_pack(cuda(masks), layout="flat"), dets, 64, 96, 2)


def test_too_small_capacity_writes_whole_strings_only():
    masks = edge_masks(33, 40)[None]
    n = masks.shape[1]
    count, idx = np.array([n], np.int32), np.arange(n, dtype=np.int32)[None]
    packed = mask_ops.mask_pack(cuda(masks), layout="flat")
    full = encode(masks, count, idx, "flat")
    ends = full[1][0] + full[2][0]
    cap = int(ends[4]) + 3                                 # strings 0..4 fit, string 5 does not
    assert ends[5] > cap
    chars = torch.full((cap,), 0xEE, dtype=torch.uint8, device=DEV)
    bufs = [torch.empty((1, n), dtype=torch.int64, device=DEV)] + [torch.empty(s, dtype=torch.int32, device=DEV)
                                                                   for s in ((1, n), (1, n), (1, n, 4))]
    need = torch.empty(2, dtype=torch.int64, device=DEV)
    mask_ops._mask_rle_into(packed, cuda(count), cuda(idx), 33, 40, None, 0, chars, *bufs, need)
    got = chars.cpu().numpy()
    np.testing.assert_array_equal(got[:ends[4]], full[0][:ends[4]])
    assert (got[ends[4]:] == 0xEE).all()
    assert int(need[0]) == int(full[5][0])
    # the host form: its first capacity (4 * (h + w) per slot) is too small for the checkerboards, the retry is exact
    big = np.stack([edge_masks(64, 64)[5]] * 3)[None]
    assert len(R.to_string(R.encode(big[0, 0]))) > 4 * 128 * 3
    dets = (cuda(np.array([3], np.int32)), cuda(np.array([[0, 0, 1]], np.int32)), cuda(np.array([[0, 1, 2]], np.int32)))
    res = postproc.segms_batched(mask_ops.mask_pack(cuda(big), layout="tiled"), dets, 64, 64, 2)
    want = R.to_string(R.encode(big[0, 0]))
    segms = res[0][0]
    assert [len(s) for s in segms] == [0, 2, 1]
    assert all(d == {"size": [64, 64], "counts": want} for d in segms[1] + segms[2])


@pytest.mark.parametrize("layout", ["tiled", "flat"])
def test_end_to_end_detections_then_segms(layout):
    B, n, C, H, W, D = 3, 96, 6, 160, 224, 20
    masks = synth_masks(B, n, H, W, seed=21)
    rs = np.random.RandomState(21)
    boxes = np.empty((B, n, 4), np.float32)
    for b in range(B):
        ys, xs = masks[b].any(2), masks[b].any(1)
        boxes[b] = np.stack([xs.argmax(1), ys.argmax(1), W - 1 - xs[:, ::-1].argmax(1), H - 1 - ys[:, ::-1].argmax(1)],
                            1)
    scores = (rs.rand(B, n, C) ** 3).astype(np.float32)
    hw = np.array([[160, 224], [150, 200], [97, 131]], np.int32)
    dets = postproc.detections_batched(cuda(scores), cuda(boxes), 1e-5, 0.3, D)
    res = postproc.segms_batched(mask_ops.mask_pack(cuda(masks), layout=layout), dets, H, W, C, mask_hw=hw)
    total = 0
    for b in range(B):
        _, o_inds = nms_oracle.results_with_nms_and_limit(scores[b], boxes[b], 1e-5, 0.3, D)
        segms, areas, bboxes = res[b]
        assert len(segms) == C + 1 and segms[0] == [] and areas[0] == [] and bboxes[0] == []
        h, w = hw[b]
        for j in range(C):
            want = [R.encode_mask(masks[b, i, :h, :w]) for i in o_inds[j]]
            assert segms[j + 1] == [d for d, _, _ in want]
            assert areas[j + 1].dtype == np.uint32 and areas[j + 1].tolist() == [a for _, a, _ in want]
            assert bboxes[j + 1].dtype == np.float64
            np.testing.assert_array_equal(bboxes[j + 1].reshape(-1, 4), np.array([bb for _, _, bb in want]).reshape(-1, 4))
            total += len(want)
    assert total == int(dets[0].sum()) and total >= B


def test_two_runs_give_identical_buffers():
    masks = synth_masks(2, 48, 480, 640, seed=9)
    count, idx = selection(np.random.RandomState(9), 2, 48, 30)
    a = encode(masks, count, idx, "tiled")
    b = encode(masks, count, idx, "tiled")
    n = int(a[5][0])
    assert np.array_equal(a[0][:n], b[0][:n])
    for x, y in zip(a[1:], b[1:]):
        np.testing.assert_array_equal(x, y)
