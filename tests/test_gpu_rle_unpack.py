"""COCO compressed RLE strings -> tiled bit masks and their metadata on the device (cim_mask_unpack_rle_tiled_meta_sparse,
mask_ops.unpack_rle, the RLE wire of CIMHeadStep.run_host).  Every comparison is bit for bit: packed words, metadata
bytes (areas, sort keys, K-block bitmaps) and the rectangles the sparse update keeps, against mask_pack + mask_meta,
the crop wire and the oracle's strings (oracle/rle_oracle.py; parity with pycocotools itself is unpinned)."""
import numpy as np
import pytest
import torch

from cim_b200 import _lib, heads, mask_ops, synth
from cim_b200.step import CIMHeadStep
from oracle import rle_oracle as R
from test_gpu_compact import real_rows
from test_gpu_roi_extents import host_problem
from test_rle_oracle_cpu import HAND

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------- helpers
def meta_parts(meta, n_img, n, words):
    """(areas, sort keys, K-block bitmaps) of a cim_mask_meta buffer as byte tensors (the padding between is not data)"""
    nm, bw = n_img * n, ((words // 4) + 31) // 32
    up = lambda v: (v + 255) & ~255
    a0, k0, b0 = 0, up(nm * 4), up(nm * 4) + up(nm * 16)
    return meta[a0:a0 + nm * 4], meta[k0:k0 + nm * 16], meta[b0:b0 + nm * bw * 4]


def dense(canvas):
    """uint8 [n_img, n, H, W] canvas masks -> (tiled packed, metadata) by mask_pack + mask_meta"""
    packed = mask_ops.mask_pack(canvas.to(DEV), layout="tiled")
    return packed, mask_ops.mask_meta(packed)


def assert_same(got, got_meta, want, want_meta):
    n_img, n, words = want.shape
    assert torch.equal(got.view(n_img, n, words), want), "packed masks differ"
    for g, w, what in zip(meta_parts(got_meta, n_img, n, words), meta_parts(want_meta, n_img, n, words),
                          ("areas", "sort keys", "K-block bitmaps")):
        assert torch.equal(g, w), f"{what} differ"


def encode_host(native, R_cap, H, W):
    """per-image uint8 [n_b, h, w] numpy masks -> host MaskRLE through the oracle's C encoder"""
    enc = R.CEncoder(max(m.shape[1] * m.shape[2] for m in native))
    per_image = [[{"size": list(m.shape), "counts": enc(np.asfortranarray(m))} for m in nm] for nm in native]
    return mask_ops.batch_rle_host(per_image, R_cap, H, W)


def to_dev(rle):
    return mask_ops.MaskRLE(rle.chars.to(DEV), rle.off.to(DEV), rle.len.to(DEV), rle.hw.to(DEV), rle.height, rle.width)


def canvas_of(native, R_cap, H, W):
    c = torch.zeros(len(native), R_cap, H, W, dtype=torch.uint8)
    for b, m in enumerate(native):
        c[b, :m.shape[0], :m.shape[1], :m.shape[2]] = torch.from_numpy(np.ascontiguousarray(m))
    return c


def device_encode(packed, H, W, mask_hw=None):
    """every proposal of packed [n_img, R, words] through mask_rle -> a device MaskRLE (the round trip)"""
    n_img, R_cap, _ = packed.shape
    cnt = torch.full((n_img,), R_cap, dtype=torch.int32, device=DEV)
    idx = torch.arange(R_cap, dtype=torch.int32, device=DEV).repeat(n_img, 1).contiguous()
    chars, off, ln, _, _, need = mask_ops.mask_rle(packed, cnt, idx, H, W, mask_hw=mask_hw)
    if int(need[0]) > chars.numel():
        chars, off, ln, _, _, need = mask_ops.mask_rle(packed, cnt, idx, H, W, mask_hw=mask_hw,
                                                      chars_cap=int(need[0]))
    hw = torch.tensor(mask_hw if mask_hw is not None else [[H, W]] * n_img, dtype=torch.int32, device=DEV)
    return mask_ops.MaskRLE(chars, off.view(-1), ln.view(-1), hw, H, W)


def synth_native(n, size, h, w, seed):
    return synth.rasterize(synth.proposal_params(n, size, seed))[:, :h, :w].numpy()


# ------------------------------------------------------------------------------------------------- 1. batches
def test_cfg2_size_proposals_equal_mask_pack_and_mask_meta():
    """8 x 2000 proposals of 512 x 512 (the bench's synthetic masks, seeds 1234 + b), strings from the device encoder;
    a sample of them equals the oracle's C encoder."""
    n_img, R_cap, S = 8, 2000, 512
    canvas = torch.stack([synth.rasterize(synth.proposal_params(R_cap, S, 1234 + b), device=DEV) for b in range(n_img)])
    want, want_meta = dense(canvas)
    rle = device_encode(want, S, S)
    got, got_meta = mask_ops.unpack_rle(rle, meta=True)
    assert_same(got, got_meta, want, want_meta)
    assert got.cim_kb_per_row == S // 16
    enc = R.CEncoder(S * S)
    chars, off, ln = rle.chars.cpu().numpy().tobytes(), rle.off.cpu().numpy(), rle.len.cpu().numpy()
    for r in range(0, n_img * R_cap, 997):
        m = canvas[r // R_cap, r % R_cap].cpu().numpy()
        assert chars[off[r]:off[r] + ln[r]] == enc(np.asfortranarray(m))


def test_cfg4_size_proposals_from_the_oracle_encoder():
    n_img, R_cap, S = 8, 2000, 128
    native = [synth.rasterize(synth.proposal_params(R_cap, 512, 1234 + b), out_size=S).numpy() for b in range(n_img)]
    want, want_meta = dense(canvas_of(native, R_cap, S, S))
    got, got_meta = mask_ops.unpack_rle(to_dev(encode_host(native, R_cap, S, S)), meta=True)
    assert_same(got, got_meta, want, want_meta)


def mixed_native():
    """500 x 375 next to 375 x 500 and a 1 x 1 image on a 512 x 512 canvas, ragged counts"""
    sizes, counts = [(500, 375), (375, 500), (1, 1)], [300, 170, 3]
    native = [synth_native(n, 512, h, w, 40 + b) for b, (n, (h, w)) in enumerate(zip(counts, sizes))]
    native[2][1] = 1
    return native, 300, 512, 512


def test_mixed_native_sizes_on_one_canvas():
    native, R_cap, H, W = mixed_native()
    want, want_meta = dense(canvas_of(native, R_cap, H, W))
    rle = encode_host(native, R_cap, H, W)
    assert rle.hw.tolist() == [[500, 375], [375, 500], [1, 1]]
    got, got_meta = mask_ops.unpack_rle(to_dev(rle), meta=True)
    assert_same(got, got_meta, want, want_meta)


# ------------------------------------------------------------------------------------------------- 2. + 3. strings
def one_row(strings_and_masks, H, W):
    """[(counts bytes, uint8 [h, w] mask)] as one image each -> (got packed, got meta, want packed, want meta)"""
    per_image = [[{"size": list(m.shape), "counts": s}] for s, m in strings_and_masks]
    rle = mask_ops.batch_rle_host(per_image, 1, H, W)
    got, got_meta = mask_ops.unpack_rle(to_dev(rle), meta=True)
    want, want_meta = dense(canvas_of([m[None] for _, m in strings_and_masks], 1, H, W))
    return got, got_meta, want, want_meta


@pytest.mark.parametrize("case", range(len(HAND)))
def test_hand_worked_strings(case):
    """negative delta, the sign continuation, a run across a column boundary, a count of 999999 (1000 x 1000 on a
    1000 x 1008 canvas: four bands of 256 rows)"""
    mask, _, string = HAND[case]
    h, w = mask.shape
    H, W = (h + 7) // 8 * 8, (w + 15) // 16 * 16
    assert_same(*one_row([(string, mask)], H, W))


def structured(h, w):
    alt = (np.arange(h * w) % 2 == 0).astype(np.uint8).reshape(w, h).T          # column-major 1, 0, 1, ...: h*w+1 counts
    out = [np.zeros((h, w), np.uint8), np.ones((h, w), np.uint8), alt, 1 - alt]
    for y, x in ((0, 0), (h - 1, 0), (0, w - 1), (h - 1, w - 1)):
        m = np.zeros((h, w), np.uint8)
        m[y, x] = 1
        out.append(m)
    return out


@pytest.mark.parametrize("h,w,H,W", [(64, 96, 64, 96), (61, 83, 64, 96), (1024, 1024, 1024, 1024),
                                     (997, 1001, 1000, 1008)])
def test_structured_masks(h, w, H, W):
    """empty (counts = [h*w]), full, alternating pixels (h*w + 1 counts), single corner pixels; the large canvases
    need several bands of the shared-memory bitmap"""
    masks = structured(h, w)
    assert R.encode(masks[2]).size == h * w + 1
    enc = R.CEncoder(h * w)
    assert_same(*one_row([(enc(np.asfortranarray(m)), m) for m in masks], H, W))


# ------------------------------------------------------------------------------------------------- 4. round trip
@pytest.mark.parametrize("with_hw", [False, True])
def test_round_trip_through_the_device_encoder(with_hw):
    native, R_cap, H, W = mixed_native()
    want, want_meta = dense(canvas_of(native, R_cap, H, W))
    rle = device_encode(want, H, W, mask_hw=[list(m.shape[1:]) for m in native] if with_hw else None)
    got, got_meta = mask_ops.unpack_rle(rle, meta=True)
    assert_same(got, got_meta, want, want_meta)


# ------------------------------------------------------------------------------------------------- 5. sparse update
def test_sparse_update_over_successive_batches_equals_the_crops_and_the_dense_path():
    """one buffer updated batch after batch by the RLE kernel, another by the crop kernel: rows grow, shrink, move, go
    empty, become padding, and the images change their native size.  After every batch both equal the dense packing,
    metadata and rectangles included."""
    n_img, n, H, W = 2, 120, 64, 96
    words = H * W // 32
    L = _lib.lib()
    st = _lib.stream_ptr(torch.device(DEV))
    bufs = {k: (torch.zeros(n_img, n, words, dtype=torch.int32, device=DEV),
                torch.zeros(n_img * n, 4, dtype=torch.int32, device=DEV),
                torch.zeros(L.cim_mask_meta_bytes(n_img, n, words), dtype=torch.uint8, device=DEV))
            for k in ("rle", "crops")}
    bad = torch.full((1,), 7, dtype=torch.int32, device=DEV)
    sizes = [[(64, 96), (50, 70)], [(33, 96), (64, 80)], [(64, 96), (64, 96)], [(8, 16), (60, 90)], [(64, 96), (1, 1)]]
    counts = [[120, 90], [60, 120], [120, 30], [5, 119], [110, 1]]
    for batch in range(len(sizes)):
        g = np.random.RandomState(100 + batch)
        native = []
        for b in range(n_img):
            h, w = sizes[batch][b]
            m = np.zeros((counts[batch][b], h, w), np.uint8)
            for i in range(m.shape[0]):
                if (i + batch) % 11 == 3:
                    continue                                             # empty in this batch
                y0, x0 = g.randint(h), g.randint(w)
                y1, x1 = g.randint(y0 + 1, h + 1), g.randint(x0 + 1, w + 1)
                m[i, y0:y1, x0:x1] = g.rand(y1 - y0, x1 - x0) < 0.5
            native.append(m)
        want, want_meta = dense(canvas_of(native, n, H, W))
        rle = to_dev(encode_host(native, n, H, W))
        packed, prev, meta = bufs["rle"]
        mask_ops._unpack_rle_into(rle, packed, prev, meta, bad, n_img, n, st)
        c = mask_ops.batch_crops_host([mask_ops.pack_crops_host(m) for m in native], n, H, W)
        cp, cprev, cmeta = bufs["crops"]
        cw, cm, co = c.words.to(DEV), c.meta.to(DEV), c.off.to(DEV)
        _lib.check(L.cim_mask_unpack_crops_tiled_meta_sparse(_lib.ptr(cw), _lib.ptr(cm), _lib.ptr(co), _lib.ptr(cp),
                                                             _lib.ptr(cprev),
                                                             _lib.ptr(cmeta), cmeta.numel(), n_img, n, H, W, words, st),
                   "crop sparse unpack")
        assert int(bad) == 0
        assert_same(packed, meta, want, want_meta)
        assert_same(cp, cmeta, want, want_meta)
        assert torch.equal(prev, cprev), f"batch {batch}: rectangles differ"
        assert torch.equal(prev.cpu(), c.meta)


# ------------------------------------------------------------------------------------------------- 6. malformed
def test_malformed_strings_give_empty_rows_and_are_counted():
    """each kind of malformed string, surrounded by valid rows, over a buffer that held masks in every row"""
    n, H, W, h, w = 12, 16, 32, 12, 20
    hw = h * w
    rs = np.random.RandomState(5)
    masks = (rs.rand(n, h, w) < 0.3).astype(np.uint8)
    enc = R.CEncoder(hw)
    good = [enc(np.asfortranarray(m)) for m in masks]
    bad_strings = {
        1: good[1][:-1] + b"/",                               # a character below 48
        3: good[3][:-1] + b"p",                               # a character above 111
        5: good[5] + b"P",                                    # the last character still has the continuation bit
        7: R.to_string(np.array([3, -1, hw - 2], np.int64)),  # a count of 2^32 - 1 after the (uint) cast
        8: R.to_string(np.array([hw + 1], np.int64)),         # a count above h * w
        9: R.to_string(np.array([1, 2], np.int64)),           # counts summing to less than h * w
    }
    strings = [bad_strings.get(i, good[i]) for i in range(n)]
    per_image = [[{"size": [h, w], "counts": s} for s in strings]]
    rle = mask_ops.batch_rle_host(per_image, n, H, W)
    rle.off[10] = rle.chars.numel() - 2                       # 10: off + len beyond the characters
    n_bad = len(bad_strings) + 1
    # the buffer first holds full masks in every row, so a malformed row must also clear what was there
    full = mask_ops.batch_rle_host([[{"size": [h, w], "counts": R.to_string(np.array([0, hw], np.int64))}] * n], n, H, W)
    words = H * W // 32
    packed = torch.zeros(1, n, words, dtype=torch.int32, device=DEV)
    prev = torch.zeros(n, 4, dtype=torch.int32, device=DEV)
    meta = torch.zeros(_lib.lib().cim_mask_meta_bytes(1, n, words), dtype=torch.uint8, device=DEV)
    bad = torch.zeros(1, dtype=torch.int32, device=DEV)
    st = _lib.stream_ptr(torch.device(DEV))
    mask_ops._unpack_rle_into(to_dev(full), packed, prev, meta, bad, 1, n, st)
    assert int(bad) == 0 and int(prev[:, 2].min()) > 0
    mask_ops._unpack_rle_into(to_dev(rle), packed, prev, meta, bad, 1, n, st)
    assert int(bad) == n_bad
    expect = masks.copy()
    for i in list(bad_strings) + [10]:
        expect[i] = 0
    want, want_meta = dense(canvas_of([expect], n, H, W))
    assert_same(packed, meta, want, want_meta)
    for i in list(bad_strings) + [10]:
        assert prev[i].tolist() == [0, 0, 0, 0]
    with pytest.raises(ValueError, match=f"{n_bad} malformed"):
        mask_ops.unpack_rle(to_dev(rle))


# ------------------------------------------------------------------------------------------------- 7. run_host
@pytest.mark.parametrize("depth", [1, 2])
def test_run_host_rle_wire_equals_the_crop_wire(depth):
    """alloc_host_io(ragged=True, compact=True) with native-size masks: the RLE wire and the crop wire give the same
    losses, valid flags, checksums and device mask buffers (masks, metadata, rectangles) step for step while the inputs
    change; a malformed string in one step raises when that step's results are collected."""
    n_img, R_cap, C, D, Cf, size = 3, 96, 20, 256, 32, 128
    probs = [host_problem(1, [96, 40, 71]), host_problem(2, [13, 96, 60]), host_problem(3, [80, 55, 96])]
    for p in probs:
        i = torch.from_numpy(real_rows(p["counts"], R_cap))
        p.update(c_rois=p["rois"][i].contiguous(), c_seg=p["seg_x"][i.to(DEV)].contiguous(),
                 c_go=p["grad_out"][i.to(DEV)].contiguous(), N=len(i),
                 rle=encode_host([m.numpy() for m in p["native"]], R_cap, size, size))
    feat = torch.randn(n_img, Cf, size // 16, size // 16, generator=torch.Generator().manual_seed(3)).to(DEV)
    torch.manual_seed(1)
    weight, bias = (t.detach().contiguous() for t in heads.cls_iou_model(D, C + 1, 3).to(DEV)._stacked())
    n_calls = 6
    fed = [probs[t % 3] for t in range(n_calls)]
    seen = [fed[max(0, t - depth)] for t in range(n_calls)]
    steps = {}
    for wire in ("crops", "rle"):
        step = CIMHeadStep(n_img, R_cap, C, Cf, size // 16, size // 16, 1.0 / 16, size * size // 32, feat_dim=D,
                           device=DEV, mask_kb_per_row=size // 16, head_grads=True)
        if wire == "crops":
            cap = max(int(p["crops"].words.numel()) for p in probs) + 64
            step.alloc_host_io(mask_hw=(size, size), crop_capacity_words=cap, prefetch_depth=depth, ragged=True,
                               compact=True)
        else:
            cap = max(int(p["rle"].chars.numel()) for p in probs) + 64
            step.alloc_host_io(rle_capacity_bytes=cap, prefetch_depth=depth, ragged=True, compact=True)
        steps[wire] = step
    got = {w: [] for w in steps}
    for wire, step in steps.items():
        np.random.seed(3)
        for t in range(n_calls):
            pr, sp = fed[t], seen[t]
            step.wait_inputs_consumed()
            step.hi_rois.zero_()
            step.hi_rois[:pr["N"]].copy_(pr["c_rois"])
            step.hi_labels.copy_(pr["labels"])
            step.hi_n_props.copy_(torch.tensor(pr["counts"], dtype=torch.int32))
            if wire == "crops":
                step.set_host_crops(pr["crops"])
            else:
                step.set_host_rle(pr["rle"])
            step.run_host(feat, sp["c_go"], sp["c_seg"], weight, bias)
            torch.cuda.synchronize()
            r = step.results_host
            got[wire].append((r["valid"], np.nan_to_num(r["losses"], nan=-7.0), r["checksum"],
                              [(b["masks"].clone(), b["meta"].clone(), b["prev_rects"].clone()) for b in step.di]))
    assert steps["rle"].results_host["bad_rle"] == 0
    assert steps["rle"].last_mask_h2d_bytes < steps["crops"].last_mask_h2d_bytes
    for t, (a, b) in enumerate(zip(got["crops"], got["rle"])):
        for x, y in zip(a[:3], b[:3]):
            np.testing.assert_array_equal(x, y, err_msg=f"call {t}")
        for (pa, ma, ra), (pb, mb, rb) in zip(a[3], b[3]):
            assert torch.equal(pa, pb) and torch.equal(ra, rb), f"call {t}: mask buffers differ"
            for x, y in zip(meta_parts(ma, n_img, R_cap, pa.shape[-1]), meta_parts(mb, n_img, R_cap, pb.shape[-1])):
                assert torch.equal(x, y), f"call {t}: metadata differs"
    assert not np.array_equal(got["rle"][0][1], got["rle"][1][1])         # the inputs do change

    # a malformed string fed at call t is decoded for step t + depth and raises at the end of that call
    step = steps["rle"]
    pr = probs[0]
    broken = mask_ops.MaskRLE(pr["rle"].chars.clone(), pr["rle"].off, pr["rle"].len, pr["rle"].hw, size, size)
    broken.chars[int(pr["rle"].off[5])] = ord("~")
    order = [broken] + [pr["rle"]] * depth
    for t, rle in enumerate(order):
        step.wait_inputs_consumed()
        step.hi_rois.zero_()
        step.hi_rois[:pr["N"]].copy_(pr["c_rois"])
        step.hi_n_props.copy_(torch.tensor(pr["counts"], dtype=torch.int32))
        step.set_host_rle(rle)
        rows = step.next_step_rows()
        src = next(p for p in probs if p["N"] == rows)
        if t < depth:
            step.run_host(feat, src["c_go"], src["c_seg"], weight, bias)
        else:
            with pytest.raises(ValueError, match="1 malformed RLE string"):
                step.run_host(feat, src["c_go"], src["c_seg"], weight, bias)
