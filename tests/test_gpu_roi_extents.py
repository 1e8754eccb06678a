"""Images of different sizes batched on one feature-map canvas: RoIAlign with per-image extents (feat_hw) on the tile,
window and generic paths against the oracle (oracle/roi_oracle.c) on each image's cropped map, the NULL case, MaskFuse,
CIMHeadStep.run with extents and proposal counts, and run_host with ragged proposal counts and crops of native-size
masks placed on a common canvas."""
import numpy as np
import pytest
import torch

import test_gpu_ragged as tr
from cim_b200 import _lib, heads, mask_ops, ops, synth
from cim_b200.step import CIMHeadStep
from oracle import roi_oracle
from test_gpu_roi import close
from test_roi_extents_cpu import extent_rois, per_image_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def per_image_grad(g, rois, hw, shape, scale, sr, aligned):
    """Backward of per_image_oracle, placed into a canvas-shaped gradient (0 outside the extents)."""
    out = np.zeros(shape, np.float64)
    for b in range(shape[0]):
        sel = np.nonzero(rois[:, 0] == b)[0]
        if len(sel):
            r = rois[sel].copy()
            r[:, 0] = 0
            gb = roi_oracle.roi_align_bwd(np.ascontiguousarray(g[sel]), r, (1, shape[1], int(hw[b, 0]), int(hw[b, 1])),
                                          scale, sr, aligned)
            out[b, :, :hw[b, 0], :hw[b, 1]] = gb[0]
    return out


def outside(a, hw):
    """The values of a [B, C, H, W] outside each image's extent, concatenated."""
    return torch.cat([torch.cat([a[b, :, h:, :].reshape(-1), a[b, :, :h, w:].reshape(-1)])
                      for b, (h, w) in enumerate(hw.tolist())])


def fill_outside(feat, hw, value):
    f = feat.clone()
    for b, (h, w) in enumerate(hw.tolist()):
        f[b, :, h:, :] = value
        f[b, :, :h, w:] = -value
    return f


def run_ops(feat, rois, scale, sr, aligned, hw, g, out_size=7):
    f = feat.to(DEV).requires_grad_(True)
    out = ops.roi_align(f, rois.to(DEV), out_size, scale, sr, "avg", aligned, feat_hw=hw)
    out.backward(g.to(DEV))
    return out.detach(), f.grad


# canvas (H, W), scale, extents, sort rois by image (tile / window paths need grouped rois)
PATHS = {
    "tile": ((32, 32), 1 / 16, [(32, 24), (24, 32), (17, 29), (32, 32), (9, 5)]),
    "window_vgg16": ((64, 64), 1 / 8, [(64, 48), (43, 64)]),
    "window_r50": ((75, 75), 1 / 16, [(75, 43), (43, 75), (60, 71), (75, 75)]),
}


def path_inputs(path, seed, K=40):
    (H, W), scale, ext = PATHS[path]
    hw = np.array(ext, np.int32)
    B, Cc = len(ext), 64
    rng = np.random.RandomState(seed)
    rois = extent_rois(rng, B, hw, scale, K)
    rois = rois[np.argsort(rois[:, 0], kind="stable")]
    feat = torch.randn(B, Cc, H, W, generator=torch.Generator().manual_seed(seed))
    return feat, torch.from_numpy(rois), hw, scale


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
def test_tile_and_window_paths_match_the_per_image_oracle(path, aligned, sr):
    feat, rois, hw, scale = path_inputs(path, 100 + 2 * sr + int(aligned))
    fn, rn = feat.numpy(), rois.numpy()
    want = per_image_oracle(fn, rn, hw, scale, sr, aligned)
    canvas = roi_oracle.roi_align_fwd(fn, rn, 7, 7, scale, sr, aligned)
    assert np.abs(canvas - want).max() > 1e-3 * np.abs(want).max(), "the inputs must discriminate"
    g = torch.randn(len(rois), feat.shape[1], 7, 7, generator=torch.Generator().manual_seed(7))
    out, grad = run_ops(feat, rois, scale, sr, aligned, hw, g)
    close(out.cpu().numpy(), want)
    want_g = per_image_grad(g.numpy(), rn, hw, tuple(feat.shape), scale, sr, aligned)
    close(grad.cpu().numpy(), want_g)
    assert not outside(grad, hw).any()                                   # exactly 0 outside the extents
    # large finite garbage outside the extents changes nothing.  The tile backward is bit-reproducible; the window
    # backward adds the partial gradients of overlapping windows with red.global.add, in no fixed order
    out2, grad2 = run_ops(fill_outside(feat, hw, 1e36), rois, scale, sr, aligned, hw, g)
    out0, grad0 = run_ops(fill_outside(feat, hw, 0.0), rois, scale, sr, aligned, hw, g)
    assert torch.equal(out, out2) and torch.equal(out, out0)
    for other in (grad2, grad0):
        assert not outside(other, hw).any()
        if path == "tile":
            assert torch.equal(grad, other)
        else:
            close(other.cpu().numpy(), grad.cpu().numpy(), elem=3e-5)


def generic_inputs(case, seed):
    """Generic kernels: unsorted rois (the tile kernel hands them over), a 14 x 14 output, extents narrower than a
    tap class."""
    H, W, scale = 32, 32, 1 / 16
    hw = np.array([(32, 5), (3, 32), (17, 2), (32, 32)], np.int32)
    rng = np.random.RandomState(seed)
    rois = extent_rois(rng, len(hw), hw, scale, 30)
    if case == "out14":
        rois = rois[np.argsort(rois[:, 0], kind="stable")]
    feat = torch.randn(len(hw), 32, H, W, generator=torch.Generator().manual_seed(seed))
    return feat, torch.from_numpy(rois), hw, scale, (14 if case == "out14" else 7)


@pytest.mark.parametrize("case", ["unsorted", "out14"])
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
def test_generic_path_matches_the_per_image_oracle(case, aligned, sr):
    feat, rois, hw, scale, o = generic_inputs(case, 200 + sr + int(aligned))
    fn, rn = feat.numpy(), rois.numpy()
    want = np.zeros((len(rn), feat.shape[1], o, o))
    want_c = roi_oracle.roi_align_fwd(fn, rn, o, o, scale, sr, aligned)
    g = torch.randn(len(rois), feat.shape[1], o, o, generator=torch.Generator().manual_seed(8))
    want_g = np.zeros(feat.shape)
    for b in range(len(hw)):
        sel = np.nonzero(rn[:, 0] == b)[0]
        r = rn[sel].copy()
        r[:, 0] = 0
        crop = np.ascontiguousarray(fn[b:b + 1, :, :hw[b, 0], :hw[b, 1]])
        want[sel] = roi_oracle.roi_align_fwd(crop, r, o, o, scale, sr, aligned)
        want_g[b, :, :hw[b, 0], :hw[b, 1]] = roi_oracle.roi_align_bwd(np.ascontiguousarray(g.numpy()[sel]), r,
                                                                       crop.shape, scale, sr, aligned)[0]
    assert np.abs(want_c - want).max() > 1e-3 * np.abs(want).max(), "the inputs must discriminate"
    out, grad = run_ops(feat, rois, scale, sr, aligned, hw, g, o)
    close(out.cpu().numpy(), want)
    close(grad.cpu().numpy(), want_g, elem=3e-5)        # fp32 atomicAdd sums in arbitrary order
    assert not outside(grad, hw).any()
    out2, _ = run_ops(fill_outside(feat, hw, 1e36), rois, scale, sr, aligned, hw, g, o)
    assert torch.equal(out, out2)


@pytest.mark.parametrize("path", sorted(PATHS) + ["generic"])
def test_full_extents_equal_no_extents_bitwise(path):
    """feat_hw = the canvas for every image (prepare_ex + the _prepared_ex calls) is bit for bit feat_hw = None (the
    self-preparing entry points), forward and backward.  On the generic path the backward adds with atomics, so its
    inputs there are exact in any order: integer roi corners in feature cells, 14 x 14 bins of one cell, one sample per
    bin, integer gradients.  The window backward adds overlapping windows in no fixed order (DESIGN.md section 4.9):
    there the two gradients agree to rounding."""
    if path == "generic":
        B, Cc, H, W, scale, sr, aligned, o = 3, 32, 32, 32, 1.0, 1, False, 14
        rng = np.random.RandomState(4)
        x1, y1 = rng.randint(-4, W - 8, 50), rng.randint(-4, H - 8, 50)
        rois = torch.from_numpy(np.stack([rng.randint(0, B, 50), x1, y1, x1 + 14, y1 + 14], 1).astype(np.float32))
        feat = torch.randn(B, Cc, H, W, generator=torch.Generator().manual_seed(4))
        g = torch.randint(-8, 9, (50, Cc, o, o), generator=torch.Generator().manual_seed(5)).float()
    else:
        feat, rois, _, scale = path_inputs(path, 300)
        B, _, H, W = feat.shape
        sr, aligned, o = 0, True, 7
        g = torch.randn(len(rois), feat.shape[1], 7, 7, generator=torch.Generator().manual_seed(9))
    full = np.array([[H, W]] * B, np.int32)
    out_n, grad_n = run_ops(feat, rois, scale, sr, aligned, None, g, o)
    for hw in (full, torch.from_numpy(full).to(DEV)):
        out_f, grad_f = run_ops(feat, rois, scale, sr, aligned, hw, g, o)
        assert torch.equal(out_n, out_f)
        if path.startswith("window"):
            close(grad_f.cpu().numpy(), grad_n.cpu().numpy(), elem=3e-5)
        else:
            assert torch.equal(grad_n, grad_f)


@pytest.mark.parametrize("path", ["tile", "window_vgg16"])
def test_maskfuse_with_extents(path):
    """MaskFuse with extents: the forward is the unfused RoIAlign with extents and its product with the mask, bit for
    bit; the backward is the unfused backward of grad[:, :C] + grad[:, C:] * mask, 0 outside the extents."""
    feat, rois, hw, scale = path_inputs(path, 400)
    K, Cc = len(rois), feat.shape[1]
    masks = (torch.rand(K, 7, 7, generator=torch.Generator().manual_seed(4)) > 0.5).float().to(DEV)
    f = feat.to(DEV).requires_grad_(True)
    r = rois.to(DEV)
    fused = ops.roi_align_maskfuse(f, r, masks, 7, scale, 0, True, feat_hw=hw)
    box = ops.roi_align(feat.to(DEV), r, 7, scale, 0, "avg", True, feat_hw=hw)
    assert torch.equal(fused[:, :Cc], box)
    assert torch.equal(fused[:, Cc:], box * masks[:, None])
    g = torch.randn(K, 2 * Cc, 7, 7, generator=torch.Generator().manual_seed(6)).to(DEV)
    fused.backward(g)
    _, grad_u = run_ops(feat, rois, scale, 0, True, hw, g[:, :Cc] + g[:, Cc:] * masks[:, None])
    close(f.grad.cpu().numpy(), grad_u.cpu().numpy())
    assert not outside(f.grad, hw).any()
    want = per_image_oracle(feat.numpy(), rois.numpy(), hw, scale, 0, True)
    close(box.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------- CIMHeadStep
def test_step_with_extents_and_counts():
    """run(feat_hw=..., n_props=...): each image's roi_out rows and grad_feat equal ops.roi_align on its cropped map;
    every other output is bit for bit that of the same run with feat_hw=None."""
    n_img, R, C, D = 3, 192, 20, 256
    n_props = [150, R, 97]
    pr = tr.step_inputs(n_props, R, C, D, 128, 32, 50)            # an 8 x 8 canvas at stride 16
    hw = np.array([(8, 6), (5, 8), (7, 7)], np.int32)
    w, b = (tr.cuda(a) for a in tr.head_params(D, C + 1, 3, 9))
    res = []
    for feat_hw in (None, hw):
        step = tr.make_step(pr, n_img, R, C, D)
        np.random.seed(3)
        for _ in range(2):
            step.run(pr["feat"], pr["rois"], pr["grad_out"], pr["packed"], pr["seg_x"], w, b, pr["labels"].to(DEV),
                     mat=pr["mat"], n_props=n_props, feat_hw=feat_hw)
        torch.cuda.synchronize()
        res.append((tr.step_outputs(step), step.roi_out.clone(), step.grad_feat.clone()))
    tr.assert_outputs_equal(res[0][0], res[1][0])
    roi_out, grad_feat = res[1][1], res[1][2]
    assert not torch.equal(res[0][1], roi_out), "the inputs must discriminate"
    for i, (h, wd) in enumerate(hw.tolist()):
        crop = pr["feat"][i:i + 1, :, :h, :wd].contiguous().requires_grad_(True)
        r = pr["rois"][i * R:(i + 1) * R].clone()
        r[:, 0] = 0
        out = ops.roi_align(crop, r, 7, 1.0 / 16, 0, "avg", True)
        out.backward(pr["grad_out"][i * R:(i + 1) * R])
        close(roi_out[i * R:(i + 1) * R].cpu().numpy(), out.detach().cpu().numpy())
        close(grad_feat[i, :, :h, :wd].cpu().numpy(), crop.grad[0].cpu().numpy())
    assert not outside(grad_feat, hw).any()


NATIVE = [(120, 96), (96, 128), (80, 128)]


def host_problem(seed, counts, R=96, C=20, D=256, Cf=32, size=128):
    """One ragged batch of images with native mask sizes NATIVE on a size x size canvas: counts, rois (padding rows
    repeat the image's first roi), labels, the per-image native masks, their crops and the canvas-padded packed
    masks run() takes."""
    n_img = len(counts)
    rois, native, labels = [], [], []
    canvas = torch.zeros(n_img, R, size, size, dtype=torch.uint8)
    for b, n in enumerate(counts):
        h, w = NATIVE[(b + seed) % len(NATIVE)]
        params = synth.proposal_params(n, size, seed * 10 + b)
        m = synth.rasterize(params)[:, :h, :w].contiguous()
        native.append(m)
        canvas[b, :n, :h, :w] = m
        r = synth.rois_from_params(params, b)
        r[:, 3].clamp_(max=w)
        r[:, 4].clamp_(max=h)
        rois.append(torch.cat([r, r[:1].expand(R - n, 5)]))
        labels.append(synth.image_labels(C, 2, seed * 10 + b))
    crops = mask_ops.batch_crops_host([mask_ops.pack_crops_host(m.numpy()) for m in native], R, size, size)
    gen = torch.Generator().manual_seed(seed)
    grad_out = torch.randn(n_img * R, Cf, 7, 7, generator=gen)
    for b, n in enumerate(counts):
        grad_out[b * R + n:(b + 1) * R] = 0
    return dict(counts=list(counts), rois=torch.cat(rois), labels=torch.cat(labels), native=native, crops=crops,
                packed=mask_ops.mask_pack(canvas.to(DEV)), grad_out=grad_out.to(DEV),
                seg_x=(torch.randn(n_img * R, D, generator=gen) * 3).to(DEV))


@pytest.mark.parametrize("depth", [1, 2])
def test_run_host_ragged_with_native_size_crops(depth):
    """run_host with alloc_host_io(ragged=True): counts, rois, labels and native-size masks (120 x 96, 96 x 128,
    80 x 128 on a 128 x 128 canvas) change from call to call.  Each call equals run() on device inputs with the same
    counts; the unpacked buffer equals the dense packing of the canvas-padded masks; each image's maps equal
    mask_overlap of its native masks alone, bit for bit."""
    n_img, R, C, D, Cf, size = 3, 96, 20, 256, 32, 128
    probs = [host_problem(1, [96, 40, 71]), host_problem(2, [13, 96, 60]), host_problem(3, [80, 55, 96])]
    kb = size // 16
    feat = torch.randn(n_img, Cf, size // 16, size // 16, generator=torch.Generator().manual_seed(3)).to(DEV)
    torch.manual_seed(1)
    model = heads.cls_iou_model(D, C + 1, 3).to(DEV)
    weight, bias = (t.detach().contiguous() for t in model._stacked())
    mk = lambda: CIMHeadStep(n_img, R, C, Cf, size // 16, size // 16, 1.0 / 16, size * size // 32, feat_dim=D,
                             device=DEV, mask_kb_per_row=kb, head_grads=True)
    n_calls = 6
    fed = [probs[t % 3] for t in range(n_calls)]
    seen = [fed[max(0, t - depth)] for t in range(n_calls)]
    ref = mk()
    want = []
    np.random.seed(3)
    for pr in seen:
        ref.run(feat, pr["rois"].to(DEV), pr["grad_out"], pr["packed"], pr["seg_x"], weight, bias,
                pr["labels"].to(DEV), n_props=pr["counts"])
        torch.cuda.synchronize()
        want.append((ref.losses.cpu().numpy().copy(), ref.valid.cpu().numpy().copy(), ref.iou.clone()))
    assert not np.array_equal(np.nan_to_num(want[0][0]), np.nan_to_num(want[3][0]))

    step = mk()
    cap = max(int(p["crops"].words.numel()) for p in probs) + 64
    step.alloc_host_io(mask_hw=(size, size), crop_capacity_words=cap, prefetch_depth=depth, ragged=True)
    assert step.hi_n_props.tolist() == [R] * n_img
    np.random.seed(3)
    for t in range(n_calls):
        pr, sp = fed[t], seen[t]
        step.wait_inputs_consumed()
        step.hi_rois.copy_(pr["rois"])
        step.hi_labels.copy_(pr["labels"])
        step.hi_n_props.copy_(torch.tensor(pr["counts"], dtype=torch.int32))
        step.set_host_crops(pr["crops"])
        step.run_host(feat, sp["grad_out"], sp["seg_x"], weight, bias)
        got = step.results_host
        w_loss, w_valid, w_iou = want[t]
        np.testing.assert_array_equal(got["valid"], w_valid)
        np.testing.assert_array_equal(np.nan_to_num(got["losses"], nan=-7.0), np.nan_to_num(w_loss, nan=-7.0))
        assert torch.equal(step.iou.view(torch.int16), w_iou.view(torch.int16))
        torch.cuda.synchronize()
        used = step.di[step._slot ^ 1]                                     # the buffer this call's step read
        assert torch.equal(used["masks"], sp["packed"])
        for b, n in enumerate(sp["counts"]):
            iou, asy = mask_ops.mask_overlap(mask_ops.mask_pack(sp["native"][b].to(DEV)))
            assert torch.equal(step.iou[b, :n, :n].view(torch.int16), iou.view(torch.int16))
            assert torch.equal(step.asy[b, :n, :n].view(torch.int16), asy.view(torch.int16))


def test_bad_feat_hw_and_host_counts_raise():
    feat = torch.randn(2, 32, 16, 16, device=DEV)
    rois = torch.tensor([[0, 0, 0, 100, 100], [1, 10, 10, 200, 120]], dtype=torch.float32, device=DEV)
    good = torch.tensor([[16, 12], [9, 16]], dtype=torch.int32, device=DEV)
    ops.roi_align(feat, rois, 7, 1 / 16, 0, "avg", True, feat_hw=good)
    bad = [([[16, 12]], ValueError), (good[:1], ValueError), (good.reshape(4), ValueError),
           (good.float(), TypeError), (good.long(), TypeError), ([[16.0, 12.0], [9.0, 16.0]], TypeError),
           ([[0, 12], [9, 16]], ValueError), ([[16, 12], [9, 17]], ValueError), ([[17, 12], [9, 16]], ValueError),
           (torch.empty((2, 2), dtype=torch.int32, device="meta"), ValueError)]
    for hw, exc in bad:
        with pytest.raises(exc):
            ops.roi_align(feat, rois, 7, 1 / 16, 0, "avg", True, feat_hw=hw)
        with pytest.raises(exc):
            ops.RoIAlign(7, 1 / 16)(feat, rois, feat_hw=hw)
        with pytest.raises(exc):
            ops.roi_align_maskfuse(feat, rois, torch.ones(2, 7, 7, device=DEV), 7, 1 / 16, feat_hw=hw)
    step = CIMHeadStep(2, 8, 20, 32, 16, 16, 1 / 16, 64, feat_dim=256, device=DEV, head_grads=True)
    with pytest.raises(ValueError):
        step.run(feat, rois.repeat(8, 1), None, None, None, None, None, None, feat_hw=[[16, 12], [9, 17]])
    step.alloc_host_io(ragged=True)
    for counts in ([0, 8], [8, 9]):
        step.hi_n_props.copy_(torch.tensor(counts, dtype=torch.int32))
        with pytest.raises(ValueError):
            step.stage_host_inputs()
