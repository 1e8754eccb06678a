"""RoIAlign / RoIPool CUDA kernels (through the mmcv-style operator surface and the C ABI) against
the oracle (oracle/roi_oracle.c), torchvision, and the reference's own vendored kernels
(oracle/_ref, aligned=False).  Tolerance from BASELINE.json: 1e-5 relative in fp32."""
import numpy as np
import pytest
import torch
from torchvision.ops import roi_align as tv_roi_align

from cim_b200 import _lib, ops, synth
from oracle import roi_oracle
from conftest import assert_close_elementwise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def close(got, want, rel=1e-5, elem=None):
    """max-norm bound AND element by element: |err| <= rel |want| + elem * rms(want), elem = rel unless given."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = max(np.abs(want).max(), 1e-30)
    err = np.abs(got - want).max() / scale
    assert err <= rel, f"max err / max|ref| = {err:.3e}"
    assert_close_elementwise(got, want, rtol=rel, atol_rms=rel if elem is None else elem)


def random_rois(seed, B, K, H, W, scale, wild=False, sort=True):
    g = torch.Generator().manual_seed(seed)
    b = torch.randint(0, B, (K,), generator=g).float()
    if sort:
        b = b.sort().values
    sw, sh = W / scale, H / scale
    x1 = torch.rand(K, generator=g) * sw * 0.8
    y1 = torch.rand(K, generator=g) * sh * 0.8
    w = torch.rand(K, generator=g) * sw * 0.6 + 0.5
    h = torch.rand(K, generator=g) * sh * 0.6 + 0.5
    if wild:
        x1 -= sw * 0.3
        y1 -= sh * 0.3
        w[::7] = 0.01
        h[::5] = 0.0
        w[3::11] = sw * 3           # far wider than the map: > 8 taps per bin -> generic path
    return torch.stack([b, x1, y1, x1 + w, y1 + h], 1)


def run_both(feat, rois, scale, sr, aligned, out_size=7):
    f = feat.to(DEV).requires_grad_(True)
    r = rois.to(DEV)
    out = ops.roi_align(f, r, out_size, scale, sr, "avg", aligned)
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(77))
    out.backward(g.to(DEV))
    oh, ow = (out_size, out_size) if isinstance(out_size, int) else out_size
    want = roi_oracle.roi_align_fwd(feat.numpy(), rois.numpy(), oh, ow, scale, sr, aligned)
    want_g = roi_oracle.roi_align_bwd(g.numpy(), rois.numpy(), feat.shape, scale, sr, aligned)
    return out.detach().cpu().numpy(), f.grad.cpu().numpy(), want, want_g


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
@pytest.mark.parametrize("wild", [False, True])
def test_tile_path_small(aligned, sr, wild):
    feat = torch.randn(3, 64, 16, 20, generator=torch.Generator().manual_seed(1))
    rois = random_rois(2, 3, 90, 16, 20, 0.25, wild)
    out, gf, want, want_g = run_both(feat, rois, 0.25, sr, aligned)
    close(out, want)
    close(gf, want_g)


def test_cfg1_resnet50_shape_against_oracle_and_torchvision():
    """BASELINE.json configs[0]: R-50 VOC, one 512x512 image, 300 mask proposals."""
    C, H, W, scale = synth.feature_shape("resnet50")
    feat = torch.randn(1, C, H, W, generator=torch.Generator().manual_seed(1234))
    rois = synth.rois_from_params(synth.proposal_params(300, 512, 1234))
    out, gf, want, want_g = run_both(feat, rois, scale, 0, True)
    close(out, want)
    close(gf, want_g)
    tv = tv_roi_align(feat, rois, (7, 7), scale, 0, True).numpy()
    close(out, tv)


@pytest.mark.parametrize("case", ["unsorted", "odd_channels", "out14", "out3x5", "big_map", "empty_image"])
def test_generic_and_mixed_paths(case):
    B, C, H, W, K, size, sort = 2, 32, 12, 12, 50, 7, True
    if case == "unsorted":
        sort = False
    elif case == "odd_channels":
        C = 5
    elif case == "out14":
        size = 14
    elif case == "out3x5":
        size = (3, 5)
    elif case == "big_map":
        H, W, C = 100, 120, 32          # 32 x 12000 floats do not fit in shared memory
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(5))
    rois = random_rois(6, B, K, H, W, 0.5, wild=True, sort=sort)
    if case == "empty_image":
        rois[:, 0] = 1                   # image 0 has no ROI at all; its gradient slab must be zero
    out, gf, want, want_g = run_both(feat, rois, 0.5, 0, True, size)
    close(out, want)
    close(gf, want_g)


def test_no_rois():
    feat = torch.randn(1, 32, 8, 8, device=DEV, requires_grad=True)
    out = ops.RoIAlign(7, 0.5, 0)(feat, torch.zeros(0, 5, device=DEV))
    assert out.shape == (0, 32, 7, 7)
    out.sum().backward()
    assert feat.grad.abs().sum().item() == 0


def test_against_reference_vendored_kernels_aligned_false():
    """oracle/_ref = lib/modeling/roi_xfrom/roi_align/src/roi_align_kernel.cu compiled as is."""
    if roi_oracle.ref_lib() is None:
        pytest.skip("oracle/_ref was not built")
    B, C, H, W, scale = 2, 256, 32, 32, 1.0 / 16
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(3)).to(DEV)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(500, 512, 40 + b), b) for b in range(B)]).to(DEV)
    mine = ops.roi_align(feat, rois, 7, scale, 0, "avg", False)
    ref = roi_oracle.ref_roi_align_fwd(feat, rois, 7, 7, scale, 0)
    # element-wise 3e-5 * rms here: `ref` is itself an fp32 kernel (sample-by-sample sums of up to 4 x 100 products,
    # FMA-contracted), not the float64-accumulating oracle the other tests compare with at 1e-5
    close(mine.cpu().numpy(), ref.cpu().numpy(), elem=3e-5)
    g = torch.randn_like(mine)
    f2 = feat.clone().requires_grad_(True)
    ops.roi_align(f2, rois, 7, scale, 0, "avg", False).backward(g)
    ref_g = roi_oracle.ref_roi_align_bwd(g, rois, feat.shape, scale, 0)
    close(f2.grad.cpu().numpy(), ref_g.cpu().numpy(), elem=3e-5)      # fp32 atomicAdd sums in arbitrary order


def test_aligned_false_against_torchvision_cuda():
    """The inputs and tolerance of the test above against torchvision's CUDA roi_align(aligned=False), which implements
    the same Caffe2-derived arithmetic as the vendored kernel (tests/test_oracle_roi.py pins the C restatement to both)
    and, unlike oracle/_ref, is available wherever the package is."""
    B, C, H, W, scale = 2, 256, 32, 32, 1.0 / 16
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(3)).to(DEV)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(500, 512, 40 + b), b) for b in range(B)]).to(DEV)
    mine = ops.roi_align(feat, rois, 7, scale, 0, "avg", False)
    close(mine.cpu().numpy(), tv_roi_align(feat, rois, (7, 7), scale, 0, False).cpu().numpy(), elem=3e-5)
    g = torch.randn(mine.shape, generator=torch.Generator().manual_seed(4)).to(DEV)
    f1, f2 = feat.clone().requires_grad_(True), feat.clone().requires_grad_(True)
    ops.roi_align(f1, rois, 7, scale, 0, "avg", False).backward(g)
    tv_roi_align(f2, rois, (7, 7), scale, 0, False).backward(g)
    close(f1.grad.cpu().numpy(), f2.grad.cpu().numpy(), elem=3e-5)    # torchvision adds with atomics, in any order


def test_backward_is_bit_reproducible():
    C, H, W, scale = 64, 32, 32, 1.0 / 16
    rois = synth.rois_from_params(synth.proposal_params(400, 512, 7)).to(DEV)
    g = torch.randn(400, C, 7, 7, device=DEV)
    outs = []
    for _ in range(3):
        f = torch.zeros(1, C, H, W, device=DEV, requires_grad=True)
        ops.roi_align(f, rois, 7, scale).backward(g)
        outs.append(f.grad.clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_full_size_cfg2_linearity_and_adjoint():
    """BASELINE.json configs[1] (8 images x 2000 proposals, R-50): size-independent properties.
    RoIAlign is linear in the features and its backward is the adjoint: <A f, g> == <f, A^T g>."""
    C, H, W, scale = synth.feature_shape("resnet50")
    B, R = 8, 2000
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(R, 512, 1234 + b), b) for b in range(B)]).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(0)
    f1 = torch.randn(B, C, H, W, device=DEV, generator=gen)
    f2 = torch.randn(B, C, H, W, device=DEV, generator=gen)
    o1 = ops.roi_align(f1, rois, 7, scale)
    o2 = ops.roi_align(f2, rois, 7, scale)
    o12 = ops.roi_align(2.5 * f1 + f2, rois, 7, scale)
    lin = (o12 - (2.5 * o1 + o2)).abs().max().item() / o12.abs().max().item()
    assert lin < 1e-5, lin
    del o2, o12
    g = torch.randn(o1.shape, device=DEV, generator=gen)
    f = f1.clone().requires_grad_(True)
    ops.roi_align(f, rois, 7, scale).backward(g)
    # the persistent backward splits tiles between two CTAs here: still bit-reproducible
    f_again = f1.clone().requires_grad_(True)
    ops.roi_align(f_again, rois, 7, scale).backward(g)
    assert torch.equal(f.grad, f_again.grad)
    del f_again
    lhs = (o1.double() * g.double()).sum().item()
    rhs = (f1.double() * f.grad.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * max(abs(lhs), abs(rhs), (o1.double().abs() * g.double().abs()).sum().item())
    # spot-check 64 random ROIs of the full run against the oracle
    idx = torch.randperm(B * R, generator=torch.Generator().manual_seed(1))[:64].sort().values
    want = roi_oracle.roi_align_fwd(f1.cpu().numpy(), rois[idx.to(DEV)].cpu().numpy(), 7, 7, scale, 0, True)
    close(o1[idx.to(DEV)].cpu().numpy(), want)


@pytest.mark.parametrize("variant", ["mmcv", "legacy"])
def test_roi_pool_exact_and_backward(variant):
    """Both bin conventions: mmcv 1.x's (the default: it is what the reference imports) and the vendored kernel's."""
    feat = torch.randn(2, 48, 20, 24, generator=torch.Generator().manual_seed(8))
    rois = random_rois(9, 2, 70, 20, 24, 0.25, wild=True)
    rois[5, 3] = rois[5, 1] - 2.0                                             # x2 + 1 < x1: mmcv pools nothing
    f = feat.to(DEV).requires_grad_(True)
    assert ops.RoIPool(7, 0.25).variant == "mmcv"
    out = ops.RoIPool(7, 0.25, variant)(f, rois.to(DEV))
    want, arg = roi_oracle.roi_pool_fwd(feat.numpy(), rois.numpy(), 7, 7, 0.25, variant)
    np.testing.assert_array_equal(out.detach().cpu().numpy(), want)          # max is exact
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(4))
    out.backward(g.to(DEV))
    close(f.grad.cpu().numpy(), roi_oracle.roi_pool_bwd(g.numpy(), arg, rois.numpy(), feat.shape))
    if variant == "legacy" and roi_oracle.ref_lib() is not None:              # the vendored kernel itself
        ref_out, _ = roi_oracle.ref_roi_pool_fwd(feat.to(DEV), rois.to(DEV), 7, 7, 0.25)
        np.testing.assert_array_equal(out.detach().cpu().numpy(), ref_out.cpu().numpy())


def _pool_raw(feat, rois, scale, variant, g=None):
    """cim_roi_pool_fwd_ex (+ cim_roi_pool_bwd) through the C ABI: pooled values, int32 argmax, grad_feat."""
    L, P = _lib.lib(), _lib.ptr
    B, C, H, W = feat.shape
    K = rois.shape[0]
    out = torch.empty(K, C, 7, 7, device=DEV)
    arg = torch.empty(K, C, 7, 7, dtype=torch.int32, device=DEV)
    st = _lib.stream_ptr(feat.device)
    _lib.check(L.cim_roi_pool_fwd_ex(P(feat), P(rois), P(out), P(arg), B, C, H, W, K, 7, 7, scale,
                                     ops.ROI_POOL_VARIANTS[variant], st), "pool fwd")
    gf = None
    if g is not None:
        gf = torch.full((B, C, H, W), float("nan"), device=DEV)       # the op must write every element
        _lib.check(L.cim_roi_pool_bwd(P(g), P(arg), P(rois), P(gf), B, C, H, W, K, 7, 7, st), "pool bwd")
    torch.cuda.synchronize()
    return out, arg, gf


@pytest.mark.parametrize("variant", ["mmcv", "legacy"])
@pytest.mark.parametrize("shape", [(3, 64, 20, 24, 300), (2, 48, 15, 17, 200), (2, 24, 40, 40, 150),
                                   (9, 32, 8, 8, 40), (1, 64, 12, 12, 9000)])
def test_roi_pool_tile_kernels_equal_simple_kernels(variant, shape):
    """The shared-memory tile kernels (32 / 16 / 8 channels per tile, odd map sizes, rois NOT grouped by image, an
    out-of-range batch index, more ROIs than one compaction round) against the thread-per-output kernels: pooled
    values and argmax bit for bit, gradients to fp32 summation order; and both against the oracle."""
    B, C, H, W, K = shape
    scale = 0.25
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(21))
    feat[:, :, 3, 4] = feat[:, :, 3, 5]                                      # ties: the first maximum must win
    rois = random_rois(31, B, K, H, W, scale, wild=True, sort=False)
    rois[7, 0] = B + 3                                                       # invalid image: pools nothing
    if K > 20:
        rois[11, 0] = -1
    f, r = feat.to(DEV), rois.to(DEV)
    g = torch.randn(K, C, 7, 7, generator=torch.Generator().manual_seed(5)).to(DEV)
    out_t, arg_t, gf_t = _pool_raw(f, r, scale, variant, g)
    with _lib.debug_flags(_lib.DBG_ROI_POOL_SIMPLE):
        out_s, arg_s, gf_s = _pool_raw(f, r, scale, variant, g)
    assert torch.equal(out_t, out_s) and torch.equal(arg_t, arg_s)
    close(gf_t.cpu().numpy(), gf_s.cpu().numpy(), rel=1e-5)
    bad = (rois[:, 0] < 0) | (rois[:, 0] >= B)
    assert (out_t[bad.to(DEV)] == 0).all() and (arg_t[bad.to(DEV)] == -1).all()
    sel = torch.nonzero(~bad).flatten()[:400]                                # the oracle does not guard the image index
    want, arg = roi_oracle.roi_pool_fwd(feat.numpy(), rois[sel].numpy(), 7, 7, scale, variant)
    np.testing.assert_array_equal(out_t[sel.to(DEV)].cpu().numpy(), want)
    np.testing.assert_array_equal(arg_t[sel.to(DEV)].cpu().numpy(), arg)


def test_roi_pool_tile_kernels_benchmarked_shape():
    """cfg2's shape (8 x 2000 proposals, 1024 x 32 x 32 map): tile kernels == simple kernels == the exact sum over the
    full output, bit for bit; oracle on sampled ROIs."""
    B, R = 8, 2000
    C, H, W, scale = synth.feature_shape("resnet50")
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(R, 512, 77 + b), b) for b in range(B)]).to(DEV)
    feat = torch.randn(B, C, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    # Both backward kernels add in an unspecified (atomic) order, and here a feature element collects hundreds of terms,
    # so fp32 sums of arbitrary values differ in their last bits from run to run.  Multiples of 1/64 in [-1, 1] sum
    # exactly in any order: at most 49 x R terms reach an element, so every partial sum is a multiple of 2^-6 below
    # 2^17, which the 24-bit fp32 significand holds.
    g = torch.randint(-64, 65, (B * R, C, 7, 7), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4),
                      dtype=torch.float32) / 64
    out_t, arg_t, gf_t = _pool_raw(feat, rois, scale, "mmcv", g)
    with _lib.debug_flags(_lib.DBG_ROI_POOL_SIMPLE):
        out_s, arg_s, gf_s = _pool_raw(feat, rois, scale, "mmcv", g)
    assert torch.equal(out_t, out_s) and torch.equal(arg_t, arg_s)
    del out_s, arg_s
    exact = torch.zeros(B, C, H * W, dtype=torch.float64, device=DEV)
    for b in range(B):
        rows = slice(b * R, (b + 1) * R)                                     # the ROIs of image b
        a = arg_t[rows].transpose(0, 1).reshape(C, -1).long()
        v = g[rows].transpose(0, 1).reshape(C, -1).double()
        exact[b].scatter_add_(1, a.clamp(min=0), torch.where(a >= 0, v, 0.0))
    del g, a, v
    exact = exact.view(B, C, H, W).float()
    assert torch.equal(gf_t, exact) and torch.equal(gf_s, exact)
    idx = torch.randperm(B * R, generator=torch.Generator().manual_seed(1))[:48].sort().values.to(DEV)
    want, arg = roi_oracle.roi_pool_fwd(feat.cpu().numpy(), rois[idx].cpu().numpy(), 7, 7, scale, "mmcv")
    np.testing.assert_array_equal(out_t[idx].cpu().numpy(), want)
    np.testing.assert_array_equal(arg_t[idx].cpu().numpy(), arg)


def test_errors_are_raised_not_printed():
    f = torch.zeros(1, 32, 8, 8, device=DEV)
    with pytest.raises(ValueError):
        ops.roi_align(f, torch.zeros(4, 4, device=DEV), 7)           # rois.size(1) != 5
    with pytest.raises(TypeError):
        ops.roi_align(f.half(), torch.zeros(4, 5, device=DEV), 7)
    with pytest.raises(NotImplementedError):
        ops.roi_align(f, torch.zeros(4, 5, device=DEV), 7, 1.0, 0, "max")


# ------------------------------------------------------------------ fused MaskFuse prologue (SURVEY 8f-1)
def maskfuse_oracle(feat, rois, masks, scale, sr, aligned, g, out_size=(7, 7)):
    """lib/modeling/resnet50.py:121-134 on top of the RoIAlign oracle: box_x, mask_x = box_x * masks,
    concat((box_x, mask_x), 1); backward: d box_x = g[:, :C] + g[:, C:] * masks."""
    oh, ow = out_size
    C = feat.shape[1]
    box = roi_oracle.roi_align_fwd(feat.numpy(), rois.numpy(), oh, ow, scale, sr, aligned)
    m = masks.numpy()[:, None]
    want = np.concatenate([box, box * m], 1)
    g_box = np.ascontiguousarray(g[:, :C] + g[:, C:] * m)
    want_g = roi_oracle.roi_align_bwd(g_box, rois.numpy(), feat.shape, scale, sr, aligned)
    return want, want_g


def run_maskfuse(feat, rois, masks, scale, sr, aligned, out_size=7):
    f = feat.to(DEV).requires_grad_(True)
    out = ops.roi_align_maskfuse(f, rois.to(DEV), masks.to(DEV), out_size, scale, sr, aligned)
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(78))
    out.backward(g.to(DEV))
    return out.detach().cpu().numpy(), f.grad.cpu().numpy(), g.numpy()


@pytest.mark.parametrize("wild", [False, True])
@pytest.mark.parametrize("aligned", [True, False])
def test_maskfuse_tile_path(aligned, wild):
    feat = torch.randn(3, 64, 16, 20, generator=torch.Generator().manual_seed(1))
    rois = random_rois(2, 3, 91, 16, 20, 0.25, wild)          # odd count: a ring slot with one ROI
    masks = (torch.rand(91, 7, 7, generator=torch.Generator().manual_seed(3)) > 0.4).float()
    out, gf, g = run_maskfuse(feat, rois, masks, 0.25, 0, aligned)
    want, want_g = maskfuse_oracle(feat, rois, masks, 0.25, 0, aligned, g)
    close(out, want)
    close(gf, want_g)


def test_maskfuse_equals_unfused_ops_bitwise_forward():
    """The fused output is the unfused RoIAlign output and its product with the mask, bit for bit."""
    C, H, W, scale = synth.feature_shape("resnet50")
    feat = torch.randn(1, C, H, W, generator=torch.Generator().manual_seed(12)).to(DEV)
    rois = synth.rois_from_params(synth.proposal_params(300, 512, 12)).to(DEV)
    masks = (torch.rand(300, 7, 7, generator=torch.Generator().manual_seed(4)) > 0.5).float().to(DEV)
    fused = ops.roi_align_maskfuse(feat, rois, masks, 7, scale, 0, True)
    box = ops.roi_align(feat, rois, 7, scale, 0, "avg", True)
    assert torch.equal(fused[:, :C], box)
    assert torch.equal(fused[:, C:], box * masks[:, None])


@pytest.mark.parametrize("case", ["unsorted", "odd_channels", "out3x5", "big_map"])
def test_maskfuse_generic_paths(case):
    B, C, H, W, K, size, sort = 2, 32, 12, 12, 50, 7, True
    if case == "unsorted":
        sort = False
    elif case == "odd_channels":
        C = 5
    elif case == "out3x5":
        size = (3, 5)
    elif case == "big_map":
        H, W = 100, 120
    oh, ow = (size, size) if isinstance(size, int) else size
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(5))
    rois = random_rois(6, B, K, H, W, 0.5, wild=True, sort=sort)
    masks = torch.rand(K, oh, ow, generator=torch.Generator().manual_seed(6))          # soft masks work too
    out, gf, g = run_maskfuse(feat, rois, masks, 0.5, 0, True, size)
    want, want_g = maskfuse_oracle(feat, rois, masks, 0.5, 0, True, g, (oh, ow))
    close(out, want)
    close(gf, want_g)


def test_maskfuse_full_size_adjoint():
    """cfg2-sized (2000 proposals, R-50 features): <fused(f), g> == <f, fused_bwd(g)> (the pair is an adjoint
    pair, a size-independent property), and the backward is bit-reproducible."""
    C, H, W, scale = synth.feature_shape("resnet50")
    K = 2000
    gen = torch.Generator(device=DEV).manual_seed(9)
    feat = torch.randn(1, C, H, W, device=DEV, generator=gen, requires_grad=True)
    rois = synth.rois_from_params(synth.proposal_params(K, 512, 9)).to(DEV)
    masks = (torch.rand(K, 7, 7, device=DEV, generator=gen) > 0.5).float()
    out = ops.roi_align_maskfuse(feat, rois, masks, 7, scale, 0, True)
    g = torch.randn(out.shape, device=DEV, generator=gen)
    (gf,) = torch.autograd.grad(out, feat, g, retain_graph=True)
    (gf2,) = torch.autograd.grad(out, feat, g)
    assert torch.equal(gf, gf2)
    lhs = (out.double() * g.double()).sum().item()
    rhs = (feat.detach().double() * gf.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * max(abs(lhs), 1.0)


# ------------------------------------------------------------------ large maps: channel-last global path
@pytest.mark.parametrize("fused", [False, True])
def test_vgg16_sized_map_uses_the_global_path_and_matches_oracle(fused):
    """BASELINE.json configs[2]: VGG-16, stride 8 -> a 64 x 64 map that does not fit the shared-memory tile.
    With the _ex workspace the sweep runs over a channel-last copy in global memory."""
    C, H, W, scale = 64, 64, 64, 1.0 / 8
    feat = torch.randn(2, C, H, W, generator=torch.Generator().manual_seed(21))
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(150, 512, 21 + b), b) for b in range(2)])
    if fused:
        masks = (torch.rand(300, 7, 7, generator=torch.Generator().manual_seed(22)) > 0.5).float()
        out, gf, g = run_maskfuse(feat, rois, masks, scale, 0, True)
        want, want_g = maskfuse_oracle(feat, rois, masks, scale, 0, True, g)
    else:
        out, gf, want, want_g = run_both(feat, rois, scale, 0, True)
    close(out, want)
    close(gf, want_g)


@pytest.mark.parametrize("fused", [False, True])
def test_vgg16_sized_map_wide_bins_stay_on_the_sweep_kernels(fused):
    """ROIs spanning most of a 64 x 64 map: 9 .. 12 collapsed taps per bin and axis.  The global-path kernels
    read WIDE descriptors (12 taps, T = 12 instance), so these no longer drop to the sample-by-sample kernel; a
    few ROIs larger than the map (> 12 taps) still do.  Same results either way."""
    C, H, W, scale = 64, 64, 64, 1.0 / 8
    feat = torch.randn(2, C, H, W, generator=torch.Generator().manual_seed(31))
    g = torch.Generator().manual_seed(32)
    K = 48
    b = torch.randint(0, 2, (K,), generator=g).float().sort().values
    w = 8 * (56 + 27 * torch.rand(K, generator=g))          # 56 .. 83 feature columns -> bins of 8 .. 11.9
    h = 8 * (40 + 43 * torch.rand(K, generator=g))
    x1 = (512 - w).clamp(min=-60) * torch.rand(K, generator=g)
    y1 = (512 - h).clamp(min=-60) * torch.rand(K, generator=g)
    w[5], h[7] = 8 * 120.0, 8 * 100.0                        # > 12 taps: generic leftover pass
    rois = torch.stack([b, x1, y1, x1 + w, y1 + h], 1)
    if fused:
        masks = (torch.rand(K, 7, 7, generator=torch.Generator().manual_seed(33)) > 0.5).float()
        out, gf, gg = run_maskfuse(feat, rois, masks, scale, 0, True)
        want, want_g = maskfuse_oracle(feat, rois, masks, scale, 0, True, gg)
    else:
        out, gf, want, want_g = run_both(feat, rois, scale, 0, True)
    close(out, want)
    close(gf, want_g)


def test_large_map_small_workspace_falls_back_to_generic():
    """The plain cim_roi_align_workspace_bytes(K) workspace is still accepted: the generic kernels run."""
    import ctypes as C_
    from cim_b200 import _lib
    L = _lib.lib()
    B, C, H, W, K, scale = 1, 32, 64, 64, 40, 1.0 / 8
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(23))
    rois = synth.rois_from_params(synth.proposal_params(K, 512, 23))
    f, r = feat.to(DEV), rois.to(DEV)
    assert L.cim_roi_align_workspace_bytes_ex(B, C, H, W, K, 7, 7) > L.cim_roi_align_workspace_bytes(K)
    assert L.cim_roi_align_workspace_bytes_ex(B, 1024, 32, 32, K, 7, 7) == L.cim_roi_align_workspace_bytes(K)
    ws = torch.empty(L.cim_roi_align_workspace_bytes(K), dtype=torch.uint8, device=DEV)
    out = torch.empty(K, C, 7, 7, device=DEV)
    _lib.check(L.cim_roi_align_fwd(_lib.ptr(f), _lib.ptr(r), _lib.ptr(out), B, C, H, W, K, 7, 7, scale, 0, 1,
                                   _lib.ptr(ws), ws.numel(), _lib.stream_ptr(torch.device(DEV))), "fwd")
    close(out.cpu().numpy(), roi_oracle.roi_align_fwd(feat.numpy(), rois.numpy(), 7, 7, scale, 0, True))


@pytest.mark.parametrize("shape", [(2, 64, 32, 32, 1.0 / 16), (1, 32, 64, 64, 1.0 / 8)])
@pytest.mark.parametrize("fused", [False, True])
def test_prepared_entry_points_equal_the_self_preparing_ones(shape, fused):
    """cim_roi_align_prepare once + the _prepared forward / backward (what CIMHeadStep and the autograd backward use)
    give bit-identical results to the calls that build their descriptors themselves -- tile path and global path."""
    from cim_b200 import _lib
    L = _lib.lib()
    B, C, H, W, scale = shape
    K = 60 * B
    dev = torch.device(DEV)
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(41)).to(dev)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(60, 512, 41 + b), b) for b in range(B)]).to(dev)
    masks = (torch.rand(K, 7, 7, generator=torch.Generator().manual_seed(42)) > 0.5).float().to(dev)
    Co = 2 * C if fused else C
    gout = torch.randn(K, Co, 7, 7, generator=torch.Generator().manual_seed(43)).to(dev)
    mk = masks if fused else None
    P, st = _lib.ptr, _lib.stream_ptr(dev)
    nbytes = L.cim_roi_align_workspace_bytes_ex(B, C, H, W, K, 7, 7)
    geo = (B, C, H, W, K, 7, 7, scale, 0, 1)

    def run(prepared):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty(K, Co, 7, 7, device=dev)
        gf = torch.empty(B, C, H, W, device=dev)
        if prepared:
            _lib.check(L.cim_roi_align_prepare(P(rois), *geo, P(ws), nbytes, st), "prepare")
            _lib.check(L.cim_roi_align_fwd_prepared(P(feat), P(rois), P(mk), P(out), *geo, P(ws), nbytes, st), "fwd")
            _lib.check(L.cim_roi_align_bwd_prepared(P(gout), P(rois), P(mk), P(gf), *geo, P(ws), nbytes, st), "bwd")
        elif fused:
            _lib.check(L.cim_roi_align_maskfuse_fwd(P(feat), P(rois), P(mk), P(out), *geo, P(ws), nbytes, st), "fwd")
            _lib.check(L.cim_roi_align_maskfuse_bwd(P(gout), P(rois), P(mk), P(gf), *geo, P(ws), nbytes, st), "bwd")
        else:
            _lib.check(L.cim_roi_align_fwd(P(feat), P(rois), P(out), *geo, P(ws), nbytes, st), "fwd")
            _lib.check(L.cim_roi_align_bwd(P(gout), P(rois), P(gf), *geo, P(ws), nbytes, st), "bwd")
        torch.cuda.synchronize()
        return out, gf

    o1, g1 = run(False)
    o2, g2 = run(True)
    assert torch.equal(o1, o2)
    if H * W <= 1024:
        assert torch.equal(g1, g2)                      # tile path: bit-reproducible
    else:
        close(g2.cpu().numpy(), g1.cpu().numpy())       # global path: red.global.add order is not fixed


@pytest.mark.parametrize("shape", [(2, 64, 32, 32, 1.0 / 16), (1, 64, 16, 16, 1.0 / 32), (1, 32, 25, 38, 1.0 / 16)])
@pytest.mark.parametrize("fused", [False, True])
def test_backward_tile_in_tensor_memory_equals_shared_memory_bitwise(shape, fused):
    """The default backward keeps its gradient tile in tensor memory (tcgen05.ld / st read-modify-write);
    cim_set_debug_flags(CIM_DBG_ROI_BWD_SMEM_TILE) selects the shared-memory tile.  Same owners, same order: bit-identical, also for odd
    map sizes (last row pair half empty, W not a multiple of 4) and the fused MaskFuse variant."""
    B, C, H, W, scale = shape
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(51))
    rois = random_rois(52, B, 90, H, W, scale)          # no leftover ROIs: their atomics have no fixed order
    masks = (torch.rand(90, 7, 7, generator=torch.Generator().manual_seed(53)) > 0.5).float()

    def grad():
        if fused:
            _, gf, _ = run_maskfuse(feat, rois, masks, scale, 0, True)
        else:
            _, gf, _, _ = run_both(feat, rois, scale, 0, True)
        return gf

    g_tm = grad()
    with _lib.debug_flags(_lib.DBG_ROI_BWD_SMEM_TILE):
        g_sm = grad()
    np.testing.assert_array_equal(g_tm, g_sm)


# ------------------------------------------------------------------ large maps: window tiles (roi_window.cuh)
WINDOW_SHAPES = [
    # B, C, H, W, scale, K
    (2, 64, 64, 64, 1.0 / 8, 120),       # VGG-16 at 512 px (cfg3)
    (1, 32, 75, 75, 1.0 / 16, 90),       # ResNet-50 at scale 1200
    (2, 32, 43, 57, 1.0 / 16, 90),       # odd sizes: padded last row, unaligned window columns
    (1, 32, 150, 112, 1.0 / 8, 60),      # VGG-16 at scale 1200: bins of up to 23 taps (3 slots per bin)
    (1, 32, 20, 90, 1.0 / 8, 60),        # one axis fits the window, the other does not
]


def window_rois(seed, B, K, H, W, scale, wild):
    rng = np.random.RandomState(seed)
    sw, sh = W / scale, H / scale
    w = rng.uniform(0.03, 1.05, K) * sw
    h = rng.uniform(0.03, 1.05, K) * sh
    x1 = rng.uniform(-0.08 if wild else 0, 1, K) * np.maximum(sw - w, 1)
    y1 = rng.uniform(-0.08 if wild else 0, 1, K) * np.maximum(sh - h, 1)
    b = np.sort(rng.randint(0, B, K))
    rois = np.stack([b, x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
    rois[0, 1:] = [0, 0, sw, sh]                                    # the whole map: the most sub-ROIs
    rois[1, 1:] = [sw * 0.4, sh * 0.4, sw * 0.4 + 3, sh * 0.4 + 2]   # a tiny one
    if wild:
        rois[2, 1:] = [-sw, -sh, -sw / 2, -sh / 2]                  # entirely outside the map: zeros
        rois[3, 1:] = [sw * 0.9, sh * 0.9, sw * 1.5, sh * 1.4]      # hanging over the far corner
        rois[4, 1:] = [0, 0, sw * 4, sh * 4]                        # bins wider than 24 taps -> generic leftover pass
    return torch.from_numpy(rois)


@pytest.mark.parametrize("shape", WINDOW_SHAPES)
@pytest.mark.parametrize("aligned,wild", [(True, False), (True, True), (False, True)])
def test_window_tiles_match_oracle(shape, aligned, wild):
    """Maps larger than the shared-memory tile: ROIs cut into sub-ROIs per 32 x 32 window, slots of <= 8 taps summed
    into bins in the epilogue (forward) / fed from their bin's gradient (backward)."""
    B, C, H, W, scale, K = shape
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(H + W))
    rois = window_rois(H * W + K, B, K, H, W, scale, wild)
    out, gf, want, want_g = run_both(feat, rois, scale, 0, aligned)
    close(out, want)
    close(gf, want_g)


@pytest.mark.parametrize("shape", WINDOW_SHAPES[:3])
def test_window_tiles_maskfuse_match_oracle(shape):
    B, C, H, W, scale, K = shape
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(H + W + 1))
    rois = window_rois(H * W + K + 1, B, K, H, W, scale, True)
    masks = (torch.rand(K, 7, 7, generator=torch.Generator().manual_seed(5)) > 0.4).float()
    out, gf, g = run_maskfuse(feat, rois, masks, scale, 0, True)
    want, want_g = maskfuse_oracle(feat, rois, masks, scale, 0, True, g)
    close(out, want)
    close(gf, want_g)


def test_window_tiles_forward_is_bitwise_reproducible_and_ungrouped_rois_work():
    """The forward of the window path writes every bin exactly once (no merging of partial sums): bit-reproducible;
    the stable sort by (image, window) does not need the rois grouped by image."""
    B, C, H, W, scale, K = WINDOW_SHAPES[0]
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(3)).to(DEV)
    rois = window_rois(77, B, K, H, W, scale, False)
    r = rois.to(DEV)
    o1 = ops.roi_align(feat, r, 7, scale, 0, "avg", True)
    o2 = ops.roi_align(feat, r, 7, scale, 0, "avg", True)
    assert torch.equal(o1, o2)
    perm = torch.randperm(K, generator=torch.Generator().manual_seed(4))
    o3 = ops.roi_align(feat, r[perm.to(DEV)], 7, scale, 0, "avg", True)
    assert torch.equal(o3, o1[perm.to(DEV)])


@pytest.mark.parametrize("shape", WINDOW_SHAPES[:2])
def test_global_pairs_path_still_matches_oracle(shape):
    """cim_set_debug_flags(CIM_DBG_ROI_NO_WINDOWS): round 1's channel-last global-memory sweep (kept for A/B timing)."""
    B, C, H, W, scale, K = shape
    if H > 64:
        K = 40
    feat = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(H))
    rois = window_rois(H + K, B, K, H, W, scale, False)
    with _lib.debug_flags(_lib.DBG_ROI_NO_WINDOWS):
        out, gf, want, want_g = run_both(feat, rois, scale, 0, True)
    close(out, want)
    close(gf, want_g)


# ------------------------------------------------------------------ the BENCHMARKED shapes, sampled channels
FULL_SHAPES = {
    # BASELINE.json config: backbone, images, proposals per image
    "cfg2_r50_8x2000": ("resnet50", 8, 2000),
    "cfg3_vgg16_8x2000": ("vgg16", 8, 2000),
    "cfg5_hrnet48_4x4000": ("hrnet48", 4, 4000),
}


@pytest.mark.parametrize("name", sorted(FULL_SHAPES))
def test_benchmarked_shapes_forward_and_backward_on_sampled_channels(name):
    """The kernels at the sizes bench.py times (they pick their code path by shape: tensor-memory tile, window tiles,
    16 x 16 maps with 2048 channels): ALL proposals of the batch, 8 sampled channels, against the oracle."""
    backbone, B, R = FULL_SHAPES[name]
    C, H, W, scale = synth.feature_shape(backbone)
    gen = torch.Generator(device=DEV).manual_seed(len(name))
    feat = torch.randn(B, C, H, W, device=DEV, generator=gen, requires_grad=True)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(R, 512, 600 + b), b) for b in range(B)])
    out = ops.roi_align(feat, rois.to(DEV), 7, scale, 0, "avg", True)
    sel = torch.tensor([0, 1, 31, 32, C // 2 + 5, C - 34, C - 2, C - 1], device=DEV)
    want = roi_oracle.roi_align_fwd(feat.detach()[:, sel].cpu().numpy(), rois.numpy(), 7, 7, scale, 0, True)
    close(out.detach()[:, sel].cpu().numpy(), want)
    g = torch.randn(out.shape, device=DEV, generator=gen)
    (gf,) = torch.autograd.grad(out, feat, g)
    del out
    want_g = roi_oracle.roi_align_bwd(g[:, sel].cpu().numpy(), rois.numpy(), (B, len(sel), H, W), scale, 0, True)
    close(gf[:, sel].cpu().numpy(), want_g)
