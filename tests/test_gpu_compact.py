"""Compact ragged batches on the GPU: rois, RoIAlign outputs and the per-proposal features hold the N = sum(n_b) real
proposals back to back (image b's at rows [off_b, off_b + n_b)), while the scores and everything after them keep the
padded capacity layout.  A compact step must compute what the padded step computes on the same ragged batch: bit for
bit wherever a row's result does not depend on the other rows, to fp32 summation order where the row count changes a
reduction (grad_feat, grad_weight, grad_bias)."""
import numpy as np
import pytest
import torch

import test_gpu_ragged as tr
from cim_b200 import _lib, heads, postproc, synth
from cim_b200.step import CIMHeadStep
from conftest import assert_close_elementwise
from oracle import heads_oracle
from test_gpu_roi_extents import host_problem, path_inputs, per_image_grad
from test_roi_extents_cpu import per_image_oracle
from test_gpu_roi import close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def real_rows(counts, R):
    """padded row of each compact row: image b's proposal r at b * R + r"""
    return np.concatenate([b * R + np.arange(n) for b, n in enumerate(counts)])


def tol(got, want):
    assert_close_elementwise(got.cpu().numpy(), want.cpu().numpy(), rtol=1e-5, atol_rms=1e-5)


@pytest.fixture(scope="module")
def cfg2_batch():
    """cfg2's batch shape (8 x 2000) with ragged_bench's seeded draw, one image at n_b = 1 and one at n_b = R"""
    n_img, R, C, D = 8, 2000, 20, 512
    counts = tr.ragged_counts(2024)
    counts[2], counts[5] = 1, R
    pr = tr.step_inputs(counts, R, C, D, 128, 32, 80)
    w, b = (tr.cuda(a) for a in tr.head_params(D, C + 1, 3, 9))
    return dict(counts=counts, pr=pr, w=w, b=b, n_img=n_img, R=R, C=C, D=D)


def run_both(bt, order, rng):
    """the padded step and the compact step on one ragged batch -> (padded step, compact step, compact row index)"""
    pr, counts, R = bt["pr"], bt["counts"], bt["R"]
    idx = torch.from_numpy(real_rows(counts, R)).to(DEV)
    steps = []
    for compact in (False, True):
        step = tr.make_step(pr, bt["n_img"], R, bt["C"], bt["D"], order=order, rng=rng)
        sel = (lambda t: t.index_select(0, idx).contiguous()) if compact else (lambda t: t)
        np.random.seed(3)
        step.run(pr["feat"], sel(pr["rois"]), sel(pr["grad_out"]), pr["packed"], sel(pr["seg_x"]), bt["w"], bt["b"],
                 pr["labels"].to(DEV), mat=pr["mat"], n_props=counts, compact=compact)
        step.sync_rng()
        torch.cuda.synchronize()
        steps.append(step)
    return steps[0], steps[1], idx


BIT_EQUAL = ("scores", "iou", "asy", "pseudo_labels", "pseudo_iou", "loss_weights", "valid", "asy_flag", "gt_count",
             "gt_keep", "losses", "pcl_loss", "grad_scores")


@pytest.mark.parametrize("order,rng", [("graph", "hop"), ("graph", "stream"), ("overlapped", "hop")])
def test_compact_step_equals_padded_step(cfg2_batch, order, rng):
    padded, compact, idx = run_both(cfg2_batch, order, rng)
    N = idx.numel()
    assert N >= 128 and N < cfg2_batch["n_img"] * cfg2_batch["R"]
    assert torch.equal(compact.roi_out[:N], padded.roi_out.index_select(0, idx))
    for name in BIT_EQUAL:
        u, v = getattr(padded, name), getattr(compact, name)
        if u.dtype == torch.float16:
            u, v = u.view(torch.int16), v.view(torch.int16)
        assert torch.equal(u, v), name
    assert int(padded.gt_count.sum()) > 0 and bool(padded.valid.any())
    assert torch.equal(compact.grad_seg_x[:N], padded.grad_seg_x.index_select(0, idx))
    for name in ("grad_feat", "grad_weight", "grad_bias"):
        tol(getattr(compact, name), getattr(padded, name))


def test_full_counts_compact_equals_no_counts():
    """n_b = R everywhere: the compact step (N = n_img * R) equals n_props = None bit for bit on every output"""
    n_img, R, C, D = 3, 192, 20, 256
    pr = tr.step_inputs([R] * n_img, R, C, D, 128, 32, 50)
    w, b = (tr.cuda(a) for a in tr.head_params(D, C + 1, 3, 9))
    outs = []
    for compact in (False, True):
        step = tr.make_step(pr, n_img, R, C, D)
        np.random.seed(3)
        for _ in range(2):
            step.run(pr["feat"], pr["rois"], pr["grad_out"], pr["packed"], pr["seg_x"], w, b, pr["labels"].to(DEV),
                     mat=pr["mat"], n_props=[R] * n_img if compact else None, compact=compact)
        torch.cuda.synchronize()
        o = tr.step_outputs(step)
        o.update(roi_out=step.roi_out.clone(), grad_feat=step.grad_feat.clone())
        outs.append(o)
    for name, u in outs[0].items():
        v = outs[1][name]
        if u.dtype == torch.float16:
            u, v = u.view(torch.int16), v.view(torch.int16)
        assert torch.equal(u, v), name


# ------------------------------------------------------------------------------------ scoring, small N and autograd
@pytest.mark.parametrize("counts,R", [([50, 1, 30], 64), ([300, 1, 137, 299], 300)])
def test_compact_scoring_against_the_oracle(counts, R):
    """forward_batched(capacity=R) on compact rows, image by image against heads_oracle (N = 81 takes the FFMA
    fallback, N = 737 the tensor cores); padding rows of the scores are 0"""
    D, C1, k, n_img = 256, 21, 3, len(counts)
    w, b = tr.head_params(D, C1, k, 3)
    x = tr.ragged_rows(counts, R, D, 10, 90)[real_rows(counts, R)]
    g = np.random.RandomState(4).randn(2 + 2 * k, n_img * R, C1).astype(np.float32)
    xt, wt, bt = (tr.cuda(a).requires_grad_(True) for a in (x, w, b))
    s = heads.ScoreHeadsFunction.apply(xt, wt, bt, n_img, k, counts, R)
    assert s.shape == (2 + 2 * k, n_img * R, C1)
    s.backward(tr.cuda(g))
    s, gx = s.detach().cpu().numpy(), xt.grad.cpu().numpy()
    assert gx.shape == x.shape
    want_w, want_b = np.zeros(w.shape, np.float64), np.zeros(b.shape, np.float64)
    off = 0
    for i, n in enumerate(counts):
        sl, cs = slice(i * R, i * R + n), slice(off, off + n)
        assert (s[:, i * R + n:(i + 1) * R] == 0).all()
        o = heads_oracle.score_heads(x[cs], list(w), list(b))
        np.testing.assert_allclose(s[:, sl], np.stack([o[0], o[1]] + o[2] + o[3]), rtol=1e-5, atol=1e-8)
        ox, ow, ob = heads_oracle.score_heads_bwd(x[cs], list(w), list(b), list(g[:, sl]))
        tr.rel(gx[cs], ox, 1e-5, 1e-5)
        want_w += np.stack(ow)
        want_b += np.stack(ob)
        off += n
    tr.rel(wt.grad.cpu().numpy(), want_w, 1e-5, 1e-5)
    tr.rel(bt.grad.cpu().numpy(), want_b, 1e-5, 1e-5)


def test_forward_batched_capacity_and_detections():
    """cls_iou_model.forward_batched(capacity=R) equals the padded ragged call: scores bit for bit, grad_x equal to
    the real rows of the padded grad_x; the detections of both score tensors are the same"""
    R, C1, D, k = 300, 21, 256, 3
    counts = [300, 1, 137, 299]
    n_img = len(counts)
    torch.manual_seed(13)
    model = heads.cls_iou_model(D, C1, k).to(DEV)
    xp = tr.cuda(tr.ragged_rows(counts, R, D, 30, 95, scale=1.0))
    idx = torch.from_numpy(real_rows(counts, R)).to(DEV)
    xc = xp.index_select(0, idx).clone()
    g = tr.cuda(np.random.RandomState(5).randn(2 + 2 * k, n_img * R, C1).astype(np.float32))
    out = []
    for x, cap in ((xp, None), (xc, R)):
        x = x.clone().requires_grad_(True)
        s = model.forward_batched(x, n_img, counts, capacity=cap)
        s.backward(g)
        out.append((s.detach(), x.grad))
    assert torch.equal(out[0][0], out[1][0])
    assert torch.equal(out[0][1].index_select(0, idx), out[1][1])
    boxes = np.concatenate([synth.rois_from_params(synth.proposal_params(R, 256, 110 + i))[:, 1:].numpy()
                            for i in range(n_img)]).reshape(n_img, R, 4)
    dets = []
    for s, _ in out:
        t = postproc.test_scores(s, k)
        dets.append(postproc.results_with_nms_and_limit_batched(t.view(n_img, R, C1 - 1), tr.cuda(boxes), 1e-5, 0.3,
                                                                100))
    n_det = 0
    for d0, d1 in zip(*dets):
        for j in range(1, C1):
            np.testing.assert_array_equal(d0[3][j], d1[3][j])
            np.testing.assert_array_equal(np.asarray(d0[2][j]).view(np.uint32), np.asarray(d1[2][j]).view(np.uint32))
            n_det += len(d0[3][j])
    assert n_det > 0


# ------------------------------------------------------------------------------------ RoIAlign on N < n_img * R rois
def roi_prepared(feat, rois, hw, scale, K_cap, g):
    """prepare / forward / backward through the _prepared_ex entry points on K = len(rois), workspace sized for K_cap"""
    L, P = _lib.lib(), _lib.ptr
    B, Cc, H, W = feat.shape
    K = rois.shape[0]
    st = _lib.stream_ptr(DEV)
    ws = torch.empty(L.cim_roi_align_workspace_bytes_ex(B, Cc, H, W, K_cap, 7, 7), dtype=torch.uint8, device=DEV)
    out = torch.empty(K, Cc, 7, 7, device=DEV)
    gf = torch.empty_like(feat)
    _lib.check(L.cim_roi_align_prepare_ex(P(rois), P(hw), B, Cc, H, W, K, 7, 7, scale, 0, 1, P(ws), ws.numel(), st),
               "prepare")
    _lib.check(L.cim_roi_align_fwd_prepared_ex(P(feat), P(rois), P(hw), None, P(out), B, Cc, H, W, K, 7, 7, scale, 0,
                                               1, P(ws), ws.numel(), st), "fwd")
    _lib.check(L.cim_roi_align_bwd_prepared_ex(P(g), P(rois), P(hw), None, P(gf), B, Cc, H, W, K, 7, 7, scale, 0, 1,
                                               P(ws), ws.numel(), st), "bwd")
    torch.cuda.synchronize()
    return out, gf


@pytest.mark.parametrize("path", ["tile", "window_vgg16", "generic"])
@pytest.mark.parametrize("extents", [False, True])
def test_roi_align_on_compact_rois(path, extents):
    """K = N rois (grouped by image, uneven counts) on a workspace sized for the padded capacity: each image's outputs
    and gradient equal the oracle on that image alone (its cropped map with extents).  "generic": the 64 x 64 map with
    the window tiles switched off (global-pairs kernels)"""
    feat, rois, hw, scale = path_inputs("window_vgg16" if path == "generic" else path, 300 + extents, K=40)
    if not extents:
        hw = np.array([feat.shape[2:]] * feat.shape[0], np.int32)
    counts = np.bincount(rois[:, 0].long().numpy(), minlength=feat.shape[0])
    K_cap = feat.shape[0] * int(counts.max()) * 2
    g = torch.randn(len(rois), feat.shape[1], 7, 7, generator=torch.Generator().manual_seed(9))
    flags = _lib.DBG_ROI_NO_WINDOWS if path == "generic" else 0
    with _lib.debug_flags(flags):
        out, gf = roi_prepared(feat.to(DEV), rois.to(DEV), tr.cuda(hw) if extents else None, scale, K_cap, g.to(DEV))
    fn, rn = feat.numpy(), rois.numpy()
    close(out.cpu().numpy(), per_image_oracle(fn, rn, hw, scale, 0, True))
    close(gf.cpu().numpy(), per_image_grad(g.numpy(), rn, hw, tuple(feat.shape), scale, 0, True))


# ------------------------------------------------------------------------------------ run_host
@pytest.mark.parametrize("depth", [1, 2])
def test_run_host_compact(depth):
    """alloc_host_io(ragged=True, compact=True): N changes every step; each call equals run(compact=True) on the same
    inputs (RoIAlign rows, losses, valid flags, maps, compact grad_seg_x)"""
    n_img, R, C, D, Cf, size = 3, 96, 20, 256, 32, 128
    probs = [host_problem(1, [96, 40, 71]), host_problem(2, [13, 96, 60]), host_problem(3, [80, 55, 96])]
    for p in probs:
        i = torch.from_numpy(real_rows(p["counts"], R))
        p.update(c_rois=p["rois"][i].contiguous(), c_seg=p["seg_x"][i.to(DEV)].contiguous(),
                 c_go=p["grad_out"][i.to(DEV)].contiguous(), N=len(i))
    kb = size // 16
    feat = torch.randn(n_img, Cf, size // 16, size // 16, generator=torch.Generator().manual_seed(3)).to(DEV)
    torch.manual_seed(1)
    weight, bias = (t.detach().contiguous() for t in heads.cls_iou_model(D, C + 1, 3).to(DEV)._stacked())
    mk = lambda: CIMHeadStep(n_img, R, C, Cf, size // 16, size // 16, 1.0 / 16, size * size // 32, feat_dim=D,
                             device=DEV, mask_kb_per_row=kb, head_grads=True)
    n_calls = 6
    fed = [probs[t % 3] for t in range(n_calls)]
    seen = [fed[max(0, t - depth)] for t in range(n_calls)]
    ref = mk()
    want = []
    np.random.seed(3)
    for pr in seen:
        ref.run(feat, pr["c_rois"].to(DEV), pr["c_go"], pr["packed"], pr["c_seg"], weight, bias, pr["labels"].to(DEV),
                n_props=pr["counts"], compact=True)
        torch.cuda.synchronize()
        want.append((ref.losses.cpu().numpy().copy(), ref.valid.cpu().numpy().copy(), ref.iou.clone(),
                     ref.roi_out[:pr["N"]].clone(), ref.grad_seg_x[:pr["N"]].clone()))
    step = mk()
    cap = max(int(p["crops"].words.numel()) for p in probs) + 64
    step.alloc_host_io(mask_hw=(size, size), crop_capacity_words=cap, prefetch_depth=depth, ragged=True, compact=True)
    np.random.seed(3)
    for t in range(n_calls):
        pr, sp = fed[t], seen[t]
        step.wait_inputs_consumed()
        step.hi_rois.zero_()
        step.hi_rois[:pr["N"]].copy_(pr["c_rois"])
        step.hi_labels.copy_(pr["labels"])
        step.hi_n_props.copy_(torch.tensor(pr["counts"], dtype=torch.int32))
        step.set_host_crops(pr["crops"])
        if t == 0:
            with pytest.raises(ValueError):
                step.run_host(feat, sp["c_go"][1:], sp["c_seg"][1:], weight, bias)
        assert step.next_step_rows() == sp["N"]
        step.run_host(feat, sp["c_go"], sp["c_seg"], weight, bias)
        got = step.results_host
        w_loss, w_valid, w_iou, w_roi, w_gx = want[t]
        np.testing.assert_array_equal(got["valid"], w_valid)
        np.testing.assert_array_equal(np.nan_to_num(got["losses"], nan=-7.0), np.nan_to_num(w_loss, nan=-7.0))
        torch.cuda.synchronize()
        assert torch.equal(step.iou.view(torch.int16), w_iou.view(torch.int16))
        assert torch.equal(step.roi_out[:sp["N"]], w_roi)
        assert torch.equal(step.grad_seg_x[:sp["N"]], w_gx)


# ------------------------------------------------------------------------------------ refusals
def test_compact_refusals():
    n_img, R, C, D = 2, 64, 20, 256
    counts = [10, 64]
    pr = tr.step_inputs(counts, R, C, D, 128, 32, 50)
    w, b = (tr.cuda(a) for a in tr.head_params(D, C + 1, 3, 9))
    idx = torch.from_numpy(real_rows(counts, R)).to(DEV)
    rois, go, x = (pr[k].index_select(0, idx) for k in ("rois", "grad_out", "seg_x"))
    step = tr.make_step(pr, n_img, R, C, D)
    run = lambda **kw: step.run(pr["feat"], kw.get("rois", rois), kw.get("go", go), pr["packed"], kw.get("x", x), w, b,
                                pr["labels"].to(DEV), n_props=kw.get("n", counts), compact=True)
    for kw, exc in ((dict(n=torch.tensor(counts, dtype=torch.int32, device=DEV)), ValueError),
                    (dict(n=None), ValueError), (dict(rois=rois[1:]), ValueError), (dict(go=go[:-1]), ValueError),
                    (dict(x=pr["seg_x"]), ValueError), (dict(n=[0, 74]), ValueError), (dict(n=[10, 65]), ValueError),
                    (dict(n=[10.0, 64.0]), TypeError)):
        with pytest.raises(exc):
            run(**kw)
    ws, wb = (t.clone().requires_grad_(True) for t in (w, b))
    for n_props, rows, exc in ((torch.tensor(counts, dtype=torch.int32, device=DEV), x, ValueError),
                               (counts, pr["seg_x"], ValueError), ([10, 65], x, ValueError), ([0, 74], x, ValueError)):
        with pytest.raises(exc):
            heads.ScoreHeadsFunction.apply(rows, ws, wb, n_img, 3, n_props, R)
    with pytest.raises(ValueError):
        CIMHeadStep(n_img, R, C, 32, 8, 8, 1.0 / 16, pr["packed"].shape[-1], feat_dim=D, device=DEV).alloc_host_io(
            compact=True)
