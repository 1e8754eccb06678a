"""Ragged batches on the GPU: images with different proposal counts n_b in one batch of capacity R (image b owns rows
[0, n_b) of its R rows).  Every result of image b must equal the oracle run on that image alone at R = n_b, no result
may depend on what the padding rows hold, padding rows of the outputs are 0, and n_props = R everywhere is
bit-identical to n_props = None."""
import numpy as np
import pytest
import torch

from cim_b200 import _lib, heads, mask_ops, postproc, synth
from cim_b200.step import CIMHeadStep
from oracle import heads_oracle, loss_oracle, nms_oracle
from conftest import assert_f16_bits_equal, assert_close_elementwise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAN16 = np.uint16(0x7E00)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def rel(got, want, rtol=2e-5, atol_rms=5e-5):
    """element-wise bound of tests/test_gpu_step.py (the chain carries three stages of fp32 rounding), then the
    max-norm error"""
    assert_close_elementwise(got, want, rtol=rtol, atol_rms=atol_rms)
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-3))


def head_params(D, C1, k, seed):
    torch.manual_seed(seed)
    w, b = heads.cls_iou_model(D, C1, k)._stacked()
    return w.detach().numpy().copy(), b.detach().numpy().copy()


def ragged_rows(n_props, R, width, seed, pad_seed, scale=3.0):
    """[n_img * R, width] float32: rows < n_b from `seed` (image by image), padding rows from `pad_seed`"""
    out = np.empty((len(n_props) * R, width), np.float32)
    for b, n in enumerate(n_props):
        out[b * R:b * R + n] = np.random.RandomState(seed + b).randn(n, width) * scale
        out[b * R + n:(b + 1) * R] = np.random.RandomState(pad_seed + b).randn(R - n, width) * scale
    return out


def score(x, w, b, n_img, k, n_props, ffma=False, grad=None):
    """ragged scoring forward (+ backward with dL/dscores = grad) -> numpy (scores, grad_x, grad_w, grad_b)"""
    xt, wt, bt = (cuda(a).requires_grad_(grad is not None) for a in (x, w, b))
    with _lib.debug_flags(_lib.DBG_SCORE_FFMA if ffma else 0):
        s = heads.ScoreHeadsFunction.apply(xt, wt, bt, n_img, k, n_props)
        if grad is None:
            return s.detach().cpu().numpy(), None, None, None
        s.backward(cuda(grad))
    return s.detach().cpu().numpy(), xt.grad.cpu().numpy(), wt.grad.cpu().numpy(), bt.grad.cpu().numpy()


# ------------------------------------------------------------------------------------ 1 + 4: scoring fwd / bwd
@pytest.mark.parametrize("ffma", [False, True])
@pytest.mark.parametrize("R,C1,n_props", [(300, 21, [300, 1, 137, 299]), (256, 81, [256, 1, 100, 255, 17])])
def test_scoring_per_image_and_zero_padding(R, C1, n_props, ffma):
    """Each image's rows against heads_oracle.score_heads / score_heads_bwd on that image alone (the detector softmax
    over its n_b rows); every head is exactly 0 on padding rows, and so is grad_x, even with NaN in grad_scores
    there; grad_W / grad_b are the sums over the images."""
    D, k, n_img = 256, 3, len(n_props)
    nh = 2 + 2 * k
    w, b = head_params(D, C1, k, 3)
    x = ragged_rows(n_props, R, D, 10, 90)
    g = np.random.RandomState(4).randn(nh, n_img * R, C1).astype(np.float32)
    pad = np.ones(n_img * R, bool)
    for i, n in enumerate(n_props):
        pad[i * R:i * R + n] = False
    g[:, pad] = np.nan                                            # must not reach anything
    s, gx, gw, gb = score(x, w, b, n_img, k, torch.tensor(n_props), ffma, g)
    assert (s[:, pad] == 0).all() and (gx[pad] == 0).all()
    want_w, want_b = np.zeros(w.shape, np.float64), np.zeros(b.shape, np.float64)
    for i, n in enumerate(n_props):
        sl = slice(i * R, i * R + n)
        o = heads_oracle.score_heads(x[sl], list(w), list(b))
        np.testing.assert_allclose(s[:, sl], np.stack([o[0], o[1]] + o[2] + o[3]), rtol=1e-5, atol=1e-8)
        ox, ow, ob = heads_oracle.score_heads_bwd(x[sl], list(w), list(b), list(g[:, sl]))
        rel(gx[sl], ox, 1e-5, 1e-5)
        want_w += np.stack(ow)
        want_b += np.stack(ob)
    rel(gw, want_w, 1e-5, 1e-5)
    rel(gb, want_b, 1e-5, 1e-5)


# ------------------------------------------------------------------------------------ the whole head chain
def chain_inputs(n_props, R, C, D, pad_seed, size=64, nan_maps=True, with_maps=True):
    """A ragged batch whose valid rows depend on fixed seeds only and whose padding rows on pad_seed: features, maps
    (valid block from the masks of the image alone; padding rows and columns NaN or random fp16), cluster matrix."""
    n_img = len(n_props)
    rs = np.random.RandomState(pad_seed)
    iou = np.empty((n_img, R, R) if with_maps else 0, np.uint16)
    asy = np.empty((n_img, R, R) if with_maps else 0, np.uint16)
    for b, n in enumerate(n_props if with_maps else ()):
        if nan_maps:
            iou[b], asy[b] = NAN16, NAN16
        else:
            iou[b] = np.float16(rs.rand(R, R)).view(np.uint16)
            asy[b] = np.float16(rs.rand(R, R)).view(np.uint16)
        m = synth.rasterize(synth.proposal_params(n, size, 500 + b), device=DEV)
        mi, ma = mask_ops.mask_overlap(mask_ops.mask_pack(m))
        iou[b, :n, :n] = mi.cpu().numpy().view(np.uint16)
        asy[b, :n, :n] = ma.cpu().numpy().view(np.uint16)
    labels = np.concatenate([synth.image_labels(C, 2, 600 + b).numpy() for b in range(n_img)])
    mat = rs.randint(0, 12, size=(n_img, R, C + 1)).astype(np.float32)
    for b, n in enumerate(n_props):
        mat[b, :n] = synth.cluster_mat(n, C, np.nonzero(labels[b])[0], 4, 700 + b).numpy()
    if not with_maps:
        iou = asy = None
    else:
        iou, asy = iou.view(np.float16), asy.view(np.float16)
    return dict(x=ragged_rows(n_props, R, D, 20, pad_seed), iou=iou, asy=asy,
                labels=labels, mat=mat)


def run_chain(inp, w, b, n_props, k, using_cim=True, anti=True, seed=3):
    """ragged scoring -> mining + assignment -> loss block + PCL_loss -> backward, through the public Python surface"""
    n_img = len(n_props)
    xt, wt, bt = (cuda(a).requires_grad_(True) for a in (inp["x"], w, b))
    s = heads.ScoreHeadsFunction.apply(xt, wt, bt, n_img, k, n_props)
    s.retain_grad()
    R = s.shape[1] // n_img
    s4 = s.detach().view(2 + 2 * k, n_img, R, -1)
    cls_l = [s4[0]] + [s4[2 + l - 1] for l in range(1, k)]
    det_l = [s4[1]] + [s4[2 + k + l - 1] for l in range(1, k)]
    labels = cuda(inp["labels"])
    np.random.seed(seed)
    a = heads.mine_and_assign(cls_l, det_l, labels, cuda(inp["iou"]), cuda(inp["asy"]),
                              [0.25 + 0.1 * l for l in range(k)], [0.5 + 0.1 * l for l in range(k)],
                              anti_noise_sampling=anti, using_cim=using_cim, n_props=n_props)
    rng = np.random.get_state()
    hl = heads.head_losses(s, a, labels, k)
    pcl = heads.PCL_loss(s[0], cuda(inp["mat"]), n_img=n_img, n_props=n_props)
    (hl["total"].mean() + pcl.mean()).backward()
    torch.cuda.synchronize()
    return dict(scores=s.detach(), assigned=a, losses=hl["losses"].detach(), pcl=pcl.detach(), grad_scores=s.grad,
                grad_x=xt.grad, grad_w=wt.grad, grad_b=bt.grad, rng=rng)


def gt_lists(a, l, b):
    c = int(a["gt_count"][l, b])
    return a["gt_rows"][l, b, :c], a["gt_class"][l, b, :c], a["gt_weight"][l, b, :c]


# ------------------------------------------------------------------------------------ 2: padding invariance
@pytest.mark.parametrize("using_cim", [True, False])
def test_results_do_not_depend_on_padding_contents(using_cim):
    """Two batches that differ only in their padding rows (x, the maps' padding rows and columns -- NaN in one, random
    fp16 in the other -- and random cluster ids in mat): every output of scoring, mining, assignment, losses, PCL and
    the backward is equal element for element, integers and fp16 bit for bit."""
    R, C, D, k = 400, 20, 256, 3
    n_props = [400, 1, 9, 233, 399]
    w, b = head_params(D, C + 1, k, 5)
    out = [run_chain(chain_inputs(n_props, R, C, D, ps, nan_maps=nm), w, b, n_props, k, using_cim)
           for ps, nm in ((31, True), (77, False))]
    a0, a1 = out[0]["assigned"], out[1]["assigned"]
    assert int(a0["gt_count"].sum()) > 0
    for key in ("scores", "losses", "pcl", "grad_scores", "grad_x", "grad_w", "grad_b"):
        assert torch.equal(out[0][key], out[1][key]), key
    for key in ("pseudo_labels", "loss_weights", "valid", "asy_iou_flag", "gt_count", "gt_keep"):
        assert torch.equal(a0[key], a1[key]), key
    assert torch.equal(a0["pseudo_iou_labels"].view(torch.int16), a1["pseudo_iou_labels"].view(torch.int16))
    for l in range(k):
        for i in range(len(n_props)):
            for u, v in zip(gt_lists(a0, l, i), gt_lists(a1, l, i)):
                assert torch.equal(u, v)
    assert np.array_equal(out[0]["rng"][1], out[1]["rng"][1])


# ------------------------------------------------------------------------------------ 3: mining + assignment
@pytest.mark.parametrize("using_cim,anti", [(True, True), (True, False), (False, True), (False, False)])
def test_mining_bit_exact_per_image(using_cim, anti):
    """mine_and_assign on one ragged batch against heads_oracle.cim_layer_forward run image by image at R = n_b, on
    the GPU's scores: gt lists, pseudo labels, fp16 IoU labels, weights and asy_flag bit for bit, and numpy's global
    RNG left where the image-by-image loop leaves it.  The counts straddle the steps of ceil(0.1 n) and 0.9 n."""
    R, C, D, k = 2000, 20, 256, 3
    n_props = [1, 9, 10, 11, 19, 20, 21, 1001, 2000]
    w, b = head_params(D, C + 1, k, 7)
    inp = chain_inputs(n_props, R, C, D, 41)
    got = run_chain(inp, w, b, n_props, k, using_cim, anti, seed=11)
    a = {key: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for key, v in got["assigned"].items()}
    s4 = got["scores"].cpu().numpy().reshape(2 + 2 * k, len(n_props), R, C + 1)
    cls_l = [s4[0]] + [s4[2 + l - 1] for l in range(1, k)]
    det_l = [s4[1]] + [s4[2 + k + l - 1] for l in range(1, k)]
    np.random.seed(11)
    n_valid = 0
    for i, n in enumerate(n_props):
        iou, asy = inp["iou"][i, :n, :n], inp["asy"][i, :n, :n]
        lab = inp["labels"][i:i + 1]
        flag = heads_oracle.big_proposal_flag(asy, 0.85)
        np.testing.assert_array_equal(a["asy_iou_flag"][i, :n], flag.astype(np.uint8))
        assert (a["asy_iou_flag"][i, n:] == 0).all()
        for l in range(k):
            cls, det = cls_l[l][i, :n], det_l[l][i, :n]
            cthr, ithr = 0.25 + 0.1 * l, 0.5 + 0.1 * l
            if using_cim:
                g_cls, g_w = heads_oracle.cim_label(cls, det, lab, iou, asy, 0.1, cthr, 0.85)[:2]
            else:
                g_cls, g_w = heads_oracle.mist_label(cls * det, lab, iou, 0.1, cthr)
            rows = np.nonzero(g_cls >= 0)[0]
            g_rows, g_c, g_wt = (t[l, i, :int(a["gt_count"][l, i])] for t in (a["gt_rows"], a["gt_class"],
                                                                             a["gt_weight"]))
            np.testing.assert_array_equal(g_rows, rows)
            np.testing.assert_array_equal(g_c, g_cls[rows])
            np.testing.assert_array_equal(g_wt.view(np.uint32), g_w[rows].view(np.uint32))
            o = heads_oracle.cim_layer_forward(cls, det, lab, iou, asy, 0.1, cthr, ithr, 0.85, anti, using_cim)
            assert a["valid"][l, i] == (o[0] is not None)
            assert (a["pseudo_labels"][l, i, n:] == 0).all() and (a["loss_weights"][l, i, n:] == 0).all()
            assert (a["pseudo_iou_labels"][l, i, n:].view(np.uint16) == 0).all()
            if o[0] is None:
                continue
            n_valid += 1
            np.testing.assert_array_equal(a["pseudo_labels"][l, i, :n], o[0])
            assert_f16_bits_equal(a["pseudo_iou_labels"][l, i, :n].view(np.uint16), o[1].view(np.uint16))
            np.testing.assert_array_equal(a["loss_weights"][l, i, :n].view(np.uint32), o[2].view(np.uint32))
    assert n_valid > 0
    want = np.random.get_state()
    assert np.array_equal(got["rng"][1], want[1]) and got["rng"][2] == want[2]


# ------------------------------------------------------------------------------------ 4: losses, PCL, backward
def test_losses_pcl_and_backward_per_image():
    """The loss block, PCL_loss and the scoring backward of a ragged batch against loss_oracle.head_losses /
    pcl_losses and heads_oracle.score_heads_bwd per image at n_b; grad_scores and grad_x are exactly 0 on padding
    rows (the loss block gets no n_props: the zeros the ragged kernels write at padding are enough)."""
    R, C, D, k = 400, 20, 256, 3
    n_props = [400, 1, 9, 233, 399]
    n_img = len(n_props)
    w, b = head_params(D, C + 1, k, 5)
    inp = chain_inputs(n_props, R, C, D, 31)
    got = run_chain(inp, w, b, n_props, k)
    s = got["scores"].cpu().numpy()
    a = {key: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for key, v in got["assigned"].items()}
    gs, gx = got["grad_scores"].cpu().numpy(), got["grad_x"].cpu().numpy()
    losses, pcl = got["losses"].cpu().numpy(), got["pcl"].cpu().numpy()
    want_w, want_b = np.zeros(w.shape, np.float64), np.zeros(b.shape, np.float64)
    assert a["valid"].any()
    for i, n in enumerate(n_props):
        sl = slice(i * R, i * R + n)
        o_loss, o_grad = loss_oracle.head_losses(s[:, sl], a["pseudo_labels"][:, i:i + 1, :n],
                                                 a["pseudo_iou_labels"][:, i:i + 1, :n], a["loss_weights"][:, i:i + 1, :n],
                                                 a["valid"][:, i:i + 1], inp["labels"][i:i + 1], k, grad_scale=1.0 / n_img)
        o_pcl, g_pcl = loss_oracle.pcl_losses(s[0, sl], inp["mat"][i:i + 1, :n], grad_scale=1.0 / n_img)
        o_grad[0] += g_pcl
        np.testing.assert_allclose(losses[i], o_loss[0], rtol=2e-5, atol=1e-7)
        np.testing.assert_allclose(pcl[i], o_pcl[0], rtol=2e-5)
        rel(gs[:, sl], o_grad)
        assert (gs[:, i * R + n:(i + 1) * R] == 0).all() and (gx[i * R + n:(i + 1) * R] == 0).all()
        ox, ow, ob = heads_oracle.score_heads_bwd(inp["x"][sl], list(w), list(b), list(gs[:, sl]),
                                                  outputs=list(s[:, sl]))
        rel(gx[sl], ox)
        want_w += np.stack(ow)
        want_b += np.stack(ob)
    rel(got["grad_w"].cpu().numpy(), want_w)
    rel(got["grad_b"].cpu().numpy(), want_b)


# ------------------------------------------------------------------------------------ the CIMHeadStep
def step_inputs(n_props, R, C, D, size, Cf, pad_seed, zero_pad_masks=False):
    """Everything CIMHeadStep.run takes for a ragged batch; valid rows from fixed seeds, padding rows from pad_seed:
    finite seg_x, the image's own rois, random (or empty) masks, random cluster ids, grad_out rows of 0."""
    n_img = len(n_props)
    inp = chain_inputs(n_props, R, C, D, pad_seed, with_maps=False)
    H = W = size // 16
    feat = torch.randn(n_img, Cf, H, W, generator=torch.Generator().manual_seed(1))
    grad_out = torch.randn(n_img * R, Cf, 7, 7, generator=torch.Generator().manual_seed(2))
    rois, masks, valid_masks = [], [], []
    for b, n in enumerate(n_props):
        pv = synth.proposal_params(n, size, 40 + b)
        pp = synth.proposal_params(max(R - n, 1), size, pad_seed + b)
        rois += [synth.rois_from_params(pv, b), synth.rois_from_params(pp, b)[:R - n]]
        mv = synth.rasterize(pv, device=DEV)
        mp = synth.rasterize(pp, device=DEV)[:R - n]
        if zero_pad_masks:
            mp = torch.zeros_like(mp)
        valid_masks.append(mv)
        masks.append(mask_ops.mask_pack(torch.cat([mv, mp])))
        grad_out[b * R + n:(b + 1) * R] = 0
    labels = torch.from_numpy(inp["labels"])
    return dict(feat=feat.to(DEV), rois=torch.cat(rois).to(DEV), grad_out=grad_out.to(DEV), packed=torch.stack(masks),
                seg_x=cuda(inp["x"]), labels=labels, mat=cuda(inp["mat"]), valid_masks=valid_masks,
                kb=size // 16 if mask_ops.tiled_ok(size, size) else 0, H=H, W=W, Cf=Cf)


def make_step(pr, n_img, R, C, D, **kw):
    return CIMHeadStep(n_img, R, C, pr["Cf"], pr["H"], pr["W"], 1.0 / 16, pr["packed"].shape[-1], feat_dim=D,
                       device=DEV, mask_kb_per_row=pr["kb"], head_grads=True, **kw)


def run_step(step, pr, w, b, n_props):
    step.run(pr["feat"], pr["rois"], pr["grad_out"], pr["packed"], pr["seg_x"], w, b, pr["labels"].to(DEV),
             mat=pr["mat"], n_props=n_props)


STEP_OUTPUTS = ("scores", "pseudo_labels", "pseudo_iou", "loss_weights", "valid", "asy_flag", "gt_count", "gt_keep",
                "losses", "pcl_loss", "grad_scores", "grad_seg_x", "grad_weight", "grad_bias")


def step_outputs(step):
    return {name: getattr(step, name).clone() for name in STEP_OUTPUTS}


def assert_outputs_equal(o0, o1):
    for name in STEP_OUTPUTS:
        u, v = o0[name], o1[name]
        if u.dtype == torch.float16:
            u, v = u.view(torch.int16), v.view(torch.int16)
        assert torch.equal(u, v), name


# ------------------------------------------------------------------------------------ 5: full counts
@pytest.mark.parametrize("rng", ["hop", "stream"])
def test_full_counts_equal_no_counts(rng):
    """n_props = R for every image through the ragged kernels is bit-identical to n_props = None, for every output of
    a CIMHeadStep with head gradients and PCL_loss, and leaves numpy's RNG in the same state."""
    n_img, R, C, D = 3, 192, 20, 256
    pr = step_inputs([R] * n_img, R, C, D, 128, 32, 50)
    w, b = (cuda(a) for a in head_params(D, C + 1, 3, 9))
    res = []
    for n_props in (None, [R] * n_img, torch.full((n_img,), R, dtype=torch.int32, device=DEV)):
        step = make_step(pr, n_img, R, C, D, rng=rng)
        np.random.seed(3)
        for _ in range(2):
            run_step(step, pr, w, b, n_props)
        step.sync_rng()
        torch.cuda.synchronize()
        res.append((step_outputs(step), np.random.get_state()[1].copy()))
    assert int(res[0][0]["gt_count"].sum()) > 0
    for o, st in res[1:]:
        assert_outputs_equal(res[0][0], o)
        assert np.array_equal(res[0][1], st)


def test_step_does_not_depend_on_padding_contents():
    """CIMHeadStep on two batches that differ only in padding rows: different seg_x, rois, masks (random in one, empty
    in the other, so the maps' padding columns are NaN there) and cluster ids -- every result is equal."""
    n_img, R, C, D = 4, 256, 20, 256
    n_props = [256, 1, 100, 255]
    w, b = (cuda(a) for a in head_params(D, C + 1, 3, 9))
    outs = []
    for pad_seed, zero in ((60, False), (61, True)):
        pr = step_inputs(n_props, R, C, D, 128, 32, pad_seed, zero_pad_masks=zero)
        step = make_step(pr, n_img, R, C, D)
        np.random.seed(3)
        run_step(step, pr, w, b, n_props)
        torch.cuda.synchronize()
        outs.append(step_outputs(step))
    assert int(outs[0]["gt_count"].sum()) > 0
    assert_outputs_equal(outs[0], outs[1])


# ------------------------------------------------------------------------------------ 6: cfg2 shape, stage by stage
def ragged_counts(seed, n_img=8, lo=200, hi=2000):
    return [int(v) for v in np.random.RandomState(seed).randint(lo, hi + 1, size=n_img)]


def test_step_cfg2_shape_stage_by_stage():
    """8 x 2000 with seeded ragged n_b >= 200, sampling through the host hop and through the device stream: maps,
    scores, pseudo labels, losses, PCL_loss and head gradients of every image against the oracles at R = n_b (fed
    the GPU's maps and scores, as tests/test_gpu_step.py does); padding rows 0; both RNG modes agree bit for bit."""
    n_img, R, C, D, k = 8, 2000, 20, 512, 3
    n_props = ragged_counts(2024)
    pr = step_inputs(n_props, R, C, D, 128, 32, 80)
    w, b = (cuda(a) for a in head_params(D, C + 1, k, 9))
    res = {}
    for mode in ("hop", "stream"):
        step = make_step(pr, n_img, R, C, D, rng=mode)
        np.random.seed(3)
        run_step(step, pr, w, b, n_props)
        step.sync_rng()
        torch.cuda.synchronize()
        res[mode] = (step_outputs(step), np.random.get_state()[1].copy(), step)
    assert_outputs_equal(res["hop"][0], res["stream"][0])
    assert np.array_equal(res["hop"][1], res["stream"][1])
    step = res["hop"][2]

    w_np, b_np = w.cpu().numpy(), b.cpu().numpy()
    x = pr["seg_x"].cpu().numpy()
    scores = step.scores.cpu().numpy()
    iou, asy = step.iou.cpu().numpy(), step.asy.cpu().numpy()
    s4 = scores.reshape(2 + 2 * k, n_img, R, C + 1)
    cls_l, det_l = [s4[0], s4[2], s4[3]], [s4[1], s4[5], s4[6]]
    labels, mat = pr["labels"].numpy(), pr["mat"].cpu().numpy()
    pl, pi, lw, valid = (t.cpu().numpy() for t in (step.pseudo_labels, step.pseudo_iou, step.loss_weights, step.valid))
    gs, gx = step.grad_scores.cpu().numpy(), step.grad_seg_x.cpu().numpy()
    np.random.seed(3)
    want_w, want_b = np.zeros(w_np.shape, np.float64), np.zeros(b_np.shape, np.float64)
    for i, n in enumerate(n_props):
        sl, pad = slice(i * R, i * R + n), slice(i * R + n, (i + 1) * R)
        mi, ma = mask_ops.mask_overlap(mask_ops.mask_pack(pr["valid_masks"][i]))
        assert_f16_bits_equal(iou[i, :n, :n].view(np.uint16), mi.cpu().numpy().view(np.uint16))
        assert_f16_bits_equal(asy[i, :n, :n].view(np.uint16), ma.cpu().numpy().view(np.uint16))
        o = heads_oracle.score_heads(x[sl], list(w_np), list(b_np))
        np.testing.assert_allclose(scores[:, sl], np.stack([o[0], o[1]] + o[2] + o[3]), rtol=1e-5, atol=1e-7)
        assert (scores[:, pad] == 0).all()
        for l in range(k):
            o = heads_oracle.cim_layer_forward(cls_l[l][i, :n], det_l[l][i, :n], labels[i:i + 1], iou[i, :n, :n],
                                               asy[i, :n, :n], 0.1, 0.25 + 0.1 * l, 0.5 + 0.1 * l, 0.85, True)
            assert valid[l, i] == (o[0] is not None)
            assert (pl[l, i, n:] == 0).all() and (lw[l, i, n:] == 0).all() and (pi[l, i, n:] == 0).all()
            if o[0] is not None:
                np.testing.assert_array_equal(pl[l, i, :n], o[0])
                assert_f16_bits_equal(pi[l, i, :n].view(np.uint16), o[1].view(np.uint16))
                np.testing.assert_array_equal(lw[l, i, :n], o[2])
        o_loss, o_grad = loss_oracle.head_losses(scores[:, sl], pl[:, i:i + 1, :n], pi[:, i:i + 1, :n],
                                                 lw[:, i:i + 1, :n], valid[:, i:i + 1], labels[i:i + 1], k,
                                                 grad_scale=1.0 / n_img)
        o_pcl, g_pcl = loss_oracle.pcl_losses(scores[0, sl], mat[i:i + 1, :n], grad_scale=1.0 / n_img)
        o_grad[0] += g_pcl
        np.testing.assert_allclose(step.losses[i].cpu().numpy(), o_loss[0], rtol=2e-5, atol=1e-7)
        np.testing.assert_allclose(step.pcl_loss[i].cpu().numpy(), o_pcl[0], rtol=2e-5)
        rel(gs[:, sl], o_grad)
        assert (gs[:, pad] == 0).all() and (gx[pad] == 0).all()
        ox, ow, ob = heads_oracle.score_heads_bwd(x[sl], list(w_np), list(b_np), list(gs[:, sl]),
                                                  outputs=list(scores[:, sl]))
        rel(gx[sl], ox)
        want_w += np.stack(ow)
        want_b += np.stack(ob)
    assert valid.any()
    assert np.array_equal(np.random.get_state()[1], res["hop"][1])
    rel(step.grad_weight.cpu().numpy(), want_w)
    rel(step.grad_bias.cpu().numpy(), want_b)


def test_stream_sampling_with_changing_counts():
    """Two consecutive steps with different n_props: rng="stream" gives what rng="hop" gives, step by step, and
    numpy's generator is where the hop leaves it after sync_rng()."""
    n_img, R, C, D = 8, 2000, 20, 256
    counts = [ragged_counts(7), ragged_counts(8)]
    pr = step_inputs([R] * n_img, R, C, D, 128, 32, 90)
    w, b = (cuda(a) for a in head_params(D, C + 1, 3, 9))
    res = {}
    for mode in ("hop", "stream"):
        step = make_step(pr, n_img, R, C, D, rng=mode)
        np.random.seed(5)
        outs = []
        for n_props in counts:
            run_step(step, pr, w, b, torch.tensor(n_props, dtype=torch.int32, device=DEV))
            outs.append(step_outputs(step))
        step.sync_rng()
        torch.cuda.synchronize()
        res[mode] = (outs, np.random.get_state()[1].copy())
    assert not torch.equal(res["hop"][0][0]["gt_count"], res["hop"][0][1]["gt_count"])
    for o0, o1 in zip(res["hop"][0], res["stream"][0]):
        assert_outputs_equal(o0, o1)
    assert np.array_equal(res["hop"][1], res["stream"][1])


# ------------------------------------------------------------------------------------ 7: inference
def test_inference_chain_per_image():
    """Ragged scoring -> test_scores -> per-class NMS -> detection limit and lists equals
    nms_oracle.results_with_nms_and_limit on each image at n_b; no padding row is ever detected."""
    R, C1, D, k = 300, 21, 256, 3
    n_props = [300, 1, 137, 299]
    n_img = len(n_props)
    w, b = head_params(D, C1, k, 13)
    x = ragged_rows(n_props, R, D, 30, 95, scale=1.0)
    s, _, _, _ = score(x, w, b, n_img, k, n_props)
    t = postproc.test_scores(cuda(s), k)
    boxes = np.concatenate([synth.rois_from_params(synth.proposal_params(R, 256, 110 + i))[:, 1:].numpy()
                            for i in range(n_img)]).reshape(n_img, R, 4)
    res = postproc.results_with_nms_and_limit_batched(t.view(n_img, R, C1 - 1), cuda(boxes), 1e-5, 0.3, 100)
    tn = t.cpu().numpy()
    detected = 0
    for i, n in enumerate(n_props):
        sl = slice(i * R, i * R + n)
        want_t = nms_oracle.test_scores(list(s[2:2 + k, sl]), list(s[2 + k:, sl]))
        np.testing.assert_array_equal(tn[sl].view(np.uint32), want_t.view(np.uint32))
        assert (tn[i * R + n:(i + 1) * R] == 0).all()
        o_boxes, o_inds = nms_oracle.results_with_nms_and_limit(want_t, boxes[i, :n], 1e-5, 0.3, 100)
        _, _, cls_boxes, cls_inds = res[i]
        for j in range(C1 - 1):
            np.testing.assert_array_equal(cls_inds[j + 1], o_inds[j])
            np.testing.assert_array_equal(cls_boxes[j + 1].view(np.uint32), o_boxes[j].view(np.uint32))
            assert (np.asarray(cls_inds[j + 1]) < n).all()
            detected += len(o_inds[j])
    assert detected > 0


# ------------------------------------------------------------------------------------ 8: errors
def test_bad_n_props_raise():
    R, C, D, k, n_img = 200, 20, 256, 3, 2
    w, b = (cuda(a) for a in head_params(D, C + 1, k, 1))
    x = cuda(np.random.RandomState(0).randn(n_img * R, D).astype(np.float32))
    fwd = lambda n: heads.ScoreHeadsFunction.apply(x, w, b, n_img, k, n)
    for bad, exc in (([200], ValueError), ([200, 0], ValueError), ([201, 5], ValueError), ([2.0, 5.0], TypeError),
                     (torch.tensor([200, 5], dtype=torch.int64, device=DEV), TypeError),
                     (torch.tensor([200, 5, 7], dtype=torch.int32, device=DEV), ValueError),
                     (torch.tensor([200, 5], dtype=torch.float32), TypeError),
                     (torch.tensor([200, 5], dtype=torch.int32, device="meta"), ValueError)):
        with pytest.raises(exc):
            fwd(bad)
    s = fwd([200, 5]).detach()
    s4 = s.view(2 + 2 * k, n_img, R, C + 1)
    maps = torch.zeros(n_img, R, R, dtype=torch.float16, device=DEV)
    labels = torch.ones(n_img, C, device=DEV)
    with pytest.raises(ValueError):
        heads.mine_and_assign([s4[0]], [s4[1]], labels, maps, maps, [0.25], [0.5], n_props=[5])
    with pytest.raises(TypeError):
        heads.mine_and_assign([s4[0]], [s4[1]], labels, maps, maps, [0.25], [0.5],
                              n_props=torch.tensor([5, 5], dtype=torch.int16, device=DEV))
    mat = torch.zeros(n_img, R, C + 1, device=DEV)
    with pytest.raises(ValueError):
        heads.PCL_loss(s[0], mat, n_img=n_img, n_props=[5, 201])
