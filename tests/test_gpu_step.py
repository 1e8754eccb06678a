"""CIMHeadStep (the fused per-batch call bench.py times) end to end against the oracle: every result buffer of
one step -- RoIAlign fwd/bwd, maps, scores, pseudo labels, losses, head gradients -- at a small size."""
import numpy as np
import pytest
import torch

from cim_b200 import heads, mask_ops, synth
from cim_b200.step import CIMHeadStep
from oracle import heads_oracle, loss_oracle, mask_oracle, roi_oracle
from conftest import assert_f16_bits_equal, assert_close_elementwise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def rel(got, want):
    """max-norm error, after an element-wise check: 2e-5 relative + 5e-5 * rms -- the oracle chain is fed the GPU's
    scores, so the head gradients carry the rounding of three stages (losses, activation backward, a 384-term fp32
    dot product per element; measured worst case 2.4e-5 * rms)."""
    assert_close_elementwise(got, want, rtol=2e-5, atol_rms=5e-5)
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-3))


@pytest.mark.parametrize("anti", [True, False])
def test_step_matches_oracle_stage_by_stage(anti):
    n_img, R, C, k, D = 2, 192, 20, 3, 256
    size, Cf = 128, 64
    H = W = size // 16
    gen = torch.Generator().manual_seed(5)
    feat = torch.randn(n_img, Cf, H, W, generator=gen)
    grad_out = torch.randn(n_img * R, Cf, 7, 7, generator=gen)
    seg_x = torch.randn(n_img * R, D, generator=gen) * 3
    rois, masks, labels = [], [], []
    for b in range(n_img):
        params = synth.proposal_params(R, size, 40 + b)
        rois.append(synth.rois_from_params(params, b))
        masks.append(synth.rasterize(params))
        labels.append(synth.image_labels(C, 2, 40 + b))
    rois, labels = torch.cat(rois), torch.cat(labels)
    packed = torch.stack([mask_ops.mask_pack(m.to(DEV)) for m in masks])
    torch.manual_seed(1)
    model = heads.cls_iou_model(D, C + 1, k).to(DEV)
    weight, bias = (t.detach().contiguous() for t in model._stacked())
    step = CIMHeadStep(n_img, R, C, Cf, H, W, 1.0 / 16, packed.shape[-1], feat_dim=D, anti_noise_sampling=anti,
                       device=DEV, mask_kb_per_row=size // 16 if mask_ops.tiled_ok(size, size) else 0, head_grads=True)
    mat = torch.stack([synth.cluster_mat(R, C, np.nonzero(labels[b].numpy())[0], 4, 40 + b) for b in range(n_img)])
    np.random.seed(3)
    step.run(feat.to(DEV), rois.to(DEV), grad_out.to(DEV), packed, seg_x.to(DEV), weight, bias, labels.to(DEV),
             labels.numpy(), mat=mat.to(DEV))
    torch.cuda.synchronize()

    want = roi_oracle.roi_align_fwd(feat.numpy(), rois.numpy(), 7, 7, 1.0 / 16, 0, True)
    assert rel(step.roi_out.cpu().numpy(), want) < 1e-5
    want = roi_oracle.roi_align_bwd(grad_out.numpy(), rois.numpy(), feat.shape, 1.0 / 16, 0, True)
    assert rel(step.grad_feat.cpu().numpy(), want) < 1e-5

    maps = [mask_oracle.mask_overlap_maps(m.numpy()) for m in masks]
    for b in range(n_img):
        assert_f16_bits_equal(step.iou[b].cpu().numpy().view(np.uint16), maps[b][0].view(np.uint16))
        assert_f16_bits_equal(step.asy[b].cpu().numpy().view(np.uint16), maps[b][1].view(np.uint16))

    w_np, b_np = weight.cpu().numpy(), bias.cpu().numpy()
    scores = step.scores.cpu().numpy()
    for b in range(n_img):
        o = heads_oracle.score_heads(seg_x[b * R:(b + 1) * R].numpy(), list(w_np), list(b_np))
        np.testing.assert_allclose(scores[:, b * R:(b + 1) * R], np.stack([o[0], o[1]] + o[2] + o[3]), rtol=1e-5,
                                   atol=1e-7)

    # mining + assignment: the oracle consumes the GPU scores (bit-exact decisions need identical inputs) and the
    # same numpy stream in the reference's order (image, layer)
    s4 = scores.reshape(2 + 2 * k, n_img, R, C + 1)
    cls_l, det_l = [s4[0], s4[2], s4[3]], [s4[1], s4[5], s4[6]]
    np.random.seed(3)
    pl = np.zeros((k, n_img, R, C + 1), np.float32)
    pi = np.zeros((k, n_img, R), np.float16)
    lw = np.zeros((k, n_img, R), np.float32)
    valid = np.zeros((k, n_img), np.uint8)
    for b in range(n_img):
        for l in range(k):
            o = heads_oracle.cim_layer_forward(cls_l[l][b], det_l[l][b], labels[b:b + 1].numpy(), maps[b][0], maps[b][1],
                                               0.1, 0.25 + 0.1 * l, 0.5 + 0.1 * l, 0.85, anti)
            if o[0] is None:
                continue
            valid[l, b], pl[l, b], pi[l, b], lw[l, b] = 1, o[0], o[1], o[2]
    np.testing.assert_array_equal(step.valid.cpu().numpy(), valid)
    assert valid.any()
    for l in range(k):
        for b in range(n_img):
            if valid[l, b]:
                np.testing.assert_array_equal(step.pseudo_labels[l, b].cpu().numpy(), pl[l, b])
                assert_f16_bits_equal(step.pseudo_iou[l, b].cpu().numpy().view(np.uint16), pi[l, b].view(np.uint16))
                np.testing.assert_array_equal(step.loss_weights[l, b].cpu().numpy(), lw[l, b])

    # losses + head gradients (batch loss = mean over the images)
    o_loss, o_grad = loss_oracle.head_losses(scores, pl, pi, lw, valid, labels.numpy(), k, grad_scale=1.0 / n_img)
    o_pcl, g_pcl = loss_oracle.pcl_losses(scores[0], mat.numpy(), grad_scale=1.0 / n_img)      # model_builder.py:203
    o_grad[0] += g_pcl
    np.testing.assert_allclose(step.pcl_loss.cpu().numpy(), o_pcl, rtol=2e-5)
    got_loss = step.losses.cpu().numpy()
    np.testing.assert_array_equal(np.isnan(got_loss), np.isnan(o_loss))
    np.testing.assert_allclose(np.nan_to_num(got_loss), np.nan_to_num(o_loss), rtol=2e-5, atol=1e-7)
    fin = np.isfinite(o_grad)
    if fin.all():
        assert rel(step.grad_scores.cpu().numpy(), o_grad) < 1e-5
        gx = np.zeros((n_img * R, D), np.float64)
        gw = np.zeros(w_np.shape, np.float64)
        gb = np.zeros(b_np.shape, np.float64)
        for b in range(n_img):
            sl = slice(b * R, (b + 1) * R)
            ox, ow, ob = heads_oracle.score_heads_bwd(seg_x[sl].numpy(), list(w_np), list(b_np), list(o_grad[:, sl]))
            gx[sl] = ox
            gw += np.stack(ow)
            gb += np.stack(ob)
        assert rel(step.grad_seg_x.cpu().numpy(), gx) < 2e-5
        assert rel(step.grad_weight.cpu().numpy(), gw) < 2e-5
        assert rel(step.grad_bias.cpu().numpy(), gb) < 2e-5


def _small_problem(seed=11):
    n_img, R, C, k, D = 2, 160, 20, 3, 256
    size, Cf = 128, 32
    H = W = size // 16
    gen = torch.Generator().manual_seed(seed)
    feat = torch.randn(n_img, Cf, H, W, generator=gen)
    grad_out = torch.randn(n_img * R, Cf, 7, 7, generator=gen)
    seg_x = torch.randn(n_img * R, D, generator=gen) * 3
    rois, masks, labels = [], [], []
    for b in range(n_img):
        params = synth.proposal_params(R, size, seed + b)
        rois.append(synth.rois_from_params(params, b))
        masks.append(synth.rasterize(params))
        labels.append(synth.image_labels(C, 2, seed + b))
    torch.manual_seed(1)
    model = heads.cls_iou_model(D, C + 1, k).to(DEV)
    weight, bias = (t.detach().contiguous() for t in model._stacked())
    packed = torch.stack([mask_ops.mask_pack(m.to(DEV)) for m in masks])
    return dict(n_img=n_img, R=R, C=C, D=D, Cf=Cf, H=H, W=W, size=size, feat=feat.to(DEV), grad_out=grad_out.to(DEV),
                seg_x=seg_x.to(DEV), rois=torch.cat(rois), labels=torch.cat(labels), packed=packed, weight=weight,
                bias=bias, masks=masks)


def test_graph_order_and_overlapped_order_give_identical_results():
    """order="graph" (the model's dependency order, model_builder.py:136-204) and order="overlapped" (round 1's:
    the sampling hop hidden behind the RoIAlign forward) run the same kernels on the same data: every output is
    bit-identical, and both leave numpy's global RNG in the same state."""
    pr = _small_problem(21)
    kb = pr["size"] // 16 if mask_ops.tiled_ok(pr["size"], pr["size"]) else 0
    outs, states = [], []
    mat = torch.stack([synth.cluster_mat(pr["R"], pr["C"], np.nonzero(pr["labels"][b].numpy())[0], 4, 5 + b)
                       for b in range(pr["n_img"])]).to(DEV)
    for order in ("graph", "overlapped"):
        step = CIMHeadStep(pr["n_img"], pr["R"], pr["C"], pr["Cf"], pr["H"], pr["W"], 1.0 / 16, pr["packed"].shape[-1],
                           feat_dim=pr["D"], device=DEV, mask_kb_per_row=kb, head_grads=True, order=order)
        np.random.seed(3)
        for _ in range(2):
            step.run(pr["feat"], pr["rois"].to(DEV), pr["grad_out"], pr["packed"], pr["seg_x"], pr["weight"],
                     pr["bias"], pr["labels"].to(DEV), mat=mat)
        torch.cuda.synchronize()
        states.append(np.random.get_state()[1].copy())
        outs.append([t.clone() for t in (step.roi_out, step.grad_feat, step.iou.view(torch.int16),
                                         step.asy.view(torch.int16), step.scores, step.pseudo_labels,
                                         step.pseudo_iou.view(torch.int16), step.loss_weights, step.valid, step.losses,
                                         step.grad_seg_x, step.grad_weight, step.grad_bias, step.gt_keep)])
        assert int(step.gt_count.sum()) > 0
    assert np.array_equal(states[0], states[1])
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("lag", [False, True])
def test_run_host_equals_run_and_lagged_results_arrive_one_call_later(lag):
    """run_host() (host rois / labels / packed masks, results read back) gives what run() gives on the same inputs;
    with lag_results the host copy of step i's losses appears during call i + 1 (or flush_results())."""
    pr = _small_problem()
    kb = pr["size"] // 16 if mask_ops.tiled_ok(pr["size"], pr["size"]) else 0
    mk = lambda: CIMHeadStep(pr["n_img"], pr["R"], pr["C"], pr["Cf"], pr["H"], pr["W"], 1.0 / 16, pr["packed"].shape[-1],
                             feat_dim=pr["D"], device=DEV, mask_kb_per_row=kb, head_grads=True)
    ref = mk()
    want = []
    np.random.seed(3)
    for i in range(3):
        ref.run(pr["feat"], pr["rois"].to(DEV), pr["grad_out"], pr["packed"], pr["seg_x"], pr["weight"], pr["bias"],
                pr["labels"].to(DEV), pr["labels"].numpy())
        torch.cuda.synchronize()
        want.append((ref.losses.cpu().numpy().copy(), ref.valid.cpu().numpy().copy()))
    step = mk()
    step.alloc_host_io()
    step.hi_rois.copy_(pr["rois"])
    step.hi_labels.copy_(pr["labels"])
    step.hi_masks.copy_(pr["packed"].cpu())
    np.random.seed(3)
    got = []
    for i in range(3):
        step.run_host(pr["feat"], pr["grad_out"], pr["seg_x"], pr["weight"], pr["bias"], lag_results=lag)
        if lag:
            if i == 0:
                assert step.results_host is None            # nothing has been read back yet
            else:
                got.append(step.results_host)
        else:
            got.append(step.results_host)
    if lag:
        got.append(step.flush_results())
    assert len(got) == 3
    for (w_loss, w_valid), g in zip(want, got):
        np.testing.assert_array_equal(g["valid"], w_valid)
        np.testing.assert_array_equal(np.nan_to_num(g["losses"], nan=-7.0), np.nan_to_num(w_loss, nan=-7.0))
    assert torch.equal(step.grad_feat, ref.grad_feat) and torch.equal(step.roi_out, ref.roi_out)


@pytest.mark.parametrize("near_ring_end,slow_host", [(False, False), (True, False), (False, True)])
def test_stream_sampling_equals_the_host_hop(near_ring_end, slow_host):
    """rng="stream" (uniforms read from a device ring the host fills ahead of time, no host sync inside the step,
    cim_anti_noise_stream) against rng="hop" over several back-to-back steps with a foreign np.random draw in the
    middle: same draws, same outputs bit for bit, and numpy's generator in the same state after sync_rng().  The
    second case starts the stream just before the end of the ring (the top-up and the kernel's reads wrap); the third
    lets the GPU finish the mining phase before the host provisions the step's uniforms (a slow host: the step's own
    count copy has landed by then)."""
    pr = _small_problem(23)
    kb = pr["size"] // 16 if mask_ops.tiled_ok(pr["size"], pr["size"]) else 0
    mat = torch.stack([synth.cluster_mat(pr["R"], pr["C"], np.nonzero(pr["labels"][b].numpy())[0], 4, 9 + b)
                       for b in range(pr["n_img"])]).to(DEV)
    res = {}
    for mode in ("hop", "stream"):
        step = CIMHeadStep(pr["n_img"], pr["R"], pr["C"], pr["Cf"], pr["H"], pr["W"], 1.0 / 16, pr["packed"].shape[-1],
                           feat_dim=pr["D"], device=DEV, mask_kb_per_row=kb, head_grads=True, rng=mode)
        if mode == "stream" and near_ring_end:
            us = step.ustream
            start = us.ring_len - 7
            us.drawn = us.consumed = us.committed = start
            step.d_cursor.fill_(start)
        np.random.seed(5)
        outs = []
        for i in range(7):
            step.run(pr["feat"], pr["rois"].to(DEV), pr["grad_out"], pr["packed"], pr["seg_x"], pr["weight"],
                     pr["bias"], pr["labels"].to(DEV), mat=mat,
                     mid_hook=torch.cuda.synchronize if slow_host and i % 2 == 0 else None)
            outs.append([t.clone() for t in (step.gt_keep, step.pseudo_labels, step.pseudo_iou.view(torch.int16),
                                             step.loss_weights, step.valid, step.losses, step.grad_weight,
                                             step.gt_count)])
            if i == 3:
                step.sync_rng()
                foreign = np.random.random_sample(4)               # e.g. the sampler's permutation at an epoch boundary
        step.sync_rng()
        torch.cuda.synchronize()
        res[mode] = (outs, foreign, np.random.get_state()[1].copy(), np.random.get_state()[2])
    assert int(res["hop"][0][0][7].sum()) > 0                      # pseudo GTs exist: uniforms were consumed
    assert not all(torch.equal(a[0], b[0]) for a, b in zip(res["hop"][0][:-1], res["hop"][0][1:]))   # draws differ by step
    for a, b in zip(res["hop"][0], res["stream"][0]):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    np.testing.assert_array_equal(res["hop"][1], res["stream"][1])
    assert np.array_equal(res["hop"][2], res["stream"][2]) and res["hop"][3] == res["stream"][3]


@pytest.mark.parametrize("depth", [1, 2])
def test_run_host_with_crops_and_changing_inputs(depth):
    """run_host() fed with bounding-box crops of the proposal masks (the bench's wire format; sparse unpack on the
    device) whose rois / labels / masks CHANGE from call to call.  prefetch_depth = 1: what is in the pinned buffers at
    call t is step t + 1's input (call 0 also serves step 0); prefetch_depth = 2: step t + 2's (call 0 also serves
    steps 0 and 1).  Every step must equal run() on the inputs it was meant to see."""
    probs = [_small_problem(31 + 7 * i) for i in range(3)]
    pr0 = probs[0]
    kb = pr0["size"] // 16 if mask_ops.tiled_ok(pr0["size"], pr0["size"]) else 0
    assert kb, "the crop path of run_host needs the tiled mask layout"
    mk = lambda: CIMHeadStep(pr0["n_img"], pr0["R"], pr0["C"], pr0["Cf"], pr0["H"], pr0["W"], 1.0 / 16,
                             pr0["packed"].shape[-1], feat_dim=pr0["D"], device=DEV, mask_kb_per_row=kb, head_grads=True)
    n_calls = 6
    fed = [probs[t % 3] for t in range(n_calls)]                       # pinned-buffer contents at call t
    seen = [fed[max(0, t - depth)] for t in range(n_calls)]            # what step t must compute on
    ref = mk()
    want = []
    np.random.seed(3)
    for pr in seen:
        ref.run(pr0["feat"], pr["rois"].to(DEV), pr0["grad_out"], pr["packed"], pr0["seg_x"], pr0["weight"], pr0["bias"],
                pr["labels"].to(DEV), pr["labels"].numpy())
        torch.cuda.synchronize()
        want.append((ref.losses.cpu().numpy().copy(), ref.valid.cpu().numpy().copy(), ref.iou.clone(),
                     ref.roi_out.clone()))
    assert not np.array_equal(np.nan_to_num(want[0][0]), np.nan_to_num(want[3][0]))     # the inputs do differ

    def crops_of(pr):
        flat = torch.stack([mask_ops.mask_pack(m.to(DEV), layout="flat").cpu() for m in pr["masks"]])
        return mask_ops.crops_from_packed_host(flat.view(pr["n_img"] * pr["R"], -1), pr["size"], pr["size"])

    crops = [crops_of(pr) for pr in probs]
    step = mk()
    cap = max(int(c.words.numel()) for c in crops) + 64
    step.alloc_host_io(mask_hw=(pr0["size"], pr0["size"]), crop_capacity_words=cap, prefetch_depth=depth)
    np.random.seed(3)
    for t in range(n_calls):
        pr = fed[t]
        step.wait_inputs_consumed()
        step.hi_rois.copy_(pr["rois"])
        step.hi_labels.copy_(pr["labels"])
        step.set_host_crops(crops[t % 3])
        step.run_host(pr0["feat"], pr0["grad_out"], pr0["seg_x"], pr0["weight"], pr0["bias"])
        got = step.results_host
        w_loss, w_valid, w_iou, w_roi = want[t]
        np.testing.assert_array_equal(got["valid"], w_valid)
        np.testing.assert_array_equal(np.nan_to_num(got["losses"], nan=-7.0), np.nan_to_num(w_loss, nan=-7.0))
        assert torch.equal(step.iou.view(torch.int16), w_iou.view(torch.int16)) and torch.equal(step.roi_out, w_roi)


def test_bench_dump_outputs_of_one_step(tmp_path):
    """bench.py --dump-outputs on a real step of its tiny workload: every result it names exists on CIMHeadStep, and
    each file holds that result whole or at bench.dump_indices, in float32."""
    import bench
    cfg = bench.WORKLOADS["tiny"]
    inp = bench.build_inputs(cfg, torch.device(DEV), 1234)
    Cf, H, W, scale = inp["shape"]
    step = CIMHeadStep(cfg["n_img"], cfg["R"], cfg["C"], Cf, H, W, scale, inp["packed"].shape[-1], device=DEV,
                       mask_kb_per_row=inp["kb_per_row"], head_grads=True)
    np.random.seed(3)
    step.run(inp["feat"], inp["rois"], inp["grad_out"], inp["packed"], inp["seg_x"], inp["weight"], inp["bias"],
             inp["labels"], mat=inp["mat"], mask_meta=inp["mask_meta"])
    torch.cuda.synchronize()
    bench.dump_outputs(step, str(tmp_path))
    names = bench.STEP_OUTPUTS + bench.STEP_OUTPUTS_HEAD_GRADS
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(f"{n}.npy" for n in names)
    for name in names:
        got = np.load(tmp_path / f"{name}.npy")
        full = getattr(step, name).float().reshape(-1).cpu().numpy()
        assert got.dtype == np.float32
        np.testing.assert_array_equal(got, full[bench.dump_indices(full.size)] if full.size > bench.DUMP_ELEMS else full)
