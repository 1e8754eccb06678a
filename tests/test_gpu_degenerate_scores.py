"""Mining, sampling, losses and scoring on the inputs a confident head produces: class scores of exactly 0 and 1,
detector scores that underflow to 0, tied scores from duplicated proposals, and scores on the loss clamp bounds.

The kernels have branches that only such inputs reach: the seed sort's tie-break (equal score -> lower index), the
containment argmax's tie-break (lowest row) and its all-zero column (torch.argmax gives row 0), the class merge's
strict '>' (on equal preds the lower class keeps the row), anti-noise sampling over zero weights, and the inclusive
clamp of the losses (torch.clamp passes the gradient at equality).  Every test first asserts that its inputs contain
the cases it targets, so a change to a generator cannot make it pass vacuously.

A present class whose pseudo GTs all weigh 0 makes the reference's np.random.choice raise; the device keeps the
class's first pseudo GT instead (heads._anti_noise_keep documents the divergence).  Where the oracle raises, the
comparison asserts that documented result."""
import ctypes
import itertools
from unittest import mock

import numpy as np
import pytest
import torch

from cim_b200 import _lib, heads, mask_ops, synth
from cim_b200.step import CIMHeadStep
from oracle import heads_oracle, loss_oracle, mask_oracle
from conftest import assert_f16_bits_equal, assert_close_elementwise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F16 = np.float16
CON = 0.85
LO32, HI32 = np.float32(1e-6), np.float32(1 - 1e-6)
# the loss clamp bounds, one float32 ulp to either side of them, and the ends of [0, 1]
EDGES = np.array([0, np.nextafter(LO32, np.float32(0)), LO32, np.nextafter(LO32, np.float32(1)), 0.5,
                  np.nextafter(HI32, np.float32(0)), HI32, np.nextafter(HI32, np.float32(1)), 1], np.float32)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ------------------------------------------------------------------------------------------------ generators
def exact_logit_inputs(g, M, D, nh, C1, logit_std, x_max):
    """x [M, D], w [nh, C1, D], b [nh, C1] whose logits x @ w^T + b every summation order computes exactly, in fp32
    FFMA and in 3xTF32 alike: x integers in [-x_max, x_max], w and b multiples of 1/64 below 1024/64 (exact in TF32),
    so every partial sum is a multiple of 1/64 below 2^18.  At logit std 40-100 the ordinary fp32 rounding of a logit
    (its ulp is ~1e-5) moves a softmax output by more than 1e-5 relative; with exact logits the float64 oracle sees
    the kernel's logits, and the comparison at 1e-5 tests the activations themselves."""
    assert D * x_max * 1023 / 64 < 2 ** 18
    x = torch.randint(-x_max, x_max + 1, (M, D), generator=g).float()
    ex2 = sum(v * v for v in range(-x_max, x_max + 1)) / (2 * x_max + 1)
    w = (torch.randn(nh, C1, D, generator=g) * (64 * logit_std / (D * ex2) ** 0.5)).round().clamp(-1023, 1023) / 64
    b = (torch.randn(nh, C1, generator=g) * 64).round() / 64
    return x, w, b


def duplicate_pairs(rs, R, n_dup):
    """(dst, src): rows dst become copies of rows src -- the same proposal listed twice."""
    src = rs.choice(R // 2, n_dup, replace=False)
    dst = R // 2 + rs.choice(R - R // 2, n_dup, replace=False)
    return dst, src


def duplicated_maps(R, seed, dst, src):
    """(b) iou / asy maps of synthetic masks with masks[dst] = masks[src]: tied rows and columns."""
    masks = synth.rasterize(synth.proposal_params(R, 512, seed), out_size=128).numpy()
    masks[dst] = masks[src]
    return mask_oracle.mask_overlap_maps(masks)


def saturated_scores(n_img, R, C1, dst, src, seed, logit_std=40.0, D=64):
    """(a) cls / det of a confident head on the GPU: logits of std `logit_std`, so the class softmax gives exact 1.0
    and 0.0 and the detector's softmax over the proposals underflows to 0; duplicated proposals get identical rows."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_img, R, D, generator=g)
    x[:, dst] = x[:, src]
    w = torch.randn(4, C1, D, generator=g) * (logit_std / D ** 0.5)
    b = torch.randn(4, C1, generator=g)
    with torch.no_grad():
        s = heads.ScoreHeadsFunction.apply(x.view(n_img * R, D).to(DEV), w.to(DEV), b.to(DEV), n_img, 1)
    s = s.view(4, n_img, R, C1).cpu().numpy()
    return s[0], s[1]


def quantized_scores(rs, labels, asys, dst, src, layer):
    """(c) cls, det in multiples of 1/16 (det 0 in half the entries), duplicated rows, det 0 in row 0 for every class,
    and per image one of two plantings (alternating over images and layers) on the two lowest present classes c0, c1:
      * det underflowed for both classes: every container set of their seeds is all zero (argmax -> row 0), both
        claim row 0 at preds 0 in CIM mode and rank the same all-zero keys in MIST mode, and all their pseudo GTs
        weigh 0;
      * c0 scores cls 0 wherever its det is non-zero (several pseudo GTs, all of weight 0), and the first row with
        cls 1 of c1 is a seed whose containers all have det 0."""
    n_img, R = len(asys), asys[0].shape[0]
    C1 = labels.shape[1] + 1
    cls = (rs.randint(0, 17, (n_img, R, C1)) / 16).astype(np.float32)
    det = (rs.randint(0, 17, (n_img, R, C1)) / 16 * (rs.rand(n_img, R, C1) < 0.5)).astype(np.float32)
    cls[:, dst], det[:, dst] = cls[:, src], det[:, src]
    det[:, 0] = 0
    for b in range(n_img):
        c0, c1 = np.nonzero(labels[b])[0][:2] + 1
        if (b + layer) % 2 == 0:
            det[b, :, [c0, c1]] = 0
        else:
            cls[b, det[b, :, c0] > 0, c0] = 0
            s = int(np.nonzero(cls[b, :, c1] == 1)[0][0])
            flag = heads_oracle.big_proposal_flag(asys[b], CON)
            det[b, (asys[b][:, s] > F16(CON)) & flag, c1] = 0
    return cls, det


def degenerate_facts(cls, det, labels, iou, asy, cls_thr, using_cim):
    """Counts of the degenerate cases in one (image, layer) of the mining input, from the oracle's own decisions:
    ties among a present class's top keep_count ranking keys, seeds whose containers all have det 0, rows claimed by
    two classes with equal preds, zero-weight pseudo GTs, and present classes whose pseudo GTs all weigh 0."""
    lab = np.asarray(labels).reshape(-1)
    present = np.nonzero(lab)[0]
    c32, d32 = cls[:, 1:], det[:, 1:]
    preds = c32 * d32
    rank = c32 if using_cim else preds
    kc = int(np.ceil(0.1 * cls.shape[0]))
    f = dict(ties=0, zero_containers=0, shared_equal=0, zero_weight=0, zero_groups=0)
    picked = {}
    if using_cim:
        gt_class, gt_weight, flag, dbg = heads_oracle.cim_label(cls, det, lab, iou, asy, 0.1, cls_thr, CON)
    else:
        gt_class, gt_weight = heads_oracle.mist_label(cls * det, lab, iou, 0.1, cls_thr)
    for c in present:
        top = heads_oracle._seed_order(rank[:, c], kc)
        f["ties"] += len(top) - len(np.unique(rank[top, c]))
        if using_cim:
            seeds = dbg[int(c)]["seeds"]
            cont = (asy[:, seeds] > F16(CON)) & flag[:, None]
            f["zero_containers"] += int(np.sum(cont.any(0) & ~(cont & (d32[:, c:c + 1] != 0)).any(0)))
            picked[c] = set(dbg[int(c)]["picked"].tolist())
        else:
            picked[c] = set(top[heads_oracle.greedy_mask_nms(iou[top][:, top], cls_thr)].tolist())
    for a, b in itertools.combinations(present, 2):
        f["shared_equal"] += sum(int(preds[r, a] == preds[r, b]) for r in picked[a] & picked[b])
    sel = gt_class >= 0
    f["zero_weight"] = int((gt_weight[sel] == 0).sum())
    f["zero_groups"] = sum(int((gt_class == c).any() and (gt_weight[gt_class == c] == 0).all()) for c in present)
    return f, gt_class, gt_weight


def _documented_keep(gt_cls, gt_w, labels):
    return heads._anti_noise_keep(gt_cls, gt_w, np.nonzero(np.asarray(labels).reshape(-1))[0]).astype(bool)


def oracle_layer(cls, det, labels, iou, asy, cls_thr, iou_thr, anti, using_cim=True):
    """heads_oracle.cim_layer_forward -> (result, raised).  Where its np.random.choice raises ValueError (a present
    class whose pseudo GTs all weigh 0, as in the reference), the layer is re-run from the same RNG state with the
    device's documented rule for that case (heads._anti_noise_keep)."""
    args = (cls, det, labels, iou, asy, 0.1, cls_thr, iou_thr, CON, anti, using_cim)
    state = np.random.get_state()
    try:
        with np.errstate(invalid="ignore"):
            return heads_oracle.cim_layer_forward(*args), False
    except ValueError:
        np.random.set_state(state)
    with mock.patch.object(heads_oracle, "anti_noise_keep", _documented_keep), np.errstate(invalid="ignore"):
        return heads_oracle.cim_layer_forward(*args), True


def assert_layer_equal(out, l, b, want):
    if want[0] is None:
        assert int(out["valid"][l, b]) == 0
        return
    assert int(out["valid"][l, b]) == 1
    np.testing.assert_array_equal(out["pseudo_labels"][l, b].cpu().numpy(), want[0])
    assert_f16_bits_equal(out["pseudo_iou_labels"][l, b].cpu().numpy().view(np.uint16), want[1].view(np.uint16))
    np.testing.assert_array_equal(out["loss_weights"][l, b].cpu().numpy().view(np.uint32), want[2].view(np.uint32))


def same_rng_state(a, b):
    return a[2] == b[2] and np.array_equal(a[1], b[1])


# ------------------------------------------------------------------------------------------------ mining
MINING_SHAPES = [(4, 333, 20), (2, 2000, 20), (1, 4000, 80)]


@pytest.mark.parametrize("using_cim", [True, False], ids=["cim", "mist"])
@pytest.mark.parametrize("n_img,R,C", MINING_SHAPES)
def test_mining_degenerate_scores_match_oracle(n_img, R, C, using_cim):
    """heads.mine_and_assign on 3 layers: layer 0 from a saturated head (a), layers 1-2 quantized (c), duplicated
    proposals (b) in all.  Against the oracle layer by layer on the same numpy stream: mined sets (rows, classes,
    weights), pseudo labels, fp16 IoU labels, loss weights and valid bit for bit, and the RNG state afterwards.
    CIM ranks seeds by cls; MIST (mode 1) by cls * det, where the quantized products tie too."""
    L = 3
    cls_thr, iou_thr = [0.25, 0.35, 0.45], [0.5, 0.6, 0.7]
    rs = np.random.RandomState(R + C + n_img)
    dst, src = duplicate_pairs(rs, R, R // 10)
    maps = [duplicated_maps(R, 700 + b, dst, src) for b in range(n_img)]
    labels = np.concatenate([synth.image_labels(C, 2 if C == 20 else 4, 700 + b).numpy() for b in range(n_img)])
    sat = saturated_scores(n_img, R, C + 1, dst, src, R + C)
    quant = [quantized_scores(rs, labels, [m[1] for m in maps], dst, src, l) for l in range(1, L)]
    cls_l, det_l = [sat[0]] + [q[0] for q in quant], [sat[1]] + [q[1] for q in quant]
    assert (sat[0] == 1).any() and (sat[0] == 0).any() and (sat[1] == 0).any()

    facts = {(l, b): degenerate_facts(cls_l[l][b], det_l[l][b], labels[b], maps[b][0], maps[b][1], cls_thr[l],
                                      using_cim) for l in range(L) for b in range(n_img)}
    total = {k: sum(f[0][k] for f in facts.values()) for k in facts[0, 0][0]}
    assert total["ties"] > 0 and total["shared_equal"] > 0 and total["zero_weight"] > 0 and total["zero_groups"] > 0
    if using_cim:
        assert total["zero_containers"] > 0

    np.random.seed(3)
    out = heads.mine_and_assign([cuda(c) for c in cls_l], [cuda(d) for d in det_l], cuda(labels),
                                cuda(np.stack([m[0] for m in maps])), cuda(np.stack([m[1] for m in maps])), cls_thr,
                                iou_thr, using_cim=using_cim)
    state_got = np.random.get_state()
    np.random.seed(3)
    raised = 0
    for b in range(n_img):
        for l in range(L):
            f, gt_class, gt_weight = facts[l, b]
            rows = np.nonzero(gt_class >= 0)[0]
            g = int(out["gt_count"][l, b])
            np.testing.assert_array_equal(out["gt_rows"][l, b, :g].cpu().numpy(), rows)
            np.testing.assert_array_equal(out["gt_class"][l, b, :g].cpu().numpy(), gt_class[rows])
            np.testing.assert_array_equal(out["gt_weight"][l, b, :g].cpu().numpy().view(np.uint32),
                                          gt_weight[rows].view(np.uint32))
            want, r = oracle_layer(cls_l[l][b], det_l[l][b], labels[b], maps[b][0], maps[b][1], cls_thr[l],
                                   iou_thr[l], True, using_cim)
            assert r == (f["zero_groups"] > 0), (b, l)          # the oracle raises exactly on an all-zero class
            raised += r
            assert_layer_equal(out, l, b, want)
    assert raised > 0
    assert same_rng_state(state_got, np.random.get_state())


# ------------------------------------------------------------------------------------------------ sampling
def _sampling_lists(rs, L, n_img, cap, C):
    """Pseudo-GT lists whose class groups hold some zero weights, all-equal weights, a single non-zero weight among
    zeros, or only zeros."""
    labels = np.zeros((n_img, C), np.float32)
    counts = np.zeros((L, n_img), np.int32)
    cls = rs.randint(0, C, (L, n_img, cap)).astype(np.int32)                 # garbage beyond the count
    w = rs.rand(L, n_img, cap).astype(np.float32)
    for b in range(n_img):
        present = np.sort(rs.choice(C, 4, replace=False))
        labels[b, present] = 1
        for l in range(L):
            g = int(rs.choice([1, 5, 40, 200, cap]))
            counts[l, b] = g
            cls[l, b, :g] = rs.choice(present, g)
            for j, c in enumerate(present):
                idx = np.nonzero(cls[l, b, :g] == c)[0]
                kind = (b + l + j) % 4
                if kind == 0:
                    w[l, b, idx[rs.rand(len(idx)) < 0.5]] = 0
                elif kind == 1:
                    w[l, b, idx] = np.float32(0.0625)
                elif kind == 2:
                    w[l, b, idx] = 0
                    if len(idx):
                        w[l, b, idx[rs.randint(len(idx))]] = np.float32(0.3)
                else:
                    w[l, b, idx] = 0
    return labels, counts, cls, w


@pytest.mark.parametrize("cap,n_img,L,C", [(300, 3, 3, 20), (1500, 2, 2, 80)])
def test_anti_noise_kernels_with_zero_and_equal_weights(cap, n_img, L, C):
    """cim_anti_noise (host uniforms) and cim_anti_noise_stream (uniforms from a device ring, read across its end)
    against heads._anti_noise_keep on the same stream, and against np.random.choice for every class group numpy
    accepts; an all-zero group makes choice raise, and both kernels keep that class's first pseudo GT."""
    rs = np.random.RandomState(cap + C)
    labels, counts, cls, w = _sampling_lists(rs, L, n_img, cap, C)
    p = _lib.MineParams()
    p.n_img, p.R, p.C, p.C1, p.n_layers, p.det_cols, p.gt_cap, p.mode, p.keep_count = n_img, cap, C, C + 1, L, C + 1, cap, 0, 8
    d_counts, d_cls, d_w, d_labels = cuda(counts), cuda(cls), cuda(w), cuda(labels)

    # expected: host restatement per (image, layer) list in the reference's order, and np.random.choice per group
    np.random.seed(99)
    want = np.ones((L, n_img, cap), np.uint8)
    kinds = dict(zeros=0, equal=0, single=0, all_zero=0)
    for b in range(n_img):
        for l in range(L):
            g = counts[l, b]
            gc, gw = cls[l, b, :g], w[l, b, :g]
            before = np.random.get_state()
            want[l, b, :g] = heads._anti_noise_keep(gc, gw, np.nonzero(labels[b])[0])
            after = np.random.get_state()
            np.random.set_state(before)
            for c in np.nonzero(labels[b])[0]:
                idx = np.nonzero(gc == c)[0]
                if len(idx) == 0:
                    continue
                wi = gw[idx]
                if wi.sum() == 0:
                    kinds["all_zero"] += len(idx) > 1
                    with pytest.raises(ValueError), np.errstate(invalid="ignore"):
                        np.random.choice(idx, len(idx), replace=True, p=wi / wi.sum())
                    np.random.random_sample(len(idx))
                    assert want[l, b, idx].tolist() == [1] + [0] * (len(idx) - 1)
                    continue
                kinds["zeros"] += bool((wi == 0).any()) and np.count_nonzero(wi) > 1
                kinds["equal"] += len(idx) > 1 and (wi == wi[0]).all()
                kinds["single"] += len(idx) > 1 and np.count_nonzero(wi) == 1
                drawn = np.random.choice(idx, len(idx), replace=True, p=wi / wi.sum())
                keep = np.zeros(len(gc), bool)
                keep[drawn] = True
                assert want[l, b, idx].astype(bool).tolist() == keep[idx].tolist(), (b, l, c)
            assert same_rng_state(after, np.random.get_state())
    state_want = np.random.get_state()
    assert all(v > 0 for v in kinds.values()), kinds
    total = int(counts.sum())

    keep = torch.full((L, n_img, cap), 7, dtype=torch.uint8, device=DEV)
    np.random.seed(99)
    heads.anti_noise_device(p, d_labels, d_counts, d_cls, d_w, keep)
    assert same_rng_state(np.random.get_state(), state_want)
    np.testing.assert_array_equal(keep.cpu().numpy(), want)

    # stream mode: the step's first double sits 5 slots before the end of the ring
    np.random.seed(99)
    u = np.random.random_sample(total)
    ring_len = L * n_img * cap + 64
    start = ring_len - 5
    ring = np.full(ring_len, 2.0)                                # 2.0 is never a uniform: a wrong read shows
    ring[(start + np.arange(total)) % ring_len] = u
    cursor = torch.tensor([start, -1], dtype=torch.int64, device=DEV)
    keep2 = torch.full((L, n_img, cap), 7, dtype=torch.uint8, device=DEV)
    d_ring = cuda(ring)
    _lib.check(_lib.lib().cim_anti_noise_stream(ctypes.byref(p), _lib.ptr(d_labels), _lib.ptr(d_counts), _lib.ptr(d_cls),
                                        _lib.ptr(d_w), _lib.ptr(d_ring), ring_len, _lib.ptr(cursor[0:]),
                                        _lib.ptr(cursor[1:]), _lib.ptr(keep2), _lib.stream_ptr(torch.device(DEV))),
               "cim_anti_noise_stream")
    np.testing.assert_array_equal(keep2.cpu().numpy(), want)
    assert int(cursor[1]) == start + total


# ------------------------------------------------------------------------------------------------ losses
def _edge_scores(rs, shape):
    return EDGES[rs.randint(0, len(EDGES), shape)]


def _check_clamped_grad(got, want, vals, what):
    """Exactly 0 outside [float32(1e-6), float32(1 - 1e-6)]; on and inside the bounds equal to the oracle."""
    out = (vals < LO32) | (vals > HI32)
    on = (vals == LO32) | (vals == HI32)
    assert (want[out] == 0).all(), what
    assert (got[out] == 0).all(), f"{what}: gradient through a clamped score"
    assert (want[on] != 0).any(), what
    np.testing.assert_array_equal(got[on] != 0, want[on] != 0, err_msg=f"{what}: gradient at the clamp bounds")
    assert_close_elementwise(got, want, rtol=1e-5, atol_rms=1e-6, what=what)


@pytest.mark.parametrize("n_img,R,C", [(2, 300, 20), (1, 2000, 80)])
def test_head_losses_at_the_clamp_bounds(n_img, R, C):
    """cim_head_losses with every score of every head drawn from EDGES (0, the clamp bounds and their float32
    neighbours, 0.5, 1) against the float64 autograd oracle.  The MIL heads enter only through column sums, so
    columns 0..5 of each image hold one non-zero product cls * det = 1 * e for e in the bounds and their neighbours
    (the sums then sit exactly on them)."""
    rs = np.random.RandomState(R + C)
    k, c1 = 3, C + 1
    scores = _edge_scores(rs, (2 + 2 * k, n_img * R, c1))
    mil = scores[:2].reshape(2, n_img, R, c1)
    sums = EDGES[[1, 2, 3, 5, 6, 7]]
    for b in range(n_img):
        mil[:, b, :, :6] = 0
        rows = rs.choice(R, 6, replace=False)
        mil[0, b, rows, np.arange(6)] = 1
        mil[1, b, rows, np.arange(6)] = sums
    scores[:2] = mil.reshape(2, n_img * R, c1)
    labels = np.zeros((n_img, C), np.float32)
    pl = np.zeros((k, n_img, R, c1), np.float32)
    for b in range(n_img):
        present = rs.choice(C, 3, replace=False)
        labels[b, present] = 1
        for l in range(k):
            kind = rs.rand(R)
            fg = kind < 0.4
            pl[l, b, fg, 1 + rs.choice(present, fg.sum())] = 1
            pl[l, b, (kind >= 0.4) & (kind < 0.8), 0] = 1
    pi = (rs.rand(k, n_img, R) > 0.5).astype(np.float16)
    lw = rs.rand(k, n_img, R).astype(np.float32)
    valid = np.ones((k, n_img), np.uint8)
    for v in EDGES:                                                       # every value in every head
        assert ((scores == v).reshape(2 + 2 * k, -1).any(1)).all(), v

    s = cuda(scores).requires_grad_(True)
    assigned = dict(pseudo_labels=cuda(pl), pseudo_iou_labels=cuda(pi), loss_weights=cuda(lw), valid=cuda(valid))
    out = heads.head_losses(s, assigned, cuda(labels), k)
    out["total"].sum().backward()
    got = s.grad.cpu().numpy()
    o_loss, o_grad = loss_oracle.head_losses(scores, pl, pi, lw, valid, labels, k)
    assert_close_elementwise(out["losses"].cpu().numpy(), o_loss, rtol=1e-5, atol_rms=1e-7, what="losses")
    for h in range(2, 2 + 2 * k):
        _check_clamped_grad(got[h], o_grad[h], scores[h], f"head {h}")
    # MIL heads: the gradient of a column is 0 when its sum lies outside the clamp, and flows when it sits on a bound
    g_mil = got[:2].reshape(2, n_img, R, c1)
    for b in range(n_img):
        for j, e in enumerate(sums):
            flows = np.abs(g_mil[:, b, :, j]).max() > 0
            assert flows == bool(LO32 <= e <= HI32), (b, j, e)
    assert_close_elementwise(got[:2], o_grad[:2], rtol=1e-5, atol_rms=1e-6, what="MIL heads")


def test_pcl_loss_at_the_clamp_bounds():
    """cim_pcl_loss with predict_cls drawn from EDGES: one-row foreground clusters (their mean is the row itself, so
    it lands exactly on the bounds), larger foreground clusters and a background cluster, against the float64
    autograd oracle."""
    rs = np.random.RandomState(12)
    n_img, R, c1 = 2, 600, 21
    p = _edge_scores(rs, (n_img * R, c1))
    mat = np.zeros((n_img, R, c1), np.float32)
    for b in range(n_img):
        order = rs.permutation(R)
        k = 1
        for j in range(60):                                               # 60 one-row clusters
            mat[b, order[j], 1 + rs.randint(c1 - 1)] = k
            k += 1
        for j in range(10):                                               # 10 clusters of 20 rows
            rows = order[60 + 20 * j:80 + 20 * j]
            mat[b, rows, 1 + rs.randint(c1 - 1)] = k
            k += 1
        mat[b, order[260:500], 0] = k                                     # background cluster
    pt = cuda(p).requires_grad_(True)
    loss = heads.PCL_loss(pt, cuda(mat), None, n_img=n_img)
    loss.sum().backward()
    o_loss, o_grad = loss_oracle.pcl_losses(p, mat)
    assert_close_elementwise(loss.detach().cpu().numpy(), o_loss, rtol=1e-5, atol_rms=0, what="loss")
    got = pt.grad.cpu().numpy()
    one_row = np.zeros(n_img * R, bool)
    bg = np.zeros(n_img * R, bool)
    for b in range(n_img):
        ids = mat[b].max(1)
        counts = np.bincount(ids.astype(np.int64))
        one_row[b * R:(b + 1) * R] = (ids > 0) & (counts[ids.astype(np.int64)] == 1) & (mat[b, :, 0] == 0)
        bg[b * R:(b + 1) * R] = mat[b, :, 0] != 0
    for sel, what in ((one_row, "one-row clusters"), (bg, "background cluster")):
        _check_clamped_grad(got[sel], o_grad[sel], p[sel], what)
    assert_close_elementwise(got, o_grad, rtol=1e-5, atol_rms=1e-6, what="PCL gradient")


# ------------------------------------------------------------------------------------------------ scoring
@pytest.mark.parametrize("C1,logit_std", [(21, 40.0), (81, 100.0)])
def test_scoring_with_large_logits(C1, logit_std):
    """cim_score_heads forward and backward at cfg2's shape (8 x 2000 proposals, D = 4096) with logits of std 40-100,
    on the 3xTF32 tcgen05 path and on the FFMA path, against the float64 oracle element by element: exact 0 and 1
    from the softmaxes, detector columns whose entries underflow, no NaN or inf."""
    n_img, R, D, K, nh = 8, 2000, 4096, 3, 8
    M = n_img * R
    g = torch.Generator().manual_seed(C1)
    x, w, b = exact_logit_inputs(g, M, D, nh, C1, logit_std, 2)
    gr = torch.randn(nh, M, C1, generator=g)
    x_np, w_np, b_np, gr_np = x.numpy(), list(w.numpy()), list(b.numpy()), gr.numpy()
    want_s = np.zeros((nh, M, C1), np.float32)
    want_x = np.zeros((M, D), np.float32)
    want_w, want_b = np.zeros((nh, C1, D)), np.zeros((nh, C1))
    for i in range(n_img):
        sl = slice(i * R, (i + 1) * R)
        o = heads_oracle.score_heads(x_np[sl], w_np, b_np)
        want_s[:, sl] = np.stack([o[0], o[1]] + o[2] + o[3])
        ox, ow, ob = heads_oracle.score_heads_bwd(x_np[sl], w_np, b_np, list(gr_np[:, sl]))
        want_x[sl] = ox
        want_w += np.stack(ow)
        want_b += np.stack(ob)
    assert (want_s[0] == 1).any() and (want_s[0] == 0).any() and (want_s[1] == 0).mean() > 0.5

    L = _lib.lib()
    st = _lib.stream_ptr(torch.device(DEV))
    dx, dw, db, dg = x.to(DEV), w.to(DEV), b.to(DEV), gr.to(DEV)
    for flags in (0, _lib.DBG_SCORE_FFMA):
        with _lib.debug_flags(flags):
            scores = torch.full((nh, M, C1), float("nan"), device=DEV)
            ws = torch.empty(L.cim_score_heads_workspace_bytes(n_img, R, D, C1, K), dtype=torch.uint8, device=DEV)
            _lib.check(L.cim_score_heads(_lib.ptr(dx), _lib.ptr(dw), _lib.ptr(db), _lib.ptr(scores), n_img, R, D, C1,
                                         K, _lib.ptr(ws), ws.numel(), st), "cim_score_heads")
            gx, gw = torch.empty(M, D, device=DEV), torch.empty(nh, C1, D, device=DEV)
            gb = torch.empty(nh, C1, device=DEV)
            ws2 = torch.empty(L.cim_score_heads_bwd_workspace_bytes(n_img, R, D, C1, K), dtype=torch.uint8, device=DEV)
            _lib.check(L.cim_score_heads_bwd(_lib.ptr(dx), _lib.ptr(dw), _lib.ptr(scores), _lib.ptr(dg), _lib.ptr(gx),
                                             _lib.ptr(gw), _lib.ptr(gb), n_img, R, D, C1, K, _lib.ptr(ws2), ws2.numel(),
                                             st), "cim_score_heads_bwd")
            torch.cuda.synchronize()
        what = "ffma" if flags else "tcgen05"
        s = scores.cpu().numpy()
        assert np.isfinite(s).all(), what
        assert_close_elementwise(s, want_s, what=f"{what} scores")
        det_sums = s[1].reshape(n_img, R, C1).astype(np.float64).sum(1)
        assert np.abs(det_sums - 1).max() <= 1e-5, what
        for got, want, name in ((gx, want_x, "grad_x"), (gw, want_w, "grad_w"), (gb, want_b, "grad_b")):
            got = got.cpu().numpy()
            assert np.isfinite(got).all(), f"{what} {name}"
            assert_close_elementwise(got, want, what=f"{what} {name}")


# ------------------------------------------------------------------------------------------------ whole step
def act_bwd_rounding(y, g, n_img, k):
    """Forward-error bound of the float32 activation backward cim_score_heads_bwd evaluates on scores y [2+2K, M, C1]
    and their gradient g: dz = y * (g - dot), dot = sum_j g_j y_j over the C1 classes in sequence (row softmaxes) or
    over the R proposals of an image in a tree (detector), and dz = g * y * (1 - y) (sigmoid).  Rounding moves dz by
    at most gamma * y * (|g| + sum_j |g_j y_j|), gamma = (terms + 2) * 2^-24.  On saturated scores the loss gradient of
    an output near 1 is ~1 / (1 - y) while dz stays O(1), so float32 loses the low digits of dz there whatever the
    implementation (torch's float32 autograd included); elsewhere the bound is far below the 2e-5 tolerance."""
    u = 2.0 ** -24
    y, g = y.astype(np.float64), g.astype(np.float64)
    nh, M, C1 = y.shape
    R = M // n_img
    a = np.abs(g * y)
    e = np.empty_like(y)
    rows = [0] + list(range(2, 2 + k))
    e[rows] = (C1 + 2) * u * y[rows] * (np.abs(g[rows]) + a[rows].sum(-1, keepdims=True))
    yd, gd = y[1].reshape(n_img, R, C1), g[1].reshape(n_img, R, C1)
    e[1] = ((np.ceil(np.log2(R)) + 3) * u * yd * (np.abs(gd) + a[1].reshape(n_img, R, C1).sum(1, keepdims=True))
            ).reshape(M, C1)
    e[2 + k:] = 4 * u * np.abs(g[2 + k:] * y[2 + k:] * (1 - y[2 + k:]))
    return e


@pytest.mark.parametrize("anti,rng", [(False, "hop"), (True, "hop"), (True, "stream")])
def test_saturated_step_matches_oracle(anti, rng):
    """CIMHeadStep with head weights large enough that its own scores saturate (logit std 60: exact 0 and 1 in the
    class softmaxes, underflowed detector entries), duplicated proposals included; every stage against the oracle fed the
    GPU's scores, as in test_gpu_step.test_step_matches_oracle_stage_by_stage."""
    n_img, R, C, k, D = 2, 192, 20, 3, 256
    size, Cf = 128, 64
    H = W = size // 16
    gen = torch.Generator().manual_seed(6)
    feat = torch.randn(n_img, Cf, H, W, generator=gen)
    grad_out = torch.randn(n_img * R, Cf, 7, 7, generator=gen)
    seg_x, weight, bias = exact_logit_inputs(gen, n_img * R, D, 2 + 2 * k, C + 1, 60.0, 4)
    rs = np.random.RandomState(6)
    dst, src = duplicate_pairs(rs, R, 20)
    rois, masks, labels = [], [], []
    for b in range(n_img):
        params = synth.proposal_params(R, size, 60 + b)
        r, m = synth.rois_from_params(params, b), synth.rasterize(params)
        r[dst], m[dst] = r[src], m[src]
        rois.append(r)
        masks.append(m)
        labels.append(synth.image_labels(C, 2, 60 + b))
        seg_x[b * R + dst] = seg_x[b * R + src]
    rois, labels = torch.cat(rois), torch.cat(labels)
    packed = torch.stack([mask_ops.mask_pack(m.to(DEV)) for m in masks])
    weight, bias = weight.to(DEV), bias.to(DEV)
    step = CIMHeadStep(n_img, R, C, Cf, H, W, 1.0 / 16, packed.shape[-1], feat_dim=D, anti_noise_sampling=anti,
                       device=DEV, mask_kb_per_row=size // 16 if mask_ops.tiled_ok(size, size) else 0, head_grads=True,
                       rng=rng)
    mat = torch.stack([synth.cluster_mat(R, C, np.nonzero(labels[b].numpy())[0], 4, 60 + b) for b in range(n_img)])
    np.random.seed(3)
    step.run(feat.to(DEV), rois.to(DEV), grad_out.to(DEV), packed, seg_x.to(DEV), weight, bias, labels.to(DEV),
             mat=mat.to(DEV))
    step.sync_rng()
    torch.cuda.synchronize()
    state_got = np.random.get_state()

    maps = [mask_oracle.mask_overlap_maps(m.numpy()) for m in masks]
    for b in range(n_img):
        assert_f16_bits_equal(step.iou[b].cpu().numpy().view(np.uint16), maps[b][0].view(np.uint16))
        assert_f16_bits_equal(step.asy[b].cpu().numpy().view(np.uint16), maps[b][1].view(np.uint16))
    w_np, b_np = weight.cpu().numpy(), bias.cpu().numpy()
    scores = step.scores.cpu().numpy()
    for b in range(n_img):
        o = heads_oracle.score_heads(seg_x[b * R:(b + 1) * R].numpy(), list(w_np), list(b_np))
        assert_close_elementwise(scores[:, b * R:(b + 1) * R], np.stack([o[0], o[1]] + o[2] + o[3]), what="scores")
    assert (scores[0] == 1).any() and (scores[0] == 0).any() and (scores[1] == 0).mean() > 0.5

    s4 = scores.reshape(2 + 2 * k, n_img, R, C + 1)
    cls_l, det_l = [s4[0], s4[2], s4[3]], [s4[1], s4[5], s4[6]]
    pl = np.zeros((k, n_img, R, C + 1), np.float32)
    pi = np.zeros((k, n_img, R), np.float16)
    lw = np.zeros((k, n_img, R), np.float32)
    valid = np.zeros((k, n_img), np.uint8)
    zero_weight = 0
    np.random.seed(3)
    for b in range(n_img):
        for l in range(k):
            f, gt_class, gt_weight = degenerate_facts(cls_l[l][b], det_l[l][b], labels[b].numpy(), maps[b][0],
                                                      maps[b][1], 0.25 + 0.1 * l, True)
            zero_weight += f["zero_weight"]
            g = int(step.gt_count[l, b])
            rows = np.nonzero(gt_class >= 0)[0]
            np.testing.assert_array_equal(step.gt_rows[l, b, :g].cpu().numpy(), rows)
            np.testing.assert_array_equal(step.gt_weight[l, b, :g].cpu().numpy().view(np.uint32),
                                          gt_weight[rows].view(np.uint32))
            o, raised = oracle_layer(cls_l[l][b], det_l[l][b], labels[b:b + 1].numpy(), maps[b][0], maps[b][1],
                                     0.25 + 0.1 * l, 0.5 + 0.1 * l, anti)
            assert raised == (anti and f["zero_groups"] > 0)
            if o[0] is None:
                continue
            valid[l, b], pl[l, b], pi[l, b], lw[l, b] = 1, o[0], o[1], o[2]
    assert zero_weight > 0
    assert same_rng_state(state_got, np.random.get_state())
    np.testing.assert_array_equal(step.valid.cpu().numpy(), valid)
    assert valid.any()
    for l in range(k):
        for b in range(n_img):
            if valid[l, b]:
                np.testing.assert_array_equal(step.pseudo_labels[l, b].cpu().numpy(), pl[l, b])
                assert_f16_bits_equal(step.pseudo_iou[l, b].cpu().numpy().view(np.uint16), pi[l, b].view(np.uint16))
                np.testing.assert_array_equal(step.loss_weights[l, b].cpu().numpy(), lw[l, b])

    o_loss, o_grad = loss_oracle.head_losses(scores, pl, pi, lw, valid, labels.numpy(), k, grad_scale=1.0 / n_img)
    o_pcl, g_pcl = loss_oracle.pcl_losses(scores[0], mat.numpy(), grad_scale=1.0 / n_img)
    o_grad[0] += g_pcl
    np.testing.assert_allclose(step.pcl_loss.cpu().numpy(), o_pcl, rtol=2e-5)
    got_loss = step.losses.cpu().numpy()
    np.testing.assert_array_equal(np.isnan(got_loss), np.isnan(o_loss))
    np.testing.assert_allclose(np.nan_to_num(got_loss), np.nan_to_num(o_loss), rtol=2e-5, atol=1e-7)
    assert np.isfinite(o_grad).all()
    assert_close_elementwise(step.grad_scores.cpu().numpy(), o_grad, rtol=2e-5, atol_rms=5e-5, what="grad_scores")
    # scoring backward: the float64 oracle is fed what cim_score_heads_bwd received (the step's scores and
    # grad_scores) and differentiates through the float32 scores as torch's softmax / sigmoid backward do
    gs = step.grad_scores.cpu().numpy()
    e = act_bwd_rounding(scores, gs, n_img, k)
    gx = np.zeros((n_img * R, D), np.float64)
    gw = np.zeros(w_np.shape, np.float64)
    gb = np.zeros(b_np.shape, np.float64)
    for b in range(n_img):
        sl = slice(b * R, (b + 1) * R)
        ox, ow, ob = heads_oracle.score_heads_bwd(seg_x[sl].numpy(), list(w_np), list(b_np), list(gs[:, sl]),
                                                  outputs=list(scores[:, sl]))
        gx[sl] = ox
        gw += np.stack(ow)
        gb += np.stack(ob)
    x_abs, w_abs = np.abs(seg_x.numpy().astype(np.float64)), np.abs(w_np.astype(np.float64))
    e_x = sum(e[h] @ w_abs[h] for h in range(2 + 2 * k))
    e_w = np.stack([e[h].T @ x_abs for h in range(2 + 2 * k)])
    e_b = e.sum(1)
    for got, want, extra, name in ((step.grad_seg_x, gx, e_x, "grad_seg_x"), (step.grad_weight, gw, e_w, "grad_weight"),
                                   (step.grad_bias, gb, e_b, "grad_bias")):
        got = got.cpu().numpy().astype(np.float64)
        rms = float(np.sqrt(np.mean(want * want)))
        err = np.abs(got - want)
        bound = 2e-5 * np.abs(want) + 5e-5 * rms + extra
        assert (err <= bound).all(), f"{name}: {int((err > bound).sum())} elements outside, worst err {err.max():.3e}"
