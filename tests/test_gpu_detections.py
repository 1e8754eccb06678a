"""Batched test-time detections on the device: the TTA score mean (cim_test_scores_tta through
postproc.TestScoreMean) and the per-image detection limit + compaction (cim_box_detections through
postproc.detections_batched / results_with_nms_and_limit_batched), bit-exact against oracle/nms_oracle.py (its
head mean and its restatement of mask_eval_utils.py:57-110, applied pass by pass and image by image).
Each test first asserts that its inputs contain the case it is about."""
import os

import numpy as np
import pytest
import torch

from cim_b200 import postproc, synth
from oracle import nms_oracle
from conftest import GOLDEN

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NPZ = np.load(os.path.join(GOLDEN, "box_nms.npz"))


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return t.cpu().numpy()


def tta_scores(passes):
    """TEST.BBOX_AUG with SCORE_HEUR 'AVG' (core/test.py:149-226): np.mean over the passes of the oracle's test
    scores, in the caller's pass order."""
    return np.mean(np.stack([nms_oracle.test_scores(cls_t, iou_t) for cls_t, iou_t in passes]), axis=0)


def oracle_batched(scores, boxes, score_thresh, nms_thresh, detections_per_im):
    """nms_oracle.results_with_nms_and_limit for each image of scores [B,n,C], boxes [B,n,4]."""
    return [nms_oracle.results_with_nms_and_limit(s, b, score_thresh, nms_thresh, detections_per_im)
            for s, b in zip(scores, boxes)]


def flat(o_boxes, o_inds):
    """The oracle's per-class lists as the device's flat order: class ascending, proposal index ascending."""
    cls = np.concatenate([np.full(len(i), j, np.int32) for j, i in enumerate(o_inds)])
    idx = np.concatenate(o_inds).astype(np.int32)
    dets = np.vstack(o_boxes).astype(np.float32) if o_boxes else np.zeros((0, 5), np.float32)
    return cls, idx, dets[:, 4].copy(), dets[:, :4].copy()


def assert_device_matches(out, oracle, keep_shape):
    """out = detections_batched(...); oracle = per image (cls_boxes, cls_inds) over the C classes."""
    count, cls, idx, score, box, keep = (host(t) for t in out)
    cap = cls.shape[1]
    assert keep.shape == keep_shape
    for b, (o_boxes, o_inds) in enumerate(oracle):
        w_cls, w_idx, w_score, w_box = flat(o_boxes, o_inds)
        assert count[b] == len(w_idx), b
        k = min(len(w_idx), cap)
        np.testing.assert_array_equal(cls[b, :k], w_cls[:k])
        np.testing.assert_array_equal(idx[b, :k], w_idx[:k])
        np.testing.assert_array_equal(score[b, :k].view(np.uint32), w_score[:k].view(np.uint32))
        np.testing.assert_array_equal(box[b, :k].view(np.uint32), w_box[:k].view(np.uint32))
        want_keep = np.zeros(keep_shape[1:], np.uint8)
        want_keep[w_cls, w_idx] = 1
        np.testing.assert_array_equal(keep[b], want_keep)


def assert_host_matches(res, oracle, c):
    for (s, bx, cls_boxes, cls_inds), (o_boxes, o_inds) in zip(res, oracle, strict=True):
        assert len(cls_boxes) == c + 1 and len(cls_boxes[0]) == 0 and len(cls_inds[0]) == 0
        for j in range(c):
            assert cls_inds[j + 1].dtype == np.intp and cls_boxes[j + 1].dtype == np.float32
            np.testing.assert_array_equal(cls_inds[j + 1], o_inds[j])
            np.testing.assert_array_equal(cls_boxes[j + 1].view(np.uint32), o_boxes[j].view(np.uint32))
        want = np.vstack([o_boxes[j] for j in range(c - 1)])                       # :108 leaves the last class out
        np.testing.assert_array_equal(s, want[:, -1])
        np.testing.assert_array_equal(bx, want[:, :-1])


def proposals(n, seed):
    return synth.rois_from_params(synth.proposal_params(n, 512, seed)).numpy()[:, 1:].copy()


def disjoint_boxes(n):
    """Boxes 6 px wide on an 8 px grid: no two overlap, so NMS keeps every candidate."""
    i = np.arange(n)
    x, y = (i % 64) * 8.0, (i // 64) * 8.0
    return np.stack([x, y, x + 5, y + 5], 1).astype(np.float32)


def sparse_scores(rs, n, c, density, levels=256):
    """Scores on a grid of `levels` values (ties within and across classes), `density` of them candidates."""
    s = (rs.randint(1, levels, size=(n, c)) / levels).astype(np.float32)
    s[rs.rand(n, c) >= density] = 0
    return s


# ------------------------------------------------------------------ TTA mean
@pytest.mark.parametrize("T", [1, 2, 10])
def test_tta_mean_bit_exact(T):
    k, m, c1 = 3, 8 * 4000, 81
    rs = np.random.RandomState(100 + T)
    mean = postproc.TestScoreMean(T)
    per_pass = []
    buf = torch.empty(2 + 2 * k, m, c1, device=DEV)                 # one scoring buffer reused by every pass
    for t in range(T):
        mag = np.float32(10.0) ** rs.randint(-3, 3, size=(2 * k, m, c1)).astype(np.float32)
        s = np.zeros((2 + 2 * k, m, c1), np.float32)
        s[2:] = rs.rand(2 * k, m, c1).astype(np.float32) * mag
        buf.copy_(cuda(s))
        with pytest.raises(RuntimeError):
            mean.scores                                               # read before the last pass
        mean.add(buf, k)
        per_pass.append((list(s[2:2 + k]), list(s[2 + k:])))
        if T == 1:
            assert torch.equal(mean.scores, postproc.test_scores(buf, k))
    got = host(mean.scores)
    want = tta_scores(per_pass)
    assert got.shape == (m, c1 - 1)
    if T > 2:                                 # the accumulation rounds: a float64 mean would differ somewhere
        wide = np.mean(np.stack([nms_oracle.test_scores(a, b) for a, b in per_pass]).astype(np.float64), 0)
        assert not np.array_equal(want, wide.astype(np.float32))
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    with pytest.raises(RuntimeError):
        mean.add(buf, k)                                              # a pass beyond n_passes


# ------------------------------------------------------------------ limit + compaction
def test_cfg5_batch_matches_oracle():
    """8 x 4000 proposals x 80 classes: limited images, an image with <= D kept, one with no candidates, a class
    with no candidates."""
    B, n, c, D = 8, 4000, 80, 100
    rs = np.random.RandomState(5)
    boxes = np.stack([proposals(n, 500 + b) for b in range(B)])
    scores = np.stack([sparse_scores(rs, n, c, 0.03, levels=1 << 20) for _ in range(B)])
    scores[0, :, 7] = 0                                               # a class without candidates
    scores[5] = 0                                                     # an image without candidates
    scores[6] = sparse_scores(rs, n, c, 0.0002)                       # an image with <= D kept
    oracle = oracle_batched(scores, boxes, 1e-5, 0.3, D)
    full = oracle_batched(scores[:1], boxes[:1], 1e-5, 0.3, 0)
    kept = [sum(len(i) for i in o[1]) for o in oracle]
    assert len(full[0][1][7]) == 0 and kept[5] == 0 and 0 < kept[6] < D
    assert sum(len(i) for i in full[0][1]) > D and sum(k == D for k in kept) >= 5
    out = postproc.detections_batched(cuda(scores), cuda(boxes), 1e-5, 0.3, D)
    assert_device_matches(out, oracle, (B, c, n))


def test_ties_at_the_limit_across_classes():
    """The D-th score is shared by entries of several classes on both sides of rank D: all of them survive, so
    count > D = cap and the host form needs its second round."""
    n, c, D = 300, 6, 100
    rs = np.random.RandomState(11)
    scores = np.full((n, c), 0.25, np.float32)
    cells = rs.permutation(n * c)
    scores.flat[cells[:90]] = 0.75
    scores.flat[cells[90:120]] = 0.5                                 # ranks 91 .. 120: the 100th is in here
    boxes = disjoint_boxes(n)
    ranked = np.sort(scores.ravel())[::-1]
    assert ranked[D - 2] == ranked[D - 1] == ranked[D] == 0.5 < ranked[89] and len(np.unique(cells[90:120] % c)) > 1
    oracle = oracle_batched(scores[None], boxes[None], 1e-5, 0.3, D)
    assert sum(len(i) for i in oracle[0][1]) == 120
    out = postproc.detections_batched(cuda(scores[None]), cuda(boxes[None]), 1e-5, 0.3, D)
    assert int(out[0][0]) == 120 and out[1].shape[1] == D
    assert_device_matches(out, oracle, (1, c, n))
    res = postproc.results_with_nms_and_limit_batched(cuda(scores[None]), cuda(boxes[None]), 1e-5, 0.3, D)
    assert_host_matches(res, oracle, c)


def test_signed_zero_ties_compare_as_floats():
    """thresh = +0.0; entries scored -0.0 are >= it as floats although their order keys are smaller."""
    n, c, D = 256, 2, 100
    rs = np.random.RandomState(12)
    scores = np.full((n, c), -0.5, np.float32)
    cells = rs.permutation(n * c)
    scores.flat[cells[:90]] = 0.5
    scores.flat[cells[90:110]] = 0.0
    scores.flat[cells[110:130]] = -0.0
    assert np.signbit(scores).sum() == n * c - 110
    boxes = disjoint_boxes(n)
    oracle = oracle_batched(scores[None], boxes[None], -1.0, 0.3, D)
    assert sum(len(i) for i in oracle[0][1]) == 130
    out = postproc.detections_batched(cuda(scores[None]), cuda(boxes[None]), -1.0, 0.3, D)
    assert int(out[0][0]) == 130
    assert_device_matches(out, oracle, (1, c, n))


def test_every_candidate_kept_worst_case():
    """Disjoint boxes and positive scores: all 4000 x 80 = 320 000 candidates of the image are kept."""
    n, c, D = 4000, 80, 100
    rs = np.random.RandomState(13)
    boxes = disjoint_boxes(n)
    scores = (rs.rand(n, c).astype(np.float32) * 0.99 + 0.01).astype(np.float32)
    assert bool(postproc.box_nms_batched(cuda(boxes[None]), cuda(scores[None]), 1e-5, 0.3).all())
    thresh = np.sort(scores.ravel())[-D]                              # mask_eval_utils.py:88, nothing suppressed
    assert (scores >= thresh).sum() == D
    inds = [np.nonzero(scores[:, j] >= thresh)[0] for j in range(c)]
    want = ([np.hstack((boxes[i], scores[i, j][:, None])).astype(np.float32) for j, i in enumerate(inds)], inds)
    out = postproc.detections_batched(cuda(scores[None]), cuda(boxes[None]), 1e-5, 0.3, D)
    assert_device_matches(out, [want], (1, c, n))
    # no limit: every one of the 320 000 detections comes back (second round of the host form, cap = count)
    res = postproc.results_with_nms_and_limit_batched(cuda(scores[None]), cuda(boxes[None]), 1e-5, 0.3, 0)
    everything = ([np.hstack((boxes, scores[:, j:j + 1])) for j in range(c)], [np.arange(n)] * c)
    assert_host_matches(res, [everything], c)
    out = postproc.detections_batched(cuda(scores[None]), cuda(boxes[None]), 1e-5, 0.3, 0)
    assert int(out[0][0]) == n * c and out[1].shape[1] == 128 and bool(out[5].all())


def test_no_limit():
    B, n, c = 3, 700, 12
    rs = np.random.RandomState(14)
    boxes = np.stack([proposals(n, 700 + b) for b in range(B)])
    scores = np.stack([sparse_scores(rs, n, c, 0.3) for _ in range(B)])
    oracle = oracle_batched(scores, boxes, 1e-5, 0.3, 0)
    assert min(sum(len(i) for i in o[1]) for o in oracle) > 128                # beyond the default cap
    out = postproc.detections_batched(cuda(scores), cuda(boxes), 1e-5, 0.3, 0)
    assert_device_matches(out, oracle, (B, c, n))
    assert_host_matches(postproc.results_with_nms_and_limit_batched(cuda(scores), cuda(boxes), 1e-5, 0.3, 0),
                        oracle, c)


@pytest.mark.parametrize("batched", [False, True])
def test_golden_coco_r500(batched):
    boxes, scores = NPZ["coco_r500/boxes"], NPZ["coco_r500/scores"]
    score_thr, nms_thr = (float(v) for v in NPZ["coco_r500/params"])
    if batched:                                                       # the fixture as the middle image of three
        rs = np.random.RandomState(15)
        n, c = scores.shape
        boxes = np.stack([proposals(n, 15), boxes, proposals(n, 16)])
        scores = np.stack([sparse_scores(rs, n, c, 0.2), scores, sparse_scores(rs, n, c, 0.2)])
    else:
        boxes, scores = boxes[None], scores[None]
    oracle = oracle_batched(scores, boxes, score_thr, nms_thr, 100)
    assert sum(len(i) for i in oracle[int(batched)][1]) == 100 < NPZ["coco_r500/keep"].sum()
    out = postproc.detections_batched(cuda(scores), cuda(boxes), score_thr, nms_thr, 100)
    assert_device_matches(out, oracle, (len(scores), scores.shape[2], scores.shape[1]))


def test_host_form_equals_per_image_calls():
    """results_with_nms_and_limit_batched == a loop of results_with_nms_and_limit, including an image whose ties
    take the batch into the second round."""
    B, n, c, D = 4, 1000, 20, 50
    rs = np.random.RandomState(16)
    boxes = np.stack([proposals(n, 800 + b) for b in range(B)])
    scores = np.stack([sparse_scores(rs, n, c, 0.1, levels=8) for _ in range(B)])
    oracle = oracle_batched(scores, boxes, 1e-5, 0.3, D)
    assert max(sum(len(i) for i in o[1]) for o in oracle) > D                  # ties: a second round
    res = postproc.results_with_nms_and_limit_batched(cuda(scores), cuda(boxes), 1e-5, 0.3, D)
    assert_host_matches(res, oracle, c)
    for b in range(B):
        one = postproc.results_with_nms_and_limit(cuda(scores[b]), cuda(boxes[b]), 1e-5, 0.3, D)
        for x, y in zip(one[:2], res[b][:2], strict=True):
            assert x.dtype == y.dtype
            np.testing.assert_array_equal(x, y)
        for xs, ys in zip(one[2:], res[b][2:], strict=True):
            for x, y in zip(xs, ys, strict=True):
                np.testing.assert_array_equal(x, y)


def test_non_default_stream():
    B, n, c = 2, 4000, 80
    rs = np.random.RandomState(17)
    boxes = cuda(np.stack([proposals(n, 900 + b) for b in range(B)]))
    scores = cuda(np.stack([sparse_scores(rs, n, c, 0.05) for _ in range(B)]))
    want = postproc.detections_batched(scores, boxes, 1e-5, 0.3, 100)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        got = postproc.detections_batched(scores, boxes, 1e-5, 0.3, 100)
    side.synchronize()
    assert int(want[0].min()) >= 100
    for g, w in zip(got, want, strict=True):
        assert torch.equal(g, w)


def test_errors():
    z = lambda *s: torch.zeros(*s, device=DEV)
    with pytest.raises(RuntimeError, match="no CPU path"):
        postproc.detections_batched(torch.zeros(1, 4, 2), torch.zeros(1, 4, 4))
    with pytest.raises(ValueError):
        postproc.detections_batched(z(1, 4, 2), z(1, 5, 4))
    with pytest.raises(ValueError):
        postproc.results_with_nms_and_limit_batched(z(2, 4, 2), z(1, 4, 4))
    with pytest.raises(RuntimeError, match="code -2"):
        postproc.detections_batched(z(1, 8193, 2), z(1, 8193, 4))    # n beyond the NMS kernel's limit
    with pytest.raises(ValueError):
        postproc.TestScoreMean(2).add(z(7, 4, 3), 3)                  # not 2 + 2K heads
    mean = postproc.TestScoreMean(2)
    mean.add(z(8, 4, 3), 3)
    with pytest.raises(ValueError):
        mean.add(z(8, 5, 3), 3)                                       # a different proposal count
