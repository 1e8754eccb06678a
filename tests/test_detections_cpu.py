"""Batched test-time detections without a GPU: argument validation of cim_test_scores_tta / cim_box_detections
(checked before anything touches CUDA), and the TTA mean the GPU tests compare with: np.mean over the passes is a
float32 sum in pass order divided once."""
import ctypes as C

import numpy as np
import pytest
import torch

from cim_b200 import _lib, postproc
from oracle import nms_oracle

NULL = C.c_void_p(0)
FAKE = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch


def tta_scores(passes):
    """TEST.BBOX_AUG with SCORE_HEUR 'AVG' (core/test.py:149-226): np.mean over the passes of the oracle's test
    scores, as tests/test_gpu_detections.py compares cim_test_scores_tta with."""
    return np.mean(np.stack([nms_oracle.test_scores(cls_t, iou_t) for cls_t, iou_t in passes]), axis=0)


def test_test_scores_tta_argument_validation():
    L = _lib.lib()
    assert L.cim_test_scores_tta(NULL, FAKE, 10, 81, 3, 0, 1, NULL) == -1
    assert L.cim_test_scores_tta(FAKE, NULL, 10, 81, 3, 0, 1, NULL) == -1
    for m, c1, k, t, T in [(-1, 81, 3, 0, 1), (10, 1, 3, 0, 1), (10, 81, 0, 0, 1), (10, 81, 9, 0, 1),
                           (10, 81, 3, 0, 0), (10, 81, 3, -1, 2), (10, 81, 3, 2, 2)]:
        assert L.cim_test_scores_tta(FAKE, FAKE, m, c1, k, t, T, NULL) == -1, (m, c1, k, t, T)
    assert L.cim_test_scores_tta(FAKE, FAKE, 0, 81, 3, 1, 2, NULL) == 0          # nothing to do


def test_box_detections_argument_validation():
    L = _lib.lib()
    call = lambda boxes=FAKE, scores=FAKE, keep=FAKE, b=8, n=4000, c=80, stride=80, d=100, cap=100, count=FAKE, \
        cls=FAKE, idx=FAKE, score=FAKE: L.cim_box_detections(boxes, scores, keep, b, n, c, stride, d, cap, NULL,
                                                             count, cls, idx, score, NULL, NULL)
    for kw in ({"boxes": NULL}, {"scores": NULL}, {"keep": NULL}, {"count": NULL}, {"cls": NULL}, {"idx": NULL},
               {"score": NULL}, {"b": -1}, {"n": -1}, {"c": -1}, {"stride": 79}, {"cap": -1}):
        assert call(**kw) == -1, kw
    assert call(cap=0, cls=NULL, idx=NULL, score=NULL, b=0) == 0              # no lists wanted, no images
    assert call(n=8193) == -2
    assert call(c=65536, stride=65536) == -2
    assert call(b=0) == 0


def test_no_cpu_path():
    with pytest.raises(RuntimeError, match="no CPU path"):
        postproc.TestScoreMean(2).add(torch.zeros(8, 4, 3), 3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        postproc.detections_batched(torch.zeros(1, 4, 2), torch.zeros(1, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU path"):
        postproc.results_with_nms_and_limit_batched(torch.zeros(1, 4, 2), torch.zeros(1, 4, 4))
    with pytest.raises(ValueError):
        postproc.TestScoreMean(0)


@pytest.mark.parametrize("T", [2, 3, 10, 17])
def test_tta_mean_is_a_sequential_float32_sum(T):
    """np.mean over the stacked passes of float32 scores is the float32 sum in pass order divided once by T, which is
    what cim_test_scores_tta computes; mixed magnitudes make the rounding of every step visible."""
    rs = np.random.RandomState(T)
    k, m, c1 = 3, 400, 81
    passes = []
    for _ in range(T):
        mag = (10.0 ** rs.uniform(-4, 2, size=(2 * k, m, c1))).astype(np.float32)
        s = (rs.rand(2 * k, m, c1).astype(np.float32) * mag).astype(np.float32)
        passes.append((list(s[:k]), list(s[k:])))
    got = tta_scores(passes)
    per = [nms_oracle.test_scores(cls_t, iou_t) for cls_t, iou_t in passes]
    assert got.dtype == np.float32
    acc = per[0].copy()
    for p in per[1:]:
        acc = acc + p
    want = acc / np.float32(T)
    assert want.dtype == np.float32
    np.testing.assert_array_equal(got, want)
    if T > 2:                     # two float32 summands round once, like the float64 sum; more do not
        assert not np.array_equal(got, (np.sum(np.stack(per).astype(np.float64), 0) / T).astype(np.float32))
