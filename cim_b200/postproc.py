"""Test-time post-processing of the CIM heads on the GPU (SURVEY.md 8f-3), with the reference's surface:

  test_scores(scores, k)                       lib/core/test.py:130-133 (mean over the refinement heads of
                                               model_builder.testing_function's (cls * iou)[:, 1:])
  box_nms(boxes, scores, score_thresh, nms)    per-class candidate filter + lib/utils/cython_nms.pyx `nms`
  results_with_nms_and_limit(...)              lib/utils/mask_eval_utils.py:57-110
                                               (mask_results_with_nms_and_limit_get_index)
  TestScoreMean(n_passes)                      lib/core/test.py:149-226 (TEST.BBOX_AUG, SCORE_HEUR 'AVG')
  detections_batched(...)                      :57-110 for a batch of images, results left on the device
  results_with_nms_and_limit_batched(...)      the same, as the reference's per-image host lists

All arithmetic runs in libcimhead.so (cim_test_scores[_tta] / cim_box_nms[_batched] / cim_box_detections); there is
no CPU path.
"""
import numpy as np
import torch

from . import _lib


def test_scores(scores, k):
    """scores [2+2K, M, C+1] (cls_iou_model.forward_batched) -> [M, C]: mean_k (ref_cls_k * ref_iou_k)[:, 1:]."""
    _lib.require_cuda(scores, "scores", torch.float32)
    scores = scores.contiguous()
    nh, m, c1 = scores.shape
    if nh != 2 + 2 * k:
        raise ValueError("scores must hold 2 + 2K heads")
    with torch.cuda.device(scores.device):
        out = torch.empty((m, c1 - 1), dtype=torch.float32, device=scores.device)
        rc = _lib.lib().cim_test_scores(_lib.ptr(scores), _lib.ptr(out), m, c1, k, _lib.stream_ptr(scores.device))
    _lib.check(rc, "cim_test_scores")
    return out


def box_nms(boxes, scores, score_thresh=1e-5, nms_thresh=0.3):
    """boxes [n,4] (x1,y1,x2,y2), scores [n,C] -> keep [C,n] uint8: proposal i survives class c's NMS."""
    _lib.require_cuda(boxes, "boxes", torch.float32)
    _lib.require_cuda(scores, "scores", torch.float32)
    boxes, scores = boxes.contiguous(), scores.contiguous()
    n, c = scores.shape
    if boxes.shape != (n, 4):
        raise ValueError("boxes must be [n, 4]")
    with torch.cuda.device(boxes.device):
        keep = torch.empty((c, n), dtype=torch.uint8, device=boxes.device)
        rc = _lib.lib().cim_box_nms(_lib.ptr(boxes), _lib.ptr(scores), n, c, c, float(score_thresh),
                                    float(nms_thresh), _lib.ptr(keep), _lib.stream_ptr(boxes.device))
    _lib.check(rc, "cim_box_nms")
    return keep


def box_nms_batched(boxes, scores, score_thresh=1e-5, nms_thresh=0.3):
    """boxes [B,n,4], scores [B,n,C] -> keep [B,C,n] uint8: box_nms for every image of a batch in one launch."""
    _lib.require_cuda(boxes, "boxes", torch.float32)
    _lib.require_cuda(scores, "scores", torch.float32)
    boxes, scores = boxes.contiguous(), scores.contiguous()
    b, n, c = scores.shape
    if boxes.shape != (b, n, 4):
        raise ValueError("boxes must be [B, n, 4]")
    with torch.cuda.device(boxes.device):
        keep = torch.empty((b, c, n), dtype=torch.uint8, device=boxes.device)
        rc = _lib.lib().cim_box_nms_batched(_lib.ptr(boxes), _lib.ptr(scores), b, n, c, c, float(score_thresh),
                                            float(nms_thresh), _lib.ptr(keep), _lib.stream_ptr(boxes.device))
    _lib.check(rc, "cim_box_nms_batched")
    return keep


class TestScoreMean:
    """Mean of the test scores over the passes of test-time augmentation (core/test.py:149-226, SCORE_HEUR 'AVG':
    np.mean(scores_ts, axis=0)), accumulated one pass at a time so that a TTA loop can reuse one scoring buffer:
    .add(scores, k) per pass ([2+2K, M, C+1], as test_scores takes it), then .scores is the [M, C] mean -- the
    float32 sum of the passes in the order they were added, divided once by n_passes."""
    __test__ = False                                   # not a pytest class

    def __init__(self, n_passes):
        if int(n_passes) < 1:
            raise ValueError("n_passes must be >= 1")
        self.n_passes, self.passes, self._acc = int(n_passes), 0, None

    def add(self, scores, k):
        _lib.require_cuda(scores, "scores", torch.float32)
        if self.passes >= self.n_passes:
            raise RuntimeError(f"TestScoreMean: all {self.n_passes} passes were already added")
        scores = scores.contiguous()
        nh, m, c1 = scores.shape
        if nh != 2 + 2 * k:
            raise ValueError("scores must hold 2 + 2K heads")
        if self._acc is None:
            self._acc = torch.empty((m, c1 - 1), dtype=torch.float32, device=scores.device)
        elif self._acc.shape != (m, c1 - 1) or self._acc.device != scores.device:
            raise ValueError("every pass must score the same proposals and classes on the same device")
        with torch.cuda.device(scores.device):
            rc = _lib.lib().cim_test_scores_tta(_lib.ptr(scores), _lib.ptr(self._acc), m, c1, k, self.passes,
                                                self.n_passes, _lib.stream_ptr(scores.device))
        _lib.check(rc, "cim_test_scores_tta")
        self.passes += 1

    @property
    def scores(self):
        if self.passes < self.n_passes:
            raise RuntimeError(f"TestScoreMean: {self.passes} of {self.n_passes} passes added")
        return self._acc


def _detections_buffer(b, cap, device):
    """One int32 device buffer holding count [B] and cls, idx, score, box [B, cap(, 4)], so that the host form can
    fetch all of it with one copy.  Returns (buffer, count, cls, idx, score, box)."""
    buf = torch.empty(b + b * cap * 7, dtype=torch.int32, device=device)
    o = [b, b + b * cap, b + 2 * b * cap, b + 3 * b * cap]
    return (buf, buf[:o[0]], buf[o[0]:o[1]].view(b, cap), buf[o[1]:o[2]].view(b, cap),
            buf[o[2]:o[3]].view(torch.float32).view(b, cap), buf[o[3]:].view(torch.float32).view(b, cap, 4))


def _box_detections(boxes, scores, keep, detections_per_im, cap, keep_out):
    b, n, c = scores.shape
    out = _detections_buffer(b, cap, boxes.device)
    _, count, cls, idx, score, box = out
    with torch.cuda.device(boxes.device):
        rc = _lib.lib().cim_box_detections(_lib.ptr(boxes), _lib.ptr(scores), _lib.ptr(keep), b, n, c, c,
                                           int(detections_per_im), cap, _lib.ptr(keep_out), _lib.ptr(count),
                                           _lib.ptr(cls), _lib.ptr(idx), _lib.ptr(score), _lib.ptr(box),
                                           _lib.stream_ptr(boxes.device))
    _lib.check(rc, "cim_box_detections")
    return out


def box_detections(boxes, scores, keep, detections_per_im=100, cap=None):
    """The limit and compaction alone (cim_box_detections) for the keep mask [B,C,n] of box_nms_batched over the
    same boxes [B,n,4] and scores [B,n,C] -> (count, cls, idx, score, box, keep) as detections_batched returns them."""
    for t, name, dt in ((boxes, "boxes", torch.float32), (scores, "scores", torch.float32), (keep, "keep", torch.uint8)):
        _lib.require_cuda(t, name, dt)
    boxes, scores, keep = boxes.contiguous(), scores.contiguous(), keep.contiguous()
    b, n, c = scores.shape
    if boxes.shape != (b, n, 4) or keep.shape != (b, c, n):
        raise ValueError("boxes must be [B, n, 4] and keep [B, C, n]")
    cap = _default_cap(detections_per_im) if cap is None else int(cap)
    if cap < 0:
        raise ValueError("cap must be >= 0")
    keep_out = torch.empty_like(keep)
    _, count, cls, idx, score, box = _box_detections(boxes, scores, keep, detections_per_im, cap, keep_out)
    return count, cls, idx, score, box, keep_out


def _default_cap(detections_per_im):
    return int(detections_per_im) if detections_per_im > 0 else 128


def detections_batched(scores, boxes, score_thresh=1e-5, nms_thresh=0.3, detections_per_im=100):
    """mask_eval_utils.py:57-110 for a batch, on the device, without a host synchronisation.  scores [B,n,C],
    boxes [B,n,4] CUDA tensors -> (count [B] int32, cls [B,cap] int32, idx [B,cap] int32, score [B,cap] fp32,
    box [B,cap,4] fp32, keep [B,C,n] uint8), cap = detections_per_im (128 when it is <= 0).  Row b holds the first
    min(count[b], cap) detections of image b, by class then proposal index; count can exceed detections_per_im
    (scores tied at the limit all survive) and cap; keep is the keep mask after the limit."""
    return box_detections(boxes, scores, box_nms_batched(boxes, scores, score_thresh, nms_thresh), detections_per_im)


def results_with_nms_and_limit_batched(scores, boxes, score_thresh=1e-5, nms_thresh=0.3, detections_per_im=100):
    """results_with_nms_and_limit for every image of a batch: scores [B,n,C], boxes [B,n,4] CUDA tensors -> a list of
    B tuples (scores, boxes, cls_boxes, cls_inds).  The NMS, the limit and the compaction run on the device; the
    detections come back in one pinned copy with one synchronisation (a second round only when an image has more
    than cap = detections_per_im detections, 128 without a limit)."""
    keep = box_nms_batched(boxes, scores, score_thresh, nms_thresh)
    scores, boxes = scores.contiguous(), boxes.contiguous()
    b, n, c = scores.shape
    stream = torch.cuda.current_stream(boxes.device)

    def fetch(cap):
        buf = _box_detections(boxes, scores, keep, detections_per_im, cap, None)[0]
        host = torch.empty(buf.shape, dtype=buf.dtype, pin_memory=True)
        host.copy_(buf, non_blocking=True)
        stream.synchronize()
        h = host.numpy()
        o = [b, b + b * cap, b + 2 * b * cap, b + 3 * b * cap]
        return (h[:o[0]], h[o[0]:o[1]].reshape(b, cap), h[o[1]:o[2]].reshape(b, cap),
                h[o[2]:o[3]].view(np.float32).reshape(b, cap), h[o[3]:].view(np.float32).reshape(b, cap, 4))

    cap = _default_cap(detections_per_im)
    count, cls, idx, score, box = fetch(cap)
    if b and int(count.max()) > cap:                      # ties at the limit, or no limit
        cap = int(count.max())
        count, cls, idx, score, box = fetch(cap)
    results = []
    for i in range(b):
        k = int(count[i])
        bounds = np.searchsorted(cls[i, :k], np.arange(c + 1))
        cls_boxes, cls_inds = [[]], [[]]
        for j in range(c):
            lo, hi = bounds[j], bounds[j + 1]
            cls_inds.append(idx[i, lo:hi].astype(np.intp))
            cls_boxes.append(np.hstack((box[i, lo:hi], score[i, lo:hi, None])).astype(np.float32, copy=False))
        im_results = np.vstack([cls_boxes[j] for j in range(1, c)]) if c > 1 else np.zeros((0, 5), np.float32)
        results.append((im_results[:, -1], im_results[:, :-1], cls_boxes, cls_inds))
    return results


def results_with_nms_and_limit(scores, boxes, score_thresh=1e-5, nms_thresh=0.3, detections_per_im=100):
    """mask_results_with_nms_and_limit_get_index (mask_eval_utils.py:57-110) for one image.
    scores [n,C], boxes [n,4] CUDA tensors.  Returns (scores, boxes, cls_boxes, cls_inds) with the reference's
    conventions: cls_boxes / cls_inds are lists of length C + 1 shifted by one (entry 0 empty, :96-105), holding
    numpy [k,5] float32 detections and the proposal indices they came from; the flat `scores` / `boxes` stack
    entries 1 .. C-1 exactly as :108-110 does (the last class is left out there too)."""
    _lib.require_cuda(boxes, "boxes", torch.float32)
    _lib.require_cuda(scores, "scores", torch.float32)
    if scores.dim() != 2 or boxes.shape != (scores.shape[0], 4):
        raise ValueError("scores must be [n, C] and boxes [n, 4]")
    return results_with_nms_and_limit_batched(scores[None], boxes[None], score_thresh, nms_thresh,
                                              detections_per_im)[0]
