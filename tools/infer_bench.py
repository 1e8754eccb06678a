#!/usr/bin/env python
"""BASELINE.json configs[4]: HRNet-W48 COCO pseudo-label generation (inference), 4000 proposals per image.
Times the test-time chain of the library per batch of images on one GPU -- RoIAlign forward
(tools/generate_mask_for_MaskRCNN.py:124-190 runs the model in eval mode), scoring heads forward, K-head score mean
(lib/core/test.py:130-133), per-class box NMS (lib/utils/mask_eval_utils.py:57-79) -- with CUDA events.
Then the detection chain with test-time augmentation: --tta T scoring passes accumulated by postproc.TestScoreMean
(core/test.py:149-226, SCORE_HEUR 'AVG'), the batched NMS, the DETECTIONS_PER_IM limit + compaction
(mask_eval_utils.py:80-110) and the copy of the detections to pinned host memory, ending in a synchronise.

    python tools/infer_bench.py [--images 4] [--props 4000] [--classes 80] [--backbone hrnet48] [--iters 10]
                                [--tta 1] [--detections 100]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cim_b200 import _lib, postproc, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=4)
    ap.add_argument("--props", type=int, default=4000)
    ap.add_argument("--classes", type=int, default=80)
    ap.add_argument("--backbone", default="hrnet48")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--tta", type=int, default=1, help="scoring passes averaged per image (TEST.BBOX_AUG: 10)")
    ap.add_argument("--detections", type=int, default=100, help="DETECTIONS_PER_IM")
    a = ap.parse_args()
    if a.tta < 1:
        ap.error("--tta must be >= 1")
    dev = torch.device("cuda:0")
    Cf, H, W, scale = synth.feature_shape(a.backbone)
    B, R, C1, K, D = a.images, a.props, a.classes + 1, 3, 4096
    L = _lib.lib()
    P, st = _lib.ptr, _lib.stream_ptr(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(R, 512, 1234 + b), b) for b in range(B)]).to(dev)
    feat = torch.randn(B, Cf, H, W, device=dev, generator=g)
    out = torch.empty(B * R, Cf, 7, 7, device=dev)
    ws = torch.empty(L.cim_roi_align_workspace_bytes_ex(B, Cf, H, W, B * R, 7, 7), dtype=torch.uint8, device=dev)
    seg_x = torch.randn(B * R, D, device=dev, generator=g)
    nh = 2 + 2 * K
    weight = torch.randn(nh, C1, D, device=dev, generator=g) * 0.02
    bias = torch.zeros(nh, C1, device=dev)
    scores = torch.empty(nh, B * R, C1, device=dev)
    sws = torch.empty(max(256, L.cim_score_heads_workspace_bytes(B, R, D, C1, K)), dtype=torch.uint8, device=dev)

    boxes = rois[:, 1:].reshape(B, R, 4).contiguous()

    def roi():
        _lib.check(L.cim_roi_align_fwd(P(feat), P(rois), P(out), B, Cf, H, W, B * R, 7, 7, scale, 0, 1, P(ws), ws.numel(),
                                       st), "roi")

    def score():
        _lib.check(L.cim_score_heads(P(seg_x), P(weight), P(bias), P(scores), B, R, D, C1, K, P(sws), sws.numel(), st),
                   "score")

    def post():
        s = postproc.test_scores(scores, K)                       # [B*R, C]
        postproc.box_nms_batched(boxes, s.view(B, R, -1), 1e-5, 0.3)

    def timeit(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.iters

    t_roi, t_score, t_post = timeit(roi), timeit(score), timeit(post)
    t_all = timeit(lambda: (roi(), score(), post()))
    print(f"{a.backbone} {B} images x {R} proposals, {a.classes} classes: RoIAlign fwd {t_roi:.3f} ms "
          f"({out.numel() * 4 / t_roi / 1e6:.0f} GB/s), scoring {t_score:.3f} ms, score mean + box NMS {t_post:.3f} ms, "
          f"chain {t_all:.3f} ms = {B / t_all * 1e3:.0f} images/s")

    # detection chain with TTA: T x (scoring + accumulate), NMS, limit + compaction, D2H of the detections
    T, Dl, C = a.tta, a.detections, C1 - 1
    mean = postproc.TestScoreMean(T)
    for _ in range(T):
        score()
        mean.add(scores, K)
    s = mean.scores.view(B, R, C)
    keep = postproc.box_nms_batched(boxes, s, 1e-5, 0.3)
    dets = postproc.box_detections(boxes, s, keep, Dl)
    pinned = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in dets[:5]]

    def accumulate():
        m = postproc.TestScoreMean(T)
        for _ in range(T):
            m.add(scores, K)

    def d2h():
        for h, t in zip(pinned, dets[:5]):
            h.copy_(t, non_blocking=True)

    def chain():
        m = postproc.TestScoreMean(T)
        for _ in range(T):
            score()
            m.add(scores, K)
        sc = m.scores.view(B, R, C)
        out = postproc.box_detections(boxes, sc, postproc.box_nms_batched(boxes, sc, 1e-5, 0.3), Dl)
        for h, t in zip(pinned, out[:5]):
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()

    t_acc = timeit(accumulate) / T
    t_nms = timeit(lambda: postproc.box_nms_batched(boxes, s, 1e-5, 0.3))
    t_lim = timeit(lambda: postproc.box_detections(boxes, s, keep, Dl))
    t_d2h = timeit(d2h)
    t_chain = timeit(chain)
    acc_bytes = 2 * K * B * R * C1 * 4 + 2 * B * R * C * 4
    name = torch.cuda.get_device_name(dev)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    counts = dets[0].tolist()
    print(f"{name}, power limit {power}: TTA x{T}, D = {Dl}: accumulate {t_acc * 1e3:.1f} us/pass "
          f"({acc_bytes / t_acc / 1e6:.0f} GB/s of {acc_bytes / 1e6:.1f} MB/pass), box NMS {t_nms:.3f} ms, "
          f"limit + compaction {t_lim * 1e3:.1f} us, D2H {t_d2h * 1e3:.1f} us, "
          f"chain (incl. {T} scoring passes, ends in a synchronise) {t_chain:.3f} ms; detections per image {counts}, "
          f"kept before the limit {keep.view(B, -1).sum(1).tolist()}")


if __name__ == "__main__":
    main()
