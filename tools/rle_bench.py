#!/usr/bin/env python
"""COCO compressed RLE of the detections' proposal masks (the last stage of pseudo-label generation,
tools/generate_mask_for_MaskRCNN.py of the reference encodes them with pycocotools.mask.encode).  Per case, in one run:
  - the device time of cim_mask_rle (mask_ops.mask_rle: length pass, scan, emit pass), CUDA events over back-to-back
    calls;
  - the host form postproc.segms_batched end to end (it ends in a synchronise);
  - the box NMS of the same batch (box_nms_batched over all proposals and classes), the yardstick it follows;
  - the packed bytes each pass reads and the resulting rate;
  - the single-threaded C restatement of rleEncode + rleToString (oracle/rle_oracle.c) on the same masks, as uint8
    Fortran arrays prepared outside the timed region -- the per-mask host loop a caller runs without the device form.
Cases: 8 images x 100 detections (detections_batched on seeded scores) at 480 x 640 tiled, 512 x 512 tiled and
375 x 500 flat, and 8 x 250 = 2000 random selections at 512 x 512 tiled.  The device strings are checked against the C
restatement.

    python tools/rle_bench.py [--props 4000] [--classes 80] [--iters 20]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cim_b200 import mask_ops, postproc, synth  # noqa: E402
from oracle import rle_oracle  # noqa: E402

CASES = [(480, 640, "tiled", None), (512, 512, "tiled", None), (375, 500, "flat", None), (512, 512, "tiled", 250)]


def events(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters                      # ms


def wall(fn, iters):
    fn()
    t = time.perf_counter()
    for _ in range(iters):
        fn()
    return (time.perf_counter() - t) / iters * 1e3         # ms; fn ends in a synchronise


def run_case(H, W, layout, per_image, a, dev):
    B, n, C = 8, a.props, a.classes
    size = max(H, W)
    params = [synth.proposal_params(n, size, seed=100 + b) for b in range(B)]
    packed = None
    for b, p in enumerate(params):                        # one image at a time: 4000 byte masks of 480 x 640 = 1.2 GB
        pb = mask_ops.mask_pack(synth.rasterize(p, device=dev)[:, :H, :W].contiguous(), layout=layout)
        if packed is None:
            packed = torch.empty((B,) + tuple(pb.shape), dtype=torch.int32, device=dev)
        packed[b] = pb
    mask_ops._tag(packed, W // 16 if layout == "tiled" else 0)
    boxes = torch.stack([synth.rois_from_params(p)[:, 1:] for p in params]).to(dev)
    boxes[..., 0::2].clamp_(max=W - 1)
    boxes[..., 1::2].clamp_(max=H - 1)
    scores = torch.rand((B, n, C), generator=torch.Generator().manual_seed(H * W)).to(dev)
    dets = postproc.detections_batched(scores, boxes, 1e-5, 0.3, 100)
    if per_image:
        rs = np.random.RandomState(7)
        idx = torch.from_numpy(rs.randint(0, n, size=(B, per_image)).astype(np.int32)).to(dev)
        count = torch.full((B,), per_image, dtype=torch.int32, device=dev)
        dets = (count, torch.zeros_like(idx), idx) + tuple(dets[3:])
    count, idx = dets[0], dets[2]
    n_sel = int(count.clamp(max=idx.shape[1]).sum())

    t_nms = events(lambda: postproc.box_nms_batched(boxes, scores, 1e-5, 0.3), a.iters)
    out = mask_ops.mask_rle(packed, count, idx, H, W)
    need = int(out[5][0])
    cap_chars = max(need, 1)
    t_rle = events(lambda: mask_ops.mask_rle(packed, count, idx, H, W, chars_cap=cap_chars), a.iters)
    t_host = wall(lambda: postproc.segms_batched(packed, dets, H, W, C), max(2, a.iters // 4))
    pass_bytes = n_sel * packed.shape[2] * 4

    # the C restatement on the same masks (uint8 Fortran arrays made before the clock starts)
    chars, off, len_ = (t.cpu().numpy() for t in mask_ops.mask_rle(packed, count, idx, H, W, chars_cap=cap_chars)[:3])
    cnt, ix = count.cpu().numpy(), idx.cpu().numpy()
    fortran, want = [], []
    for b in range(B):
        k = min(int(cnt[b]), ix.shape[1])
        p = params[b]
        sel = ix[b, :k]
        sub = synth.ProposalParams(p.cx[sel], p.cy[sel], p.ax[sel], p.ay[sel], p.size)
        m = synth.rasterize(sub, device=dev)[:, :H, :W].cpu().numpy() if k else np.zeros((0, H, W), np.uint8)
        fortran += [np.asfortranarray(x) for x in m]
        want += [chars[off[b, j]:off[b, j] + len_[b, j]].tobytes() for j in range(k)]
    enc = rle_oracle.CEncoder(H * W)
    t = time.perf_counter()
    got = [enc(x) for x in fortran]
    t_c = (time.perf_counter() - t) * 1e3
    assert got == want, "device strings differ from the C restatement"
    return (f"{B} x {'%d random' % per_image if per_image else 'detections'} ({n_sel} masks) at {H} x {W} {layout}: "
            f"cim_mask_rle {t_rle * 1e3:.1f} us ({pass_bytes / 1e6:.1f} MB packed per pass, "
            f"{2 * pass_bytes / t_rle / 1e6:.0f} GB/s over both passes), segms_batched end to end {t_host:.3f} ms, "
            f"box NMS of the batch ({n} proposals x {C} classes) {t_nms:.3f} ms, C restatement (1 thread) "
            f"{t_c:.1f} ms; {need} characters")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--props", type=int, default=4000)
    ap.add_argument("--classes", type=int, default=80)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    name = torch.cuda.get_device_name(dev)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(f"{name}, power limit {power}")
    for H, W, layout, per_image in CASES:
        print(run_case(H, W, layout, per_image, a, dev), flush=True)


if __name__ == "__main__":
    main()
