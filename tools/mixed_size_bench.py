"""Cost of batching differently sized images on one feature-map canvas (RoIAlign with per-image extents, feat_hw) in
CIMHeadStep.run, at bench.py's inputs: cfg2 (ResNet-50, VOC, 8 images x 2000 proposals, 32 x 32 canvas, tile kernels)
and cfg3 (VGG-16, 64 x 64 canvas, window tiles).  Head gradients and PCL_loss on.  Three forms of the step run
alternately in one process, on the same inputs and buffers:
  none    feat_hw = None (every image fills the canvas; the entry points' NULL case)
  full    feat_hw = the canvas for every image, through the _ex path
  mixed   seeded VOC-like extents: the longest side fills the canvas, the other side is 5/8 .. 1 of it (20 .. 32
          cells at cfg2); each image's rois are scaled into its extent
Next to them, the RoIAlign forward + backward of the mixed batch two ways: in one batched call with feat_hw
(`batched`), and image by image on the cropped maps (`per_image`), the only exact way without extents.
Prints the card, its power limit and the median / spread of each form.

    python tools/mixed_size_bench.py [--steps 20] [--rounds 5] [--sampling stream|hop]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from cim_b200 import ops  # noqa: E402
from cim_b200.step import CIMHeadStep  # noqa: E402


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True,
                              timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def voc_extents(rng, n_img, H, W):
    """Longest side = the canvas, the other side uniform in [5/8, 1] of it; landscape and portrait alternate."""
    hw = np.zeros((n_img, 2), np.int32)
    for b in range(n_img):
        if b % 2 == 0:
            hw[b] = (rng.randint((5 * H + 7) // 8, H + 1), W)
        else:
            hw[b] = (H, rng.randint((5 * W + 7) // 8, W + 1))
    return hw


def measure(name, a, dev):
    cfg = bench.WORKLOADS[name]
    inp = bench.build_inputs(cfg, dev, 1234)
    Cf, H, W, scale = inp["shape"]
    n_img, R = cfg["n_img"], cfg["R"]
    step = CIMHeadStep(n_img, R, cfg["C"], Cf, H, W, scale, inp["packed"].shape[-1], device=dev,
                       mask_kb_per_row=inp["kb_per_row"], head_grads=True, order="graph", rng=a.sampling)
    hw = voc_extents(np.random.RandomState(a.seed), n_img, H, W)
    rois_mixed = inp["rois"].clone()
    b = rois_mixed[:, 0].long()
    fy = torch.from_numpy(hw[:, 0] / H).float().to(dev)[b]
    fx = torch.from_numpy(hw[:, 1] / W).float().to(dev)[b]
    rois_mixed[:, 1] *= fx
    rois_mixed[:, 3] *= fx
    rois_mixed[:, 2] *= fy
    rois_mixed[:, 4] *= fy
    hw_dev = torch.from_numpy(hw).to(dev)
    forms = {"none": (inp["rois"], None),
             "full": (inp["rois"], torch.tensor([[H, W]] * n_img, dtype=torch.int32, device=dev)),
             "mixed": (rois_mixed, hw_dev)}

    def run(rois, feat_hw):
        step.run(inp["feat"], rois, inp["grad_out"], inp["packed"], inp["seg_x"], inp["weight"], inp["bias"],
                 inp["labels"], mat=inp["mat"], mask_meta=inp["mask_meta"], feat_hw=feat_hw)

    # RoIAlign forward + backward of the mixed batch: batched with feat_hw, or image by image on the cropped maps
    feat = inp["feat"]
    crops = [feat[i:i + 1, :, :hw[i, 0], :hw[i, 1]].contiguous() for i in range(n_img)]
    per_rois = []
    for i in range(n_img):
        r = rois_mixed[i * R:(i + 1) * R].clone()
        r[:, 0] = 0
        per_rois.append(r)
    grads = [inp["grad_out"][i * R:(i + 1) * R] for i in range(n_img)]
    feat_g = feat.detach().requires_grad_(True)
    crops_g = [c.requires_grad_(True) for c in crops]

    def roi_batched(_rois, _hw):
        out = ops.roi_align(feat_g, rois_mixed, 7, scale, 0, "avg", True, feat_hw=hw_dev)
        out.backward(inp["grad_out"])

    def roi_per_image(_rois, _hw):
        for c, r, g in zip(crops_g, per_rois, grads):
            out = ops.roi_align(c, r, 7, scale, 0, "avg", True)
            out.backward(g)

    roi_forms = {"batched": roi_batched, "per_image": roi_per_image}
    everything = [(k, run, v) for k, v in forms.items()] + [(k, f, (None, None)) for k, f in roi_forms.items()]

    np.random.seed(3)
    for _, fn, args in everything:
        for _ in range(a.warmup):
            fn(*args)
    torch.cuda.synchronize()
    step.sync_rng()
    times = {k: [] for k, _, _ in everything}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.rounds):
        for key, fn, args in everything:
            ev0.record()
            for _ in range(a.steps):
                fn(*args)
            ev1.record()
            ev1.synchronize()
            step.sync_rng()
            times[key].append(ev0.elapsed_time(ev1) / a.steps)
    print(f"{name}: {n_img} x {R}, canvas {Cf} x {H} x {W}, {a.rounds} rounds x {a.steps} steps, "
          f"sampling {a.sampling}; mixed extents {[tuple(x) for x in hw.tolist()]}")
    med = {k: float(np.median(v)) for k, v in times.items()}
    for key, v in times.items():
        what = "CIMHeadStep.run" if key in forms else "RoIAlign fwd + bwd"
        print(f"  {key:9s} {what:18s} median {med[key]:.3f} ms  (min {min(v):.3f}, max {max(v):.3f})")
    print(f"  full / none = {med['full'] / med['none']:.4f}; mixed / none = {med['mixed'] / med['none']:.4f}; "
          f"per_image / batched = {med['per_image'] / med['batched']:.2f}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="steps per form and round")
    ap.add_argument("--rounds", type=int, default=5, help="rounds; each runs every form once, in turn")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sampling", default="stream", choices=["stream", "hop"])
    ap.add_argument("--seed", type=int, default=2024, help="seed of the mixed extents")
    ap.add_argument("--workloads", default="cfg2_r50_voc_8x2000,cfg3_vgg16_voc_8x2000")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mixed_size_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    print(f"{torch.cuda.get_device_name(dev)}, power limit {power_limit()}")
    for name in a.workloads.split(","):
        measure(name, a, dev)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
