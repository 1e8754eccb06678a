"""Cost of ragged batches in CIMHeadStep.run at one of bench.py's 8 x 2000 shapes (default cfg2: ResNet-50, VOC; cfg3:
VGG-16, whose 64 x 64 maps take the RoIAlign window path), head gradients and PCL_loss on.  Four forms run alternately
in one process, on the same inputs and buffers:
  none     n_props = None (every image has R proposals; the entry points' NULL case)
  full     n_props = R for every image, through the ragged kernels
  ragged   a seeded draw of n_b uniform in [200, 2000] in the padded layout: every stage but mining still does the
           work of n_img x R rows
  compact  the same draw in the compact layout (run(compact=True)): rois, RoIAlign outputs and seg_x hold the
           sum(n_b) real rows only
Prints the card, its power limit, the median / spread of the per-step times of each form, and the rows that RoIAlign,
the scoring GEMMs and a caller's MaskFuse process in each form (a count: MaskFuse is not part of the step).

    python tools/ragged_bench.py [--workload cfg3_vgg16_voc_8x2000] [--steps 20] [--rounds 5] [--sampling stream|hop]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from cim_b200.step import CIMHeadStep  # noqa: E402


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True,
                              timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="steps per form and round")
    ap.add_argument("--rounds", type=int, default=5, help="rounds; each runs every form once, in turn")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sampling", default="stream", choices=["stream", "hop"])
    ap.add_argument("--seed", type=int, default=2024, help="seed of the ragged draw")
    ap.add_argument("--workload", default="cfg2_r50_voc_8x2000", choices=["cfg2_r50_voc_8x2000", "cfg3_vgg16_voc_8x2000"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ragged_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    cfg = bench.WORKLOADS[a.workload]
    inp = bench.build_inputs(cfg, dev, 1234)
    Cf, H, W, scale = inp["shape"]
    n_img, R = cfg["n_img"], cfg["R"]
    step = CIMHeadStep(n_img, R, cfg["C"], Cf, H, W, scale, inp["packed"].shape[-1], device=dev,
                       mask_kb_per_row=inp["kb_per_row"], head_grads=True, order="graph", rng=a.sampling)
    ragged = np.random.RandomState(a.seed).randint(200, R + 1, size=n_img).astype(np.int32)
    forms = {"none": None,
             "full": torch.full((n_img,), R, dtype=torch.int32, device=dev),
             "ragged": torch.from_numpy(ragged).to(dev),
             "compact": ragged}
    # the compact form's inputs: the real rows of the padded ones (rois keep their image index)
    idx = torch.from_numpy(np.concatenate([b * R + np.arange(n) for b, n in enumerate(ragged)])).to(dev)
    comp = {k: inp[k].index_select(0, idx).contiguous() for k in ("rois", "grad_out", "seg_x")}
    n_rows = int(ragged.sum())

    def run(n_props):
        src = comp if isinstance(n_props, np.ndarray) else inp
        step.run(inp["feat"], src["rois"], src["grad_out"], inp["packed"], src["seg_x"], inp["weight"], inp["bias"],
                 inp["labels"], mat=inp["mat"], mask_meta=inp["mask_meta"], n_props=n_props,
                 compact=src is comp)

    np.random.seed(3)
    for n_props in forms.values():
        for _ in range(a.warmup):
            run(n_props)
    torch.cuda.synchronize()
    step.sync_rng()
    times = {k: [] for k in forms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.rounds):
        for name, n_props in forms.items():
            ev0.record()
            for _ in range(a.steps):
                run(n_props)
            ev1.record()
            ev1.synchronize()
            step.sync_rng()
            times[name].append(ev0.elapsed_time(ev1) / a.steps)
    print(f"{torch.cuda.get_device_name(dev)}, power limit {power_limit()}: CIMHeadStep.run at {a.workload} "
          f"({n_img} x {R}, head gradients, PCL_loss, sampling {a.sampling}), {a.rounds} rounds x {a.steps} steps")
    print(f"ragged n_b = {ragged.tolist()}: {int(ragged.sum())} of {n_img * R} rows "
          f"({100.0 * (1 - ragged.sum() / (n_img * R)):.1f} % padding)")
    med = {k: float(np.median(v)) for k, v in times.items()}
    for name, v in times.items():
        rows = n_rows if name == "compact" else n_img * R
        print(f"  {name:7s} median {med[name]:.3f} ms/step  (min {min(v):.3f}, max {max(v):.3f}); "
              f"{n_img / med[name] * 1e3:.0f} images/s; rows through RoIAlign, scoring GEMMs and MaskFuse: {rows}")
    print(f"  full / none = {med['full'] / med['none']:.4f}; ragged / none = {med['ragged'] / med['none']:.4f}; "
          f"compact / ragged = {med['compact'] / med['ragged']:.4f}")


if __name__ == "__main__":
    main()
