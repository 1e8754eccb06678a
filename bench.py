#!/usr/bin/env python
"""bench.py -- CIM-head images/s on B200 (BASELINE.json metric).

A step = one pass of the hot path over one batch of synthetic images:
RoIAlign fwd + RoIAlign bwd + mask IoU/containment + scoring heads fwd + 3 x (mining + assignment) + the loss
block incl. PCL_loss (fwd + bwd) + scoring heads bwd (head gradients, averaged over the ranks with one NCCL allreduce when N > 1).
Workload = BASELINE.json configs[1]: ResNet-50 VOC, 8 images x 2000 mask proposals per GPU
(512x512 images -> 1024x32x32 features, 512x512 bit-packed proposal masks, 20 classes).

    python bench.py [--gpus N] [--steps K] [--warmup W]          one JSON line on rank 0
    python bench.py --impl reference ...                          the CPU restatement, host cores
    python bench.py --dump-outputs DIR ...                        + the last timed step's results as DIR/<name>.npy

Weak scaling: every rank owns its own 8 images (the path shards per image, no data-path
collective; SURVEY.md section 8e).  Timing: CUDA events on the launching stream, barrier +
synchronize on both sides, MAX over ranks.  The per-step working set (>3 GB of RoI gradients
alone) is far larger than the 126 MB L2, so no explicit flush is needed between iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The CPU arm uses every host core whatever the launcher exported: torchrun sets OMP_NUM_THREADS=1 for its workers,
# which made the N > 1 reference lines 3.5x slower than the N = 1 line in round 1.  BLAS / OpenMP read these when
# numpy / torch load, so they are set before either is imported.
if "reference" in sys.argv[1:] and "--impl" in sys.argv[1:] or any(a.startswith("--impl=reference") for a in sys.argv[1:]):
    for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "CIM-head images/s (ROIAlign fwd+bwd + mask IoU + scoring fwd+bwd + mining + losses incl. PCL)"
WORKLOADS = {
    # name: backbone, images per GPU, proposals, classes, present classes, mask side
    "cfg2_r50_voc_8x2000": dict(backbone="resnet50", n_img=8, R=2000, C=20, present=2, mask=512),
    "cfg3_vgg16_voc_8x2000": dict(backbone="vgg16", n_img=8, R=2000, C=20, present=2, mask=512),
    # BASELINE.json configs[2]: a batch of 64 images sharded per image over 2/4/8 GPUs (64 / N per rank; N = 1: 8)
    "cfg3_vgg16_voc_64": dict(backbone="vgg16", n_img=8, total_images=64, R=2000, C=20, present=2, mask=512),
    # configs[4]: HRNet-W48 COCO pseudo-label generation, forward only
    "cfg5_hrnet48_coco_infer_8x4000": dict(backbone="hrnet48", n_img=8, R=4000, C=80, present=4, mask=128,
                                           inference=True),
    "cfg4_r50_coco_8x2000_q": dict(backbone="resnet50", n_img=8, R=2000, C=80, present=4, mask=128),
    "cfg1_r50_voc_1x300": dict(backbone="resnet50", n_img=1, R=300, C=20, present=2, mask=512),
    "tiny": dict(backbone="resnet50", n_img=2, R=200, C=20, present=2, mask=128),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def algorithmic_bytes(cfg, Cf, H, W):
    """SURVEY.md section 8d, bytes per image and stage."""
    R, C, hwm = cfg["R"], cfg["C"], cfg["mask"] ** 2
    F, O = Cf * H * W * 4, R * Cf * 49 * 4
    return {
        "roi_align_fwd": F + 20 * R + O,
        "roi_align_bwd": O + 20 * R + F,
        "mask_overlap": R * hwm // 8 + 2 * R * R * 2,
        "score_heads": R * 4096 * 4 + 8 * (C + 1) * 4097 * 4 + 8 * R * (C + 1) * 4,
        "mine_assign": 3 * (2 * R * R * 2 + R * (C + 1) * 4 + R * 6),
        # scoring backward: x read, grad_x written, scores and grad_scores read, weights read and head
        # gradients written
        "score_heads_bwd": 2 * R * 4096 * 4 + 2 * 8 * R * (C + 1) * 4 + 2 * 8 * (C + 1) * 4097 * 4,
        # loss block: scores read, pseudo labels / weights read, grad_scores written
        "head_losses": 2 * 8 * R * (C + 1) * 4 + 3 * R * (C + 1) * 4 + 3 * R * 6 + R * (C + 1) * 4,
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, smax, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons),
                    samples=len(sm))


# ------------------------------------------------------------------------------------ CPU arm
def literal_mask_utils(cfg):
    """The reference's LITERAL mask_utils double loop (one Python-level pair at a time, create_cob_iou.py:43-48)
    extrapolated to this workload by its pair count from the us/pair measured in the build container with the
    unmodified reference file (tools/literal_mask_utils_timing.py -> profiles/literal_mask_utils.json; the reference
    tree does not travel to the GPU box).  The CPU arm itself times the vectorised restatement (M . M^T)."""
    try:
        with open(os.path.join(ROOT, "profiles", "literal_mask_utils.json")) as f:
            t = json.load(f)
        us = t["sizes"][str(cfg["mask"])]["us_per_pair_both_maps"]
    except (OSError, ValueError, KeyError):
        return None
    return {"s_per_image": us * 1e-6 * cfg["R"] ** 2, "us_per_pair_iou_plus_asy": us,
            "measured_on": f"build container, 1 of {t['host_cores']} cores (the loop is single-threaded numpy), "
                           f"{t['n_masks']} masks of {cfg['mask']}^2", "pairs_per_image": cfg["R"] ** 2}


def cpu_reference(cfg, steps, warmup, sample_rois=128, head_grads=True):
    """The reference's algorithm for the path, restated for CPU (oracle/), timed on the host cores
    on a BOUNDED sample of the workload: one image; RoIAlign fwd+bwd and the mask overlap on
    `sample_rois` of its R proposals (cost scaled by R / sample_rois: both are linear in the
    number of rows processed); scoring and the 3 mining layers at full R."""
    import torch
    from cim_b200 import synth
    from oracle import heads_oracle, loss_oracle, roi_oracle
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    R, C, S = cfg["R"], cfg["C"], min(sample_rois, cfg["R"])
    Cf, H, W, scale = synth.feature_shape(cfg["backbone"])
    params = synth.proposal_params(R, 512, 1234)
    rois = synth.rois_from_params(params).numpy()
    feat = np.random.RandomState(0).randn(1, Cf, H, W).astype(np.float32)
    g_out = np.random.RandomState(1).randn(S, Cf, 7, 7).astype(np.float32)
    masks = synth.rasterize(params, out_size=cfg["mask"]).numpy().reshape(R, -1)
    mf = masks.astype(np.float32)
    torch.manual_seed(0)
    w = [np.random.RandomState(10 + i).uniform(-1 / 64, 1 / 64, (C + 1, 4096)).astype(np.float32) for i in range(8)]
    b = [np.zeros(C + 1, np.float32) for _ in range(8)]
    x = np.random.RandomState(2).randn(R, 4096).astype(np.float32)
    labels = synth.image_labels(C, cfg["present"], 1234).numpy()
    cmat = synth.cluster_mat(R, C, np.nonzero(labels[0])[0], 6, 1234).numpy()
    from oracle import mask_oracle
    iou16, asy16 = mask_oracle.mask_overlap_maps(masks[:, ::max(1, masks.shape[1] // 4096)])   # setup only

    def one_step():
        t0 = time.perf_counter()
        roi_oracle.roi_align_fwd(feat, rois[:S], 7, 7, scale, 0, True)
        roi_oracle.roi_align_bwd(g_out, rois[:S], feat.shape, scale, 0, True)
        t_roi = time.perf_counter() - t0
        t0 = time.perf_counter()
        inter = mf[:S] @ mf.T                                       # S x R intersection counts
        area = mf.sum(1)
        with np.errstate(divide="ignore", invalid="ignore"):
            (inter / (area[:S, None] + area[None, :] - inter)).astype(np.float16)
            (inter / area[None, :]).astype(np.float16)
        t_mask = time.perf_counter() - t0
        t0 = time.perf_counter()
        p_cls, p_det, r_cls, r_iou = heads_oracle.score_heads(x, w, b)
        t_score = time.perf_counter() - t0
        t0 = time.perf_counter()
        cls_l, det_l = [p_cls, r_cls[0], r_cls[1]], [p_det, r_iou[0], r_iou[1]]
        assigned = []
        for l in range(3):
            assigned.append(heads_oracle.cim_layer_forward(cls_l[l], det_l[l], labels, iou16, asy16, 0.1,
                                                           0.25 + 0.1 * l, 0.5 + 0.1 * l, 0.85, True))
        t_mine = time.perf_counter() - t0
        if head_grads:                                   # loss block fwd+bwd, then the scoring backward
            t0 = time.perf_counter()
            ok = [a[0] is not None for a in assigned]
            pl = np.stack([a[0] if o else np.zeros((R, C + 1), np.float32) for a, o in zip(assigned, ok)])[:, None]
            pi = np.stack([a[1] if o else np.zeros(R, np.float16) for a, o in zip(assigned, ok)])[:, None]
            lw = np.stack([a[2] if o else np.zeros(R, np.float32) for a, o in zip(assigned, ok)])[:, None]
            sc = np.stack([p_cls, p_det] + r_cls + r_iou)
            _, g = loss_oracle.head_losses(sc, pl, pi, lw, np.array(ok, np.uint8)[:, None], labels.reshape(1, -1), 3,
                                           dtype=torch.float32)
            _, g_pcl = loss_oracle.pcl_losses(p_cls, cmat[None], dtype=torch.float32)
            g[0] += g_pcl
            heads_oracle.score_heads_bwd(x, w, b, list(g))
            t_score += time.perf_counter() - t0
        return (t_roi + t_mask) * (R / S) + t_score + t_mine, dict(roi=t_roi * R / S, mask=t_mask * R / S,
                                                                   score=t_score, mine=t_mine)

    np.random.seed(3)
    for _ in range(warmup):
        one_step()
    per_image, parts = [], None
    t_wall = time.perf_counter()
    for _ in range(steps):
        t, parts = one_step()
        per_image.append(t)
    wall = time.perf_counter() - t_wall
    sec = float(np.mean(per_image))
    return dict(images_per_s=1.0 / sec, sec_per_image=sec, cores=ncpu, wall_s=wall, parts=parts,
                literal=literal_mask_utils(cfg),
                sample=f"1 image of {cfg['R']} proposals; RoIAlign fwd+bwd and mask overlap on {S} proposal rows "
                       f"(x{R / S:.1f}), scoring {'fwd+bwd + loss block' if head_grads else 'fwd'} + 3 mining layers at full size; "
                       f"numpy/OpenMP on all host cores")


# ------------------------------------------------------------------------------------ GPU arm
def build_inputs(cfg, dev, seed_base):
    import torch
    from cim_b200 import heads, mask_ops, synth
    n_img, R, C = cfg["n_img"], cfg["R"], cfg["C"]
    Cf, H, W, scale = synth.feature_shape(cfg["backbone"])
    gen = torch.Generator(device=dev).manual_seed(seed_base)
    feat = torch.randn(n_img, Cf, H, W, device=dev, generator=gen)
    grad_out = torch.randn(n_img * R, Cf, 7, 7, device=dev, generator=gen)
    seg_x = torch.randn(n_img * R, 4096, device=dev, generator=gen)
    rois, packed, packed_flat, labels, mats = [], [], [], [], []
    kb_per_row = cfg["mask"] // 16 if mask_ops.tiled_ok(cfg["mask"], cfg["mask"]) else 0
    for b in range(n_img):
        params = synth.proposal_params(R, 512, seed_base + b)
        rois.append(synth.rois_from_params(params, b))
        m = synth.rasterize(params, device=dev, out_size=cfg["mask"])
        packed.append(mask_ops.mask_pack(m))                         # tiled 8 x 16 patches when the size allows
        packed_flat.append(mask_ops.mask_pack(m, layout="flat").cpu())   # only to derive the host wire format
        labels.append(synth.image_labels(C, cfg["present"], seed_base + b))
        mats.append(synth.cluster_mat(R, C, np.nonzero(labels[-1][0].numpy())[0], 6, seed_base + b))
    torch.manual_seed(0)
    model = heads.cls_iou_model(4096, C + 1, 3).to(dev)
    weight, bias = (t.detach().contiguous() for t in model._stacked())
    labels = torch.cat(labels)
    packed_all = torch.stack(packed)
    # the resident input = the packed masks AND their metadata (areas, K-block occupancy), produced when the masks
    # are packed (mask_ops.mask_meta); the e2e path produces both on the copy stream of its input prefetch
    meta = mask_ops.mask_meta(packed_all, kb_per_row) if packed_all.shape[-1] % 4 == 0 else None
    return dict(feat=feat, rois=torch.cat(rois).to(dev), grad_out=grad_out, packed=packed_all, mask_meta=meta,
                packed_flat=torch.stack(packed_flat), kb_per_row=kb_per_row, mat=torch.stack(mats).to(dev),
                seg_x=seg_x, weight=weight, bias=bias, labels=labels.to(dev), labels_host=labels.numpy(),
                shape=(Cf, H, W, scale))


def measured_traffic(workload, stage):
    """DRAM bytes per launch of the stage's main kernel from the committed ncu --set full capture
    (profiles/traffic.json), or None when there is no capture for this workload / stage."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if t.get("workload") != workload or stage not in t or t.get("kernel_source_sha16") != source_sha16():
            return None                                  # no capture of THESE kernels on this workload: not a number
        return int(t[stage]["dram_read"] + t[stage]["dram_write"])
    except (OSError, ValueError, KeyError):
        return None


def visited_kblocks(step, cfg):
    """Number of 128-pixel K-blocks the tensor-core overlap kernel visited in its last launch (it leaves the
    count in the first 8 bytes of its workspace, include/cimhead.h) and the dense total: 128 x 256 tiles on or
    right of the diagonal x all K-blocks."""
    import torch
    torch.cuda.synchronize()
    visited = int(step.overlap_ws[:8].view(torch.int64).item())
    n, kblocks = cfg["R"], step.words // 4
    nrb, ncb = (n + 127) // 128, (n + 255) // 256
    tiles = sum(ncb - (i >> 1) for i in range(nrb))
    return visited, tiles * cfg["n_img"] * kblocks


def time_stages(step, inp, iters=5):
    """Per-stage device time (ms) with CUDA events, each stage launched back to back `iters` times."""
    import ctypes as C
    import torch
    from cim_b200 import _lib
    L, P, p = step.L, _lib.ptr, step.p
    st = _lib.stream_ptr(step.dev)
    n_img, R = step.n_img, step.R
    calls = {
        "roi_align_fwd": lambda: L.cim_roi_align_fwd(P(inp["feat"]), P(inp["rois"]), P(step.roi_out), n_img, step.Cf,
                                                     step.H, step.W, n_img * R, 7, 7, step.scale, 0, 1,
                                                     P(step.roi_ws), step.roi_ws.numel(), st),
        "roi_align_bwd": lambda: L.cim_roi_align_bwd(P(inp["grad_out"]), P(inp["rois"]), P(step.grad_feat), n_img,
                                                     step.Cf, step.H, step.W, n_img * R, 7, 7, step.scale, 0, 1,
                                                     P(step.roi_ws), step.roi_ws.numel(), st),
        "mask_overlap": lambda: L.cim_mask_overlap_meta(P(inp["packed"]), P(inp["mask_meta"]), n_img, R, step.words,
                                                        step.kb_per_row, None, P(step.area), P(step.iou), P(step.asy),
                                                        P(step.overlap_ws), step.overlap_ws.numel(), 0, st),
        "mask_meta": lambda: L.cim_mask_meta(P(inp["packed"]), n_img, R, step.words, step.kb_per_row,
                                             P(inp["mask_meta"]), inp["mask_meta"].numel(), st),
        "score_heads": lambda: L.cim_score_heads(P(inp["seg_x"]), P(inp["weight"]), P(inp["bias"]), P(step.scores),
                                                 n_img, R, step.D, step.C + 1, step.K, P(step.score_ws),
                                                 step.score_ws.numel(), st),
        "score_heads_bwd": lambda: L.cim_score_heads_bwd(P(inp["seg_x"]), P(inp["weight"]), P(step.scores),
                                                         P(step.grad_scores), P(step.grad_seg_x), P(step.grad_weight),
                                                         P(step.grad_bias), n_img, R, step.D, step.C + 1, step.K,
                                                         P(step.score_bwd_ws), step.score_bwd_ws.numel(), st),
        "head_losses": lambda: (L.cim_head_losses(P(step.scores), P(step.pseudo_labels), P(step.pseudo_iou),
                                                  P(step.loss_weights), P(step.valid), P(inp["labels"]), P(step.losses),
                                                  P(step.grad_scores), n_img, R, step.C, step.K, step.K, 3.0, 1.0, 3.0,
                                                  1.0 / n_img, st) or
                                L.cim_pcl_loss(P(step.scores), P(inp["mat"]), P(step.pcl_loss), P(step.grad_scores), n_img,
                                               R, step.C + 1, 255, 1.0 / n_img, 1, st)),
        "mine": lambda: L.cim_mine(C.byref(p), step.cls_ptrs, step.det_ptrs, P(inp["labels"]), P(step.iou),
                                   P(step.asy), P(step.gt_count), P(step.gt_rows), P(step.gt_class),
                                   P(step.gt_weight), P(step.asy_flag), P(step.mine_ws), step.mine_ws.numel(), st),
        "assign": lambda: L.cim_assign(C.byref(p), P(step.iou), P(step.gt_count), P(step.gt_rows), P(step.gt_class),
                                       P(step.gt_weight), None, P(step.pseudo_labels), P(step.pseudo_iou),
                                       P(step.loss_weights), P(step.valid), st),
    }
    if not step.head_grads:
        del calls["score_heads_bwd"], calls["head_losses"]
    if inp["mask_meta"] is None:
        del calls["mask_meta"]
    out = {}
    for name, fn in calls.items():
        _lib.check(fn(), name)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            _lib.check(fn(), name)
        e1.record()
        torch.cuda.synchronize()
        out[name] = e0.elapsed_time(e1) / iters
    return out


def source_sha16():
    """sha256[:16] over the CUDA sources: profiles/traffic.json records the value it was captured with, so a number
    measured on other kernels reads as stale instead of being copied into the bench line."""
    import glob
    import hashlib
    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(ROOT, "cim_b200", "csrc", "*.cu*"))):
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def timed(fn, steps, warmup, dev, cdist=None, finish=None):
    """CUDA events on the launching stream around `steps` calls, barrier + synchronize on both sides, max over ranks
    (cdist=None: this rank alone, no barrier).  finish: host work that belongs to the timed region's end (the RNG
    commit of the sync-free sampling mode)."""
    import torch
    for _ in range(warmup):
        fn()
    if finish is not None:
        finish()
    torch.cuda.synchronize()
    if cdist is not None:
        cdist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if finish is not None:
        finish()
    e1.record()
    torch.cuda.synchronize()
    if cdist is None:
        return e0.elapsed_time(e1) / steps
    cdist.barrier()
    return cdist.max_over_ranks(e0.elapsed_time(e1) / steps, dev)


#: the results CIMHeadStep.run leaves for its caller (see its docstring); the second group with head_grads=True
STEP_OUTPUTS = ("roi_out", "grad_feat", "iou", "asy", "scores", "pseudo_labels", "pseudo_iou", "loss_weights", "valid")
STEP_OUTPUTS_HEAD_GRADS = ("losses", "pcl_loss", "grad_scores", "grad_seg_x", "grad_weight", "grad_bias")
DUMP_ELEMS = 1 << 19


def dump_outputs(step, out_dir):
    """Write the results of the last step run on `step` to out_dir/<name>.npy as float32 (the float16 and uint8 ones
    convert exactly).  An array of more than DUMP_ELEMS elements is written as the DUMP_ELEMS elements at flat indices
    drawn from a fixed seed and sorted: the same indices in every run, so that two builds can be compared output for
    output.  At most 15 x 2 MiB in all."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name in STEP_OUTPUTS + (STEP_OUTPUTS_HEAD_GRADS if step.head_grads else ()):
        t = getattr(step, name).reshape(-1)
        if t.numel() > DUMP_ELEMS:
            t = t[torch.from_numpy(dump_indices(t.numel())).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def dump_indices(n):
    """The sorted flat indices dump_outputs writes of an array of n > DUMP_ELEMS elements."""
    # a generator of its own: numpy's global one drives the step's anti-noise sampling
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ELEMS, replace=False))


SAMPLING_NOTE = {
    "stream": "anti-noise sampling without a host hop: the device reads numpy's random stream from a ring the host "
              "fills ahead of time (cim_anti_noise_stream), pseudo-GT counts are read back with a lag, np.random is "
              "advanced at the end of the timed region (CIMHeadStep.sync_rng); bit-identical to the hop "
              "(tests/test_gpu_step.py); ms_per_step_sampling_hop = the same step with the hop",
    "hop": "pseudo-GT counts D2H, one np.random.random_sample call, uniforms H2D, cim_anti_noise",
}


def stage_table(stage_ms, bytes_img, n_img, peaks):
    table = {}
    for name, ms in stage_ms.items():
        gbs = bytes_img[name] * n_img / (ms * 1e-3) / 1e9
        table[name] = dict(ms=round(ms, 4), algorithmic_mb=round(bytes_img[name] * n_img / 1e6, 2),
                           gb_per_s=round(gbs, 1), hbm_frac=round(gbs / peaks["hbm_gbs"], 4))
    return table


def images_per_rank(name, cfg, world):
    """cfg3 (BASELINE.json configs[2]) is a FIXED batch of 64 images sharded per image over 2/4/8 GPUs: 64 / N images
    per rank (strong scaling); at N = 1 it runs the 8-GPU per-rank batch.  Every other workload is weak: its own
    n_img per rank."""
    if cfg.get("total_images") and world > 1:
        return max(1, cfg["total_images"] // world)
    return cfg["n_img"]


def measure_training(name, cfg, args, dev, rank, world, peaks, cdist, headline):
    """One training workload: the step in the model's dependency order (and, for the headline, in the overlapped
    order and end to end with host inputs), the per-stage table and the roofline of its dominant stage."""
    import torch
    from cim_b200 import mask_ops
    from cim_b200.step import CIMHeadStep, KERNELS_HEAD_GRADS, KERNELS_PCL, KERNELS_PER_STEP
    cfg = dict(cfg, n_img=images_per_rank(name, cfg, world))
    inp = build_inputs(cfg, dev, 1234 + 1000 * rank)
    Cf, H, W, scale = inp["shape"]
    words = inp["packed"].shape[-1]
    step = CIMHeadStep(cfg["n_img"], cfg["R"], cfg["C"], Cf, H, W, scale, words,
                       anti_noise_sampling=not args.no_anti_noise, device=dev, mask_kb_per_row=inp["kb_per_row"],
                       head_grads=not args.no_head_grads, order="graph", rng=args.sampling)
    mat = None if args.no_head_grads else inp["mat"]
    run = lambda order: step.run(inp["feat"], inp["rois"], inp["grad_out"], inp["packed"], inp["seg_x"], inp["weight"],
                                 inp["bias"], inp["labels"], mat=mat, order=order, mask_meta=inp["mask_meta"])
    steps, warmup = (args.steps, max(args.warmup, 3)) if headline else (max(3, min(args.steps, 10)), 3)
    np.random.seed(3)
    sampler = ClockSampler(dev.index or 0)
    if headline and rank == 0:
        sampler.start()
    ms_graph = timed(lambda: run("graph"), steps, warmup, dev, cdist, finish=step.sync_rng)
    clocks = sampler.stop() if headline and rank == 0 else None
    if headline and rank == 0 and args.dump_outputs:
        dump_outputs(step, args.dump_outputs)          # before the runs below overwrite the step's buffers
    ms_hop = None
    if args.sampling == "stream" and not args.no_anti_noise:
        step.rng = "hop"                       # same step, same buffers, the host hop instead of the device ring
        ms_hop = timed(lambda: run("graph"), steps, 2, dev, cdist)
        step.rng = "stream"
    ms_over = timed(lambda: run("overlapped"), steps, 2, dev, cdist, finish=step.sync_rng)
    n_images = cfg["n_img"] * world
    res = {"workload": name, "images_per_gpu": cfg["n_img"], "steps": steps, "warmup": warmup,
           "ms_per_step": ms_graph, "images_per_s": n_images / (ms_graph * 1e-3),
           "order": "graph: RoIAlign fwd -> scoring -> mining -> sampling hop -> assignment -> losses -> scoring bwd -> "
                    "RoIAlign bwd (model_builder.py:136-204); mask maps on a side stream next to the RoIAlign forward",
           "ms_per_step_overlapped_order": ms_over,
           "overlapped_order_note": "round-1 order: maps, scoring and mining first, the sampling hop hidden behind the "
                                    "RoIAlign forward; needs seg_x independent of this step's RoIAlign output",
           "sampling": SAMPLING_NOTE[args.sampling]}
    if ms_hop is not None:
        res["ms_per_step_sampling_hop"] = ms_hop
    if headline:
        res["clocks"] = clocks
        # end to end through the public call with HOST inputs (rois, labels, bbox-cropped bit-packed masks) and
        # results read back to the host every step
        crops = mask_ops.crops_from_packed_host(inp.pop("packed_flat").view(cfg["n_img"] * cfg["R"], -1), cfg["mask"],
                                                cfg["mask"])
        step.alloc_host_io(mask_hw=(cfg["mask"], cfg["mask"]),
                           crop_capacity_words=int(crops.words.numel() * 1.25) + 1024, prefetch_depth=args.prefetch_depth)
        step.hi_rois.copy_(inp["rois"])
        step.hi_labels.copy_(inp["labels"])
        step.set_host_crops(crops)
        if args.e2e_diag == "no-wait":         # diagnostic: the host never waits for a step's results
            step._collect_results = lambda: None
        run_host = lambda: step.run_host(inp["feat"], inp["grad_out"], inp["seg_x"], inp["weight"], inp["bias"],
                                         mat=mat, lag_results=True)
        # the step runs on a HIGH-priority stream: the prefetch of the next step's inputs (H2D + the crop-unpack kernel
        # on the step's low-priority copy stream) then only takes SMs the step's own kernels are not waiting for
        hp = torch.cuda.Stream(device=dev, priority=-1)
        hp.wait_stream(torch.cuda.current_stream(dev))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(hp):
            for _ in range(3):
                run_host()
            step.flush_results()
            step.sync_rng()
            cdist.barrier()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                run_host()             # reads the previous step's results on the host while this step computes
            step.flush_results()       # ... and the last step's: every timed step's H2D, D2H and host wait are inside
            step.sync_rng()            # sampling "stream": numpy's generator brought to where the steps left it
            e1.record()
            torch.cuda.synchronize()
        ms_e2e = cdist.max_over_ranks(e0.elapsed_time(e1) / steps, dev)
        res["e2e"] = {"value": n_images / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                      "h2d_bytes_per_step": int(step.h2d_bytes + step.last_mask_h2d_bytes +
                                                (step.last_uniform_bytes if step.rng == "hop" else 0)),
                      "uniform_ring": (None if step.rng == "hop" or args.no_anti_noise else
                                       f"{step.last_uniform_bytes} B per top-up of the device ring of random doubles; a top-up "
                                       f"lasts for {step.max_uniforms * 4} consumed doubles (a step consumes one per pseudo GT), "
                                       "not counted per step"),
                      "d2h_bytes_per_step": int(step.d2h_bytes),
                      "host_inputs": "rois, labels, bbox-cropped bit-packed proposal masks (unpacked on the device), the "
                                     "uniform doubles of the sampling hop; features/seg_x/grad_out are device-produced",
                      "host_outputs": "per-image losses [n_img, K+1, 3], valid flags, two checksums of the RoIAlign outputs, "
                                      "the pseudo-GT counts of the sampling hop" if not args.no_head_grads else
                                      "pseudo labels / IoU labels / loss weights, valid flags, checksums, pseudo-GT counts",
                      "pipelining": ("every call copies one full set of inputs host->device on a copy stream while the "
                                     "kernels of the current step run" +
                                     (" -- two steps ahead (prefetch_depth 2: into a pre-stage buffer, moved device-to-"
                                      "device into the next step's input buffer, whose crop unpack then always finds its "
                                      "data when the mining phase leaves the SMs idle)" if args.prefetch_depth == 2 else
                                      " -- one step ahead") +
                                     "; the results of step i are copied D2H at its end and read by the host (one event "
                                     "wait per step) while step i+1 runs; the last step's wait is inside the timed region"),
                      "prefetch_depth": args.prefetch_depth,
                      **({"DIAGNOSTIC": args.e2e_diag + ": not a result"} if args.e2e_diag else {}),
                      "order": "graph"}
        if step.trace is not None and rank == 0:             # host timeline of the last e2e steps (CIM_STEP_TRACE=1)
            ev = step.trace[-5 * 3:]
            for nm, t in ev:
                print(f"trace {nm:16s} {(t - ev[0][1]) * 1e3:8.3f} ms", file=sys.stderr)
        res["gpu_launches"] = (KERNELS_PER_STEP + (0 if args.no_head_grads else KERNELS_HEAD_GRADS + KERNELS_PCL)) * steps
        res["collective"] = (("none (single process)" if world == 1 else
                              f"NCCL allreduce (avg) of the {step.head_bucket.numel() * 4} B head-gradient bucket per "
                              "step, inside the timed region, overlapped with the RoIAlign backward")
                             if not args.no_head_grads else "none (head gradients excluded)")
    stages = time_stages(step, inp) if rank == 0 else None
    cdist.barrier()
    if rank == 0:
        bytes_img = algorithmic_bytes(cfg, Cf, H, W)
        if args.no_head_grads:
            del bytes_img["score_heads_bwd"], bytes_img["head_losses"]
        stage_ms = dict(stages)
        stage_ms["mine_assign"] = stage_ms.pop("mine") + stage_ms.pop("assign")
        if "mask_meta" in stage_ms:
            # NOT a stage of the step: per-mask areas / K-block occupancy are produced with the masks (data-set
            # packing; in the e2e path on the copy stream of the input prefetch, inside its timed region)
            res["mask_meta"] = {"ms": round(stage_ms.pop("mask_meta"), 4),
                                "note": "produced with the packed masks, outside the device-timed step; inside the "
                                        "e2e timed region (copy stream)"}
        table = stage_table(stage_ms, bytes_img, cfg["n_img"], peaks)
        dominant = max(stage_ms, key=stage_ms.get)
        total_bytes = sum(bytes_img.values())
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": table[dominant]["gb_per_s"],
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": table[dominant]["hbm_frac"],
                    "traffic": measured_traffic(name, dominant), "peak_source": peaks["source"],
                    "share_of_step": round(stage_ms[dominant] / sum(stage_ms.values()), 3)}
        visited, total = visited_kblocks(step, cfg)
        ov = {"executed_kblock_fraction": round(visited / max(total, 1), 4)}
        if visited:
            # a dense R x HW x R contraction of 0/1 operands (SURVEY 8d).  `executed` = the MMA flops actually issued
            # (visited K-blocks x 2*128*256*128); the kernel's instruction is tcgen05.mma.kind::mxf4 (E2M1 nibbles),
            # whose dense rate on this chip tools/micro/mxf4_check.cu measured (profiles/mxf4_peak.json).  The kernel is
            # NOT tensor-bound any more (DESIGN 4.3: operand loads, expansion and epilogue bound it), so this fraction
            # is reported for the record, next to the int8 rate the previous kernel was measured against.
            secs = stage_ms["mask_overlap"] * 1e-3
            executed = visited * 2.0 * 128 * 256 * 128
            peak_i8, note = tensor_peak(peaks)
            ov.update({"executed_tops": round(executed / secs / 1e12, 1), "tensor_peak_tops": round(peak_i8, 1),
                       "tensor_peak_source": note, "tensor_frac": round(executed / secs / 1e12 / peak_i8, 4),
                       "algorithmic_equivalent_tops": round(float(cfg["R"]) ** 2 * cfg["mask"] ** 2 * cfg["n_img"]
                                                            / secs / 1e12, 1)})
        table["mask_overlap"].update(ov)
        if dominant == "mask_overlap" and visited:
            roofline.update({"bound": "tensor", "achieved": ov["executed_tops"], "peak": ov["tensor_peak_tops"],
                             "unit": "TFLOP/s", "frac": ov["tensor_frac"], "peak_note": ov["tensor_peak_source"]})
        res.update({"roofline": roofline, "stages": table,
                    "step_roofline": {"algorithmic_mb_per_image": round(total_bytes / 1e6, 1),
                                      "hbm_frac": round(res["images_per_s"] / world * total_bytes / 1e9 / peaks["hbm_gbs"], 4)}})
    del step, inp
    torch.cuda.empty_cache()
    return res


def tensor_peak(peaks):
    """Dense tensor peak of THIS chip for the overlap kernel's instruction (tcgen05.mma.kind::mxf4, E2M1 operands):
    tools/micro/mxf4_check.cu's measurement when committed (profiles/mxf4_peak.json), else 4 x the measured bf16
    burst (the nominal fp4 : bf16 ratio), labelled as an assumption."""
    try:
        with open(os.path.join(ROOT, "profiles", "mxf4_peak.json")) as f:
            t = json.load(f)
        return float(t["mxf4_tops"]), f"measured, tools/micro/mxf4_check.cu ({t.get('how', '')})"
    except (OSError, ValueError, KeyError):
        return 4 * peaks["bf16_tflops"], "ASSUMED 4 x measured bf16 burst (no committed mxf4 measurement)"


def measure_inference(name, cfg, args, dev, rank, world, peaks, cdist):
    """BASELINE.json configs[4]: HRNet-W48 COCO pseudo-label generation, forward only (model_builder.py:209-211 returns
    after the heads in eval mode; tools/generate_mask_for_MaskRCNN.py:124-190): RoIAlign forward, scoring heads
    forward, K-head score mean (core/test.py:130-133) + per-class box NMS (mask_eval_utils.py:57-79)."""
    import torch
    from cim_b200 import _lib, postproc, synth
    Cf, H, W, scale = synth.feature_shape(cfg["backbone"])
    B, R, C1, K, D = cfg["n_img"], cfg["R"], cfg["C"] + 1, 3, 4096
    L = _lib.lib()
    P, st = _lib.ptr, _lib.stream_ptr(dev)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    rois = torch.cat([synth.rois_from_params(synth.proposal_params(R, 512, 1234 + 1000 * rank + b), b)
                      for b in range(B)]).to(dev)
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
        _lib.check(L.cim_roi_align_fwd(P(feat), P(rois), P(out), B, Cf, H, W, B * R, 7, 7, scale, 0, 1, P(ws),
                                       ws.numel(), st), "roi")

    def score():
        _lib.check(L.cim_score_heads(P(seg_x), P(weight), P(bias), P(scores), B, R, D, C1, K, P(sws), sws.numel(), st),
                   "score")

    def post():
        s = postproc.test_scores(scores, K)                       # [B*R, C]
        postproc.box_nms_batched(boxes, s.view(B, R, -1), 1e-5, 0.3)

    steps = max(3, min(args.steps, 10))
    ms = timed(lambda: (roi(), score(), post()), steps, 3, dev, cdist)
    res = {"workload": name, "images_per_gpu": B, "steps": steps, "warmup": 3, "ms_per_step": ms,
           "images_per_s": B * world / (ms * 1e-3), "order": "forward only: RoIAlign fwd -> scoring fwd -> K-head mean + "
           "per-class box NMS (80 classes x 4000 candidates with random-init scores: the NMS's worst case)"}
    if rank == 0:
        one = lambda fn: timed(fn, 5, 2, dev)
        stage_ms = {"roi_align_fwd": one(roi), "score_heads": one(score), "postproc": one(post)}
        F, O = Cf * H * W * 4, R * Cf * 49 * 4
        bytes_img = {"roi_align_fwd": F + 20 * R + O,
                     "score_heads": R * D * 4 + nh * C1 * (D + 1) * 4 + nh * R * C1 * 4,
                     "postproc": nh * R * C1 * 4 // 2 + R * 16 + R * (C1 - 1) * 5}
        table = stage_table(stage_ms, bytes_img, B, peaks)
        dominant = max(stage_ms, key=stage_ms.get)
        total_bytes = sum(bytes_img.values())
        res.update({"stages": table,
                    "roofline": {"kernel": dominant, "bound": "hbm", "achieved": table[dominant]["gb_per_s"],
                                 "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": table[dominant]["hbm_frac"],
                                 "traffic": None, "peak_source": peaks["source"]},
                    "step_roofline": {"algorithmic_mb_per_image": round(total_bytes / 1e6, 1),
                                      "hbm_frac": round(res["images_per_s"] / world * total_bytes / 1e9 / peaks["hbm_gbs"], 4)}})
    cdist.barrier()
    del out, seg_x, scores, feat
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline workload; the --also workloads time between 3 and 10 of "
                         "them, --impl reference at most 3")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_r50_voc_8x2000", choices=sorted(WORKLOADS))
    ap.add_argument("--also", default="cfg3_vgg16_voc_64,cfg4_r50_coco_8x2000_q,cfg5_hrnet48_coco_infer_8x4000",
                    help="comma-separated workloads measured after the headline one and reported under `workloads` "
                         "('' for none)")
    ap.add_argument("--sampling", default="stream", choices=["stream", "hop"],
                    help="anti-noise sampling: uniforms from a device ring filled ahead (no host sync inside the step) "
                         "or the host hop (counts down, draw, uniforms up)")
    ap.add_argument("--prefetch-depth", type=int, default=1, choices=[1, 2],
                    help="e2e input pipeline: host->device copies one or two steps ahead of the step that uses them")
    ap.add_argument("--e2e-diag", default="", choices=["", "no-wait"],
                    help="DIAGNOSTIC ONLY (the e2e number is then not a result): switch a piece of the host path off")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-anti-noise", action="store_true")
    ap.add_argument("--no-head-grads", action="store_true",
                    help="leave the loss block, the scoring backward and the allreduce of the head gradients out of the step")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps of the headline workload, write what its last timed step computed (rank "
                         f"0) as DIR/<name>.npy in float32; arrays of more than {DUMP_ELEMS} elements as a fixed, seeded "
                         "sample of that many")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path")
    # stdout carries exactly ONE line, the JSON result: everything else a library may write to fd 1 (NCCL prints its
    # version banner there on the first collective) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    cfg = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = dict(workload=args.workload, images_per_gpu=cfg["n_img"], proposals_per_image=cfg["R"],
                  classes=cfg["C"], backbone=cfg["backbone"], mask_px=cfg["mask"], sharding="per image, weak",
                  l2="per-step working set > 3 GB >> 126 MB L2, no explicit flush")

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = max(1, min(args.steps, 3)), 1          # bounded; one untimed pass warms BLAS / pages
        r = cpu_reference(cfg, steps, warmup, head_grads=not args.no_head_grads)
        emit(({
            "impl": "reference", "metric": METRIC, "value": r["images_per_s"], "unit": "images/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * r["sec_per_image"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": r["images_per_s"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                             "sample": r["sample"], "parts_s_per_image": r["parts"],
                             "literal_mask_utils_s_per_image": r["literal"]},
            "e2e": {"value": r["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    import torch
    from cim_b200 import dist as cdist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    rank, world, local = cdist.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    peaks = load_peaks()
    # one slice of the host cores per rank (before any pinned buffer is allocated) and as many numpy / torch host
    # threads as the slice has: eight ranks otherwise share cores for their launch loops and sampling hops
    cores = cdist.pin_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if cores:
        torch.set_num_threads(max(1, min(4, len(cores))))

    head = measure_training(args.workload, cfg, args, dev, rank, world, peaks, cdist, headline=True)
    others = {}
    for name in [n for n in args.also.split(",") if n and n != args.workload]:
        c = WORKLOADS[name]
        try:
            if c.get("inference"):
                others[name] = measure_inference(name, c, args, dev, rank, world, peaks, cdist)
            else:
                others[name] = measure_training(name, c, args, dev, rank, world, peaks, cdist, headline=False)
        except RuntimeError as exc:                              # e.g. out of memory on a smaller part: say so, go on
            others[name] = {"workload": name, "error": str(exc)[:300]}
            torch.cuda.empty_cache()
    cdist.barrier()
    cdist.shutdown()
    if rank != 0:
        return

    result = {
        "metric": METRIC, "value": head["images_per_s"], "unit": "images/s", "n_gpus": world, "steps": head["steps"],
        "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
        "step_order": head["order"], "ms_per_step_graph_order": head["ms_per_step"],
        "ms_per_step_overlapped_order": head["ms_per_step_overlapped_order"],
        "overlapped_order_note": head["overlapped_order_note"], "sampling": head["sampling"],
        "ms_per_step_sampling_hop": head.get("ms_per_step_sampling_hop"),
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "collective": head["collective"],
        "roofline": head["roofline"], "step_roofline": head["step_roofline"], "stages": head["stages"],
        "clocks": head["clocks"], "kernel_source_sha16": source_sha16(),
        "workloads": others,
    }
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(cfg, 1, 0, head_grads=not args.no_head_grads)
        result["cpu_baseline"] = {"value": r["images_per_s"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                                  "sample": r["sample"], "parts_s_per_image": r["parts"],
                                  "literal_mask_utils_s_per_image": r["literal"]}
    emit(result)


if __name__ == "__main__":
    main()
