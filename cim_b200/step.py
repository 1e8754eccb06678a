"""CIMHeadStep -- one CIM head step for a batch of images with every buffer pre-allocated.

This is the call a training loop makes per iteration once the backbone has produced its feature
map and MaskFuse its 4096-d proposal features; it covers the span of
Generalized_RCNN.forward / backward of the reference that BASELINE.json names
(lib/modeling/model_builder.py:136-204 + the RoIAlign backward inside loss.backward(),
tools/train.py:436):

    RoIAlign forward            model_builder.py:230-231
    mask IoU + containment maps model_builder.py:148-156 (there: two pickle loads per step)
    scoring heads               model_builder.py:143
    3 x mining + assignment     model_builder.py:170-187
    RoIAlign backward           autograd of the first line
    scoring heads backward      autograd of the third line (loss.backward(), tools/train.py:436) -> head
                                gradients, all-reduced over the ranks of a data-parallel run
                                (reference: comm.reduce_add_coalesced, lib/nn/parallel/_functions.py:39)

All device work goes through the C ABI (include/cimhead.h) on the current CUDA stream.  The one
host hop is the anti-noise sampling (heads.py:451-466, numpy global RNG); it is overlapped with
the RoIAlign kernels, which do not depend on it.
"""
import collections
import ctypes as C
import os
import time

import numpy as np
import torch

from . import _lib
from . import dist as cdist
from .heads import PCL_MAX_ID, UniformStream, draw_uniforms


class _nvtx:
    """NVTX range around a stage of the step (shows up in nsys / ncu --nvtx timelines of the REAL step)."""
    __slots__ = ("name",)

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_pop()
        return False

#: kernels (not memsets / copies) libcimhead launches in one run(): roi_align prep 1 + fwd 2 + bwd 2,
#: mask area + sort + overlap + 2 un-permutes = 5, scoring 3, mining 3, anti-noise sampling 1, assignment 1
KERNELS_PER_STEP = 18
#: + with head_grads: loss block (fwd + bwd), detector dot, activation backward, bias, W^T split, grad_x GEMM,
#: grad_W GEMM, reduce
KERNELS_HEAD_GRADS = 8
#: + with a cluster matrix: PCL_loss forward + backward
KERNELS_PCL = 1


class CIMHeadStep:
    def __init__(self, n_img, n_props, n_classes, feat_channels, feat_h, feat_w, spatial_scale, mask_words,
                 feat_dim=4096, refine_times=3, p_seed=0.1, step_rate=0.1, con_thr=0.85, anti_noise_sampling=True,
                 max_present=None, device="cuda:0", sampling_ratio=0, aligned=True, mask_kb_per_row=0,
                 head_grads=False, order="graph", rng="hop"):
        self.dev = torch.device(device)
        self.n_img, self.R, self.C, self.K = n_img, n_props, n_classes, refine_times
        self.Cf, self.H, self.W, self.scale = feat_channels, feat_h, feat_w, float(spatial_scale)
        self.words, self.D = mask_words, feat_dim
        # pixel order of the packed masks given to run(): W // 16 for the tiled 8 x 16 layout
        # (mask_ops.mask_pack's default whenever H % 8 == W % 16 == 0), 0 for flat row-major
        self.kb_per_row = int(mask_kb_per_row)
        self.sr, self.aligned = int(sampling_ratio), int(bool(aligned))
        self.anti = anti_noise_sampling
        self.p_seed = float(p_seed)
        self.n_props = None             # the device counts of the last run(): kept alive while its kernels may run
        self.feat_hw = None             # the device image extents of the last run(), likewise
        self.order = order
        if rng not in ("hop", "stream"):
            raise ValueError("rng must be 'hop' or 'stream'")
        self.rng = rng
        self.L = _lib.lib()
        R, C1, nh, k = n_props, n_classes + 1, 2 + 2 * refine_times, refine_times
        dev = self.dev
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
        with torch.cuda.device(dev):
            self.roi_out = e((n_img * R, feat_channels, 7, 7), torch.float32)
            self.grad_feat = e((n_img, feat_channels, feat_h, feat_w), torch.float32)
            self.roi_ws = e((self.L.cim_roi_align_workspace_bytes_ex(n_img, feat_channels, feat_h, feat_w, n_img * R,
                                                                     7, 7),), torch.uint8)
            self.iou = e((n_img, R, R), torch.float16)
            self.asy = e((n_img, R, R), torch.float16)
            self.area = e((n_img, R), torch.int32)
            self.overlap_ws = e((self.L.cim_mask_overlap_workspace_bytes(n_img, R, mask_words, 0),), torch.uint8)
            self.scores = e((nh, n_img * R, C1), torch.float32)
            # large enough for the padded and the compact form (the latter at N = n_img * R covers every N)
            self.score_ws = e((max(256, self.L.cim_score_heads_workspace_bytes(n_img, R, feat_dim, C1, k),
                                   self.L.cim_score_heads_compact_workspace_bytes(n_img, R, n_img * R, feat_dim, C1,
                                                                                  k)),), torch.uint8)
            self.head_grads = bool(head_grads)
            if self.head_grads:
                # grad_weight and grad_bias share one buffer: the bucket of the data-parallel allreduce
                self.head_bucket = e((nh * C1 * feat_dim + nh * C1,), torch.float32)
                self.grad_weight = self.head_bucket[:nh * C1 * feat_dim].view(nh, C1, feat_dim)
                self.grad_bias = self.head_bucket[nh * C1 * feat_dim:].view(nh, C1)
                self.grad_seg_x = e((n_img * R, feat_dim), torch.float32)
                self.score_bwd_ws = e((max(self.L.cim_score_heads_bwd_workspace_bytes(n_img, R, feat_dim, C1, k),
                                           self.L.cim_score_heads_bwd_compact_workspace_bytes(n_img, R, n_img * R,
                                                                                              feat_dim, C1, k)),),
                                      torch.uint8)
                self.losses = e((n_img, k + 1, 3), torch.float32)
                self.pcl_loss = torch.zeros((n_img,), dtype=torch.float32, device=dev)
                self.grad_scores = e((nh, n_img * R, C1), torch.float32)
                self.pcl_grad = e((n_img * R, C1), torch.float32)
            p = _lib.MineParams()
            p.n_img, p.R, p.C, p.C1, p.n_layers = n_img, R, n_classes, C1, k
            p.det_cols, p.mode = C1, 0
            p.keep_count = int(np.ceil(p_seed * R))                 # heads.py:332; the capacity for ragged batches
            # the pseudo-GT lists stay on the device (the sampling runs there, cim_anti_noise), so they get the full
            # capacity R: no overflow whatever the number of present classes (max_present is accepted and ignored)
            gcap = R
            p.gt_cap = gcap
            p.big_thr = float(np.float32(0.9 * R))                  # heads.py:338
            p.con_thr = con_thr
            for l in range(k):                                      # model_builder.py:90-93
                p.cls_thr[l], p.iou_thr[l] = 0.25 + step_rate * l, 0.5 + step_rate * l
            self.p = p
            self.mine_ws = e((max(256, self.L.cim_mine_workspace_bytes(C.byref(p))),), torch.uint8)
            self.gt_count = e((k, n_img), torch.int32)
            self.gt_rows = e((k, n_img, gcap), torch.int32)
            self.gt_class = e((k, n_img, gcap), torch.int32)
            self.gt_weight = e((k, n_img, gcap), torch.float32)
            self.asy_flag = e((n_img, R), torch.uint8)
            self.gt_keep = torch.ones((k, n_img, gcap), dtype=torch.uint8, device=dev)
            self.pseudo_labels = e((k, n_img, R, C1), torch.float32)
            self.pseudo_iou = e((k, n_img, R), torch.float16)
            self.loss_weights = e((k, n_img, R), torch.float32)
            self.valid = e((k, n_img), torch.uint8)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        self.h_count = pin((k, n_img), torch.int32)
        self.h_uniform = pin((k * n_img * gcap,), torch.float64)       # one double per pseudo GT at most
        with torch.cuda.device(dev):
            self.d_uniform = e((k * n_img * gcap,), torch.float64)
        self.ev = torch.cuda.Event()
        self.last_uniform_bytes = 0
        if self.rng == "stream" and self.anti:
            # sync-free sampling (cim_anti_noise_stream): a device ring of uniforms drawn ahead, two cursor words the
            # steps alternate between, the pseudo-GT counts read back with a lag of up to 2 steps
            self.max_uniforms = k * n_img * gcap
            ring_len = 16 * self.max_uniforms
            self.ustream = UniformStream(ring_len, self.max_uniforms)
            with torch.cuda.device(dev):
                self.d_ring = torch.zeros((ring_len,), dtype=torch.float64, device=dev)
                self.d_cursor = torch.zeros((2,), dtype=torch.int64, device=dev)
            self.h_ring = pin((8 * self.max_uniforms,), torch.float64)      # staging of one top-up
            self.ring_ev = torch.cuda.Event()
            self._ring_pending = False
            self._cursor_idx = 0
            self._cnt_slots = [(pin((k, n_img), torch.int32), torch.cuda.Event()) for _ in range(3)]
            self._cnt_next = 0
            self._cnt_q = collections.deque()
        self.side = torch.cuda.Stream(device=self.dev, priority=-2)     # scoring GEMM next to the overlap helpers: above the step
        self.side2 = torch.cuda.Stream(device=self.dev, priority=-2)    # graph order: PCL_loss next to the mining kernels
        self.ev_score = torch.cuda.Event()
        self.ev_premine = torch.cuda.Event()
        self.ev_prep = torch.cuda.Event()
        self.trace = [] if os.environ.get("CIM_STEP_TRACE") else None
        # layer l reads (cls, det) = (predict_cls, predict_det) for l = 0, else (ref_cls[l-1], ref_iou[l-1])
        s = self.scores.view(nh, n_img, R, C1)
        cls_src = [s[0]] + [s[2 + l - 1] for l in range(1, k)]
        det_src = [s[1]] + [s[2 + k + l - 1] for l in range(1, k)]
        PtrArr = C.c_void_p * k
        self.cls_ptrs = PtrArr(*[t.data_ptr() for t in cls_src])
        self.det_ptrs = PtrArr(*[t.data_ptr() for t in det_src])

    # -------------------------------------------------------------------------------------
    def run(self, feat, rois, grad_out, packed_masks, seg_x, weight, bias, labels, labels_host=None, grad_scores=None,
            mat=None, mid_hook=None, order=None, mask_meta=None, n_props=None, feat_hw=None, compact=False):
        """feat [n_img,Cf,H,W] f32, rois [n_img*R,5] f32 grouped by image, grad_out [n_img*R,Cf,7,7]
        f32, packed_masks [n_img,R,words] i32, seg_x [n_img*R,D] f32, weight [2+2K,C+1,D],
        bias [2+2K,C+1], labels [n_img,C] f32 (labels_host is no longer needed: the sampling runs on the device).
        Results land in self.roi_out, grad_feat, iou, asy, scores, pseudo_labels, pseudo_iou,
        loss_weights, valid.  With head_grads=True also losses [n_img, K+1, 3], grad_scores (the loss
        block's backward; pass grad_scores to supply dL/dscores yourself instead), grad_seg_x, grad_weight,
        grad_bias; in a multi-process run the head-gradient bucket is averaged over the ranks (one NCCL
        allreduce, overlapped with the RoIAlign backward).  mat [n_img, R, C+1] (the dataset's proposal-cluster
        matrix, model_builder.py:125,203) adds PCL_loss: pcl_loss [n_img] and its gradient on the classifier head.
        mask_meta: mask_ops.mask_meta(packed_masks), produced with the masks (data-set packing / input prefetch): the
        overlap stage then skips its own pass over the 524 MB of packed masks.
        n_props: proposals per image of a ragged batch (a host sequence / CPU tensor, validated and copied, or a CUDA
        int32 [n_img] tensor used as is; it may change from step to step).  R is then a capacity: image b owns rows
        [0, n_b) of its R rows, and every result of image b equals that of the image run alone at R = n_b (scores,
        pseudo labels, losses, PCL_loss, gradients; padding rows of all of them are 0).  Padding rows must hold finite
        seg_x, rois with the image's own index and finite coordinates, and grad_out rows of 0; the maps are computed
        for them but never read.  None: every image has R proposals.
        feat_hw: image sizes of a batch of differently sized images (a host [n_img, 2] sequence / array / CPU tensor,
        validated and copied, or a CUDA int32 [n_img, 2] tensor used as is; it may change from step to step).  feat is
        then a canvas of the constructor's (feat_h, feat_w): image b occupies feat[b, :, :H_b, :W_b], and its roi_out
        rows and grad_feat equal RoIAlign of that map alone (grad_feat is 0 outside it; the canvas there must be
        finite).  Nothing else of the step depends on it.  None: every image fills the canvas.
        compact: a compact ragged batch.  n_props must then be host counts (a sequence, numpy array or CPU tensor); with
        N = sum(n_props), image b's proposals are rows [off_b, off_b + n_b) (off_b = n_0 + ... + n_{b-1}) of rois,
        grad_out and seg_x, which have exactly N rows, and the results of those rows land in roi_out[:N] and
        grad_seg_x[:N].  RoIAlign, the scoring GEMMs and the caller's per-proposal head then process N rows instead of
        n_img * R; everything from the scores on (maps, mining, losses, PCL) keeps the padded capacity layout, with the
        same values as a padded call.  The buffers stay allocated at capacity, so N may change from step to step.

        order (default: the constructor's):
          "graph"      the model's dependency order (model_builder.py:136-204): RoIAlign forward -> scoring heads ->
                       mining -> sampling hop -> assignment -> losses -> scoring backward -> RoIAlign backward.  In
                       the real graph seg_x = Box_Head(RoIAlign output) feeds the heads, so nothing of the step can
                       hide the hop; the mask maps (which depend on the proposals only) run on the side stream next to
                       the RoIAlign forward and the scoring GEMM.
          "overlapped" mask maps, scoring and mining first, the RoIAlign forward launched BEFORE the host waits for
                       the mining result, so the hop hides behind it.  Only possible when seg_x does not depend on
                       this step's RoIAlign output (a bench with synthetic seg_x; features cached from an earlier
                       pass)."""
        L, p, dev = self.L, self.p, self.dev
        P, n_img, R, k = _lib.ptr, self.n_img, self.R, self.K
        order = order or self.order
        if order not in ("graph", "overlapped"):
            raise ValueError("order must be 'graph' or 'overlapped'")
        tr = self.trace                                         # host timeline (CIM_STEP_TRACE=1), else None
        if tr is not None:
            tr.append(("run", time.perf_counter()))
        st = _lib.stream_ptr(dev)
        side_st = C.c_void_p(self.side.cuda_stream)
        ck = _lib.check
        cur = torch.cuda.current_stream(dev)
        pcl_early = self.head_grads and grad_scores is None and mat is not None
        if compact:
            np_dev, n_rows = _lib.compact_rows_arg(n_props, n_img, R, dev)
            self.n_props = np_dev
            for name, t in (("rois", rois), ("grad_out", grad_out), ("seg_x", seg_x)):
                if t.shape[0] != n_rows:
                    raise ValueError(f"{name} of a compact batch must have sum(n_props) = {n_rows} rows, "
                                     f"got {t.shape[0]}")
        else:
            self.n_props = np_dev = _lib.n_props_arg(n_props, n_img, R, dev)
            n_rows = n_img * R
        self.feat_hw = hw = _lib.feat_hw_arg(feat_hw, n_img, self.H, self.W, dev)

        def pcl(stream):
            # PCL_loss (model_builder.py:203) needs predict_cls and the cluster matrix only: 8 CTAs of pure latency;
            # its gradient is added to head 0's after the loss block
            with _nvtx("cim/pcl_loss"):
                ck(L.cim_pcl_loss_ex(P(self.scores), P(mat), P(np_dev), P(self.pcl_loss), P(self.pcl_grad), n_img, R,
                                     self.C + 1, PCL_MAX_ID, 1.0 / n_img, 0, stream), "cim_pcl_loss")

        def score_fwd(stream, with_pcl):
            with _nvtx("cim/score_heads"):
                if compact:
                    ck(L.cim_score_heads_compact(P(seg_x), P(weight), P(bias), P(self.scores), P(np_dev), n_img, R,
                                                 n_rows, self.D, self.C + 1, k, P(self.score_ws),
                                                 self.score_ws.numel(), stream), "cim_score_heads_compact")
                else:
                    ck(L.cim_score_heads_ex(P(seg_x), P(weight), P(bias), P(self.scores), P(np_dev), n_img, R, self.D,
                                            self.C + 1, k, P(self.score_ws), self.score_ws.numel(), stream),
                       "cim_score_heads")
            if with_pcl and pcl_early:
                pcl(stream)

        def overlap(stream):
            with _nvtx("cim/mask_overlap"):
                ck(L.cim_mask_overlap_meta(P(packed_masks), P(mask_meta), n_img, R, self.words, self.kb_per_row, None,
                                           P(self.area), P(self.iou), P(self.asy), P(self.overlap_ws),
                                           self.overlap_ws.numel(), 0, stream), "cim_mask_overlap_meta")

        def roi_fwd():
            with _nvtx("cim/roi_align_fwd"):
                ck(L.cim_roi_align_fwd_prepared_ex(P(feat), P(rois), P(hw), None, P(self.roi_out), n_img, self.Cf,
                                                   self.H, self.W, n_rows, 7, 7, self.scale, self.sr, self.aligned,
                                                   P(self.roi_ws), self.roi_ws.numel(), st), "cim_roi_align_fwd")

        def mine():
            self.ev_premine.record(cur)        # from here on the GPU is mostly idle until the hop is over
            with _nvtx("cim/mine"):
                ck(L.cim_mine_ex(C.byref(p), P(np_dev), self.p_seed, self.cls_ptrs, self.det_ptrs, P(labels),
                                 P(self.iou), P(self.asy), P(self.gt_count), P(self.gt_rows), P(self.gt_class),
                                 P(self.gt_weight), P(self.asy_flag), P(self.mine_ws), self.mine_ws.numel(), st),
                   "cim_mine")
                if self.anti and self.rng == "stream":
                    hbuf, hev = self._cnt_slots[self._cnt_next]
                    self._cnt_next = (self._cnt_next + 1) % len(self._cnt_slots)
                    hbuf.copy_(self.gt_count, non_blocking=True)
                    hev.record(cur)
                    self._cnt_q.append((hbuf, hev))
                elif self.anti:
                    self.h_count.copy_(self.gt_count, non_blocking=True)
                    self.ev.record(cur)

        self.side.wait_stream(cur)
        if order == "graph":
            # the mask maps depend on the proposals only: side stream, next to the RoIAlign forward + scoring GEMM.
            # The side stream starts behind the ROI descriptors (window plans on large maps: six small kernels), so
            # the persistent RoIAlign forward is on the SMs before the overlap's tensor kernel asks for them -- which of
            # the two went first used to depend on launch timing (cfg3: 5.67 or 5.85 ms)
            with _nvtx("cim/roi_prepare"):
                ck(L.cim_roi_align_prepare_ex(P(rois), P(hw), n_img, self.Cf, self.H, self.W, n_rows, 7, 7,
                                              self.scale, self.sr, self.aligned, P(self.roi_ws), self.roi_ws.numel(),
                                              st), "cim_roi_align_prepare")
            self.ev_prep.record(cur)
            roi_fwd()
            self.side.wait_event(self.ev_prep)
            overlap(side_st)
            score_fwd(st, False)
            if pcl_early:
                # PCL on its own stream, next to the (equally latency-bound) mining kernels; joined before the losses
                self.ev_score.record(cur)
                self.side2.wait_event(self.ev_score)
                pcl(C.c_void_p(self.side2.cuda_stream))
            cur.wait_stream(self.side)
            mine()
        else:
            # the scoring GEMM (independent of the maps) runs on a side stream next to the overlap stage, whose small
            # serial helpers leave most of the GPU idle; RoI descriptors once per step, also off the critical path
            score_fwd(side_st, True)
            ck(L.cim_roi_align_prepare_ex(P(rois), P(hw), n_img, self.Cf, self.H, self.W, n_rows, 7, 7, self.scale,
                                          self.sr, self.aligned, P(self.roi_ws), self.roi_ws.numel(), side_st),
               "cim_roi_align_prepare")
            overlap(st)
            cur.wait_stream(self.side)
            mine()
            roi_fwd()
        if mid_hook is not None:
            mid_hook()                                          # host work that should hide behind the kernels in flight
        keep = None
        if tr is not None:
            tr.append(("launched_phase1", time.perf_counter()))
        if self.anti and self.rng == "stream":
            # no hop: the device takes its uniforms from the ring; the host only keeps the ring ahead of the steps
            with _nvtx("cim/sampling_stream"):
                self._ring_top_up(cur)
                ci = self._cursor_idx
                ck(L.cim_anti_noise_stream(C.byref(p), P(labels), P(self.gt_count), P(self.gt_class),
                                           P(self.gt_weight), P(self.d_ring), self.d_ring.numel(),
                                           P(self.d_cursor[ci:]), P(self.d_cursor[ci ^ 1:]), P(self.gt_keep), st),
                   "cim_anti_noise_stream")
                self._cursor_idx = ci ^ 1
            keep = self.gt_keep
        elif self.anti:
            # the sampling hop: pseudo-GT counts down (K * n_img ints), one random_sample call from numpy's global
            # RNG (heads.draw_uniforms), the uniforms up, cim_anti_noise on the device
            with _nvtx("cim/sampling_hop"):
                self.ev.synchronize()                           # mining is done
                if tr is not None:
                    tr.append(("mining_done", time.perf_counter()))
                u = draw_uniforms(self.h_count.numpy())
                self.last_uniform_bytes = int(u.size) * 8
                if u.size:
                    self.h_uniform.numpy()[:u.size] = u
                    self.d_uniform[:u.size].copy_(self.h_uniform[:u.size], non_blocking=True)
                ck(L.cim_anti_noise(C.byref(p), P(labels), P(self.gt_count), P(self.gt_class), P(self.gt_weight),
                                    P(self.d_uniform), P(self.gt_keep), st), "cim_anti_noise")
            keep = self.gt_keep
            if tr is not None:
                tr.append(("sampled", time.perf_counter()))
        if getattr(self, "_res_guard", False):
            cur.wait_event(self.res_ev)                         # run_host: the previous step's results have been read
            self._res_guard = False
        with _nvtx("cim/assign"):
            ck(L.cim_assign_ex(C.byref(p), P(np_dev), P(self.iou), P(self.gt_count), P(self.gt_rows),
                               P(self.gt_class), P(self.gt_weight), P(keep), P(self.pseudo_labels), P(self.pseudo_iou),
                               P(self.loss_weights), P(self.valid), st), "cim_assign")
        reduce_work = None
        if self.head_grads:
            if grad_scores is None:
                # losses forward + backward (model_builder.py:170-202): total of an image = sum_l cls + 3 iou + bag
                # + mil_bag; the batch loss is the mean over this rank's images
                with _nvtx("cim/head_losses"):
                    ck(L.cim_head_losses(P(self.scores), P(self.pseudo_labels), P(self.pseudo_iou),
                                         P(self.loss_weights), P(self.valid), P(labels), P(self.losses),
                                         P(self.grad_scores), n_img, R, self.C, k, k, 3.0, 1.0, 3.0, 1.0 / n_img, st),
                       "cim_head_losses")
                    if pcl_early:                                    # + PCL_loss on predict_cls
                        if order == "graph":
                            cur.wait_stream(self.side2)
                        self.grad_scores[0].add_(self.pcl_grad)
                grad_scores = self.grad_scores
            with _nvtx("cim/score_heads_bwd"):
                if compact:
                    ck(L.cim_score_heads_bwd_compact(P(seg_x), P(weight), P(self.scores), P(grad_scores), P(np_dev),
                                                     P(self.grad_seg_x), P(self.grad_weight), P(self.grad_bias), n_img,
                                                     R, n_rows, self.D, self.C + 1, k, P(self.score_bwd_ws),
                                                     self.score_bwd_ws.numel(), st), "cim_score_heads_bwd_compact")
                else:
                    ck(L.cim_score_heads_bwd_ex(P(seg_x), P(weight), P(self.scores), P(grad_scores), P(np_dev),
                                                P(self.grad_seg_x), P(self.grad_weight), P(self.grad_bias), n_img, R,
                                                self.D, self.C + 1, k, P(self.score_bwd_ws), self.score_bwd_ws.numel(),
                                                st), "cim_score_heads_bwd")
                reduce_work = cdist.allreduce_mean_async_(self.head_bucket)     # overlaps the RoIAlign backward
        with _nvtx("cim/roi_align_bwd"):
            ck(L.cim_roi_align_bwd_prepared_ex(P(grad_out), P(rois), P(hw), None, P(self.grad_feat), n_img, self.Cf,
                                               self.H, self.W, n_rows, 7, 7, self.scale, self.sr, self.aligned,
                                               P(self.roi_ws), self.roi_ws.numel(), st), "cim_roi_align_bwd")
        if reduce_work is not None:
            reduce_work()                                       # current stream waits for the allreduce
        if tr is not None:
            tr.append(("launched_phase2", time.perf_counter()))
        return self

    # -------------------------------------------------------------------------------------
    def _drain_counts(self, keep_unknown, keep_newest=0):
        """Read the pseudo-GT counts of finished steps (rng="stream"); wait until at most `keep_unknown` steps are
        left whose consumption is unknown.  keep_newest = 1 leaves the newest entry alone even if its copy has
        already landed: inside a step that entry is the step's OWN count, whose uniforms are only provisioned after
        this call."""
        q, us = self._cnt_q, self.ustream
        while len(q) > keep_newest and (len(q) > keep_unknown or q[0][1].query()):
            hbuf, hev = q.popleft()
            hev.synchronize()
            us.note_consumed(int(np.minimum(hbuf.numpy(), self.p.gt_cap).sum()))

    def _ring_top_up(self, cur):
        """Called once per step before cim_anti_noise_stream is enqueued (the step's own count copy is already in the
        queue): learn what finished steps consumed, draw ahead if the reserve could run out, upload in stream order
        (the ring slots overwritten belong to positions below `consumed`, i.e. to kernels that precede the copy)."""
        us = self.ustream
        self._drain_counts(keep_unknown=2, keep_newest=1)   # this step + at most one earlier step still running
        if not us.attached:
            us.attach()
        n = us.need(len(self._cnt_q))
        if n <= 0:
            return
        if self._ring_pending:
            self.ring_ev.synchronize()                  # the staging buffer of the previous top-up has been read
        pos, u = us.draw(n)
        self.h_ring.numpy()[:n] = u
        lo = pos % us.ring_len
        first = min(n, us.ring_len - lo)
        self.d_ring[lo:lo + first].copy_(self.h_ring[:first], non_blocking=True)
        if first < n:
            self.d_ring[:n - first].copy_(self.h_ring[first:n], non_blocking=True)
        self.ring_ev.record(cur)
        self._ring_pending = True
        self.last_uniform_bytes = n * 8

    def sync_rng(self):
        """rng="stream": wait for the steps in flight, advance numpy's global RandomState by the doubles they consumed
        (it is then where the reference's np.random.choice calls would have left it) and detach from it.  Call it
        before anything else draws from np.random (epoch boundaries: lib/roi_data/loader.py:_shuffle_roidb_inds) and
        before reading the generator's state.  No-op for rng="hop"."""
        if self.rng != "stream" or not self.anti:
            return
        self._drain_counts(keep_unknown=0)
        self.ustream.commit()

    # -------------------------------------------------------------------------------------
    def alloc_host_io(self, mask_hw=None, crop_capacity_words=0, prefetch_depth=1, ragged=False, compact=False,
                      rle_capacity_bytes=0):
        """Pinned host buffers of the end-to-end call: inputs that originate on the host in the
        reference's pipeline (rois, labels: lib/roi_data/minibatch.py:45-61; proposal masks:
        the COB .mat files of tools/pre) and the step's results.  Device-side input buffers are
        DOUBLE buffered and filled on a separate copy stream, so the host->device copy of step
        i+1 overlaps the kernels of step i (what a prefetching data loader does).
        rle_capacity_bytes > 0: the masks arrive as COCO compressed RLE strings instead (mask_ops.MaskRLE, set_host_rle:
        ~11x fewer bytes than the crops for COB-like proposals at 512 x 512), decoded on the device by
        cim_mask_unpack_rle_tiled_meta_sparse into the same buffer; it excludes crop_capacity_words and needs the tiled
        layout.  A malformed string gives an empty mask, and the step's results raise ValueError when they are
        collected: at the end of the run_host() call that ran the step, or with lag_results one call later (or in
        flush_results()), after that call's step has been enqueued.
        prefetch_depth = 2 (crops or RLE only): the host->device copy runs TWO steps ahead, into a third set of (small)
        wire buffers on its own stream; the copy into the step's input buffer is then a device-to-device copy at the start
        of the previous step, so the crop unpack can always run in that step's idle mining phase -- with eight ranks
        copying at once a rank's 60 MB take 2.5 ms instead of 1.3 (tools/h2d_bw.py) and the unpack used to slip behind
        the RoIAlign backward.  What run_host() finds in the pinned buffers at call t is then the input of step t + 2
        (the first call also uses it for steps t and t + 1).
        ragged: a pinned hi_n_props int32 [n_img] (initialised to R) joins the inputs: the proposal counts of the step,
        filled by the caller like hi_rois, validated when staged and carried with that step's rois, labels and masks
        through the double buffer and the pre-stage (run(n_props=...) for what a padding row must hold; with crops,
        mask_ops.batch_crops_host builds the wire format with empty crops for the padding rows).
        compact (with ragged): the batch is compact (run(compact=True)).  hi_rois holds the N = sum(hi_n_props) real rois
        in its first N rows and only those are copied; each staged step keeps its own host counts and N, and run_host()
        runs it with them (next_step_rows() tells how many rows its seg_x / grad_out need).  The masks stay padded."""
        k, n_img, R, C1 = self.K, self.n_img, self.R, self.C + 1
        if crop_capacity_words and rle_capacity_bytes:
            raise ValueError("the masks arrive as crops or as RLE strings, not both")
        if rle_capacity_bytes and not self.kb_per_row:
            raise ValueError("the RLE wire needs the tiled mask layout (mask_kb_per_row = W // 16)")
        if prefetch_depth not in (1, 2) or (prefetch_depth == 2 and not (crop_capacity_words or rle_capacity_bytes)):
            raise ValueError("prefetch_depth must be 1, or 2 with crop_capacity_words > 0 or rle_capacity_bytes > 0")
        self.prefetch_depth = prefetch_depth
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        self.hi_rois = pin((n_img * R, 5), torch.float32)
        self.hi_labels = pin((n_img, self.C), torch.float32)
        self.ragged = bool(ragged)
        if compact and not self.ragged:
            raise ValueError("compact host I/O needs ragged=True")
        self.compact = bool(compact)
        self.hi_n_props = pin((n_img,), torch.int32).fill_(R) if self.ragged else None
        # masks arrive either as full bit masks (hi_masks) or, with crop_capacity_words > 0, as
        # bounding-box crops (mask_ops.MaskCrops: ~8x fewer bytes over PCIe) that the device unpacks
        self.crop_cap = int(crop_capacity_words)
        self.rle_cap = int(rle_capacity_bytes)
        self.mask_hw = mask_hw
        if self.crop_cap:
            self.hi_masks = None
            self.hi_crop_words = pin((self.crop_cap,), torch.int32)
            self.hi_crop_meta = pin((n_img * R, 4), torch.int32)
            self.hi_crop_off = pin((n_img * R,), torch.int64)
            self.n_crop_words = 0
        elif self.rle_cap:
            self.hi_masks = None
            self.hi_rle_chars = pin((self.rle_cap,), torch.uint8)
            self.hi_rle_off = pin((n_img * R,), torch.int64)
            self.hi_rle_len = pin((n_img * R,), torch.int32).zero_()
            self.hi_rle_hw = pin((n_img, 2), torch.int32)
            self.n_rle_chars = 0
        else:
            self.hi_masks = pin((n_img, R, self.words), torch.int32)
        # what the host reads back every step: with the loss block in the step (head_grads) the step's result
        # is its losses -- the pseudo labels stay on the device, where the reference keeps them too
        # (model_builder.py:192-196); without it, the pseudo labels themselves
        self.ho_valid = pin((k, n_img), torch.uint8)
        if self.head_grads:
            self.ho_losses = pin((n_img, k + 1, 3), torch.float32)
            results = (self.ho_losses, self.ho_valid)
        else:
            self.ho_labels = pin((k, n_img, R, C1), torch.float32)
            self.ho_iou = pin((k, n_img, R), torch.float16)
            self.ho_weights = pin((k, n_img, R), torch.float32)
            results = (self.ho_labels, self.ho_iou, self.ho_weights, self.ho_valid)
        self.ho_checksum = pin((2,), torch.float32)
        if self.rle_cap:
            self.ho_bad = pin((1,), torch.int32)              # malformed strings among the step's masks
            results = results + (self.ho_bad,)
        with torch.cuda.device(self.dev):
            dv = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.dev)
            # masks: ZERO-filled when they are produced from crops or RLE -- the fused unpack is a sparse update that
            # only touches the rectangles of the mask a row held before (prev_rects) and of the new one
            mk = torch.zeros if self.crop_cap or self.rle_cap else torch.empty
            self.di = [dict(rois=dv((n_img * R, 5), torch.float32), labels=dv((n_img, self.C), torch.float32),
                            masks=mk((n_img, R, self.words), dtype=torch.int32, device=self.dev),
                            ready=torch.cuda.Event(), free=torch.cuda.Event()) for _ in range(2)]
            if self.ragged:
                for buf in self.di:
                    buf["n_props"] = dv((n_img,), torch.int32)
            if self.crop_cap:
                for buf in self.di:
                    buf.update(crop_words=dv((self.crop_cap,), torch.int32), crop_meta=dv((n_img * R, 4), torch.int32),
                               crop_off=dv((n_img * R,), torch.int64),
                               prev_rects=torch.zeros((n_img * R, 4), dtype=torch.int32, device=self.dev))
            if self.rle_cap:
                for buf in self.di:
                    buf.update(rle_chars=dv((self.rle_cap,), torch.uint8), rle_off=dv((n_img * R,), torch.int64),
                               rle_len=dv((n_img * R,), torch.int32), rle_hw=dv((n_img, 2), torch.int32),
                               prev_rects=torch.zeros((n_img * R, 4), dtype=torch.int32, device=self.dev),
                               bad=dv((1,), torch.int32))
                self.d_bad = torch.zeros((1,), dtype=torch.int32, device=self.dev)
            # mask metadata (areas, K-block bitmaps) produced on the copy stream right after the masks land
            self.use_meta = self.words % 4 == 0
            if self.use_meta:
                for buf in self.di:
                    buf["meta"] = dv((self.L.cim_mask_meta_bytes(n_img, R, self.words),), torch.uint8)
            self.d_checksum = dv((2,), torch.float32)
            self.copy_stream = torch.cuda.Stream(device=self.dev)
            if prefetch_depth == 2:
                self.pre = dict(rois=dv((n_img * R, 5), torch.float32), labels=dv((n_img, self.C), torch.float32),
                                n_words=0, valid=False, filled=torch.cuda.Event())
                if self.crop_cap:
                    self.pre.update(crop_words=dv((self.crop_cap,), torch.int32),
                                    crop_meta=dv((n_img * R, 4), torch.int32), crop_off=dv((n_img * R,), torch.int64))
                else:
                    self.pre.update(rle_chars=dv((self.rle_cap,), torch.uint8), rle_off=dv((n_img * R,), torch.int64),
                                    rle_len=dv((n_img * R,), torch.int32), rle_hw=dv((n_img, 2), torch.int32))
                if self.ragged:
                    self.pre["n_props"] = dv((n_img,), torch.int32)
                self.copy_stream2 = torch.cuda.Stream(device=self.dev)
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in (self.hi_rois, self.hi_labels))
        if self.ragged:
            self.h2d_bytes += self.hi_n_props.numel() * 4
        if self.hi_masks is not None:
            self.h2d_bytes += self.hi_masks.numel() * 4
        self.d2h_bytes = sum(t.numel() * t.element_size() for t in results + (self.ho_checksum,))
        # the sampling hop: pseudo-GT counts down, one double per pseudo GT up (self.last_uniform_bytes, set by run())
        self.d2h_bytes += self.h_count.numel() * 4
        self._slot = 0
        self._staged = False
        self.res_ev = torch.cuda.Event()
        self.ev_done = torch.cuda.Event()
        with torch.cuda.device(self.dev):
            self.res_stream = torch.cuda.Stream(device=self.dev)
        self._res_guard = False
        self.h2d_ev = torch.cuda.Event()
        self._h2d_pending = False
        self._pending = False
        self._bad_rle = 0
        self.results_host = None

    def wait_inputs_consumed(self):
        """Block until the last stage_host_inputs() has finished READING the pinned input buffers (hi_rois, hi_labels,
        hi_masks / hi_crop_* / hi_rle_*, hi_n_props).  The copies are asynchronous: refill those buffers for the following
        step only after this returns (set_host_crops() and set_host_rle() call it themselves)."""
        if getattr(self, "_h2d_pending", False):
            self.h2d_ev.synchronize()
            self._h2d_pending = False

    def set_host_crops(self, crops):
        """Copy a MaskCrops (CPU) of the n_img * R proposal masks into the pinned input buffers."""
        self.wait_inputs_consumed()
        n = crops.words.numel()
        if n > self.crop_cap:
            raise ValueError(f"{n} crop words exceed the capacity {self.crop_cap}")
        self.hi_crop_words[:n].copy_(crops.words)
        self.hi_crop_meta.copy_(crops.meta)
        self.hi_crop_off.copy_(crops.off)
        self.n_crop_words = n
        self.mask_hw = (crops.height, crops.width)

    def set_host_rle(self, rle):
        """Copy a MaskRLE (CPU; mask_ops.batch_rle_host) of the n_img * R proposal masks into the pinned input buffers
        (alloc_host_io(rle_capacity_bytes=...)).  Its canvas must be the step's: height * width == 32 * mask_words and
        width == 16 * mask_kb_per_row."""
        self.wait_inputs_consumed()
        n, rows = rle.chars.numel(), self.n_img * self.R
        if n > self.rle_cap:
            raise ValueError(f"{n} RLE characters exceed the capacity {self.rle_cap}")
        if rle.off.numel() != rows or rle.len.numel() != rows or tuple(rle.hw.shape) != (self.n_img, 2):
            raise ValueError(f"the RLE batch must have {rows} rows and {self.n_img} image sizes")
        if rle.height * rle.width != 32 * self.words or rle.width != 16 * self.kb_per_row:
            raise ValueError(f"the RLE canvas {rle.height} x {rle.width} is not the step's tiled mask canvas")
        self.hi_rle_chars[:n].copy_(rle.chars)
        self.hi_rle_off.copy_(rle.off)
        self.hi_rle_len.copy_(rle.len)
        self.hi_rle_hw.copy_(rle.hw)
        self.n_rle_chars = n
        self.mask_hw = (rle.height, rle.width)

    def stage_host_inputs(self, defer_kernels=False, direct=False):
        """Enqueue the host->device copy of the CURRENT contents of hi_rois / hi_labels / hi_masks
        into the idle device buffer, on the copy stream.  Call it for step i+1 before (or while)
        step i computes; run_host() consumes the staged buffer.
        defer_kernels: only the copies (copy engine) are enqueued now; the returned callable enqueues the kernels that
        turn them into the step's input (crop unpack + mask metadata) -- run_host() calls it from inside the step,
        behind `ev_premine`, so that they run next to the mining kernels and the sampling hop, which leave most SMs idle,
        instead of competing with the RoIAlign kernels (0.31 ms -> measured in tools/e2e_diag.py).
        direct (prefetch_depth = 2 only): copy the pinned buffers straight into the device buffer, bypassing and
        invalidating the pre-stage (a step that was not prefetched)."""
        buf = self.di[self._slot ^ 1] if self._staged else self.di[self._slot]
        if self.ragged:
            n = self.hi_n_props.numpy()
            if n.min() < 1 or n.max() > self.R:
                raise ValueError(f"hi_n_props must lie in [1, {self.R}], got [{n.min()}, {n.max()}]")

        def kernels(after=None):
            with torch.cuda.stream(self.copy_stream):
                if after is not None:
                    self.copy_stream.wait_event(after)
                if self.rle_cap:
                    # RLE strings -> tiled bit masks + their metadata, the same sparse update as the crops'
                    rc = self.L.cim_mask_unpack_rle_tiled_meta_sparse(
                        _lib.ptr(buf["rle_chars"]), buf["n_chars"], _lib.ptr(buf["rle_off"]), _lib.ptr(buf["rle_len"]),
                        _lib.ptr(buf["rle_hw"]), _lib.ptr(buf["masks"]), _lib.ptr(buf["prev_rects"]),
                        _lib.ptr(buf["meta"]), buf["meta"].numel(), self.n_img, self.R, self.mask_hw[0],
                        self.mask_hw[1], self.words, _lib.ptr(buf["bad"]), C.c_void_p(self.copy_stream.cuda_stream))
                    _lib.check(rc, "cim_mask_unpack_rle_tiled_meta_sparse")
                    buf["meta_done"] = True
                elif self.crop_cap:
                    fused = bool(self.kb_per_row) and self.use_meta and \
                        self.words * 32 == self.mask_hw[0] * self.mask_hw[1]
                    if fused:
                        # crops -> tiled bit masks + their metadata in one pass, as a sparse update of the buffer:
                        # the patches of the crops it held two steps ago are cleared, those of the new crops written
                        rc = self.L.cim_mask_unpack_crops_tiled_meta_sparse(
                            _lib.ptr(buf["crop_words"]), _lib.ptr(buf["crop_meta"]), _lib.ptr(buf["crop_off"]),
                            _lib.ptr(buf["masks"]), _lib.ptr(buf["prev_rects"]), _lib.ptr(buf["meta"]),
                            buf["meta"].numel(), self.n_img, self.R, self.mask_hw[0], self.mask_hw[1], self.words,
                            C.c_void_p(self.copy_stream.cuda_stream))
                        _lib.check(rc, "cim_mask_unpack_crops_tiled_meta_sparse")
                        buf["meta_done"] = True
                    else:
                        unpack = self.L.cim_mask_unpack_crops_tiled if self.kb_per_row else self.L.cim_mask_unpack_crops
                        buf["prev_rects"].zero_()     # (these entry points zero `masks` themselves; no rectangle list)
                        rc = unpack(_lib.ptr(buf["crop_words"]), _lib.ptr(buf["crop_meta"]), _lib.ptr(buf["crop_off"]),
                                    _lib.ptr(buf["masks"]), self.n_img * self.R, self.mask_hw[0], self.mask_hw[1],
                                    self.words, C.c_void_p(self.copy_stream.cuda_stream))
                        _lib.check(rc, "cim_mask_unpack_crops")
                        buf["meta_done"] = False
                if self.use_meta and not buf["meta_done"]:
                    _lib.check(self.L.cim_mask_meta(_lib.ptr(buf["masks"]), self.n_img, self.R, self.words,
                                                    self.kb_per_row, _lib.ptr(buf["meta"]), buf["meta"].numel(),
                                                    C.c_void_p(self.copy_stream.cuda_stream)), "cim_mask_meta")
                buf["ready"].record(self.copy_stream)

        def h2d(dst, stream):
            """pinned input buffers -> dst (a device input buffer or the pre-stage); returns the crop word / RLE
            character count"""
            if self.compact:
                dst["counts"] = self.hi_n_props.numpy().copy()        # this step's host counts travel with it
                dst["N"] = int(dst["counts"].sum())
                dst["rois"][:dst["N"]].copy_(self.hi_rois[:dst["N"]], non_blocking=True)
            else:
                dst["rois"].copy_(self.hi_rois, non_blocking=True)
            dst["labels"].copy_(self.hi_labels, non_blocking=True)
            if self.ragged:
                dst["n_props"].copy_(self.hi_n_props, non_blocking=True)
            n = 0
            if self.crop_cap:
                n = self.n_crop_words
                dst["crop_words"][:n].copy_(self.hi_crop_words[:n], non_blocking=True)
                dst["crop_meta"].copy_(self.hi_crop_meta, non_blocking=True)
                dst["crop_off"].copy_(self.hi_crop_off, non_blocking=True)
                self.last_mask_h2d_bytes = n * 4 + self.hi_crop_meta.numel() * 4 + self.hi_crop_off.numel() * 8
            elif self.rle_cap:
                n = self.n_rle_chars
                dst["rle_chars"][:n].copy_(self.hi_rle_chars[:n], non_blocking=True)
                for key in ("rle_off", "rle_len", "rle_hw"):
                    dst[key].copy_(getattr(self, "hi_" + key), non_blocking=True)
                self.last_mask_h2d_bytes = n + sum(getattr(self, "hi_" + k).numel() * getattr(self, "hi_" + k).element_size()
                                                   for k in ("rle_off", "rle_len", "rle_hw"))
            else:
                dst["masks"].copy_(self.hi_masks, non_blocking=True)
                dst["meta_done"] = False
            self.h2d_ev.record(stream)                         # the pinned input buffers have been read
            self._h2d_pending = True
            return n

        pre = getattr(self, "pre", None) if self.prefetch_depth == 2 else None
        if pre is not None and direct:
            pre["valid"] = False
            pre = None
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(buf["free"])          # its previous consumer has finished
            if pre is not None and pre["valid"]:
                # the input of this buffer's step arrived a step ago: device-to-device
                self.copy_stream.wait_event(pre["filled"])
                n = pre["n_words"]
                wire = ("crop_meta", "crop_off") if self.crop_cap else ("rle_off", "rle_len", "rle_hw")
                for key in ("rois", "labels") + wire + (("n_props",) if self.ragged else ()):
                    buf[key].copy_(pre[key], non_blocking=True)
                if self.compact:
                    buf["counts"], buf["N"] = pre["counts"], pre["N"]
                big = "crop_words" if self.crop_cap else "rle_chars"
                buf[big][:n].copy_(pre[big][:n], non_blocking=True)
                buf["n_chars"] = n
            else:
                buf["n_chars"] = h2d(buf, self.copy_stream)
        if pre is not None:
            # ... and the pinned buffers (the input of the step after that one) go to the pre-stage on their own stream,
            # so that a slow copy never sits in front of the unpack kernel
            with torch.cuda.stream(self.copy_stream2):
                # after the device-to-device copy out of the pre-stage / after the copy stream's own read of the
                # pinned buffers (h2d_ev, recorded below, then covers both readers)
                self.copy_stream2.wait_stream(self.copy_stream)
                pre["n_words"] = h2d(pre, self.copy_stream2)
                pre["filled"].record(self.copy_stream2)
                pre["valid"] = True
        if defer_kernels:
            return kernels
        kernels()
        return self

    def _collect_results(self):
        """Host side of the result read-back: wait for the D2H copies of the last enqueued step and keep a
        host copy of what the training loop logs (losses / valid flags / checksums)."""
        if not self._pending:
            return
        self.res_ev.synchronize()
        self.results_host = {"valid": self.ho_valid.numpy().copy(), "checksum": self.ho_checksum.numpy().copy()}
        if self.head_grads:
            self.results_host["losses"] = self.ho_losses.numpy().copy()
        if self.rle_cap:
            self._bad_rle = self.results_host["bad_rle"] = int(self.ho_bad[0])
        self._pending = False

    def _raise_bad_rle(self):
        """The RLE wire: raise for the malformed strings of the step whose results were collected last."""
        n, self._bad_rle = self._bad_rle, 0
        if n:
            raise ValueError(f"{n} malformed RLE string(s) among the step's proposal masks: those masks were empty")

    def flush_results(self):
        """With lag_results: wait for the results of the last run_host() call (self.results_host)."""
        self._collect_results()
        self._raise_bad_rle()
        return self.results_host

    def next_step_rows(self):
        """alloc_host_io(compact=True): N, the rows of seg_x / grad_out that the next run_host() call needs -- the
        proposal count of the step it runs (staged earlier, or the pinned buffers' if nothing is staged)."""
        if self._staged:
            return self.di[self._slot]["N"]
        return int(self.hi_n_props.numpy().sum())

    def run_host(self, feat, grad_out, seg_x, weight, bias, prefetch_next=True, grad_scores=None, mat=None,
                 lag_results=False, feat_hw=None):
        """End-to-end step: host rois / labels / bit-packed masks -> device, the step, results ->
        host.  With alloc_host_io(ragged=True) the proposal counts (hi_n_props) travel with the step's inputs and the
        batch is ragged (run(n_props=...)).  feat / seg_x / grad_out are produced on the device by the backbone, MaskFuse
        and autograd in the real pipeline and therefore stay device tensors; so does feat_hw, the image sizes of a
        canvas-padded feat (run(feat_hw=...)), which goes straight through to run().  With alloc_host_io(compact=True)
        the step runs compact with the counts staged with its inputs: seg_x and grad_out must have that step's N rows
        (next_step_rows()), else ValueError before the step is enqueued.
        With prefetch_next the copy of the NEXT step's inputs (whatever is in the pinned input
        buffers now) is enqueued on the copy stream first, so it overlaps this step's kernels;
        every call therefore moves one full set of inputs host->device."""
        cur_stream = torch.cuda.current_stream(self.dev)
        if not self._staged:                                   # first call: nothing was prefetched
            self.stage_host_inputs(direct=True)
            self._staged = True
        buf = self.di[self._slot]
        if self.compact:
            for name, t in (("seg_x", seg_x), ("grad_out", grad_out)):
                if t.shape[0] != buf["N"]:
                    raise ValueError(f"{name} must have the {buf['N']} rows of the step being run, got {t.shape[0]}")
        finish_stage = None
        if prefetch_next:
            finish_stage = self.stage_host_inputs(defer_kernels=True)      # copies now, the other buffer
        cur_stream.wait_event(buf["ready"])
        compact = self.compact
        self.run(feat, buf["rois"][:buf["N"]] if compact else buf["rois"], grad_out, buf["masks"], seg_x, weight, bias,
                 buf["labels"], None, grad_scores=grad_scores, mat=mat, mask_meta=buf.get("meta"),
                 n_props=buf["counts"] if compact else buf.get("n_props"), feat_hw=feat_hw, compact=compact,
                 mid_hook=lambda: ((finish_stage(self.ev_premine) if finish_stage else None),
                                   (self._collect_results() if lag_results else None)))
        if self.rle_cap:
            self.d_bad.copy_(buf["bad"])                       # read before the buffer's next unpack overwrites it
        buf["free"].record(cur_stream)
        # two sparse checksums of the RoIAlign outputs ride along with the losses (a few hundred elements each, summed
        # straight into the result buffer).  roi_out is the first thing the next step overwrites, so its checksum stays on
        # the step's stream; everything else of the read-back -- the other checksum and the device -> host copies --
        # runs on a results stream behind `ev_done`, so the next step's first kernels do not queue behind the copies.
        # The next step waits for `res_ev` right before the first kernel that overwrites a result (cim_assign).
        ro, gf = (self.roi_out[:buf["N"]] if compact else self.roi_out).reshape(-1), self.grad_feat.view(-1)
        torch.sum(ro[::max(1, ro.numel() // 509)], dim=0, out=self.d_checksum[0])
        self.ev_done.record(cur_stream)
        with torch.cuda.stream(self.res_stream):
            self.res_stream.wait_event(self.ev_done)
            torch.sum(gf[::max(1, gf.numel() // 251)], dim=0, out=self.d_checksum[1])
            if self.head_grads:
                self.ho_losses.copy_(self.losses, non_blocking=True)
            else:
                self.ho_labels.copy_(self.pseudo_labels, non_blocking=True)
                self.ho_iou.copy_(self.pseudo_iou, non_blocking=True)
                self.ho_weights.copy_(self.loss_weights, non_blocking=True)
            self.ho_valid.copy_(self.valid, non_blocking=True)
            self.ho_checksum.copy_(self.d_checksum, non_blocking=True)
            if self.rle_cap:
                self.ho_bad.copy_(self.d_bad, non_blocking=True)
            self.res_ev.record(self.res_stream)
        self._res_guard = True
        self._pending = True
        if not lag_results:
            self._collect_results()                            # the host reads the results every step
        if prefetch_next:
            self._slot ^= 1
        else:
            self._staged = False
        self._raise_bad_rle()
        return self
