"""CIM heads with the reference's Python surface, backed by libcimhead.so.

Mirrors lib/modeling/heads.py of the reference:
  * cls_iou_model (heads.py:168-219): same constructor, same parameter names (`classifier`,
    `detector`, `refine_cls.k`, `refine_iou.k`, so reference checkpoints load), same forward
    return convention; the 2+2K linear layers + softmax / column-softmax / sigmoid run as one
    fused scoring call (cim_score_heads).
  * CIM_layer (heads.py:222-503): same constructor and forward signature, same return
    convention ((pseudo_labels, pseudo_iou_labels, loss_weights) or (None, None, None));
    mining, mask NMS and assignment run in cim_mine / cim_assign.
  * mine_and_assign(): the batched entry point (all images x all refinement layers in one go)
    that model_builder.py:170-187 would call instead of looping over CIM_layer objects.

Anti-noise sampling (heads.py:440-473) draws from numpy's GLOBAL RandomState on the host in the
reference.  To reproduce its pseudo labels bit for bit the same uniform doubles are drawn here from
the same global stream (one random_sample call per step, the reference's order: image-major, then
layer, then ascending class) between the two device phases, and cim_anti_noise restates
RandomState.choice's arithmetic on the device; that costs one small device->host->device hop per
step (the pseudo-GT counts down, the uniforms up).  _anti_noise_keep is the host restatement of the
same draw the tests compare the kernel with.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib


# ------------------------------------------------------------------------------- scoring
class ScoreHeadsFunction(Function):
    """scores[h] = act_h(x @ W_h^T + b_h) for the 2+2K heads; see cim_score_heads in cimhead.h.
    n_props (optional): proposals per image of a ragged batch (_lib.n_props_arg); image b owns rows [0, n_b) of its R
    rows, the detector softmax runs over those and every head is 0 on the others (cim_score_heads_ex).
    capacity (compact ragged batch, cim_score_heads_compact): x holds only the N = sum(n_props) real rows, image b's at
    [off_b, off_b + n_b); n_props must then be host counts (_lib.compact_rows_arg).  The scores come back padded to
    [2+2K, n_img * capacity, C1] as with n_props alone, and the backward returns grad_x [N, D]."""

    @staticmethod
    def forward(ctx, x, weight, bias, n_img, k, n_props=None, capacity=None):
        _lib.require_cuda(x, "seg_feature", torch.float32)
        _lib.require_cuda(weight, "weight", torch.float32)
        _lib.require_cuda(bias, "bias", torch.float32)
        x, weight, bias = x.contiguous(), weight.contiguous(), bias.contiguous()
        m, d = x.shape
        nh, c1, _ = weight.shape
        L = _lib.lib()
        if capacity is not None:
            R = int(capacity)
            with torch.cuda.device(x.device):
                n_props, n = _lib.compact_rows_arg(n_props, n_img, R, x.device)
                if m != n:
                    raise ValueError(f"a compact seg_feature must have sum(n_props) = {n} rows, got {m}")
                scores = torch.empty((nh, n_img * R, c1), dtype=torch.float32, device=x.device)
                ws = torch.empty(L.cim_score_heads_compact_workspace_bytes(n_img, R, n, d, c1, k), dtype=torch.uint8,
                                 device=x.device)
                rc = L.cim_score_heads_compact(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(scores),
                                               _lib.ptr(n_props), n_img, R, n, d, c1, k, _lib.ptr(ws), ws.numel(),
                                               _lib.stream_ptr(x.device))
            _lib.check(rc, "cim_score_heads_compact")
            ctx.save_for_backward(x, weight, scores)
            ctx.cfg = (n_img, k, n_props, R)
            return scores
        if m % n_img:
            raise ValueError("rows of seg_feature must be n_img * R")
        with torch.cuda.device(x.device):
            n_props = _lib.n_props_arg(n_props, n_img, m // n_img, x.device)
            scores = torch.empty((nh, m, c1), dtype=torch.float32, device=x.device)
            ws = torch.empty(L.cim_score_heads_workspace_bytes(n_img, m // n_img, d, c1, k), dtype=torch.uint8,
                             device=x.device)
            rc = L.cim_score_heads_ex(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(scores),
                                      _lib.ptr(n_props), n_img, m // n_img, d, c1, k, _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr(x.device))
        _lib.check(rc, "cim_score_heads")
        ctx.save_for_backward(x, weight, scores)
        ctx.cfg = (n_img, k, n_props, None)
        return scores

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        """cim_score_heads_bwd: activation backward + grad_x / grad_weight / grad_bias in one call
        (autograd of heads.py:194-219)."""
        x, weight, s = ctx.saved_tensors
        n_img, k, n_props, capacity = ctx.cfg
        nh, m, c1 = s.shape
        n, d = x.shape
        grad = _lib.require_cuda(grad, "grad_scores", torch.float32).contiguous()
        L = _lib.lib()
        need_x, need_w, need_b = ctx.needs_input_grad[:3]
        with torch.cuda.device(x.device):
            gx = torch.empty_like(x) if need_x else None
            gw = torch.empty_like(weight) if need_w else None
            gb = torch.empty((nh, c1), dtype=torch.float32, device=x.device) if need_b else None
            if capacity is not None:
                ws = torch.empty(L.cim_score_heads_bwd_compact_workspace_bytes(n_img, capacity, n, d, c1, k),
                                 dtype=torch.uint8, device=x.device)
                rc = L.cim_score_heads_bwd_compact(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(s), _lib.ptr(grad),
                                                   _lib.ptr(n_props), _lib.ptr(gx), _lib.ptr(gw), _lib.ptr(gb), n_img,
                                                   capacity, n, d, c1, k, _lib.ptr(ws), ws.numel(),
                                                   _lib.stream_ptr(x.device))
            else:
                ws = torch.empty(L.cim_score_heads_bwd_workspace_bytes(n_img, m // n_img, d, c1, k), dtype=torch.uint8,
                                 device=x.device)
                rc = L.cim_score_heads_bwd_ex(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(s), _lib.ptr(grad),
                                              _lib.ptr(n_props), _lib.ptr(gx), _lib.ptr(gw), _lib.ptr(gb), n_img,
                                              m // n_img, d, c1, k, _lib.ptr(ws), ws.numel(), _lib.stream_ptr(x.device))
        _lib.check(rc, "cim_score_heads_bwd")
        return gx, gw, gb, None, None, None, None


class cls_iou_model(nn.Module):
    """heads.cls_iou_model(dim_in, dim_out, refine_times, class_agnostic=False) (heads.py:168-219)."""

    def __init__(self, dim_in, dim_out, refine_times, class_agnostic=False):
        super().__init__()
        self.classifier = nn.Linear(dim_in, dim_out)
        self.detector = nn.Linear(dim_in, dim_out)
        self.refine_cls = nn.ModuleList([nn.Linear(dim_in, dim_out) for _ in range(refine_times)])
        self.refine_iou = nn.ModuleList([nn.Linear(dim_in, dim_out) for _ in range(refine_times)])

    def detectron_weight_mapping(self):
        return {name: name for name, _ in self.named_parameters()}, []

    def _stacked(self):
        layers = [self.classifier, self.detector, *self.refine_cls, *self.refine_iou]
        return torch.stack([l.weight for l in layers]), torch.stack([l.bias for l in layers])

    def forward_batched(self, seg_feature, n_img=1, n_props=None, capacity=None):
        """seg_feature [n_img*R, D] -> scores [2+2K, n_img*R, C1] (detector softmax per image).  n_props: proposals
        per image of a ragged batch (R is then a capacity; see ScoreHeadsFunction).  capacity=R: a compact ragged batch,
        seg_feature [sum(n_props), D] holds the real proposals only (image b's at rows [off_b, off_b + n_b)), n_props
        are host counts, and the scores come back padded [2+2K, n_img*R, C1]."""
        if seg_feature.dim() == 4:
            seg_feature = seg_feature.squeeze(3).squeeze(2)
        weight, bias = self._stacked()
        return ScoreHeadsFunction.apply(seg_feature, weight, bias, n_img, len(self.refine_cls), n_props, capacity)

    def forward(self, seg_feature):
        k = len(self.refine_cls)
        s = self.forward_batched(seg_feature, 1)
        return s[0], s[1], [s[2 + i] for i in range(k)], [s[2 + k + i] for i in range(k)]


# ------------------------------------------------------------------- mining + assignment
def _anti_noise_keep(gt_cls, gt_w, present):
    """heads.py:451-466 on the host: per present class (ascending) with at least one pseudo GT,
    np.random.choice(class_idx, size=n, replace=True, p=w / w.sum()) from the GLOBAL numpy RNG;
    the unique draws survive.

    The draw is spelled out the way RandomState.choice makes it for replace=True with p given
    (numpy/random/mtrand.pyx: cdf = p.cumsum(); cdf /= cdf[-1]; uniform = random_sample(n);
    idx = cdf.searchsorted(uniform, side='right')): it consumes the same n doubles of the global stream and
    returns the same indices, without choice()'s argument validation, which is 2/3 of its cost at these sizes
    (this hop sits on the step's critical path).  tests/test_host_logic.py checks the equivalence.

    A class whose pseudo GTs ALL have weight 0 (cls * det underflowed to 0 for every one of them, which a confident
    head produces) is a deliberate divergence: np.random.choice raises ValueError on p = 0/0 and stops the reference's
    training; here the class keeps its first pseudo GT and still consumes its n doubles, so the classes and steps
    after it draw the doubles they would draw had the class been sampled.  cim_anti_noise does the same on the
    device."""
    keep = np.ones(gt_cls.shape[0], dtype=np.uint8)
    for c in present:
        class_idx = np.nonzero(gt_cls == c)[0]
        if len(class_idx) == 0:
            continue
        prob = gt_w[class_idx]
        if prob.sum() == 0:
            np.random.random_sample(len(class_idx))
            keep[class_idx] = 0
            keep[class_idx[0]] = 1
            continue
        cdf = (prob / prob.sum()).astype(np.float64).cumsum()
        cdf /= cdf[-1]
        drawn = class_idx[cdf.searchsorted(np.random.random_sample(len(class_idx)), side="right")]
        keep[class_idx] = 0
        keep[drawn] = 1
    return keep


def draw_uniforms(counts):
    """The host half of the sampling hop: ONE np.random.random_sample(T) call from numpy's GLOBAL RandomState with
    T = total number of pseudo GTs.  The reference calls np.random.choice(idx, size=n, p=...) once per (image, layer,
    present class) (heads.py:459); each of those consumes exactly n doubles of the stream (mtrand.pyx: uniform =
    random_sample(n)), n summing to T over the step, so one call of T doubles leaves the global stream where the
    reference leaves it and hands out the same numbers in the same order (tests/test_host_logic.py)."""
    return np.random.random_sample(int(counts.sum()))


class UniformStream:
    """Host half of the sync-free sampling mode (cim_anti_noise_stream, CIMHeadStep(rng="stream")): doubles of numpy's
    GLOBAL RandomState stream drawn ahead of time through a clone of its state.

    Positions are absolute indices into the stream numpy's global generator will produce from the moment of
    attach(); `drawn` = first position not handed out yet, `consumed` = first position no FINISHED step has used
    (learned from lagged read-backs of the pseudo-GT counts), `committed` = position the global generator itself
    has been advanced to.  commit() advances the global generator by consumed - committed doubles -- after it
    np.random is exactly where the reference's per-class np.random.choice calls (heads.py:459) would have left it --
    and detaches: if other code draws from np.random BETWEEN commit() and the next step, the values drawn ahead but not
    consumed are dropped and the next step clones the global state again, so those draws keep their place in the stream
    (if nobody drew, the reserve is still the stream's continuation and is kept).  Other
    code must not draw from np.random between a step and the following commit()."""

    def __init__(self, ring_len, max_per_step):
        if ring_len < 16 * max_per_step:
            raise ValueError("ring_len must be >= 16 * max_per_step")
        self.ring_len, self.max_per_step = int(ring_len), int(max_per_step)
        self.rs = None
        self.drawn = self.consumed = self.committed = 0
        self._left_at = None            # np.random's state right after the last commit()

    @property
    def attached(self):
        return self.rs is not None and self._left_at is None

    def attach(self):
        """Follow numpy's global generator from its CURRENT state; the stream continues at `consumed`.  If the
        generator is still where the last commit() left it (nobody else drew from it), the reserve drawn ahead before
        that commit is still the continuation of the stream and is kept; otherwise it is dropped and the state is
        cloned again (the next draw() then refills the ring from position `consumed`)."""
        assert self.consumed == self.committed, "commit() before attaching again"
        if self.rs is not None and self._left_at is not None and _same_state(np.random.get_state(), self._left_at):
            self._left_at = None
            return
        self.rs = np.random.RandomState()
        self.rs.set_state(np.random.get_state())
        self.drawn = self.consumed
        self._left_at = None

    def need(self, steps_unknown):
        """Doubles to draw now so that a step launched next cannot run past `drawn`, whatever the `steps_unknown`
        steps in flight (consumption not read back yet) and the step itself consume; 0 if the reserve suffices.
        Top-ups come in blocks of 4 * max_per_step (numpy draws ~8 ns per double: a rare burst, off the GPU's path)."""
        want = (steps_unknown + 1) * self.max_per_step
        have = self.drawn - self.consumed
        if have >= want:
            return 0
        n = max(want - have, 4 * self.max_per_step)
        assert have + n <= self.ring_len - self.max_per_step, "ring too small for the steps in flight"
        return n

    def draw(self, n):
        """n more doubles of the stream -> (absolute position of the first, float64 array)."""
        pos = self.drawn
        out = self.rs.random_sample(int(n))
        self.drawn += int(n)
        return pos, out

    def note_consumed(self, n):
        self.consumed += int(n)
        assert self.consumed <= self.drawn, "a step consumed more uniforms than were drawn ahead"

    def commit(self):
        """Every step's consumption is known (the caller waited for the read-backs): bring np.random there and detach
        (the reserve survives if the generator is found in this very state at the next attach())."""
        n = self.consumed - self.committed
        if n:
            np.random.random_sample(n)
        self.committed = self.consumed
        self._left_at = np.random.get_state() if self.rs is not None else None


def _same_state(a, b):
    return a[0] == b[0] and a[2:] == b[2:] and np.array_equal(a[1], b[1])


def anti_noise_device(p, labels, gt_count, gt_class, gt_weight, gt_keep, stream=None):
    """Anti-noise sampling (heads.py:440-473) with only the random numbers coming from the host: read the pseudo-GT
    counts (sync point; the reference syncs per class, heads.py:453,457), draw the uniforms, run cim_anti_noise."""
    dev = gt_count.device
    counts = gt_count.cpu().numpy()
    u = draw_uniforms(np.minimum(counts, p.gt_cap))
    uni = torch.from_numpy(u if u.size else np.zeros(1)).to(dev)
    rc = _lib.lib().cim_anti_noise(C.byref(p), _lib.ptr(labels), _lib.ptr(gt_count), _lib.ptr(gt_class),
                                   _lib.ptr(gt_weight), _lib.ptr(uni), _lib.ptr(gt_keep),
                                   stream if stream is not None else _lib.stream_ptr(dev))
    _lib.check(rc, "cim_anti_noise")
    return gt_keep


def mine_and_assign(cls_scores, det_scores, labels, iou_map, asy_iou_map, cls_thr, iou_thr, p_seed=0.1,
                    con_thr=0.85, anti_noise_sampling=True, using_cim=True, n_props=None):
    """All images x all refinement layers of CIM_layer.forward in two device phases.

    cls_scores / det_scores: lists (one per layer) of [n_img, R, C1] float32 CUDA tensors -- layer 0
    gets (predict_cls, predict_det), layer l > 0 gets (ref_cls[l-1], ref_iou[l-1])
    (model_builder.py:176-187).  labels [n_img, C]; iou_map / asy_iou_map [n_img, R, R] float16.
    cls_thr / iou_thr: per-layer thresholds (model_builder.py:90-93).
    Returns dict(pseudo_labels [L,n_img,R,C+1] f32, pseudo_iou_labels [L,n_img,R] f16,
    loss_weights [L,n_img,R] f32, valid [L,n_img] uint8 (0 where the reference returns None),
    asy_iou_flag [n_img,R] uint8, gt_count [L,n_img] int32).
    n_props: proposals per image of a ragged batch (_lib.n_props_arg).  Image b is then mined from rows [0, n_b) as
    if it were alone at R = n_b (keep_count and the big-proposal threshold from n_b, the same numpy stream); its rows
    >= n_b get the ignore row and asy_iou_flag 0, and the maps' rows and columns >= n_b are never read."""
    n_layers = len(cls_scores)
    if n_layers < 1 or n_layers > _lib.MAX_LAYERS:
        raise ValueError(f"1..{_lib.MAX_LAYERS} layers supported")
    cls_scores = [_lib.require_cuda(t, "cls_scores", torch.float32).contiguous() for t in cls_scores]
    dev = cls_scores[0].device
    n_img, R, c1 = cls_scores[0].shape
    labels = _lib.require_cuda(labels, "labels").to(torch.float32).reshape(n_img, -1).contiguous()
    n_cls = labels.shape[1]
    if using_cim:
        if asy_iou_map is None:
            raise ValueError("CIM_label needs asy_iou_map (heads.py:383)")
        det_scores = [_lib.require_cuda(t, "det_scores", torch.float32).contiguous() for t in det_scores]
    elif det_scores is not None and det_scores[0] is not None:
        det_scores = [_lib.require_cuda(t, "det_scores", torch.float32).contiguous() for t in det_scores]
    else:
        det_scores = None
    if iou_map is None:
        raise NotImplementedError("the box-IoU fallback of heads.py:287-289,375-377 is not on the CIM path")
    iou_map = _lib.require_cuda(iou_map, "iou_map", torch.float16).contiguous()
    if asy_iou_map is not None:
        asy_iou_map = _lib.require_cuda(asy_iou_map, "asy_iou_map", torch.float16).contiguous()
    if tuple(iou_map.shape) != (n_img, R, R):
        raise ValueError("iou_map must be [n_img, R, R]")

    p = _lib.MineParams()
    p.n_img, p.R, p.C, p.C1, p.n_layers = n_img, R, n_cls, c1, n_layers
    p.det_cols = det_scores[0].shape[-1] if det_scores is not None else c1
    p.gt_cap = R
    p.mode = 0 if using_cim else 1
    p.keep_count = int(np.ceil(p_seed * R))                      # heads.py:332 (with n_props: the capacity)
    p.big_thr = float(np.float32(0.9 * R))                       # heads.py:338
    p.con_thr = con_thr
    for l in range(n_layers):
        p.cls_thr[l], p.iou_thr[l] = cls_thr[l], iou_thr[l]

    L = _lib.lib()
    n_props = _lib.n_props_arg(n_props, n_img, R, dev)
    PtrArr = C.c_void_p * n_layers
    cls_ptrs = PtrArr(*[t.data_ptr() for t in cls_scores])
    det_ptrs = PtrArr(*[t.data_ptr() for t in det_scores]) if det_scores is not None else None
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        ws = torch.empty(max(L.cim_mine_workspace_bytes(C.byref(p)), 256), dtype=torch.uint8, device=dev)
        gt_count = torch.empty((n_layers, n_img), dtype=torch.int32, device=dev)
        gt_rows = torch.empty((n_layers, n_img, R), dtype=torch.int32, device=dev)
        gt_class = torch.empty((n_layers, n_img, R), dtype=torch.int32, device=dev)
        gt_weight = torch.empty((n_layers, n_img, R), dtype=torch.float32, device=dev)
        asy_flag = torch.ones((n_img, R), dtype=torch.uint8, device=dev)
        if n_props is not None and asy_iou_map is None:
            asy_flag[:, :] = (torch.arange(R, device=dev) < n_props[:, None]).to(torch.uint8)
        rc = L.cim_mine_ex(C.byref(p), _lib.ptr(n_props), float(p_seed), cls_ptrs, det_ptrs, _lib.ptr(labels),
                           _lib.ptr(iou_map), _lib.ptr(asy_iou_map), _lib.ptr(gt_count), _lib.ptr(gt_rows),
                           _lib.ptr(gt_class), _lib.ptr(gt_weight), _lib.ptr(asy_flag), _lib.ptr(ws), ws.numel(), st)
        _lib.check(rc, "cim_mine")

        gt_keep = None
        if anti_noise_sampling:
            gt_keep = torch.empty((n_layers, n_img, R), dtype=torch.uint8, device=dev)
            anti_noise_device(p, labels, gt_count, gt_class, gt_weight, gt_keep)

        pseudo_labels = torch.empty((n_layers, n_img, R, n_cls + 1), dtype=torch.float32, device=dev)
        pseudo_iou = torch.empty((n_layers, n_img, R), dtype=torch.float16, device=dev)
        loss_weights = torch.empty((n_layers, n_img, R), dtype=torch.float32, device=dev)
        valid = torch.empty((n_layers, n_img), dtype=torch.uint8, device=dev)
        rc = L.cim_assign_ex(C.byref(p), _lib.ptr(n_props), _lib.ptr(iou_map), _lib.ptr(gt_count), _lib.ptr(gt_rows),
                             _lib.ptr(gt_class), _lib.ptr(gt_weight), _lib.ptr(gt_keep), _lib.ptr(pseudo_labels),
                             _lib.ptr(pseudo_iou), _lib.ptr(loss_weights), _lib.ptr(valid), st)
        _lib.check(rc, "cim_assign")
    return dict(pseudo_labels=pseudo_labels, pseudo_iou_labels=pseudo_iou, loss_weights=loss_weights,
                valid=valid, asy_iou_flag=asy_flag, gt_count=gt_count, gt_rows=gt_rows, gt_class=gt_class,
                gt_weight=gt_weight, gt_keep=gt_keep)


class CIM_layer(nn.Module):
    """heads.CIM_layer(p_seed=0.1, cls_thr=0.25, iou_thr=0.5, con_thr=0.85, Anti_noise_sampling=True)
    (heads.py:222-235); forward signature and return convention of heads.py:409-503."""

    def __init__(self, p_seed=0.1, cls_thr=0.25, iou_thr=0.5, con_thr=0.85, Anti_noise_sampling=True):
        super().__init__()
        self.p_seed = p_seed
        self.cls_thr = cls_thr
        self.nms_thr = cls_thr          # heads.py:227
        self.iou_thr = iou_thr
        self.con_thr = con_thr
        self.Anti_noise_sampling = Anti_noise_sampling

    @torch.no_grad()
    def forward(self, predict_cls, predict_det, rois, labels, iou_map=None, asy_iou_map=None, using_CIM=True):
        # rois only feed gt_boxes in the reference, which nothing downstream reads when maps are given
        out = mine_and_assign([predict_cls.unsqueeze(0)],
                              [predict_det.unsqueeze(0)] if predict_det is not None else None,
                              labels.reshape(1, -1), iou_map.unsqueeze(0) if iou_map is not None else None,
                              asy_iou_map.unsqueeze(0) if asy_iou_map is not None else None,
                              [self.cls_thr], [self.iou_thr], p_seed=self.p_seed, con_thr=self.con_thr,
                              anti_noise_sampling=self.Anti_noise_sampling, using_cim=using_CIM)
        if int(out["valid"][0, 0].item()) == 0:                   # heads.py:429-430
            return None, None, None
        return out["pseudo_labels"][0, 0], out["pseudo_iou_labels"][0, 0], out["loss_weights"][0, 0]


# ------------------------------------------------------------------------------- losses
class HeadLossFunction(Function):
    """cim_head_losses: the loss block of model_builder.py:170-202 (heads.cls_iou_loss per refinement layer +
    heads.mil_bag_loss) forward AND backward in one launch.  Returns (total [n_img], losses [n_img, K+1, 3]);
    only `total` = sum_l cls + iou_weight * sum_l iou + sum_l bag + mil_bag per image is differentiable."""

    @staticmethod
    def forward(ctx, scores, pseudo_labels, pseudo_iou, loss_weights, valid, labels, k, lmda0, lmda_rest, iou_weight):
        _lib.require_cuda(scores, "scores", torch.float32)
        _lib.require_cuda(pseudo_labels, "pseudo_labels", torch.float32)
        _lib.require_cuda(pseudo_iou, "pseudo_iou_labels", torch.float16)
        _lib.require_cuda(loss_weights, "loss_weights", torch.float32)
        _lib.require_cuda(valid, "valid", torch.uint8)
        scores, pseudo_labels, pseudo_iou = scores.contiguous(), pseudo_labels.contiguous(), pseudo_iou.contiguous()
        loss_weights, valid = loss_weights.contiguous(), valid.contiguous()
        n_layers, n_img, R, c1 = pseudo_labels.shape
        labels = _lib.require_cuda(labels, "labels").to(torch.float32).reshape(n_img, c1 - 1).contiguous()
        if tuple(scores.shape) != (2 + 2 * k, n_img * R, c1):
            raise ValueError("scores must be [2+2K, n_img*R, C+1]")
        with torch.cuda.device(scores.device):
            losses = torch.empty((n_img, k + 1, 3), dtype=torch.float32, device=scores.device)
            grad = torch.empty_like(scores)
            rc = _lib.lib().cim_head_losses(_lib.ptr(scores), _lib.ptr(pseudo_labels), _lib.ptr(pseudo_iou),
                                            _lib.ptr(loss_weights), _lib.ptr(valid), _lib.ptr(labels), _lib.ptr(losses),
                                            _lib.ptr(grad), n_img, R, c1 - 1, k, n_layers, float(lmda0),
                                            float(lmda_rest), float(iou_weight), 1.0, _lib.stream_ptr(scores.device))
        _lib.check(rc, "cim_head_losses")
        ctx.save_for_backward(grad)
        ctx.shape = (n_img, R)
        total = losses[:, :, 0].sum(1) + iou_weight * losses[:, :, 1].sum(1) + losses[:, :, 2].sum(1)
        ctx.mark_non_differentiable(losses)
        return total, losses

    @staticmethod
    @once_differentiable
    def backward(ctx, g_total, _g_losses):
        (grad,) = ctx.saved_tensors
        n_img, R = ctx.shape
        nh, _, c1 = grad.shape
        g = grad.view(nh, n_img, R, c1) * g_total.view(1, n_img, 1, 1)
        return (g.view_as(grad),) + (None,) * 9


def head_losses(scores, assigned, labels, k, lmda=(3.0, 1.0), iou_weight=3.0):
    """Loss block for a batch: `scores` from cls_iou_model.forward_batched, `assigned` the dict returned by
    mine_and_assign.  Returns dict(total [n_img] (differentiable), cls_loss, iou_loss, bag_loss [n_img] as
    model_builder.py:198-202 accumulates them (iou_loss already x iou_weight), losses [n_img, K+1, 3])."""
    total, losses = HeadLossFunction.apply(scores, assigned["pseudo_labels"], assigned["pseudo_iou_labels"],
                                           assigned["loss_weights"], assigned["valid"], labels, k, lmda[0], lmda[1],
                                           iou_weight)
    return dict(total=total, losses=losses, cls_loss=losses[:, :, 0].sum(1), iou_loss=iou_weight * losses[:, :, 1].sum(1),
                bag_loss=losses[:, :, 2].sum(1))


class PCLLossFunction(Function):
    """cim_pcl_loss: heads.PCL_loss (heads.py:10-41) forward + backward in one launch, n_img images at once."""

    @staticmethod
    def forward(ctx, predict_cls, mat, n_img, max_id, n_props=None):
        _lib.require_cuda(predict_cls, "predict_cls", torch.float32)
        _lib.require_cuda(mat, "mat", torch.float32)
        predict_cls, mat = predict_cls.contiguous(), mat.contiguous()
        m, c1 = predict_cls.shape
        R = m // n_img
        if mat.numel() != m * c1 or m % n_img:
            raise ValueError("mat must be [n_img, R, C+1] matching predict_cls [n_img*R, C+1]")
        with torch.cuda.device(predict_cls.device):
            n_props = _lib.n_props_arg(n_props, n_img, R, predict_cls.device)
            loss = torch.empty((n_img,), dtype=torch.float32, device=predict_cls.device)
            grad = torch.empty_like(predict_cls)
            rc = _lib.lib().cim_pcl_loss_ex(_lib.ptr(predict_cls), _lib.ptr(mat), _lib.ptr(n_props), _lib.ptr(loss),
                                            _lib.ptr(grad), n_img, R, c1, int(max_id), 1.0, 0,
                                            _lib.stream_ptr(predict_cls.device))
        _lib.check(rc, "cim_pcl_loss")
        ctx.save_for_backward(grad)
        ctx.shape = (n_img, R)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        n_img, R = ctx.shape
        return (grad.view(n_img, R, -1) * g.view(n_img, 1, 1)).view_as(grad), None, None, None, None


#: cluster ids cim_pcl_loss accepts (its per-row id lists hold 8-bit ids); CIMHeadStep passes the same constant
PCL_MAX_ID = 255


def PCL_loss(predict_cls, mat, labels=None, n_img=1, max_id=PCL_MAX_ID, strict=False, n_props=None):
    """heads.PCL_loss(predict_cls, mat, labels) (heads.py:10-41; `labels` only supplied the device there).
    n_img = 1 returns a 0-d loss like the reference; n_img > 1 (predict_cls [n_img*R, C+1], mat [n_img, R, C+1])
    returns one loss per image.  A cluster matrix the kernel cannot take (an id above max_id, a non-integer id, more
    than four distinct ids in a row, two background ids -- the reference asserts on the last) gives a NaN loss and a
    zero gradient for that image; strict=True turns that into a RuntimeError (one host sync).  n_props: proposals per
    image of a ragged batch (_lib.n_props_arg); rows r >= n_b of an image join no cluster whatever mat holds there."""
    loss = PCLLossFunction.apply(predict_cls, mat, n_img, max_id, n_props)
    if strict and bool(torch.isnan(loss.detach()).any()):
        raise RuntimeError("cim_pcl_loss: cluster matrix outside what the kernel supports (ids must be integers in "
                           f"[0, {max_id}], at most 4 distinct ids per row, one background id), or NaN scores")
    return loss[0] if n_img == 1 else loss


def refine_scores(ref_cls_score, ref_iou_score):
    """testing_function of lib/modeling/model_builder.py:60-68: per head (cls * iou)[:, 1:]."""
    return [(c * i)[:, 1:] for c, i in zip(ref_cls_score, ref_iou_score)]
