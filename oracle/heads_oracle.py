"""oracle/heads_oracle.py -- CPU (numpy) restatement of the reference's CIM heads.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under cim_b200/ may import it.

Restates, function by function, lib/modeling/heads.py of the reference:
  * score_heads        <- cls_iou_model.forward            heads.py:194-219
  * greedy_mask_nms    <- CIM_layer.instance_nms           heads.py:237-258
  * cim_label          <- CIM_layer.CIM_label              heads.py:318-407
  * mist_label         <- CIM_layer.MIST_label             heads.py:260-316
  * cim_layer_forward  <- CIM_layer.forward                heads.py:409-503
  * refine_scores      <- testing_function                 lib/modeling/model_builder.py:60-68

Facts of the reference this file reproduces on purpose (SURVEY.md, "five facts"):
  - iou_map / asy_iou_map are float16; every `map < thr` / `map > thr` is evaluated in
    float16 against float16(thr) (heads.py:250-251, 338, 387, 489, 500-501).
  - `0.9 * R` (heads.py:338) is compared with an integer count after promotion to float32.
  - heads.py:493-498 (`pseudo_labels[big_proposal, :] = 0`) raises inside a bare
    try/except and therefore changes nothing; it is NOT applied here either.
  - Anti-noise sampling (heads.py:451-466) draws from numpy's GLOBAL RandomState, one
    np.random.choice per present class in ascending class order.
  - argsort / argmax / max ties: lowest index wins (what torch returns on CPU and what
    its CUDA reductions return); NaN handling of torch.max(dim) = first NaN wins.

Pinning: oracle/make_golden.py imports the reference's heads.py unmodified from
/root/reference, runs it on seeded synthetic inputs and stores inputs + outputs under
tests/golden/; tests/test_oracle_heads.py replays them through this file bit for bit.
"""
import numpy as np

F16 = np.float16


# --------------------------------------------------------------------------- scoring
def _softmax(z, axis):
    z = z - z.max(axis=axis, keepdims=True)
    e = np.exp(z)
    return e / e.sum(axis=axis, keepdims=True)


def score_heads(x, weights, biases):
    """cls_iou_model.forward (heads.py:194-219).

    x [R,D]; weights/biases: lists of 2+2K arrays ordered
    [classifier, detector, refine_cls.0..K-1, refine_iou.0..K-1], each [C1,D] / [C1].
    Evaluated in float64 and rounded once to float32, so both an fp32 CPU run of the
    reference and the CUDA kernel sit within ~1e-6 relative of it.
    Returns (predict_cls, predict_det, [ref_cls_k], [ref_iou_k]) as float32 arrays [R,C1].
    """
    x = np.asarray(x, dtype=np.float64)
    k = (len(weights) - 2) // 2
    logits = [x @ np.asarray(w, np.float64).T + np.asarray(b, np.float64)
              for w, b in zip(weights, biases)]
    predict_cls = _softmax(logits[0], axis=-1)           # over classes   (:199-200)
    predict_det = _softmax(logits[1], axis=0)            # over PROPOSALS (:202-203)
    ref_cls = [_softmax(logits[2 + i], axis=-1) for i in range(k)]          # :211-212
    ref_iou = [1.0 / (1.0 + np.exp(-logits[2 + k + i])) for i in range(k)]  # :215-216
    f = lambda a: a.astype(np.float32)
    return f(predict_cls), f(predict_det), [f(a) for a in ref_cls], [f(a) for a in ref_iou]


def score_heads_bwd(x, weights, biases, grads, outputs=None):
    """Backward of cls_iou_model.forward (autograd of heads.py:194-219) in float64.

    grads: 2+2K arrays [R,C1] = dL/d(output) in the order of `weights`.  Returns
    (grad_x [R,D], [grad_W_h [C1,D]], [grad_b_h [C1]]) as float32.  Pinned by oracle/make_golden.py
    against torch autograd through the reference's own cls_iou_model.
    outputs: optionally the forward's float32 outputs (2+2K arrays [R,C1]) to differentiate through, as torch's
    softmax / sigmoid backward does with its saved outputs; by default they are recomputed in float64.  On saturated
    scores the difference matters: near y = 1 the float32 rounding of y changes 1 - y by percents."""
    x = np.asarray(x, dtype=np.float64)
    k = (len(weights) - 2) // 2
    gx = np.zeros_like(x)
    gws, gbs = [], []
    for h, (w, b, g) in enumerate(zip(weights, biases, grads)):
        w, g = np.asarray(w, np.float64), np.asarray(g, np.float64)
        z = x @ w.T + np.asarray(b, np.float64) if outputs is None else None
        if h == 1:                                    # softmax over proposals (:203)
            y = _softmax(z, axis=0) if z is not None else np.asarray(outputs[h], np.float64)
            dz = y * (g - (g * y).sum(0, keepdims=True))
        elif h < 2 + k:                               # softmax over classes (:200, :212)
            y = _softmax(z, axis=-1) if z is not None else np.asarray(outputs[h], np.float64)
            dz = y * (g - (g * y).sum(-1, keepdims=True))
        else:                                         # sigmoid (:216)
            y = 1.0 / (1.0 + np.exp(-z)) if z is not None else np.asarray(outputs[h], np.float64)
            dz = g * y * (1.0 - y)
        gx += dz @ w
        gws.append((dz.T @ x).astype(np.float32))
        gbs.append(dz.sum(0).astype(np.float32))
    return gx.astype(np.float32), gws, gbs


def refine_scores(ref_cls, ref_iou):
    """testing_function (model_builder.py:60-68): per refinement head (cls*iou)[:,1:]."""
    return [(c * i)[:, 1:] for c, i in zip(ref_cls, ref_iou)]


# --------------------------------------------------------------------------- mining
def _drop_bg(a, n_cls):
    a = np.asarray(a, dtype=np.float32)
    return a[:, 1:] if a.shape[1] - 1 == n_cls else a


def _seed_order(scores, keep_count):
    """`argsort(descending=True)[:keep_count]` (heads.py:279,354); ties -> lower index."""
    return np.argsort(-scores, kind="stable")[:keep_count]


def greedy_mask_nms(sub_iou, thr):
    """instance_nms (heads.py:237-258) on candidates already in descending-score order.
    sub_iou[a,b] = iou_map[seed_a, seed_b] (float16).  A later candidate b survives an
    earlier kept a only if `sub_iou[a,b] < float16(thr)` is True (so NaN suppresses)."""
    thr = F16(thr)
    n = sub_iou.shape[0]
    alive = np.ones(n, dtype=bool)
    kept = []
    for a in range(n):
        if not alive[a]:
            continue
        kept.append(a)
        ok = sub_iou[a] < thr
        ok[: a + 1] = True            # only later entries are filtered
        alive &= ok
    return np.asarray(kept, dtype=np.int64)


def big_proposal_flag(asy_map, con_thr):
    """asy_iou_flag (heads.py:338): proposals that contain (> con_thr) fewer than 90% of
    all proposals.  int64 count vs python float -> torch compares in float32."""
    r = asy_map.shape[-1]
    cnt = (asy_map > F16(con_thr)).sum(axis=-1)
    return cnt.astype(np.float32) < np.float32(0.9 * r)


def cim_label(predict_cls, predict_det, labels, iou_map, asy_map,
              p_seed=0.1, nms_thr=0.25, con_thr=0.85):
    """CIM_label (heads.py:318-407).  Returns (gt_class [R] int64, -1 = not mined,
    otherwise the 0-based foreground class; gt_weight [R] float32, -1 where not mined;
    asy_iou_flag [R] bool; per_class debug dict)."""
    labels = np.asarray(labels).reshape(-1)
    n_cls = labels.shape[0]
    cls = _drop_bg(predict_cls, n_cls)
    det = _drop_bg(predict_det, n_cls)
    preds = cls * det                                            # :330 (fp32 product)
    r = cls.shape[0]
    keep_count = int(np.ceil(p_seed * r))                         # :332
    flag = big_proposal_flag(asy_map, con_thr)                    # :338
    gt_class = np.full(r, -1, dtype=np.int64)
    gt_weight = np.full(r, -1.0, dtype=np.float32)
    debug = {}
    for c in np.nonzero(labels)[0]:                               # :340 ascending
        det_c = det[:, c] if det.shape[1] == n_cls else det[:, 0]  # :343-349
        order = _seed_order(cls[:, c], keep_count)                # :354
        kept = greedy_mask_nms(iou_map[order][:, order], nms_thr)  # :361-372
        seeds = order[kept]                                       # :380
        contain = (asy_map[:, seeds] > F16(con_thr)) & flag[:, None]   # :386-390
        entry = {"order": order, "seeds": seeds, "picked": np.zeros(0, np.int64)}
        if contain.any():                                         # :391
            contain = contain[:, contain.any(axis=0)]             # :392
            weighted = np.where(contain, det_c[:, None], np.float32(0))   # :393
            picked = np.unique(np.argmax(weighted, axis=0))        # :394-395
            better = preds[picked, c] > gt_weight[picked]          # :397
            take = picked[better]
            gt_class[take] = c                                    # :400-401
            gt_weight[take] = preds[take, c]                       # :402
            entry["picked"] = picked
        debug[int(c)] = entry
    return gt_class, gt_weight, flag, debug


def mist_label(preds, labels, iou_map, p_seed=0.1, nms_thr=0.25):
    """MIST_label (heads.py:260-316): the NMS survivors themselves become pseudo GT."""
    labels = np.asarray(labels).reshape(-1)
    n_cls = labels.shape[0]
    p = np.asarray(preds, dtype=np.float32)
    p = p if p.shape[1] == n_cls else p[:, 1:]                    # :269
    r = p.shape[0]
    keep_count = int(np.ceil(p_seed * r))
    gt_class = np.full(r, -1, dtype=np.int64)
    gt_weight = np.full(r, -1.0, dtype=np.float32)
    for c in np.nonzero(labels)[0]:
        order = _seed_order(p[:, c], keep_count)
        kept = greedy_mask_nms(iou_map[order][:, order], nms_thr)
        seeds = order[kept]
        better = p[seeds, c] > gt_weight[seeds]                   # :307
        take = seeds[better]
        gt_class[take] = c
        gt_weight[take] = p[take, c]
    return gt_class, gt_weight


def anti_noise_keep(gt_cls_list, gt_w_list, labels):
    """Anti-noise sampling (heads.py:440-473).  gt_*_list are the mined pseudo GTs in
    ascending proposal order.  Uses numpy's global RNG exactly like the reference:
    one np.random.choice(class_idx, size=n, replace=True, p=w/w.sum()) per present
    class (ascending) that has at least one pseudo GT."""
    labels = np.asarray(labels).reshape(-1)
    keep = np.ones(len(gt_cls_list), dtype=bool)
    for c in np.nonzero(labels)[0]:
        class_idx = np.nonzero(gt_cls_list == c)[0]
        if len(class_idx) == 0:
            continue
        prob = gt_w_list[class_idx]                               # float32
        drawn = np.random.choice(class_idx, size=len(class_idx), replace=True,
                                 p=prob / prob.sum())
        keep[class_idx] = False
        keep[np.unique(drawn)] = True
    return keep


def _rowmax_first(a):
    """torch.max(a, dim=-1) on CPU: strict '>' scan, first NaN wins and stops the scan."""
    a32 = a.astype(np.float32)
    nan = np.isnan(a32)
    idx = np.argmax(np.where(nan, np.inf, a32), axis=-1)
    has_nan = nan.any(axis=-1)
    idx = np.where(has_nan, np.argmax(nan, axis=-1), idx)
    val = np.take_along_axis(a, idx[:, None], axis=-1)[:, 0]
    return val, idx


def cim_layer_forward(predict_cls, predict_det, labels, iou_map, asy_map,
                      p_seed=0.1, cls_thr=0.25, iou_thr=0.5, con_thr=0.85,
                      anti_noise_sampling=True, using_cim=True):
    """CIM_layer.forward (heads.py:409-503).  Returns (pseudo_labels [R,C+1] float32,
    pseudo_iou_labels [R] float16, loss_weights [R] float32) or (None, None, None)."""
    labels = np.asarray(labels).reshape(-1)
    n_cls = labels.shape[0]
    if using_cim:
        gt_class, gt_weight, _flag, _ = cim_label(predict_cls, predict_det, labels, iou_map,
                                                  asy_map, p_seed, cls_thr, con_thr)
    else:                                                         # :421-427
        preds = (np.asarray(predict_cls, np.float32) * np.asarray(predict_det, np.float32)
                 if predict_det is not None else np.asarray(predict_cls, np.float32))
        gt_class, gt_weight = mist_label(preds, labels, iou_map, p_seed, cls_thr)
    gt_rows = np.nonzero(gt_class >= 0)[0]                        # boolean-mask order
    if len(gt_rows) == 0:                                         # :429-430
        return None, None, None
    g_cls, g_w = gt_class[gt_rows], gt_weight[gt_rows]
    if anti_noise_sampling:
        keep = anti_noise_keep(g_cls, g_w, labels)
        gt_rows, g_cls, g_w = gt_rows[keep], g_cls[keep], g_w[keep]
    overlaps = iou_map[:, gt_rows]                                # :435,473
    max_v, max_i = _rowmax_first(overlaps)                        # :477
    r = overlaps.shape[0]
    pseudo = np.zeros((r, n_cls + 1), dtype=np.float32)
    pseudo[np.arange(r), g_cls[max_i] + 1] = 1.0                  # :479
    loss_w = g_w[max_i].copy()                                    # :480
    ignore = max_v == F16(0)                                      # :484-486
    pseudo[ignore] = 0
    loss_w[ignore] = 0
    bg = (max_v < F16(cls_thr)) & ~ignore                         # :489-491
    pseudo[bg] = 0
    pseudo[bg, 0] = 1
    # heads.py:493-498 is a swallowed IndexError -> no relabelling of big proposals.
    piou = max_v.copy()                                           # :481,500-501
    hi = piou > F16(iou_thr)
    lo = piou <= F16(iou_thr)
    piou[hi] = 1
    piou[lo] = 0
    return pseudo, piou.astype(F16), loss_w
