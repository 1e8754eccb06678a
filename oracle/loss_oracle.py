"""oracle/loss_oracle.py -- CPU restatement of the CIM loss block and its gradient.  TEST INFRASTRUCTURE:
imported only by tests/, __graft_entry__.smoke() and bench.py's CPU legs, never by the product path.

Restates (torch on CPU, float64 by default; the gradient comes from autograd over the restated forward, which
is what loss.backward() does in the reference, tools/train.py:436):
  * heads.loss_weight_bag_loss   lib/modeling/heads.py:43-74
  * heads.cls_iou_loss           lib/modeling/heads.py:78-138 (class-specific IoU branch)
  * heads.mil_bag_loss           lib/modeling/heads.py:149-166
  * heads.PCL_loss               lib/modeling/heads.py:10-41
  * the wiring of lib/modeling/model_builder.py:170-202 (lmda = 3 for layer 0, iou_loss x 3, skipped layers)
Pinned: oracle/make_golden.py runs the reference's own heads.cls_iou_loss / heads.mil_bag_loss (imported
unmodified) with autograd on seeded inputs and stores losses + gradients in tests/golden/head_losses.npz; this
restatement reproduces them within 1e-6 relative (make_golden asserts it, tests/test_oracle_losses.py re-checks).
"""
import numpy as np
import torch

# The reference clamps float32 tensors, so torch rounds the bounds 1e-6 and 1 - 1e-6 to float32 first (both roundings
# go down).  At float64 the unrounded bound 1e-6 would lie above float32(1e-6) and zero the gradient of a score that
# sits exactly on it, where the reference passes the gradient (torch.clamp is inclusive).
LO, HI = float(np.float32(1e-6)), float(np.float32(1 - 1e-6))


def weighted_bag_loss(pred, pseudo, label_tmp, w):
    """heads.py:43-74.  pred [R,C1] (already clamped products), pseudo [R,C1], label_tmp [C1] 0/1, w [R]."""
    p = (pseudo != 0).to(pred.dtype)                                      # :50
    ind = (p.sum(-1) != 0).to(pred.dtype)                                 # :49
    fg_val, fg_idx = torch.max(ind[:, None] * pred * p, dim=0)            # :55
    un_val, un_idx = torch.max(pred, dim=0)                               # :57
    agg = (fg_val * label_tmp + un_val * (1 - label_tmp)).clamp(LO, HI)   # :60-61
    present = label_tmp == 1
    idx = torch.where(present, fg_idx, un_idx)                            # :64-67
    lw = torch.where(present, w[idx], torch.ones_like(agg))               # :69-70
    return (-(label_tmp * torch.log(agg) + (1 - label_tmp) * torch.log(1 - agg)) * lw).mean()   # :72-74


def cls_iou_loss(cls, iou, pseudo, pseudo_iou, w, labels):
    """heads.py:78-138 -> (cls_loss, iou_loss, bag_loss).  labels [C] 0/1 image labels."""
    cls, iou = cls.clamp(LO, HI), iou.clamp(LO, HI)                       # :80-81
    label_tmp = torch.cat([torch.ones(1, dtype=cls.dtype), labels.to(cls.dtype)])   # :83-84
    bag = weighted_bag_loss(cls * iou, pseudo, label_tmp, w)              # :100
    ind = (pseudo != 0).sum(-1) != 0                                      # :86
    zero = torch.zeros((), dtype=cls.dtype)
    if ind.sum() == 0:
        return zero, zero, bag
    p = (pseudo[ind] != 0).to(cls.dtype)                                  # :106
    w_i = w[ind]
    cls_loss = (-p * torch.log(cls[ind]) * w_i[:, None]).sum() / p.sum()  # :115-116
    fg = (p[:, 1:] != 0).sum(-1) != 0                                     # :118
    if fg.sum() == 0:
        return cls_loss, zero, bag
    s = (p[fg] * iou[ind][fg]).sum(-1)                                    # :127
    t = pseudo_iou.flatten()[ind][fg].to(cls.dtype)
    iou_loss = (torch.nn.functional.smooth_l1_loss(s, t, reduction="none") * w_i[fg]).sum() / p[fg].sum()   # :134-135
    return cls_loss, iou_loss, bag


def mil_bag_loss(p_cls, p_det, labels):
    """heads.py:149-166 (background column present in the prediction)."""
    pred = (p_cls * p_det).sum(0).clamp(LO, HI)
    label_tmp = torch.cat([torch.ones(1, dtype=pred.dtype), labels.to(pred.dtype)])
    return (-(label_tmp * torch.log(pred) + (1 - label_tmp) * torch.log(1 - pred))).mean()


def head_losses(scores, pseudo_labels, pseudo_iou, loss_weights, valid, labels, k, lmda=(3.0, 1.0), iou_weight=3.0,
                grad_scale=1.0, dtype=torch.float64):
    """model_builder.py:170-202 for n_img images.  scores [2+2K, n_img*R, C1]; pseudo_labels [L,n_img,R,C1];
    pseudo_iou [L,n_img,R] (float16 array); loss_weights [L,n_img,R]; valid [L,n_img]; labels [n_img,C].
    Returns (losses [n_img, K+1, 3] float64, grad_scores like scores, float64): slot l = (cls, iou, bag) of layer l,
    slot K = (0, 0, mil_bag); grad = grad_scale * d(sum_l cls + iou_weight sum_l iou + sum_l bag + mil) / d scores."""
    scores = torch.as_tensor(np.asarray(scores), dtype=dtype).clone().requires_grad_(True)
    n_layers, n_img, R, c1 = pseudo_labels.shape
    s = scores.view(2 + 2 * k, n_img, R, c1)
    pl = torch.as_tensor(np.asarray(pseudo_labels), dtype=dtype)
    pi = torch.as_tensor(np.asarray(pseudo_iou).astype(np.float32), dtype=dtype)
    lw = torch.as_tensor(np.asarray(loss_weights), dtype=dtype)
    lab = torch.as_tensor(np.asarray(labels), dtype=dtype)
    losses = torch.zeros(n_img, k + 1, 3, dtype=dtype)
    total = torch.zeros((), dtype=dtype)
    for b in range(n_img):
        for l in range(n_layers):
            if not valid[l][b]:
                continue                                                  # :189-190
            m = lmda[0] if l == 0 else lmda[1]                            # :172
            c, i, g = cls_iou_loss(s[2 + l, b], s[2 + k + l, b], pl[l, b], pi[l, b], m * lw[l, b], lab[b])
            losses[b, l] = torch.stack([c, i, g]).detach()
            total = total + c + iou_weight * i + g                        # :198-200
        mil = mil_bag_loss(s[0, b], s[1, b], lab[b])                      # :202
        losses[b, k, 2] = mil.detach()
        total = total + mil
    (total * grad_scale).backward()
    return losses.numpy(), scores.grad.numpy()


def pcl_loss(predict_cls, mat):
    """heads.py:10-41 for one image.  predict_cls [R,C1] (requires_grad allowed), mat [R,C1] cluster ids."""
    mat = torch.as_tensor(mat)
    col0 = np.setdiff1d(mat[:, 0].numpy(), [0])                         # :13
    if len(col0) > 1:
        raise AssertionError("more than one background cluster id")      # :20
    bg = col0[0] if len(col0) else None
    loss = torch.zeros((), dtype=predict_cls.dtype)
    count = 1e-6                                                         # :22
    for k in np.unique(mat.numpy()):                                     # :23, ascending
        if k == 0:
            continue
        hit = mat == float(k)
        rows = hit.sum(1) != 0
        sel = predict_cls[rows]
        n = sel.shape[0]
        count += n
        if bg is None or k != bg:                                        # foreground cluster, :25-32
            v = sel.mean(0).clamp(LO, HI)
            t = (hit.sum(0) != 0).to(predict_cls.dtype)
            loss = loss + n * (-(t * torch.log(v) + (1 - t) * torch.log(1 - v))).mean()
        else:                                                            # background cluster, :34-39
            p = sel.clamp(LO, HI)
            t = (mat[rows] != 0).to(predict_cls.dtype)
            loss = loss + n * (-(t * torch.log(p) + (1 - t) * torch.log(1 - p))).mean()
    return 12 * (loss / count)                                           # :40-41


def pcl_losses(predict_cls, mat, grad_scale=1.0, dtype=torch.float64):
    """n_img images: predict_cls [n_img*R, C1], mat [n_img, R, C1] -> (loss [n_img], grad like predict_cls)."""
    n_img, R, c1 = np.asarray(mat).shape
    p = torch.as_tensor(np.asarray(predict_cls), dtype=dtype).clone().requires_grad_(True)
    m = torch.as_tensor(np.asarray(mat), dtype=dtype)
    losses = [pcl_loss(p[b * R:(b + 1) * R], m[b]) for b in range(n_img)]
    total = sum(losses) * grad_scale
    if total.requires_grad:                           # images without any cluster contribute a constant 0
        total.backward()
    grad = p.grad.numpy() if p.grad is not None else np.zeros(tuple(p.shape))
    return np.array([float(l.detach()) for l in losses]), grad
