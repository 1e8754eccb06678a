"""oracle/mask_oracle.py -- CPU restatement of the reference's pairwise mask overlap maps.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under cim_b200/ may import it.

Restates (numpy, integer counts then the reference's float casts):
  * mask_iou            lib/utils/mask_utils.py:6-18
        iou[n,k] = sum(m_a[n] & m_b[k]) / sum(m_a[n] | m_b[k])      (int / int -> float64,
        stored into a float32 array, :12,17)
  * mask_asymmetric_iou lib/utils/mask_utils.py:20-32
        asy[n,k] = sum(m_a[n] & m_b[k]) / sum(m_b)                  (denominator: the COLUMN mask)
  * the column-by-column driver + float16 cast of the offline scripts
        tools/pre/create_cob_iou.py:43-48, tools/pre/create_cob_asy_iou.py:43-51

Pinning: tests/golden/mask_overlap_*.npz were produced by oracle/make_golden.py running the
reference's own lib/utils/mask_utils.py (unmodified, behind a 3-line
chainer.backends.cuda.get_array_module -> numpy shim) and tests/test_oracle_masks.py checks
this restatement against them bit for bit (fp16 payload compared as uint16).
"""
import numpy as np


def _as_bool(masks):
    m = np.asarray(masks)
    return m.reshape(m.shape[0], -1) != 0


def overlap_counts(masks):
    """Integer intersection counts [N,N] (int64) and areas [N] (int64)."""
    m = _as_bool(masks)
    # 0/1 float32 matmul is exact while counts stay below 2**24 (512x512 masks: 2**18).
    if m.shape[1] < (1 << 24):
        f = m.astype(np.float32)
        inter = np.rint(f @ f.T).astype(np.int64)
    else:  # pragma: no cover - never reached at the sizes we run
        f = m.astype(np.float64)
        inter = np.rint(f @ f.T).astype(np.int64)
    area = np.diagonal(inter).copy()
    return inter, area


def maps_from_counts(inter, area, row_area=None):
    """(iou_fp16, asy_fp16) from integer counts with the reference's rounding chain:
    python/numpy int / int -> float64, assignment into a float32 array, `.astype(float16)`.
    row_area: areas of the rows when inter holds only some rows of the map (default: area, a square map)."""
    inter = np.asarray(inter, dtype=np.int64)
    area = np.asarray(area, dtype=np.int64)
    row_area = area if row_area is None else np.asarray(row_area, dtype=np.int64)
    union = row_area[:, None] + area[None, :] - inter
    with np.errstate(divide="ignore", invalid="ignore"):
        iou32 = (inter.astype(np.float64) / union.astype(np.float64)).astype(np.float32)
        asy32 = (inter.astype(np.float64) / area[None, :].astype(np.float64)).astype(np.float32)
        # float32 -> float16 overflow cannot happen (values in [0,1] or NaN)
        return iou32.astype(np.float16), asy32.astype(np.float16)


def mask_overlap_maps(masks):
    """iou_map[i,j], asy_iou_map[i,j] (both float16 [N,N]) for byte/bool masks [N,H,W] or [N,HW].
    asy[i,j] = |m_i & m_j| / |m_j|: how much of proposal j lies inside proposal i."""
    inter, area = overlap_counts(masks)
    return maps_from_counts(inter, area)


def mask_overlap_maps_literal(masks):
    """The reference's literal per-pair loops (slow; small N only).  Same arithmetic as
    mask_utils.py called one column at a time as in create_cob_iou.py:44-46."""
    m = _as_bool(masks)
    n = m.shape[0]
    iou = np.empty((n, n), dtype=np.float32)
    asy = np.empty((n, n), dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        for k in range(n):
            col = m[k]
            col_area = col.sum()
            for i in range(n):
                inter = np.bitwise_and(m[i], col).sum()
                union = np.bitwise_or(m[i], col).sum()
                iou[i, k] = inter / union
                asy[i, k] = inter / col_area
    return iou.astype(np.float16), asy.astype(np.float16)


def pair_ratio(mask_a, mask_b, mode="iou"):
    """The four rectangular functions of lib/utils/mask_utils.py between two mask sets -> float32 [Na, Nb]:
    "iou" (:6-18), "asymmetric" (:20-32, denominator mask_b.sum() over ALL of b), "inside" (:35-47, |b_k|),
    "outside" (:50-62, |a_n|).  int / int in float64, stored to float32, like the reference's result array.
    Pinned by tests/golden/mask_pair.npz (reference's own mask_utils.py through the numpy shim)."""
    a, b = _as_bool(mask_a), _as_bool(mask_b)
    inter = a.astype(np.float64) @ b.astype(np.float64).T
    area_a, area_b = a.sum(1).astype(np.float64), b.sum(1).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        if mode == "iou":
            out = inter / (area_a[:, None] + area_b[None, :] - inter)
        elif mode == "asymmetric":
            out = inter / np.float64(b.sum())
        elif mode == "inside":
            out = inter / area_b[None, :]
        elif mode == "outside":
            out = inter / area_a[:, None]
        else:
            raise ValueError(mode)
    return out.astype(np.float32)
