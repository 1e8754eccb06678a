"""Ragged batches without a GPU: argument validation of the _ex entry points (refused before anything touches CUDA),
the per-image mining constants the kernels compute against the reference's numpy arithmetic, and the host-side
validation of n_props."""
import ctypes as C

import numpy as np
import pytest
import torch

from cim_b200 import _lib

NULL = C.c_void_p(0)
FAKE = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch
ODD = C.c_void_p(4098)            # an n_props pointer that is not 4-byte aligned


def _params(R=2000, p_seed=0.1):
    p = _lib.MineParams()
    p.n_img, p.R, p.C, p.C1, p.n_layers, p.det_cols, p.gt_cap, p.mode = 8, R, 20, 21, 3, 21, R, 0
    p.keep_count = int(np.ceil(p_seed * R))
    p.big_thr = float(np.float32(0.9 * R))
    p.con_thr = 0.85
    return p


def test_score_heads_ex_argument_validation():
    L = _lib.lib()
    call = lambda x=FAKE, w=FAKE, b=FAKE, s=FAKE, n=FAKE, n_img=8, R=2000, D=4096, C1=21, K=3: \
        L.cim_score_heads_ex(x, w, b, s, n, n_img, R, D, C1, K, NULL, 0, NULL)
    for kw in ({"x": NULL}, {"w": NULL}, {"b": NULL}, {"s": NULL}, {"n_img": -1}, {"R": -1}, {"D": 0}, {"C1": 0},
               {"K": -1}, {"K": 9}):
        assert call(**kw) == -1, kw
    assert call(n=ODD) == -4
    assert call(n_img=65536) == -2
    assert call(n_img=0) == 0 and call(R=0) == 0                  # nothing to do


def test_score_heads_bwd_ex_argument_validation():
    L = _lib.lib()
    call = lambda x=FAKE, w=FAKE, s=FAKE, g=FAKE, n=FAKE, gx=FAKE, ws=FAKE, n_img=8, R=2000, K=3, ws_bytes=1 << 40: \
        L.cim_score_heads_bwd_ex(x, w, s, g, n, gx, NULL, NULL, n_img, R, 4096, 21, K, ws, ws_bytes, NULL)
    for kw in ({"x": NULL}, {"w": NULL}, {"s": NULL}, {"g": NULL}, {"ws": NULL}, {"n_img": -1}, {"R": -1}, {"K": 9}):
        assert call(**kw) == -1, kw
    assert call(n=ODD) == -4
    assert call(ws_bytes=1024) == -3
    assert call(gx=NULL) == 0                                       # no gradient wanted


def test_mine_ex_and_assign_ex_argument_validation():
    L = _lib.lib()
    p = _params()
    ptrs = (C.c_void_p * 3)(4096, 4096, 4096)
    mine = lambda p=p, n=FAKE, p_seed=0.1, ws=FAKE, ws_bytes=1 << 40: L.cim_mine_ex(
        C.byref(p), n, p_seed, ptrs, ptrs, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, ws, ws_bytes, NULL)
    for p_seed in (0.0, -0.1, 1.5, float("nan"), float("inf")):
        assert mine(p_seed=p_seed) == -1, p_seed
    small = _params()
    small.keep_count = 199                                          # ceil(0.1 * 2000) = 200 seeds at n_b = R
    assert mine(p=small) == -1
    assert mine(p=small, p_seed=0.05, n=ODD) == -4                  # ... which p_seed = 0.05 fits
    assert mine(n=ODD) == -4
    assert mine(ws=NULL) == -3 and mine(ws_bytes=16) == -3
    bad = _params()
    bad.R = 20000
    assert mine(p=bad) == -2
    assert mine(n=NULL, p_seed=0.0, ws=NULL) == -3                  # NULL n_props: cim_mine, p_seed not looked at

    assign = lambda p=p, n=FAKE, iou=FAKE, out=FAKE: L.cim_assign_ex(C.byref(p), n, iou, FAKE, FAKE, FAKE, FAKE, NULL,
                                                                     out, FAKE, FAKE, FAKE, NULL)
    assert assign(iou=NULL) == -1 and assign(out=NULL) == -1
    assert assign(n=ODD) == -4
    assert assign(p=bad) == -2


def test_pcl_loss_ex_argument_validation():
    L = _lib.lib()
    call = lambda pc=FAKE, mat=FAKE, n=FAKE, loss=FAKE, n_img=8, R=2000, C1=21, max_id=255: L.cim_pcl_loss_ex(
        pc, mat, n, loss, NULL, n_img, R, C1, max_id, 1.0, 0, NULL)
    for kw in ({"pc": NULL}, {"mat": NULL}, {"loss": NULL}, {"n_img": -1}, {"R": 0}, {"C1": 1}, {"max_id": 0}):
        assert call(**kw) == -1, kw
    assert call(C1=129) == -2 and call(max_id=256) == -2 and call(R=16385) == -2
    assert call(n=ODD) == -4
    assert call(n_img=0) == 0


@pytest.mark.parametrize("p_seed", [0.1, 0.05, 0.15, 0.3, 1 / 3])
def test_image_constants_equal_the_reference_arithmetic(p_seed):
    """keep_count = int(np.ceil(p_seed * n)) (heads.py:332) and big_thr = np.float32(0.9 * n) (heads.py:338) for every
    n up to the mining limit, from the function the kernels run."""
    L = _lib.lib()
    kc, bt = C.c_int(), C.c_float()
    got_k = np.empty(10240, np.int64)
    got_b = np.empty(10240, np.float32)
    for n in range(1, 10241):
        assert L.cim_mine_image_constants(p_seed, n, C.byref(kc), C.byref(bt)) == 0
        got_k[n - 1], got_b[n - 1] = kc.value, bt.value
    n = np.arange(1, 10241)
    want_k = np.array([int(np.ceil(p_seed * int(i))) for i in n])
    want_b = np.array([np.float32(0.9 * int(i)) for i in n], np.float32)
    np.testing.assert_array_equal(got_k, want_k)
    np.testing.assert_array_equal(got_b.view(np.uint32), want_b.view(np.uint32))
    # the cases the rounding decides: products that land next to an integer in float64
    assert (p_seed * n != np.round(p_seed * n)).any()


def test_image_constants_argument_validation():
    L = _lib.lib()
    kc, bt = C.c_int(), C.c_float()
    assert L.cim_mine_image_constants(0.1, 0, C.byref(kc), C.byref(bt)) == -1
    assert L.cim_mine_image_constants(0.0, 10, C.byref(kc), C.byref(bt)) == -1
    assert L.cim_mine_image_constants(1.01, 10, C.byref(kc), C.byref(bt)) == -1
    assert L.cim_mine_image_constants(float("nan"), 10, C.byref(kc), C.byref(bt)) == -1
    assert L.cim_mine_image_constants(0.1, 10, None, C.byref(bt)) == -1
    assert L.cim_mine_image_constants(0.1, 10, C.byref(kc), None) == -1
    assert L.cim_mine_image_constants(1.0, 7, C.byref(kc), C.byref(bt)) == 0 and kc.value == 7


@pytest.mark.parametrize("bad,exc", [([5, 6, 7], ValueError), ([0, 5, 6, 7], ValueError), ([5, 6, 7, 2001], ValueError),
                                     ([-1, 5, 6, 7], ValueError), ([5.0, 6.0, 7.0, 8.0], TypeError),
                                     (torch.tensor([5, 6, 7, 8], dtype=torch.float32), TypeError),
                                     (np.array([[5, 6], [7, 8]]), ValueError),
                                     (torch.tensor([5, 6, 7, 8], dtype=torch.int32, device="meta"), ValueError)])
def test_host_n_props_are_validated(bad, exc):
    """Host counts are checked before anything is copied: length n_img, integers, 1 <= n_b <= R; a tensor on a device
    other than the call's is refused."""
    with pytest.raises(exc):
        _lib.n_props_arg(bad, 4, 2000, "cuda:0")
    assert _lib.n_props_arg(None, 4, 2000, "cuda:0") is None
