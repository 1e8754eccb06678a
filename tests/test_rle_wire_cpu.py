"""The RLE wire of the proposal masks without a GPU: mask_ops.batch_rle_host against the oracle's decoder, its
refusals, and the argument refusals of cim_mask_unpack_rle_tiled_meta_sparse (checked before anything touches CUDA)."""
import ctypes as C

import numpy as np
import pytest
import torch

from cim_b200 import _lib, mask_ops
from oracle import rle_oracle as R

NULL = C.c_void_p(0)
FAKE = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch


def native_masks(seed, n, h, w):
    rs = np.random.RandomState(seed)
    m = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        y0, x0 = rs.randint(h), rs.randint(w)
        m[i, y0:rs.randint(y0, h + 1), x0:rs.randint(x0, w + 1)] = 1
        m[i] &= (rs.rand(h, w) < 0.9).astype(np.uint8)
    return m


def test_batch_rle_host_slots_decode_to_the_canvas_padded_masks():
    H, W, Rcap = 48, 64, 7
    sizes = [(40, 33), (48, 64), (1, 1), (17, 50)]
    counts = [5, 7, 1, 0]
    native = [native_masks(b, n, h, w) for b, (n, (h, w)) in enumerate(zip(counts, sizes))]
    per_image = [[R.encode_mask(m)[0] for m in nm] for nm in native]
    per_image[1] = [dict(d, counts=d["counts"].decode()) for d in per_image[1]]       # str counts are taken too
    rle = mask_ops.batch_rle_host(per_image, Rcap, H, W)
    assert rle.chars.dtype == torch.uint8 and rle.off.shape == (4 * Rcap,) and rle.len.shape == (4 * Rcap,)
    assert rle.hw.tolist() == [[40, 33], [48, 64], [1, 1], [H, W]]
    assert rle.nbytes == rle.chars.numel() + 4 * Rcap * 12 + 4 * 2 * 4
    chars = rle.chars.numpy().tobytes()
    for b in range(4):
        h, w = rle.hw[b].tolist()
        for i in range(Rcap):
            r = b * Rcap + i
            o, n = int(rle.off[r]), int(rle.len[r])
            if i >= counts[b]:
                assert n == 0                                              # padding row
                continue
            canvas = np.zeros((H, W), np.uint8)
            canvas[:h, :w] = R.decode(R.fr_string(chars[o:o + n]), h, w)
            want = np.zeros((H, W), np.uint8)
            want[:h, :w] = native[b][i]
            np.testing.assert_array_equal(canvas, want)


def test_batch_rle_host_refusals():
    d = R.encode_mask(np.ones((4, 6), np.uint8))[0]
    with pytest.raises(ValueError, match="exceed R"):
        mask_ops.batch_rle_host([[d, d, d]], 2, 8, 16)
    with pytest.raises(ValueError, match="different sizes"):
        mask_ops.batch_rle_host([[d, R.encode_mask(np.ones((5, 6), np.uint8))[0]]], 4, 8, 16)
    with pytest.raises(ValueError, match="exceeds the canvas"):
        mask_ops.batch_rle_host([[d]], 4, 8, 4)
    with pytest.raises(ValueError, match="exceeds the canvas"):
        mask_ops.batch_rle_host([[d]], 4, 3, 16)
    with pytest.raises(ValueError, match="uncompressed"):
        mask_ops.batch_rle_host([[{"size": [4, 6], "counts": [0, 24]}]], 4, 8, 16)


def test_unpack_rle_argument_validation():
    L = _lib.lib()

    def call(chars=FAKE, n_chars=100, off=FAKE, len_=FAKE, hw=NULL, packed=FAKE, prev=FAKE, meta=FAKE,
             meta_bytes=1 << 30, n_img=2, n=10, h=512, w=512, words=8192, bad=NULL):
        return L.cim_mask_unpack_rle_tiled_meta_sparse(chars, n_chars, off, len_, hw, packed, prev, meta, meta_bytes,
                                                       n_img, n, h, w, words, bad, NULL)

    for kw in ({"chars": NULL}, {"off": NULL}, {"len_": NULL}, {"packed": NULL}, {"prev": NULL}, {"meta": NULL},
               {"n_chars": -1}, {"n_img": -1}, {"n": -1}, {"h": 0}, {"w": 0}):
        assert call(**kw) == -1, kw
    for kw in ({"h": 500, "words": 8000}, {"w": 504, "words": 8064}, {"h": 8, "w": 8208, "words": 2052},
               {"h": 65536, "w": 32768, "words": 2 ** 26}):
        assert call(**kw) == -2, kw
    for kw in ({"words": 8191}, {"packed": C.c_void_p(4104)}, {"prev": C.c_void_p(4104)}, {"off": C.c_void_p(4100)},
               {"len_": C.c_void_p(4097)}, {"hw": C.c_void_p(4098)}, {"bad": C.c_void_p(4098)}):
        assert call(**kw) == -4, kw
    assert call(meta_bytes=16) == -3
    assert call(meta=C.c_void_p(4096 + 128)) == -3
