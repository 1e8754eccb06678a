"""Compact ragged batches without a GPU: the row map of cim_debug_compact_row_map (the code the device builder runs)
against a numpy restatement of the layout, and the argument checks of _lib.compact_rows_arg."""
import numpy as np
import pytest
import torch

from cim_b200 import _lib


def numpy_row_map(n_props, n_img, R, N):
    """compact row off_b + r -> padded row b * R + r for r < n_b (n_b clamped to [1, R]); rows past sum(n_b) -> -1,
    proposals past row N dropped"""
    n = np.full(n_img, R) if n_props is None else np.clip(np.asarray(n_props, np.int64), 1, R)
    padded = np.concatenate([b * R + np.arange(v) for b, v in enumerate(n)])
    out = np.full(N, -1, np.int32)
    out[:min(N, padded.size)] = padded[:N]
    return out


@pytest.mark.parametrize("n_props,R", [([2000, 1, 137, 1999, 200], 2000), ([1], 1), ([3, 3, 3], 3),
                                       (list(np.random.RandomState(2024).randint(200, 2001, size=8)), 2000)])
def test_row_map_exact_counts(n_props, R):
    N = int(np.sum(n_props))
    got = _lib.compact_row_map(n_props, len(n_props), R, N)
    np.testing.assert_array_equal(got, numpy_row_map(n_props, len(n_props), R, N))
    assert (got >= 0).all() and len(np.unique(got)) == N


def test_row_map_extra_rows_are_minus_one():
    n_props, R = [5, 1, 7], 8
    got = _lib.compact_row_map(n_props, 3, R, 20)
    np.testing.assert_array_equal(got, numpy_row_map(n_props, 3, R, 20))
    assert (got[13:] == -1).all() and (got[:13] >= 0).all()


def test_row_map_over_count_drops_the_tail():
    n_props, R = [5, 6, 7], 8
    got = _lib.compact_row_map(n_props, 3, R, 9)
    np.testing.assert_array_equal(got, [0, 1, 2, 3, 4, 8, 9, 10, 11])


def test_row_map_clamps_like_the_kernels():
    n_props, R = [0, -3, 50, 2], 4
    got = _lib.compact_row_map(n_props, 4, R, 16)
    np.testing.assert_array_equal(got, numpy_row_map(n_props, 4, R, 16))
    np.testing.assert_array_equal(got[:8], [0, 4, 8, 9, 10, 11, 12, 13])


def test_row_map_null_counts_is_identity():
    np.testing.assert_array_equal(_lib.compact_row_map(None, 3, 5, 15), np.arange(15))


def test_row_map_refuses_bad_sizes():
    for n_img, R, N in ((0, 4, 1), (2, 0, 1), (2, 4, 0), (2, 4, 9)):
        with pytest.raises(RuntimeError):
            _lib.compact_row_map([1] * max(n_img, 1), n_img, R, N)


def test_compact_rows_arg_validation():
    dev = torch.device("cpu")                                   # the copy target is not used by the refusals
    with pytest.raises(ValueError):
        _lib.compact_rows_arg(None, 2, 10, dev)
    with pytest.raises(ValueError):
        _lib.compact_rows_arg(torch.tensor([3, 4], dtype=torch.int32, device="meta"), 2, 10, dev)
    with pytest.raises(ValueError):
        _lib.compact_rows_arg([3], 2, 10, dev)
    with pytest.raises(ValueError):
        _lib.compact_rows_arg([0, 4], 2, 10, dev)
    with pytest.raises(ValueError):
        _lib.compact_rows_arg([11, 4], 2, 10, dev)
    with pytest.raises(TypeError):
        _lib.compact_rows_arg([1.0, 4.0], 2, 10, dev)
    counts, n = _lib.compact_rows_arg(np.array([3, 10], np.int64), 2, 10, dev)
    assert n == 13 and counts.dtype == torch.int32 and counts.tolist() == [3, 10]
    counts, n = _lib.compact_rows_arg(torch.tensor([1, 2]), 2, 10, dev)
    assert n == 3


def test_abi_version_and_symbols():
    assert _lib.lib().cim_abi_version() == _lib.ABI_VERSION == 7
    for name in ("cim_score_heads_compact", "cim_score_heads_bwd_compact", "cim_score_heads_compact_workspace_bytes",
                 "cim_score_heads_bwd_compact_workspace_bytes", "cim_debug_compact_row_map"):
        assert name in _lib.EXPORTED_SYMBOLS


def test_compact_workspace_covers_smaller_batches():
    L = _lib.lib()
    for fn in (L.cim_score_heads_compact_workspace_bytes, L.cim_score_heads_bwd_compact_workspace_bytes):
        full = fn(8, 2000, 16000, 4096, 21, 3)
        assert all(fn(8, 2000, n, 4096, 21, 3) <= full for n in (8, 127, 128, 9000, 15999))
