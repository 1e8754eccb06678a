"""ctypes binding of libcimhead.so (the C ABI declared in include/cimhead.h).

There is no CPU or PyTorch fallback anywhere in this package: if the shared library has not
been built, or a tensor is not on a CUDA device, the call raises.
Build with `python -c "import __graft_entry__ as g; g.build()"` or `make -C cim_b200/csrc`.
"""
import ctypes as C
import os
import threading

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcimhead.so")
ABI_VERSION = 7
MAX_LAYERS = 4
OVERLAP_ALGOS = {"auto": 0, "popc": 1, "tensor": 2}
#: cim_set_debug_flags bits (include/cimhead.h): diagnostic kernel selection for A/B timing and bit-identity tests
DBG_ROI_BWD_SMEM_TILE, DBG_OVERLAP_LOADER_WARP, DBG_SCORE_FFMA, DBG_ROI_NO_WINDOWS, DBG_ROI_BWD_ONE_CHUNK = 1, 2, 4, 8, 16
DBG_ROI_POOL_SIMPLE = 32

_lock = threading.Lock()
_lib = None


class MineParams(C.Structure):
    """cim_mine_params of include/cimhead.h (field order and types must match)."""
    _fields_ = [
        ("n_img", C.c_int), ("R", C.c_int), ("C", C.c_int), ("C1", C.c_int), ("n_layers", C.c_int),
        ("det_cols", C.c_int), ("gt_cap", C.c_int), ("mode", C.c_int), ("keep_count", C.c_int),
        ("big_thr", C.c_float), ("con_thr", C.c_float),
        ("cls_thr", C.c_float * MAX_LAYERS), ("iou_thr", C.c_float * MAX_LAYERS),
    ]


_P, _I, _F, _SZ, _I64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64
_SIGNATURES = {
    "cim_abi_version": (C.c_int, []),
    "cim_error_string": (C.c_char_p, [_I]),
    "cim_set_debug_flags": (None, [C.c_uint]),
    "cim_get_debug_flags": (C.c_uint, []),
    "cim_debug_roi_window_plan": (_I, [_P, _I, _I, _I, _I, _F, _I, _I, _P, _P, _I, _P, _P]),
    "cim_debug_roi_window_plan_ex": (_I, [_P, _P, _I, _I, _I, _I, _F, _I, _I, _P, _P, _I, _P, _P]),
    "cim_roi_align_workspace_bytes": (_SZ, [_I]),
    "cim_roi_align_workspace_bytes_ex": (_SZ, [_I, _I, _I, _I, _I, _I, _I]),
    "cim_roi_align_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_prepare": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_fwd_prepared": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_bwd_prepared": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_prepare_ex": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_fwd_prepared_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_bwd_prepared_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_maskfuse_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_align_maskfuse_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _SZ, _P]),
    "cim_roi_pool_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _P]),
    "cim_roi_pool_fwd_ex": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _P]),
    "cim_roi_pool_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "cim_mask_pack": (_I, [_P, _P, _I64, _I64, _I64, _P]),
    "cim_mask_unpack_crops": (_I, [_P, _P, _P, _P, _I64, _I, _I, _I64, _P]),
    "cim_mask_pack_tiled": (_I, [_P, _P, _I64, _I, _I, _I64, _P]),
    "cim_mask_unpack_crops_tiled": (_I, [_P, _P, _P, _P, _I64, _I, _I, _I64, _P]),
    "cim_mask_overlap_workspace_bytes": (_SZ, [_I, _I, _I64, _I]),
    "cim_mask_overlap": (_I, [_P, _I, _I, _I64, _P, _P, _P, _P, _P, _SZ, _P]),
    "cim_mask_overlap_algo": (_I, [_P, _I, _I, _I64, _P, _P, _P, _P, _P, _SZ, _I, _P]),
    "cim_mask_overlap_ex": (_I, [_P, _I, _I, _I64, _I, _P, _P, _P, _P, _P, _SZ, _I, _P]),
    "cim_mask_meta_bytes": (_SZ, [_I, _I, _I64]),
    "cim_mask_unpack_crops_tiled_meta": (_I, [_P, _P, _P, _P, _P, _SZ, _I, _I, _I, _I, _I64, _P]),
    "cim_mask_unpack_crops_tiled_meta_sparse": (_I, [_P, _P, _P, _P, _P, _P, _SZ, _I, _I, _I, _I, _I64, _P]),
    "cim_mask_unpack_rle_tiled_meta_sparse": (_I, [_P, _I64, _P, _P, _P, _P, _P, _P, _SZ, _I, _I, _I, _I, _I64, _P,
                                                    _P]),
    "cim_mask_meta": (_I, [_P, _I, _I, _I64, _I, _P, _SZ, _P]),
    "cim_mask_overlap_meta": (_I, [_P, _P, _I, _I, _I64, _I, _P, _P, _P, _P, _P, _SZ, _I, _P]),
    "cim_mask_pair_ratio": (_I, [_P, _P, _I, _I, _I64, _I, _P, _P, _P, _P, _P]),
    "cim_mask_rle": (_I, [_P, _I, _I, _I64, _I, _I, _I, _P, _P, _P, _I, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "cim_score_heads_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "cim_score_heads": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_score_heads_bwd_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "cim_score_heads_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_score_heads_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_score_heads_bwd_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_score_heads_compact_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "cim_score_heads_compact": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_score_heads_bwd_compact_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "cim_score_heads_bwd_compact": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "cim_debug_compact_row_map": (_I, [_P, _I, _I, _I, _P]),
    "cim_head_losses": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _F, _F, _F, _P]),
    "cim_pcl_loss": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _F, _I, _P]),
    "cim_pcl_loss_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _I, _P]),
    "cim_test_scores": (_I, [_P, _P, _I64, _I, _I, _P]),
    "cim_box_nms": (_I, [_P, _P, _I, _I, _I, _F, _F, _P, _P]),
    "cim_box_nms_batched": (_I, [_P, _P, _I, _I, _I, _I, _F, _F, _P, _P]),
    "cim_test_scores_tta": (_I, [_P, _P, _I64, _I, _I, _I, _I, _P]),
    "cim_box_detections": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "cim_sizeof_mine_params": (_SZ, []),
    "cim_mine_workspace_bytes": (_SZ, [C.POINTER(MineParams)]),
    "cim_mine": (_I, [C.POINTER(MineParams), C.POINTER(_P), C.POINTER(_P), _P, _P, _P, _P, _P, _P, _P, _P,
                      _P, _SZ, _P]),
    "cim_anti_noise_uniform_count_max": (_SZ, [C.POINTER(MineParams)]),
    "cim_anti_noise": (_I, [C.POINTER(MineParams), _P, _P, _P, _P, _P, _P, _P]),
    "cim_anti_noise_stream": (_I, [C.POINTER(MineParams), _P, _P, _P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "cim_assign": (_I, [C.POINTER(MineParams), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cim_mine_ex": (_I, [C.POINTER(MineParams), _P, C.c_double, C.POINTER(_P), C.POINTER(_P), _P, _P, _P, _P, _P, _P,
                         _P, _P, _P, _SZ, _P]),
    "cim_mine_image_constants": (_I, [C.c_double, _I, C.POINTER(_I), C.POINTER(_F)]),
    "cim_assign_ex": (_I, [C.POINTER(MineParams), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    """The loaded library; raises (loudly) if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: the CUDA extension has not been built and this package "
                        "has no fallback path.  Run `make -C cim_b200/csrc` (needs nvcc, sm_100a).")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in _SIGNATURES.items():
                    fn = getattr(handle, name)          # AttributeError if the symbol is missing
                    fn.restype, fn.argtypes = res, args
                if handle.cim_abi_version() != ABI_VERSION:
                    raise RuntimeError("libcimhead.so ABI version mismatch; rebuild it")
                if handle.cim_sizeof_mine_params() != C.sizeof(MineParams):
                    raise RuntimeError("cim_mine_params layout mismatch between cimhead.h and _lib.py")
                _lib = handle
    return _lib


class debug_flags:
    """with _lib.debug_flags(_lib.DBG_...): the library's diagnostic kernel selection for the calls inside the
    block (process-wide; tests and A/B timing only).  The library never reads the environment."""

    def __init__(self, flags):
        self.flags = int(flags)

    def __enter__(self):
        self.prev = lib().cim_get_debug_flags()
        lib().cim_set_debug_flags(self.flags)
        return self

    def __exit__(self, *exc):
        lib().cim_set_debug_flags(self.prev)
        return False


def check(rc, what):
    if rc != 0:
        msg = lib().cim_error_string(rc).decode()
        raise RuntimeError(f"{what} failed with code {rc}: {msg}")


def stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def n_props_arg(n_props, n_img, R, device):
    """The n_props argument of the ragged entry points -> None (every image has R proposals) or a CUDA int32 [n_img]
    tensor on `device`.  A host sequence, numpy array or CPU tensor is validated (length n_img, integers in [1, R]) and
    copied to the device once; a CUDA tensor must be int32 [n_img] on `device` and is used as is (its values cannot be
    checked without a synchronisation: the kernels clamp them to [1, R])."""
    if n_props is None:
        return None
    if isinstance(n_props, torch.Tensor) and n_props.device.type != "cpu":
        if not n_props.is_cuda or n_props.device != torch.device(device):
            raise ValueError(f"n_props must be on {device} or on the host, got {n_props.device}")
        if n_props.dtype != torch.int32:
            raise TypeError(f"n_props must be int32 on the device, got {n_props.dtype}")
        if n_props.numel() != n_img or n_props.dim() != 1:
            raise ValueError(f"n_props must have shape [{n_img}], got {tuple(n_props.shape)}")
        return n_props.contiguous()
    return torch.from_numpy(host_counts(n_props, n_img, R)).to(device, non_blocking=True)


def host_counts(n_props, n_img, R):
    """Validated host copy of proposal counts (a sequence, numpy array or CPU tensor: integers in [1, R], shape
    [n_img]) -> int32 numpy array."""
    a = n_props.numpy() if isinstance(n_props, torch.Tensor) else np.asarray(n_props)
    if a.dtype.kind not in "iu":
        raise TypeError(f"n_props must hold integers, got {a.dtype}")
    if a.shape != (n_img,):
        raise ValueError(f"n_props must have shape [{n_img}], got {a.shape}")
    if a.size and (a.min() < 1 or a.max() > R):
        raise ValueError(f"n_props must lie in [1, {R}], got [{a.min()}, {a.max()}]")
    return a.astype(np.int32)


def compact_rows_arg(n_props, n_img, R, device):
    """The counts of a compact ragged batch -> (CUDA int32 [n_img] counts on `device`, N = their sum).  Image b's
    proposals are then rows [off_b, off_b + n_b) of the per-proposal tensors, off_b = n_0 + ... + n_{b-1}.  N sizes
    host-side tensors, so the counts must come from the host (a sequence, numpy array or CPU tensor, validated as by
    n_props_arg); a CUDA tensor is refused, because reading it would cost a synchronisation."""
    if n_props is None:
        raise ValueError("a compact batch needs its proposal counts")
    if isinstance(n_props, torch.Tensor) and n_props.device.type != "cpu":
        raise ValueError("the counts of a compact batch must be on the host (N = their sum sizes the tensors); "
                         f"got a tensor on {n_props.device}")
    a = host_counts(n_props, n_img, R)
    return torch.from_numpy(a).to(device, non_blocking=True), int(a.sum(dtype=np.int64))


def compact_row_map(n_props, n_img, R, N):
    """cim_debug_compact_row_map (host, no GPU): padded row of each compact row, -1 past the counts' sum."""
    a = None if n_props is None else np.ascontiguousarray(n_props, dtype=np.int32)
    out = np.empty(N, np.int32)
    check(lib().cim_debug_compact_row_map(a.ctypes.data_as(C.c_void_p) if a is not None else None, n_img, R, N,
                                          out.ctypes.data_as(C.c_void_p)), "cim_debug_compact_row_map")
    return out


def feat_hw_arg(feat_hw, B, H, W, device):
    """The feat_hw argument of the RoIAlign _ex entry points -> None (every image fills the [H, W] canvas) or a CUDA
    int32 [B, 2] tensor of the per-image extents (H_b, W_b) on `device`.  A host sequence, numpy array or CPU tensor is
    validated (shape [B, 2], integers, 1 <= H_b <= H, 1 <= W_b <= W) and copied to the device once; a CUDA tensor must be
    int32 [B, 2] on `device` and is used as is (the kernels clamp its values to [1, H] x [1, W])."""
    if feat_hw is None:
        return None
    if isinstance(feat_hw, torch.Tensor) and feat_hw.device.type != "cpu":
        if not feat_hw.is_cuda or feat_hw.device != torch.device(device):
            raise ValueError(f"feat_hw must be on {device} or on the host, got {feat_hw.device}")
        if feat_hw.dtype != torch.int32:
            raise TypeError(f"feat_hw must be int32 on the device, got {feat_hw.dtype}")
        if tuple(feat_hw.shape) != (B, 2):
            raise ValueError(f"feat_hw must have shape [{B}, 2], got {tuple(feat_hw.shape)}")
        return feat_hw.contiguous()
    a = feat_hw.numpy() if isinstance(feat_hw, torch.Tensor) else np.asarray(feat_hw)
    if a.dtype.kind not in "iu":
        raise TypeError(f"feat_hw must hold integers, got {a.dtype}")
    if a.shape != (B, 2):
        raise ValueError(f"feat_hw must have shape [{B}, 2], got {a.shape}")
    if a.size and (a[:, 0].min() < 1 or a[:, 0].max() > H or a[:, 1].min() < 1 or a[:, 1].max() > W):
        raise ValueError(f"feat_hw must lie in [1, {H}] x [1, {W}], got heights [{a[:, 0].min()}, {a[:, 0].max()}] "
                         f"and widths [{a[:, 1].min()}, {a[:, 1].max()}]")
    return torch.from_numpy(a.astype(np.int32)).to(device, non_blocking=True)


def require_cuda(t, name, dtype=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: cim_b200 has no CPU path")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t
