"""ROI operators with mmcv.ops' Python surface, backed by libcimhead.so.

The reference imports `RoIPool, RoIAlign, roi_pool, roi_align, nms, soft_nms` from mmcv.ops
(lib/ops/__init__.py:6) and calls `RoIAlign(resolution, spatial_scale, sampling_ratio)(feat, rois)`
/ `RoIPool(resolution, spatial_scale)(feat, rois)` at lib/modeling/model_builder.py:227-231, building
a fresh module per call with positional arguments.  Same names, argument order and defaults here
(mmcv 1.x: `aligned=True`, `pool_mode='avg'`), so the reference files stay unchanged once
`cim_b200/shim` is on PYTHONPATH (INTEGRATION.md).

rois: [K, 5] float32 rows (batch_idx, x1, y1, x2, y2) in input-image pixels.

feat_hw (keyword, RoIAlign only): images of different sizes batched on one canvas.  input [N, C, H, W] is the canvas
and image b occupies input[b, :, :H_b, :W_b]; feat_hw [N, 2] holds the (H_b, W_b) (see _lib.feat_hw_arg).  Each
image's outputs and gradient then equal RoIAlign of its own map alone; the canvas outside the extents must be finite
and gets a gradient of exactly 0.  None: every image fills the canvas.
"""
import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib


def _pair(v):
    if isinstance(v, (tuple, list)):
        if len(v) != 2:
            raise ValueError("output_size must be an int or a pair")
        return int(v[0]), int(v[1])
    return int(v), int(v)


def _check_inputs(feat, rois):
    _lib.require_cuda(feat, "input", torch.float32)
    _lib.require_cuda(rois, "rois", torch.float32)
    if feat.dim() != 4:
        raise ValueError("input must be [N, C, H, W]")
    if rois.dim() != 2 or rois.size(1) != 5:
        raise ValueError("rois must be [K, 5] (batch_idx, x1, y1, x2, y2)")
    if rois.device != feat.device:
        raise ValueError("input and rois must be on the same device")


class RoIAlignFunction(Function):
    @staticmethod
    def forward(ctx, feat, rois, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode="avg", aligned=True,
                feat_hw=None):
        if pool_mode != "avg":
            raise NotImplementedError("only pool_mode='avg' is implemented (the reference never uses 'max')")
        _check_inputs(feat, rois)
        oh, ow = _pair(output_size)
        feat, rois = feat.contiguous(), rois.contiguous()
        B, Cc, H, W = feat.shape
        K = rois.size(0)
        hw = _lib.feat_hw_arg(feat_hw, B, H, W, feat.device)
        L = _lib.lib()
        with torch.cuda.device(feat.device):
            ws = torch.empty(L.cim_roi_align_workspace_bytes_ex(B, Cc, H, W, K, oh, ow), dtype=torch.uint8,
                             device=feat.device)
            out = torch.empty((K, Cc, oh, ow), dtype=torch.float32, device=feat.device)
            if hw is None:
                rc = L.cim_roi_align_fwd(_lib.ptr(feat), _lib.ptr(rois), _lib.ptr(out), B, Cc, H, W, K, oh, ow,
                                         float(spatial_scale), int(sampling_ratio), int(bool(aligned)),
                                         _lib.ptr(ws), ws.numel(), _lib.stream_ptr(feat.device))
            else:
                rc = _fwd_ex(L, feat, rois, hw, None, out, oh, ow, spatial_scale, sampling_ratio, aligned, ws)
        _lib.check(rc, "cim_roi_align_fwd")
        ctx.save_for_backward(rois)
        ctx.ws = ws                 # the backward reuses the forward's ROI descriptors (cim_roi_align_bwd_prepared)
        ctx.hw = hw
        ctx.cfg = (tuple(feat.shape), oh, ow, float(spatial_scale), int(sampling_ratio), int(bool(aligned)))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        (rois,) = ctx.saved_tensors
        (B, Cc, H, W), oh, ow, scale, sr, aligned = ctx.cfg
        grad_out = grad_out.contiguous()
        K = rois.size(0)
        L = _lib.lib()
        ws = ctx.ws
        with torch.cuda.device(grad_out.device):
            grad_feat = torch.empty((B, Cc, H, W), dtype=torch.float32, device=grad_out.device)
            rc = L.cim_roi_align_bwd_prepared_ex(_lib.ptr(grad_out), _lib.ptr(rois), _lib.ptr(ctx.hw), None,
                                                 _lib.ptr(grad_feat), B, Cc, H, W, K, oh, ow, scale, sr, aligned,
                                                 _lib.ptr(ws), ws.numel(), _lib.stream_ptr(grad_out.device))
        _lib.check(rc, "cim_roi_align_bwd")
        return grad_feat, None, None, None, None, None, None, None


def _fwd_ex(L, feat, rois, hw, masks, out, oh, ow, spatial_scale, sampling_ratio, aligned, ws):
    """Descriptors with the image extents hw, then the forward that reuses them (the backward does too)."""
    B, Cc, H, W = feat.shape
    K = rois.size(0)
    st = _lib.stream_ptr(feat.device)
    args = (B, Cc, H, W, K, oh, ow, float(spatial_scale), int(sampling_ratio), int(bool(aligned)), _lib.ptr(ws),
            ws.numel(), st)
    rc = L.cim_roi_align_prepare_ex(_lib.ptr(rois), _lib.ptr(hw), *args)
    if rc == 0:
        rc = L.cim_roi_align_fwd_prepared_ex(_lib.ptr(feat), _lib.ptr(rois), _lib.ptr(hw), _lib.ptr(masks),
                                             _lib.ptr(out), *args)
    return rc


#: RoIPool bin conventions (cim_roi_pool_fwd_ex): "mmcv" = mmcv 1.x's RoIPool, the op the reference imports
#: (lib/ops/__init__.py:6) and therefore the default of this drop-in; "legacy" = the reference's vendored
#: lib/model/roi_pooling kernel == torchvision.ops.roi_pool.  They differ for most ROIs (float vs rounded corners).
ROI_POOL_VARIANTS = {"legacy": 0, "mmcv": 1}


class RoIPoolFunction(Function):
    @staticmethod
    def forward(ctx, feat, rois, output_size, spatial_scale=1.0, variant="mmcv"):
        if variant not in ROI_POOL_VARIANTS:
            raise ValueError("variant must be 'mmcv' or 'legacy'")
        _check_inputs(feat, rois)
        oh, ow = _pair(output_size)
        feat, rois = feat.contiguous(), rois.contiguous()
        B, Cc, H, W = feat.shape
        K = rois.size(0)
        L = _lib.lib()
        with torch.cuda.device(feat.device):
            out = torch.empty((K, Cc, oh, ow), dtype=torch.float32, device=feat.device)
            argmax = torch.empty((K, Cc, oh, ow), dtype=torch.int32, device=feat.device)
            rc = L.cim_roi_pool_fwd_ex(_lib.ptr(feat), _lib.ptr(rois), _lib.ptr(out), _lib.ptr(argmax), B, Cc, H, W,
                                       K, oh, ow, float(spatial_scale), ROI_POOL_VARIANTS[variant],
                                       _lib.stream_ptr(feat.device))
        _lib.check(rc, "cim_roi_pool_fwd")
        ctx.save_for_backward(rois, argmax)
        ctx.cfg = (tuple(feat.shape), oh, ow)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        rois, argmax = ctx.saved_tensors
        (B, Cc, H, W), oh, ow = ctx.cfg
        grad_out = grad_out.contiguous()
        L = _lib.lib()
        with torch.cuda.device(grad_out.device):
            grad_feat = torch.empty((B, Cc, H, W), dtype=torch.float32, device=grad_out.device)
            rc = L.cim_roi_pool_bwd(_lib.ptr(grad_out), _lib.ptr(argmax), _lib.ptr(rois), _lib.ptr(grad_feat), B,
                                    Cc, H, W, rois.size(0), oh, ow, _lib.stream_ptr(grad_out.device))
        _lib.check(rc, "cim_roi_pool_bwd")
        return grad_feat, None, None, None, None


class RoIAlignMaskFuseFunction(Function):
    """RoIAlign + the MaskFuse prologue in one kernel: concat(box_x, box_x * masks) of
    lib/modeling/resnet50.py:121-134 (vgg16.py:172-175, HRNet.py:625-628).  masks [K, oh, ow] carry no gradient
    (the reference passes masks.detach(), model_builder.py:136)."""

    @staticmethod
    def forward(ctx, feat, rois, masks, output_size, spatial_scale=1.0, sampling_ratio=0, aligned=True, feat_hw=None):
        _check_inputs(feat, rois)
        _lib.require_cuda(masks, "masks", torch.float32)
        oh, ow = _pair(output_size)
        feat, rois = feat.contiguous(), rois.contiguous()
        B, Cc, H, W = feat.shape
        K = rois.size(0)
        masks = masks.reshape(K, oh, ow).contiguous()
        hw = _lib.feat_hw_arg(feat_hw, B, H, W, feat.device)
        L = _lib.lib()
        with torch.cuda.device(feat.device):
            ws = torch.empty(L.cim_roi_align_workspace_bytes_ex(B, Cc, H, W, K, oh, ow), dtype=torch.uint8,
                             device=feat.device)
            out = torch.empty((K, 2 * Cc, oh, ow), dtype=torch.float32, device=feat.device)
            if hw is None:
                rc = L.cim_roi_align_maskfuse_fwd(_lib.ptr(feat), _lib.ptr(rois), _lib.ptr(masks), _lib.ptr(out), B,
                                                  Cc, H, W, K, oh, ow, float(spatial_scale), int(sampling_ratio),
                                                  int(bool(aligned)), _lib.ptr(ws), ws.numel(),
                                                  _lib.stream_ptr(feat.device))
            else:
                rc = _fwd_ex(L, feat, rois, hw, masks, out, oh, ow, spatial_scale, sampling_ratio, aligned, ws)
        _lib.check(rc, "cim_roi_align_maskfuse_fwd")
        ctx.save_for_backward(rois, masks)
        ctx.ws = ws
        ctx.hw = hw
        ctx.cfg = (tuple(feat.shape), oh, ow, float(spatial_scale), int(sampling_ratio), int(bool(aligned)))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        rois, masks = ctx.saved_tensors
        (B, Cc, H, W), oh, ow, scale, sr, aligned = ctx.cfg
        grad_out = grad_out.contiguous()
        K = rois.size(0)
        L = _lib.lib()
        ws = ctx.ws
        with torch.cuda.device(grad_out.device):
            grad_feat = torch.empty((B, Cc, H, W), dtype=torch.float32, device=grad_out.device)
            rc = L.cim_roi_align_bwd_prepared_ex(_lib.ptr(grad_out), _lib.ptr(rois), _lib.ptr(ctx.hw), _lib.ptr(masks),
                                                 _lib.ptr(grad_feat), B, Cc, H, W, K, oh, ow, scale, sr, aligned,
                                                 _lib.ptr(ws), ws.numel(), _lib.stream_ptr(grad_out.device))
        _lib.check(rc, "cim_roi_align_maskfuse_bwd")
        return grad_feat, None, None, None, None, None, None, None


def roi_align_maskfuse(input, rois, masks, output_size, spatial_scale=1.0, sampling_ratio=0, aligned=True, *,
                       feat_hw=None):
    """[K, 2C, oh, ow] = concat(RoIAlign(input, rois), RoIAlign(input, rois) * masks[:, None]) in one pass."""
    return RoIAlignMaskFuseFunction.apply(input, rois, masks, output_size, spatial_scale, sampling_ratio, aligned,
                                          feat_hw)


def roi_align(input, rois, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode="avg", aligned=True, *,
              feat_hw=None):
    return RoIAlignFunction.apply(input, rois, output_size, spatial_scale, sampling_ratio, pool_mode, aligned,
                                  feat_hw)


def roi_pool(input, rois, output_size, spatial_scale=1.0, variant="mmcv"):
    return RoIPoolFunction.apply(input, rois, output_size, spatial_scale, variant)


class RoIAlign(nn.Module):
    """mmcv.ops.RoIAlign(output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode='avg',
    aligned=True, use_torchvision=False).  Holds no parameters or buffers."""

    def __init__(self, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode="avg", aligned=True,
                 use_torchvision=False):
        super().__init__()
        if use_torchvision:
            raise NotImplementedError("use_torchvision=True would bypass the sm_100a kernels")
        self.output_size = _pair(output_size)
        self.spatial_scale = float(spatial_scale)
        self.sampling_ratio = int(sampling_ratio)
        self.pool_mode = pool_mode
        self.aligned = aligned

    def forward(self, input, rois, *, feat_hw=None):
        return roi_align(input, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.pool_mode,
                         self.aligned, feat_hw=feat_hw)

    def __repr__(self):
        return (f"{self.__class__.__name__}(output_size={self.output_size}, spatial_scale={self.spatial_scale}, "
                f"sampling_ratio={self.sampling_ratio}, pool_mode={self.pool_mode}, aligned={self.aligned})")


class RoIPool(nn.Module):
    """mmcv.ops.RoIPool(output_size, spatial_scale=1.0), with mmcv 1.x's bins by default (float ROI corners
    x1 * s .. (x2 + 1) * s, floor / ceil of p * bin + start; restated from mmcv's published kernel, parity unpinned
    because mmcv is absent here); variant="legacy" gives the bins of the reference's vendored roi_pooling kernel
    (== torchvision.ops.roi_pool), which is pinned against both."""

    def __init__(self, output_size, spatial_scale=1.0, variant="mmcv"):
        super().__init__()
        if variant not in ROI_POOL_VARIANTS:
            raise ValueError("variant must be 'mmcv' or 'legacy'")
        self.output_size = _pair(output_size)
        self.spatial_scale = float(spatial_scale)
        self.variant = variant

    def forward(self, input, rois):
        return roi_pool(input, rois, self.output_size, self.spatial_scale, self.variant)

    def __repr__(self):
        return f"{self.__class__.__name__}(output_size={self.output_size}, spatial_scale={self.spatial_scale})"


def nms(*args, **kwargs):
    """Imported by lib/ops/__init__.py:6 but never called on the CIM path (box NMS only runs in
    test-time post-processing through Cython, lib/utils/mask_eval_utils.py:71)."""
    raise NotImplementedError("box nms is outside the CIM head path; see SURVEY.md section 8f")


def soft_nms(*args, **kwargs):
    raise NotImplementedError("soft_nms is outside the CIM head path; see SURVEY.md section 8f")
