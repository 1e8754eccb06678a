"""Pairwise mask-proposal overlap maps on the GPU.

Replaces the reference's offline `mask_iou` / `mask_asymmetric_iou` (lib/utils/mask_utils.py:6-32,
driven by tools/pre/create_cob_iou.py:43-48 and create_cob_asy_iou.py:43-51) and the two pickle
loads + H2D copies per training step that consume them (lib/modeling/model_builder.py:148-156).

    packed = mask_pack(masks_u8)                 # [..., N, H, W] uint8 -> [..., N, words] int32 bits
    iou_map, asy_iou_map = mask_overlap(packed)  # float16 [..., N, N] each, the reference's dtype
asy_iou_map[i, j] = |m_i & m_j| / |m_j| (how much of proposal j lies inside proposal i).
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib


@dataclass
class MaskCrops:
    """Compact wire format of N proposal masks: bounding-box crops, bit-packed, 32-pixel aligned in x.
    words [total] int32, meta [N,4] int32 = (wx0, y0, ww, h), off [N] int64 (word offset of each crop).
    Host (numpy / pinned torch) or device tensors."""
    words: torch.Tensor
    meta: torch.Tensor
    off: torch.Tensor
    height: int
    width: int

    @property
    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.words, self.meta, self.off))


def pack_crops_host(masks):
    """numpy/CPU: uint8 / bool masks [N, H, W] -> MaskCrops (CPU tensors).  What a data-loader worker
    would produce from the COB proposals instead of full-image byte masks."""
    m = np.asarray(masks) != 0
    n, h, w = m.shape
    wpad = (w + 31) // 32 * 32
    rows = np.zeros((n, h, wpad), dtype=bool)
    rows[:, :, :w] = m
    bits = np.packbits(rows, axis=2, bitorder="little").view("<u4").reshape(n, h, wpad // 32)   # word k = px 32k..
    meta = np.zeros((n, 4), np.int32)
    off = np.zeros(n, np.int64)
    chunks, total = [], 0
    for i in range(n):
        ys, xs = np.nonzero(m[i].any(1))[0], np.nonzero(m[i].any(0))[0]
        if len(ys) == 0:
            off[i] = total
            continue
        y0, y1, wx0, wx1 = ys[0], ys[-1] + 1, xs[0] // 32, xs[-1] // 32 + 1
        meta[i] = (wx0, y0, wx1 - wx0, y1 - y0)
        off[i] = total
        c = bits[i, y0:y1, wx0:wx1].reshape(-1)
        chunks.append(c)
        total += c.size
    words = np.concatenate(chunks) if chunks else np.zeros(0, np.uint32)
    return MaskCrops(torch.from_numpy(words.view(np.int32).copy()), torch.from_numpy(meta), torch.from_numpy(off),
                     h, w)


def crops_from_packed_host(packed, height, width):
    """CPU: full bit masks [N, H*W/32] (int32, W % 32 == 0) -> MaskCrops, without going through
    byte masks (used by bench.py to derive the wire format from its synthetic packed masks)."""
    if width % 32:
        raise ValueError("crops_from_packed_host needs width % 32 == 0; use pack_crops_host")
    p = np.ascontiguousarray(packed.cpu().numpy() if isinstance(packed, torch.Tensor) else packed)
    p = p.view(np.uint32).reshape(p.shape[0], height, width // 32)
    n = p.shape[0]
    nz = p != 0
    row_any, col_any = nz.any(2), nz.any(1)
    y0 = row_any.argmax(1)
    y1 = height - row_any[:, ::-1].argmax(1)
    x0 = col_any.argmax(1)
    x1 = width // 32 - col_any[:, ::-1].argmax(1)
    empty = ~row_any.any(1)
    meta = np.stack([x0, y0, x1 - x0, y1 - y0], 1).astype(np.int32)
    meta[empty] = 0
    sizes = meta[:, 2].astype(np.int64) * meta[:, 3]
    off = np.zeros(n, np.int64)
    off[1:] = np.cumsum(sizes)[:-1]
    words = np.empty(int(sizes.sum()), np.uint32)
    for i in range(n):
        if sizes[i]:
            words[off[i]:off[i] + sizes[i]] = p[i, y0[i]:y1[i], x0[i]:x1[i]].reshape(-1)
    return MaskCrops(torch.from_numpy(words.view(np.int32)), torch.from_numpy(meta), torch.from_numpy(off),
                     height, width)


def batch_crops_host(crops, R, height, width):
    """CPU: the wire format of a batch of differently sized images.  crops: one MaskCrops per image (n_b <= R masks of
    that image at its native size, e.g. from pack_crops_host), each image placed at the top left of a common
    (height, width) canvas -> one MaskCrops of len(crops) * R rows, image b in rows [b * R, b * R + n_b) and EMPTY crops
    (meta 0) in its padding rows, which the unpack turns into all-zero masks.  Zero padding changes neither
    |a & b|, |a | b| nor |b|, so the overlap maps of an image on the canvas are those of the image alone.  A crop
    that does not fit the canvas (rows, or 32-pixel words in x) raises."""
    n_img = len(crops)
    canvas_words = (width + 31) // 32
    meta = np.zeros((n_img * R, 4), np.int32)
    off = np.zeros(n_img * R, np.int64)
    chunks, total = [], 0
    for b, c in enumerate(crops):
        m = np.asarray(c.meta, dtype=np.int64).reshape(-1, 4)
        o = np.asarray(c.off, dtype=np.int64).reshape(-1)
        w = np.asarray(c.words).view(np.int32).reshape(-1)
        n = m.shape[0]
        if n > R:
            raise ValueError(f"image {b}: {n} masks exceed R = {R}")
        if c.height > height or c.width > width:
            raise ValueError(f"image {b}: native size {c.height} x {c.width} exceeds the canvas {height} x {width}")
        full = (m[:, 2] > 0) & (m[:, 3] > 0)
        if np.any(full & ((m[:, 0] < 0) | (m[:, 1] < 0) | (m[:, 0] + m[:, 2] > canvas_words) |
                          (m[:, 1] + m[:, 3] > height))):
            raise ValueError(f"image {b}: a crop does not fit the {height} x {width} canvas")
        for i in range(R):
            r = b * R + i
            off[r] = total                                  # (empty and padding rows: no words)
            if i < n and full[i]:
                size = int(m[i, 2] * m[i, 3])
                meta[r] = m[i]
                chunks.append(w[o[i]:o[i] + size])
                total += size
    words = np.concatenate(chunks) if chunks else np.zeros(0, np.int32)
    return MaskCrops(torch.from_numpy(words.astype(np.int32, copy=True)), torch.from_numpy(meta),
                     torch.from_numpy(off), height, width)


@dataclass
class MaskRLE:
    """Proposal masks as COCO compressed RLE strings (what pycocotools.mask.encode returns as 'counts'), the other wire
    format: row m's string is chars[off[m] : off[m] + len[m]], len 0 = a row of zeros.  chars uint8 [total], off int64
    [rows], len int32 [rows], hw int32 [n_img, 2] = each image's native (h, w) on the (height, width) canvas, where its
    masks sit at the top left.  Host (pinned torch) or device tensors.  mask_rle's device outputs (chars, off, len) plug
    in directly."""
    chars: torch.Tensor
    off: torch.Tensor
    len: torch.Tensor
    hw: torch.Tensor
    height: int
    width: int

    @property
    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.chars, self.off, self.len, self.hw))


def batch_rle_host(per_image, R, height, width):
    """CPU: the RLE wire format of a batch.  per_image: one list per image of COCO dicts {'size': [h, w], 'counts':
    bytes | str} (compressed strings, e.g. from pycocotools.mask.encode), n_b <= R of them, all of one size -> a
    MaskRLE of len(per_image) * R rows, image b in rows [b * R, b * R + n_b) and len 0 in its padding rows.  An image
    whose masks differ in size or exceed the (height, width) canvas raises, and so do uncompressed (list) counts.  An
    image without masks takes the canvas size."""
    n_img = len(per_image)
    off = np.zeros(n_img * R, np.int64)
    lens = np.zeros(n_img * R, np.int32)
    hw = np.zeros((n_img, 2), np.int32)
    chunks, total = [], 0
    for b, dicts in enumerate(per_image):
        if len(dicts) > R:
            raise ValueError(f"image {b}: {len(dicts)} masks exceed R = {R}")
        sizes = {tuple(int(v) for v in d["size"]) for d in dicts}
        if len(sizes) > 1:
            raise ValueError(f"image {b}: masks of different sizes {sorted(sizes)}")
        h, w = sizes.pop() if sizes else (height, width)
        if not (1 <= h <= height and 1 <= w <= width):
            raise ValueError(f"image {b}: native size {h} x {w} exceeds the canvas {height} x {width}")
        hw[b] = (h, w)
        for i, d in enumerate(dicts):
            c = d["counts"]
            if isinstance(c, str):
                c = c.encode("ascii")
            if not isinstance(c, (bytes, bytearray)):
                raise ValueError(f"image {b}, mask {i}: uncompressed (list) counts; only compressed RLE strings "
                                 "(bytes or str) are taken")
            r = b * R + i
            off[r], lens[r] = total, len(c)
            chunks.append(np.frombuffer(bytes(c), np.uint8))
            total += len(c)
        off[b * R + len(dicts):(b + 1) * R] = total
    chars = np.concatenate(chunks) if chunks else np.zeros(0, np.uint8)
    return MaskRLE(torch.from_numpy(chars.copy()), torch.from_numpy(off), torch.from_numpy(lens), torch.from_numpy(hw),
                   int(height), int(width))


def _unpack_rle_into(rle, packed, prev_rects, meta, bad, n_img, n, stream):
    """cim_mask_unpack_rle_tiled_meta_sparse of a device MaskRLE into packed [n_img * n, words] (sparse update against
    prev_rects), metadata into meta, the malformed-string count into bad (int32 [1])."""
    words = rle.height * rle.width // 32
    rc = _lib.lib().cim_mask_unpack_rle_tiled_meta_sparse(
        _lib.ptr(rle.chars), rle.chars.numel(), _lib.ptr(rle.off), _lib.ptr(rle.len), _lib.ptr(rle.hw),
        _lib.ptr(packed), _lib.ptr(prev_rects), _lib.ptr(meta), meta.numel(), n_img, n, rle.height, rle.width, words,
        _lib.ptr(bad), stream)
    _lib.check(rc, "cim_mask_unpack_rle_tiled_meta_sparse")


def unpack_rle(rle, out=None, meta=None):
    """MaskRLE on the device -> tiled bit masks [n_img, R, H*W/32] int32 (tagged kb_per_row = W // 16), or (masks,
    metadata) when meta is True or a uint8 tensor to fill (mask_meta's format, tied to those masks).  out: a buffer to
    overwrite.  Needs H % 8 == 0 and W % 16 == 0.  A malformed string raises ValueError with their number (a host
    synchronisation); its row would be all zero."""
    _lib.require_cuda(rle.chars, "rle.chars", torch.uint8)
    _lib.require_cuda(rle.off, "rle.off", torch.int64)
    _lib.require_cuda(rle.len, "rle.len", torch.int32)
    _lib.require_cuda(rle.hw, "rle.hw", torch.int32)
    if not tiled_ok(rle.height, rle.width):
        raise ValueError("unpack_rle writes the tiled layout: it needs height % 8 == 0 and width % 16 == 0")
    n_img = rle.hw.shape[0]
    rows = rle.off.numel()
    if rle.hw.shape != (n_img, 2) or rle.len.numel() != rows or (n_img and rows % n_img):
        raise ValueError(f"rle.hw must be [n_img, 2] and rle.off / rle.len [n_img * R], got {tuple(rle.hw.shape)}, "
                         f"{rows} and {rle.len.numel()}")
    n = rows // n_img if n_img else 0
    words = rle.height * rle.width // 32
    dev = rle.chars.device
    if out is None:
        out = torch.empty((n_img, n, words), dtype=torch.int32, device=dev)
    if out.shape != (n_img, n, words) or out.dtype != torch.int32 or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous int32 [{n_img}, {n}, {words}] tensor")
    want_meta = meta is not None and meta is not False
    L = _lib.lib()
    with torch.cuda.device(dev):
        out.zero_()
        prev = torch.zeros((max(rows, 1), 4), dtype=torch.int32, device=dev)
        nbytes = L.cim_mask_meta_bytes(n_img, n, words)
        if meta is True or not want_meta:
            meta = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _unpack_rle_into(rle, out, prev, meta, bad, n_img, n, _lib.stream_ptr(dev))
    n_bad = int(bad.item())
    if n_bad:
        raise ValueError(f"{n_bad} malformed RLE string(s): those rows are empty")
    _tag(out, rle.width // 16)
    return (out, meta) if want_meta else out


def tiled_ok(height, width):
    """The 8 x 16 patch pixel order (cim_mask_pack_tiled) needs whole patches."""
    return height % 8 == 0 and width % 16 == 0


def _tag(packed, kb_per_row):
    packed.cim_kb_per_row = kb_per_row      # read back by mask_overlap (plain attribute, lost on views / copies)
    return packed


def unpack_crops(crops, out=None, layout="auto"):
    """MaskCrops on the device -> full bit masks [N, ceil(H*W/32)] int32 (the input of mask_overlap).
    layout: "flat" (row-major pixels), "tiled" (8 x 16 patches) or "auto" (tiled whenever H % 8 == W % 16 == 0)."""
    _lib.require_cuda(crops.words, "crops.words", torch.int32)
    _lib.require_cuda(crops.meta, "crops.meta", torch.int32)
    _lib.require_cuda(crops.off, "crops.off", torch.int64)
    n = crops.meta.shape[0]
    words = (crops.height * crops.width + 31) // 32
    dev = crops.words.device
    if out is None:
        out = torch.empty((n, words), dtype=torch.int32, device=dev)
    tiled = _want_tiled(layout, crops.height, crops.width)
    L = _lib.lib()
    fn = L.cim_mask_unpack_crops_tiled if tiled else L.cim_mask_unpack_crops
    with torch.cuda.device(dev):
        rc = fn(_lib.ptr(crops.words), _lib.ptr(crops.meta.contiguous()), _lib.ptr(crops.off.contiguous()),
                _lib.ptr(out), n, crops.height, crops.width, words, _lib.stream_ptr(dev))
    _lib.check(rc, "cim_mask_unpack_crops")
    return _tag(out, crops.width // 16 if tiled else 0)


def _want_tiled(layout, height, width):
    if layout not in ("auto", "flat", "tiled"):
        raise ValueError("layout must be 'auto', 'flat' or 'tiled'")
    if layout == "tiled" and not tiled_ok(height, width):
        raise ValueError("the tiled layout needs H % 8 == 0 and W % 16 == 0")
    return layout == "tiled" or (layout == "auto" and tiled_ok(height, width))


def mask_pack(masks, layout="auto"):
    """uint8/bool masks [..., H, W] (non-zero = inside) -> bit masks [..., ceil(H*W/32)] int32.
    layout: "flat" = pixel p = y*W + x is bit p & 31 of word p >> 5; "tiled" = 8 x 16 pixel patches (see
    include/cimhead.h), which lets the tensor-core overlap kernel skip the empty parts of the image; "auto" =
    tiled whenever H % 8 == W % 16 == 0.  The overlap maps do not depend on the layout."""
    _lib.require_cuda(masks, "masks")
    if masks.dtype == torch.bool:
        masks = masks.view(torch.uint8)
    if masks.dtype != torch.uint8:
        raise TypeError("masks must be uint8 or bool")
    if masks.dim() < 3:
        raise ValueError("masks must be [..., H, W]")
    masks = masks.contiguous()
    lead = masks.shape[:-2]
    hw = masks.shape[-1] * masks.shape[-2]
    n = 1
    for s in lead:
        n *= s
    words = (hw + 31) // 32
    packed = torch.empty(lead + (words,), dtype=torch.int32, device=masks.device)
    height, width = masks.shape[-2], masks.shape[-1]
    tiled = _want_tiled(layout, height, width)
    with torch.cuda.device(masks.device):
        if tiled:
            rc = _lib.lib().cim_mask_pack_tiled(_lib.ptr(masks), _lib.ptr(packed), n, height, width, words,
                                                _lib.stream_ptr(masks.device))
        else:
            rc = _lib.lib().cim_mask_pack(_lib.ptr(masks), _lib.ptr(packed), n, hw, words,
                                          _lib.stream_ptr(masks.device))
    _lib.check(rc, "cim_mask_pack")
    return _tag(packed, width // 16 if tiled else 0)


def mask_meta(packed, kb_per_row=None, out=None, stream=None):
    """Per-mask metadata of bit masks [n_img, N, words] (areas, occupancy bitmaps over 128-pixel K-blocks, sort keys)
    for mask_overlap(..., meta=...) / CIMHeadStep.run(mask_meta=...): produced once WITH the masks (when a data set is
    packed, or on the copy stream right after cim_mask_unpack_crops) instead of by a pass over all packed masks inside
    every overlap call.  Opaque uint8 tensor (cim_mask_meta_bytes)."""
    _lib.require_cuda(packed, "packed", torch.int32)
    if kb_per_row is None:
        kb_per_row = int(getattr(packed, "cim_kb_per_row", 0))
    if packed.dim() == 2:
        packed = packed.unsqueeze(0)
    packed = packed.contiguous()
    n_img, n, words = packed.shape
    L = _lib.lib()
    with torch.cuda.device(packed.device):
        nbytes = L.cim_mask_meta_bytes(n_img, n, words)
        if out is None:
            out = torch.empty(nbytes, dtype=torch.uint8, device=packed.device)
        rc = L.cim_mask_meta(_lib.ptr(packed), n_img, n, words, int(kb_per_row), _lib.ptr(out), out.numel(),
                             stream if stream is not None else _lib.stream_ptr(packed.device))
    _lib.check(rc, "cim_mask_meta")
    return out


def mask_overlap(packed, return_counts=False, algo="auto", kb_per_row=None, return_visited=False, meta=None):
    """Bit masks [N, words] or [n_img, N, words] (int32) -> (iou_map, asy_iou_map) float16
    [.., N, N]; with return_counts also (inter int32 [.., N, N], area int32 [.., N]).
    algo: "auto" | "popc" (AND + POPC kernel) | "tensor" (tcgen05 int8 kernel).
    kb_per_row: W // 16 for masks in the tiled pixel order, 0 for flat; None = what mask_pack / unpack_crops
    recorded on the tensor (0 if nothing was).  It only steers the locality sort of the tensor path.
    return_visited: also return the number of K-blocks the tensor path visited (int, 0 on the popc path).
    meta: the tensor mask_meta(packed) returned (same packed / kb_per_row): the call then skips its own pass over the
    packed masks."""
    _lib.require_cuda(packed, "packed", torch.int32)
    if kb_per_row is None:
        kb_per_row = int(getattr(packed, "cim_kb_per_row", 0))
    squeeze = packed.dim() == 2
    if squeeze:
        packed = packed.unsqueeze(0)
    if packed.dim() != 3:
        raise ValueError("packed must be [N, words] or [n_img, N, words]")
    packed = packed.contiguous()
    n_img, n, words = packed.shape
    dev = packed.device
    L = _lib.lib()
    iou = torch.empty((n_img, n, n), dtype=torch.float16, device=dev)
    asy = torch.empty((n_img, n, n), dtype=torch.float16, device=dev)
    area = torch.empty((n_img, n), dtype=torch.int32, device=dev)
    inter = torch.empty((n_img, n, n), dtype=torch.int32, device=dev) if return_counts else None
    with torch.cuda.device(dev):
        ws = torch.empty(L.cim_mask_overlap_workspace_bytes(n_img, n, words, int(return_counts)), dtype=torch.uint8,
                         device=dev)
        if return_visited:
            ws[:8].zero_()
        rc = L.cim_mask_overlap_meta(_lib.ptr(packed), _lib.ptr(meta), n_img, n, words, int(kb_per_row),
                                     _lib.ptr(inter), _lib.ptr(area), _lib.ptr(iou), _lib.ptr(asy), _lib.ptr(ws),
                                     ws.numel(), _lib.OVERLAP_ALGOS[algo], _lib.stream_ptr(dev))
    _lib.check(rc, "cim_mask_overlap_meta")
    outs = (iou, asy, inter, area) if return_counts else (iou, asy)
    outs = tuple(o.squeeze(0) for o in outs) if squeeze else outs
    if return_visited:
        outs = outs + (int(ws[:8].view(torch.int64).item()),)
    return outs


def mask_overlap_maps(masks):
    """Convenience: uint8 masks [N, H, W] -> (iou_map, asy_iou_map), i.e. what the reference
    un-pickles from cfg.iou_dir / cfg.asy_iou_dir for one image."""
    return mask_overlap(mask_pack(masks))


# ------------------------------------------------------------------ COCO RLE of selected masks
def rle_chars_cap(n_slots, height, width):
    """Default string capacity of mask_rle: 4 * (height + width) characters per slot, enough for masks with a couple
    of runs per column (need[0] tells the exact total)."""
    return int(n_slots) * 4 * (int(height) + int(width))


def _mask_rle_into(packed, sel_count, sel_idx, height, width, mask_hw, kb_per_row, chars, off, len_, area, bbox,
                   need):
    n_img, R, words = packed.shape
    cap = sel_idx.shape[1]
    with torch.cuda.device(packed.device):
        rc = _lib.lib().cim_mask_rle(_lib.ptr(packed), n_img, R, words, int(height), int(width), int(kb_per_row),
                                     _lib.ptr(mask_hw), _lib.ptr(sel_count), _lib.ptr(sel_idx), cap, _lib.ptr(chars),
                                     chars.numel(), _lib.ptr(off), _lib.ptr(len_), _lib.ptr(area), _lib.ptr(bbox),
                                     _lib.ptr(need), _lib.stream_ptr(packed.device))
    _lib.check(rc, "cim_mask_rle")


def _rle_args(packed, sel_count, sel_idx, height, width, mask_hw, kb_per_row):
    _lib.require_cuda(packed, "packed", torch.int32)
    _lib.require_cuda(sel_count, "sel_count", torch.int32)
    _lib.require_cuda(sel_idx, "sel_idx", torch.int32)
    if kb_per_row is None:
        kb_per_row = int(getattr(packed, "cim_kb_per_row", 0))
    if packed.dim() == 2:
        packed = packed.unsqueeze(0)
    if packed.dim() != 3:
        raise ValueError("packed must be [N, words] or [n_img, N, words]")
    n_img = packed.shape[0]
    if sel_count.shape != (n_img,) or sel_idx.dim() != 2 or sel_idx.shape[0] != n_img:
        raise ValueError(f"sel_count must be [{n_img}] and sel_idx [{n_img}, cap]")
    mask_hw = _lib.feat_hw_arg(mask_hw, n_img, height, width, packed.device)
    return packed.contiguous(), sel_count.contiguous(), sel_idx.contiguous(), mask_hw, int(kb_per_row)


def mask_rle(packed, sel_count, sel_idx, height, width, mask_hw=None, kb_per_row=None, chars_cap=None):
    """Selected bit masks as COCO compressed RLE on the device (cim_mask_rle): what pycocotools.mask.encode returns
    as 'counts', with mask.area and mask.toBbox, for every slot of a selection.
      packed [n_img, R, words] int32 on a height x width canvas (mask_pack / unpack_crops, flat or tiled order;
        kb_per_row = W // 16 for tiled, 0 for flat, None = what mask_pack / unpack_crops recorded);
      sel_count [n_img], sel_idx [n_img, cap] int32 CUDA tensors (count / idx of postproc.detections_batched): slot
        (b, j), j < min(sel_count[b], cap), selects mask sel_idx[b, j] of image b;
      mask_hw: per-image native (h, w) [n_img, 2] (None: the canvas); set bits outside it are ignored.
    Returns device tensors (chars uint8 [chars_cap], off int64 [n_img, cap], len int32 [n_img, cap], area int32
    [n_img, cap], bbox int32 [n_img, cap, 4] (x, y, w, h), need int64 [2]): slot (b, j)'s string is
    chars[off : off + len] when off + len <= chars_cap; need[0] = total characters, need[1] = selected indices
    outside [0, R) (their slots get len 0).  No host synchronisation.  chars_cap None: rle_chars_cap(...)."""
    packed, sel_count, sel_idx, mask_hw, kb_per_row = _rle_args(packed, sel_count, sel_idx, height, width, mask_hw,
                                                                kb_per_row)
    n_img, cap = sel_idx.shape
    if chars_cap is None:
        chars_cap = rle_chars_cap(n_img * cap, height, width)
    if int(chars_cap) < 0:
        raise ValueError("chars_cap must be >= 0")
    dev = packed.device
    chars = torch.empty(int(chars_cap), dtype=torch.uint8, device=dev)
    off = torch.empty((n_img, cap), dtype=torch.int64, device=dev)
    len_ = torch.empty((n_img, cap), dtype=torch.int32, device=dev)
    area = torch.empty((n_img, cap), dtype=torch.int32, device=dev)
    bbox = torch.empty((n_img, cap, 4), dtype=torch.int32, device=dev)
    need = torch.empty(2, dtype=torch.int64, device=dev)
    _mask_rle_into(packed, sel_count, sel_idx, height, width, mask_hw, kb_per_row, chars, off, len_, area, bbox, need)
    return chars, off, len_, area, bbox, need


# ------------------------------------------------------------------ offline callers of lib/utils/mask_utils.py
_RATIO_MODES = {"iou": 0, "asymmetric": 1, "inside": 2, "outside": 3}


def _as_packed_flat(m, name):
    """uint8/bool [N, H, W] -> flat bit masks [N, words] (already packed int32 [N, words] passes through)."""
    _lib.require_cuda(m, name)
    if m.dtype == torch.int32 and m.dim() == 2:
        return m.contiguous(), None
    if m.dim() != 3:
        raise ValueError(f"{name} must be [N, H, W] masks or [N, words] packed int32")
    return mask_pack(m, layout="flat"), tuple(m.shape[1:])


def mask_pair_ratio(mask_a, mask_b, mode="iou", return_counts=False):
    """float32 [Na, Nb] ratio between every mask of a and every mask of b: the four functions of
    lib/utils/mask_utils.py in one kernel (cim_mask_pair_ratio).  Inputs: uint8/bool [N, H, W] CUDA tensors or
    flat bit masks [N, words] from mask_pack(layout="flat")."""
    pa, sa = _as_packed_flat(mask_a, "mask_a")
    pb, sb = _as_packed_flat(mask_b, "mask_b")
    if (sa is not None and sb is not None and sa != sb) or pa.shape[1] != pb.shape[1]:
        raise IndexError("mask shapes differ")                   # mask_utils.py:7-8
    na, nb, words = pa.shape[0], pb.shape[0], pa.shape[1]
    dev = pa.device
    with torch.cuda.device(dev):
        ratio = torch.empty((na, nb), dtype=torch.float32, device=dev)
        inter = torch.empty((na, nb), dtype=torch.int32, device=dev) if return_counts else None
        area_a = torch.empty((na,), dtype=torch.int32, device=dev)
        area_b = torch.empty((nb,), dtype=torch.int32, device=dev)
        rc = _lib.lib().cim_mask_pair_ratio(_lib.ptr(pa), _lib.ptr(pb), na, nb, words, _RATIO_MODES[mode],
                                            _lib.ptr(ratio), _lib.ptr(inter), _lib.ptr(area_a), _lib.ptr(area_b),
                                            _lib.stream_ptr(dev))
    _lib.check(rc, "cim_mask_pair_ratio")
    return (ratio, inter, area_a, area_b) if return_counts else ratio


def mask_iou(mask_a, mask_b):
    """lib/utils/mask_utils.py:6-18."""
    return mask_pair_ratio(mask_a, mask_b, "iou")


def mask_asymmetric_iou(mask_a, mask_b):
    """lib/utils/mask_utils.py:20-32 (the denominator is mask_b.sum() over ALL masks of b, as written there)."""
    return mask_pair_ratio(mask_a, mask_b, "asymmetric")


def mask_inside(mask_a, mask_b):
    """lib/utils/mask_utils.py:35-47."""
    return mask_pair_ratio(mask_a, mask_b, "inside")


def mask_outside(mask_a, mask_b):
    """lib/utils/mask_utils.py:50-62."""
    return mask_pair_ratio(mask_a, mask_b, "outside")


# ------------------------------------------------------------------ on-disk formats
def load_map_pickle(path, device="cuda:0", index=None):
    """Read a cob_iou / cob_asy_iou pickle written by the reference's tools/pre/create_cob_iou.py:48-49 /
    create_cob_asy_iou.py (one float16 [N, N] numpy array, pickle.HIGHEST_PROTOCOL) the way
    lib/modeling/model_builder.py:148-156 does: tensor on `device`, re-indexed [index][:, index] when given.
    Lets maps computed by the reference be replayed against the mining kernels, or compared with cim_mask_overlap."""
    import pickle
    with open(path, "rb") as f:
        arr = pickle.load(f)
    t = torch.as_tensor(arr, device=device)
    if t.dtype != torch.float16 or t.dim() != 2 or t.shape[0] != t.shape[1]:
        raise ValueError(f"{path}: expected a float16 [N, N] map, got {t.dtype} {tuple(t.shape)}")
    if index is not None:
        index = torch.as_tensor(index, device=device).long()
        t = t[index][:, index]
    return t.contiguous()


def save_map_pickle(path, map_f16):
    """Write a map in the reference's format (create_cob_iou.py:48-49), e.g. the output of mask_overlap, so the
    reference's training loop can consume maps produced here."""
    import pickle
    arr = map_f16.detach().cpu().numpy()
    if arr.dtype.name != "float16" or arr.ndim != 2:
        raise ValueError("expected a float16 [N, N] map")
    with open(path, "wb") as f:
        pickle.dump(arr, f, pickle.HIGHEST_PROTOCOL)


def save_packed_masks(path, packed, height, width, layout="flat"):
    """Bit-packed proposal-mask store (1 bit / pixel instead of the uint8 [N, H, W] arrays the reference keeps in
    COB .mat files: 8x smaller on disk and on the PCIe bus).  .npz with the words, the image size and the pixel
    order; load_packed_masks() returns what mask_overlap() takes."""
    import numpy as np
    np.savez_compressed(path, words=packed.detach().cpu().numpy(), height=np.int64(height), width=np.int64(width),
                        layout=np.bytes_(layout))


def load_packed_masks(path, device="cuda:0"):
    import numpy as np
    z = np.load(path)
    height, width = int(z["height"]), int(z["width"])
    layout = bytes(z["layout"]).decode()
    packed = torch.from_numpy(z["words"]).to(device)
    return _tag(packed, width // 16 if layout == "tiled" else 0), height, width, layout
