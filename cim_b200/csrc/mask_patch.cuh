// mask_patch.cuh -- the sparse update of one tiled bit mask and its metadata, shared by the two wires that fill the
// packed proposal-mask buffer from the host (bounding-box crops in mask_overlap.cu, COCO RLE strings in mask_rle.cu).
//
// A row of the buffer holds zeros outside the rectangle its last mask was written from (prev_rects: (wx0, y0, ww, h)
// in 32-pixel words x rows, all zero for a row of zeros).  An update visits the 8 x 16 patches of the union of the old
// and the new rectangle, stores every one of them (zeros where only the old mask was) and keeps what cim_mask_meta
// would compute: popcount, the K-block bitmap (rebuilt from zero in shared memory) and the occupied patch range.
#pragma once
#include "common.cuh"

// Column words of the RLE decoder's band bitmap in shared memory (32 KB): a 512 x 512 image is one band; the canvas
// width is limited to this many pixels.
constexpr int CIM_RLE_UNPACK_BITMAP_WORDS = 8192;

// Patch range [bx_lo, bx_hi) x [by_lo, by_hi) of the union of two rectangles, clipped to the bpr x nby patch grid.
__device__ __forceinline__ void patch_union(int4 a, int4 b, int bpr, int nby, int *bx_lo, int *bx_hi, int *by_lo,
                                            int *by_hi) {
    int xl = bpr, xh = 0, yl = nby, yh = 0;
    if (a.z > 0 && a.w > 0) { xl = min(xl, 2 * a.x); xh = max(xh, 2 * (a.x + a.z)); yl = min(yl, a.y >> 3); yh = max(yh, ((a.y + a.w - 1) >> 3) + 1); }
    if (b.z > 0 && b.w > 0) { xl = min(xl, 2 * b.x); xh = max(xh, 2 * (b.x + b.z)); yl = min(yl, b.y >> 3); yh = max(yh, ((b.y + b.w - 1) >> 3) + 1); }
    *bx_lo = max(xl, 0); *by_lo = max(yl, 0); *bx_hi = min(xh, bpr); *by_hi = min(yh, nby);
}

struct PatchMeta {
    int s = 0, alo = 0x7fffffff, ahi = -1, blo = 0x7fffffff, bhi = -1;

    // store patch (bx, by) = K-block kb of the row and account for it; bm = the row's K-block bitmap in shared memory
    __device__ __forceinline__ void store(uint4 *row4, uint32_t *bm, int kb, int bx, int by, uint4 v) {
        row4[kb] = v;
        s += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
        if ((v.x | v.y | v.z | v.w) != 0u) {
            atomicOr(bm + (kb >> 5), 1u << (kb & 31));
            alo = min(alo, bx); ahi = max(ahi, bx); blo = min(blo, by); bhi = max(bhi, by);
        }
    }

    __device__ __forceinline__ void warp_reduce() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            alo = min(alo, __shfl_xor_sync(0xffffffffu, alo, o));
            ahi = max(ahi, __shfl_xor_sync(0xffffffffu, ahi, o));
            blo = min(blo, __shfl_xor_sync(0xffffffffu, blo, o));
            bhi = max(bhi, __shfl_xor_sync(0xffffffffu, bhi, o));
        }
    }

    // the row's area and sort-key inputs (cim_mask_meta's kinfo)
    __device__ __forceinline__ void write(int32_t *area, int4 *kinfo, long long m) const {
        area[m] = s;
        kinfo[m] = ahi >= 0 ? make_int4(1, alo + ahi, blo + bhi, 0) : make_int4(0, 0, 0, 0);
    }
};
