// mask_overlap.cu -- pairwise mask-proposal IoU and containment maps for sm_100a.
//
// Replaces lib/utils/mask_utils.py:6-18 (mask_iou) and :20-32 (mask_asymmetric_iou) of the
// reference as driven by tools/pre/create_cob_iou.py:43-48 / create_cob_asy_iou.py:43-51
// (N^2 pairs, two cupy reductions each, float16 cast, pickled, re-loaded every training step
// at lib/modeling/model_builder.py:148-156).
//
//   inter[i,j] = |m_i & m_j|         exact integer
//   iou[i,j]   = fp16( fp32(inter) / fp32(area_i + area_j - inter) )
//   asy[i,j]   = fp16( fp32(inter) / fp32(area_j) )                  0/0 -> NaN like numpy
//
// The reference divides in float64 and stores into float32 before the float16 cast; for integer
// operands below 2^24 the float64 quotient can never sit close enough to a float32 rounding
// boundary for the double rounding to matter, so one IEEE fp32 division gives the same float32
// (tests/test_oracle_masks.py checks this exhaustively for small counts).  The fp32 -> fp16 step
// is kept as a second rounding exactly as in the reference.
//
// Kernels in this file:
//   mask_pack_kernel      byte masks -> bit masks (32 pixels per word), HBM-bound streaming
//   mask_area_kernel      per-mask popcount
//   mask_overlap_popc     64x64 output tile per CTA over bit-packed rows: AND + POPC, only the
//                         upper triangle of tiles is computed, the mirror tile is written from
//                         the same counts (inter is symmetric, asy is not)
#include "common.cuh"
#include "mask_patch.cuh"

// mask_overlap_tc.cu: the tcgen05 (tensor core) path for large problems
bool cim_mask_overlap_tc_eligible(int n, long long words);
int cim_mask_overlap_tc_launch(const uint32_t *packed, const int32_t *area, const int32_t *perm,
                               const uint32_t *umap_a, const uint32_t *umap_b, int bw, unsigned long long *visited,
                               const int32_t *tile_order, int n_img, int n, long long words, int32_t *inter,
                               __half *iou, __half *asy, cudaStream_t st);
// mask_rle.cu: COCO RLE strings -> tiled bit masks + metadata (cim_mask_unpack_rle_tiled_meta_sparse)
int cim_mask_unpack_rle_launch(const uint8_t *chars, long long n_chars, const int64_t *off, const int32_t *len,
                               const int32_t *mask_hw, uint32_t *packed, int32_t *prev_rects, int32_t *area,
                               uint32_t *kbmap, int4 *kinfo, long long n_masks, int n, int H, int W, long long words,
                               int bw, int32_t *bad, cudaStream_t st);

namespace {

// ---------------------------------------------------------------------------------------- pack
__device__ __forceinline__ uint32_t nibble_of(uint32_t four_bytes) {
    // 0xFF per non-zero byte, keep bit i of byte i, add the bytes up in the top byte
    uint32_t m = __vcmpne4(four_bytes, 0u) & 0x08040201u;
    return (m * 0x01010101u) >> 24;
}

__global__ void mask_pack_kernel(const uint8_t *__restrict__ masks, uint32_t *__restrict__ packed,
                                 long long n_masks, long long hw, long long words) {
    const long long total = n_masks * words;
    const bool vec = (hw % 16) == 0 && (((uintptr_t)masks) % 16) == 0;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long m = idx / words, w = idx - m * words;
        const long long p0 = w * 32;
        const uint8_t *src = masks + m * hw + p0;
        uint32_t bits = 0;
        if (vec && p0 + 32 <= hw) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(src));
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(src) + 1);
            bits = nibble_of(a.x) | (nibble_of(a.y) << 4) | (nibble_of(a.z) << 8) | (nibble_of(a.w) << 12) |
                   (nibble_of(b.x) << 16) | (nibble_of(b.y) << 20) | (nibble_of(b.z) << 24) |
                   (nibble_of(b.w) << 28);
        } else {
            for (int i = 0; i < 32; ++i)
                if (p0 + i < hw && src[i] != 0) bits |= 1u << i;
        }
        packed[idx] = bits;
    }
}

// Tiled layout ("8 x 16"): pixel (y, x) of an H x W mask (H % 8 == 0, W % 16 == 0) sits at flat position
//   q = ((y >> 3) * (W >> 4) + (x >> 4)) * 128 + (y & 7) * 16 + (x & 15),   bit q & 31 of word q >> 5,
// so 4 consecutive words (one 128-pixel K-block of the tensor-core overlap kernel) are one 8 x 16 pixel
// patch.  Counts and overlaps do not depend on the pixel order; the patch order makes the set of K-blocks a
// mask touches follow its 2-D footprint, which lets the overlap kernel skip far more of them.
__device__ __forceinline__ uint32_t bits16_of(const uint4 a) {
    return nibble_of(a.x) | (nibble_of(a.y) << 4) | (nibble_of(a.z) << 8) | (nibble_of(a.w) << 12);
}
__global__ void mask_pack_tiled_kernel(const uint8_t *__restrict__ masks, uint32_t *__restrict__ packed,
                                       long long n_masks, int H, int W, long long words) {
    const long long total = n_masks * words;
    const long long used = (long long)H * W / 32;
    const int bpr = W >> 4;
    const bool vec = (((uintptr_t)masks) % 16) == 0;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long m = idx / words, w = idx - m * words;
        uint32_t bits = 0;
        if (w < used) {
            const int blk = (int)(w >> 2), wi = (int)(w & 3), by = blk / bpr, bx = blk - by * bpr;
            const uint8_t *src = masks + m * (long long)H * W + (long long)(8 * by + 2 * wi) * W + 16 * bx;
            if (vec) {
                bits = bits16_of(__ldg(reinterpret_cast<const uint4 *>(src))) |
                       (bits16_of(__ldg(reinterpret_cast<const uint4 *>(src + W))) << 16);
            } else {
                for (int i = 0; i < 16; ++i) {
                    if (src[i] != 0) bits |= 1u << i;
                    if (src[W + i] != 0) bits |= 1u << (16 + i);
                }
            }
        }
        packed[idx] = bits;
    }
}

// crop word (row y, pixels 32 X .. 32 X + 31) -> two 16-pixel halves = one half-word each in the tiled layout
__global__ void mask_unpack_crops_tiled_kernel(const uint32_t *__restrict__ crop_words, const int32_t *__restrict__ meta,
                                               const long long *__restrict__ off, uint32_t *__restrict__ packed,
                                               int H, int W, long long words) {
    const long long m = blockIdx.x;
    const int wx0 = meta[4 * m], y0 = meta[4 * m + 1], ww = meta[4 * m + 2], h = meta[4 * m + 3];
    const uint32_t *src = crop_words + off[m];
    unsigned short *dst = reinterpret_cast<unsigned short *>(packed + m * words);
    const int bpr = W >> 4;
    for (int e = threadIdx.x; e < ww * h; e += blockDim.x) {
        const int r = e / ww, k = e - r * ww;
        const int y = y0 + r, x = 32 * (wx0 + k);
        if (y < 0 || y >= H || x < 0 || x >= W) continue;
        const uint32_t w = __ldg(src + e);
        if (w == 0u) continue;
        const long long blk = (long long)(y >> 3) * bpr + (x >> 4);
        const int hw = ((y & 7) >> 1) * 2 + (y & 1);                 // half-word inside the block
        if (w & 0xffffu) dst[blk * 8 + hw] = (unsigned short)(w & 0xffffu);
        if ((w >> 16) && x + 16 < W) dst[(blk + 1) * 8 + hw] = (unsigned short)(w >> 16);
    }
}

// Crops -> tiled bit masks AND their metadata in ONE pass, one warp per mask: a lane builds one K-block (an 8 x 16
// pixel patch = 4 words = rows 2j, 2j + 1 of the patch per word) from the crop words that cover it (or zeros outside
// the crop: no memset of the 524 MB beforehand), stores it with one 16-byte store, and keeps what mask_area_kernel
// would have to re-read the masks for: popcount, the ballot of "patch not empty" (= one word of the K-block bitmap)
// and the occupied block range (sort key).
__global__ void mask_unpack_crops_tiled_meta_kernel(const uint32_t *__restrict__ crop_words, const int32_t *__restrict__ meta,
                                                    const long long *__restrict__ off, uint32_t *__restrict__ packed,
                                                    int32_t *__restrict__ area, uint32_t *__restrict__ kbmap,
                                                    int4 *__restrict__ kinfo, long long n_masks, int H, int W,
                                                    long long words, int bw) {
    const long long m = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= n_masks) return;
    const int lane = threadIdx.x & 31;
    const int wx0 = meta[4 * m], y0 = meta[4 * m + 1], ww = meta[4 * m + 2], h = meta[4 * m + 3];
    const uint32_t *src = crop_words + off[m];
    uint4 *row4 = reinterpret_cast<uint4 *>(packed + m * words);
    const int bpr = W >> 4, nkb = (int)(words >> 2), nblk = (H >> 3) * bpr;
    int s = 0, alo = 0x7fffffff, ahi = -1, blo = 0x7fffffff, bhi = -1;
    for (int j = 0; j < bw; ++j) {
        const int kb = j * 32 + lane;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (kb < nblk) {
            const int by = kb / bpr, bx = kb - by * bpr;
            const int k = (bx >> 1) - wx0;                       // crop word column holding these 16 pixels
            if (k >= 0 && k < ww) {
                const int sh = (bx & 1) * 16;
                uint32_t o[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int r0 = 8 * by + 2 * q - y0, r1 = r0 + 1;
                    const uint32_t lo = (r0 >= 0 && r0 < h) ? (__ldg(src + (long long)r0 * ww + k) >> sh) & 0xffffu : 0u;
                    const uint32_t hi = (r1 >= 0 && r1 < h) ? (__ldg(src + (long long)r1 * ww + k) >> sh) & 0xffffu : 0u;
                    o[q] = lo | (hi << 16);
                }
                v = make_uint4(o[0], o[1], o[2], o[3]);
            }
        }
        if (kb < nkb) row4[kb] = v;
        s += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
        const bool nz = (v.x | v.y | v.z | v.w) != 0u;
        const uint32_t bm = __ballot_sync(0xffffffffu, nz);
        if (lane == 0) kbmap[m * bw + j] = bm;
        if (nz) {
            const int by = kb / bpr, bx = kb - by * bpr;
            alo = min(alo, bx); ahi = max(ahi, bx); blo = min(blo, by); bhi = max(bhi, by);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        alo = min(alo, __shfl_xor_sync(0xffffffffu, alo, o));
        ahi = max(ahi, __shfl_xor_sync(0xffffffffu, ahi, o));
        blo = min(blo, __shfl_xor_sync(0xffffffffu, blo, o));
        bhi = max(bhi, __shfl_xor_sync(0xffffffffu, bhi, o));
    }
    if (lane == 0) {
        area[m] = s;
        kinfo[m] = ahi >= 0 ? make_int4(1, alo + ahi, blo + bhi, 0) : make_int4(0, 0, 0, 0);
    }
}

// The same, as a SPARSE UPDATE of a buffer that already holds an earlier batch of unpacked crops (and zeros everywhere
// else): prev[m] = the crop rectangle (wx0, y0, ww, h) of the mask currently stored in row m, all zero for an empty row.
// A warp only visits the patches of the bounding rectangle of the old and the new crop -- it writes the new patch
// (zeros where only the old crop was) -- instead of all H * W / 128 of them: masks cover a few percent of the image, so
// a step re-writes ~10 % of the 524 MB instead of all of it.  The K-block bitmap (64 words per mask) is rebuilt in
// shared memory and written whole; prev[m] becomes the new rectangle.
__global__ void mask_unpack_crops_tiled_meta_sparse_kernel(const uint32_t *__restrict__ crop_words,
                                                           const int32_t *__restrict__ meta, const long long *__restrict__ off,
                                                           uint32_t *__restrict__ packed, int4 *__restrict__ prev,
                                                           int32_t *__restrict__ area, uint32_t *__restrict__ kbmap,
                                                           int4 *__restrict__ kinfo, long long n_masks, int H, int W,
                                                           long long words, int bw) {
    extern __shared__ uint32_t s_bitmaps[];                      // [warps][bw]
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long m = blockIdx.x * (long long)(blockDim.x >> 5) + wib;
    if (m >= n_masks) return;
    uint32_t *bm = s_bitmaps + wib * bw;
    for (int j = lane; j < bw; j += 32) bm[j] = 0u;
    const int wx0 = meta[4 * m], y0 = meta[4 * m + 1], ww = meta[4 * m + 2], h = meta[4 * m + 3];
    const int4 pv = prev[m];
    const uint32_t *src = crop_words + off[m];
    uint4 *row4 = reinterpret_cast<uint4 *>(packed + m * words);
    const int bpr = W >> 4, nby = H >> 3;
    // patch rectangle (16-pixel columns x 8-pixel rows) of the new and the old crop, clipped to the image
    int bx_lo, bx_hi, by_lo, by_hi;                              // [lo, hi)
    patch_union(make_int4(wx0, y0, ww, h), pv, bpr, nby, &bx_lo, &bx_hi, &by_lo, &by_hi);
    const int nx = max(bx_hi - bx_lo, 0), cells = nx * max(by_hi - by_lo, 0);
    PatchMeta acc;
    __syncwarp();
    for (int e = lane; e < cells; e += 32) {
        const int by = by_lo + e / nx, bx = bx_lo + e % nx, kb = by * bpr + bx;
        const int k = (bx >> 1) - wx0;                           // crop word column holding these 16 pixels
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (k >= 0 && k < ww) {
            const int sh = (bx & 1) * 16;
            uint32_t o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int r0 = 8 * by + 2 * q - y0, r1 = r0 + 1;
                const uint32_t lo = (r0 >= 0 && r0 < h) ? (__ldg(src + (long long)r0 * ww + k) >> sh) & 0xffffu : 0u;
                const uint32_t hi = (r1 >= 0 && r1 < h) ? (__ldg(src + (long long)r1 * ww + k) >> sh) & 0xffffu : 0u;
                o[q] = lo | (hi << 16);
            }
            v = make_uint4(o[0], o[1], o[2], o[3]);
        }
        acc.store(row4, bm, kb, bx, by, v);
    }
    acc.warp_reduce();
    __syncwarp();
    for (int j = lane; j < bw; j += 32) kbmap[m * bw + j] = bm[j];
    if (lane == 0) {
        acc.write(area, kinfo, m);
        prev[m] = make_int4(wx0, y0, ww, h);
    }
}

// ------------------------------------------------------------------------------- unpack crops
// Wire format for proposal masks (host -> device): only the bounding box of every mask is sent.
// crop row r, word k holds pixels (y0 + r, 32 * wx0 + 32 k .. + 31); it is OR-ed into the flat
// bit-packed mask (pixel p = y * W + x -> bit p & 31 of word p >> 5) with a funnel shift when the
// image width is not a multiple of 32.  One CTA per mask; `packed` is zeroed beforehand.
__global__ void mask_unpack_crops_kernel(const uint32_t *__restrict__ crop_words, const int32_t *__restrict__ meta,
                                         const long long *__restrict__ off, uint32_t *__restrict__ packed,
                                         int H, int W, long long words) {
    const long long m = blockIdx.x;
    const int wx0 = meta[4 * m], y0 = meta[4 * m + 1], ww = meta[4 * m + 2], h = meta[4 * m + 3];
    const uint32_t *src = crop_words + off[m];
    uint32_t *dst = packed + m * words;
    const bool aligned = (W & 31) == 0;
    for (int e = threadIdx.x; e < ww * h; e += blockDim.x) {
        const int r = e / ww, k = e - r * ww;
        const int y = y0 + r, x = 32 * (wx0 + k);
        if (y < 0 || y >= H || x < 0 || x >= W) continue;
        uint32_t w = __ldg(src + e);
        if (x + 32 > W) w &= (1u << (W - x)) - 1u;             // bits beyond the image row are dropped
        if (w == 0u) continue;
        const long long p = (long long)y * W + x;
        const long long wi = p >> 5;
        const int sh = (int)(p & 31);
        if (aligned) {
            dst[wi] = w;                                        // every output word has one source word
        } else {
            atomicOr(dst + wi, w << sh);
            if (sh != 0 && (w >> (32 - sh)) != 0u) atomicOr(dst + wi + 1, w >> (32 - sh));
        }
    }
}

// ---------------------------------------------------------------------------------------- area
// per mask (one warp): popcount; for the tensor path also the occupancy bitmap over K-blocks of 4 words
// (bit kb & 31 of kbmap word kb >> 5) and the sort key inputs: kinfo = (any, a, b) with
//   kb_per_row == 0 (flat pixel order):  a = first + last occupied K-block, b = 0
//   kb_per_row  > 0 (tiled layout)    :  a = min + max block column, b = min + max block row
__global__ void mask_area_kernel(const uint32_t *__restrict__ packed, int32_t *__restrict__ area,
                                 uint32_t *__restrict__ kbmap, int4 *__restrict__ kinfo, long long n_masks,
                                 long long words, int bw, int kb_per_row) {
    const long long m = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= n_masks) return;
    const int lane = threadIdx.x & 31;
    const uint32_t *row = packed + m * words;
    int s = 0;
    if (!kbmap) {                                    // popcount only (popc path)
        for (long long w = lane; w < words; w += 32) s += __popc(__ldg(row + w));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) area[m] = s;
        return;
    }
    // tensor path: words % 4 == 0 and 16-byte aligned rows; a lane takes one K-block (4 words) per round, so
    // the ballot of "non-zero" IS the bitmap word of the round
    int alo = 0x7fffffff, ahi = -1, blo = 0x7fffffff, bhi = -1;
    const int nkb = (int)(words >> 2);
    const uint4 *row4 = reinterpret_cast<const uint4 *>(row);
    for (int j = 0; j < bw; ++j) {
        const int kb = j * 32 + lane;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (kb < nkb) v = __ldg(row4 + kb);
        s += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
        const bool nz = (v.x | v.y | v.z | v.w) != 0u;
        const uint32_t bm = __ballot_sync(0xffffffffu, nz);
        if (lane == 0) kbmap[m * bw + j] = bm;
        if (nz) {
            if (kb_per_row > 0) {
                const int by = kb / kb_per_row, bx = kb - by * kb_per_row;
                alo = min(alo, bx); ahi = max(ahi, bx); blo = min(blo, by); bhi = max(bhi, by);
            } else {
                alo = min(alo, kb); ahi = max(ahi, kb);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        alo = min(alo, __shfl_xor_sync(0xffffffffu, alo, o));
        ahi = max(ahi, __shfl_xor_sync(0xffffffffu, ahi, o));
        blo = min(blo, __shfl_xor_sync(0xffffffffu, blo, o));
        bhi = max(bhi, __shfl_xor_sync(0xffffffffu, bhi, o));
    }
    if (lane == 0) {
        area[m] = s;
        kinfo[m] = ahi >= 0 ? make_int4(1, alo + ahi, bhi >= 0 ? blo + bhi : 0, 0) : make_int4(0, 0, 0, 0);
    }
}

// ------------------------------------------------------------------------- locality sort + unions
// One CTA per image.  Masks are sorted by position so that the 128 / 256 masks of a tile block cover a small
// part of the image: flat pixel order -> by the centre of the occupied K-block range (= vertical position);
// tiled layout -> three vertical stripes by block-column centre, inside a stripe by block-row centre
// (alternating direction, so neighbours in the order stay neighbours in the image).
// perm[k] = original index of the k-th mask in sorted order, inv = inverse.  For every block of 128 (A
// operand) and 256 (B operand) sorted masks the union of the masks' K-block bitmaps is stored; a tile only
// has to visit the K-blocks set in BOTH unions: everywhere else one operand is all zero.
__global__ void __launch_bounds__(1024)
mask_sort_kernel(const int4 *__restrict__ kinfo_all, int n, int npad, int kb_per_row, int nkb,
                 int32_t *__restrict__ perm_all, int32_t *__restrict__ inv_all) {
    extern __shared__ __align__(16) unsigned char sort_smem[];
    int *key = reinterpret_cast<int *>(sort_smem);        // [npad]
    int *idx = key + npad;                                // [npad]
    const int img = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int4 *ki = kinfo_all + (size_t)img * n;
    const int nby = kb_per_row > 0 ? (nkb + kb_per_row - 1) / kb_per_row : 0;
    for (int i = tid; i < npad; i += nthr) {
        int k = 0x7fffffff;
        if (i < n) {
            const int4 v = ki[i];
            if (!v.x) k = 0;                               // empty masks first
            else if (kb_per_row > 0) {
                const int st = min(2, (v.y * 3) / (2 * kb_per_row));
                k = (st << 24) | ((st & 1) ? (2 * nby - v.z) : v.z);
            } else k = v.y;
        }
        key[i] = k;
        idx[i] = i < n ? i : 0x7fffffff;
    }
    __syncthreads();
    for (int size = 2; size <= npad; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (npad >> 1); t += nthr) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const int ka = key[lo], kb = key[hi], ia = idx[lo], ib = idx[hi];
                const bool a_first = ka < kb || (ka == kb && ia < ib);
                if (asc ? !a_first : a_first) { key[lo] = kb; key[hi] = ka; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    int32_t *perm = perm_all + (size_t)img * n, *inv = inv_all + (size_t)img * n;
    for (int i = tid; i < n; i += nthr) { perm[i] = idx[i]; inv[idx[i]] = i; }
}

// union bitmaps of the sorted 128- (A operand) and 256-mask (B operand) blocks: one CTA per (block, image), one
// thread per bitmap word (the sort kernel used to do this with its 8 CTAs: 55 us of the stage)
__global__ void __launch_bounds__(128)
mask_union_kernel(const uint32_t *__restrict__ kbmap_all, const int32_t *__restrict__ perm_all, int n, int bw,
                  uint32_t *__restrict__ umap_a, uint32_t *__restrict__ umap_b, int nrb, int ncb) {
    const int blk = blockIdx.x, img = blockIdx.y;
    const bool is_a = blk < nrb;
    const int bs = is_a ? 128 : 256, b0 = (is_a ? blk : blk - nrb) * bs, b1 = min(n, b0 + bs);
    const uint32_t *kbm = kbmap_all + (size_t)img * n * bw;
    const int32_t *perm = perm_all + (size_t)img * n;
    __shared__ int s_idx[256];
    for (int i = threadIdx.x; i < b1 - b0; i += blockDim.x) s_idx[i] = perm[b0 + i];
    __syncthreads();
    for (int j = threadIdx.x; j < bw; j += blockDim.x) {
        uint32_t u = 0;
#pragma unroll 8
        for (int i = 0; i < b1 - b0; ++i) u |= __ldg(kbm + (size_t)s_idx[i] * bw + j);
        if (is_a) umap_a[((size_t)img * nrb + blk) * bw + j] = u;
        else umap_b[((size_t)img * ncb + (blk - nrb)) * bw + j] = u;
    }
}

// Longest tile first, per image: the CTA ranks ITS image's tiles by the number of K-blocks they visit and writes rank
// r to tile_order[r * n_img + img] -- the images' rankings interleaved, which starts the long tiles of every image
// first without a single-CTA sort over all tiles (mask_tile_order_kernel: 28 us at cfg2).
__global__ void __launch_bounds__(256)
mask_rank_kernel(const uint32_t *__restrict__ umap_a, const uint32_t *__restrict__ umap_b, int bw, int nrb, int ncb,
                 int per_img, int tpad, int32_t *__restrict__ tile_order) {
    extern __shared__ __align__(16) unsigned char sort_smem[];
    int *key = reinterpret_cast<int *>(sort_smem);        // [tpad]
    int *idx = key + tpad;                                // [tpad]
    const int img = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    for (int t = tid; t < tpad; t += nthr) { key[t] = t < per_img ? 0 : 0x7fffffff; idx[t] = -1; }
    __syncthreads();
    for (int e = tid; e < per_img * bw; e += nthr) {      // (tile, bitmap word): coalesced over the words
        const int t = e / bw, j = e - t * bw;
        int rem = t, ti = 0;
        while (rem >= ncb - (ti >> 1)) { rem -= ncb - (ti >> 1); ++ti; }
        const int tj = (ti >> 1) + rem;
        const int c = __popc(__ldg(umap_a + ((size_t)img * nrb + ti) * bw + j) &
                             __ldg(umap_b + ((size_t)img * ncb + tj) * bw + j));
        if (c) atomicSub(&key[t], c);
        if (j == 0) idx[t] = (img << 16) | (ti << 8) | tj;
    }
    __syncthreads();
    for (int size = 2; size <= tpad; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (tpad >> 1); t += nthr) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const int ka = key[lo], kb = key[hi], ia = idx[lo], ib = idx[hi];
                const bool a_first = ka < kb || (ka == kb && ia < ib);
                if (asc ? !a_first : a_first) { key[lo] = kb; key[hi] = ka; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    for (int t = tid; t < per_img; t += nthr) tile_order[(size_t)t * gridDim.x + img] = idx[t];
}

// out[i][j] = tmp[inv[i]][inv[j]] for both fp16 maps: one CTA per output row, the source rows go through smem
__global__ void __launch_bounds__(256)
mask_unpermute2_kernel(const __half *__restrict__ tmp_a, const __half *__restrict__ tmp_b,
                       const int32_t *__restrict__ inv_all, __half *__restrict__ out_a, __half *__restrict__ out_b,
                       int n) {
    extern __shared__ __align__(16) unsigned char unp_smem[];
    __half *ra = reinterpret_cast<__half *>(unp_smem), *rb = ra + n;
    const int i = blockIdx.x, img = blockIdx.y;
    const int32_t *inv = inv_all + (size_t)img * n;
    const size_t so = ((size_t)img * n + inv[i]) * n, d_o = ((size_t)img * n + i) * n;
    if ((n & 7) == 0) {
        const uint4 *sa = reinterpret_cast<const uint4 *>(tmp_a + so), *sb = reinterpret_cast<const uint4 *>(tmp_b + so);
        for (int j = threadIdx.x; j < n / 8; j += blockDim.x) {
            reinterpret_cast<uint4 *>(ra)[j] = __ldg(sa + j);
            reinterpret_cast<uint4 *>(rb)[j] = __ldg(sb + j);
        }
    } else {
        for (int j = threadIdx.x; j < n; j += blockDim.x) { ra[j] = tmp_a[so + j]; rb[j] = tmp_b[so + j]; }
    }
    __syncthreads();
    if ((n & 1) == 0) {
        for (int j = threadIdx.x; j < n / 2; j += blockDim.x) {
            const int c0 = inv[2 * j], c1 = inv[2 * j + 1];
            reinterpret_cast<__half2 *>(out_a + d_o)[j] = __halves2half2(ra[c0], ra[c1]);
            reinterpret_cast<__half2 *>(out_b + d_o)[j] = __halves2half2(rb[c0], rb[c1]);
        }
    } else {
        for (int j = threadIdx.x; j < n; j += blockDim.x) { out_a[d_o + j] = ra[inv[j]]; out_b[d_o + j] = rb[inv[j]]; }
    }
}

// out[i][j] = tmp[inv[i]][inv[j]]: one CTA per output row, the source row goes through smem
template <typename T>
__global__ void __launch_bounds__(256)
mask_unpermute_kernel(const T *__restrict__ tmp_all, const int32_t *__restrict__ inv_all, T *__restrict__ out_all,
                      int n) {
    extern __shared__ __align__(16) unsigned char unp_smem[];
    T *row = reinterpret_cast<T *>(unp_smem);
    const int i = blockIdx.x, img = blockIdx.y;
    const int32_t *inv = inv_all + (size_t)img * n;
    const T *src = tmp_all + ((size_t)img * n + inv[i]) * n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) row[j] = src[j];
    __syncthreads();
    T *dst = out_all + ((size_t)img * n + i) * n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) dst[j] = row[inv[j]];
}

// --------------------------------------------------------------------------------- popc overlap
constexpr int TS = 64;      // output tile side
constexpr int KC = 32;      // words per k-chunk
constexpr int KP = KC + 1;  // padded smem pitch

__device__ __forceinline__ void write_pair(int32_t *inter, __half *iou, __half *asy, size_t idx, int I,
                                           int a_row, int a_col) {
    const float fi = (float)I;
    if (inter) inter[idx] = I;
    iou[idx] = __float2half_rn(__fdiv_rn(fi, (float)(a_row + a_col - I)));
    asy[idx] = __float2half_rn(__fdiv_rn(fi, (float)a_col));
}

__global__ void __launch_bounds__(256)
mask_overlap_popc_kernel(const uint32_t *__restrict__ packed, const int32_t *__restrict__ area_all,
                         int n, long long words, int32_t *__restrict__ inter_all, __half *__restrict__ iou_all,
                         __half *__restrict__ asy_all) {
    __shared__ uint32_t As[TS][KP];
    __shared__ uint32_t Bs[TS][KP];
    const int img = blockIdx.y;
    // linear id -> (ti, tj) with ti <= tj
    const int nt = (n + TS - 1) / TS;
    int ti = 0, rem = blockIdx.x;
    while (rem >= nt - ti) { rem -= nt - ti; ++ti; }
    const int tj = ti + rem;

    const uint32_t *base = packed + (size_t)img * n * words;
    const int32_t *area = area_all + (size_t)img * n;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0;

    for (long long k0 = 0; k0 < words; k0 += KC) {
        // 64 rows x 32 words per operand, 256 threads: 8 words each, coalesced along k
#pragma unroll
        for (int it = 0; it < (TS * KC) / 256; ++it) {
            const int e = it * 256 + tid, row = e / KC, kk = e % KC;
            const long long kw = k0 + kk;
            const int ra = ti * TS + row, rb = tj * TS + row;
            As[row][kk] = (ra < n && kw < words) ? __ldg(base + (size_t)ra * words + kw) : 0u;
            Bs[row][kk] = (rb < n && kw < words) ? __ldg(base + (size_t)rb * words + kw) : 0u;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < KC; ++kk) {
            uint32_t a[4], b[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) a[r] = As[ty + 16 * r][kk];
#pragma unroll
            for (int c = 0; c < 4; ++c) b[c] = Bs[tx + 16 * c][kk];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] += __popc(a[r] & b[c]);
        }
        __syncthreads();
    }

    int32_t *inter = inter_all ? inter_all + (size_t)img * n * n : nullptr;
    __half *iou = iou_all + (size_t)img * n * n;
    __half *asy = asy_all + (size_t)img * n * n;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = ti * TS + ty + 16 * r;
        if (i >= n) continue;
        const int ai = area[i];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = tj * TS + tx + 16 * c;
            if (j >= n) continue;
            const int aj = area[j];
            write_pair(inter, iou, asy, (size_t)i * n + j, acc[r][c], ai, aj);
            if (ti != tj) write_pair(inter, iou, asy, (size_t)j * n + i, acc[r][c], aj, ai);
        }
    }
}

}  // namespace

CIM_API int cim_mask_pack(const uint8_t *masks, uint32_t *packed, int64_t n_masks, int64_t hw, int64_t words,
                          cim_stream_t stream) {
    if (!masks || !packed || n_masks < 0 || hw <= 0 || words * 32 < hw) return CIM_ERR_ARG;
    if (n_masks == 0) return CIM_OK;
    const long long total = n_masks * words;
    const int blocks = (int)min((long long)cim_num_sms() * 16, (total + 255) / 256);
    mask_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(masks, packed, n_masks, hw, words);
    return cim_launch_status();
}

CIM_API int cim_mask_pack_tiled(const uint8_t *masks, uint32_t *packed, int64_t n_masks, int H, int W, int64_t words,
                                cim_stream_t stream) {
    if (!masks || !packed || n_masks < 0 || H <= 0 || W <= 0 || words * 32 < (int64_t)H * W) return CIM_ERR_ARG;
    if ((H & 7) || (W & 15)) return CIM_ERR_SHAPE;
    if (n_masks == 0) return CIM_OK;
    const long long total = n_masks * words;
    const int blocks = (int)min((long long)cim_num_sms() * 16, (total + 255) / 256);
    mask_pack_tiled_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(masks, packed, n_masks, H, W, words);
    return cim_launch_status();
}

CIM_API int cim_mask_unpack_crops_tiled(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                        uint32_t *packed, int64_t n_masks, int H, int W, int64_t words,
                                        cim_stream_t stream) {
    if (!crop_words || !crop_meta || !crop_off || !packed || n_masks < 0 || H <= 0 || W <= 0) return CIM_ERR_ARG;
    if (words * 32 < (int64_t)H * W) return CIM_ERR_ARG;
    if ((H & 7) || (W & 15)) return CIM_ERR_SHAPE;
    if (n_masks == 0) return CIM_OK;
    if (n_masks > 0x7fffffffLL) return CIM_ERR_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(packed, 0, sizeof(uint32_t) * (size_t)n_masks * words, st);
    mask_unpack_crops_tiled_kernel<<<(unsigned)n_masks, 128, 0, st>>>(crop_words, crop_meta,
                                                                      reinterpret_cast<const long long *>(crop_off),
                                                                      packed, H, W, words);
    return cim_launch_status();
}

CIM_API int cim_mask_unpack_crops(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                  uint32_t *packed, int64_t n_masks, int H, int W, int64_t words,
                                  cim_stream_t stream) {
    if (!crop_words || !crop_meta || !crop_off || !packed || n_masks < 0 || H <= 0 || W <= 0) return CIM_ERR_ARG;
    if (words * 32 < (int64_t)H * W) return CIM_ERR_ARG;
    if (n_masks == 0) return CIM_OK;
    if (n_masks > 0x7fffffffLL) return CIM_ERR_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(packed, 0, sizeof(uint32_t) * (size_t)n_masks * words, st);
    mask_unpack_crops_kernel<<<(unsigned)n_masks, 128, 0, st>>>(crop_words, crop_meta,
                                                                reinterpret_cast<const long long *>(crop_off), packed,
                                                                H, W, words);
    return cim_launch_status();
}

namespace {
struct OverlapWs {
    unsigned long long *visited;      // word 0 of the workspace: K-blocks visited by the tensor path (diagnostic)
    int32_t *area;
    int4 *kinfo;
    uint32_t *kbmap, *umap_a, *umap_b;
    int32_t *perm, *inv, *tmp_inter, *tile_order;
    __half *tmp_iou, *tmp_asy;
    int bw;
    size_t bytes;
};
inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }
OverlapWs carve_overlap_ws(void *base, int n_img, int n, long long words, int want_inter) {
    OverlapWs w{};
    const size_t nm = (size_t)(n_img > 0 ? n_img : 0) * (size_t)(n > 0 ? n : 0), nn = nm * (size_t)(n > 0 ? n : 0);
    const size_t nrb = (size_t)n_img * ((n + 127) / 128), ncb = (size_t)n_img * ((n + 255) / 256);
    const long long nkb = (words + 3) / 4;
    w.bw = (int)((nkb + 31) / 32);
    char *p = (char *)base;
    size_t o = 0;
    auto take = [&](size_t bytes) { char *q = p ? p + o : nullptr; o += up256(bytes); return q; };
    w.visited = (unsigned long long *)take(8);
    w.area = (int32_t *)take(nm * 4);
    w.kinfo = (int4 *)take(nm * 16);
    w.kbmap = (uint32_t *)take(nm * w.bw * 4);
    w.perm = (int32_t *)take(nm * 4);
    w.inv = (int32_t *)take(nm * 4);
    w.umap_a = (uint32_t *)take(nrb * w.bw * 4);
    w.umap_b = (uint32_t *)take(ncb * w.bw * 4);
    w.tile_order = (int32_t *)take(nrb * ((size_t)(n + 255) / 256) * 4);
    w.tmp_iou = (__half *)take(nn * 2);
    w.tmp_asy = (__half *)take(nn * 2);
    w.tmp_inter = want_inter ? (int32_t *)take(nn * 4) : nullptr;
    w.bytes = o + 256;
    return w;
}
}  // namespace

namespace {
struct MaskMeta {
    int32_t *area;
    int4 *kinfo;
    uint32_t *kbmap;
    size_t bytes;
};
MaskMeta carve_meta(void *base, int n_img, int n, long long words) {
    MaskMeta m{};
    const size_t nm = (size_t)(n_img > 0 ? n_img : 0) * (size_t)(n > 0 ? n : 0);
    const int bw = (int)(((words + 3) / 4 + 31) / 32);
    char *p = (char *)base;
    size_t o = 0;
    auto take = [&](size_t bytes) { char *q = p ? p + o : nullptr; o += up256(bytes); return q; };
    m.area = (int32_t *)take(nm * 4);
    m.kinfo = (int4 *)take(nm * 16);
    m.kbmap = (uint32_t *)take(nm * bw * 4);
    m.bytes = o;
    return m;
}
}  // namespace

CIM_API size_t cim_mask_meta_bytes(int n_img, int n, int64_t words) { return carve_meta(nullptr, n_img, n, words).bytes; }

CIM_API int cim_mask_meta(const uint32_t *packed, int n_img, int n, int64_t words, int kb_per_row, void *meta,
                          size_t meta_bytes, cim_stream_t stream) {
    if (!packed || !meta || n_img < 0 || n < 0 || words <= 0 || kb_per_row < 0) return CIM_ERR_ARG;
    if ((words & 3) || !cim_aligned(packed, 16)) return CIM_ERR_ALIGN;
    if (meta_bytes < cim_mask_meta_bytes(n_img, n, words) || !cim_aligned(meta, 256)) return CIM_ERR_WORKSPACE;
    if (n_img == 0 || n == 0) return CIM_OK;
    const MaskMeta m = carve_meta(meta, n_img, n, words);
    const long long n_masks = (long long)n_img * n;
    const int bw = (int)(((words + 3) / 4 + 31) / 32);
    mask_area_kernel<<<(unsigned)((n_masks + 7) / 8), 256, 0, (cudaStream_t)stream>>>(packed, m.area, m.kbmap, m.kinfo,
                                                                                       n_masks, words, bw, kb_per_row);
    return cim_launch_status();
}

CIM_API int cim_mask_unpack_crops_tiled_meta(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                             uint32_t *packed, void *meta, size_t meta_bytes, int n_img, int n, int H,
                                             int W, int64_t words, cim_stream_t stream) {
    if (!crop_words || !crop_meta || !crop_off || !packed || !meta || n_img < 0 || n < 0 || H <= 0 || W <= 0)
        return CIM_ERR_ARG;
    if ((H & 7) || (W & 15)) return CIM_ERR_SHAPE;
    if (words * 32 != (int64_t)H * W || (words & 3) || !cim_aligned(packed, 16)) return CIM_ERR_ALIGN;
    if (meta_bytes < cim_mask_meta_bytes(n_img, n, words) || !cim_aligned(meta, 256)) return CIM_ERR_WORKSPACE;
    if (n_img == 0 || n == 0) return CIM_OK;
    const MaskMeta mm = carve_meta(meta, n_img, n, words);
    const long long n_masks = (long long)n_img * n;
    const int bw = (int)(((words + 3) / 4 + 31) / 32);
    mask_unpack_crops_tiled_meta_kernel<<<(unsigned)((n_masks + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        crop_words, crop_meta, reinterpret_cast<const long long *>(crop_off), packed, mm.area, mm.kbmap, mm.kinfo,
        n_masks, H, W, words, bw);
    return cim_launch_status();
}

CIM_API int cim_mask_unpack_crops_tiled_meta_sparse(const uint32_t *crop_words, const int32_t *crop_meta,
                                                    const int64_t *crop_off, uint32_t *packed, int32_t *prev_rects,
                                                    void *meta, size_t meta_bytes, int n_img, int n, int H, int W,
                                                    int64_t words, cim_stream_t stream) {
    if (!crop_words || !crop_meta || !crop_off || !packed || !prev_rects || !meta || n_img < 0 || n < 0 || H <= 0 || W <= 0)
        return CIM_ERR_ARG;
    if ((H & 7) || (W & 15)) return CIM_ERR_SHAPE;
    if (words * 32 != (int64_t)H * W || (words & 3) || !cim_aligned(packed, 16) || !cim_aligned(prev_rects, 16))
        return CIM_ERR_ALIGN;
    if (meta_bytes < cim_mask_meta_bytes(n_img, n, words) || !cim_aligned(meta, 256)) return CIM_ERR_WORKSPACE;
    if (n_img == 0 || n == 0) return CIM_OK;
    const MaskMeta mm = carve_meta(meta, n_img, n, words);
    const long long n_masks = (long long)n_img * n;
    const int bw = (int)(((words + 3) / 4 + 31) / 32);
    if ((size_t)bw * 8 * 4 > 48 * 1024) return CIM_ERR_SHAPE;          // bitmap of 8 masks in static-limit shared memory
    mask_unpack_crops_tiled_meta_sparse_kernel<<<(unsigned)((n_masks + 7) / 8), 256, (size_t)bw * 8 * 4, (cudaStream_t)stream>>>(
        crop_words, crop_meta, reinterpret_cast<const long long *>(crop_off), packed, reinterpret_cast<int4 *>(prev_rects),
        mm.area, mm.kbmap, mm.kinfo, n_masks, H, W, words, bw);
    return cim_launch_status();
}

CIM_API int cim_mask_unpack_rle_tiled_meta_sparse(const uint8_t *chars, int64_t n_chars, const int64_t *off,
                                                  const int32_t *len, const int32_t *mask_hw, uint32_t *packed,
                                                  int32_t *prev_rects, void *meta, size_t meta_bytes, int n_img, int n,
                                                  int H, int W, int64_t words, int32_t *bad, cim_stream_t stream) {
    if (!off || !len || !packed || !prev_rects || !meta || (n_chars > 0 && !chars) || n_chars < 0 || n_img < 0 ||
        n < 0 || H <= 0 || W <= 0)
        return CIM_ERR_ARG;
    if ((H & 7) || (W & 15) || (int64_t)H * W > 0x7fffffffLL || ((W + 31) & ~31) > CIM_RLE_UNPACK_BITMAP_WORDS)
        return CIM_ERR_SHAPE;
    if (words * 32 != (int64_t)H * W || (words & 3) || !cim_aligned(packed, 16) || !cim_aligned(prev_rects, 16) ||
        !cim_aligned(off, 8) || !cim_aligned(len, 4) || (mask_hw && !cim_aligned(mask_hw, 4)) ||
        (bad && !cim_aligned(bad, 4)))
        return CIM_ERR_ALIGN;
    if (meta_bytes < cim_mask_meta_bytes(n_img, n, words) || !cim_aligned(meta, 256)) return CIM_ERR_WORKSPACE;
    const long long n_masks = (long long)n_img * n;
    if (n_masks > 0x7fffffffLL) return CIM_ERR_SHAPE;
    const int bw = (int)(((words + 3) / 4 + 31) / 32);
    if (bw > 2048) return CIM_ERR_SHAPE;                                // the row's K-block bitmap in shared memory
    const MaskMeta mm = carve_meta(meta, n_img, n, words);
    return cim_mask_unpack_rle_launch(chars, n_chars, off, len, mask_hw, packed, prev_rects, mm.area, mm.kbmap,
                                      mm.kinfo, n_masks, n, H, W, words, bw, bad, (cudaStream_t)stream);
}

CIM_API size_t cim_mask_overlap_workspace_bytes(int n_img, int n, int64_t words, int want_inter) {
    return carve_overlap_ws(nullptr, n_img, n, words, want_inter).bytes;
}

CIM_API int cim_mask_overlap(const uint32_t *packed, int n_img, int n, int64_t words, int32_t *inter,
                             int32_t *area, void *iou_f16, void *asy_f16, void *workspace, size_t ws_bytes,
                             cim_stream_t stream) {
    return cim_mask_overlap_ex(packed, n_img, n, words, 0, inter, area, iou_f16, asy_f16, workspace, ws_bytes,
                               CIM_OVERLAP_AUTO, stream);
}

CIM_API int cim_mask_overlap_algo(const uint32_t *packed, int n_img, int n, int64_t words, int32_t *inter,
                                  int32_t *area, void *iou_f16, void *asy_f16, void *workspace, size_t ws_bytes,
                                  int algo, cim_stream_t stream) {
    return cim_mask_overlap_ex(packed, n_img, n, words, 0, inter, area, iou_f16, asy_f16, workspace, ws_bytes, algo,
                               stream);
}

CIM_API int cim_mask_overlap_ex(const uint32_t *packed, int n_img, int n, int64_t words, int kb_per_row,
                                int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16, void *workspace,
                                size_t ws_bytes, int algo, cim_stream_t stream) {
    return cim_mask_overlap_meta(packed, nullptr, n_img, n, words, kb_per_row, inter, area, iou_f16, asy_f16, workspace,
                                 ws_bytes, algo, stream);
}

CIM_API int cim_mask_overlap_meta(const uint32_t *packed, const void *meta, int n_img, int n, int64_t words,
                                  int kb_per_row, int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16,
                                  void *workspace, size_t ws_bytes, int algo, cim_stream_t stream) {
    if (algo != CIM_OVERLAP_AUTO && algo != CIM_OVERLAP_POPC && algo != CIM_OVERLAP_TENSOR) return CIM_ERR_ARG;
    if (!packed || !iou_f16 || !asy_f16 || n_img < 0 || n < 0 || words <= 0 || kb_per_row < 0) return CIM_ERR_ARG;
    if (words * 32 >= (1LL << 24)) return CIM_ERR_SHAPE;      // counts must stay exact in fp32
    if (n_img == 0 || n == 0) return CIM_OK;
    if (n_img > 65535 || n > 16384) return CIM_ERR_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool tc_ok = cim_mask_overlap_tc_eligible(n, words) && cim_aligned(packed, 16);
    if (algo == CIM_OVERLAP_TENSOR && !tc_ok) return CIM_ERR_SHAPE;
    // the tensor path pays off once a 128 x 256 tile is reasonably full and K is long
    const bool use_tc = algo == CIM_OVERLAP_TENSOR || (algo == CIM_OVERLAP_AUTO && tc_ok && n >= 256 && words >= 128);
    const size_t need = use_tc ? cim_mask_overlap_workspace_bytes(n_img, n, words, inter != nullptr)
                               : (area ? 0 : 2 * up256(sizeof(int32_t) * (size_t)n_img * n) + 512);
    if (need && (!workspace || ws_bytes < need || !cim_aligned(workspace, 256))) return CIM_ERR_WORKSPACE;
    OverlapWs w = carve_overlap_ws(workspace, n_img, n, words, inter != nullptr);
    const long long n_masks = (long long)n_img * n;
    int rc;
    if (meta) {
        // areas, K-block occupancy bitmaps and sort keys were produced with the masks (cim_mask_meta): no pass over
        // the packed masks here.  (meta must come from the same packed / words / kb_per_row; tensor-path layout.)
        if (!cim_aligned(meta, 256) || (words & 3)) return CIM_ERR_ALIGN;
        const MaskMeta mm = carve_meta(const_cast<void *>(meta), n_img, n, words);
        if (area) cudaMemcpyAsync(area, mm.area, sizeof(int32_t) * (size_t)n_masks, cudaMemcpyDeviceToDevice, st);
        area = mm.area;
        w.kinfo = mm.kinfo;
        w.kbmap = mm.kbmap;
    } else {
        if (!area) area = w.area;
        mask_area_kernel<<<(unsigned)((n_masks + 7) / 8), 256, 0, st>>>(packed, area, use_tc ? w.kbmap : nullptr,
                                                                        use_tc ? w.kinfo : nullptr, n_masks, words, w.bw,
                                                                        kb_per_row);
        if ((rc = cim_launch_status())) return rc;
    }
    __half *iou = reinterpret_cast<__half *>(iou_f16), *asy = reinterpret_cast<__half *>(asy_f16);
    if (use_tc) {
        int npad = 1;
        while (npad < n) npad <<= 1;
        const int nrb = (n + 127) / 128, ncb = (n + 255) / 256;
        int per_img = 0;
        for (int i = 0; i < nrb; ++i) per_img += ncb - (i >> 1);
        int tpad = 1;
        while (tpad < per_img) tpad <<= 1;
        // longest tiles first: ranked per image inside the sort kernel, the images' rankings interleaved
        const bool ordered = n_img < 32768 && nrb < 256 && ncb < 256 && (size_t)tpad * 8 <= 48 * 1024;
        const size_t smem_sort = (size_t)npad * 8;
        cudaFuncSetAttribute(mask_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sort);
        mask_sort_kernel<<<n_img, 1024, smem_sort, st>>>(w.kinfo, n, npad, kb_per_row, (int)((words + 3) / 4), w.perm,
                                                         w.inv);
        mask_union_kernel<<<dim3((unsigned)(nrb + ncb), (unsigned)n_img), 128, 0, st>>>(w.kbmap, w.perm, n, w.bw,
                                                                                        w.umap_a, w.umap_b, nrb, ncb);
        if (ordered)
            mask_rank_kernel<<<n_img, 256, (size_t)tpad * 8, st>>>(w.umap_a, w.umap_b, w.bw, nrb, ncb, per_img, tpad,
                                                                    w.tile_order);
        if ((rc = cim_launch_status())) return rc;
        cudaMemsetAsync(w.visited, 0, 8, st);
        const int32_t *order = ordered ? w.tile_order : nullptr;
        // the tensor kernel works in sorted index space and writes sorted-order maps
        rc = cim_mask_overlap_tc_launch(packed, area, w.perm, w.umap_a, w.umap_b, w.bw, w.visited, order, n_img, n,
                                        words, w.tmp_inter, w.tmp_iou, w.tmp_asy, st);
        if (rc) return rc;
        dim3 g((unsigned)n, (unsigned)n_img);
        if ((size_t)n * 4 > 48 * 1024)
            cudaFuncSetAttribute(mask_unpermute2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, n * 4);
        mask_unpermute2_kernel<<<g, 256, (size_t)n * 4, st>>>(w.tmp_iou, w.tmp_asy, w.inv, iou, asy, n);
        if (inter) {
            cudaFuncSetAttribute(mask_unpermute_kernel<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, n * 4);
            mask_unpermute_kernel<int32_t><<<g, 256, (size_t)n * 4, st>>>(w.tmp_inter, w.inv, inter, n);
        }
        return cim_launch_status();
    }
    const int nt = (n + TS - 1) / TS;
    dim3 grid((unsigned)(nt * (nt + 1) / 2), (unsigned)n_img);
    mask_overlap_popc_kernel<<<grid, 256, 0, st>>>(packed, area, n, words, inter, iou, asy);
    return cim_launch_status();
}
