// mask_rle.cu -- selected proposal masks as COCO compressed RLE (pycocotools maskApi.c: rleEncode + rleToString,
// rleArea, rleToBbox), for the detections of cim_box_detections.
//
//  cim_mask_rle : one CTA per selected (image, slot).  The mask is walked in COCO's column-major order (pixel
//                 j = x*h + y over the image's native h x w) one 32-bit COLUMN WORD at a time (32 rows of one column,
//                 bit r = row 32*rb + r).  A warp builds the column words of a 32 x 32 block of the packed mask with
//                 32 __ballot_sync (a bit transpose of the row words), into a shared-memory run of consecutive column
//                 words (a "unit": whole columns, or a row range of one column when a column alone is too tall).
//                 Per chunk of 256 column words the transition words w ^ (w << 1 | carry) are ranked by a block scan
//                 of their popcounts; transition i ends count i, and its string needs count i and count i-2, i.e.
//                 transition positions i .. i-3, so the CTA keeps the last three positions across chunks and stores
//                 no counts.  The same template runs twice: a length pass (string length, area, box), a scan of
//                 the lengths over all slots (offsets, need[]), then an emit pass that writes the characters.
#include "common.cuh"

#include <limits.h>

namespace {

constexpr int RLE_THREADS = 256;
constexpr int RLE_WARPS = RLE_THREADS / 32;
constexpr int RLE_ELEMS = 4096;                       // column words staged per unit (16 KB)
constexpr int RLE_POS = 3 + 32 * RLE_THREADS;         // three carried positions + every transition of a chunk
constexpr size_t RLE_SMEM = (size_t)RLE_ELEMS * 4 + (size_t)RLE_POS * 4;
constexpr int SCAN_THREADS = 1024;

// Columns 32s .. 32s+31 of row y of the packed canvas as one word (bit c = column 32s + c).  Bits of columns >= W
// are whatever follows in memory; the caller never uses them.
__device__ __forceinline__ uint32_t row_word(const uint32_t *__restrict__ m, int64_t words, int W, int kbr, int y,
                                             int s) {
    if (kbr == 0) {                                    // flat: pixel p = y*W + x is bit p & 31 of word p >> 5
        const int64_t p = (int64_t)y * W + 32 * s;
        const int64_t q = p >> 5;
        const int sh = (int)(p & 31);
        uint32_t v = __ldg(m + q) >> sh;
        if (sh && q + 1 < words) v |= __ldg(m + q + 1) << (32 - sh);
        return v;
    }
    // tiled: q = ((y>>3)*kbr + (x>>4))*128 + (y&7)*16 + (x&15); both 16-pixel halves share q & 31
    const int64_t q0 = ((int64_t)(y >> 3) * kbr + 2 * s) * 128 + (y & 7) * 16;
    const int sh = (int)(q0 & 31);
    uint32_t v = (__ldg(m + (q0 >> 5)) >> sh) & 0xffffu;
    if (2 * s + 1 < kbr) v |= ((__ldg(m + ((q0 + 128) >> 5)) >> sh) & 0xffffu) << 16;
    return v;
}

// rleToString for one count: x = cnts[i] (- cnts[i-2] when i > 2), 5 bits per character, the last one sign-extends.
// Writes the characters to out when out != nullptr; returns their number (1 .. 7).
__device__ __forceinline__ int rle_chars(long long x, uint8_t *out) {
    int n = 0;
    bool more = true;
    while (more) {
        int c = (int)(x & 0x1f);
        x >>= 5;
        more = (c & 0x10) ? x != -1 : x != 0;
        if (more) c |= 0x20;
        if (out) out[n] = (uint8_t)(c + 48);
        ++n;
    }
    return n;
}

// Exclusive block scan of v; *total = the block's sum.  Every thread of the block calls it.
template <typename T>
__device__ __forceinline__ T block_scan(T v, T *s_w, T *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nw = blockDim.x >> 5;
    T inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) s_w[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        T t = lane < nw ? s_w[lane] : T(0);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const T o = __shfl_up_sync(0xffffffffu, t, d);
            if (lane >= d) t += o;
        }
        if (lane < nw) s_w[lane] = t;
    }
    __syncthreads();
    const T before = wid ? s_w[wid - 1] : T(0);
    *total = s_w[nw - 1];
    __syncthreads();
    return before + inc - v;
}

__device__ __forceinline__ bool rle_selected(const int32_t *sel_count, const int32_t *sel_idx, int cap, int R,
                                             int e, int *idx, bool *invalid) {
    const int b = e / cap, j = e - b * cap;
    const int n_sel = min(max(sel_count[b], 0), cap);
    *invalid = false;
    if (j >= n_sel) return false;
    *idx = sel_idx[e];
    *invalid = *idx < 0 || *idx >= R;
    return !*invalid;
}

template <bool EMIT>
__global__ void __launch_bounds__(RLE_THREADS)
cim_mask_rle_kernel(const uint32_t *__restrict__ packed, int R, int64_t words, int H, int W, int kbr,
                    const int32_t *__restrict__ mask_hw, const int32_t *__restrict__ sel_count,
                    const int32_t *__restrict__ sel_idx, int cap, uint8_t *__restrict__ chars, int64_t chars_cap,
                    const int64_t *__restrict__ off, int32_t *__restrict__ len, int32_t *__restrict__ area,
                    int32_t *__restrict__ bbox) {
    extern __shared__ uint32_t s_colw[];                       // [RLE_ELEMS] column words of the current unit
    int *const s_pos = (int *)(s_colw + RLE_ELEMS);            // [RLE_POS]: t_{i-3}, t_{i-2}, t_{i-1}, then the chunk's
    __shared__ int s_wi[32];
    __shared__ long long s_wl[32];
    __shared__ int s_red[5];                                   // area, xmin, xmax, ymin, ymax
    __shared__ uint32_t s_carry;                               // last pixel of the previous unit
    const int e = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = e / cap;
    int idx = 0;
    bool invalid;
    const bool ok = rle_selected(sel_count, sel_idx, cap, R, e, &idx, &invalid);
    if (!ok) {
        if (!EMIT && tid == 0) {
            len[e] = 0;
            if (area) area[e] = 0;
            if (bbox) reinterpret_cast<int4 *>(bbox)[e] = make_int4(0, 0, 0, 0);
        }
        return;
    }
    uint8_t *out = nullptr;
    if (EMIT) {
        const int64_t o = off[e];
        if (o + len[e] > chars_cap) return;                   // only whole strings below chars_cap are written
        out = chars + o;
    }
    int h = H, w = W;
    if (mask_hw) {
        h = min(max(mask_hw[2 * b], 1), H);
        w = min(max(mask_hw[2 * b + 1], 1), W);
    }
    const uint32_t *m = packed + ((int64_t)b * R + idx) * words;
    const int nb = (h + 31) >> 5;
    const uint32_t last_mask = (h & 31) ? (1u << (h & 31)) - 1u : 0xffffffffu;   // valid rows of block nb-1
    const int last_bit = (h - 1) & 31;
    // a unit is a run of consecutive column words: whole columns when a column has <= RLE_ELEMS words, else a row
    // range of one column
    const int cpu = nb <= RLE_ELEMS ? RLE_ELEMS / nb : 1;
    const int rpu = nb <= RLE_ELEMS ? nb : RLE_ELEMS;

    if (tid < 3) s_pos[tid] = 0;                               // t_{-1} = 0 (pixel 0 follows a virtual 0)
    if (tid == 0) s_carry = 0u;
    long long rank = 0, cbase = 0, len_acc = 0;                // transitions / characters before the chunk
    int my_area = 0, xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;

    for (int x0 = 0; x0 < w; x0 += cpu) {
        const int x1 = min(w, x0 + cpu);
        for (int rb0 = 0; rb0 < nb; rb0 += rpu) {
            const int rb1 = min(nb, rb0 + rpu), nrb = rb1 - rb0;
            const int n_el = (x1 - x0) * nrb;
            const int s_lo = x0 >> 5, ntiles = (((x1 - 1) >> 5) - s_lo + 1) * nrb;
            __syncthreads();                                   // the previous unit is done with s_colw
            for (int t = warp; t < ntiles; t += RLE_WARPS) {
                const int s = s_lo + t / nrb, rb = rb0 + t % nrb;
                const int y = rb * 32 + lane;
                const uint32_t rw = y < h ? row_word(m, words, W, kbr, y, s) : 0u;
                uint32_t mine = 0u;
                if (__ballot_sync(0xffffffffu, rw != 0u)) {     // (most blocks of a proposal mask are empty)
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const uint32_t bal = __ballot_sync(0xffffffffu, (rw >> c) & 1u);
                        if (lane == c) mine = bal;
                    }
                }
                const int x = 32 * s + lane;
                if (x >= x0 && x < x1) s_colw[(x - x0) * nrb + (rb - rb0)] = mine;
            }
            __syncthreads();
            for (int c0 = 0; c0 < n_el; c0 += RLE_THREADS) {
                const int el = c0 + tid;
                uint32_t tr = 0u;
                int x = 0, rb = 0;
                if (el < n_el) {
                    const int col = el / nrb;
                    rb = rb0 + (el - col * nrb);
                    x = x0 + col;
                    const uint32_t wv = s_colw[el];
                    uint32_t carry;
                    if (el == 0) {
                        carry = s_carry;
                    } else {
                        const int prb = rb > rb0 ? rb - 1 : rb1 - 1;
                        carry = (s_colw[el - 1] >> (prb == nb - 1 ? last_bit : 31)) & 1u;
                    }
                    tr = (wv ^ ((wv << 1) | carry)) & (rb == nb - 1 ? last_mask : 0xffffffffu);
                    if (!EMIT && wv) {
                        my_area += __popc(wv);
                        xmin = min(xmin, x);
                        xmax = max(xmax, x);
                        ymin = min(ymin, 32 * rb + __ffs(wv) - 1);
                        ymax = max(ymax, 32 * rb + 31 - __clz(wv));
                    }
                }
                if (!__syncthreads_or(tr != 0u)) continue;     // no transition in the chunk: nothing changes
                int n_tr;
                const int r0 = block_scan<int>(__popc(tr), s_wi, &n_tr);
                {
                    int q = 3 + r0;
                    const int pbase = x * h + 32 * rb;
                    for (uint32_t r = tr; r; r &= r - 1u) s_pos[q++] = pbase + __ffs(r) - 1;
                }
                __syncthreads();
                auto delta = [&](int q) {                       // cnts[i] - cnts[i-2] (i > 2) of transition i
                    const long long i = rank + (q - 3);
                    long long xv = (long long)s_pos[q] - s_pos[q - 1];
                    if (i > 2) xv -= (long long)s_pos[q - 2] - s_pos[q - 3];
                    return xv;
                };
                const int q1 = 3 + r0 + __popc(tr);
                long long my_len = 0;
                for (int q = 3 + r0; q < q1; ++q) my_len += rle_chars(delta(q), nullptr);
                if (EMIT) {
                    long long chunk_len;
                    long long at = cbase + block_scan<long long>(my_len, s_wl, &chunk_len);
                    for (int q = 3 + r0; q < q1; ++q) at += rle_chars(delta(q), out + at);
                    cbase += chunk_len;
                } else {
                    len_acc += my_len;                          // summed over the block once, at the end
                }
                __syncthreads();                                // every read of s_pos is done
                if (tid == 0) {                                 // keep the last three positions
                    const int a = s_pos[n_tr], bb = s_pos[n_tr + 1], c = s_pos[n_tr + 2];
                    s_pos[0] = a;
                    s_pos[1] = bb;
                    s_pos[2] = c;
                }
                rank += n_tr;
                __syncthreads();
            }
            if (tid == 0) s_carry = (s_colw[n_el - 1] >> (rb1 - 1 == nb - 1 ? last_bit : 31)) & 1u;
        }
    }
    __syncthreads();
    if (!EMIT) {
        block_scan<long long>(len_acc, s_wl, &cbase);
        if (tid == 0) {
            s_red[0] = 0;
            s_red[1] = INT_MAX;
            s_red[2] = -1;
            s_red[3] = INT_MAX;
            s_red[4] = -1;
        }
        __syncthreads();
        if (my_area) {
            atomicAdd(&s_red[0], my_area);
            atomicMin(&s_red[1], xmin);
            atomicMax(&s_red[2], xmax);
            atomicMin(&s_red[3], ymin);
            atomicMax(&s_red[4], ymax);
        }
        __syncthreads();
    }
    if (tid == 0) {                                             // the last count: from t_{K-1} to the end
        const long long i = rank;
        long long xv = (long long)h * w - s_pos[2];
        if (i > 2) xv -= (long long)s_pos[1] - s_pos[0];
        const int n = rle_chars(xv, EMIT ? out + cbase : nullptr);
        if (!EMIT) {
            len[e] = (int32_t)(cbase + n);
            if (area) area[e] = s_red[0];
            if (bbox) {
                const bool any = s_red[0] > 0;
                reinterpret_cast<int4 *>(bbox)[e] =
                    any ? make_int4(s_red[1], s_red[3], s_red[2] - s_red[1] + 1, s_red[4] - s_red[3] + 1)
                        : make_int4(0, 0, 0, 0);
            }
        }
    }
}

// off = exclusive scan of len over all slots; need[0] = total characters, need[1] = selected indices outside [0, R).
__global__ void __launch_bounds__(SCAN_THREADS)
cim_mask_rle_scan_kernel(const int32_t *__restrict__ sel_count, const int32_t *__restrict__ sel_idx, int n_img,
                         int cap, int R, const int32_t *__restrict__ len, int64_t *__restrict__ off,
                         int64_t *__restrict__ need) {
    __shared__ long long s_wl[32];
    const int total = n_img * cap;
    long long base = 0, bad = 0;
    for (int c0 = 0; c0 < total; c0 += SCAN_THREADS) {
        const int e = c0 + threadIdx.x;
        long long l = 0, inv = 0;
        if (e < total) {
            int idx;
            bool invalid;
            rle_selected(sel_count, sel_idx, cap, R, e, &idx, &invalid);
            l = len[e];
            inv = invalid;
        }
        long long sum, nbad;
        const long long ex = block_scan<long long>(l, s_wl, &sum);
        block_scan<long long>(inv, s_wl, &nbad);
        if (e < total) off[e] = base + ex;
        base += sum;
        bad += nbad;
    }
    if (threadIdx.x == 0) {
        need[0] = base;
        need[1] = bad;
    }
}

}  // namespace

CIM_API int cim_mask_rle(const uint32_t *packed, int n_img, int R, int64_t words, int H, int W, int kb_per_row,
                         const int32_t *mask_hw, const int32_t *sel_count, const int32_t *sel_idx, int cap,
                         uint8_t *chars, int64_t chars_cap, int64_t *off, int32_t *len, int32_t *area, int32_t *bbox,
                         int64_t *need, cim_stream_t stream) {
    if (n_img < 0 || R < 0 || cap < 0 || words < 0 || chars_cap < 0 || H < 1 || W < 1) return CIM_ERR_ARG;
    if (!packed || !sel_count || !sel_idx || !off || !len || !need || (chars_cap > 0 && !chars)) return CIM_ERR_ARG;
    if ((int64_t)H * W > INT_MAX || (int64_t)n_img * cap > INT_MAX || (int64_t)n_img * R > INT_MAX)
        return CIM_ERR_SHAPE;
    if (words < ((int64_t)H * W + 31) / 32) return CIM_ERR_SHAPE;
    if (kb_per_row != 0 && (kb_per_row < 0 || H % 8 || W % 16 || kb_per_row != W / 16)) return CIM_ERR_ARG;
    if (!cim_aligned(packed, 4) || !cim_aligned(sel_count, 4) || !cim_aligned(sel_idx, 4) || !cim_aligned(off, 8) ||
        !cim_aligned(len, 4) || !cim_aligned(need, 8) || (mask_hw && !cim_aligned(mask_hw, 4)) ||
        (area && !cim_aligned(area, 4)) || (bbox && !cim_aligned(bbox, 16)))
        return CIM_ERR_ALIGN;
    const int n = n_img * cap;
    if (n > 0) {
        cudaFuncSetAttribute(cim_mask_rle_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RLE_SMEM);
        cudaFuncSetAttribute(cim_mask_rle_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RLE_SMEM);
        cim_mask_rle_kernel<false><<<n, RLE_THREADS, RLE_SMEM, stream>>>(
            packed, R, words, H, W, kb_per_row, mask_hw, sel_count, sel_idx, cap, chars, chars_cap, off, len, area,
            bbox);
    }
    cim_mask_rle_scan_kernel<<<1, SCAN_THREADS, 0, stream>>>(sel_count, sel_idx, n_img, cap, R, len, off, need);
    if (n > 0 && chars_cap > 0)
        cim_mask_rle_kernel<true><<<n, RLE_THREADS, RLE_SMEM, stream>>>(
            packed, R, words, H, W, kb_per_row, mask_hw, sel_count, sel_idx, cap, chars, chars_cap, off, len, area,
            bbox);
    return cim_launch_status();
}
