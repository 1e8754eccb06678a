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
//
//  cim_mask_unpack_rle_kernel : the way back, COCO compressed RLE strings (rleFrString + rleDecode) -> tiled bit masks
//                 and their metadata, as the sparse update of mask_patch.cuh.  One CTA per row.  The string is parsed
//                 256 characters at a time: a ballot over the continuation bit finds where counts end, a block scan
//                 numbers them, and the count's value is read from its first (at most 7) characters -- only the low
//                 32 bits of rleFrString's long survive its (uint) cast.  The delta coding (x += cnts[m-2], m > 2) is
//                 two interleaved prefix sums (even and odd counts), a third scan gives the run boundaries; the last
//                 count index, the two chain sums and the running position are carried across chunks.  The ones-runs
//                 are painted as column intervals into a column-major bitmap of a band of rows in shared memory (32
//                 rows per word), 32 x 32 blocks are transposed back with ballots into 8 x 16 patches, and the union
//                 of the old and the new rectangle is written.  An image too large for one band re-walks the string
//                 per band.  A malformed string gives an empty row and is counted.
#include "common.cuh"
#include "mask_patch.cuh"

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

// ------------------------------------------------------------------------------- RLE strings -> tiled bit masks
constexpr int RU_THREADS = 256;
constexpr int RU_WARPS = RU_THREADS / 32;
// 4 CTAs per SM: 64 registers (no spills) and 32 KB of band bitmap + the K-block bitmap + 3.6 KB static each

__global__ void __launch_bounds__(RU_THREADS, 4)
cim_mask_unpack_rle_kernel(const uint8_t *__restrict__ chars, long long n_chars, const long long *__restrict__ off,
                           const int32_t *__restrict__ len, const int32_t *__restrict__ mask_hw,
                           uint32_t *__restrict__ packed, int4 *__restrict__ prev, int32_t *__restrict__ area,
                           uint32_t *__restrict__ kbmap, int4 *__restrict__ kinfo, int n, int H, int W,
                           long long words, int bw, int32_t *__restrict__ bad) {
    extern __shared__ uint32_t s_dyn[];
    uint32_t *const s_bmp = s_dyn;                       // [RLE_UNPACK_BITMAP_WORDS] word (rb, x) = rows 32 rb.. of x
    uint32_t *const s_kb = s_dyn + CIM_RLE_UNPACK_BITMAP_WORDS;     // [bw] the row's K-block bitmap
    __shared__ int s_wi[32];
    __shared__ unsigned s_wu[32];
    __shared__ long long s_wl[32];
    __shared__ int s_wlast[RU_WARPS];                   // last count-ending character of each warp of the chunk
    __shared__ int s_seg[RU_THREADS], s_ra[RU_THREADS], s_rb[RU_THREADS];   // column segments (inclusive scan), runs
    __shared__ int s_box[4];                            // xmin, xmax, ymin, ymax of the ones
    __shared__ int s_acc[5];                            // PatchMeta of the CTA
    const long long m = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = (int)(m / n);
    int h = H, w = W;
    if (mask_hw) {
        h = min(max(mask_hw[2 * b], 1), H);
        w = min(max(mask_hw[2 * b + 1], 1), W);
    }
    const long long hw = (long long)h * w;
    const long long o = off[m];
    const int L = len[m];
    bool row_bad = L < 0 || o < 0 || o > n_chars - L;
    const uint8_t *s = chars + (row_bad ? 0 : o);
    const int bpr = W >> 4, nby = H >> 3;
    const int bc = (w + 31) & ~31;                                   // bitmap columns
    const int nrb = min(CIM_RLE_UNPACK_BITMAP_WORDS / bc, (h + 31) >> 5);   // 32-row blocks per band
    const int BR = 32 * nrb;

    for (int i = tid; i < nrb * bc; i += RU_THREADS) s_bmp[i] = 0u;
    for (int i = tid; i < bw; i += RU_THREADS) s_kb[i] = 0u;
    if (tid == 0) {
        s_box[0] = INT_MAX; s_box[1] = -1; s_box[2] = INT_MAX; s_box[3] = -1;
        s_acc[0] = 0; s_acc[1] = INT_MAX; s_acc[2] = -1; s_acc[3] = INT_MAX; s_acc[4] = -1;
    }
    __syncthreads();

    int xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;
    // rleFrString + rleDecode over the whole string: paints the ones of rows [yb0, yb1) into s_bmp; with `first` also
    // validates and records the box.  Returns true (block-uniform) for a malformed string.
    auto walk = [&](int yb0, int yb1, bool first) {
        unsigned cE = 0u, cO = 0u;                      // sums of the even (m >= 2) / odd deltas before the chunk
        long long pos = 0, mbase = 0;                   // pixels / counts before the chunk
        int last_end = -1;                              // last count-ending character before the chunk
        for (int c0 = 0; c0 < L; c0 += RU_THREADS) {
            const int i = c0 + tid;
            const bool have = i < L;
            const int v = have ? (int)__ldg(s + i) - 48 : 0;
            bool my_bad = have && (v < 0 || v > 63);
            const bool cont = have && (v & 0x20);
            const bool end = have && !cont;
            if (i == L - 1 && cont) my_bad = true;      // the string stops inside a count
            const unsigned eb = __ballot_sync(0xffffffffu, end);
            if (lane == 0) s_wlast[warp] = eb ? c0 + 32 * warp + 31 - __clz(eb) : -1;
            int n_end;
            const int r0 = block_scan<int>(end ? 1 : 0, s_wi, &n_end);   // (its barriers publish s_wlast)
            unsigned x = 0u;
            if (end) {                                  // the count spans characters st .. i
                const unsigned below = eb & ((1u << lane) - 1u);
                int pe = last_end;
                if (below) {
                    pe = c0 + 32 * warp + 31 - __clz(below);
                } else {
                    for (int q = 0; q < warp; ++q) pe = max(pe, s_wlast[q]);
                }
                const int st = pe + 1, K = i - st + 1;
                for (int k = 0; k < min(K, 7); ++k) x |= (unsigned)((__ldg(s + st + k) - 48) & 0x1f) << (5 * k);
                if ((v & 0x10) && K <= 6) x |= 0xffffffffu << (5 * K);     // sign extension (mod 2^32)
            }
            const long long mi = mbase + r0;            // count index
            const unsigned ev = (end && mi >= 2 && !(mi & 1)) ? x : 0u, ov = (end && (mi & 1)) ? x : 0u;
            unsigned tE, tO;
            const unsigned E = cE + block_scan<unsigned>(ev, s_wu, &tE) + ev;
            const unsigned O = cO + block_scan<unsigned>(ov, s_wu, &tO) + ov;
            const unsigned cnt = mi == 0 ? x : ((mi & 1) ? O : E);
            long long tP;
            const long long c64 = end ? (long long)cnt : 0;
            const long long P = pos + block_scan<long long>(c64, s_wl, &tP) + c64;   // end of run mi
            if (end && (c64 > hw || P > hw)) my_bad = true;
            const bool run = end && (mi & 1) && cnt > 0u && c64 <= hw && P <= hw;
            const int ra = run ? (int)(P - c64) : 0, rb = run ? (int)P : 0;
            const int xa = run ? ra / h : 0, xb = run ? (rb - 1) / h : -1;
            if (first && run) {
                xmin = min(xmin, xa);
                xmax = max(xmax, xb);
                if (xa == xb) {
                    ymin = min(ymin, ra - xa * h);
                    ymax = max(ymax, rb - 1 - xb * h);
                } else {                                // a run across a column boundary covers rows 0 and h-1
                    ymin = 0;
                    ymax = h - 1;
                }
            }
            int n_seg;
            const int sg = block_scan<int>(xb - xa + 1, s_wi, &n_seg);
            s_seg[tid] = sg + xb - xa + 1;
            s_ra[tid] = ra;
            s_rb[tid] = rb;
            if (n_end) {                                // (s_wlast is rewritten only after the barrier below)
                int le = -1;
                for (int q = 0; q < RU_WARPS; ++q) le = max(le, s_wlast[q]);
                last_end = le;
            }
            __syncthreads();
            for (int j = tid; j < n_seg; j += RU_THREADS) {     // one column segment of one run per iteration
                int lo = 0, hi = RU_THREADS - 1;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (s_seg[mid] > j) hi = mid; else lo = mid + 1;
                }
                const int a = s_ra[lo], e = s_rb[lo], ca = a / h, ce = (e - 1) / h;
                const int xc = ce + 1 + j - s_seg[lo];
                const int y0 = max(xc == ca ? a - ca * h : 0, yb0), y1 = min(xc == ce ? e - 1 - ce * h : h - 1, yb1 - 1);
                for (int y = y0; y <= y1;) {
                    const int r = (y - yb0) >> 5, ye = min(y1, yb0 + 32 * r + 31);
                    const unsigned bits = (0xffffffffu >> (31 - ((ye - yb0) & 31))) & (0xffffffffu << ((y - yb0) & 31));
                    uint32_t *wp = s_bmp + r * bc + xc;
                    if (bits == 0xffffffffu) *wp = bits;        // no other run touches a word this one fills
                    else atomicOr(wp, bits);
                    y = ye + 1;
                }
            }
            if (__syncthreads_or(my_bad)) return true;
            cE += tE;
            cO += tO;
            pos += tP;
            mbase += n_end;
        }
        return pos != hw;
    };

    uint4 *row4 = reinterpret_cast<uint4 *>(packed + m * words);
    const int4 pv = prev[m];
    int4 nr = make_int4(0, 0, 0, 0);
    int ytop = 0, bx_lo = 0, bx_hi = 0, by_lo = 0, by_hi = 0;
    PatchMeta acc;
    for (int yb0 = 0;; yb0 += BR) {
        // band 0: the walk that validates and finds the box; later bands re-walk only where the new mask has rows
        if (yb0 == 0 ? !row_bad && L > 0 : nr.w > 0 && yb0 < nr.y + nr.w && yb0 + BR > nr.y) {
            const bool wb = walk(yb0, yb0 + BR, yb0 == 0);
            if (yb0 == 0) row_bad = wb;
        }
        if (yb0 == 0) {
            if (row_bad) {
                for (int i = tid; i < nrb * bc; i += RU_THREADS) s_bmp[i] = 0u;
            } else if (xmax >= 0) {
                atomicMin(&s_box[0], xmin);
                atomicMax(&s_box[1], xmax);
                atomicMin(&s_box[2], ymin);
                atomicMax(&s_box[3], ymax);
            }
            __syncthreads();
            if (s_box[1] >= 0 && !row_bad)
                nr = make_int4(s_box[0] >> 5, s_box[2], (s_box[1] >> 5) - (s_box[0] >> 5) + 1, s_box[3] - s_box[2] + 1);
            if (nr.z > 0 && nr.w > 0) ytop = nr.y + nr.w;
            if (pv.z > 0 && pv.w > 0) ytop = max(ytop, pv.y + pv.w);
            patch_union(nr, pv, bpr, nby, &bx_lo, &bx_hi, &by_lo, &by_hi);
        }
        // the union's patches in this band: 32 x 32 blocks of the bitmap (cleared as they are read) -> 8 patches each
        const int pl = max(by_lo, yb0 >> 3), ph = min(by_hi, (yb0 + BR) >> 3);
        if (bx_hi > bx_lo && ph > pl) {
            const int wx_lo = bx_lo >> 1, nwx = ((bx_hi + 1) >> 1) - wx_lo;
            const int rb_lo = (8 * pl - yb0) >> 5, nblk = nwx * (((8 * ph - 1 - yb0) >> 5) + 1 - rb_lo);
            for (int t = warp; t < nblk; t += RU_WARPS) {
                const int r = rb_lo + t / nwx, wx = wx_lo + t % nwx;
                const int col = 32 * wx + lane;
                uint32_t cw = 0u;
                if (col < bc) {
                    cw = s_bmp[r * bc + col];
                    s_bmp[r * bc + col] = 0u;
                }
                uint32_t rw = 0u;                       // row yb0 + 32 r + lane, columns 32 wx ..
                if (__ballot_sync(0xffffffffu, cw != 0u)) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const uint32_t bal = __ballot_sync(0xffffffffu, (cw >> c) & 1u);
                        if (lane == c) rw = bal;
                    }
                }
                const int pr = (lane >> 1) & 3, sh = 16 * (lane & 1);      // lanes 0..7: patch row pr, left / right
                uint32_t q[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) q[j] = (__shfl_sync(0xffffffffu, rw, 8 * pr + j) >> sh) & 0xffffu;
                const int by = (yb0 >> 3) + 4 * r + pr, bx = 2 * wx + (lane & 1);
                if (lane < 8 && by >= pl && by < ph && bx >= bx_lo && bx < bx_hi)
                    acc.store(row4, s_kb, by * bpr + bx, bx, by,
                              make_uint4(q[0] | (q[1] << 16), q[2] | (q[3] << 16), q[4] | (q[5] << 16), q[6] | (q[7] << 16)));
            }
        }
        __syncthreads();                                // the bitmap is clear again
        if (yb0 + BR >= ytop) break;
    }
    acc.warp_reduce();
    if (lane == 0 && acc.ahi >= 0) {
        atomicAdd(&s_acc[0], acc.s);
        atomicMin(&s_acc[1], acc.alo);
        atomicMax(&s_acc[2], acc.ahi);
        atomicMin(&s_acc[3], acc.blo);
        atomicMax(&s_acc[4], acc.bhi);
    }
    __syncthreads();
    for (int j = tid; j < bw; j += RU_THREADS) kbmap[m * bw + j] = s_kb[j];
    if (tid == 0) {
        PatchMeta tot;
        tot.s = s_acc[0]; tot.alo = s_acc[1]; tot.ahi = s_acc[2]; tot.blo = s_acc[3]; tot.bhi = s_acc[4];
        tot.write(area, kinfo, m);
        prev[m] = nr;
        if (row_bad && bad) atomicAdd(bad, 1);
    }
}

}  // namespace

// The launch behind cim_mask_unpack_rle_tiled_meta_sparse (mask_overlap.cu, which owns the metadata layout); the
// arguments are checked there.
int cim_mask_unpack_rle_launch(const uint8_t *chars, long long n_chars, const int64_t *off, const int32_t *len,
                               const int32_t *mask_hw, uint32_t *packed, int32_t *prev_rects, int32_t *area,
                               uint32_t *kbmap, int4 *kinfo, long long n_masks, int n, int H, int W, long long words,
                               int bw, int32_t *bad, cudaStream_t st) {
    if (bad) cudaMemsetAsync(bad, 0, sizeof(int32_t), st);
    if (n_masks > 0)
        cim_mask_unpack_rle_kernel<<<(unsigned)n_masks, RU_THREADS,
                                     ((size_t)CIM_RLE_UNPACK_BITMAP_WORDS + bw) * sizeof(uint32_t), st>>>(
            chars, n_chars, reinterpret_cast<const long long *>(off), len, mask_hw, packed,
            reinterpret_cast<int4 *>(prev_rects), area, kbmap, kinfo, n, H, W, words, bw, bad);
    return cim_launch_status();
}

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
