// box_nms.cu -- test-time post-processing of the CIM heads on the GPU (SURVEY.md 8f-3).
//
//  cim_test_scores : lib/core/test.py:130-133 + lib/modeling/model_builder.py:60-68 -- the refinement heads'
//                    (cls * iou)[:, 1:] averaged over the K heads: out[r][c] = mean_k cls_k[r][c+1] * iou_k[r][c+1]
//                    (summed in head order then divided by K, as `scores += ...; scores /= K` does).
//  cim_box_nms     : the per-class loop of lib/utils/mask_eval_utils.py:57-79 (and box_results_with_nms_and_limit):
//                    candidates = scores[:, c] > score_thresh, greedy NMS of lib/utils/cython_nms.pyx:37-87:
//                    areas (x2-x1+1)(y2-y1+1), boxes visited by descending score, a later box is suppressed when
//                    inter / (area_i + area_j - inter) >= nms_thresh, all in float32.  One CTA per class:
//                    bitonic sort of the candidates in shared memory, then rounds over a compacted list of the
//                    candidates that are still alive (64-box chunk -> hit matrix -> kept members -> applied to
//                    the later live candidates -> compaction).
//                    Equal scores are visited by descending proposal index (what a stable ascending argsort,
//                    reversed, yields; numpy's default argsort leaves the order of ties unspecified).
//  cim_test_scores_tta : one pass of the TEST.BBOX_AUG score mean (core/test.py:149-226, SCORE_HEUR 'AVG':
//                    np.mean over the passes' test scores), accumulated in place pass by pass.
//  cim_box_detections : DETECTIONS_PER_IM limit over all classes of an image (mask_eval_utils.py:80-93) and the
//                    per-class detection lists (:96-110) compacted on the device, for a batch of images.
#include "common.cuh"

namespace {

// Pass t of T of a test-time-augmentation mean (T = 1: the plain head mean): s = the head mean of this pass,
// acc = s (t = 0) or fl(acc + s), and on the last pass of T > 1 acc = fl(acc / T) -- np.mean over the stacked
// passes, which sums float32 slices in pass order and divides once.
__global__ void cim_test_scores_kernel(const float *__restrict__ scores, float *__restrict__ acc, long long M, int C1,
                                       int K, int t, int T) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int C = C1 - 1;
    if (idx >= M * C) return;
    const long long r = idx / C;
    const int c = (int)(idx - r * C) + 1;
    float s = 0.f;
    for (int k = 0; k < K; ++k) {
        const float cls = scores[((size_t)(2 + k) * M + r) * C1 + c];
        const float iou = scores[((size_t)(2 + K + k) * M + r) * C1 + c];
        s = __fadd_rn(s, __fmul_rn(cls, iou));
    }
    s = __fdiv_rn(s, (float)K);
    if (t > 0) s = __fadd_rn(acc[idx], s);
    if (T > 1 && t == T - 1) s = __fdiv_rn(s, (float)T);
    acc[idx] = s;
}

constexpr int NMS_THREADS = 1024;
constexpr int CHUNK = 64;

// total order on floats as unsigned keys (larger float -> larger key) and back
__device__ __forceinline__ uint32_t score_key(float s) {
    const uint32_t b = __float_as_uint(s);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_score(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// float32 arithmetic of cython_nms.pyx:76-84, no contraction
__device__ __forceinline__ float box_area(float4 b) {
    return __fmul_rn(__fadd_rn(__fsub_rn(b.z, b.x), 1.f), __fadd_rn(__fsub_rn(b.w, b.y), 1.f));
}
__device__ __forceinline__ bool nms_hit(float4 a, float aarea, float4 b, float barea, float thr) {
    const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y), xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    const float w = fmaxf(0.f, __fadd_rn(__fsub_rn(xx2, xx1), 1.f)), h = fmaxf(0.f, __fadd_rn(__fsub_rn(yy2, yy1), 1.f));
    const float inter = __fmul_rn(w, h);
    const float uni = __fsub_rn(__fadd_rn(aarea, barea), inter);
    // fl(inter / uni) >= thr decided without the division when inter is not within 2^-20 (relative) of thr * uni:
    // the rounding errors of the product and of the quotient are < 2^-22, so both shortcuts agree with the division
    if (thr > 0.f && uni > 1e-30f && uni < 3.0e38f) {
        const float t = thr * uni;
        if (inter > t * 1.00000095367431640625f) return true;
        if (inter < t * 0.99999904632568359375f) return false;
    }
    return __fdiv_rn(inter, uni) >= thr;
}

// One CTA per (class, image).  After the sort the kernel works on a LIVE list (positions in score order of the
// candidates no kept box has suppressed yet) and proceeds in rounds:
//   A  the first <= 64 live candidates form the chunk; all threads fill its 64 x 64 hit matrix (row i = the later
//      chunk members box i would suppress), one 64-bit word per row
//   B  one thread walks the rows in score order: a member still alive is KEPT and clears the members it hits
//   C  every later live candidate is tested against the kept members only, and the live list is compacted (order
//      preserved by a block-wide scan) for the next round
// A chunk member is alive w.r.t. all earlier kept boxes by construction, so it is either kept or suppressed by a
// kept member of its own chunk: the number of rounds is ~ (kept + suppressed-inside-chunks) / 64 instead of m / 64,
// and the tests are those of the sequential algorithm (box i of cython_nms.pyx:60-87 only meets boxes that are
// still alive) plus the <= 2016 pairs of each chunk.  Round 2's first kernel walked all m / 64 chunks and scanned
// 64 (mostly dead) members per later box: 2.1 ms for 640 lists of 4000 candidates; this one: see DESIGN 4.10.
__global__ void __launch_bounds__(NMS_THREADS)
cim_box_nms_kernel(const float *__restrict__ boxes, const float *__restrict__ scores, int n, int ncls, int score_stride,
                   float score_thresh, float nms_thresh, int npad, uint8_t *__restrict__ keep) {
    extern __shared__ unsigned char smem_raw[];
    unsigned long long *key = reinterpret_cast<unsigned long long *>(smem_raw);      // [npad] (score bits, index)
    float4 *box = reinterpret_cast<float4 *>(key + npad);                            // [npad] sorted order
    uint16_t *live0 = reinterpret_cast<uint16_t *>(box + npad);                      // [npad] live list, ping
    uint16_t *live1 = live0 + npad;                                                  // [npad] pong
    __shared__ unsigned long long s_row[CHUNK];
    __shared__ unsigned long long s_kept;
    __shared__ int s_count, s_wtot[NMS_THREADS / 32];
    const int c = blockIdx.x, tid = threadIdx.x;
    // blockIdx.y = image of a batch: boxes [n_img][n][4], scores [n_img][n][score_stride], keep [n_img][ncls][n]
    boxes += (size_t)blockIdx.y * n * 4;
    scores += (size_t)blockIdx.y * n * score_stride;
    uint8_t *kout = keep + ((size_t)blockIdx.y * ncls + c) * n;

    // candidates: score > thresh (mask_eval_utils.py:64).  Key = (orderable score bits << 32) | index, sorted
    // descending; non-candidates get key 0 and sink to the end.
    int local = 0;
    for (int i = tid; i < npad; i += NMS_THREADS) {
        unsigned long long k = 0ull;
        if (i < n) {
            const float s = scores[(size_t)i * score_stride + c];
            if (s > score_thresh) {
                k = ((unsigned long long)score_key(s) << 32) | (uint32_t)(i + 1);    // + 1: 0 is "none"
                ++local;
            }
            kout[i] = 0;
        }
        key[i] = k;
    }
    if (tid == 0) s_count = 0;
    __syncthreads();
    if (local) atomicAdd(&s_count, local);
    // bitonic sort, descending; thread t owns compare-exchange t of the npad / 2 of a pass (i = t with a zero bit
    // inserted at bit log2(j), partner i | j), so every thread of a pass does useful work
    for (int k = 2; k <= npad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
            for (int t = tid; t < (npad >> 1); t += NMS_THREADS) {
                const int lo = t & (j - 1), i = ((t - lo) << 1) | lo, p = i | j;
                const unsigned long long a = key[i], b = key[p];
                const bool desc = (i & k) == 0;
                if (desc ? (a < b) : (a > b)) { key[i] = b; key[p] = a; }
            }
        }
    __syncthreads();
    int m = s_count;                                       // live candidates of the current round
    for (int i = tid; i < m; i += NMS_THREADS) {
        const int src = (int)(uint32_t)(key[i] & 0xFFFFFFFFull) - 1;
        box[i] = *reinterpret_cast<const float4 *>(boxes + (size_t)src * 4);
        live0[i] = (uint16_t)i;
    }
    const int lane = tid & 31, warp = tid >> 5;
    uint16_t *cur = live0, *nxt = live1;
    while (m > 0) {
        if (tid < CHUNK) s_row[tid] = 0ull;
        __syncthreads();                                   // live list / boxes of this round, s_row zeroed
        const int nc = min(m, CHUNK);
        // A: hit matrix of the chunk, 16 threads per row, 4 columns each
        {
            const int i = tid >> 4, j0 = (tid & 15) * 4;
            if (i < nc && j0 + 3 > i) {
                const float4 bi = box[cur[i]];
                const float ai = box_area(bi);
                unsigned long long bits = 0ull;
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    const int j = j0 + d;
                    if (j > i && j < nc) {
                        const float4 bj = box[cur[j]];
                        if (nms_hit(bi, ai, bj, box_area(bj), nms_thresh)) bits |= 1ull << j;
                    }
                }
                if (bits) atomicOr(&s_row[i], bits);
            }
        }
        __syncthreads();
        // B: sequential resolution in score order
        if (tid == 0) {
            unsigned long long alive = nc == 64 ? ~0ull : ((1ull << nc) - 1ull), kept = 0ull;
            while (alive) {
                const int i = __ffsll((long long)alive) - 1;
                kept |= 1ull << i;
                alive &= ~(s_row[i] | (1ull << i));
            }
            s_kept = kept;
        }
        __syncthreads();
        const unsigned long long kept = s_kept;
        if (tid < nc && ((kept >> tid) & 1ull)) kout[(int)(uint32_t)(key[cur[tid]] & 0xFFFFFFFFull) - 1] = 1;
        // C: later live candidates against the kept members; thread t owns a contiguous run so that one scan of the
        // per-thread counts keeps the score order
        const int rest = m - nc;
        const int per = (rest + NMS_THREADS - 1) / NMS_THREADS;             // <= npad / 1024
        const int b0 = nc + tid * per, b1 = min(b0 + per, m);
        uint32_t alive_bits = 0;
        int cnt = 0;
        for (int j = b0; j < b1; ++j) {
            const float4 bj = box[cur[j]];
            const float aj = box_area(bj);
            bool dead = false;
            unsigned long long km = kept;
            while (km && !dead) {
                const int i = __ffsll((long long)km) - 1;
                km &= km - 1ull;
                const float4 bi = box[cur[i]];
                dead = nms_hit(bi, box_area(bi), bj, aj, nms_thresh);
            }
            if (!dead) { alive_bits |= 1u << (j - b0); ++cnt; }
        }
        int incl = cnt;                                    // inclusive scan over the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_wtot[warp] = incl;
        __syncthreads();
        int wsum = s_wtot[lane];                           // every warp scans the 32 warp totals
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, wsum, d);
            if (lane >= d) wsum += v;
        }
        const int total = __shfl_sync(0xffffffffu, wsum, 31);
        int pos = incl - cnt + (warp ? __shfl_sync(0xffffffffu, wsum, (warp + 31) & 31) : 0);
        for (int j = b0; j < b1; ++j)
            if ((alive_bits >> (j - b0)) & 1u) nxt[pos++] = cur[j];
        m = total;
        uint16_t *t = cur; cur = nxt; nxt = t;
        // the __syncthreads at the top of the next round orders these writes (and the reads of s_wtot / s_kept)
        // before their next use
    }
}

// ---- detection limit + compaction (mask_eval_utils.py:80-110), one CTA per image
// The image's keep mask [C][n] is read as one flat byte range (position p = c * n + i, so ascending p is the
// reference's order: class, then proposal index) in 16-byte units: unit 0 = the bytes before the first 16-byte
// boundary, units 1 .. nv = aligned uint4 loads, unit nv + 1 = the tail.  Every pass re-reads the mask (L2-resident
// right after the NMS); nothing is staged, so the worst case -- all C * n candidates kept -- needs no other path.
constexpr int DET_THREADS = 1024;
constexpr int DET_UNITS = 4;                              // consecutive units per thread and tile: loads in flight

struct MaskUnits {
    const uint8_t *p;
    int L, head, nv;
    __device__ MaskUnits(const uint8_t *p_, int L_) : p(p_), L(L_) {
        head = min(L, (int)((16u - (unsigned)((uintptr_t)p & 15u)) & 15u));
        nv = (L - head) >> 4;
    }
    __device__ int count() const { return nv + 2; }
    __device__ int start(int u) const { return u == 0 ? 0 : head + 16 * (u - 1); }
    __device__ bool vector(int u) const { return u >= 1 && u <= nv; }
    __device__ int len(int u) const { return u == 0 ? head : vector(u) ? 16 : u == nv + 1 ? L - start(u) : 0; }
    // bit j = byte j of the unit is non-zero
    __device__ unsigned kept(int u) const {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (vector(u)) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p + start(u)));
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        } else {
            const int s = start(u), l = len(u);
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (j < l) w[j >> 2] |= (uint32_t)p[s + j] << (8 * (j & 3));
        }
        unsigned m = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) m |= ((w[j >> 2] >> (8 * (j & 3))) & 0xffu) ? (1u << j) : 0u;
        return m;
    }
};

// exclusive scan of v over the 1024 threads; every thread must call it
__device__ __forceinline__ int block_exclusive_scan(int v, int *s_wtot, int &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += x;
    }
    if (lane == 31) s_wtot[warp] = incl;
    __syncthreads();
    int w = s_wtot[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += x;
    }
    total = __shfl_sync(0xffffffffu, w, 31);
    const int before = __shfl_sync(0xffffffffu, w, (warp + 31) & 31);
    __syncthreads();                                       // s_wtot free for the next call
    return (warp ? before : 0) + incl - v;
}

// total = kept entries of the image.  With limit > 0 and total > limit, thresh = the limit-th largest kept score
// (with multiplicity), found by a radix select over score_key() in 8-bit digits: pass 1 counts and histograms the
// top digit, each later pass histograms the next digit of the entries that match the digits chosen so far.
// Survivors: kept and score >= thresh as a float32 comparison (so -0 and +0 tie as in numpy).  The compaction pass
// scans the survivor counts of each tile block-wide, which keeps ascending position order; entries of rank < cap
// are written, count gets the full number.
__global__ void __launch_bounds__(DET_THREADS)
cim_box_detections_kernel(const float *__restrict__ boxes, const float *__restrict__ scores,
                          const uint8_t *__restrict__ keep, int n, int ncls, int score_stride, int limit, int cap,
                          uint8_t *__restrict__ keep_out, int *__restrict__ count, int *__restrict__ det_cls,
                          int *__restrict__ det_idx, float *__restrict__ det_score, float *__restrict__ det_box) {
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_sel[2];                          // chosen key prefix, rank still to find inside it
    __shared__ int s_wtot[32];
    __shared__ int s_total;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int L = ncls * n;
    const MaskUnits mu(keep + (size_t)b * L, L);
    scores += (size_t)b * n * score_stride;
    boxes += (size_t)b * n * 4;
    const int units = mu.count(), step = DET_THREADS * DET_UNITS;
    auto score_at = [&](int pos) {
        const int c = pos / n, i = pos - c * n;
        return scores[(size_t)i * score_stride + c];
    };
    // one pass over the kept entries; shift >= 0: histogram of digit `shift` of the entries whose digits above it
    // equal prefix's.  Returns this thread's number of kept entries.
    auto hist_pass = [&](int shift, uint32_t prefix) {
        int local = 0;
        for (int u0 = tid * DET_UNITS; u0 < units; u0 += step) {
            unsigned m[DET_UNITS];
#pragma unroll
            for (int q = 0; q < DET_UNITS; ++q) m[q] = mu.kept(u0 + q);
#pragma unroll
            for (int q = 0; q < DET_UNITS; ++q) {
                local += __popc(m[q]);
                if (shift < 0) continue;
                const int s0 = mu.start(u0 + q);
                for (unsigned r = m[q]; r; r &= r - 1u) {
                    const uint32_t k = score_key(score_at(s0 + __ffs(r) - 1));
                    if (shift == 24 || (k >> (shift + 8)) == (prefix >> (shift + 8)))
                        atomicAdd(&s_hist[(k >> shift) & 255u], 1u);
                }
            }
        }
        return local;
    };

    if (tid < 256) s_hist[tid] = 0u;
    if (tid == 0) s_total = 0;
    __syncthreads();
    const int local = hist_pass(limit > 0 ? 24 : -1, 0u);
    if (local) atomicAdd(&s_total, local);
    __syncthreads();
    const bool limited = limit > 0 && s_total > limit;
    float thresh = 0.f;
    if (limited) {
        uint32_t prefix = 0u;
        unsigned need = (unsigned)limit;
        for (int shift = 24;; shift -= 8) {
            if (tid < 32) {                                // highest digit d with #(digit >= d) >= need
                unsigned sum = 0u;
#pragma unroll
                for (int e = 0; e < 8; ++e) sum += s_hist[255 - 8 * lane - e];
                unsigned incl = sum;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const unsigned x = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += x;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, incl >= need);
                if (lane == __ffs(hit) - 1) {
                    unsigned above = incl - sum;
                    for (int e = 0; e < 8; ++e) {
                        const int d = 255 - 8 * lane - e;
                        const unsigned h = s_hist[d];
                        if (above + h >= need) {
                            s_sel[0] = prefix | ((uint32_t)d << shift);
                            s_sel[1] = need - above;
                            break;
                        }
                        above += h;
                    }
                }
            }
            __syncthreads();
            prefix = s_sel[0];
            need = s_sel[1];
            if (shift == 0) break;
            if (tid < 256) s_hist[tid] = 0u;
            __syncthreads();
            hist_pass(shift - 8, prefix);
            __syncthreads();
        }
        thresh = key_score(prefix);
    }

    uint8_t *ko = keep_out ? keep_out + (size_t)b * L : nullptr;
    const bool ko_vec = ko && (((uintptr_t)ko ^ (uintptr_t)mu.p) & 15u) == 0;     // same alignment as the input
    int base = 0;
    for (int t0 = 0; t0 < units; t0 += step) {
        const int u0 = t0 + tid * DET_UNITS;
        unsigned m[DET_UNITS];
#pragma unroll
        for (int q = 0; q < DET_UNITS; ++q) m[q] = mu.kept(u0 + q);
        int cnt = 0;
#pragma unroll
        for (int q = 0; q < DET_UNITS; ++q) {
            const int u = u0 + q, s0 = mu.start(u);
            if (limited)
                for (unsigned r = m[q]; r; r &= r - 1u) {
                    const int j = __ffs(r) - 1;
                    if (!(score_at(s0 + j) >= thresh)) m[q] &= ~(1u << j);
                }
            cnt += __popc(m[q]);
            if (ko && u < units) {
                if (ko_vec && mu.vector(u)) {
                    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                    for (int j = 0; j < 16; ++j) w[j >> 2] |= ((m[q] >> j) & 1u) << (8 * (j & 3));
                    *reinterpret_cast<uint4 *>(ko + s0) = make_uint4(w[0], w[1], w[2], w[3]);
                } else {
                    const int l = mu.len(u);
                    for (int j = 0; j < l; ++j) ko[s0 + j] = (uint8_t)((m[q] >> j) & 1u);
                }
            }
        }
        int tile_total;
        int rank = base + block_exclusive_scan(cnt, s_wtot, tile_total);
#pragma unroll
        for (int q = 0; q < DET_UNITS; ++q) {
            const int s0 = mu.start(u0 + q);
            for (unsigned r = m[q]; r && rank < cap; r &= r - 1u, ++rank) {
                const int pos = s0 + __ffs(r) - 1, c = pos / n, i = pos - c * n;
                const size_t o = (size_t)b * cap + rank;
                det_cls[o] = c;
                det_idx[o] = i;
                det_score[o] = scores[(size_t)i * score_stride + c];
                if (det_box)
#pragma unroll
                    for (int e = 0; e < 4; ++e) det_box[o * 4 + e] = boxes[(size_t)i * 4 + e];
            }
        }
        base += tile_total;
    }
    if (tid == 0) count[b] = base;
}

inline int next_pow2(int v) {
    int p = 64;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace

CIM_API int cim_test_scores_tta(const float *scores, float *acc, int64_t M, int C1, int K, int t, int T,
                                cim_stream_t stream) {
    if (!scores || !acc) return CIM_ERR_ARG;
    if (M < 0 || C1 < 2 || K < 1 || K > 8 || T < 1 || t < 0 || t >= T) return CIM_ERR_ARG;
    if (M == 0) return CIM_OK;
    const long long n = M * (C1 - 1);
    cim_test_scores_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scores, acc, M, C1, K, t, T);
    return cim_launch_status();
}

CIM_API int cim_test_scores(const float *scores, float *out, int64_t M, int C1, int K, cim_stream_t stream) {
    return cim_test_scores_tta(scores, out, M, C1, K, 0, 1, stream);
}

CIM_API int cim_box_detections(const float *boxes, const float *scores, const uint8_t *keep, int n_img, int n,
                               int n_classes, int score_stride, int detections_per_im, int cap, uint8_t *keep_out,
                               int32_t *count, int32_t *det_cls, int32_t *det_idx, float *det_score, float *det_box,
                               cim_stream_t stream) {
    if (!boxes || !scores || !keep || !count) return CIM_ERR_ARG;
    if (cap > 0 && (!det_cls || !det_idx || !det_score)) return CIM_ERR_ARG;
    if (n_img < 0 || n < 0 || n_classes < 0 || score_stride < n_classes || cap < 0) return CIM_ERR_ARG;
    if (n_img == 0) return CIM_OK;
    if (n > 8192 || n_classes > 65535 || n_img > 65535) return CIM_ERR_SHAPE;
    cim_box_detections_kernel<<<(unsigned)n_img, DET_THREADS, 0, (cudaStream_t)stream>>>(
        boxes, scores, keep, n, n_classes, score_stride, detections_per_im, cap, keep_out, count, det_cls, det_idx,
        det_score, det_box);
    return cim_launch_status();
}

CIM_API int cim_box_nms(const float *boxes, const float *scores, int n, int n_classes, int score_stride,
                        float score_thresh, float nms_thresh, uint8_t *keep, cim_stream_t stream) {
    return cim_box_nms_batched(boxes, scores, 1, n, n_classes, score_stride, score_thresh, nms_thresh, keep, stream);
}

CIM_API int cim_box_nms_batched(const float *boxes, const float *scores, int n_img, int n, int n_classes,
                                int score_stride, float score_thresh, float nms_thresh, uint8_t *keep,
                                cim_stream_t stream) {
    if (!boxes || !scores || !keep) return CIM_ERR_ARG;
    if (n_img < 0 || n < 0 || n_classes < 0 || score_stride < n_classes) return CIM_ERR_ARG;
    if (n_img == 0 || n == 0 || n_classes == 0) return CIM_OK;
    if (n > 8192 || n_classes > 65535 || n_img > 65535) return CIM_ERR_SHAPE;
    if (!cim_aligned(boxes, 16)) return CIM_ERR_ALIGN;
    const int npad = next_pow2(n);
    const size_t smem = (size_t)npad * (8 + 16 + 2 + 2);
    if ((int)smem > cim_max_smem_optin()) return CIM_ERR_SHAPE;
    cudaFuncSetAttribute(cim_box_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cim_box_nms_kernel<<<dim3((unsigned)n_classes, (unsigned)n_img), NMS_THREADS, smem, (cudaStream_t)stream>>>(
        boxes, scores, n, n_classes, score_stride, score_thresh, nms_thresh, npad, keep);
    return cim_launch_status();
}
