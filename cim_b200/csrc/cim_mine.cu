// cim_mine.cu -- complete-instance mining, mask NMS and pseudo-label assignment for sm_100a.
//
// Replaces heads.CIM_layer of the reference (lib/modeling/heads.py:222-503): instance_nms
// (:237-258, a Python while/filter loop with one device sync per compared pair), CIM_label
// (:318-407), MIST_label (:260-316) and the assignment half of forward (:475-501), for all
// images of the batch and all refinement layers at once (the layers only depend on the scores,
// never on each other's pseudo labels: model_builder.py:170-187).
//
// Kernels (one launch each per step):
//   cim_seed_kernel     block = (class, layer, image), skipped when the image label is 0:
//                       bitonic sort of the class scores in smem (descending, ties -> lower index),
//                       top keep_count seeds, k x k suppression bitmask from iou_map, greedy scan
//                       by one warp -> kept seeds in score order.                (:354-380)
//   cim_contain_kernel  warp = one asy_map row, read once for everything: the big-proposal
//                       count (:338) and, for every (layer, class, kept seed), the containment
//                       test (:386-390); containers race with a 64-bit atomicMax on
//                       (det score, ~row) = argmax with lowest-index ties       (:393-394).
//   cim_merge_kernel    block = (layer, image): classes in ascending order, a proposal is taken
//                       by class c iff preds > current weight (:397-402); compaction in
//                       ascending proposal order (:405).
//   cim_assign_kernel   warp = one iou_map row: max over the kept pseudo GTs with torch.max
//                       semantics (first maximum, first NaN wins), labels / weights / fp16 IoU
//                       labels (:477-501; :493-498 is a swallowed exception in the reference and
//                       is deliberately not applied).
// Every comparison on a map value is made in fp16 against fp16(threshold).
//
// Ragged batches (cim_mine_ex / cim_assign_ex): image b owns rows [0, n_b) of its R rows.  Its seeds are sorted from
// rows < n_b only, its containment counts run over columns < n_b, and keep_count / big_thr are evaluated for n_b on
// the device by cim_image_constants(); rows >= n_b get asy_flag 0 and the ignore row of the assignment.
#include "common.cuh"

// heads.py:332 and :338 for an image of n proposals, in the reference's arithmetic: int(np.ceil(p_seed * n)) and
// np.float32(0.9 * n), a float64 product rounded once.  Shared by the kernels and cim_mine_image_constants().
__host__ __device__ inline void cim_image_constants(double p_seed, int n, int *keep_count, float *big_thr) {
#ifdef __CUDA_ARCH__
    *keep_count = (int)ceil(__dmul_rn(p_seed, (double)n));
    *big_thr = __double2float_rn(__dmul_rn(0.9, (double)n));
#else
    volatile double kp = p_seed * (double)n, bp = 0.9 * (double)n;      // volatile: no contraction, no x87 excess
    *keep_count = (int)ceil(kp);
    *big_thr = (float)bp;
#endif
}

namespace {

constexpr int MAX_LAYERS = 4;

struct LayerPtrs {
    const float *cls[MAX_LAYERS];
    const float *det[MAX_LAYERS];
};

struct MineWs {
    int *nkept;                    // [L*n_img*C]
    int *kept;                     // [L*n_img*C][kc]
    unsigned long long *best;      // [L*n_img*C][kc]
};

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// rows, seed count and big-proposal threshold of image img: n_props[img] clamped to [1, R] and the constants for it,
// or R and the host-evaluated p.keep_count / p.big_thr when n_props is NULL.  keep_count never exceeds p.keep_count,
// the capacity the workspace was sized for.
struct ImageRows {
    int n, keep_count;
    float big_thr;
};
__device__ __forceinline__ ImageRows image_rows(const cim_mine_params &p, const int32_t *n_props, double p_seed,
                                                int img) {
    ImageRows r{p.R, p.keep_count, p.big_thr};
    if (n_props) {
        r.n = min(max(n_props[img], 1), p.R);
        cim_image_constants(p_seed, r.n, &r.keep_count, &r.big_thr);
        r.keep_count = min(max(r.keep_count, 1), p.keep_count);
    }
    return r;
}

__host__ inline MineWs carve_ws(void *ws, const cim_mine_params &p) {
    const size_t slots = (size_t)p.n_layers * p.n_img * p.C;
    char *b = (char *)ws;
    MineWs w;
    w.best = (unsigned long long *)b;
    b += align_up(slots * p.keep_count * 8, 256);
    w.kept = (int *)b;
    b += align_up(slots * p.keep_count * 4, 256);
    w.nkept = (int *)b;
    return w;
}

// "a sorts before b": higher score first, equal scores by lower index
__device__ __forceinline__ bool before(float ka, int ia, float kb, int ib) {
    return ka > kb || (ka == kb && ia < ib);
}

// ------------------------------------------------------------------------------ seeds + NMS
__global__ void __launch_bounds__(512, 4)
cim_seed_kernel(LayerPtrs ptrs, const float *__restrict__ labels, const __half *__restrict__ iou_all,
                cim_mine_params p, int npad, MineWs ws, const int32_t *__restrict__ n_props, double p_seed) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int c = blockIdx.x, l = blockIdx.y, img = blockIdx.z;
    if (labels[(size_t)img * p.C + c] == 0.f) return;
    const int R = p.R, kc = p.keep_count, tid = threadIdx.x, nthr = blockDim.x;
    const int slot = (l * p.n_img + img) * p.C + c;
    const ImageRows ir = image_rows(p, n_props, p_seed, img);
    const int n = ir.n;
    while ((npad >> 1) >= n) npad >>= 1;                              // the image's own power of two

    int *seeds = reinterpret_cast<int *>(smem_raw);                   // [kc]
    unsigned char *big = smem_raw + align_up((size_t)kc * 4, 16);
    float *key = reinterpret_cast<float *>(big);                      // [npad]
    int *idx = reinterpret_cast<int *>(big + (size_t)npad * 4);       // [npad]

    const int bg = (p.C1 == p.C + 1) ? 1 : 0;
    const float *cls = ptrs.cls[l] + (size_t)img * R * p.C1;
    const float *det = ptrs.det[l] ? ptrs.det[l] + (size_t)img * R * p.det_cols : nullptr;
    const int dcol = p.det_cols == 1 ? 0 : c + (p.det_cols == p.C + 1 ? 1 : 0);
    for (int i = tid; i < npad; i += nthr) {
        float v = -INFINITY;
        if (i < n) {
            v = cls[(size_t)i * p.C1 + c + bg];
            if (p.mode == 1 && det) v = __fmul_rn(v, det[(size_t)i * p.det_cols + dcol]);   // MIST ranks cls*det
        }
        key[i] = v;
        idx[i] = i < n ? i : 0x7fffffff;
    }
    __syncthreads();
    for (int size = 2; size <= npad; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (npad >> 1); t += nthr) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;       // "ascending" = sorted by before()
                const float ka = key[lo], kb = key[hi];
                const int ia = idx[lo], ib = idx[hi];
                const bool swap = asc ? before(kb, ib, ka, ia) : before(ka, ia, kb, ib);
                if (swap) { key[lo] = kb; key[hi] = ka; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    const int k = min(ir.keep_count, n);
    for (int i = tid; i < k; i += nthr) seeds[i] = idx[i];
    __syncthreads();

    // suppression bitmask over the sort buffer: supp[a][w] bit b set <=> NOT (iou[a][b] < thr)
    const int kw = (k + 31) >> 5;
    uint32_t *supp = reinterpret_cast<uint32_t *>(big);               // [k][kw]
    const __half *iou = iou_all + (size_t)img * R * R;
    const __half thr = __float2half_rn(p.cls_thr[l]);
    const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
    // 4 (seed a, word w) entries per warp and round: the gathers are dependent loads of L2 latency, so they are all
    // issued before the first ballot (one entry at a time this loop was half of the kernel)
    constexpr int SU = 4;
    for (int e0 = warp * SU; e0 < k * kw; e0 += nwarp * SU) {
        __half v[SU];
        bool ok[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const int e = e0 + u, a = e / kw, w = e - a * kw, b = w * 32 + lane;
            ok[u] = e < k * kw && b < k && b > a;
            v[u] = ok[u] ? iou[(size_t)seeds[a] * R + seeds[b]] : __float2half_rn(0.f);
        }
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const bool s = ok[u] && !__hlt(v[u], thr);
            const uint32_t word = __ballot_sync(0xffffffffu, s);
            if (lane == 0 && e0 + u < k * kw) supp[e0 + u] = word;
        }
    }
    __syncthreads();
    if (warp == 0) {
        uint32_t alive = 0xffffffffu;            // lane j: candidates 32j .. 32j+31 (kw <= 32)
        int nk = 0;
        int *kept = ws.kept + (size_t)slot * kc;
        for (int a = 0; a < k; ++a) {
            const uint32_t wa = __shfl_sync(0xffffffffu, alive, a >> 5);
            if ((wa >> (a & 31)) & 1u) {
                if (lane == 0) kept[nk] = seeds[a];
                ++nk;
                if (lane < kw) alive &= ~supp[a * kw + lane];
            }
        }
        if (lane == 0) ws.nkept[slot] = nk;
    }
}

// ------------------------------------------------------------------------- containment pass
__global__ void __launch_bounds__(256)
cim_contain_kernel(LayerPtrs ptrs, const float *__restrict__ labels, const __half *__restrict__ asy_all,
                   cim_mine_params p, MineWs ws, uint8_t *__restrict__ asy_flag, const int32_t *__restrict__ n_props,
                   double p_seed) {
    const int img = blockIdx.y, lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int R = p.R;
    if (i >= R) return;
    const int n = n_props ? min(max(n_props[img], 1), R) : R;
    if (i >= n) {                                                   // padding row: never big, never a container
        if (lane == 0 && asy_flag) asy_flag[(size_t)img * R + i] = 0;
        return;
    }
    const __half *row = asy_all + ((size_t)img * R + i) * R;
    const __half con = __float2half_rn(p.con_thr);
    int cnt = 0;
    if ((R & 1) == 0 && (((uintptr_t)row) & 3) == 0) {
        const __half2 *row2 = reinterpret_cast<const __half2 *>(row);
        for (int j = lane; j < (n >> 1); j += 32) {
            const __half2 v = row2[j];
            cnt += (int)__hgt(__low2half(v), con) + (int)__hgt(__high2half(v), con);
        }
        if ((n & 1) && lane == 0) cnt += (int)__hgt(row[n - 1], con);
    } else {
        for (int j = lane; j < n; j += 32) cnt += (int)__hgt(row[j], con);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const float big_thr = n_props ? image_rows(p, n_props, p_seed, img).big_thr : p.big_thr;
    const bool flag = (float)cnt < big_thr;                         // heads.py:338
    if (lane == 0 && asy_flag) asy_flag[(size_t)img * R + i] = flag ? 1 : 0;
    if (!flag || p.mode != 0) return;

    for (int l = 0; l < p.n_layers; ++l) {
        const float *det = ptrs.det[l] + ((size_t)img * R + i) * p.det_cols;
        for (int c = 0; c < p.C; ++c) {
            if (labels[(size_t)img * p.C + c] == 0.f) continue;
            const int slot = (l * p.n_img + img) * p.C + c;
            const int nk = ws.nkept[slot];
            const int *kept = ws.kept + (size_t)slot * p.keep_count;
            unsigned long long *best = ws.best + (size_t)slot * p.keep_count;
            const float d = det[p.det_cols == 1 ? 0 : c + (p.det_cols == p.C + 1 ? 1 : 0)];
            // key: (det score bits, ~row) -> max score, ties to the lowest row; the low word is
            // never 0, so key != 0 also means "this seed has at least one container"
            const unsigned long long keyv =
                ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)(0xffffffffu - (unsigned)i);
            for (int s = lane; s < nk; s += 32)
                if (__hgt(row[kept[s]], con)) atomicMax(best + s, keyv);
        }
    }
}

// ------------------------------------------------------------------- class arbitration + lists
__global__ void __launch_bounds__(1024)
cim_merge_kernel(LayerPtrs ptrs, const float *__restrict__ labels, cim_mine_params p, MineWs ws,
                 int32_t *__restrict__ gt_count, int32_t *__restrict__ gt_rows, int32_t *__restrict__ gt_class,
                 float *__restrict__ gt_weight) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int l = blockIdx.x, img = blockIdx.y, tid = threadIdx.x, nthr = blockDim.x, R = p.R;
    int *g_cls = reinterpret_cast<int *>(smem_raw);          // [R]
    float *g_w = reinterpret_cast<float *>(g_cls + R);       // [R]
    __shared__ int scan[1024];
    for (int i = tid; i < R; i += nthr) { g_cls[i] = -1; g_w[i] = -1.f; }
    __syncthreads();

    const int bg = (p.C1 == p.C + 1) ? 1 : 0;
    const float *cls = ptrs.cls[l] + (size_t)img * R * p.C1;
    const float *det = ptrs.det[l] ? ptrs.det[l] + (size_t)img * R * p.det_cols : nullptr;
    for (int c = 0; c < p.C; ++c) {
        if (labels[(size_t)img * p.C + c] == 0.f) continue;          // uniform
        const int slot = (l * p.n_img + img) * p.C + c;
        const int nk = ws.nkept[slot];
        const int dcol = p.det_cols == 1 ? 0 : c + (p.det_cols == p.C + 1 ? 1 : 0);
        int row = -1;
        float pv = 0.f;
        bool take = false;
        if (tid < nk) {
            if (p.mode == 0) {
                const unsigned long long key = ws.best[(size_t)slot * p.keep_count + tid];
                if (key != 0ull) {
                    // all containers scored exactly 0: torch.argmax over the zero column -> row 0
                    row = (key >> 32) == 0ull ? 0 : (int)(0xffffffffu - (unsigned)(key & 0xffffffffull));
                }
            } else {
                row = ws.kept[(size_t)slot * p.keep_count + tid];
            }
            if (row >= 0) {
                const float cv = cls[(size_t)row * p.C1 + c + bg];
                pv = det ? __fmul_rn(cv, det[(size_t)row * p.det_cols + dcol]) : cv;   // preds = cls*det
                take = pv > g_w[row];
            }
        }
        __syncthreads();
        if (take) { g_cls[row] = c; g_w[row] = pv; }    // duplicates write identical values
        __syncthreads();
    }

    // compaction in ascending proposal order
    const int per = (R + nthr - 1) / nthr, s0 = min(R, tid * per), s1 = min(R, s0 + per);
    int cnt = 0;
    for (int i = s0; i < s1; ++i) cnt += g_cls[i] >= 0;
    scan[tid] = cnt;
    __syncthreads();
    for (int o = 1; o < nthr; o <<= 1) {
        int v = tid >= o ? scan[tid - o] : 0;
        __syncthreads();
        scan[tid] += v;
        __syncthreads();
    }
    int pos = scan[tid] - cnt;
    const size_t base = ((size_t)l * p.n_img + img) * p.gt_cap;
    for (int i = s0; i < s1; ++i)
        if (g_cls[i] >= 0) {
            if (pos < p.gt_cap) {
                gt_rows[base + pos] = i;
                gt_class[base + pos] = g_cls[i];
                gt_weight[base + pos] = g_w[i];
            }
            ++pos;
        }
    if (tid == nthr - 1) gt_count[l * p.n_img + img] = min(scan[tid], p.gt_cap);
}

// ------------------------------------------------------------------------------- assignment
__global__ void __launch_bounds__(256)
cim_assign_kernel(cim_mine_params p, const __half *__restrict__ iou_all, const int32_t *__restrict__ gt_count,
                  const int32_t *__restrict__ gt_rows, const int32_t *__restrict__ gt_class,
                  const float *__restrict__ gt_weight, const uint8_t *__restrict__ gt_keep,
                  float *__restrict__ pseudo_labels, __half *__restrict__ pseudo_iou,
                  float *__restrict__ loss_weights, uint8_t *__restrict__ valid, const int32_t *__restrict__ n_props) {
    const int l = blockIdx.y, img = blockIdx.z, lane = threadIdx.x & 31, R = p.R;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= R) return;
    const int li = l * p.n_img + img;
    const int C1o = p.C + 1;
    if (n_props && i >= min(max(n_props[img], 1), R)) {             // padding row: the ignore row (heads.py:484-486)
        float *pl = pseudo_labels + ((size_t)li * R + i) * C1o;
        for (int c = lane; c < C1o; c += 32) pl[c] = 0.f;
        if (lane == 0) {
            pseudo_iou[(size_t)li * R + i] = __float2half_rn(0.f);
            loss_weights[(size_t)li * R + i] = 0.f;
        }
        return;
    }
    const int G = gt_count[li];
    const size_t gbase = (size_t)li * p.gt_cap;
    const __half *row = iou_all + ((size_t)img * R + i) * R;

    // torch.max(dim=-1): first maximum; a NaN beats everything and the first NaN wins
    float bv = -INFINITY;
    int bg_ = 0x7fffffff, nan_g = 0x7fffffff, seen = 0;
    __half bh = __float2half_rn(0.f);
    for (int g = lane; g < G; g += 32) {
        if (gt_keep && !gt_keep[gbase + g]) continue;
        seen = 1;
        const __half h = row[gt_rows[gbase + g]];
        const float v = __half2float(h);
        if (v != v) { if (nan_g == 0x7fffffff) nan_g = g; continue; }
        if (bg_ == 0x7fffffff || v > bv) { bv = v; bg_ = g; bh = h; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int og = __shfl_xor_sync(0xffffffffu, bg_, o);
        const unsigned short oh = __shfl_xor_sync(0xffffffffu, __half_as_ushort(bh), o);
        const int on = __shfl_xor_sync(0xffffffffu, nan_g, o);
        seen |= __shfl_xor_sync(0xffffffffu, seen, o);
        nan_g = min(nan_g, on);
        if (og != 0x7fffffff && (bg_ == 0x7fffffff || ov > bv || (ov == bv && og < bg_))) {
            bv = ov; bg_ = og; bh = __ushort_as_half(oh);
        }
    }
    float *pl = pseudo_labels + ((size_t)li * R + i) * C1o;
    if (!seen) {                                  // nothing mined for this (layer, image)
        for (int c = lane; c < C1o; c += 32) pl[c] = 0.f;
        if (lane == 0) {
            pseudo_iou[(size_t)li * R + i] = __float2half_rn(0.f);
            loss_weights[(size_t)li * R + i] = 0.f;
            if (i == 0) valid[li] = 0;
        }
        return;
    }
    int g;
    __half mv;
    if (nan_g != 0x7fffffff) { g = nan_g; mv = row[gt_rows[gbase + g]]; }
    else { g = bg_; mv = bh; }
    const __half zero = __float2half_rn(0.f);
    const __half cthr = __float2half_rn(p.cls_thr[l]), ithr = __float2half_rn(p.iou_thr[l]);
    const bool ignore = __heq(mv, zero);                              // heads.py:484
    const bool bgrow = __hlt(mv, cthr) && !ignore;                    // heads.py:489
    const int hot = ignore ? -1 : (bgrow ? 0 : gt_class[gbase + g] + 1);
    for (int c = lane; c < C1o; c += 32) pl[c] = c == hot ? 1.f : 0.f;
    if (lane == 0) {
        loss_weights[(size_t)li * R + i] = ignore ? 0.f : gt_weight[gbase + g];
        __half out = mv;                                              // NaN stays NaN (:500-501)
        if (__hgt(mv, ithr)) out = __float2half_rn(1.f);
        else if (__hle(mv, ithr)) out = zero;
        pseudo_iou[(size_t)li * R + i] = out;
        if (i == 0) valid[li] = 1;
    }
}


// ------------------------------------------------------------------------------ anti-noise sampling
// heads.py:440-473 with the arithmetic of numpy's RandomState.choice(replace=True, p=...) on the device; only the
// uniform doubles come from the host (numpy's GLOBAL RNG, so that the stream stays in step with the reference).
// numpy's float32 add.reduce (pairwise summation, loops_utils.h.src): n < 8 sequential from 0; n <= 128 eight
// running sums + the rest sequentially; above that halves, the left one a multiple of 8.
__device__ float np_pairwise_sum_f32(const float *a, int n) {
    if (n < 8) {
        float r = 0.f;
        for (int i = 0; i < n; ++i) r = __fadd_rn(r, a[i]);
        return r;
    }
    if (n <= 128) {
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = a[j];
        int i = 8;
        for (; i < n - (n % 8); i += 8)
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], a[i + j]);
        float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                              __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
        for (; i < n; ++i) res = __fadd_rn(res, a[i]);
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return __fadd_rn(np_pairwise_sum_f32(a, n2), np_pairwise_sum_f32(a + n2, n - n2));
}

// One warp per (layer, image).  For every present class c (ascending) with n > 0 pseudo GTs at list positions
// idx[0..n): p = w[idx] / sum(w[idx]) (float32) -> float64 cumsum -> / last -> j_t = #{cdf <= u_t} for the class's n
// uniforms; keep[idx] = 0, keep[idx[j_t]] = 1.  The uniforms of (image b, layer l, class c) follow those of every
// earlier (image, layer) -- image-major, the order in which the reference's training loop reaches np.random.choice --
// and of the smaller present classes of the same list.
__global__ void __launch_bounds__(32)
cim_anti_noise_kernel(cim_mine_params p, const float *__restrict__ labels, const int *__restrict__ gt_count,
                      const int *__restrict__ gt_class, const float *__restrict__ gt_weight,
                      const double *__restrict__ uniforms, unsigned char *__restrict__ gt_keep,
                      const long long *__restrict__ cursor_in, long long *__restrict__ cursor_out, long long ring_len) {
    extern __shared__ __align__(16) unsigned char an_smem[];
    const int l = blockIdx.x, img = blockIdx.y, lane = threadIdx.x;
    const int g = min(gt_count[l * p.n_img + img], p.gt_cap);
    // stream mode (cim_anti_noise_stream): `uniforms` is a ring holding a stretch of the host's random stream, the
    // step's first double sits at absolute position *cursor_in; the first block leaves *cursor_in + (doubles this
    // step consumes) in *cursor_out for the next step (a different word: the other blocks still read *cursor_in)
    const long long cbase = cursor_in ? *cursor_in : 0;
    if (cursor_out && l == 0 && img == 0) {
        long long tot = 0;
        for (int t = lane; t < p.n_img * p.n_layers; t += 32) tot += min(gt_count[t], p.gt_cap);
#pragma unroll
        for (int s = 16; s; s >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, s);
        if (lane == 0) *cursor_out = cbase + tot;
    }
    double *cdf = reinterpret_cast<double *>(an_smem);                 // [gt_cap]
    int *idx = reinterpret_cast<int *>(cdf + p.gt_cap);                // [gt_cap]
    float *prob = reinterpret_cast<float *>(idx + p.gt_cap);           // [gt_cap]
    const size_t base = ((size_t)l * p.n_img + img) * p.gt_cap;
    for (int i = lane; i < p.gt_cap; i += 32) gt_keep[base + i] = 1;
    if (g == 0) return;
    // first uniform of this list: lists of earlier images (all layers) and of earlier layers of this image
    long long off = 0;
    for (int t = lane; t < img * p.n_layers + l; t += 32) {
        const int bb = t / p.n_layers, ll = t - bb * p.n_layers;
        off += min(gt_count[ll * p.n_img + bb], p.gt_cap);
    }
#pragma unroll
    for (int s = 16; s; s >>= 1) off += __shfl_xor_sync(0xffffffffu, off, s);
    __syncwarp();
    for (int c = 0; c < p.C; ++c) {
        if (labels[(size_t)img * p.C + c] == 0.f) continue;            // warp-uniform
        int n = 0;
        for (int i0 = 0; i0 < g; i0 += 32) {                           // stable compaction of the class's positions
            const int i = i0 + lane;
            const bool hit = i < g && gt_class[base + i] == c;
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (hit) {
                const int pos = n + __popc(m & ((1u << lane) - 1u));
                idx[pos] = i;
                prob[pos] = gt_weight[base + i];
            }
            n += __popc(m);
        }
        __syncwarp();
        if (n == 0) continue;
        if (lane == 0) {
            const float s = np_pairwise_sum_f32(prob, n);
            if (s == 0.f) {
                // every weight of the class is 0: np.random.choice raises there (p = 0/0).  Deliberate divergence,
                // shared with heads._anti_noise_keep: all n draws pick the class's first pseudo GT (cdf = 1 > u),
                // and the class still consumes its n uniforms, so the stream stays in step for the classes after it
                for (int i = 0; i < n; ++i) cdf[i] = 1.0;
            } else {
                double acc = 0.0;
                for (int i = 0; i < n; ++i) {                          // np.cumsum: sequential, float64
                    const double v = (double)__fdiv_rn(prob[i], s);
                    acc = i == 0 ? v : __dadd_rn(acc, v);
                    cdf[i] = acc;
                }
                const double last = cdf[n - 1];
                for (int i = 0; i < n; ++i) cdf[i] = __ddiv_rn(cdf[i], last);
            }
        }
        __syncwarp();
        for (int i = lane; i < n; i += 32) gt_keep[base + idx[i]] = 0;
        __syncwarp();
        for (int t = lane; t < n; t += 32) {
            const double u = ring_len ? uniforms[(cbase + off + t) % ring_len] : uniforms[off + t];
            int lo = 0, hi = n;                                        // searchsorted(side='right'): first cdf > u
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
            }
            gt_keep[base + idx[min(lo, n - 1)]] = 1;
        }
        __syncwarp();
        off += n;
    }
}

int check_params(const cim_mine_params *p) {
    if (!p) return CIM_ERR_ARG;
    if (p->n_img <= 0 || p->R <= 0 || p->C <= 0 || p->n_layers <= 0 || p->gt_cap <= 0) return CIM_ERR_ARG;
    if (p->n_layers > MAX_LAYERS || p->R > 10240 || p->keep_count < 1 || p->keep_count > 1024) return CIM_ERR_SHAPE;
    if (p->C1 != p->C && p->C1 != p->C + 1) return CIM_ERR_ARG;
    if (p->det_cols != p->C && p->det_cols != p->C + 1 && p->det_cols != 1) return CIM_ERR_ARG;
    if (p->mode != 0 && p->mode != 1) return CIM_ERR_ARG;
    if (p->n_img > 65535 || p->C > 65535) return CIM_ERR_SHAPE;
    return CIM_OK;
}

}  // namespace

CIM_API size_t cim_mine_workspace_bytes(const cim_mine_params *p) {
    if (check_params(p)) return 0;
    const size_t slots = (size_t)p->n_layers * p->n_img * p->C;
    return align_up(slots * p->keep_count * 8, 256) + align_up(slots * p->keep_count * 4, 256) +
           align_up(slots * 4, 256);
}

CIM_API int cim_mine_image_constants(double p_seed, int n, int *keep_count, float *big_thr) {
    if (!keep_count || !big_thr || n < 1 || !(p_seed > 0.0 && p_seed <= 1.0)) return CIM_ERR_ARG;
    cim_image_constants(p_seed, n, keep_count, big_thr);
    return CIM_OK;
}

CIM_API int cim_mine_ex(const cim_mine_params *p, const int32_t *n_props, double p_seed, const float *const *cls,
                        const float *const *det, const float *labels, const void *iou_f16, const void *asy_f16,
                        int32_t *gt_count, int32_t *gt_rows, int32_t *gt_class, float *gt_weight, uint8_t *asy_flag,
                        void *workspace, size_t ws_bytes, cim_stream_t stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if (n_props) {
        if (!(p_seed > 0.0 && p_seed <= 1.0)) return CIM_ERR_ARG;
        int kc_full;
        float bt;
        cim_image_constants(p_seed, p->R, &kc_full, &bt);
        if (p->keep_count < kc_full) return CIM_ERR_ARG;          // the capacity must hold a full image's seeds
        if (!cim_aligned(n_props, 4)) return CIM_ERR_ALIGN;
    }
    if (!cls || !labels || !iou_f16 || !gt_count || !gt_rows || !gt_class || !gt_weight) return CIM_ERR_ARG;
    if (p->mode == 0 && (!det || !asy_f16)) return CIM_ERR_ARG;
    if (!workspace || ws_bytes < cim_mine_workspace_bytes(p) || !cim_aligned(workspace, 256)) return CIM_ERR_WORKSPACE;
    LayerPtrs ptrs{};
    for (int l = 0; l < p->n_layers; ++l) {
        if (!cls[l] || (p->mode == 0 && !det[l])) return CIM_ERR_ARG;
        ptrs.cls[l] = cls[l];
        ptrs.det[l] = det ? det[l] : nullptr;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const MineWs ws = carve_ws(workspace, *p);
    cudaMemsetAsync(workspace, 0, cim_mine_workspace_bytes(p), st);

    int npad = 1;
    while (npad < p->R) npad <<= 1;
    const int k = p->keep_count < p->R ? p->keep_count : p->R, kw = (k + 31) / 32;
    size_t big = (size_t)npad * 8;
    if ((size_t)k * kw * 4 > big) big = (size_t)k * kw * 4;
    const size_t smem_seed = align_up((size_t)p->keep_count * 4, 16) + big;
    if (smem_seed > (size_t)cim_max_smem_optin()) return CIM_ERR_SHAPE;
    cudaFuncSetAttribute(cim_seed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_seed);
    cim_seed_kernel<<<dim3(p->C, p->n_layers, p->n_img), 512, smem_seed, st>>>(
        ptrs, labels, reinterpret_cast<const __half *>(iou_f16), *p, npad, ws, n_props, p_seed);
    if ((rc = cim_launch_status())) return rc;

    if (p->mode == 0 || asy_flag) {
        if (asy_f16) {
            cim_contain_kernel<<<dim3((p->R + 7) / 8, p->n_img), 256, 0, st>>>(
                ptrs, labels, reinterpret_cast<const __half *>(asy_f16), *p, ws, asy_flag, n_props, p_seed);
            if ((rc = cim_launch_status())) return rc;
        }
    }
    const size_t smem_merge = (size_t)p->R * 8;
    cudaFuncSetAttribute(cim_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_merge);
    cim_merge_kernel<<<dim3(p->n_layers, p->n_img), 1024, smem_merge, st>>>(ptrs, labels, *p, ws, gt_count, gt_rows,
                                                                            gt_class, gt_weight);
    return cim_launch_status();
}

CIM_API int cim_mine(const cim_mine_params *p, const float *const *cls, const float *const *det,
                     const float *labels, const void *iou_f16, const void *asy_f16, int32_t *gt_count,
                     int32_t *gt_rows, int32_t *gt_class, float *gt_weight, uint8_t *asy_flag, void *workspace,
                     size_t ws_bytes, cim_stream_t stream) {
    return cim_mine_ex(p, nullptr, 0.0, cls, det, labels, iou_f16, asy_f16, gt_count, gt_rows, gt_class, gt_weight,
                       asy_flag, workspace, ws_bytes, stream);
}

CIM_API int cim_assign_ex(const cim_mine_params *p, const int32_t *n_props, const void *iou_f16,
                          const int32_t *gt_count, const int32_t *gt_rows, const int32_t *gt_class,
                          const float *gt_weight, const uint8_t *gt_keep, float *pseudo_labels, void *pseudo_iou_f16,
                          float *loss_weights, uint8_t *valid, cim_stream_t stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if (!iou_f16 || !gt_count || !gt_rows || !gt_class || !gt_weight || !pseudo_labels || !pseudo_iou_f16 ||
        !loss_weights || !valid)
        return CIM_ERR_ARG;
    if (!cim_aligned(n_props, 4)) return CIM_ERR_ALIGN;
    cim_assign_kernel<<<dim3((p->R + 7) / 8, p->n_layers, p->n_img), 256, 0, (cudaStream_t)stream>>>(
        *p, reinterpret_cast<const __half *>(iou_f16), gt_count, gt_rows, gt_class, gt_weight, gt_keep,
        pseudo_labels, reinterpret_cast<__half *>(pseudo_iou_f16), loss_weights, valid, n_props);
    return cim_launch_status();
}

CIM_API int cim_assign(const cim_mine_params *p, const void *iou_f16, const int32_t *gt_count,
                       const int32_t *gt_rows, const int32_t *gt_class, const float *gt_weight,
                       const uint8_t *gt_keep, float *pseudo_labels, void *pseudo_iou_f16, float *loss_weights,
                       uint8_t *valid, cim_stream_t stream) {
    return cim_assign_ex(p, nullptr, iou_f16, gt_count, gt_rows, gt_class, gt_weight, gt_keep, pseudo_labels,
                         pseudo_iou_f16, loss_weights, valid, stream);
}

CIM_API size_t cim_anti_noise_uniform_count_max(const cim_mine_params *p) {
    if (check_params(p)) return 0;
    return (size_t)p->n_layers * p->n_img * p->gt_cap;
}

CIM_API int cim_anti_noise(const cim_mine_params *p, const float *labels, const int32_t *gt_count,
                           const int32_t *gt_class, const float *gt_weight, const double *uniforms,
                           uint8_t *gt_keep, cim_stream_t stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if (!labels || !gt_count || !gt_class || !gt_weight || !uniforms || !gt_keep) return CIM_ERR_ARG;
    if (!cim_aligned(uniforms, 8)) return CIM_ERR_ALIGN;
    const size_t smem = (size_t)p->gt_cap * 16;
    if (smem > (size_t)cim_max_smem_optin()) return CIM_ERR_SHAPE;
    cudaFuncSetAttribute(cim_anti_noise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cim_anti_noise_kernel<<<dim3(p->n_layers, p->n_img), 32, smem, (cudaStream_t)stream>>>(
        *p, labels, gt_count, gt_class, gt_weight, uniforms, gt_keep, nullptr, nullptr, 0);
    return cim_launch_status();
}

CIM_API int cim_anti_noise_stream(const cim_mine_params *p, const float *labels, const int32_t *gt_count,
                                  const int32_t *gt_class, const float *gt_weight, const double *ring,
                                  int64_t ring_len, const int64_t *cursor_in, int64_t *cursor_out, uint8_t *gt_keep,
                                  cim_stream_t stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if (!labels || !gt_count || !gt_class || !gt_weight || !ring || !gt_keep || !cursor_in || !cursor_out)
        return CIM_ERR_ARG;
    if (cursor_in == cursor_out) return CIM_ERR_ARG;
    if (ring_len < (int64_t)p->n_layers * p->n_img * p->gt_cap) return CIM_ERR_SHAPE;
    if (!cim_aligned(ring, 8) || !cim_aligned(cursor_in, 8) || !cim_aligned(cursor_out, 8)) return CIM_ERR_ALIGN;
    const size_t smem = (size_t)p->gt_cap * 16;
    if (smem > (size_t)cim_max_smem_optin()) return CIM_ERR_SHAPE;
    cudaFuncSetAttribute(cim_anti_noise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cim_anti_noise_kernel<<<dim3(p->n_layers, p->n_img), 32, smem, (cudaStream_t)stream>>>(
        *p, labels, gt_count, gt_class, gt_weight, ring, gt_keep, reinterpret_cast<const long long *>(cursor_in),
        reinterpret_cast<long long *>(cursor_out), (long long)ring_len);
    return cim_launch_status();
}
