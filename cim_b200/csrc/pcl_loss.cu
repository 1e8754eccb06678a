// pcl_loss.cu -- PCL_loss (lib/modeling/heads.py:10-41 of the reference, the proposal-cluster loss of
// https://arxiv.org/abs/1807.03342 as CIM uses it) forward + backward in one launch (SURVEY.md 8f-2).
//
//   mat [R, C+1] holds cluster ids written by tools/pre/AGPL_label_assign.py:60-96: a foreground cluster k > 0 sits in
//   the class column of its peak for the proposals assigned to it; the background cluster's id sits in column 0.
//   Reference, per image:
//     bg_ind = the single non-zero value of mat[:, 0] (none: no background cluster)                       (:13-21)
//     for every distinct id k != 0 in ascending order:                                                     (:23)
//       rows_k = rows of mat containing k,  n_k = |rows_k|
//       foreground k != bg_ind:  v = mean over rows_k of predict_cls,  t = columns of mat containing k,
//                                loss += n_k * mean_c BCE(clamp(v_c), t_c)                                 (:25-32)
//       background k == bg_ind:  loss += n_k * mean_{r in rows_k, c} BCE(clamp(p[r][c]), mat[r][c] != 0)    (:34-39)
//     return 12 * loss / (1e-6 + sum_k n_k)                                                                (:40-41)
//   The reference loops over `mat.unique()` on the host with ~10 launches and two syncs per cluster; here one CTA
//   per image makes three passes over its [R, C+1] slices (8 rows in flight per thread: the work is latency bound):
//   ids -> per-row id lists and cluster tables in shared memory; cluster sums in 2^-44 fixed point, so the
//   shared-memory atomics commute exactly (deterministic); gradients.
// Cluster ids must be integers in [1, max_id] (they are small counters); anything else, or two different ids in
// column 0 (the reference asserts there), yields a NaN loss and zero gradient.
// Ragged batches (cim_pcl_loss_ex): mat is read as 0 for rows r >= n_props[b], so those rows join no cluster and get
// a zero gradient (or keep what grad_cls held, with accumulate).
#include "common.cuh"

namespace {

constexpr int PT = 1024;
constexpr int MAX_ROW_IDS = 4;
constexpr float LO = 1e-6f, HI = 1.f - 1e-6f;

__device__ __forceinline__ float clampf(float v) { return fminf(fmaxf(v, LO), HI); }
__device__ __forceinline__ bool in_clamp(float v) { return v >= LO && v <= HI; }
__device__ __forceinline__ float bce(float p, float t) { return -t * logf(p) - (1.f - t) * logf(1.f - p); }
__device__ __forceinline__ float dbce(float p, float t) { return -(t / p - (1.f - t) / (1.f - p)); }

__device__ float block_sum_p(float v, float *red) {
    const int tid = threadIdx.x;
    __syncthreads();
    red[tid] = v;
    __syncthreads();
    for (int o = PT / 2; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    return red[0];
}

constexpr int UN = 8;                                   // rows in flight per thread: the passes are latency bound
// Cluster sums are accumulated in fixed point (units of 2^-44), so the shared-memory atomics commute exactly
// (deterministic).  Every float32 at or above 2^-21 is a whole number of units, so a cluster of one row has exactly
// that row's scores as its mean and the clamp at float32(1e-6) decides as the reference does (with 2^-40 units a score
// one ulp below the bound was rounded up onto the other side of it).  16384 rows of scores <= 1 stay below 2^58.
constexpr float FIX = 17592186044416.f;                 // 2^44

// insert `id` into the row's list of distinct ids (4 x 8 bit in one word); true if this call added it
__device__ __forceinline__ bool row_add_id(uint32_t *slot, int id, int *err) {
    uint32_t cur = *reinterpret_cast<volatile uint32_t *>(slot);
    while (true) {
        int free_j = -1;
        for (int j = 0; j < MAX_ROW_IDS; ++j) {
            const int v = (cur >> (8 * j)) & 255;
            if (v == id) return false;
            if (v == 0 && free_j < 0) free_j = j;
        }
        if (free_j < 0) { atomicOr(err, 1); return false; }
        const uint32_t old = atomicCAS(slot, cur, cur | ((uint32_t)id << (8 * free_j)));
        if (old == cur) return true;
        cur = old;
    }
}

__global__ void __launch_bounds__(PT)
cim_pcl_loss_kernel(const float *__restrict__ pcls, const float *__restrict__ mat, float *__restrict__ loss_out,
                    float *__restrict__ grad, const int32_t *__restrict__ n_props, int R, int C1, int max_id,
                    float grad_scale, int accumulate) {
    extern __shared__ __align__(16) unsigned char dyn[];
    // layout: sum64 [max_id+1][C1] i64 (later re-used as vgrad f32) | cnt [max_id+1] i32 | colmask [max_id+1][4] u32 |
    //         lk [max_id+1] f32 | rowids [R] u32 (4 x 8-bit distinct ids of the row)
    const int NI = max_id + 1;
    unsigned long long *sum64 = reinterpret_cast<unsigned long long *>(dyn);
    int *cnt = reinterpret_cast<int *>(sum64 + (size_t)NI * C1);
    uint32_t *colmask = reinterpret_cast<uint32_t *>(cnt + NI);
    float *lk = reinterpret_cast<float *>(colmask + (size_t)NI * 4);
    uint32_t *rowids = reinterpret_cast<uint32_t *>(lk + NI);
    __shared__ float red[PT];
    __shared__ int s_bgmin, s_bgmax, s_err;

    const int b = blockIdx.x, tid = threadIdx.x;
    const float *p = pcls + (size_t)b * R * C1;
    const float *m = mat + (size_t)b * R * C1;
    float *g = grad ? grad + (size_t)b * R * C1 : nullptr;
    const int G = PT / C1, rg = tid / C1, c = tid - rg * C1;
    const bool elem = tid < G * C1;
    const int n = n_props ? min(max(n_props[b], 1), R) : R;          // rows of this image; the rest read as mat = 0

    for (int i = tid; i < NI * C1; i += PT) sum64[i] = 0ull;
    for (int i = tid; i < NI; i += PT) { cnt[i] = 0; lk[i] = 0.f; }
    for (int i = tid; i < NI * 4; i += PT) colmask[i] = 0u;
    for (int i = tid; i < R; i += PT) rowids[i] = 0u;
    if (tid == 0) { s_bgmin = 0x7fffffff; s_bgmax = 0; s_err = 0; }
    __syncthreads();

    // pass 1, thread = (row group, class): cluster ids -> per-row id lists, cluster sizes, class columns, background id
    if (elem)
        for (int r0 = rg; r0 < R; r0 += G * UN) {
            float v[UN];
#pragma unroll
            for (int i = 0; i < UN; ++i) {
                const int r = r0 + i * G;
                v[i] = r < n ? __ldg(m + (size_t)r * C1 + c) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < UN; ++i) {
                if (v[i] == 0.f) continue;
                const int r = r0 + i * G, id = (int)v[i];
                if (!(v[i] > 0.f) || (float)id != v[i] || id > max_id) { atomicOr(&s_err, 1); continue; }
                atomicOr(&colmask[id * 4 + (c >> 5)], 1u << (c & 31));
                if (c == 0) { atomicMin(&s_bgmin, id); atomicMax(&s_bgmax, id); }
                if (row_add_id(&rowids[r], id, &s_err)) atomicAdd(&cnt[id], 1);
            }
        }
    __syncthreads();
    const int bg = s_bgmax > 0 ? s_bgmin : -1;
    if (s_err || (s_bgmax > 0 && s_bgmin != s_bgmax)) {               // heads.py:20 asserts a single background id
        if (tid == 0) loss_out[b] = __int_as_float(0x7fc00000);
        if (g && !accumulate)
            for (int e = tid; e < R * C1; e += PT) g[e] = 0.f;
        return;
    }

    // pass 2: foreground cluster sums (fixed point), background BCE
    float bsum = 0.f;
    if (elem)
        for (int r0 = rg; r0 < R; r0 += G * UN) {
            float pv[UN], mv[UN];
            uint32_t ids[UN];
#pragma unroll
            for (int i = 0; i < UN; ++i) {
                const int r = r0 + i * G;
                ids[i] = r < R ? rowids[r] : 0u;
                pv[i] = (r < R && ids[i]) ? __ldg(p + (size_t)r * C1 + c) : 0.f;
                mv[i] = (r < R && ids[i]) ? __ldg(m + (size_t)r * C1 + c) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < UN; ++i)
                for (uint32_t w = ids[i]; w; w >>= 8) {
                    const int id = w & 255;
                    if (id == bg) bsum += bce(clampf(pv[i]), mv[i] != 0.f ? 1.f : 0.f);
                    else atomicAdd(&sum64[id * C1 + c], (unsigned long long)(long long)__float2ll_rn(pv[i] * FIX));
                }
        }
    bsum = block_sum_p(bsum, red);                                     // (syncs: the sums are complete)

    // per cluster and class: mean -> BCE against the cluster's class columns, and its derivative
    for (int i = tid; i < NI * C1; i += PT) {
        const int k = i / C1, cc = i - k * C1;
        float gk = 0.f, lkc = 0.f;
        if (k >= 1 && k != bg && cnt[k] > 0) {
            const float v = (float)((double)(long long)sum64[i] * (1.0 / (double)FIX) / (double)cnt[k]);
            const float vc = clampf(v), tgt = (colmask[k * 4 + (cc >> 5)] >> (cc & 31)) & 1u ? 1.f : 0.f;
            gk = in_clamp(v) ? dbce(vc, tgt) / C1 : 0.f;
            lkc = bce(vc, tgt);
        }
        // sum64[i] (8 bytes) is replaced by (gradient coefficient, loss term) of the same entry
        reinterpret_cast<float2 *>(sum64)[i] = make_float2(gk, lkc);
    }
    __syncthreads();
    for (int k = tid; k < NI; k += PT) {                               // per cluster: class order
        float l = 0.f;
        if (k >= 1 && k != bg && cnt[k] > 0)
            for (int cc = 0; cc < C1; ++cc) l += reinterpret_cast<const float2 *>(sum64)[k * C1 + cc].y;
        lk[k] = (float)cnt[k] * (l / C1);                              // heads.py:32
    }
    __syncthreads();
    float ntot = 1e-6f, fg_loss = 0.f;
    for (int k = 1; k <= max_id; ++k) {                                // ascending, as the reference accumulates
        ntot += (float)cnt[k];
        fg_loss += lk[k];
    }
    const float total = fg_loss + bsum / C1;                           // n_b * mean over n_b * C1 elements
    if (tid == 0) loss_out[b] = 12.f * (total / ntot);
    if (!g) return;
    const float sc = 12.f / ntot * grad_scale;
    const float2 *vg = reinterpret_cast<const float2 *>(sum64);
    if (elem)
        for (int r0 = rg; r0 < R; r0 += G * UN) {
            float pv[UN], mv[UN], go[UN];
            uint32_t ids[UN];
#pragma unroll
            for (int i = 0; i < UN; ++i) {
                const int r = r0 + i * G;
                ids[i] = r < R ? rowids[r] : 0u;
                const bool need = r < R && ids[i] != 0u;
                pv[i] = need ? __ldg(p + (size_t)r * C1 + c) : 0.f;
                mv[i] = need ? __ldg(m + (size_t)r * C1 + c) : 0.f;
                go[i] = (accumulate && r < R) ? g[(size_t)r * C1 + c] : 0.f;
            }
#pragma unroll
            for (int i = 0; i < UN; ++i) {
                const int r = r0 + i * G;
                if (r >= R) continue;
                float gv = 0.f;
                for (uint32_t w = ids[i]; w; w >>= 8) {
                    const int id = w & 255;
                    if (id == bg) {
                        if (in_clamp(pv[i])) gv += dbce(clampf(pv[i]), mv[i] != 0.f ? 1.f : 0.f) / C1;
                    } else {
                        gv += vg[id * C1 + c].x;
                    }
                }
                g[(size_t)r * C1 + c] = go[i] + gv * sc;
            }
        }
}

}  // namespace

CIM_API int cim_pcl_loss_ex(const float *predict_cls, const float *mat, const int32_t *n_props, float *loss,
                            float *grad_cls, int n_img, int R, int C1, int max_id, float grad_scale, int accumulate,
                            cim_stream_t stream) {
    if (!predict_cls || !mat || !loss) return CIM_ERR_ARG;
    if (n_img < 0 || R <= 0 || C1 < 2 || max_id < 1) return CIM_ERR_ARG;
    if (n_img == 0) return CIM_OK;
    if (C1 > 128 || max_id > 255 || R > 16384) return CIM_ERR_SHAPE;
    if (!cim_aligned(n_props, 4)) return CIM_ERR_ALIGN;
    const size_t NI = (size_t)max_id + 1;
    const size_t smem = NI * C1 * 8 + NI * 4 + NI * 16 + NI * 4 + (size_t)R * 4 + 16;
    if ((int)smem + 8192 > cim_max_smem_optin()) return CIM_ERR_SHAPE;
    cudaFuncSetAttribute(cim_pcl_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cim_pcl_loss_kernel<<<(unsigned)n_img, PT, smem, (cudaStream_t)stream>>>(predict_cls, mat, loss, grad_cls, n_props, R,
                                                                            C1, max_id, grad_scale, accumulate);
    return cim_launch_status();
}

CIM_API int cim_pcl_loss(const float *predict_cls, const float *mat, float *loss, float *grad_cls, int n_img, int R,
                         int C1, int max_id, float grad_scale, int accumulate, cim_stream_t stream) {
    return cim_pcl_loss_ex(predict_cls, mat, nullptr, loss, grad_cls, n_img, R, C1, max_id, grad_scale, accumulate,
                           stream);
}
