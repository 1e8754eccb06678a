// score_heads.cu -- the CIM scoring heads for sm_100a.
//
// Replaces heads.cls_iou_model.forward (lib/modeling/heads.py:194-219 of the reference): there,
// 2 + 2K separate nn.Linear(4096 -> C+1) calls (tiny-N cuBLAS GEMMs) followed by 2 + 2K separate
// softmax / sigmoid launches.  Here: ONE fp32 GEMM  [n_img*R, D] x [D, (2+2K)*(C+1)]  that reads
// the features once, bias fused, then the activations in place:
//   head 0 (classifier), heads 2..2+K-1 (refine_cls): softmax over classes      (heads.py:200,212)
//   head 1 (detector): softmax over the PROPOSALS of each image, per class       (heads.py:203)
//   heads 2+K..2+2K-1 (refine_iou): sigmoid                                      (heads.py:216)
// fp32 FFMA accumulation (TF32 would miss the 1e-5 parity bar).
#include "common.cuh"
#include "ragged.cuh"

// score_heads_tc.cu: 3xTF32 tcgen05 + TMA path
bool cim_score_tc_eligible(long long M, int D, int C1, int n_ref);
size_t cim_score_tc_workspace_bytes(int D, int C1, int n_ref);
int cim_score_tc_launch(const float *x, const float *weight, const float *bias, float *scores, long long M, int D,
                        int C1, int n_ref, void *workspace, cudaStream_t st, const int32_t *row_map,
                        long long M_out);

namespace {

constexpr int BM = 128, BN = 64, BK = 16;
constexpr int APITCH = BM + 4, BPITCH = BN + 4;

// logits[h][m][c] = sum_k x[m][k] * w[h*C1 + c][k] + bias[h*C1 + c].  REMAP (compact ragged rows, ragged.cuh): row m
// goes to row row_map[m] of heads of M_out rows, nowhere for row_map[m] < 0.
template <bool REMAP>
__global__ void __launch_bounds__(256)
score_gemm_kernel(const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ bias,
                  float *__restrict__ out, int M, int N, int D, int C1, const int32_t *__restrict__ row_map,
                  int M_out) {
    __shared__ __align__(16) float As[BK][APITCH];
    __shared__ __align__(16) float Bs[BK][BPITCH];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const bool vec = (D & 3) == 0;
    for (int k0 = 0; k0 < D; k0 += BK) {
        // A tile: 128 rows x 16 k  (2 float4 per thread); B tile: 64 rows x 16 k (1 float4)
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            const int e = it * 256 + tid, row = e >> 2, k4 = (e & 3) * 4;
            const int m = m0 + row, k = k0 + k4;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (m < M) {
                if (vec && k + 3 < D) {
                    const float4 t = __ldg(reinterpret_cast<const float4 *>(x + (size_t)m * D + k));
                    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
                } else {
                    for (int i = 0; i < 4; ++i) if (k + i < D) v[i] = __ldg(x + (size_t)m * D + k + i);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) As[k4 + i][row] = v[i];
        }
        {
            const int row = tid >> 2, k4 = (tid & 3) * 4;
            const int n = n0 + row, k = k0 + k4;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (n < N) {
                if (vec && k + 3 < D) {
                    const float4 t = __ldg(reinterpret_cast<const float4 *>(w + (size_t)n * D + k));
                    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
                } else {
                    for (int i = 0; i < 4; ++i) if (k + i < D) v[i] = __ldg(w + (size_t)n * D + k + i);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) Bs[k4 + i][row] = v[i];
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8 + 4]);
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + ty * 8 + i;
        if (m >= M) continue;
        int out_row = m, out_rows = M;
        if constexpr (REMAP) {
            out_row = row_map[m];
            out_rows = M_out;
            if (out_row < 0) continue;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            const int h = n / C1, c = n - h * C1;
            out[((size_t)h * out_rows + out_row) * C1 + c] = acc[i][j] + __ldg(bias + n);
        }
    }
}

// softmax over classes / sigmoid, in place, one thread per (head, row); the detector head (1)
// is left as logits for the column pass below.  REMAP: M compact rows, whose rows in heads of M_out rows row_map gives.
template <bool REMAP>
__global__ void score_row_act_kernel(float *__restrict__ s, int M, int C1, int K, const int32_t *__restrict__ row_map,
                                     int M_out) {
    const int nheads = 2 + 2 * K;
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= (long long)nheads * M) return;
    const int h = (int)(idx / M);
    if (h == 1) return;
    float *row = s + (size_t)idx * C1;
    if constexpr (REMAP) {
        const int r = row_map[idx - (long long)h * M];
        if (r < 0) return;
        row = s + ((size_t)h * M_out + r) * C1;
    }
    if (h == 0 || h < 2 + K) {
        float mx = -INFINITY;
        for (int c = 0; c < C1; ++c) mx = fmaxf(mx, row[c]);
        float sum = 0.f;
        for (int c = 0; c < C1; ++c) sum += expf(row[c] - mx);
        for (int c = 0; c < C1; ++c) row[c] = expf(row[c] - mx) / sum;
    } else {
        for (int c = 0; c < C1; ++c) row[c] = 1.f / (1.f + expf(-row[c]));
    }
}

// detector head: softmax over the n proposals of one image for one class; block = (class, image).  n = n_props[img]
// clamped to [1, R] (R when n_props is NULL): the partial sums run over r < n in the order of a launch with R = n, and
// the block writes 0 into column c of every head for the padding rows r >= n.
__global__ void __launch_bounds__(256)
score_col_softmax_kernel(float *__restrict__ scores, const int32_t *__restrict__ n_props, long long M, int nheads,
                         int R, int C1) {
    __shared__ float red[8];
    __shared__ float bcast;
    const int c = blockIdx.x, img = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = n_props ? min(max(n_props[img], 1), R) : R;
    float *col = scores + ((size_t)M + (size_t)img * R) * C1 + c;
    float mx = -INFINITY;
    for (int r = tid; r < n; r += 256) mx = fmaxf(mx, col[(size_t)r * C1]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    if (tid == 0) {
        float m = red[0];
        for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
        bcast = m;
    }
    __syncthreads();
    mx = bcast;
    float sum = 0.f;
    for (int r = tid; r < n; r += 256) sum += expf(col[(size_t)r * C1] - mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    __syncthreads();
    if (lane == 0) red[warp] = sum;
    __syncthreads();
    if (tid == 0) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += red[i];
        bcast = t;
    }
    __syncthreads();
    sum = bcast;
    for (int r = tid; r < n; r += 256) col[(size_t)r * C1] = expf(col[(size_t)r * C1] - mx) / sum;
    for (int h = 0; h < nheads; ++h) {
        float *hc = scores + ((size_t)h * M + (size_t)img * R) * C1 + c;
        for (int r = n + tid; r < R; r += 256) hc[(size_t)r * C1] = 0.f;
    }
}

}  // namespace

CIM_API size_t cim_score_heads_workspace_bytes(int n_img, int R, int D, int C1, int K) {
    (void)n_img; (void)R;
    if (D <= 0 || C1 <= 0 || K < 0) return 256;
    return cim_score_tc_workspace_bytes(D, C1, K);          // W_hi / W_lo of the tensor-core path
}

// the FFMA / tensor-core GEMM + activations into padded scores [nheads, n_img*R, C1]: x has n_img*R rows, or with a
// row map (compact ragged rows) M = N rows
static int score_heads_run(const float *x, const float *weight, const float *bias, float *scores,
                           const int32_t *n_props, int n_img, int R, long long M, const int32_t *row_map, int D, int C1,
                           int K, void *workspace, size_t ws_bytes, size_t tc_ws_bytes, cudaStream_t st) {
    const int nheads = 2 + 2 * K, N = nheads * C1;
    const long long M_out = (long long)n_img * R;
    const dim3 col_grid((unsigned)C1, (unsigned)n_img);
    // tensor cores (3xTF32, fp32-accurate) when the shape allows and the caller gave the workspace;
    // CIM_DBG_SCORE_FFMA forces the FFMA kernel (tuning / A-B aid)
    if (!(cim_get_debug_flags() & CIM_DBG_SCORE_FFMA) && cim_score_tc_eligible(M, D, C1, K) && workspace &&
        ws_bytes >= tc_ws_bytes) {
        int rc2 = cim_score_tc_launch(x, weight, bias, scores, M, D, C1, K, workspace, st, row_map, M_out);
        if (rc2) return rc2;
        score_col_softmax_kernel<<<col_grid, 256, 0, st>>>(scores, n_props, M_out, nheads, R, C1);
        return cim_launch_status();
    }
    dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN));
    if (row_map) score_gemm_kernel<true><<<grid, 256, 0, st>>>(x, weight, bias, scores, (int)M, N, D, C1, row_map, (int)M_out);
    else score_gemm_kernel<false><<<grid, 256, 0, st>>>(x, weight, bias, scores, (int)M, N, D, C1, nullptr, 0);
    int rc = cim_launch_status();
    if (rc) return rc;
    const long long rows = (long long)nheads * M;
    if (row_map)
        score_row_act_kernel<true><<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(scores, (int)M, C1, K, row_map,
                                                                                   (int)M_out);
    else
        score_row_act_kernel<false><<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(scores, (int)M, C1, K, nullptr, 0);
    if ((rc = cim_launch_status())) return rc;
    score_col_softmax_kernel<<<col_grid, 256, 0, st>>>(scores, n_props, M_out, nheads, R, C1);
    return cim_launch_status();
}

CIM_API int cim_score_heads_ex(const float *x, const float *weight, const float *bias, float *scores,
                               const int32_t *n_props, int n_img, int R, int D, int C1, int K, void *workspace,
                               size_t ws_bytes, cim_stream_t stream) {
    if (!x || !weight || !bias || !scores) return CIM_ERR_ARG;
    if (n_img < 0 || R < 0 || D <= 0 || C1 <= 0 || K < 0 || K > 8) return CIM_ERR_ARG;
    if (n_img == 0 || R == 0) return CIM_OK;
    if (!cim_aligned(x, 16) || !cim_aligned(weight, 16) || !cim_aligned(n_props, 4)) return CIM_ERR_ALIGN;
    if (n_img > 65535 || C1 > 65535) return CIM_ERR_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const long long M = (long long)n_img * R;
    if (M > (1LL << 30)) return CIM_ERR_SHAPE;
    return score_heads_run(x, weight, bias, scores, n_props, n_img, R, M, nullptr, D, C1, K, workspace, ws_bytes,
                           cim_score_tc_workspace_bytes(D, C1, K), st);
}

// compact ragged rows: the tensor-core workspace, then the row map (ragged.cuh), each 256-byte aligned
static size_t tc_part_bytes(int D, int C1, int K) {
    return (cim_score_tc_workspace_bytes(D, C1, K) + 255) & ~(size_t)255;
}

CIM_API size_t cim_score_heads_compact_workspace_bytes(int n_img, int R, int N, int D, int C1, int K) {
    (void)R;
    if (n_img <= 0 || N <= 0 || D <= 0 || C1 <= 0 || K < 0) return 256;
    return 256 + tc_part_bytes(D, C1, K) + compact_map_bytes(n_img, N);
}

CIM_API int cim_score_heads_compact(const float *x, const float *weight, const float *bias, float *scores,
                                    const int32_t *n_props, int n_img, int R, int N, int D, int C1, int K,
                                    void *workspace, size_t ws_bytes, cim_stream_t stream) {
    if (!x || !weight || !bias || !scores || !workspace) return CIM_ERR_ARG;
    if (n_img <= 0 || R <= 0 || N <= 0 || D <= 0 || C1 <= 0 || K < 0 || K > 8) return CIM_ERR_ARG;
    if (!cim_aligned(x, 16) || !cim_aligned(weight, 16) || !cim_aligned(n_props, 4)) return CIM_ERR_ALIGN;
    if (n_img > 65535 || C1 > 65535) return CIM_ERR_SHAPE;
    if ((long long)n_img * R > (1LL << 30) || N > n_img * R) return CIM_ERR_SHAPE;
    if (ws_bytes < cim_score_heads_compact_workspace_bytes(n_img, R, N, D, C1, K)) return CIM_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char *base = reinterpret_cast<unsigned char *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    unsigned char *map_ws = base + tc_part_bytes(D, C1, K);
    int rc = compact_row_map_launch(n_props, n_img, R, N, map_ws, st);
    if (rc) return rc;
    // the tensor-core operands at `base` (cim_score_tc_launch aligns `workspace` the same way)
    return score_heads_run(x, weight, bias, scores, n_props, n_img, R, N, reinterpret_cast<const int32_t *>(map_ws),
                           D, C1, K, base, tc_part_bytes(D, C1, K), cim_score_tc_workspace_bytes(D, C1, K), st);
}

CIM_API int cim_score_heads(const float *x, const float *weight, const float *bias, float *scores, int n_img,
                            int R, int D, int C1, int K, void *workspace, size_t ws_bytes, cim_stream_t stream) {
    return cim_score_heads_ex(x, weight, bias, scores, nullptr, n_img, R, D, C1, K, workspace, ws_bytes, stream);
}
