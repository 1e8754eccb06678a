// score_heads_bwd.cu -- backward of the CIM scoring heads (autograd of heads.cls_iou_model.forward,
// lib/modeling/heads.py:194-219 of the reference) for sm_100a.
//
// With z = x W^T + b the [M, N] logits of all 2 + 2K heads (N = (2 + 2K)(C + 1)) and y the activations
// the forward stored, the upstream gradient g = dL/dy turns into
//     dz = y * (g - sum_c g y)          softmax over classes   (classifier, refine_cls)
//     dz = y * (g - sum_r g y)          softmax over the PROPOSALS of one image (detector, heads.py:203)
//     dz = g * y * (1 - y)              sigmoid                (refine_iou)
// and the three products
//     grad_x = dz W        [M, N] x [N, D]      -> score_dx_tc_kernel
//     grad_W = dz^T x      [N, M] x [M, D]      -> score_dw_tc_kernel  (split over M, partials summed in order)
//     grad_b = sum_m dz                         -> score_bias_grad_kernel
// are what the reference gets from eight nn.Linear backward calls (16 cuBLAS GEMMs with N = 21).
// grad_W / grad_b are the "head gradients" the data-parallel run all-reduces (SURVEY.md 8e).
//
// Both GEMMs run on the tensor cores as 3xTF32 (operands split into hi + lo TF32 numbers, three
// tcgen05.mma.kind::tf32 products, see score_heads_tc.cu) with the same short-chain discipline: a TMEM
// accumulator only ever sums <= 128 k, chunk sums are added in registers with round-to-nearest.
//   score_dx_tc_kernel: CTA = 128 rows of dz; loops over 128-column tiles of D.  A = dz_hi / dz_lo
//     [128 x 32], B = W^T_hi / W^T_lo [128 x 32], all four pre-split in the workspace and loaded by TMA
//     (SWIZZLE_128B); K = N is small (168 / 648), so the operands stream from L2.
//   score_dw_tc_kernel: CTA = (128 columns of D, one slice of M, 176 logit columns).  The A operand is
//     x^T: TMA brings the raw [32 m x 128 d] tile, four warps transpose + split it into the K-major
//     swizzled layout (x_hi, x_lo); B = dz^T_hi / dz^T_lo [176 x 32 m] by TMA.  D[128 d, 176 n] leaves
//     TMEM chunk by chunk into registers; the epilogue writes grad_W^T coalesced.
// Shapes the tensor path does not take (M < 128, D % 4 != 0, no TMA driver entry) run two plain fp32
// kernels (correctness path for tiny problems).
#include "common.cuh"
#include "ragged.cuh"
#include "score_tc.cuh"

namespace {

constexpr int BM = 128;
constexpr int BK = TC_BK;
constexpr int A_TILE = BM * BK * 4;                 // 16 KB
constexpr int THREADS_TC = 6 * 32;
constexpr uint32_t HI_MASK = 0xFFFFE000u;           // keeps the 10 mantissa bits TF32 has

__device__ __forceinline__ void split_tf32(float v, float &hi, float &lo) {
    hi = __uint_as_float(__float_as_uint(v) & HI_MASK);
    lo = v - hi;
}
__device__ __forceinline__ void commit_to(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ uint32_t tf32_idesc(int n) {       // F32 accumulate, TF32 x TF32, K-major, M = 128
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// ------------------------------------------------------------------------------- activations
// image row count n_props[img] clamped to [1, R]; R when n_props is NULL
__device__ __forceinline__ int image_rows(const int32_t *n_props, int img, int R) {
    return n_props ? min(max(n_props[img], 1), R) : R;
}

// detector head: dot[img][c] = sum_r g[r][c] * y[r][c] over the n proposals of one image (fixed order)
__global__ void __launch_bounds__(256)
score_det_dot_kernel(const float *__restrict__ g, const float *__restrict__ y, const int32_t *__restrict__ n_props,
                     float *__restrict__ dot, int R, int C1) {
    __shared__ float red[256];
    const int c = blockIdx.x, img = blockIdx.y, tid = threadIdx.x;
    const size_t base = (size_t)img * R * C1 + c;
    const int n = image_rows(n_props, img, R);
    float s = 0.f;
    for (int r = tid; r < n; r += 256) s = fmaf(g[base + (size_t)r * C1], y[base + (size_t)r * C1], s);
    red[tid] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) dot[img * C1 + c] = red[0];
}

// dz for 32 proposals x one head per warp (lane = proposal), written hi/lo-split as dz [M][NP] (row = proposal) and
// dz^T [N][MP].  The warp parks its 32 x C1 values in a private smem tile so that both layouts leave in contiguous
// runs: dz rows in C1-float runs, dz^T rows as 128 B (32 proposals) per class -- one thread per (head, row) writing
// its row with a 768-byte stride took 57 us at cfg2 for 43 MB.  Padding rows (r >= n of their image) get dz = 0
// whatever grad_scores holds there, so their grad_x rows and their share of grad_W / grad_b are 0.
// COMPACT (compact ragged rows, ragged.cuh): dz row m is read from y / g row row_map[m] of heads of M_in rows; a row
// with row_map[m] < 0 gets dz = 0 and reads nothing.
template <bool COMPACT>
__global__ void __launch_bounds__(256)
score_act_bwd_kernel(const float *__restrict__ y_all, const float *__restrict__ g_all,
                     const float *__restrict__ det_dot, const int32_t *__restrict__ n_props, float *__restrict__ dz_hi, float *__restrict__ dz_lo,
                     float *__restrict__ dzT_hi, float *__restrict__ dzT_lo, int M, int R, int C1, int K, int NP,
                     long long MP, const int32_t *__restrict__ row_map, int M_in) {
    extern __shared__ float act_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int pitch = C1 | 1;                                  // odd: lane = row reads / writes conflict-free
    float *tile = act_smem + (size_t)warp * 32 * pitch;
    const int nheads = 2 + 2 * K;
    const int m0 = blockIdx.x * 32;
    for (int h = warp; h < nheads; h += nw) {
        const int m = m0 + lane;
        if constexpr (COMPACT) {
            const int pm = m < M ? row_map[m] : -1;
            if (pm >= 0) {
                const size_t row = (size_t)h * M_in + pm;
                const float *y = y_all + row * C1, *g = g_all + row * C1;
                float dot = 0.f;
                const bool row_softmax = (h == 0) || (h >= 2 && h < 2 + K);
                if (row_softmax)
                    for (int c = 0; c < C1; ++c) dot = fmaf(g[c], y[c], dot);
                const float *ddot = det_dot + (size_t)(pm / R) * C1;
                for (int c = 0; c < C1; ++c) {
                    const float yy = y[c], gg = g[c];
                    float v;
                    if (row_softmax) v = yy * (gg - dot);
                    else if (h == 1) v = yy * (gg - ddot[c]);
                    else v = gg * yy * (1.f - yy);
                    tile[lane * pitch + c] = v;
                }
            } else if (m < M) {
                for (int c = 0; c < C1; ++c) tile[lane * pitch + c] = 0.f;
            }
        } else if (m < M) {
            const size_t row = (size_t)h * M + m;
            const float *y = y_all + row * C1, *g = g_all + row * C1;
            float dot = 0.f;
            const bool row_softmax = (h == 0) || (h >= 2 && h < 2 + K);
            if (row_softmax)
                for (int c = 0; c < C1; ++c) dot = fmaf(g[c], y[c], dot);
            const int img = m / R;
            const float *ddot = det_dot + (size_t)img * C1;
            const bool pad = m - img * R >= image_rows(n_props, img, R);
            for (int c = 0; c < C1; ++c) {
                const float yy = y[c], gg = g[c];
                float v;
                if (pad) v = 0.f;
                else if (row_softmax) v = yy * (gg - dot);
                else if (h == 1) v = yy * (gg - ddot[c]);
                else v = gg * yy * (1.f - yy);
                tile[lane * pitch + c] = v;
            }
        }
        __syncwarp();
        const int rows = min(32, M - m0);
        if (dz_hi) {
            for (int i = lane; i < rows * C1; i += 32) {
                const int r = i / C1, c = i - r * C1;
                float hi, lo;
                split_tf32(tile[r * pitch + c], hi, lo);
                const size_t o = (size_t)(m0 + r) * NP + h * C1 + c;
                dz_hi[o] = hi;
                dz_lo[o] = lo;
            }
        }
        if (dzT_hi && lane < rows) {
            for (int c = 0; c < C1; ++c) {
                float hi, lo;
                split_tf32(tile[lane * pitch + c], hi, lo);
                const size_t o = (size_t)(h * C1 + c) * MP + m0 + lane;
                dzT_hi[o] = hi;
                dzT_lo[o] = lo;
            }
        }
        __syncwarp();
    }
}

// grad_bias[n] = sum_m dz[m][n], read from dz^T (contiguous in m); fixed summation order
__global__ void __launch_bounds__(256)
score_bias_grad_kernel(const float *__restrict__ dzT_hi, const float *__restrict__ dzT_lo, float *__restrict__ gb,
                       int M, long long MP) {
    __shared__ float red[256];
    const int n = blockIdx.x, tid = threadIdx.x;
    const float *h = dzT_hi + (size_t)n * MP, *l = dzT_lo + (size_t)n * MP;
    float s = 0.f;
    for (int m = tid; m < M; m += 256) s += h[m] + l[m];
    red[tid] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) gb[n] = red[0];
}

// W [N][D] -> W^T_hi / W^T_lo [D][NP]
__global__ void __launch_bounds__(256)
score_wT_split_kernel(const float *__restrict__ w, float *__restrict__ wT_hi, float *__restrict__ wT_lo, int N, int D,
                      int NP) {
    __shared__ float tile[32][33];
    const int d0 = blockIdx.x * 32, n0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int i = ty; i < 32; i += 8) {
        const int n = n0 + i, d = d0 + tx;
        tile[i][tx] = (n < N && d < D) ? w[(size_t)n * D + d] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int d = d0 + i, n = n0 + tx;
        if (d < D && n < N) {
            float hi, lo;
            split_tf32(tile[tx][i], hi, lo);
            wT_hi[(size_t)d * NP + n] = hi;
            wT_lo[(size_t)d * NP + n] = lo;
        }
    }
}

// ------------------------------------------------------------------------------- grad_x = dz W
constexpr int DX_BN = 128;                            // columns of D per accumulator tile (UMMA N)
constexpr int DX_B_TILE = DX_BN * BK * 4;             // 16 KB
constexpr int DX_STAGE = 2 * A_TILE + 2 * DX_B_TILE;  // dz_hi | dz_lo | W^T_hi | W^T_lo = 64 KB
constexpr int DX_NSTAGE = 3;
constexpr int DX_CH = 3;                              // k-blocks per accumulation chunk (K = 96)

__global__ void __launch_bounds__(THREADS_TC, 1)
score_dx_tc_kernel(const __grid_constant__ CUtensorMap tm_dzh, const __grid_constant__ CUtensorMap tm_dzl,
                   const __grid_constant__ CUtensorMap tm_wth, const __grid_constant__ CUtensorMap tm_wtl,
                   float *__restrict__ grad_x, int M, int D, int nkb) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)DX_NSTAGE * DX_STAGE);
    uint64_t *empty = full + DX_NSTAGE;
    uint64_t *chunk_full = empty + DX_NSTAGE;
    uint64_t *chunk_empty = chunk_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(chunk_empty + 2);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = blockIdx.x * BM;
    const int ntiles = (D + DX_BN - 1) / DX_BN;
    const int nchunks = (nkb + DX_CH - 1) / DX_CH;

    if (tid == 0) {
        for (int s = 0; s < DX_NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int p = 0; p < 2; ++p) { mbar_init(&chunk_full[p], 1); mbar_init(&chunk_empty[p], 4); }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(256u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;            // accumulator p at columns 128 p
    const uint32_t idesc = tf32_idesc(DX_BN);

    if (warp == 0) {
        if (elect_one()) {
            int it = 0;
            for (int nt = 0; nt < ntiles; ++nt)
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % DX_NSTAGE;
                    if (it >= DX_NSTAGE) mbar_wait(&empty[s], ((it / DX_NSTAGE) - 1) & 1);
                    unsigned char *st = smem + (size_t)s * DX_STAGE;
                    mbar_expect_tx(&full[s], (uint32_t)DX_STAGE);
                    tma_load_2d(st, &tm_dzh, kb * BK, m0, &full[s]);
                    tma_load_2d(st + A_TILE, &tm_dzl, kb * BK, m0, &full[s]);
                    tma_load_2d(st + 2 * A_TILE, &tm_wth, kb * BK, nt * DX_BN, &full[s]);
                    tma_load_2d(st + 2 * A_TILE + DX_B_TILE, &tm_wtl, kb * BK, nt * DX_BN, &full[s]);
                }
        }
    } else if (warp == 1) {
        if (elect_one()) {                            // one elected thread runs the whole issue loop (common.cuh)
            int it = 0, g = 0;                        // g: running chunk index, accumulator g & 1
            for (int nt = 0; nt < ntiles; ++nt)
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % DX_NSTAGE, p = g & 1;
                    const bool first = (kb % DX_CH) == 0, last = (kb % DX_CH) == DX_CH - 1 || kb == nkb - 1;
                    if (first && g >= 2) mbar_wait(&chunk_empty[p], ((g >> 1) - 1) & 1);
                    mbar_wait(&full[s], (it / DX_NSTAGE) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t base = smem_u32(smem + (size_t)s * DX_STAGE), acc = tmem_base + (uint32_t)DX_BN * p;
                    const uint64_t ah = smem_desc128(base), al = smem_desc128(base + A_TILE);
                    const uint64_t bh = smem_desc128(base + 2 * A_TILE), bl = smem_desc128(base + 2 * A_TILE + DX_B_TILE);
#pragma unroll
                    for (int k = 0; k < BK / 8; ++k) {
                        mma_tf32(acc, ah + 2 * k, bh + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
                        mma_tf32(acc, ah + 2 * k, bl + 2 * k, idesc, 1u);
                        mma_tf32(acc, al + 2 * k, bh + 2 * k, idesc, 1u);
                    }
                    commit_to(&empty[s]);
                    if (last) { commit_to(&chunk_full[p]); ++g; }
                }
        }
        __syncwarp();
    } else {
        const int q4 = warp & 3;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q4) << 16);
        const int m = m0 + 32 * q4 + lane;
        int g = 0;
        for (int nt = 0; nt < ntiles; ++nt) {
            float acc[DX_BN];
#pragma unroll
            for (int j = 0; j < DX_BN; ++j) acc[j] = 0.f;
            for (int c = 0; c < nchunks; ++c, ++g) {
                const int p = g & 1;
                mbar_wait(&chunk_full[p], (g >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int cc = 0; cc < DX_BN / 32; ++cc) {
                    float v[32];
                    tmem_ld32(lane_addr + (uint32_t)DX_BN * p + 32u * cc, v);
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[cc * 32 + j] += v[j];
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive1(&chunk_empty[p]);
            }
            if (m < M) {
                float *dst = grad_x + (size_t)m * D + (size_t)nt * DX_BN;
                const int left = D - nt * DX_BN;                     // D % 4 == 0
#pragma unroll
                for (int j = 0; j < DX_BN; j += 4)
                    if (j < left) *reinterpret_cast<float4 *>(dst + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
    }
}

// ------------------------------------------------------------------------------- grad_W = dz^T x
constexpr int DW_NT = 176;                            // logit columns per CTA (UMMA N), 8 x 21 = 168 for VOC
constexpr int DW_B_TILE = DW_NT * BK * 4;             // 22 KB
constexpr int DW_RAW = 32 * BM * 4;                   // raw x tile [32 m][128 d], 16 KB
constexpr int DW_STAGE = 2 * A_TILE + 2 * DW_B_TILE;     // x^T_hi | x^T_lo | dz^T_hi | dz^T_lo = 76 KB
constexpr int DW_NSTAGE = 2;
constexpr int DW_NRAW = 4;                            // raw x tiles in flight ahead of the transpose (HBM latency)
constexpr int DW_THREADS = 7 * 32;                    // x producer, MMA issuer, 4 transpose/epilogue warps, dz^T producer
constexpr int DW_CHK = 4;                             // k-blocks per accumulation chunk (128 proposals)
constexpr int DW_LAG = 2;

__global__ void __launch_bounds__(DW_THREADS, 1)
score_dw_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_bh,
                   const __grid_constant__ CUtensorMap tm_bl, float *__restrict__ partial, int M, int N, int D,
                   int kb_per_split) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char *rawring = smem + (size_t)DW_NSTAGE * DW_STAGE;                     // [DW_NRAW][DW_RAW]
    uint64_t *tma_full = reinterpret_cast<uint64_t *>(rawring + (size_t)DW_NRAW * DW_RAW);   // [NSTAGE] dz^T tiles landed
    uint64_t *raw_full = tma_full + DW_NSTAGE;                   // [DW_NRAW] raw x tile landed
    uint64_t *raw_empty = raw_full + DW_NRAW;                    // [DW_NRAW] raw x tile read by the 4 transpose warps
    uint64_t *lo_ready = raw_empty + DW_NRAW;
    uint64_t *empty = lo_ready + DW_NSTAGE;
    uint64_t *chunk_full = empty + DW_NSTAGE;
    uint64_t *chunk_empty = chunk_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(chunk_empty + 2);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d0 = blockIdx.x * BM, n0 = blockIdx.z * DW_NT;
    const int nkb_total = (M + BK - 1) / BK;
    const int kb0 = blockIdx.y * kb_per_split;
    const int nkb = min(kb_per_split, nkb_total - kb0);          // >= 1 by construction of the grid
    const int nchunks = (nkb + DW_CHK - 1) / DW_CHK;

    if (tid == 0) {
        for (int s = 0; s < DW_NSTAGE; ++s) { mbar_init(&tma_full[s], 1); mbar_init(&lo_ready[s], 4); mbar_init(&empty[s], 1); }
        for (int p = 0; p < 2; ++p) { mbar_init(&chunk_full[p], 1); mbar_init(&chunk_empty[p], 4); }
        for (int r = 0; r < DW_NRAW; ++r) { mbar_init(&raw_full[r], 1); mbar_init(&raw_empty[r], 4); }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;                       // accumulator p at columns 256 p
    const uint32_t idesc = tf32_idesc(DW_NT);

    if (warp == 0) {
        if (elect_one()) {                                 // x producer: the HBM stream, DW_NRAW tiles ahead
            for (int kb = 0; kb < nkb; ++kb) {
                const int r = kb % DW_NRAW;
                if (kb >= DW_NRAW) mbar_wait(&raw_empty[r], ((kb / DW_NRAW) - 1) & 1);
                mbar_expect_tx(&raw_full[r], (uint32_t)DW_RAW);
                tma_load_2d(rawring + (size_t)r * DW_RAW, &tm_x, d0, (kb0 + kb) * BK, &raw_full[r]);   // [32 m][128 d]
            }
        }
    } else if (warp == 6) {
        if (elect_one()) {                                 // dz^T producer (L2 hits), tied to the MMA stage
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % DW_NSTAGE;
                if (kb >= DW_NSTAGE) mbar_wait(&empty[s], ((kb / DW_NSTAGE) - 1) & 1);
                unsigned char *st = smem + (size_t)s * DW_STAGE;
                mbar_expect_tx(&tma_full[s], (uint32_t)(2 * DW_B_TILE));
                tma_load_2d(st + 2 * A_TILE, &tm_bh, (kb0 + kb) * BK, n0, &tma_full[s]);
                tma_load_2d(st + 2 * A_TILE + DW_B_TILE, &tm_bl, (kb0 + kb) * BK, n0, &tma_full[s]);
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {                                 // one elected thread runs the whole issue loop
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % DW_NSTAGE, c = kb / DW_CHK, p = c & 1;
                if (kb % DW_CHK == 0 && c >= 2) mbar_wait(&chunk_empty[p], ((c >> 1) - 1) & 1);
                mbar_wait(&tma_full[s], (kb / DW_NSTAGE) & 1);
                mbar_wait(&lo_ready[s], (kb / DW_NSTAGE) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t base = smem_u32(smem + (size_t)s * DW_STAGE), acc = tmem_base + 256u * p;
                const uint64_t ah = smem_desc128(base), al = smem_desc128(base + A_TILE);
                const uint64_t bh = smem_desc128(base + 2 * A_TILE), bl = smem_desc128(base + 2 * A_TILE + DW_B_TILE);
#pragma unroll
                for (int k = 0; k < BK / 8; ++k) {
                    mma_tf32(acc, ah + 2 * k, bh + 2 * k, idesc, ((kb % DW_CHK) | k) != 0);
                    mma_tf32(acc, ah + 2 * k, bl + 2 * k, idesc, 1u);
                    mma_tf32(acc, al + 2 * k, bh + 2 * k, idesc, 1u);
                }
                commit_to(&empty[s]);
                if (kb % DW_CHK == DW_CHK - 1 || kb == nkb - 1) commit_to(&chunk_full[p]);
            }
        }
        __syncwarp();
    } else {
        // transpose + split warps: thread t owns column d0 + t of x = row t of the A operand
        const int t = tid - 64;
        const uint32_t row_off = (t >> 3) * 1024 + (t & 7) * 128, sw = t & 7;
        const int q4 = warp & 3;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q4) << 16);
        float acc[DW_NT];
#pragma unroll
        for (int j = 0; j < DW_NT; ++j) acc[j] = 0.f;
        auto drain = [&](int c) {
            const int p = c & 1;
            mbar_wait(&chunk_full[p], (c >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int cc = 0; cc < DW_NT / 32; ++cc) {
                float v[32];
                tmem_ld32(lane_addr + 256u * p + 32u * cc, v);
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[cc * 32 + j] += v[j];
            }
            if (DW_NT % 32) {
                float v[16];
                tmem_ld16(lane_addr + 256u * p + (uint32_t)(DW_NT / 32 * 32), v);
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[DW_NT / 32 * 32 + j] += v[j];
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive1(&chunk_empty[p]);
        };
        int next_drain = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % DW_NSTAGE, r = kb % DW_NRAW;
            mbar_wait(&raw_full[r], (kb / DW_NRAW) & 1);
            if (kb >= DW_NSTAGE) mbar_wait(&empty[s], ((kb / DW_NSTAGE) - 1) & 1);     // the stage's last MMAs are done
            unsigned char *st = smem + (size_t)s * DW_STAGE;
            const float *raw = reinterpret_cast<const float *>(rawring + (size_t)r * DW_RAW) + t;      // raw[mm * 128]
            unsigned char *xh = st + row_off, *xl = xh + A_TILE;
#pragma unroll
            for (int c = 0; c < 8; ++c) {                    // 4 proposals per 16 B chunk of the operand row
                float h[4], l[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) split_tf32(raw[(4 * c + i) * BM], h[i], l[i]);
                const uint32_t o = (uint32_t)((c ^ sw) << 4);
                *reinterpret_cast<float4 *>(xh + o) = make_float4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<float4 *>(xl + o) = make_float4(l[0], l[1], l[2], l[3]);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) { mbar_arrive1(&lo_ready[s]); mbar_arrive1(&raw_empty[r]); }
            while (next_drain < nchunks && min((next_drain + 1) * DW_CHK, nkb) - 1 + DW_LAG <= kb) drain(next_drain++);
        }
        while (next_drain < nchunks) drain(next_drain++);

        const int d = d0 + 32 * q4 + lane;
        if (d < D) {
            float *dst = partial + ((size_t)blockIdx.y * N + n0) * D + d;
            const int nn = min(DW_NT, N - n0);
#pragma unroll
            for (int j = 0; j < DW_NT; ++j)
                if (j < nn) dst[(size_t)j * D] = acc[j];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// grad_W = sum of the split partials, in split order
__global__ void score_dw_reduce_kernel(const float *__restrict__ partial, float *__restrict__ gw, long long n, int S) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float s = partial[i];
        for (int k = 1; k < S; ++k) s += partial[(size_t)k * n + i];
        gw[i] = s;
    }
}

// ------------------------------------------------------------------------------- plain fp32 kernels
__global__ void score_dx_plain_kernel(const float *__restrict__ dz_hi, const float *__restrict__ dz_lo,
                                      const float *__restrict__ w, float *__restrict__ gx, int M, int N, int D, int NP) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= (long long)M * D) return;
    const int m = (int)(idx / D), d = (int)(idx - (long long)m * D);
    float s = 0.f;
    for (int n = 0; n < N; ++n) s = fmaf(dz_hi[(size_t)m * NP + n] + dz_lo[(size_t)m * NP + n], w[(size_t)n * D + d], s);
    gx[idx] = s;
}
__global__ void score_dw_plain_kernel(const float *__restrict__ dzT_hi, const float *__restrict__ dzT_lo,
                                      const float *__restrict__ x, float *__restrict__ gw, int M, int N, int D,
                                      long long MP) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= (long long)N * D) return;
    const int n = (int)(idx / D), d = (int)(idx - (long long)n * D);
    float s = 0.f;
    for (int m = 0; m < M; ++m) s = fmaf(dzT_hi[(size_t)n * MP + m] + dzT_lo[(size_t)n * MP + m], x[(size_t)m * D + d], s);
    gw[idx] = s;
}

struct BwdLayout {
    int N, NP, S, dtiles, ntiles;
    long long M, MP;
    size_t off_dot, off_dzh, off_dzl, off_dth, off_dtl, off_wth, off_wtl, off_part, total;
};
inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }
// M rows of x and dz: n_img * R, or N with compact ragged rows (their row map then follows at `total`)
BwdLayout bwd_layout(int n_img, long long M, int D, int C1, int K) {
    BwdLayout L;
    L.M = M;
    L.N = (2 + 2 * K) * C1;
    L.NP = (L.N + 31) & ~31;
    L.MP = (L.M + 31) & ~31LL;
    L.dtiles = (D + BM - 1) / BM;
    L.ntiles = (L.N + DW_NT - 1) / DW_NT;
    const int nkb_total = (int)((L.M + BK - 1) / BK);
    int S = cim_num_sms() / (L.dtiles * L.ntiles);
    S = S < 1 ? 1 : (S > 8 ? 8 : S);
    if (S > nkb_total) S = nkb_total > 0 ? nkb_total : 1;
    L.S = S;
    size_t o = 256;                                    // slack to align the base
    L.off_dot = o; o += up256(sizeof(float) * (size_t)n_img * C1);
    L.off_dzh = o; o += up256(sizeof(float) * (size_t)L.M * L.NP);
    L.off_dzl = o; o += up256(sizeof(float) * (size_t)L.M * L.NP);
    L.off_dth = o; o += up256(sizeof(float) * (size_t)L.N * L.MP);
    L.off_dtl = o; o += up256(sizeof(float) * (size_t)L.N * L.MP);
    L.off_wth = o; o += up256(sizeof(float) * (size_t)D * L.NP);
    L.off_wtl = o; o += up256(sizeof(float) * (size_t)D * L.NP);
    L.off_part = o; o += up256(sizeof(float) * (size_t)L.S * L.N * D);
    L.total = o;
    return L;
}

}  // namespace

CIM_API size_t cim_score_heads_bwd_workspace_bytes(int n_img, int R, int D, int C1, int K) {
    if (n_img <= 0 || R <= 0 || D <= 0 || C1 <= 0 || K < 0) return 256;
    return bwd_layout(n_img, (long long)n_img * R, D, C1, K).total;
}

// everything after the argument checks: scores / grad_scores padded (heads of n_img * R rows), x / grad_x / dz of L.M
// rows; row_map (compact ragged rows) maps dz row m to its padded row, NULL when L.M = n_img * R rows are padded rows
static int score_heads_bwd_run(const float *x, const float *weight, const float *scores, const float *grad_scores,
                               const int32_t *n_props, const int32_t *row_map, float *grad_x, float *grad_weight,
                               float *grad_bias, int n_img, int R, int D, int C1, int K, const BwdLayout &L,
                               unsigned char *ws, cudaStream_t st) {
    const int nheads = 2 + 2 * K;
    auto F = [&](size_t off) { return reinterpret_cast<float *>(ws + off - 256); };
    float *dot = F(L.off_dot), *dzh = F(L.off_dzh), *dzl = F(L.off_dzl), *dth = F(L.off_dth), *dtl = F(L.off_dtl);
    float *wth = F(L.off_wth), *wtl = F(L.off_wtl), *part = F(L.off_part);
    const int M = (int)L.M, N = L.N, M_in = n_img * R;
    const bool want_t = grad_weight || grad_bias;

    score_det_dot_kernel<<<dim3((unsigned)C1, (unsigned)n_img), 256, 0, st>>>(grad_scores + (size_t)M_in * C1,
                                                                             scores + (size_t)M_in * C1, n_props, dot, R, C1);
    int rc = cim_launch_status();
    if (rc) return rc;
    const long long rows = (long long)nheads * M;
    int act_warps = 8;                                           // one head per warp, 32 proposals per CTA
    while (act_warps > 1 && (size_t)act_warps * 32 * (C1 | 1) * sizeof(float) > 96 * 1024) act_warps >>= 1;
    const size_t act_smem = (size_t)act_warps * 32 * (C1 | 1) * sizeof(float);
    if (act_smem > (size_t)cim_max_smem_optin()) return CIM_ERR_SHAPE;         // C1 > ~1700
    if (row_map) {
        if (act_smem > 48 * 1024)
            cudaFuncSetAttribute(score_act_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)act_smem);
        score_act_bwd_kernel<true><<<(unsigned)((M + 31) / 32), act_warps * 32, act_smem, st>>>(
            scores, grad_scores, dot, n_props, grad_x ? dzh : nullptr, dzl, want_t ? dth : nullptr, dtl, M, R, C1, K,
            L.NP, L.MP, row_map, M_in);
    } else {
        if (act_smem > 48 * 1024)
            cudaFuncSetAttribute(score_act_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)act_smem);
        score_act_bwd_kernel<false><<<(unsigned)((M + 31) / 32), act_warps * 32, act_smem, st>>>(
            scores, grad_scores, dot, n_props, grad_x ? dzh : nullptr, dzl, want_t ? dth : nullptr, dtl, M, R, C1, K,
            L.NP, L.MP, nullptr, 0);
    }
    if ((rc = cim_launch_status())) return rc;
    if (grad_bias) {
        score_bias_grad_kernel<<<(unsigned)N, 256, 0, st>>>(dth, dtl, grad_bias, M, L.MP);
        if ((rc = cim_launch_status())) return rc;
    }
    const bool tc = !(cim_get_debug_flags() & CIM_DBG_SCORE_FFMA) && M >= BM && (D % 4) == 0 && D >= BK && encode_tiled() != nullptr &&
                    (size_t)cim_max_smem_optin() >= 1024 + (size_t)DW_NSTAGE * DW_STAGE + (size_t)DW_NRAW * DW_RAW + 256;
    if (grad_x) {
        if (tc) {
            score_wT_split_kernel<<<dim3((unsigned)((D + 31) / 32), (unsigned)((N + 31) / 32)), 256, 0, st>>>(
                weight, wth, wtl, N, D, L.NP);
            if ((rc = cim_launch_status())) return rc;
            CUtensorMap ta, tb, tc_, td;
            if (!make_map_ex(&ta, dzh, M, N, L.NP, BM, BK, true) || !make_map_ex(&tb, dzl, M, N, L.NP, BM, BK, true) ||
                !make_map_ex(&tc_, wth, D, N, L.NP, DX_BN, BK, true) || !make_map_ex(&td, wtl, D, N, L.NP, DX_BN, BK, true))
                return CIM_ERR_ARG;
            const size_t smem = 1024 + (size_t)DX_NSTAGE * DX_STAGE + 256;
            cudaFuncSetAttribute(score_dx_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            score_dx_tc_kernel<<<(unsigned)((M + BM - 1) / BM), THREADS_TC, smem, st>>>(ta, tb, tc_, td, grad_x, M, D,
                                                                                         (N + BK - 1) / BK);
        } else {
            const long long n = (long long)M * D;
            score_dx_plain_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dzh, dzl, weight, grad_x, M, N, D, L.NP);
        }
        if ((rc = cim_launch_status())) return rc;
    }
    if (grad_weight) {
        if (tc) {
            const int nkb_total = (M + BK - 1) / BK;
            const int per = (nkb_total + L.S - 1) / L.S, S = (nkb_total + per - 1) / per;
            CUtensorMap tx, tb, tl;
            if (!make_map_ex(&tx, x, M, D, D, 32, BM, false) || !make_map_ex(&tb, dth, N, M, L.MP, DW_NT, BK, true) ||
                !make_map_ex(&tl, dtl, N, M, L.MP, DW_NT, BK, true))
                return CIM_ERR_ARG;
            const size_t smem = 1024 + (size_t)DW_NSTAGE * DW_STAGE + (size_t)DW_NRAW * DW_RAW + 256;
            cudaFuncSetAttribute(score_dw_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            float *out = S == 1 ? grad_weight : part;
            score_dw_tc_kernel<<<dim3((unsigned)L.dtiles, (unsigned)S, (unsigned)L.ntiles), DW_THREADS, smem, st>>>(
                tx, tb, tl, out, M, N, D, per);
            if ((rc = cim_launch_status())) return rc;
            if (S > 1) score_dw_reduce_kernel<<<592, 256, 0, st>>>(part, grad_weight, (long long)N * D, S);
        } else {
            const long long n = (long long)N * D;
            score_dw_plain_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dth, dtl, x, grad_weight, M, N, D, L.MP);
        }
        if ((rc = cim_launch_status())) return rc;
    }
    return CIM_OK;
}

// the checks both entry points make; rows = n_img * R (padded) or N (compact)
static int score_heads_bwd_args(const float *x, const float *weight, const float *scores, const float *grad_scores,
                                const int32_t *n_props, const float *grad_x, int n_img, int R, int D, int C1, int K,
                                const void *workspace) {
    if (!x || !weight || !scores || !grad_scores || !workspace) return CIM_ERR_ARG;
    if (n_img < 0 || R < 0 || D <= 0 || C1 <= 0 || K < 0 || K > 8) return CIM_ERR_ARG;
    if (n_img > 65535 || C1 > 65535) return CIM_ERR_SHAPE;
    if ((long long)n_img * R > (1LL << 30)) return CIM_ERR_SHAPE;
    if (!cim_aligned(x, 16) || !cim_aligned(weight, 16) || (grad_x && !cim_aligned(grad_x, 16)) ||
        !cim_aligned(n_props, 4))
        return CIM_ERR_ALIGN;
    return CIM_OK;
}

CIM_API int cim_score_heads_bwd_ex(const float *x, const float *weight, const float *scores, const float *grad_scores,
                                   const int32_t *n_props, float *grad_x, float *grad_weight, float *grad_bias,
                                   int n_img, int R, int D, int C1, int K, void *workspace, size_t ws_bytes,
                                   cim_stream_t stream) {
    if (!x || !weight || !scores || !grad_scores || !workspace) return CIM_ERR_ARG;
    if (n_img < 0 || R < 0 || D <= 0 || C1 <= 0 || K < 0 || K > 8) return CIM_ERR_ARG;
    if (!grad_x && !grad_weight && !grad_bias) return CIM_OK;
    if (n_img > 65535 || C1 > 65535) return CIM_ERR_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const int nheads = 2 + 2 * K;
    if (n_img == 0 || R == 0) {                        // no proposals: the parameter gradients are zero
        if (grad_weight) cudaMemsetAsync(grad_weight, 0, sizeof(float) * (size_t)nheads * C1 * D, st);
        if (grad_bias) cudaMemsetAsync(grad_bias, 0, sizeof(float) * (size_t)nheads * C1, st);
        return cim_launch_status();
    }
    const BwdLayout L = bwd_layout(n_img, (long long)n_img * R, D, C1, K);
    if (L.M > (1LL << 30)) return CIM_ERR_SHAPE;
    if (ws_bytes < L.total) return CIM_ERR_WORKSPACE;
    int rc = score_heads_bwd_args(x, weight, scores, grad_scores, n_props, grad_x, n_img, R, D, C1, K, workspace);
    if (rc) return rc;
    unsigned char *ws = reinterpret_cast<unsigned char *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    return score_heads_bwd_run(x, weight, scores, grad_scores, n_props, nullptr, grad_x, grad_weight, grad_bias, n_img,
                               R, D, C1, K, L, ws, st);
}

CIM_API size_t cim_score_heads_bwd_compact_workspace_bytes(int n_img, int R, int N, int D, int C1, int K) {
    (void)R;
    if (n_img <= 0 || N <= 0 || D <= 0 || C1 <= 0 || K < 0) return 256;
    return bwd_layout(n_img, N, D, C1, K).total + compact_map_bytes(n_img, N);
}

CIM_API int cim_score_heads_bwd_compact(const float *x, const float *weight, const float *scores,
                                        const float *grad_scores, const int32_t *n_props, float *grad_x,
                                        float *grad_weight, float *grad_bias, int n_img, int R, int N, int D, int C1,
                                        int K, void *workspace, size_t ws_bytes, cim_stream_t stream) {
    int rc = score_heads_bwd_args(x, weight, scores, grad_scores, n_props, grad_x, n_img, R, D, C1, K, workspace);
    if (rc) return rc;
    if (n_img <= 0 || R <= 0 || N <= 0) return CIM_ERR_ARG;
    if (N > n_img * R) return CIM_ERR_SHAPE;
    if (!grad_x && !grad_weight && !grad_bias) return CIM_OK;
    if (ws_bytes < cim_score_heads_bwd_compact_workspace_bytes(n_img, R, N, D, C1, K)) return CIM_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const BwdLayout L = bwd_layout(n_img, N, D, C1, K);
    unsigned char *ws = reinterpret_cast<unsigned char *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    unsigned char *map_ws = ws + L.total - 256;                  // offsets in the layout count the 256 B of slack
    if ((rc = compact_row_map_launch(n_props, n_img, R, N, map_ws, st))) return rc;
    return score_heads_bwd_run(x, weight, scores, grad_scores, n_props, reinterpret_cast<const int32_t *>(map_ws),
                               grad_x, grad_weight, grad_bias, n_img, R, D, C1, K, L, ws, st);
}

CIM_API int cim_score_heads_bwd(const float *x, const float *weight, const float *scores, const float *grad_scores,
                                float *grad_x, float *grad_weight, float *grad_bias, int n_img, int R, int D, int C1,
                                int K, void *workspace, size_t ws_bytes, cim_stream_t stream) {
    return cim_score_heads_bwd_ex(x, weight, scores, grad_scores, nullptr, grad_x, grad_weight, grad_bias, n_img, R, D,
                                  C1, K, workspace, ws_bytes, stream);
}
