// score_heads_tc.cu -- the scoring GEMM of cls_iou_model on the 5th-gen tensor cores (sm_100a).
//
// logits[m][n] = sum_k x[m][k] * W[n][k] + b[n]  with  M = n_img * R (16000), K = 4096 and
// N = (2 + 2K_ref) * (C + 1) = 168 (VOC): 22 GFLOP per step that the fp32 FFMA kernel
// (score_heads.cu) needs 0.83 ms for.  Parity demands fp32-like accuracy (1e-5 relative), which a
// plain TF32 GEMM misses, so every operand is split into two TF32 numbers
//     x = x_hi + x_lo,  x_hi = x with the low 13 mantissa bits cleared,  x_lo = x - x_hi (exact)
// and   x * w  ~=  x_hi w_hi + x_hi w_lo + x_lo w_hi      (the dropped x_lo w_lo term is ~2^-22),
// three tcgen05.mma.kind::tf32 products accumulated in fp32 in tensor memory.
//
// The tensor core's fp32 accumulator TRUNCATES on every add (measured: the error of a single long
// chain grows linearly with K, 4.5e-6 at K = 128 -> 9e-5 at K = 4096, tools/score_err.py), so
// chains are kept short: K is cut into chunks of 128, each chunk accumulates from zero in one of
// two TMEM accumulators, and the chunk sums are added in registers with round-to-nearest while
// the next chunk is being multiplied.
//
// One CTA per 128 rows of x and per group of heads (all 8 heads at once when 8 (C+1) <= 256).
//   warp 0      x producer: cp.async.bulk.tensor (SWIZZLE_128B) of the raw x tile [128 x 32 fp32] into a ring of
//               NRAW buffers that runs ahead of everything else -- x comes from HBM (the 262 MB stream that
//               bounds the kernel), its latency must not sit inside the 2-stage MMA ring.
//   warp 6      W producer: the W_hi / W_lo tiles [NT x 32] of a k-block (L2 hits) into the MMA stage, as soon as
//               the MMAs that read the stage before have completed.
//   warps 2..5  split: read the raw x tile, write x_hi and x_lo into the MMA stage (generic proxy ->
//               fence.proxy.async); later the epilogue (TMEM lane quarter = warp % 4).
//   warp 1      MMA issuer: 3 products x 4 k-steps per k-block, tcgen05.commit frees the stage.
// Epilogue: tcgen05.ld per head, bias, softmax over classes / sigmoid in registers, one contiguous
// store per (head, row).  The detector head keeps its logits (softmax over the proposals of an
// image runs in score_col_softmax_kernel).
#include "common.cuh"
#include "score_tc.cuh"

namespace {

constexpr int BM = 128;                  // rows of x per CTA (UMMA M)
constexpr int BK = 32;                   // fp32 elements per k-block = 128 B = one SW128 atom row
constexpr int NSTAGE = 2;
constexpr int A_TILE = BM * BK * 4;      // 16 KB
constexpr int THREADS_TC = 7 * 32;
constexpr int NRAW = 4;                  // raw x tiles in flight ahead of the split (HBM latency)
constexpr int NT = 176;                  // UMMA N = logit columns per CTA (8 heads x 21 = 168 for VOC)
constexpr int W_TILE = NT * BK * 4;      // 22 KB
constexpr int STAGE = 2 * A_TILE + 2 * W_TILE;            // x_hi | x_lo | W_hi | W_lo
constexpr int CHK = 4;                   // k-blocks per accumulation chunk (K = 128)
constexpr int LAG = 2;                   // a chunk is drained this many k-blocks after its last split
constexpr int ZP = NT + 1;               // float pitch of the epilogue staging (odd: lanes = rows)

// W -> (W_hi, W_lo), both exactly representable... W_hi in TF32, W_lo = W - W_hi (the MMA drops its
// low mantissa bits, an error of 2^-21 |W|)
__global__ void score_split_w_kernel(const float *__restrict__ w, float *__restrict__ w_hi, float *__restrict__ w_lo,
                                     long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = w[i], h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
        w_hi[i] = h;
        w_lo[i] = v - h;
    }
}

// REMAP (compact ragged rows, ragged.cuh): x row m is written to scores row row_map[m] of heads of M_out rows, and
// not at all for row_map[m] < 0; without it, to row m of heads of M rows (row_map / M_out unused).
template <bool REMAP>
__global__ void __launch_bounds__(THREADS_TC, 1)
score_gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_whi,
                     const __grid_constant__ CUtensorMap tm_wlo, const float *__restrict__ bias,
                     float *__restrict__ scores, int M, int D, int C1, int n_ref, int heads_per_tile,
                     const int32_t *__restrict__ row_map, int M_out) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char *raw = smem + (size_t)NSTAGE * STAGE;                 // [NRAW][A_TILE]
    uint64_t *tma_full = reinterpret_cast<uint64_t *>(raw + (size_t)NRAW * A_TILE);   // [NSTAGE] W tiles landed
    uint64_t *raw_full = tma_full + NSTAGE;                     // [NRAW] raw x tile landed
    uint64_t *raw_empty = raw_full + NRAW;                      // [NRAW] raw x tile read by the 4 split warps
    uint64_t *lo_ready = raw_empty + NRAW;
    uint64_t *empty = lo_ready + NSTAGE;
    uint64_t *chunk_full = empty + NSTAGE;                      // [2] accumulator p holds a finished chunk
    uint64_t *chunk_empty = chunk_full + 2;                     // [2] accumulator p has been drained
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(chunk_empty + 2);
    float *s_bias = reinterpret_cast<float *>(tmem_slot + 2);   // [heads_per_tile * C1]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // head groups vary FASTEST over the grid: the CTAs that read the same 2 MB x row-block (one per head group, 4 at
    // COCO's 81 classes) run side by side and share it through L2 instead of streaming it from HBM once each
    const int m0 = blockIdx.y * BM;
    const int h0 = blockIdx.x * heads_per_tile;                 // first head of this CTA
    const int nheads = 2 + 2 * n_ref;
    const int nh = min(heads_per_tile, nheads - h0);
    const int n0 = h0 * C1;                                     // first row of W / first logit column
    const int nkb = D / BK, nchunks = (nkb + CHK - 1) / CHK;

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&tma_full[s], 1); mbar_init(&lo_ready[s], 4); mbar_init(&empty[s], 1); }
        for (int p = 0; p < 2; ++p) { mbar_init(&chunk_full[p], 1); mbar_init(&chunk_empty[p], 4); }
        for (int r = 0; r < NRAW; ++r) { mbar_init(&raw_full[r], 1); mbar_init(&raw_empty[r], 4); }
        fence_mbar_init();
    }
    for (int i = tid; i < nh * C1; i += THREADS_TC) s_bias[i] = bias[n0 + i];
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;                      // accumulator p at columns 256 p
    // instruction descriptor: F32 accumulate, TF32 x TF32, K-major, N = NT, M = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

    if (warp == 0) {
        // ------------------------------------------------------------------ x producer (HBM stream)
        if (elect_one()) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int r = kb % NRAW;
                if (kb >= NRAW) mbar_wait(&raw_empty[r], ((kb / NRAW) - 1) & 1);
                mbar_expect_tx(&raw_full[r], (uint32_t)A_TILE);
                tma_load_2d(raw + (size_t)r * A_TILE, &tm_x, kb * BK, m0, &raw_full[r]);
            }
        }
    } else if (warp == 6) {
        // ------------------------------------------------------------------ W producer (L2 hits)
        if (elect_one()) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % NSTAGE;
                if (kb >= NSTAGE) mbar_wait(&empty[s], ((kb / NSTAGE) - 1) & 1);
                unsigned char *st = smem + (size_t)s * STAGE;
                mbar_expect_tx(&tma_full[s], (uint32_t)(2 * W_TILE));
                tma_load_2d(st + 2 * A_TILE, &tm_whi, kb * BK, n0, &tma_full[s]);
                tma_load_2d(st + 2 * A_TILE + W_TILE, &tm_wlo, kb * BK, n0, &tma_full[s]);
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (one elected thread)
        if (elect_one()) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % NSTAGE, c = kb / CHK, p = c & 1;
                if (kb % CHK == 0 && c >= 2) mbar_wait(&chunk_empty[p], ((c >> 1) - 1) & 1);   // accumulator p drained
                mbar_wait(&tma_full[s], (kb / NSTAGE) & 1);
                mbar_wait(&lo_ready[s], (kb / NSTAGE) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t base = smem_u32(smem + (size_t)s * STAGE), acc = tmem_base + 256u * p;
                const uint64_t xh = smem_desc128(base), xl = smem_desc128(base + A_TILE);
                const uint64_t wh = smem_desc128(base + 2 * A_TILE), wl = smem_desc128(base + 2 * A_TILE + W_TILE);
#pragma unroll
                for (int k = 0; k < BK / 8; ++k) {        // K = 8 tf32 = 32 B per instruction: +2 in 16 B units
                    mma_tf32(acc, xh + 2 * k, wh + 2 * k, idesc, ((kb % CHK) | k) != 0);   // a chunk starts from 0
                    mma_tf32(acc, xh + 2 * k, wl + 2 * k, idesc, 1u);
                    mma_tf32(acc, xl + 2 * k, wh + 2 * k, idesc, 1u);
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                                 smem_u32(&empty[s]))
                             : "memory");
                if (kb % CHK == CHK - 1 || kb == nkb - 1)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                                     smem_u32(&chunk_full[p]))
                                 : "memory");
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------ split warps (+ chunk drains)
        const int row = tid - 64;                              // 0..127: one x row per thread
        const uint32_t row_off = (row >> 3) * 1024 + (row & 7) * 128, sw = row & 7;
        const int q4 = warp & 3;                               // TMEM lane quarter this warp may read
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q4) << 16);
        float acc[NT];                                         // logits of TMEM lane 32 q4 + lane, RN-accumulated
#pragma unroll
        for (int j = 0; j < NT; ++j) acc[j] = 0.f;
        auto drain = [&](int c) {
            const int p = c & 1;
            mbar_wait(&chunk_full[p], (c >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int cc = 0; cc < NT / 32; ++cc) {
                float v[32];
                tmem_ld32(lane_addr + 256u * p + 32u * cc, v);
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[cc * 32 + j] += v[j];
            }
            if (NT % 32) {
                float v[16];
                tmem_ld16(lane_addr + 256u * p + (uint32_t)(NT / 32 * 32), v);
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[NT / 32 * 32 + j] += v[j];
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive1(&chunk_empty[p]);
        };
        int next_drain = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % NSTAGE, r = kb % NRAW;
            mbar_wait(&raw_full[r], (kb / NRAW) & 1);
            if (kb >= NSTAGE) mbar_wait(&empty[s], ((kb / NSTAGE) - 1) & 1);       // the stage's last MMAs are done
            const unsigned char *xr = raw + (size_t)r * A_TILE + row_off;
            unsigned char *xh = smem + (size_t)s * STAGE + row_off, *xl = xh + A_TILE;
#pragma unroll
            for (int c = 0; c < 8; ++c) {                      // the row's eight 16 B chunks (swizzled position)
                const uint32_t o = (uint32_t)((c ^ sw) << 4);
                const uint4 v = *reinterpret_cast<const uint4 *>(xr + o);
                const uint4 h = make_uint4(v.x & 0xFFFFE000u, v.y & 0xFFFFE000u, v.z & 0xFFFFE000u, v.w & 0xFFFFE000u);
                float4 l;
                l.x = __uint_as_float(v.x) - __uint_as_float(h.x);
                l.y = __uint_as_float(v.y) - __uint_as_float(h.y);
                l.z = __uint_as_float(v.z) - __uint_as_float(h.z);
                l.w = __uint_as_float(v.w) - __uint_as_float(h.w);
                *reinterpret_cast<uint4 *>(xh + o) = h;
                *reinterpret_cast<float4 *>(xl + o) = l;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) { mbar_arrive1(&lo_ready[s]); mbar_arrive1(&raw_empty[r]); }
            // drain the chunks whose last k-block was split LAG iterations ago (their MMAs are done or
            // nearly done by now, so this does not hold up the split of the next stages)
            while (next_drain < nchunks && min((next_drain + 1) * CHK, nkb) - 1 + LAG <= kb) drain(next_drain++);
        }
        while (next_drain < nchunks) drain(next_drain++);

        // ------------------------------------------------------------------ epilogue
        // every MMA has completed (the last chunk was drained): the stage memory is free.  Each thread
        // parks its row in smem (so that the heads can be indexed at run time), adds the bias and applies
        // the activation: softmax over classes / sigmoid; the detector head keeps its logits.
        asm volatile("bar.sync 1, 128;" ::: "memory");
        float *zrow = reinterpret_cast<float *>(smem) + (size_t)(32 * q4 + lane) * ZP;
#pragma unroll
        for (int j = 0; j < NT; ++j) zrow[j] = acc[j];
        const int m = m0 + 32 * q4 + lane;
        int out_row = m, out_rows = M;
        bool live = m < M;
        if constexpr (REMAP) {
            out_row = live ? row_map[m] : -1;
            out_rows = M_out;
            live = out_row >= 0;
        }
        if (live) {
            for (int hh = 0; hh < nh; ++hh) {
                const int h = h0 + hh;
                float *z = zrow + hh * C1;
                const float *bh = s_bias + hh * C1;
                float *dst = scores + ((size_t)h * out_rows + out_row) * C1;
                const bool softmax = (h == 0) || (h >= 2 && h < 2 + n_ref);
                if (softmax) {
                    float mx = -INFINITY;
                    for (int j = 0; j < C1; ++j) { z[j] += bh[j]; mx = fmaxf(mx, z[j]); }
                    float sum = 0.f;
                    for (int j = 0; j < C1; ++j) { z[j] = expf(z[j] - mx); sum += z[j]; }
                    for (int j = 0; j < C1; ++j) dst[j] = z[j] / sum;
                } else if (h == 1) {                           // detector: logits, column softmax follows
                    for (int j = 0; j < C1; ++j) dst[j] = z[j] + bh[j];
                } else {                                       // refine_iou: sigmoid
                    for (int j = 0; j < C1; ++j) dst[j] = 1.f / (1.f + expf(-(z[j] + bh[j])));
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

}  // namespace

static size_t score_tc_smem_bytes(int bias_floats) {
    const size_t ring = (size_t)NSTAGE * STAGE + (size_t)NRAW * A_TILE;
    static_assert((size_t)NSTAGE * STAGE + (size_t)NRAW * A_TILE >= (size_t)BM * ZP * 4, "the epilogue staging aliases the rings");
    return 1024 + ring + 256 + sizeof(float) * (size_t)bias_floats;
}

// can the tensor-core path take this shape?  (else score_heads.cu's FFMA kernel runs)
bool cim_score_tc_eligible(long long M, int D, int C1, int n_ref) {
    (void)n_ref;
    return M >= BM && (D % BK) == 0 && D >= BK && C1 >= 1 && C1 <= NT && encode_tiled() != nullptr &&
           (size_t)cim_max_smem_optin() >= score_tc_smem_bytes(NT);
}
size_t cim_score_tc_workspace_bytes(int D, int C1, int n_ref) {
    return 2 * sizeof(float) * (size_t)(2 + 2 * n_ref) * C1 * D + 512;
}

// logits + row activations for every head into `scores`; the detector head (1) is left as logits.  row_map != NULL:
// x holds M compact rows, scores heads of M_out padded rows (ragged.cuh)
int cim_score_tc_launch(const float *x, const float *weight, const float *bias, float *scores, long long M, int D,
                        int C1, int n_ref, void *workspace, cudaStream_t st, const int32_t *row_map,
                        long long M_out) {
    const int nheads = 2 + 2 * n_ref, N = nheads * C1;
    float *w_hi = reinterpret_cast<float *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    float *w_lo = w_hi + (size_t)N * D;
    score_split_w_kernel<<<256, 256, 0, st>>>(weight, w_hi, w_lo, (long long)N * D);
    int rc = cim_launch_status();
    if (rc) return rc;
    const int heads_per_tile = min(nheads, NT / C1);
    const int ntiles = (nheads + heads_per_tile - 1) / heads_per_tile;
    CUtensorMap tx, twh, twl;
    if (!make_map(&tx, x, M, D, BM) || !make_map(&twh, w_hi, N, D, NT) || !make_map(&twl, w_lo, N, D, NT))
        return CIM_ERR_ARG;
    const size_t smem = score_tc_smem_bytes(heads_per_tile * C1);
    if ((M + BM - 1) / BM > 65535) return CIM_ERR_SHAPE;
    dim3 grid((unsigned)ntiles, (unsigned)((M + BM - 1) / BM));
    if (row_map) {
        cudaFuncSetAttribute(score_gemm_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        score_gemm_tc_kernel<true><<<grid, THREADS_TC, smem, st>>>(tx, twh, twl, bias, scores, (int)M, D, C1, n_ref,
                                                                   heads_per_tile, row_map, (int)M_out);
    } else {
        cudaFuncSetAttribute(score_gemm_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        score_gemm_tc_kernel<false><<<grid, THREADS_TC, smem, st>>>(tx, twh, twl, bias, scores, (int)M, D, C1, n_ref,
                                                                    heads_per_tile, nullptr, 0);
    }
    return cim_launch_status();
}
