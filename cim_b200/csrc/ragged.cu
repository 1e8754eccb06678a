// ragged.cu -- builder of the compact row map of ragged batches (rule: ragged.cuh).
#include <vector>

#include "common.cuh"
#include "ragged.cuh"

namespace {

constexpr int MAP_THREADS = 1024;

// One CTA: the exclusive scan of the clamped counts, 1024 images per pass, into off[0..n_img], then map[0, N).
// A few microseconds for a batch of 8 x 2000 proposals: the scan is over n_img numbers and the map is N ints.
__global__ void __launch_bounds__(MAP_THREADS)
compact_row_map_kernel(const int32_t *__restrict__ n_props, int n_img, int R, int N, int32_t *__restrict__ map,
                       int32_t *__restrict__ off) {
    __shared__ int32_t warp_sum[MAP_THREADS / 32];
    __shared__ int32_t carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n_img; b0 += MAP_THREADS) {
        const int b = b0 + tid;
        const int v = b < n_img ? ragged_count(n_props, b, R) : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_sum[lane] = w;                                  // inclusive over warps
        }
        __syncthreads();
        const int base = carry + (warp ? warp_sum[warp - 1] : 0);
        if (b < n_img) off[b] = base + incl - v;
        __syncthreads();
        if (tid == MAP_THREADS - 1) carry = base + incl;
        __syncthreads();
    }
    if (tid == 0) off[n_img] = carry;
    __syncthreads();                                             // off[] is visible to the whole CTA
    for (int m = tid; m < N; m += MAP_THREADS) map[m] = compact_row_to_padded(m, off, n_img, R);
}

}  // namespace

int compact_row_map_launch(const int32_t *n_props, int n_img, int R, int N, void *ws, cudaStream_t st) {
    if (n_img <= 0 || R <= 0 || N <= 0) return CIM_ERR_ARG;
    if (!cim_aligned(ws, 256)) return CIM_ERR_ALIGN;
    int32_t *map = reinterpret_cast<int32_t *>(ws);
    int32_t *off = reinterpret_cast<int32_t *>(reinterpret_cast<unsigned char *>(ws) +
                                               ((sizeof(int32_t) * (size_t)N + 255) & ~(size_t)255));
    compact_row_map_kernel<<<1, MAP_THREADS, 0, st>>>(n_props, n_img, R, N, map, off);
    return cim_launch_status();
}

// Test hook, HOST memory only: the map the device builder writes, from host counts (NULL: R for every image).
CIM_API int cim_debug_compact_row_map(const int32_t *n_props, int n_img, int R, int N, int32_t *map_out) {
    if (!map_out || n_img <= 0 || R <= 0 || N <= 0) return CIM_ERR_ARG;
    if ((long long)n_img * R > (1LL << 30) || N > n_img * R) return CIM_ERR_SHAPE;
    std::vector<int32_t> off((size_t)n_img + 1, 0);
    for (int b = 0; b < n_img; ++b) off[b + 1] = off[b] + ragged_count(n_props, b, R);
    for (int m = 0; m < N; ++m) map_out[m] = compact_row_to_padded(m, off.data(), n_img, R);
    return CIM_OK;
}
