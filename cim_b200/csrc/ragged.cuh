// ragged.cuh -- the compact row layout of ragged batches (include/cimhead.h, "Compact ragged batches").
//
// Image b has n_b = n_props[b] proposals, clamped to [1, R] (R when n_props is NULL).  In the compact layout its
// proposal r sits at row off_b + r, off_b = sum_{i<b} n_i; in the padded layout at row b * R + r.  The row map
// map[m] (m < N) is the padded row of compact row m, or -1 for rows m >= sum_b n_b.  If sum_b n_b > N, the proposals
// past row N have no compact row, and their padded rows are treated as padding.  These functions are the one
// statement of that rule: the device builder (ragged.cu) and the host test hook both call them.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

__host__ __device__ __forceinline__ int ragged_count(const int32_t *n_props, int b, int R) {
    const int n = n_props ? n_props[b] : R;
    return n < 1 ? 1 : (n > R ? R : n);
}

// padded row of compact row m, given the exclusive scan off[0..n_img] of the clamped counts (off[n_img] = total)
__host__ __device__ __forceinline__ int32_t compact_row_to_padded(int m, const int32_t *off, int n_img, int R) {
    if (m >= off[n_img]) return -1;
    int lo = 0, hi = n_img - 1;                 // the last image b with off[b] <= m
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= m) lo = mid;
        else hi = mid - 1;
    }
    return lo * R + (m - off[lo]);
}

// workspace of the row map: int32 map[N] and the scan off[n_img + 1], each 256-byte aligned
inline size_t compact_map_bytes(int n_img, int N) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    return up(sizeof(int32_t) * (size_t)(N > 0 ? N : 0)) + up(sizeof(int32_t) * ((size_t)n_img + 1));
}

// Enqueues the builder of map[N] (and the scan after it) at `ws`, 256-byte aligned, compact_map_bytes() bytes.
// No host synchronisation: the offsets are computed on the device.  Returns a CIM_* code.
int compact_row_map_launch(const int32_t *n_props, int n_img, int R, int N, void *ws, cudaStream_t st);
