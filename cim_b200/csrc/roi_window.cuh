// roi_window.cuh -- RoIAlign on feature maps that do not fit the shared-memory tile: WINDOW TILES.
//
// The tile kernels of roi_align.cu keep [32 channels x H x W] of one image in shared memory, which caps the map at
// about 32 x 32 cells; VGG-16 at stride 8 (64 x 64 .. 150 x 150) and ResNet-50 at the training scales 688 .. 1200
// (43 .. 75 cells, lib/utils/blob.py:162-169 of the reference) are larger.  Here the shared-memory tile is a WINDOW of
// the map -- WIN_DIM x WIN_DIM cells whose origin is a multiple of WIN_G cells -- and every ROI is cut into SUB-ROIs that
// each fit one window, with NO partial sums to merge between them:
//
//   * per axis a ROI is 7 bins; a bin touches `n` consecutive rows (columns) with collapsed weights (roi_prep_kernel's
//     arithmetic).  A bin becomes ceil(n / 8) SLOTS of <= 8 taps, so the 8-tap inner loops of the tile kernels take
//     bins of any width up to WIN_MTB taps;
//   * consecutive bins are packed greedily into SEGMENTS of <= 7 slots whose extent fits a window; a sub-ROI is one row
//     segment x one column segment.  It is described by an ordinary NARROW tile descriptor in window-relative
//     coordinates whose 7 x 7 "bins" are its slots, so fwd_pairs / bwd_pairs / build_wyd run unchanged;
//   * the 7 x 7 VIRTUAL outputs of a sub-ROI are summed slot -> bin in the epilogue and written to the bins the
//     sub-ROI owns (distinct sub-ROIs own distinct bins); the backward reads the gradient of a slot from its bin;
//   * sub-ROIs are sorted by (image, window) with a stable counting sort, so the order in which a tile applies its
//     ROIs is fixed; the units are processed image -> channel chunk -> window -> sub-ROI, which keeps the pieces of one
//     (roi, chunk) output (and the re-reads of its gradient block by the backward) within a few MB of each other in L2.
//
// The split logic is __host__ __device__: cim_debug_roi_window_plan() runs it on the CPU so that tests can rebuild the
// forward from the descriptors without a GPU (tests/test_roi_window_plan.py).
#pragma once

namespace {

constexpr int WIN_DIM = 32;     // window rows / columns
constexpr int WIN_G = 8;        // granularity of the window origins
constexpr int WIN_MTB = 24;     // max taps per bin and axis on this path (3 slots); wider bins -> generic kernel
constexpr int WIN_KEYBITS = 10; // window coordinate index per axis < 1024

struct WinGeom {
    int Hp, W, wh, ww, nwy, nwx;
};
__host__ __device__ inline WinGeom win_geom(int H, int W) {
    WinGeom g;
    g.Hp = (H + 1) & ~1;
    g.W = W;
    g.wh = g.Hp < WIN_DIM ? g.Hp : WIN_DIM;
    g.ww = W < WIN_DIM ? W : WIN_DIM;
    g.nwy = (g.Hp - g.wh + WIN_G - 1) / WIN_G + 1;
    g.nwx = (W - g.ww + WIN_G - 1) / WIN_G + 1;
    return g;
}
// origin of window coordinate i along an axis of (padded) length L with window length wl; even for rows
__host__ __device__ inline int win_origin(int i, int L, int wl) {
    const int o = i * WIN_G;
    return o < L - wl ? o : L - wl;
}

__host__ __device__ inline float win_sample_coord(float start, float bin, int p, int s, int grid) {
#ifdef __CUDA_ARCH__
    float a = __fadd_rn(start, __fmul_rn((float)p, bin));
    float b = __fdiv_rn(__fmul_rn(__fadd_rn((float)s, .5f), bin), (float)grid);
    return __fadd_rn(a, b);
#else
    volatile float m = (float)p * bin;
    volatile float a = start + m;
    volatile float t = ((float)s + .5f) * bin;
    volatile float b = t / (float)grid;
    return a + b;
#endif
}

// one bin of one axis: first map row / column touched, number touched, collapsed weights (already / grid).
// Same arithmetic as roi_prep_kernel; returns false when the bin needs more than WIN_MTB taps.
__host__ __device__ inline bool win_bin_taps(float c1, float bin, int p, int grid, int L, int &lo, int &n, float *w) {
    int lo0 = -1;
    n = 0;
    for (int i = 0; i < WIN_MTB; ++i) w[i] = 0.f;
    for (int s = 0; s < grid; ++s) {
        float t = win_sample_coord(c1, bin, p, s, grid);
        if (t < -1.f || t > (float)L) continue;
        if (t <= 0.f) t = 0.f;
        int l0 = (int)t, h0;
        if (l0 >= L - 1) { h0 = l0 = L - 1; t = (float)l0; } else { h0 = l0 + 1; }
        const float fl = t - (float)l0, fh = 1.f - fl;
        if (lo0 < 0) lo0 = l0;
        const int i0 = l0 - lo0, i1 = h0 - lo0;
        if (i1 >= WIN_MTB) return false;
        w[i0] += fh;
        w[i1] += fl;
        n = n > i1 + 1 ? n : i1 + 1;
    }
    const float g = (float)(grid > 0 ? grid : 1);
    for (int i = 0; i < WIN_MTB; ++i) w[i] = w[i] / g;
    lo = lo0 < 0 ? -1 : lo0;
    return true;
}

struct AxisGeom {      // ROI extent along one axis in map cells
    float c1, bin;
    int grid;
    bool bad;
};
__host__ __device__ inline AxisGeom win_axis_geom(const float *r, int axis, int nb, float scale, int sr, int aligned) {
    AxisGeom a;
    const float off = aligned ? .5f : 0.f;
#ifdef __CUDA_ARCH__
    const float c1 = __fsub_rn(__fmul_rn(r[1 + (axis == 0 ? 1 : 0)], scale), off);
    const float c2 = __fsub_rn(__fmul_rn(r[3 + (axis == 0 ? 1 : 0)], scale), off);
    float ext = __fsub_rn(c2, c1);
    if (!aligned) ext = fmaxf(ext, 1.f);
    a.bin = __fdiv_rn(ext, (float)nb);
    a.grid = sr > 0 ? sr : (int)ceilf(__fdiv_rn(ext, (float)nb));
#else
    volatile float m1 = r[1 + (axis == 0 ? 1 : 0)] * scale, m2 = r[3 + (axis == 0 ? 1 : 0)] * scale;
    const float c1 = m1 - off, c2 = m2 - off;
    volatile float ext = c2 - c1;
    if (!aligned && ext < 1.f) ext = 1.f;
    volatile float q = ext / (float)nb;
    a.bin = q;
    a.grid = sr > 0 ? sr : (int)ceilf(q);
#endif
    a.c1 = c1;
    a.bad = a.grid > 64;
    return a;
}

// Border length of image b along an axis (0 = rows) of a canvas of length L: feat_hw [B][2] = (H_b, W_b), clamped to
// [1, L]; NULL: every image fills the canvas.  Only the border rule (clamp to L_b - 1, drop beyond L_b) uses it; window
// geometry, tile layout and addressing stay on the canvas.
__host__ __device__ inline int img_extent(const int *feat_hw, int b, int axis, int L) {
    if (!feat_hw) return L;
#ifdef __CUDA_ARCH__
    const int v = __ldg(feat_hw + 2 * b + axis);
#else
    const int v = feat_hw[2 * b + axis];
#endif
    return v < 1 ? 1 : v > L ? L : v;
}

// Plan of one (roi, axis): bins -> slots -> segments.
struct AxisPlan {
    int nseg;              // 0: this ROI takes the generic kernel
    int lo[7], n[7];       // per bin (empty bins: n = 0, lo = a neighbour's)
    int first_bin[8];      // segment s covers bins [first_bin[s], first_bin[s + 1])
    int nslots[7];         // slots of segment s
    int wcoord[7];         // window coordinate index of segment s
};
__host__ __device__ inline int win_slots_of(int n) { return n <= 8 ? 1 : (n + 7) >> 3; }

// L: the image's length along the axis (border rule), Lp: padded canvas length (rows: even), wl: window length,
// nw: window positions
__host__ __device__ inline void win_axis_plan(const AxisGeom &a, int L, int Lp, int wl, int nw, AxisPlan &pl) {
    pl.nseg = 0;
    if (a.bad) return;
    float w[WIN_MTB];
    for (int p = 0; p < 7; ++p)
        if (!win_bin_taps(a.c1, a.bin, p, a.grid, L, pl.lo[p], pl.n[p], w)) return;
    // empty bins sit where a neighbour is (they own an all-zero slot, so that their outputs are written as zeros)
    int next = -1;
    for (int p = 6; p >= 0; --p) {
        if (pl.lo[p] >= 0) next = pl.lo[p];
        else if (next >= 0) pl.lo[p] = next;
    }
    int prev = 0;
    for (int p = 0; p < 7; ++p) {
        if (pl.lo[p] < 0) pl.lo[p] = prev;
        prev = pl.lo[p];
    }
    int nseg = 0, sc = 0, smin = 0, emax = 0;
    for (int p = 0; p < 7; ++p) {
        const int ns = win_slots_of(pl.n[p]);
        const int end = pl.lo[p] + (pl.n[p] > 0 ? pl.n[p] : 1);
        bool fits = false;
        if (sc > 0 && sc + ns <= 7) {
            const int lo_min = smin < pl.lo[p] ? smin : pl.lo[p];
            int wi = lo_min / WIN_G;
            if (wi > nw - 1) wi = nw - 1;
            const int e = emax > end ? emax : end;
            fits = e - win_origin(wi, Lp, wl) <= wl;
        }
        if (!fits) {                       // open a new segment with this bin
            if (nseg == 7) { pl.nseg = 0; return; }
            pl.first_bin[nseg] = p;
            pl.nslots[nseg] = 0;
            ++nseg;
            sc = 0;
            smin = pl.lo[p];
            emax = end;
            int wi = smin / WIN_G;
            if (wi > nw - 1) wi = nw - 1;
            if (ns > 7 || end - win_origin(wi, Lp, wl) > wl) { pl.nseg = 0; return; }     // a single bin must fit
        }
        sc += ns;
        if (pl.lo[p] < smin) smin = pl.lo[p];
        if (end > emax) emax = end;
        pl.nslots[nseg - 1] = sc;
        int wi = smin / WIN_G;
        if (wi > nw - 1) wi = nw - 1;
        pl.wcoord[nseg - 1] = wi;
    }
    pl.first_bin[nseg] = 7;
    pl.nseg = nseg;
}

// Descriptor words the window path adds to the NARROW layout (they are spare there)
enum { DW_ROI = D_B, DW_YMAP = D_YLO + 7, DW_XMAP = D_XLO + 7, DW_FLAGS = D_YN + 7 };
// DW_YMAP / DW_XMAP: nibble s = bin of slot s (15: unused), bits 28..30 = number of slots.  DW_FLAGS bit 0: SIMPLE
// (one sub-ROI covers the ROI with 7 one-slot bins per axis: the 49 virtual outputs ARE the outputs).

// Write one axis' part of the descriptor of the sub-ROI that pairs segment `seg` of this axis with any segment of the
// other axis.  d: the 168-word descriptor.  axis 0 = rows.
__host__ __device__ inline void win_axis_emit(const AxisGeom &a, const AxisPlan &pl, int seg, int axis, int L, int Lp,
                                              int wl, int roi, bool simple, int *d) {
    float w[WIN_MTB];
    const int org = win_origin(pl.wcoord[seg], Lp, wl);
    int s_lo[7], s_n[7], s_bin[7];
    float s_w[7][8];
    int ns = 0;
    for (int p = pl.first_bin[seg]; p < pl.first_bin[seg + 1]; ++p) {
        int lo, n;
        win_bin_taps(a.c1, a.bin, p, a.grid, L, lo, n, w);
        lo = pl.lo[p];                                     // (empty bins: the neighbour's position)
        // a bin of n > 8 taps is cut into k slots of nearly equal width (9 -> 4 + 5, not 8 + 1): the slots' first and
        // last rows then ascend from slot to slot across bins too (adjacent bins overlap by at most 2 taps), which the
        // row-pair lists of the backward (a contiguous slot range per pair) and its XINC fast path rely on
        const int k = win_slots_of(n);
        for (int j = 0; j < k; ++j, ++ns) {
            const int t0 = (j * n) / k, t1 = ((j + 1) * n) / k;
            s_bin[ns] = p;
            s_lo[ns] = lo + t0 - org;
            s_n[ns] = t1 - t0;
            for (int i = 0; i < 8; ++i) s_w[ns][i] = (t0 + i < t1) ? w[t0 + i] : 0.f;
        }
    }
    unsigned map = (unsigned)ns << 28;
    for (int s = 0; s < 7; ++s) map |= (unsigned)(s < ns ? s_bin[s] : 15) << (4 * s);
    float *df = reinterpret_cast<float *>(d);
    if (axis == 0) {
        d[DW_ROI] = roi;
        d[D_FLAGY] = 0;
        d[DW_YMAP] = (int)map;
        d[DW_FLAGS] = simple ? 1 : 0;
        int y0 = 1 << 30, y1 = 0;
        for (int s = 0; s < 7; ++s) {
            const int lo = s < ns ? s_lo[s] : 0, n = s < ns ? s_n[s] : 0;
            d[D_YLO + s] = lo;
            d[D_YN + s] = n;
            if (n > 0) { y0 = y0 < lo ? y0 : lo; y1 = y1 > lo + n ? y1 : lo + n; }
            float *wy = df + D_WY + s * WYP;
            wy[0] = 0.f;
            wy[WYP - 1] = 0.f;
            for (int i = 0; i < MAXT; ++i) wy[1 + i] = s < ns ? s_w[s][i] : 0.f;
        }
        if (y1 == 0) y0 = 0;
        d[D_Y0] = y0;
        d[D_Y1] = y1;
        int own = 0;
        for (int y = y0; y < y1 && own != 0xffff; ++y) own |= 1 << ((y >> 1) & 15);
        d[D_OWN] = own;
        unsigned char *phr = reinterpret_cast<unsigned char *>(d + D_PHR);
        const int pb = y0 >> 1, pe = (y1 + 1) >> 1;
        for (int j = 0; j < 32; ++j) {
            int first = 0, cnt = 0;
            if (pb + j < pe)
                for (int s = 0; s < ns; ++s) {
                    const int rel = 2 * (pb + j) - s_lo[s];
                    if (s_n[s] > 0 && rel + 1 >= 0 && rel < s_n[s]) { if (cnt == 0) first = s; cnt = s - first + 1; }
                }
            phr[j] = (unsigned char)(first | (cnt << 4));
        }
    } else {
        // tap class T in {2,3,4,6,8}: the forward's x loops are unrolled T times.  (The backward updates a slot with one
        // 8-tap-wide tensor-memory access whatever T is; its tile rows carry 8 spare columns for slots that start
        // fewer than 8 columns from the window's right edge.)
        int nmax = 0;
        for (int s = 0; s < ns; ++s) nmax = nmax > s_n[s] ? nmax : s_n[s];
        const int T = nmax <= 2 ? 2 : nmax <= 3 ? 3 : nmax <= 4 ? 4 : nmax <= 6 ? 6 : 8;
        d[D_FLAGX] = 0;
        d[D_TX] = T;
        d[DW_XMAP] = (int)map;
        int inc = 1, prev = -1;
        for (int s = 0; s < 7; ++s) {
            const int lo = s < ns ? s_lo[s] : 0;
            int lo2 = lo < wl - T ? lo : wl - T;
            if (lo2 < 0) lo2 = 0;
            const int sh = lo - lo2;
            d[D_XLO + s] = lo2;
            for (int i = 0; i < MAXT; ++i) {
                const int src = i - sh;
                df[D_WX + s * MAXT + i] = (s < ns && src >= 0 && src < MAXT) ? s_w[s][src] : 0.f;
            }
            if (s < ns) {
                if (lo2 <= prev) inc = 0;
                prev = lo2;
            }
        }
        d[D_XINC] = inc;
    }
}

// ---------------------------------------------------------------------------------------------- prep kernels
// Workspace of the window path (after the common header): per-ROI records, keys, bucket tables, sorted descriptors.
struct WinWs {
    int *rec;          // [K][2][4]  per (roi, axis): nseg | simple << 8, wcoord[0..3] / [4..6] packed in 3 more ints
    int *item_base;    // [K + 1]    first item (sub-ROI) of each ROI, ROI order
    int *flags;        // [K][4]     word 1 = 1: the ROI takes the generic kernel (layout the leftover pass reads)
    int *keys;         // [cap]      bucket (image * NW + window) of each item, ROI order
    int *slot;         // [cap]      sorted position of each item
    int *bucket;       // [B * NW + 1] first sorted position of each bucket; hist during the count
    int *desc;         // [cap][DESC_WORDS] descriptors in sorted order
    int cap;
};

__device__ __forceinline__ void win_pack_rec(const AxisPlan &pl, int *r) {
    r[0] = pl.nseg | ((pl.nseg == 1 && pl.nslots[0] == 7) ? 256 : 0);
    r[1] = pl.nseg > 0 ? (pl.wcoord[0] | (pl.nseg > 1 ? pl.wcoord[1] << WIN_KEYBITS : 0) |
                          (pl.nseg > 2 ? pl.wcoord[2] << (2 * WIN_KEYBITS) : 0)) : 0;
    r[2] = pl.nseg > 3 ? (pl.wcoord[3] | (pl.nseg > 4 ? pl.wcoord[4] << WIN_KEYBITS : 0) |
                          (pl.nseg > 5 ? pl.wcoord[5] << (2 * WIN_KEYBITS) : 0)) : 0;
    r[3] = pl.nseg > 6 ? pl.wcoord[6] : 0;
}
__device__ __forceinline__ int win_rec_coord(const int *r, int s) {
    return (r[1 + s / 3] >> ((s % 3) * WIN_KEYBITS)) & ((1 << WIN_KEYBITS) - 1);
}

// pass 1: thread per (roi, axis): plan -> record
__global__ void roi_win_plan_kernel(const float *__restrict__ rois, const int *__restrict__ feat_hw, int K, int B, int H,
                                    int W, float scale, int sr, int aligned, WinWs ws) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = gid >> 1, axis = gid & 1;
    if (k >= K) return;
    const float *r = rois + 5 * (size_t)k;
    const WinGeom g = win_geom(H, W);
    const AxisGeom a = win_axis_geom(r, axis, 7, scale, sr, aligned);
    AxisPlan pl;
    const int b = (int)r[0];
    if (b < 0 || b >= B) pl.nseg = 0;
    else if (axis == 0) win_axis_plan(a, img_extent(feat_hw, b, 0, H), g.Hp, g.wh, g.nwy, pl);
    else win_axis_plan(a, img_extent(feat_hw, b, 1, W), W, g.ww, g.nwx, pl);
    win_pack_rec(pl, ws.rec + ((size_t)k * 2 + axis) * 4);
}

// pass 2: one CTA: items per ROI, exclusive scan in ROI order, overflow / flagged ROIs -> generic kernel
__global__ void __launch_bounds__(1024)
roi_win_scan_kernel(int K, WinWs ws) {
    __shared__ int s_sum[32];
    __shared__ int s_carry, s_total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_carry = 0; s_total = 0x7fffffff; }
    __syncthreads();
    for (int k0 = 0; k0 < K; k0 += 1024) {
        const int k = k0 + tid;
        int cnt = 0;
        if (k < K) {
            const int ny = ws.rec[((size_t)k * 2) * 4] & 255, nx = ws.rec[((size_t)k * 2 + 1) * 4] & 255;
            cnt = ny * nx;
        }
        int v = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        if (lane == 31) s_sum[warp] = v;
        __syncthreads();
        if (warp == 0) {
            int t = s_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int q = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += q;
            }
            s_sum[lane] = t;
        }
        __syncthreads();
        const int carry = s_carry;
        int excl = carry + v - cnt + (warp > 0 ? s_sum[warp - 1] : 0);
        if (k < K) {
            if (excl + cnt > ws.cap) {                      // no room left (cannot happen with the workspace
                atomicMin(&s_total, excl);                  // cim_roi_align_workspace_bytes_ex asks for): generic kernel
                cnt = 0;
                excl = 0;
            }
            ws.item_base[k] = excl;
            int *f = ws.flags + (size_t)k * 4;
            f[0] = 0; f[1] = cnt == 0; f[2] = 0; f[3] = 0;
        }
        __syncthreads();
        if (tid == 1023) s_carry = carry + s_sum[31];
        __syncthreads();
    }
    if (tid == 0) ws.item_base[K] = s_carry < s_total ? s_carry : s_total;
}

// pass 3: thread per ROI: bucket key of each of its items + bucket histogram
__global__ void roi_win_keys_kernel(const float *__restrict__ rois, int K, int NW, int nwx, WinWs ws) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    if (ws.flags[(size_t)k * 4 + 1]) return;
    const int *ry = ws.rec + ((size_t)k * 2) * 4, *rx = ry + 4;
    const int ny = ry[0] & 255, nx = rx[0] & 255, b = (int)rois[5 * (size_t)k];
    const int base = ws.item_base[k];
    for (int sy = 0; sy < ny; ++sy)
        for (int sx = 0; sx < nx; ++sx) {
            const int key = b * NW + win_rec_coord(ry, sy) * nwx + win_rec_coord(rx, sx);
            ws.keys[base + sy * nx + sx] = key;
            atomicAdd(ws.bucket + key + 1, 1);            // bucket[0] stays 0; scanned in place by the next kernel
        }
}

// pass 4: one CTA: inclusive scan of the histogram in place -> bucket[j] = first sorted position of bucket j
__global__ void __launch_bounds__(1024)
roi_win_bucket_kernel(int nb, WinWs ws) {
    __shared__ int s_sum[32];
    __shared__ int s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int j0 = 1; j0 <= nb; j0 += 1024) {
        const int j = j0 + tid;
        const int cnt = j <= nb ? ws.bucket[j] : 0;
        int v = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        if (lane == 31) s_sum[warp] = v;
        __syncthreads();
        if (warp == 0) {
            int t = s_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int q = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += q;
            }
            s_sum[lane] = t;
        }
        __syncthreads();
        const int carry = s_carry;
        if (j <= nb) ws.bucket[j] = carry + v + (warp > 0 ? s_sum[warp - 1] : 0);
        __syncthreads();
        if (tid == 1023) s_carry = carry + s_sum[31];
        __syncthreads();
    }
}

// pass 5: CTA per bucket: STABLE placement -- the items whose key is this bucket, in ROI order (the rois need not be
// grouped by image on this path; every CTA scans all keys: a few tens of thousands of ints from L2)
__global__ void __launch_bounds__(256)
roi_win_place_kernel(int K, WinWs ws) {
    __shared__ int s_w[8];
    __shared__ int s_base;
    const int key = blockIdx.x;
    const int first = ws.bucket[key], n = ws.bucket[key + 1] - first;
    if (n == 0) return;
    const int i1 = ws.item_base[K];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < i1; c0 += 256) {
        const int i = c0 + tid;
        const bool hit = i < i1 && ws.keys[i] == key;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_w[warp] = __popc(m);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < warp; ++w) before += s_w[w];
        if (hit) ws.slot[i] = first + before + __popc(m & ((1u << lane) - 1u));
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int w = 0; w < 8; ++w) t += s_w[w];
            s_base += t;
        }
        __syncthreads();
    }
}

// pass 6: thread per (roi, axis): the axis' part of the descriptors of every sub-ROI of the ROI
__global__ void roi_win_emit_kernel(const float *__restrict__ rois, const int *__restrict__ feat_hw, int K, int H, int W,
                                    float scale, int sr, int aligned, WinWs ws) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = gid >> 1, axis = gid & 1;
    if (k >= K) return;
    if (ws.flags[(size_t)k * 4 + 1]) return;
    const float *r = rois + 5 * (size_t)k;
    const WinGeom g = win_geom(H, W);
    const AxisGeom a = win_axis_geom(r, axis, 7, scale, sr, aligned);
    const int Lb = img_extent(feat_hw, (int)r[0], axis, axis == 0 ? H : W);    // (flagged: b out of range, above)
    AxisPlan pl;
    if (axis == 0) win_axis_plan(a, Lb, g.Hp, g.wh, g.nwy, pl);
    else win_axis_plan(a, Lb, W, g.ww, g.nwx, pl);
    const int *ry = ws.rec + ((size_t)k * 2) * 4, *rx = ry + 4;
    const int ny = ry[0] & 255, nx = rx[0] & 255;
    const bool simple = (ry[0] & 256) && (rx[0] & 256);
    const int base = ws.item_base[k];
    const int nmine = axis == 0 ? ny : nx, nother = axis == 0 ? nx : ny;
    for (int s = 0; s < nmine; ++s) {
        int *d0 = nullptr;
        for (int t = 0; t < nother; ++t) {
            const int item = base + (axis == 0 ? s * nx + t : t * nx + s);
            int *d = ws.desc + (size_t)ws.slot[item] * DESC_WORDS;
            if (t == 0) {
                if (axis == 0) win_axis_emit(a, pl, s, 0, Lb, g.Hp, g.wh, k, simple, d);
                else win_axis_emit(a, pl, s, 1, Lb, W, g.ww, k, simple, d);
                d0 = d;
            } else if (axis == 0) {            // the row part: words 0, 1, 4, 5, 7, 8..23, 32..109
                d[0] = d0[0]; d[1] = d0[1]; d[4] = d0[4]; d[5] = d0[5]; d[7] = d0[7];
                for (int i = D_YLO; i < D_XLO; ++i) d[i] = d0[i];
                for (int i = D_PHR; i < D_WY + 7 * WYP; ++i) d[i] = d0[i];
            } else {                           // the column part: words 2, 3, 6, 24..31, 112..167
                d[2] = d0[2]; d[3] = d0[3]; d[6] = d0[6];
                for (int i = D_XLO; i < D_PHR; ++i) d[i] = d0[i];
                for (int i = D_WX; i < DESC_WORDS; ++i) d[i] = d0[i];
            }
        }
    }
}

}  // namespace
