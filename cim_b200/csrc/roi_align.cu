// roi_align.cu -- RoIAlign forward / backward for sm_100a.
//
// Replaces mmcv.ops.RoIAlign at lib/modeling/model_builder.py:230-231 of the reference
// (arithmetic: lib/modeling/roi_xfrom/roi_align/src/roi_align_kernel.cu:16-121 fwd,
// :150-270 bwd, plus mmcv's `aligned` half-pixel shift).
//
// Design (DESIGN.md "RoIAlign"):
//   1. roi_prep_kernel turns every ROI into a descriptor: per output bin and axis the first
//      feature row/column touched, the number touched and the COLLAPSED bilinear weights
//      (all samples of the bin folded into <= 8 taps per axis; the 2-D weight of a tap is the
//      product of its row and column weight, already divided by the sample count).  It also
//      checks that rois are grouped by image and records each image's ROI range.
//   2. Tile kernels: a CTA keeps the [32 channels x H x W] feature (or gradient) tile of one
//      image in shared memory and sweeps the image's ROIs, lane = channel.  The tile is stored
//      ROW-PAIR INTERLEAVED: rows 2p and 2p+1 of a channel alternate element by element, so one
//      LDS.64 / STS.64 moves (f[2p][x], f[2p+1][x]) and one FFMA2 (fma.rn.f32x2, weight as the
//      scalar-broadcast operand) does the arithmetic of both rows.  The channel pitch is 2 x odd
//      words, which makes the 64-bit accesses of a warp bank-conflict free.
//        forward : persistent, one CTA per SM, (roi, chunk) units split evenly; a warp owns one
//                  ROI at a time, its descriptor is prefetched into smem with cp.async (LDGSTS)
//                  one ROI ahead; ROW-PAIR SWEEP: per row pair the 7 column sums (x pass) are
//                  formed once and added into all 7 output rows with a dense, branch-free y pass
//                  (per-warp smem table of the pair's 7 x 2 row weights); 49 float2 accumulators
//                  (even row / odd row partial sums) in registers; the 32 x 49 outputs are staged
//                  in smem and leave with one 6272-byte cp.async.bulk (UBLKCP) per (roi, 32 ch).
//        backward: gradients + descriptors stream through a 3-slot mbarrier ring of 4 ROIs each
//                  (cp.async.bulk, no CTA-wide barrier); warp w of 16 owns the tile row pairs
//                  p % 16 == w, so every tile address has exactly one writer and ROIs are
//                  applied in index order: no atomics, bit-reproducible.
//   3. Generic kernels (one thread per output element, sample by sample) take whatever the
//      tile kernels cannot: other output sizes, feature maps too large for shared memory,
//      bins wider than 8 taps, ROIs not grouped by image.
#include "common.cuh"
#include <algorithm>

namespace {

constexpr int PH = 7, PW = 7, NBIN = 49;
// Descriptor layouts.  NARROW (tile kernels: the map sits in shared memory, every byte next to it counts): up to 8
// collapsed taps per bin and axis, 672 B per ROI.  WIDE (global-pairs kernels, large maps such as VGG-16's 64 x 64 at
// stride 8, where a bin of a full-image ROI spans 11 taps): up to 12 taps, 896 B per ROI.  Words 0..39 are common.
template <bool WIDE>
struct DescL {
    static constexpr int MT = WIDE ? 12 : 8;        // max collapsed taps per bin and axis
    static constexpr int WYP = MT + 2;              // row weights of a bin, padded: [0, w_0 .. w_{MT-1}, 0]
    static constexpr int WX = WIDE ? 140 : 112;     // first word of the column weights [7][MT]
    static constexpr int WORDS = WX + 7 * MT;       // 224 : 168
};
constexpr int MAXT = DescL<false>::MT;
constexpr int WYP = DescL<false>::WYP;
constexpr int DESC_WORDS = DescL<false>::WORDS;     // 672 B per ROI (tile kernels)
constexpr int DESC_WORDS_MAX = DescL<true>::WORDS;  // what the workspace reserves per ROI
enum {
    D_B = 0, D_FLAGY = 1, D_FLAGX = 2, D_TX = 3, D_Y0 = 4, D_Y1 = 5, D_XINC = 6, D_OWN = 7,
    D_YLO = 8, D_YN = 16, D_XLO = 24, D_PHR = 32 /* 32 bytes */, D_WY = 40 /* [7][WYP] */, D_WX = DescL<false>::WX
};
static_assert(D_WY + 7 * DescL<false>::WYP <= DescL<false>::WX && DescL<false>::WORDS == 168, "narrow descriptor");
static_assert(D_WY + 7 * DescL<true>::WYP <= DescL<true>::WX && (DescL<true>::WX % 4) == 0 &&
              (DescL<true>::WORDS % 4) == 0 && DescL<true>::WORDS / 4 <= 64, "wide descriptor");
constexpr int WS_HDR_BYTES = 256;   // word 0: "rois not grouped by image" flag
constexpr int CH = 32;              // channels per tile (= lanes)
constexpr int STAGE_FLOATS = CH * NBIN;          // 1568 floats = 6272 B

}  // namespace
#include "roi_window.cuh"
namespace {

struct RoiWs {
    int *hdr;          // [64]
    int *img_start;    // [B+1]
    int *desc;         // [K][DESC_WORDS]
    float *maskpad;    // [K][52]  fused MaskFuse backward: the ROI masks padded to 208 B rows
};

__host__ __device__ inline size_t ws_img_off() { return WS_HDR_BYTES; }
__host__ __device__ inline size_t ws_desc_off(int B) {
    size_t o = WS_HDR_BYTES + sizeof(int) * (size_t)(B + 1);
    return (o + 15) & ~(size_t)15;
}

// ------------------------------------------------------------------------------------ prep
// One sample coordinate, evaluated exactly like the reference expression
//   start + p * bin + (s + .5f) * bin / grid          (roi_align_kernel.cu:103-108)
// with every operation individually rounded (no FMA contraction), so that the integer
// decisions (floor, border tests) agree with a plain C evaluation.
__device__ __forceinline__ float sample_coord(float start, float bin, int p, int s, int grid) {
    float a = __fadd_rn(start, __fmul_rn((float)p, bin));
    float b = __fdiv_rn(__fmul_rn(__fadd_rn((float)s, .5f), bin), (float)grid);
    return __fadd_rn(a, b);
}

template <bool WIDE>
__global__ void roi_prep_kernel(const float *__restrict__ rois, const int *__restrict__ feat_hw, int K, int B, int H,
                                int W, int oh, int ow, float scale, int sampling_ratio, int aligned,
                                int *__restrict__ hdr, int *__restrict__ img_start,
                                int *__restrict__ desc) {
    int gid = blockIdx.x * blockDim.x + threadIdx.x;
    int k = gid >> 1, axis = gid & 1;          // axis 0 = y (rows), 1 = x (columns)
    if (k >= K) return;
    const float *r = rois + 5 * (size_t)k;
    constexpr int MAXT = DescL<WIDE>::MT, WYP = DescL<WIDE>::WYP, D_WX = DescL<WIDE>::WX;
    int *d = desc + (size_t)k * DescL<WIDE>::WORDS;
    int b = (int)r[0];

    if (axis == 0) {
        d[D_B] = b;
        // image ranges + grouping check (rois of one image must be contiguous, ascending)
        int bprev = k > 0 ? (int)rois[5 * (size_t)(k - 1)] : -1;
        if (k > 0 && b < bprev) atomicOr(hdr, 1);
        int lo = max(bprev + 1, 0), hi = min(b, B);
        if (k == 0) lo = 0;
        for (int j = lo; j <= hi; ++j) img_start[j] = k;
        if (k == K - 1)
            for (int j = max(b + 1, 0); j <= B; ++j) img_start[j] = K;
    }

    const int nb = axis == 0 ? oh : ow;       // bins along this axis (7 on the tile path)
    // border rule on the image's own extent; the x-window shift below stays on the canvas width W
    const int L = (b >= 0 && b < B) ? img_extent(feat_hw, b, axis, axis == 0 ? H : W) : (axis == 0 ? H : W);
    const float off = aligned ? .5f : 0.f;
    float c1 = __fsub_rn(__fmul_rn(r[1 + (axis == 0 ? 1 : 0)], scale), off);
    float c2 = __fsub_rn(__fmul_rn(r[3 + (axis == 0 ? 1 : 0)], scale), off);
    float ext = __fsub_rn(c2, c1);
    if (!aligned) ext = fmaxf(ext, 1.f);
    float bin = __fdiv_rn(ext, (float)nb);
    int grid = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(ext, (float)nb));

    int flag = 0;
    if (nb != 7 || grid > 64 || b < 0 || b >= B) flag = 1;

    int lo_[7], n_[7];
    float w_[7][MAXT];
    int nmax = 0;
    if (!flag) {
        for (int p = 0; p < 7; ++p) {
            int lo0 = -1, n = 0;
            float w[MAXT];
#pragma unroll
            for (int i = 0; i < MAXT; ++i) w[i] = 0.f;
            for (int s = 0; s < grid; ++s) {
                float t = sample_coord(c1, bin, p, s, grid);
                if (t < -1.f || t > (float)L) continue;
                if (t <= 0.f) t = 0.f;
                int l0 = (int)t, h0;
                if (l0 >= L - 1) { h0 = l0 = L - 1; t = (float)l0; } else { h0 = l0 + 1; }
                float fl = t - (float)l0, fh = 1.f - fl;
                if (lo0 < 0) lo0 = l0;
                int i0 = l0 - lo0, i1 = h0 - lo0;
                if (i1 >= MAXT) { flag = 1; break; }
                w[i0] += fh;
                w[i1] += fl;
                n = max(n, i1 + 1);
            }
            if (flag) break;
            lo_[p] = lo0 < 0 ? 0 : lo0;
            n_[p] = n;
            nmax = max(nmax, n);
            float g = (float)(grid > 0 ? grid : 1);
#pragma unroll
            for (int i = 0; i < MAXT; ++i) w_[p][i] = w[i] / g;
        }
    }

    if (axis == 0) {
        d[D_FLAGY] = flag;
        int y0 = 1 << 30, y1 = 0;
        for (int p = 0; p < 7; ++p) {
            int lo = flag ? 0 : lo_[p], n = flag ? 0 : n_[p];
            d[D_YLO + p] = lo;
            d[D_YN + p] = n;
            if (n > 0) { y0 = min(y0, lo); y1 = max(y1, lo + n); }
            float *wy = reinterpret_cast<float *>(d) + D_WY + p * WYP;
            wy[0] = 0.f;
            wy[WYP - 1] = 0.f;
            for (int i = 0; i < MAXT; ++i) wy[1 + i] = flag ? 0.f : w_[p][i];
        }
        if (y1 == 0) y0 = 0;
        d[D_Y0] = y0;
        d[D_Y1] = y1;
        // backward: which of the 16 warps own a row of [y0, y1)?  warp w owns the row pairs p = y >> 1 with p % 16 == w
        int own = 0;
        for (int y = y0; y < y1 && own != 0xffff; ++y) own |= 1 << ((y >> 1) & 15);
        d[D_OWN] = flag ? 0 : own;
        d[D_YLO + 7] = 0;
        d[D_YN + 7] = 0;
        // backward: byte j of D_PHR = first | count << 4 of the bins whose row window meets row pair
        // (y0 >> 1) + j (windows are monotone in the bin index, so the set is a contiguous range)
        unsigned char *phr = reinterpret_cast<unsigned char *>(d + D_PHR);
        const int pb = y0 >> 1, pe = (y1 + 1) >> 1;
        if (pe - pb > 32) {                       // more row pairs than the table holds (H > 64): generic path
            d[D_FLAGY] = 1;
            d[D_OWN] = 0;
        }
        for (int j = 0; j < 32; ++j) {
            int first = 0, cnt = 0;
            if (!flag && pb + j < pe)
                for (int p = 0; p < 7; ++p) {
                    const int rel = 2 * (pb + j) - lo_[p];       // window index of row 2 (pb + j)
                    if (n_[p] > 0 && rel + 1 >= 0 && rel < n_[p]) { if (cnt == 0) first = p; cnt = p - first + 1; }
                }
            phr[j] = (unsigned char)(first | (cnt << 4));
        }
    } else {
        // tap class T in {2,3,4,6,8(,12)}: the x loops of the tile kernels are unrolled T times.
        int T = nmax <= 2 ? 2 : nmax <= 3 ? 3 : nmax <= 4 ? 4 : nmax <= 6 ? 6 : nmax <= 8 ? 8 : 12;
        if (W < T) flag = 1;
        d[D_FLAGX] = flag;
        d[D_TX] = T;
        int inc = 1, prev = -1;
        for (int p = 0; p < 7; ++p) {
            int lo = flag ? 0 : lo_[p];
            // shift the window left so that lo + T - 1 stays inside the row; the padding
            // taps get weight 0 but must still address valid shared memory
            int lo2 = min(lo, W - T);
            if (lo2 < 0) lo2 = 0;
            int sh = lo - lo2;
            d[D_XLO + p] = lo2;
            for (int i = 0; i < MAXT; ++i) {
                int src = i - sh;
                float v = (!flag && src >= 0 && src < MAXT) ? w_[p][src] : 0.f;
                reinterpret_cast<float *>(d)[D_WX + p * MAXT + i] = v;
            }

            if (lo2 <= prev) inc = 0;
            prev = lo2;
        }
        // 1: window starts strictly increase -> taps of one l never alias.  3: in addition the T-wide windows of bins
        // p and p + 3 never overlap, so the bins can be updated in the three groups {0,3,6}, {1,4}, {2,5} with
        // whole-window accesses (tensor-memory backward)
        if (inc && !flag) {
            int g3 = 1;
            for (int p = 0; p + 3 < 7; ++p)
                if (d[D_XLO + p + 3] - d[D_XLO + p] < T) g3 = 0;
            if (g3) inc = 3;
        }
        d[D_XINC] = inc;
        d[D_XLO + 7] = 0;
    }
}

// ------------------------------------------------------------------------------ tile: forward
// Tile layout (both directions): element (c, y, x) lives at tile[c * pitch + ((y >> 1) * W + x) * 2 + (y & 1)],
// i.e. as float2 index c * pitch / 2 + (y >> 1) * W + x  ->  (f[2p][x], f[2p+1][x]).  H odd: the missing
// row of the last pair is zero (its weights are zero too, but it must be finite).
__device__ __forceinline__ int tile_off(int y, int x, int W) { return (((y >> 1) * W + x) << 1) + (y & 1); }

__device__ __forceinline__ void load_tile(float *tile, const float *__restrict__ src, int H, int W,
                                          int pitch, int tid, int nthr) {
    const int HW = H * W;
    if ((W & 3) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        const int n4 = CH * HW / 4;
        for (int e = tid; e < n4; e += nthr) {
            const float4 v = __ldg(s4 + e);
            const int idx = e * 4, c = idx / HW, rem = idx - c * HW, y = rem / W, x = rem - y * W;
            float *dst = tile + c * pitch + tile_off(y, x, W);
            dst[0] = v.x; dst[2] = v.y; dst[4] = v.z; dst[6] = v.w;
        }
    } else {
        for (int e = tid; e < CH * HW; e += nthr) {
            const int c = e / HW, rem = e - c * HW, y = rem / W, x = rem - y * W;
            tile[c * pitch + tile_off(y, x, W)] = __ldg(src + e);
        }
    }
    if (H & 1)
        for (int e = tid; e < CH * W; e += nthr) {
            const int c = e / W, x = e - c * W;
            tile[c * pitch + tile_off(H, x, W)] = 0.f;
        }
}

// 16-byte async copy global -> shared (LDGSTS), per-thread completion groups
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ float2 bcast2(float w) { return make_float2(w, w); }   // FFMA2 takes it as R.F32

// One ROI x 32 channels (lane = channel), row-pair sweep.  Per pair p of the ROI's rows:
//   x pass: r[pw] = sum_l wx[pw][l] * (f[2p][xo+l], f[2p+1][xo+l])        7T LDS.64 + 7T FFMA2
//   y pass: (out[2q][pw], out[2q+1][pw]) += (wy[2q][y], wy[2q+1][y]) * r_y[pw]  for y = 2p, 2p+1 and ALL q:
//           56 FFMA2 with r_y as the scalar-broadcast operand; the weights (mostly zero) come from the warp's
//           dense per-row table wyd[y][8] -- no data-dependent branch in the loop, 28 float2 accumulators.
// All control flow depends only on the descriptor (warp-uniform).  T >= 6 keeps the x weights in smem.
// GLB: the feature map does not fit in shared memory (VGG-16: 64 x 64 x 32 ch = 512 KB); the same sweep reads a
// channel-last copy of the map in global memory instead -- element (p, x, c) = (f[2p][x], f[2p+1][x]) of channel c
// at float2 index (p * W + x) * C + c, so the 32 lanes (= channels) of a warp read 256 contiguous bytes per tap
// (L1 / L2 resident: a map is a few MB).  xs = float2 stride between neighbouring columns (1 in smem, C in global).
template <int T, bool GLB>
__device__ __forceinline__ void fwd_pairs(const float *__restrict__ tile_c, int W, int xs_rt, const int *__restrict__ d,
                                          float *__restrict__ stage_c, const float4 *__restrict__ wyd, int lane) {
    const int xs = GLB ? xs_rt : 1;
    constexpr bool WREG = T <= 4;
    constexpr int TR = WREG ? T : 1;
    constexpr int MAXT = DescL<GLB>::MT;                  // GLB kernels read WIDE descriptors
    float wx[PW][TR];
    int xo[PW];
    const float *dwx = reinterpret_cast<const float *>(d + DescL<GLB>::WX);
    {
        int4 a = *reinterpret_cast<const int4 *>(d + D_XLO), b = *reinterpret_cast<const int4 *>(d + D_XLO + 4);
        xo[0] = a.x; xo[1] = a.y; xo[2] = a.z; xo[3] = a.w; xo[4] = b.x; xo[5] = b.y; xo[6] = b.z;
    }
    if (WREG) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            const float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
            const float t4[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int l = 0; l < TR; ++l) wx[pw][l] = t4[l];
        }
    }
    float2 acc[4][PW];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) acc[q][pw] = make_float2(0.f, 0.f);

    const int p0 = d[D_Y0] >> 1, p1 = (d[D_Y1] + 1) >> 1;
    const unsigned char *phr = reinterpret_cast<const unsigned char *>(d + D_PHR);
    const float2 *tile2 = reinterpret_cast<const float2 *>(tile_c);
#pragma unroll 1
    if (GLB) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) xo[pw] *= xs;
    }
    for (int p = p0; p < p1; ++p) {
        const float2 *row = tile2 + (size_t)p * W * xs;
        float2 r[PW];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            float2 t = make_float2(0.f, 0.f);
            if (WREG) {
#pragma unroll
                for (int l = 0; l < T; ++l) t = __ffma2_rn(bcast2(wx[pw][l]), row[xo[pw] + l * xs], t);
            } else {
                const float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
                const float4 b = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
                float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
                if (T > 8) c = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 8);
                const float t12[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
#pragma unroll
                for (int l = 0; l < T; ++l) t = __ffma2_rn(bcast2(t12[l]), row[xo[pw] + l * xs], t);
            }
            r[pw] = t;
        }
        const float4 *wq = wyd + (p - p0) * 4;             // rows 2p (wq[0..1]) and 2p+1 (wq[2..3])
        const float4 e0 = wq[0], e1 = wq[1], o0 = wq[2], o1 = wq[3];
        const float2 we[4] = {make_float2(e0.x, e0.y), make_float2(e0.z, e0.w), make_float2(e1.x, e1.y),
                              make_float2(e1.z, e1.w)};
        const float2 wo[4] = {make_float2(o0.x, o0.y), make_float2(o0.z, o0.w), make_float2(o1.x, o1.y),
                              make_float2(o1.z, o1.w)};
        // only the output-row pairs q whose bins (2q, 2q + 1) meet this row pair: byte p - p0 of D_PHR lists them as
        // first | count << 4 (a contiguous range, usually 1-2 bins of 7) -- everywhere else the weights are zero.  The
        // branches are warp-uniform; the dense form (56 FFMA2 per pair, no branch) was a fifth of the kernel.
        const int code = phr[p - p0];
        const int qlo = (code & 15) >> 1, qhi = ((code & 15) + (code >> 4) - 1) >> 1;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q >= qlo && q <= qhi) {
#pragma unroll
                for (int pw = 0; pw < PW; ++pw) {
                    acc[q][pw] = __ffma2_rn(bcast2(r[pw].x), we[q], acc[q][pw]);
                    acc[q][pw] = __ffma2_rn(bcast2(r[pw].y), wo[q], acc[q][pw]);
                }
            }
    }
    if (elect_one()) bulk_wait_read<0>();            // the previous bulk store has drained this stage
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            stage_c[(2 * q) * PW + pw] = acc[q][pw].x;
            if (q < 3) stage_c[(2 * q + 1) * PW + pw] = acc[q][pw].y;
        }
}

// The warp's dense y-weight table for one ROI: wyd[(y - 2 p0) * 8 + ph] = weight of tile row y in output row
// ph (0 where row y is outside the bin's window; word 7 of a row is 0, it feeds the unused half of acc[3]).
template <bool WIDE>
__device__ __forceinline__ void build_wyd(float *wyd, const int *__restrict__ d, int lane) {
    constexpr int MAXT = DescL<WIDE>::MT, WYP = DescL<WIDE>::WYP;
    const int p0 = d[D_Y0] >> 1, np = ((d[D_Y1] + 1) >> 1) - p0;
    float4 *w4 = reinterpret_cast<float4 *>(wyd);
    for (int i = lane; i < np * 4; i += 32) w4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    const float *dwy = reinterpret_cast<const float *>(d + D_WY);
    for (int t = lane; t < PH * MAXT; t += 32) {
        const int ph = t / MAXT, i = t - ph * MAXT;
        if (i < d[D_YN + ph]) {
            const int y = d[D_YLO + ph] + i;
            wyd[(y - 2 * p0) * 8 + ph] = dwy[ph * WYP + 1 + i];
        }
    }
    __syncwarp();
}

constexpr int FWD_MAX_WARPS = 11;

constexpr int FWD_GLOB_WARPS = 8;   // the global-memory variant trades warps for registers (64-bit addressing)
template <bool GLB>
__global__ void __launch_bounds__((GLB ? FWD_GLOB_WARPS : FWD_MAX_WARPS) * 32, 1)
roi_align_fwd_tile_kernel(const float *__restrict__ feat, const int *__restrict__ hdr,
                          const int *__restrict__ img_start, const int *__restrict__ descs,
                          const float *__restrict__ mask7, float *__restrict__ out, int B, int C, int H, int W,
                          int pitch, int wyd_floats) {
    constexpr int FWD_DESC_WORDS = DescL<GLB>::WORDS;          // GLB kernels read WIDE descriptors
    extern __shared__ __align__(128) float smem[];
    const int nw = blockDim.x >> 5;
    float *tile = smem;
    float *stage = smem + (GLB ? 0 : (size_t)CH * pitch);                        // [nw][1568]
    int *dslots = reinterpret_cast<int *>(stage + (size_t)nw * STAGE_FLOATS);   // [nw][2][FWD_DESC_WORDS]
    float *wyds = reinterpret_cast<float *>(dslots + (size_t)nw * 2 * FWD_DESC_WORDS);   // [nw][wyd_floats]
    __shared__ int s_next;                    // next ROI of the segment nobody has taken yet
    if (__ldg(hdr) != 0) return;              // rois not grouped by image: generic kernel runs

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = C / CH;
    const size_t HW = (size_t)H * W;
    const int s0 = __ldg(img_start), sB = __ldg(img_start + B);
    const long long U = (long long)nchunks * (sB - s0);     // (roi, chunk) units
    long long u = U * blockIdx.x / gridDim.x;
    const long long u_end = U * (blockIdx.x + 1) / gridDim.x;
    float *stage_w = stage + warp * STAGE_FLOATS;
    float *stage_c = stage_w + lane * NBIN;
    int *my_slots = dslots + warp * 2 * FWD_DESC_WORDS;
    float *my_wyd = wyds + (size_t)warp * wyd_floats;

    // descriptor prefetch: 672 B = 42 x 16 B per ROI, lanes 0..31 + lanes 0..9 again
    auto prefetch = [&](int roi, int slot) {
        const int *src = descs + (size_t)roi * FWD_DESC_WORDS;
        int *dst = my_slots + slot * FWD_DESC_WORDS;
        cp_async16(dst + lane * 4, src + lane * 4);
        if (lane < FWD_DESC_WORDS / 4 - 32) cp_async16(dst + (32 + lane) * 4, src + (32 + lane) * 4);
        cp_async_commit();
    };

    int b = 0;
    while (u < u_end) {
        // locate the tile (image b, channel chunk ch) that unit u falls into
        while (b < B && (long long)nchunks * (__ldg(img_start + b + 1) - s0) <= u) ++b;
        const int is = __ldg(img_start + b), nroi = __ldg(img_start + b + 1) - is;
        const long long base = (long long)nchunks * (is - s0);
        const int ch = (int)((u - base) / nroi);
        const int r0 = (int)((u - base) - (long long)ch * nroi);
        const int r1 = (int)min((long long)nroi, r0 + (u_end - u));
        const int c0 = ch * CH;

        int r = r0 + warp, slot = 0;
        if (r < r1) prefetch(is + r, 0);       // overlaps the tile load below
        const float *tile_c;
        if (GLB) {                             // feat = the channel-last pair copy [B][Hp/2][W][C][2]
            tile_c = feat + (((size_t)b * ((H + 1) >> 1) * W) * C + c0 + lane) * 2;
        } else {
            __syncthreads();                   // everyone is done with the previous tile (and has read s_next)
            if (tid == 0) s_next = r0 + nw;    // ROIs of the segment are handed out dynamically (their cost varies)
            load_tile(tile, feat + ((size_t)b * C + c0) * HW, H, W, pitch, tid, blockDim.x);
            __syncthreads();
            tile_c = tile + lane * pitch;
        }
        while (r < r1) {
            int rn = r + nw;
            if (!GLB) {
                if (lane == 0) rn = atomicAdd(&s_next, 1);
                rn = __shfl_sync(0xffffffffu, rn, 0);
            }
            if (rn < r1) { prefetch(is + rn, slot ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
            __syncwarp();
            const int *d = my_slots + slot * FWD_DESC_WORDS;
            const int roi = is + r;
            if ((d[D_FLAGY] | d[D_FLAGX]) == 0) {
                build_wyd<GLB>(my_wyd, d, lane);
                const float4 *wyd4 = reinterpret_cast<const float4 *>(my_wyd);
                switch (d[D_TX]) {
                    case 2: fwd_pairs<2, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                    case 3: fwd_pairs<3, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                    case 4: fwd_pairs<4, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                    case 6: fwd_pairs<6, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                    case 8: fwd_pairs<8, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                    default: fwd_pairs<GLB ? 12 : 8, GLB>(tile_c, W, C, d, stage_c, wyd4, lane); break;
                }
                fence_proxy_async_smem();
                __syncwarp();
                // MaskFuse prologue (mask7 != null): out is [K][2C][49], channels [0, C) = the pooled features,
                // [C, 2C) = the same times the ROI's 7 x 7 mask (lib/modeling/resnet50.py:131-134)
                const size_t orow = mask7 ? (size_t)roi * 2 * C : (size_t)roi * C;
                if (elect_one()) {
                    bulk_s2g(out + (orow + c0) * NBIN, stage_w, STAGE_FLOATS * 4);
                    bulk_commit();
                }
                if (mask7) {
                    float m[NBIN];
                    const float *mp = mask7 + (size_t)roi * NBIN;
#pragma unroll
                    for (int i = 0; i < NBIN; ++i) m[i] = __ldg(mp + i);
                    if (elect_one()) bulk_wait_read<0>();        // the stage has been read by the store above
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < NBIN; ++i) stage_c[i] *= m[i];
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (elect_one()) {
                        bulk_s2g(out + (orow + C + c0) * NBIN, stage_w, STAGE_FLOATS * 4);
                        bulk_commit();
                    }
                }
            }
            __syncwarp();                      // slot is re-filled two iterations from now
            slot ^= 1;
            r = rn;
        }
        u += r1 - r0;
    }
    if (elect_one()) bulk_wait_read<0>();
}

// ------------------------------------------------------------------------- window tiles: forward
// Window (b, oy, ox) x 32 channels of the map -> the row-pair interleaved smem tile (rows beyond H: zero).
__device__ __forceinline__ void load_window(float *tile, const float *__restrict__ src /* (b, c0) plane */, int H, int W,
                                            int oy, int ox, int wh, int ww, int pitch, int tid, int nthr) {
    const size_t HW = (size_t)H * W;
    const int area = wh * ww;
    if (((W | ox | ww) & 3) == 0) {
        const int q = ww >> 2, n4 = CH * wh * q;
        for (int e = tid; e < n4; e += nthr) {
            const int c = e / (wh * q), rem = e - c * wh * q, y = rem / q, x = (rem - y * q) << 2;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (oy + y < H) v = __ldg(reinterpret_cast<const float4 *>(src + c * HW + (size_t)(oy + y) * W + ox + x));
            float *dst = tile + c * pitch + tile_off(y, x, ww);
            dst[0] = v.x; dst[2] = v.y; dst[4] = v.z; dst[6] = v.w;
        }
    } else {
        for (int e = tid; e < CH * area; e += nthr) {
            const int c = e / area, rem = e - c * area, y = rem / ww, x = rem - y * ww;
            tile[c * pitch + tile_off(y, x, ww)] = oy + y < H ? __ldg(src + c * HW + (size_t)(oy + y) * W + ox + x) : 0.f;
        }
    }
}

// bucket (image * NW + window) that holds sorted position s: the last k with bucket[k] <= s
__device__ __forceinline__ int win_find_bucket(const int *__restrict__ bucket, int lo, int hi, int s) {
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(bucket + mid) <= s) lo = mid; else hi = mid;
    }
    return lo;
}

// Epilogue of a sub-ROI that is NOT the whole ROI: sum the virtual outputs (slots) of each bin and write the bins this
// sub-ROI owns.  stage_c: this lane's 49 virtual outputs [row slot][column slot]; lane = channel.
__device__ __forceinline__ void win_store_partial(float *stage_c, const int *d, float *__restrict__ out_c,
                                                  const float *__restrict__ mask, float *__restrict__ out2_c) {
    const unsigned ym = (unsigned)d[DW_YMAP], xm = (unsigned)d[DW_XMAP];
    const int ny = (ym >> 28) & 7, nx = (xm >> 28) & 7;
    for (int ys = 0; ys < ny; ++ys) {                       // column slots of one bin -> its first slot
        int first = 0;
        for (int xs = 1; xs < nx; ++xs) {
            if (((xm >> (4 * xs)) & 15u) == ((xm >> (4 * (xs - 1))) & 15u)) stage_c[ys * PW + first] += stage_c[ys * PW + xs];
            else first = xs;
        }
    }
    int firsty = 0;
    for (int ys = 1; ys < ny; ++ys) {                       // row slots of one bin -> its first slot
        if (((ym >> (4 * ys)) & 15u) == ((ym >> (4 * (ys - 1))) & 15u)) {
            for (int xs = 0; xs < nx; ++xs) stage_c[firsty * PW + xs] += stage_c[ys * PW + xs];
        } else firsty = ys;
    }
    for (int ys = 0; ys < ny; ++ys) {
        const int by = (ym >> (4 * ys)) & 15;
        if (ys > 0 && (int)((ym >> (4 * (ys - 1))) & 15u) == by) continue;
        for (int xs = 0; xs < nx; ++xs) {
            const int bx = (xm >> (4 * xs)) & 15;
            if (xs > 0 && (int)((xm >> (4 * (xs - 1))) & 15u) == bx) continue;
            const float v = stage_c[ys * PW + xs];
            out_c[by * PW + bx] = v;
            if (mask) out2_c[by * PW + bx] = v * __ldg(mask + by * PW + bx);
        }
    }
}

// Forward over WINDOW tiles (roi_window.cuh): units = (sub-ROI, channel chunk) in the order image -> chunk -> window ->
// sub-ROI, split evenly over the persistent CTAs; per (window, chunk) segment the CTA stages the window in shared
// memory and its warps sweep the segment's sub-ROIs with the same fwd_pairs as the whole-map tile kernel.
__global__ void __launch_bounds__(FWD_MAX_WARPS * 32, 1)
roi_align_fwd_win_kernel(const float *__restrict__ feat, const int *__restrict__ bucket, const int *__restrict__ descs,
                         const float *__restrict__ mask7, float *__restrict__ out, int B, int C, int H, int W,
                         WinGeom g, int pitch, int wyd_floats) {
    extern __shared__ __align__(128) float smem[];
    const int nw = blockDim.x >> 5;
    float *tile = smem;
    float *stage = smem + (size_t)CH * pitch;                                    // [nw][1568]
    int *dslots = reinterpret_cast<int *>(stage + (size_t)nw * STAGE_FLOATS);   // [nw][2][DESC_WORDS]
    float *wyds = reinterpret_cast<float *>(dslots + (size_t)nw * 2 * DESC_WORDS);
    __shared__ int s_next;                     // next sub-ROI of the segment nobody has taken yet

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = C / CH, NW = g.nwy * g.nwx;
    const size_t HW = (size_t)H * W;
    const long long U = (long long)nchunks * __ldg(bucket + B * NW);
    long long u = U * blockIdx.x / gridDim.x;
    const long long u_end = U * (blockIdx.x + 1) / gridDim.x;
    float *stage_w = stage + warp * STAGE_FLOATS;
    float *stage_c = stage_w + lane * NBIN;
    int *my_slots = dslots + warp * 2 * DESC_WORDS;
    float *my_wyd = wyds + (size_t)warp * wyd_floats;

    auto prefetch = [&](int pos, int slot) {
        const int *src = descs + (size_t)pos * DESC_WORDS;
        int *dst = my_slots + slot * DESC_WORDS;
        cp_async16(dst + lane * 4, src + lane * 4);
        if (lane < DESC_WORDS / 4 - 32) cp_async16(dst + (32 + lane) * 4, src + (32 + lane) * 4);
        cp_async_commit();
    };

    int b = 0;
    while (u < u_end) {
        while (b < B && (long long)nchunks * __ldg(bucket + (b + 1) * NW) <= u) ++b;
        const int ib0 = __ldg(bucket + b * NW), nit = __ldg(bucket + (b + 1) * NW) - ib0;
        const long long base = (long long)nchunks * ib0;
        const int ch = (int)((u - base) / nit);
        const int s0 = ib0 + (int)((u - base) - (long long)ch * nit);          // sorted position of the first unit
        const int k = win_find_bucket(bucket, b * NW, (b + 1) * NW, s0);
        const int s1 = (int)min((long long)__ldg(bucket + k + 1), s0 + (u_end - u));
        const int wy = (k - b * NW) / g.nwx, wx = (k - b * NW) - wy * g.nwx;
        const int oy = win_origin(wy, g.Hp, g.wh), ox = win_origin(wx, W, g.ww);
        const int c0 = ch * CH;

        // sub-ROIs are handed out dynamically (their cost varies 10x with their size: with a fixed stride the warps
        // reached the barrier of the next window load far apart -- 18 % of the samples at VGG-16 size)
        int r = s0 + warp, slot = 0;
        if (r < s1) prefetch(r, 0);            // overlaps the window load below
        __syncthreads();                       // everyone is done with the previous window (and has read s_next)
        if (tid == 0) s_next = s0 + nw;
        load_window(tile, feat + ((size_t)b * C + c0) * HW, H, W, oy, ox, g.wh, g.ww, pitch, tid, blockDim.x);
        __syncthreads();
        const float *tile_c = tile + lane * pitch;
        while (r < s1) {
            int rn = 0;
            if (lane == 0) rn = atomicAdd(&s_next, 1);
            rn = __shfl_sync(0xffffffffu, rn, 0);
            if (rn < s1) { prefetch(rn, slot ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
            __syncwarp();
            const int *d = my_slots + slot * DESC_WORDS;
            const int roi = d[DW_ROI];
            build_wyd<false>(my_wyd, d, lane);
            const float4 *wyd4 = reinterpret_cast<const float4 *>(my_wyd);
            switch (d[D_TX]) {
                case 2: fwd_pairs<2, false>(tile_c, g.ww, C, d, stage_c, wyd4, lane); break;
                case 3: fwd_pairs<3, false>(tile_c, g.ww, C, d, stage_c, wyd4, lane); break;
                case 4: fwd_pairs<4, false>(tile_c, g.ww, C, d, stage_c, wyd4, lane); break;
                case 6: fwd_pairs<6, false>(tile_c, g.ww, C, d, stage_c, wyd4, lane); break;
                default: fwd_pairs<8, false>(tile_c, g.ww, C, d, stage_c, wyd4, lane); break;
            }
            const size_t orow = mask7 ? (size_t)roi * 2 * C : (size_t)roi * C;
            if (d[DW_FLAGS] & 1) {             // the sub-ROI is the whole ROI: one bulk store, as on the whole-map path
                fence_proxy_async_smem();
                __syncwarp();
                if (elect_one()) {
                    bulk_s2g(out + (orow + c0) * NBIN, stage_w, STAGE_FLOATS * 4);
                    bulk_commit();
                }
                if (mask7) {
                    float m[NBIN];
                    const float *mp = mask7 + (size_t)roi * NBIN;
#pragma unroll
                    for (int i = 0; i < NBIN; ++i) m[i] = __ldg(mp + i);
                    if (elect_one()) bulk_wait_read<0>();
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < NBIN; ++i) stage_c[i] *= m[i];
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (elect_one()) {
                        bulk_s2g(out + (orow + C + c0) * NBIN, stage_w, STAGE_FLOATS * 4);
                        bulk_commit();
                    }
                }
            } else {
                win_store_partial(stage_c, d, out + (orow + c0 + lane) * NBIN,
                                  mask7 ? mask7 + (size_t)roi * NBIN : nullptr, out + (orow + C + c0 + lane) * NBIN);
            }
            __syncwarp();                      // slot is re-filled two iterations from now
            slot ^= 1;
            r = rn;
        }
        u += s1 - s0;
    }
    if (elect_one()) bulk_wait_read<0>();
}

// ----------------------------------------------------------------------------- tile: backward
constexpr int WIN_TM_PAD = 8;       // window path: spare tensor-memory columns per tile row (bwd_pairs_win)
constexpr int NWB_DEFAULT = 16;     // consumer warps of the backward CTA; warp w owns row pairs
                                    // {y : (y >> 1) % 16 == w}  (D_OWN is computed for exactly this map)
constexpr int NBR = 4;              // ROIs per ring slot: one full/empty barrier round per 4 ROIs
constexpr int NS = 3;               // ring slots
// tensor-memory variant: the tile's 128 KB of shared memory go to the ring -- as LARGER slots (16 ROIs per barrier
// round, 2 slots) rather than more of them: cfg2 backward 1.57 ms (4 ROIs x 3 slots) -> 1.49 (4 x 6) -> 1.385 (8 x 4)
// -> 1.34 (16 x 2)
constexpr int NS_TM_EXTRA = -1;
constexpr int NBR_TM_MUL = 4;
constexpr int SLOT_FLOATS = NBR * (STAGE_FLOATS + DESC_WORDS);
// fused MaskFuse backward: two gradient blocks per ROI (d/d pooled, d/d pooled*mask)
// and the ROI's 7 x 7 mask (padded to 52 floats = 208 B so that it can travel by cp.async.bulk); the owners fold
// g + g2 * mask while they read the gradient in their y pass
constexpr int MASK_PAD = 52;
constexpr int NBR_F = 2, NS_F = 3;
constexpr int SLOT_FLOATS_F = NBR_F * (2 * STAGE_FLOATS + DESC_WORDS + MASK_PAD);

// One ROI x 32 channels x the row pairs this warp owns.  Per owned pair p:
//   y pass: r[pw] = sum_ph (wy[ph][2p], wy[ph][2p+1]) * g[ph][pw]   over the bins D_PHR lists for the pair
//   x pass: (t[2p][xo+l], t[2p+1][xo+l]) += wx[pw][l] * r[pw]       7T x (LDS.64, FFMA2, STS.64)
// FUSED (MaskFuse prologue): the gradient of the pooled value is g[ph][pw] + g2[ph][pw] * m[ph][pw] with g2 the
// gradient block of the masked copy (STAGE_FLOATS further on in the slot) and m the ROI's 7 x 7 mask (smem).
// tensor-memory accessors of the backward's TM variant: lane = channel, 2 columns = (g[2p][x], g[2p+1][x])
__device__ __forceinline__ float2 tm_ld2(uint32_t taddr) {
    uint32_t a, b;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "r"(taddr) : "memory");
    return make_float2(__uint_as_float(a), __uint_as_float(b));
}
__device__ __forceinline__ void tm_st2(uint32_t taddr, float2 v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__float_as_uint(v.x)),
                 "r"(__float_as_uint(v.y))
                 : "memory");
}
// N column pairs (row 2p, row 2p + 1) starting at taddr
template <int N>
__device__ __forceinline__ void tm_ld_n(uint32_t taddr, float2 *v) {
    static_assert(N == 1 || N == 2 || N == 4 || N == 8, "tcgen05.ld.32x32b shapes");
    uint32_t *u = reinterpret_cast<uint32_t *>(v);
    if constexpr (N == 1)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(u[0]), "=r"(u[1]) : "r"(taddr) : "memory");
    else if constexpr (N == 2)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "r"(taddr) : "memory");
    else if constexpr (N == 4)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                     : "r"(taddr) : "memory");
    else
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
                       "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                     : "r"(taddr) : "memory");
}
template <int N>
__device__ __forceinline__ void tm_st_n(uint32_t taddr, const float2 *v) {
    const uint32_t *u = reinterpret_cast<const uint32_t *>(v);
    if constexpr (N == 1)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(u[0]), "r"(u[1]) : "memory");
    else if constexpr (N == 2)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(u[0]), "r"(u[1]),
                     "r"(u[2]), "r"(u[3]) : "memory");
    else if constexpr (N == 4)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(u[0]),
                     "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
    else
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                     ::"r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]),
                     "r"(u[9]), "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]) : "memory");
}
// the T-wide column window of a bin: T = 2, 4, 8 one access, T = 3 and 6 two (a power of two and its half)
template <int T>
__device__ __forceinline__ void tm_ld_win(uint32_t taddr, float2 *v) {
    if constexpr (T == 3) { tm_ld_n<2>(taddr, v); tm_ld_n<1>(taddr + 4u, v + 2); }
    else if constexpr (T == 6) { tm_ld_n<4>(taddr, v); tm_ld_n<2>(taddr + 8u, v + 4); }
    else tm_ld_n<T>(taddr, v);
}
template <int T>
__device__ __forceinline__ void tm_st_win(uint32_t taddr, const float2 *v) {
    if constexpr (T == 3) { tm_st_n<2>(taddr, v); tm_st_n<1>(taddr + 4u, v + 2); }
    else if constexpr (T == 6) { tm_st_n<4>(taddr, v); tm_st_n<2>(taddr + 8u, v + 4); }
    else tm_st_n<T>(taddr, v);
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// TM: the gradient tile lives in TENSOR MEMORY instead of shared memory (tmem_w = first column of this warp's
// region, pair p of the warp at columns 2 W (p / NW) ..): the x pass becomes tcgen05.ld / FFMA2 / tcgen05.st.
// tools/micro/tmem_rmw.cu: this read-modify-write pattern runs at 98 B/clk/SM in tensor memory against the 64 B/clk
// of shared memory (128 B/clk port, read + write), and the port stays free for the y pass.
template <int T, bool XINC, bool FUSED, int NW, bool TM = false>
__device__ __forceinline__ void bwd_pairs(float *__restrict__ tile_c, int W, const int *d,
                                          const float *__restrict__ g, const float *__restrict__ m, int warp, int y0,
                                          int y1, uint32_t tmem_w = 0) {
    // column weights in registers -- except for the wide tap classes of the tensor-memory variant, whose 16-register
    // accesses leave no room for 56 weights: those read a bin's weights (two LDS.128, broadcast) when they need them
    constexpr bool WREG = !(TM && T > 4);
    float wx[PW][WREG ? T : 1];
    int xo[PW];
    const float *dwx = reinterpret_cast<const float *>(d + D_WX);
    const float *dwy = reinterpret_cast<const float *>(d + D_WY);
    const unsigned char *phr = reinterpret_cast<const unsigned char *>(d + D_PHR);
    {
        int4 a = *reinterpret_cast<const int4 *>(d + D_XLO), b = *reinterpret_cast<const int4 *>(d + D_XLO + 4);
        xo[0] = a.x; xo[1] = a.y; xo[2] = a.z; xo[3] = a.w; xo[4] = b.x; xo[5] = b.y; xo[6] = b.z;
    }
    if constexpr (WREG) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
            float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
            if (T > 4) b = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
            float t8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int l = 0; l < T; ++l) wx[pw][l] = t8[l];
        }
    }
    float2 *tile2 = reinterpret_cast<float2 *>(tile_c);
    const int pb = y0 >> 1, p1 = (y1 + 1) >> 1;
    // first owned pair >= pb: pairs p with p % NW == warp
    int p = pb + ((warp - pb) & (NW - 1));
#pragma unroll 1
    for (; p < p1; p += NW) {
        float2 r[PW];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) r[pw] = make_float2(0.f, 0.f);
        const int code = phr[p - pb];
        const int ph_end = (code & 15) + (code >> 4);
#pragma unroll 1
        for (int ph = code & 15; ph < ph_end; ++ph) {
            const int dd = 2 * p - d[D_YLO + ph];    // window index of row 2p, in [-1, yn): padded weights
            const float2 w = make_float2(dwy[ph * WYP + dd + 1], dwy[ph * WYP + dd + 2]);
            const float *gp = g + ph * PW;
#pragma unroll
            for (int pw = 0; pw < PW; ++pw) {
                float gv = gp[pw];
                if (FUSED) gv = fmaf(gp[STAGE_FLOATS + pw], m[ph * PW + pw], gv);
                r[pw] = __ffma2_rn(bcast2(gv), w, r[pw]);
            }
        }
        if (TM) {
            // whole-window accesses: the T columns x 2 rows of a bin are ONE (T = 3, 6: two) tensor-memory load and
            // store, addressed off one base per bin.  (Per-tap .x2 accesses cost an R2UR per access on top of the
            // LDTM / STTM: the address has to sit in a uniform register, and ptxas re-materialises it at every use --
            // R2UR was 12 % of the issued instructions of this issue-bound kernel.)
            const uint32_t trow = tmem_w + (uint32_t)((p / NW) * W) * 2u;
            if (XINC) {
                // descriptor flag 3: bins p and p + 3 never share a column -> three groups, each loaded, updated and
                // stored as a whole (T <= 4), 6 waits per row pair
#pragma unroll
                for (int g0 = 0; g0 < 3; ++g0) {
                    if (T <= 4) {
                        float2 v[3][T];
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                            if (g0 + 3 * i < PW) tm_ld_win<T>(trow + 2u * (uint32_t)xo[g0 + 3 * i], v[i]);
                        tm_wait_ld();
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            const int pw = g0 + 3 * i;
                            if (pw < PW) {
#pragma unroll
                                for (int l = 0; l < T; ++l) v[i][l] = __ffma2_rn(bcast2(wx[pw][l]), r[pw], v[i][l]);
                                tm_st_win<T>(trow + 2u * (uint32_t)xo[pw], v[i]);
                            }
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            const int pw = g0 + 3 * i;
                            if (pw < PW) {
                                float2 v[T];
                                tm_ld_win<T>(trow + 2u * (uint32_t)xo[pw], v);
                                const float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
                                const float4 b = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
                                const float w8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                                tm_wait_ld();
#pragma unroll
                                for (int l = 0; l < T; ++l) v[l] = __ffma2_rn(bcast2(w8[l]), r[pw], v[l]);
                                tm_st_win<T>(trow + 2u * (uint32_t)xo[pw], v);
                            }
                        }
                    }
                    tm_wait_st();                       // the next group (and the next ROI) may read these columns
                }
            } else {
#pragma unroll
                for (int pw = 0; pw < PW; ++pw) {
                    float2 v[T];
                    tm_ld_win<T>(trow + 2u * (uint32_t)xo[pw], v);
                    float w8[8];
                    if constexpr (WREG) {
#pragma unroll
                        for (int l = 0; l < T; ++l) w8[l] = wx[pw][l];
                    } else {
                        const float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
                        const float4 b = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
                        w8[0] = a.x; w8[1] = a.y; w8[2] = a.z; w8[3] = a.w; w8[4] = b.x; w8[5] = b.y; w8[6] = b.z; w8[7] = b.w;
                    }
                    tm_wait_ld();
#pragma unroll
                    for (int l = 0; l < T; ++l) v[l] = __ffma2_rn(bcast2(w8[l]), r[pw], v[l]);
                    tm_st_win<T>(trow + 2u * (uint32_t)xo[pw], v);
                    tm_wait_st();                       // the next bin may alias these columns
                }
            }
            continue;
        }
        float2 *row = tile2 + p * W;
        if (XINC) {
            // descriptor flag 3: the windows of bins p and p + 3 are disjoint, so the bins of a group {0,3,6}, {1,4},
            // {2,5} can be loaded, updated and stored together; groups in this order = the order of the additions into
            // an element, the same as in the tensor-memory variant (the two are bit-identical)
#pragma unroll
            for (int g0 = 0; g0 < 3; ++g0) {
                float2 v[3][T];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    if (g0 + 3 * i < PW) {
#pragma unroll
                        for (int l = 0; l < T; ++l) v[i][l] = row[xo[g0 + 3 * i] + l];
                    }
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const int pw = g0 + 3 * i;
                    if (pw < PW) {
#pragma unroll
                        for (int l = 0; l < T; ++l) row[xo[pw] + l] = __ffma2_rn(bcast2(wx[pw][l]), r[pw], v[i][l]);
                    }
                }
                asm volatile("" ::: "memory");          // the next group may alias these columns
            }
        } else {
            // windows may coincide (tiny ROIs): bins strictly in program order; the T taps of one bin
            // are distinct columns
#pragma unroll
            for (int pw = 0; pw < PW; ++pw) {
                float2 v[T];
#pragma unroll
                for (int l = 0; l < T; ++l) v[l] = row[xo[pw] + l];
#pragma unroll
                for (int l = 0; l < T; ++l) row[xo[pw] + l] = __ffma2_rn(bcast2(wx[pw][l]), r[pw], v[l]);
                asm volatile("" ::: "memory");          // the next bin may alias these columns
            }
        }
    }
}

// WIN (window tiles, roi_window.cuh): the descriptor's 7 x 7 "bins" are SLOTS of a sub-ROI; slot (ys, xs) takes the
// gradient of bin (ymap[ys], xmap[xs]) of the ROI, and only the first nx column slots exist.  One instance for every
// tap class (the ten unrolled T x XINC instances of bwd_pairs made this kernel 118 KB of SASS: a third of all warp
// samples were instruction-fetch stalls).  The x pass goes SLOT BY SLOT: the 8 (T <= 4: 4) columns of a slot x 2 rows
// are one 16- (8-) column tensor-memory load, 8 (4) FFMA2 with the slot's weights (two LDS.128 from the descriptor),
// one store -- nx round trips per row pair instead of T rounds of 7 + 7 narrow accesses; consecutive slots may share
// columns, so each store is waited for.  W = columns of a tile row in tensor memory = window width + WIN_TM_PAD: a slot
// that starts fewer than 8 columns from the window's right edge runs into the (never drained, always zero) padding.
__device__ __forceinline__ void tm_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tm_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
                   "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
                 : "memory");
}
__device__ __forceinline__ void tm_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tm_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
                 "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

template <bool FUSED, int NW>
__device__ __forceinline__ void bwd_pairs_win(int W, const int *d, const float *__restrict__ g,
                                              const float *__restrict__ m, int warp, int y0, int y1, uint32_t tmem_w) {
    int xo[PW];
    const unsigned ymap = (unsigned)d[DW_YMAP], xmap = (unsigned)d[DW_XMAP];
    const int nx = (int)((xmap >> 28) & 7u);
    const bool narrow = d[D_TX] <= 4;                 // every slot has its weights in taps 0..3
    const float *dwx = reinterpret_cast<const float *>(d + D_WX);
    const float *dwy = reinterpret_cast<const float *>(d + D_WY);
    const unsigned char *phr = reinterpret_cast<const unsigned char *>(d + D_PHR);
    {
        int4 a = *reinterpret_cast<const int4 *>(d + D_XLO), b = *reinterpret_cast<const int4 *>(d + D_XLO + 4);
        xo[0] = a.x; xo[1] = a.y; xo[2] = a.z; xo[3] = a.w; xo[4] = b.x; xo[5] = b.y; xo[6] = b.z;
    }
    const int pb = y0 >> 1, p1 = (y1 + 1) >> 1;
    int p = pb + ((warp - pb) & (NW - 1));
#pragma unroll 1
    for (; p < p1; p += NW) {
        float2 r[PW];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) r[pw] = make_float2(0.f, 0.f);
        const int code = phr[p - pb];
        const int ph_end = (code & 15) + (code >> 4);
#pragma unroll 1
        for (int ph = code & 15; ph < ph_end; ++ph) {
            const int dd = 2 * p - d[D_YLO + ph];    // window index of row 2p, in [-1, yn): padded weights
            const float2 w = make_float2(dwy[ph * WYP + dd + 1], dwy[ph * WYP + dd + 2]);
            const int phb = (int)((ymap >> (4 * ph)) & 7u);
            const float *gp = g + phb * PW;
#pragma unroll
            for (int pw = 0; pw < PW; ++pw) {
                const int pwb = (int)((xmap >> (4 * pw)) & 7u);           // (unused slots: any valid column)
                float gv = gp[pwb];
                if (FUSED) gv = fmaf(gp[STAGE_FLOATS + pwb], m[phb * PW + pwb], gv);
                r[pw] = __ffma2_rn(bcast2(gv), w, r[pw]);
            }
        }
        const uint32_t trow = tmem_w + (uint32_t)((p / NW) * W) * 2u;
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            if (pw >= nx) break;
            const uint32_t ta = trow + 2u * (uint32_t)xo[pw];
            const float4 wa = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
            if (narrow) {
                uint32_t v[8];
                tm_ld8(ta, v);
                tm_wait_ld();
                const float wl[4] = {wa.x, wa.y, wa.z, wa.w};
#pragma unroll
                for (int l = 0; l < 4; ++l) {
                    const float2 t = __ffma2_rn(bcast2(wl[l]), r[pw],
                                                make_float2(__uint_as_float(v[2 * l]), __uint_as_float(v[2 * l + 1])));
                    v[2 * l] = __float_as_uint(t.x);
                    v[2 * l + 1] = __float_as_uint(t.y);
                }
                tm_st8(ta, v);
            } else {
                const float4 wb = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
                uint32_t v[16];
                tm_ld16(ta, v);
                tm_wait_ld();
                const float wl[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                for (int l = 0; l < 8; ++l) {
                    const float2 t = __ffma2_rn(bcast2(wl[l]), r[pw],
                                                make_float2(__uint_as_float(v[2 * l]), __uint_as_float(v[2 * l + 1])));
                    v[2 * l] = __float_as_uint(t.x);
                    v[2 * l + 1] = __float_as_uint(t.y);
                }
                tm_st16(ta, v);
            }
            tm_wait_st();                               // the next slot (and the next ROI) may share these columns
        }
    }
}

__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 4 floats added to global memory with one reduction (RED.E.ADD.F32x4)
__device__ __forceinline__ void red_add4(float *gptr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gptr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Persistent: one CTA per SM.  The (roi, channel-chunk) units of the whole batch are split evenly and
// contiguously over the CTAs (like the forward), so a CTA works through 1-3 tile SEGMENTS: zero the
// smem tile, apply the ROIs of the segment, add the tile to grad_feat with red.global.add.  grad_feat
// is zeroed beforehand and every tile is touched by at most TWO CTAs (a CTA's share is larger than one
// tile), i.e. each element is 0 + a (+ b): exact and independent of the order -> still bit-reproducible.
// FUSED (MaskFuse prologue): grad_out is [K][2C][49]; the effective gradient of the pooled features is
// g[c] + g[C + c] * mask[roi].  Both gradient blocks and the (padded) mask of a ROI travel in the ring slot;
// mask7 points at the PADDED masks [K][MASK_PAD] in the workspace.
// TM: the gradient tile is kept in tensor memory (see bwd_pairs); shared memory then only holds the ring.
// WIN (window tiles, roi_window.cuh): the tile is a wg.wh x wg.ww WINDOW of the map; img_start is the bucket table
// [B * NW + 1] of the sorted sub-ROI descriptors `descs`, the segments are (image, chunk, window, sub-ROI range), a
// sub-ROI's gradient block is its ROI's (descriptor word DW_ROI), and the tile is added to its window of grad_feat
// (windows overlap, so on this path the order of the global additions is not fixed).
// NCH = 2 (tensor-memory variant, whole map, C % 64 == 0): a CTA carries TWO 32-channel chunks at once.  Warp w owns
// row pair w of chunk 0 and row pair (w + 8) % 16 of chunk 1, so maps of 8 row pairs (HRNet, 16 x 16) keep all 16
// warps busy instead of 8 (the host selects it for those).  Both chunks of a ROI's gradient are contiguous in
// grad_out and travel with one bulk copy; a slot holds half as many ROIs.
template <bool FUSED, int NWB, bool TM, bool WIN = false, int NCH = 1>
__global__ void __launch_bounds__(NWB * 32, 1)
roi_align_bwd_tile_kernel(const float *__restrict__ grad_out, const int *__restrict__ hdr,
                          const int *__restrict__ img_start, const int *__restrict__ descs,
                          const float *__restrict__ mask7, float *__restrict__ grad_feat, int B, int C, int Hmap, int Wmap,
                          int pitch, WinGeom wg = WinGeom()) {
    const int H = WIN ? wg.wh : Hmap, W = WIN ? wg.ww : Wmap;          // tile rows / columns
    static_assert(NCH == 1 || (NCH == 2 && TM && !FUSED && !WIN && NWB == 16), "two chunks: whole-map tensor-memory variant");
    constexpr int NBR = (FUSED ? NBR_F : ::NBR) * (TM ? NBR_TM_MUL : 1) / NCH;   // ROIs per slot
    constexpr int NS = (FUSED ? NS_F : ::NS) + (TM ? NS_TM_EXTRA : 0);   // ring slots (TM: the tile's smem is free)
    constexpr int GSTRIDE = (FUSED ? 2 : NCH) * STAGE_FLOATS;             // gradient floats per ROI in a slot
    constexpr int SLOT_FLOATS = NBR * (GSTRIDE + DESC_WORDS + (FUSED ? MASK_PAD : 0));
    const int Cg = FUSED ? 2 * C : C;                         // channels of grad_out
    extern __shared__ __align__(128) float smem[];
    float *tile = smem;
    float *ring = smem + (TM ? 0 : (size_t)CH * pitch);      // [NS][NBR x grads | NBR x DESC_WORDS]
    __shared__ uint32_t tmem_slot;
    __shared__ int done_cnt[4];                                // LASTP: warps that have finished the batch in each slot
    constexpr bool LASTP = WIN;     // (measured on the whole-map path too: 1.18 -> 1.38 ms, the fast warps no longer run ahead)
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + (size_t)NS * SLOT_FLOATS);
    uint64_t *empty = full + NS;
    if (!WIN && __ldg(hdr) != 0) return;      // rois not grouped by image: the generic kernel does it all

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int HW = Hmap * Wmap, nchunks = C / (CH * NCH);
    const int NWIN = WIN ? wg.nwy * wg.nwx : 1;
    if (tid == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NWB); done_cnt[s] = 0; }
        fence_mbar_init();
    }
    if (TM && warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (TM) asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (TM) asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // TM: warp w reaches the TMEM lanes of its quarter (w % 4) only; lane = channel.  Its region holds the row
    // pairs it owns (p % NWB == w), 2 W columns each; the 4 warps of a quarter sit side by side.
    const int npw = (((H + 1) >> 1) + NWB - 1) / NWB;        // row pairs per warp
    const int TW = WIN ? W + WIN_TM_PAD : W;                 // columns of a tile row in tensor memory (bwd_pairs_win)
    const uint32_t tmem_cols_w = (uint32_t)(npw * TW * 2);
    const uint32_t tmem_w = TM ? tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(warp >> 2) * tmem_cols_w * NCH : 0u;

    const int s0 = __ldg(img_start), sB = __ldg(img_start + B * NWIN);
    const long long U = (long long)nchunks * (sB - s0);
    // Even split of the units only if a CTA's share covers the largest tile (then a tile is shared by
    // at most two CTAs and the merge is order-independent); otherwise whole tiles, round-robin.
    int maxroi = 0;
    if (!WIN)
        for (int i = 0; i < B; ++i) maxroi = max(maxroi, __ldg(img_start + i + 1) - __ldg(img_start + i));
    const bool split = WIN || U / gridDim.x >= maxroi;
    long long u = split ? U * blockIdx.x / gridDim.x : 0;
    const long long u_end = split ? U * (blockIdx.x + 1) / gridDim.x : 0;
    int tile_id = blockIdx.x;                 // whole-tile mode: tiles blockIdx.x, + gridDim.x, ...
    float *tile_c = tile + lane * pitch;
    int gb = 0;                               // batches consumed so far (all segments): slot / phase bookkeeping
    int issued = 0;                           // batches issued so far (producer thread only)
    int b = 0;
    int oy = 0, ox = 0;                       // WIN: origin of the segment's window
    while (true) {
        int is, nroi, ch, r0, r1;
        if (WIN) {
            if (u >= u_end) break;
            while (b < B && (long long)nchunks * (__ldg(img_start + (b + 1) * NWIN) - s0) <= u) ++b;
            const int ib0 = __ldg(img_start + b * NWIN), nit = __ldg(img_start + (b + 1) * NWIN) - ib0;
            const long long base = (long long)nchunks * (ib0 - s0);
            ch = (int)((u - base) / nit);
            const int p0 = ib0 + (int)((u - base) - (long long)ch * nit);        // sorted position of the first unit
            const int k = win_find_bucket(img_start, b * NWIN, (b + 1) * NWIN, p0);
            const int p1 = (int)min((long long)__ldg(img_start + k + 1), p0 + (u_end - u));
            const int wy = (k - b * NWIN) / wg.nwx, wx = (k - b * NWIN) - wy * wg.nwx;
            oy = win_origin(wy, wg.Hp, wg.wh);
            ox = win_origin(wx, Wmap, wg.ww);
            is = 0; r0 = p0; r1 = p1; nroi = p1 - p0;                             // "ROIs" = sorted positions
            u += p1 - p0;
        } else if (split) {
            if (u >= u_end) break;
            while (b < B && (long long)nchunks * (__ldg(img_start + b + 1) - s0) <= u) ++b;
            is = __ldg(img_start + b);
            nroi = __ldg(img_start + b + 1) - is;
            const long long base = (long long)nchunks * (is - s0);
            ch = (int)((u - base) / nroi);
            r0 = (int)((u - base) - (long long)ch * nroi);
            r1 = (int)min((long long)nroi, r0 + (u_end - u));
            u += r1 - r0;
        } else {
            if (tile_id >= B * nchunks) break;
            b = tile_id / nchunks;
            ch = tile_id - b * nchunks;
            tile_id += gridDim.x;
            is = __ldg(img_start + b);
            nroi = __ldg(img_start + b + 1) - is;
            r0 = 0;
            r1 = nroi;
            if (nroi == 0) continue;          // its slab stays zero
        }
        const int c0 = ch * CH * NCH;
        const int first_roi = is + r0, n = r1 - r0;
        const int nbatch = (n + NBR - 1) / NBR, gb0 = gb;

        if (TM) {
            for (uint32_t cc = 0; cc < tmem_cols_w * NCH; cc += 2) tm_st2(tmem_w + cc, make_float2(0.f, 0.f));
            tm_wait_st();
        } else {
            for (int e = tid; e < CH * pitch; e += NWB * 32) tile[e] = 0.f;
        }
        __syncthreads();

        // producer duty (lane 0 of warp 0): batch j of this segment (NBR consecutive ROIs: gradients +
        // descriptors) goes to slot (gb0 + j) % NS once every warp has released the batch that used
        // the slot before.  `must` = the batch warp 0 itself is about to read: blocking wait.
        auto issue_batch = [&](int gbatch) {              // one thread: the bulk copies of batch `gbatch` (global index)
            {
                const int s = gbatch % NS;
                float *slot = ring + (size_t)s * SLOT_FLOATS;
                const int first = (gbatch - gb0) * NBR, cnt = min(NBR, n - first);
                mbar_expect_tx(&full[s], (uint32_t)cnt * (GSTRIDE + DESC_WORDS + (FUSED ? MASK_PAD : 0)) * 4);
                int rois_j[NBR];
                if (WIN) {                    // the ROI of each sub-ROI: word DW_ROI of its descriptor (loads in flight together)
#pragma unroll
                    for (int j = 0; j < NBR; ++j)
                        rois_j[j] = j < cnt ? __ldg(descs + (size_t)(first_roi + first + j) * DESC_WORDS + DW_ROI) : 0;
                }
#pragma unroll
                for (int j = 0; j < NBR; ++j) {
                    if (j < cnt) {
                        const int roi = WIN ? rois_j[j] : first_roi + first + j;
                        const float *src = grad_out + ((size_t)roi * Cg + c0) * NBIN;
                        bulk_g2s(slot + j * GSTRIDE, src, NCH * STAGE_FLOATS * 4, &full[s]);   // NCH = 2: both chunks
                        if (FUSED)
                            bulk_g2s(slot + j * GSTRIDE + STAGE_FLOATS, src + (size_t)C * NBIN, STAGE_FLOATS * 4, &full[s]);
                        if (FUSED && WIN)
                            bulk_g2s(slot + NBR * (GSTRIDE + DESC_WORDS) + j * MASK_PAD, mask7 + (size_t)roi * MASK_PAD,
                                     MASK_PAD * 4, &full[s]);
                    }
                }
                bulk_g2s(slot + NBR * GSTRIDE, descs + (size_t)(first_roi + first) * DESC_WORDS,
                         (uint32_t)cnt * DESC_WORDS * 4, &full[s]);
                if (FUSED && !WIN)
                    bulk_g2s(slot + NBR * (GSTRIDE + DESC_WORDS), mask7 + (size_t)(first_roi + first) * MASK_PAD,
                             (uint32_t)cnt * MASK_PAD * 4, &full[s]);
            }
        };
        auto produce = [&](int want, int must) {
            while (issued < want && issued < gb0 + nbatch) {
                const int s = issued % NS;
                if (issued >= NS) {
                    const uint32_t par = ((issued / NS) - 1) & 1;
                    if (issued <= must) mbar_wait(&empty[s], par);
                    else if (!mbar_test(&empty[s], par)) break;
                }
                issue_batch(issued);
                ++issued;
            }
        };
        // LASTP: the warp that finishes a batch LAST refills its slot (batch + NS) at once.  With the refill left to
        // warp 0 (which owns the lightly loaded top row pair) its non-blocking look at the slot usually came too early,
        // and the batch was only fetched when warp 0 needed it itself: every batch then waited for its data.
        if (LASTP) {
            if (tid == 0)
                for (int j = 0; j < NS && j < nbatch; ++j) issue_batch(gb0 + j);      // all slots are free (CTA barrier above)
        } else if (tid == 0) produce(gb0 + NS, -1);

        for (int bi = 0; bi < nbatch; ++bi, ++gb) {
            if (!LASTP && tid == 0) produce(gb + NS, gb);
            const int s = gb % NS;
            mbar_wait(&full[s], (gb / NS) & 1);
            const float *slot = ring + (size_t)s * SLOT_FLOATS;
            const int cnt = min(NBR, n - bi * NBR);
            // which of the slot's ROIs touch a row pair of this warp (lane j looks at ROI j)
            const int *dbase = reinterpret_cast<const int *>(slot + NBR * GSTRIDE);
            bool mine = false;
            if (lane < cnt) {
                const int2 ff = *reinterpret_cast<const int2 *>(dbase + lane * DESC_WORDS + D_XINC);   // (xinc, own)
                const int own = NWB == 16 ? ff.y : (ff.y | (ff.y >> 8));       // D_OWN: bit (pair & 15)
                const int mybits = NCH == 2 ? (1 << warp) | (1 << ((warp + 8) & 15)) : 1 << warp;
                mine = (own & mybits) != 0 && dbase[lane * DESC_WORDS + D_FLAGX] == 0;   // (WIN: always 0)
            }
            unsigned todo = __ballot_sync(0xffffffffu, mine);
            while (todo) {
                const int j = __ffs(todo) - 1;
                todo &= todo - 1;
                const int *d = dbase + j * DESC_WORDS;
                const int2 yr = *reinterpret_cast<const int2 *>(d + D_Y0);
                const int y0 = yr.x, y1 = yr.y;
                const float *g = slot + j * GSTRIDE + lane * NBIN;
                const float *m = slot + NBR * (GSTRIDE + DESC_WORDS) + j * MASK_PAD;
                if constexpr (WIN) {
                    bwd_pairs_win<FUSED, NWB>(TW, d, g, m, warp, y0, y1, tmem_w);
                    continue;
                }
                const int own_j = NCH == 2 ? d[D_OWN] : 0;
#pragma unroll 1
                for (int cch = 0; cch < NCH; ++cch) {
                    // chunk 1 of the two-chunk variant: this warp stands in for warp (w + 8) % 16 of the one-chunk layout
                    const int vw = cch ? (warp + 8) & 15 : warp;
                    if (NCH == 2 && !((own_j >> vw) & 1)) continue;
                    const float *gc = g + cch * STAGE_FLOATS;
                    const uint32_t tmem_c = tmem_w + (uint32_t)cch * tmem_cols_w;
                    const int T = d[D_TX];
                    if (d[D_XINC] == 3) {      // groups of bins with disjoint windows; otherwise bin by bin
                        switch (T) {
                            case 2: bwd_pairs<2, true, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 3: bwd_pairs<3, true, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 4: bwd_pairs<4, true, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 6: bwd_pairs<6, true, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            default: bwd_pairs<8, true, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                        }
                    } else {
                        switch (T) {
                            case 2: bwd_pairs<2, false, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 3: bwd_pairs<3, false, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 4: bwd_pairs<4, false, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            case 6: bwd_pairs<6, false, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                            default: bwd_pairs<8, false, FUSED, NWB, TM>(tile_c, W, d, gc, m, vw, y0, y1, tmem_c); break;
                        }
                    }
                }
            }
            __syncwarp();
            if (LASTP) {
                if (lane == 0) {
                    __threadfence_block();                   // this warp's reads of slot s are done
                    if (atomicAdd(&done_cnt[s], 1) == NWB - 1) {
                        done_cnt[s] = 0;
                        if (bi + NS < nbatch) {
                            fence_proxy_async_smem();
                            issue_batch(gb + NS);
                        }
                    }
                }
            } else if (lane == 0) mbar_arrive_cta(&empty[s]);       // this warp is done reading slot s
        }
        __syncthreads();

        // tile -> grad_feat (+=): the slab is zero or holds the other CTA's partial sum
        float *dst = grad_feat + ((size_t)b * C + c0) * HW;
        if (WIN) {
            // the window's rows [oy, oy + H) x columns [ox, ox + W) of the map; rows beyond the map are padding
            float *dl = dst + (size_t)lane * HW + (size_t)oy * Wmap + ox;
            const bool v4 = ((Wmap | ox | W) & 3) == 0;
            for (int pl = 0; pl < npw; ++pl) {
                const int pp = warp + NWB * pl, y = 2 * pp;
                if (y >= H || oy + y >= Hmap) break;
                const bool row1 = oy + y + 1 < Hmap;
                if (TM) {
                    const uint32_t trow = tmem_w + (uint32_t)(pl * TW) * 2u;
                    if (v4) {
                        for (int x = 0; x < W; x += 4) {
                            uint32_t v[8];
                            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                                         : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]),
                                           "=r"(v[6]), "=r"(v[7])
                                         : "r"(trow + 2u * (uint32_t)x)
                                         : "memory");
                            tm_wait_ld();
                            red_add4(dl + (size_t)y * Wmap + x, __uint_as_float(v[0]), __uint_as_float(v[2]),
                                     __uint_as_float(v[4]), __uint_as_float(v[6]));
                            if (row1)
                                red_add4(dl + (size_t)(y + 1) * Wmap + x, __uint_as_float(v[1]), __uint_as_float(v[3]),
                                         __uint_as_float(v[5]), __uint_as_float(v[7]));
                        }
                    } else {
                        for (int x = 0; x < W; ++x) {
                            const float2 v = tm_ld2(trow + 2u * (uint32_t)x);
                            tm_wait_ld();
                            atomicAdd(dl + (size_t)y * Wmap + x, v.x);
                            if (row1) atomicAdd(dl + (size_t)(y + 1) * Wmap + x, v.y);
                        }
                    }
                } else {
                    const float2 *row = reinterpret_cast<const float2 *>(tile_c) + pp * W;
                    for (int x = 0; x < W; ++x) {
                        const float2 v = row[x];
                        atomicAdd(dl + (size_t)y * Wmap + x, v.x);
                        if (row1) atomicAdd(dl + (size_t)(y + 1) * Wmap + x, v.y);
                    }
                }
            }
        } else if (TM) {
            // every warp drains its own row pairs: lane = channel, 8 columns = 4 x-positions x (row 2p, row 2p+1)
            for (int cch = 0; cch < NCH; ++cch) {
            float *dl = dst + ((size_t)cch * CH + lane) * HW;
            const int vw = cch ? (warp + 8) & 15 : warp;
            for (int pl = 0; pl < npw; ++pl) {
                const int pp = vw + NWB * pl, y = 2 * pp;
                if (y >= H) break;
                const uint32_t trow = tmem_w + (uint32_t)cch * tmem_cols_w + (uint32_t)(pl * W) * 2u;
                if ((W & 3) == 0) {
                    for (int x = 0; x < W; x += 4) {
                        uint32_t v[8];
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
                                       "=r"(v[7])
                                     : "r"(trow + 2u * (uint32_t)x)
                                     : "memory");
                        tm_wait_ld();
                        red_add4(dl + (size_t)y * W + x, __uint_as_float(v[0]), __uint_as_float(v[2]),
                                 __uint_as_float(v[4]), __uint_as_float(v[6]));
                        if (y + 1 < H)
                            red_add4(dl + (size_t)(y + 1) * W + x, __uint_as_float(v[1]), __uint_as_float(v[3]),
                                     __uint_as_float(v[5]), __uint_as_float(v[7]));
                    }
                } else {
                    for (int x = 0; x < W; ++x) {
                        const float2 v = tm_ld2(trow + 2u * (uint32_t)x);
                        tm_wait_ld();
                        atomicAdd(dl + (size_t)y * W + x, v.x);
                        if (y + 1 < H) atomicAdd(dl + (size_t)(y + 1) * W + x, v.y);
                    }
                }
            }
            }
        } else if ((W & 3) == 0) {
            for (int e = tid * 4; e < CH * HW; e += NWB * 32 * 4) {
                const int c = e / HW, rem = e - c * HW, y = rem / W, x = rem - y * W;
                const float *t = tile + c * pitch + tile_off(y, x, W);
                red_add4(dst + e, t[0], t[2], t[4], t[6]);
            }
        } else {
            for (int e = tid; e < CH * HW; e += NWB * 32) {
                const int c = e / HW, rem = e - c * HW, y = rem / W, x = rem - y * W;
                atomicAdd(dst + e, tile[c * pitch + tile_off(y, x, W)]);
            }
        }
        __syncthreads();
    }
    if (TM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
        }
    }
}

// ------------------------------------------------------------------- large maps: channel-last global copy
// NCHW -> pairs layout [B][Hp/2][W][C] of float2 = (f[2p][x], f[2p+1][x]) and back (fwd_pairs GLB comment).
__global__ void __launch_bounds__(256)
nchw_to_pairs_kernel(const float *__restrict__ src, float2 *__restrict__ dst, int C, int H, int W) {
    __shared__ float t0[32][33], t1[32][33];
    const int hp2 = (H + 1) >> 1;
    const int b = blockIdx.z / hp2, p = blockIdx.z - b * hp2;
    const int x0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int c = ty; c < 32; c += 8) {
        const int cc = c0 + c, x = x0 + tx;
        float a = 0.f, bb = 0.f;
        if (cc < C && x < W) {
            const float *r = src + (((size_t)b * C + cc) * H + 2 * p) * W + x;
            a = __ldg(r);
            if (2 * p + 1 < H) bb = __ldg(r + W);
        }
        t0[c][tx] = a;
        t1[c][tx] = bb;
    }
    __syncthreads();
    for (int x = ty; x < 32; x += 8) {
        const int xx = x0 + x, cc = c0 + tx;
        if (xx < W && cc < C) dst[(((size_t)b * hp2 + p) * W + xx) * C + cc] = make_float2(t0[tx][x], t1[tx][x]);
    }
}
__global__ void __launch_bounds__(256)
pairs_to_nchw_kernel(const float2 *__restrict__ src, float *__restrict__ dst, int C, int H, int W) {
    __shared__ float t0[32][33], t1[32][33];
    const int hp2 = (H + 1) >> 1;
    const int b = blockIdx.z / hp2, p = blockIdx.z - b * hp2;
    const int x0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int x = ty; x < 32; x += 8) {
        const int xx = x0 + x, cc = c0 + tx;
        float2 v = make_float2(0.f, 0.f);
        if (xx < W && cc < C) v = src[(((size_t)b * hp2 + p) * W + xx) * C + cc];
        t0[tx][x] = v.x;
        t1[tx][x] = v.y;
    }
    __syncthreads();
    for (int c = ty; c < 32; c += 8) {
        const int cc = c0 + c, x = x0 + tx;
        if (cc < C && x < W) {
            float *r = dst + (((size_t)b * C + cc) * H + 2 * p) * W + x;
            r[0] = t0[c][tx];
            if (2 * p + 1 < H) r[W] = t1[c][tx];
        }
    }
}

__device__ __forceinline__ void red_add2(float2 *gptr, float2 v) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(gptr), "f"(v.x), "f"(v.y) : "memory");
}

// Backward over the global pairs copy: one ROI x 32 channels x ALL its row pairs per warp; the x pass is a
// red.global.add.v2.f32 per tap (256 contiguous bytes per warp instruction).  Summation order across ROIs is
// not fixed, like the reference's atomicAdd backward (roi_align_kernel.cu:237-267).
template <int T, bool FUSED>
__device__ __forceinline__ void bwd_pairs_glob(float2 *__restrict__ base2, int W, int xs, const int *d,
                                               const float *__restrict__ g, const float *__restrict__ m) {
    // WIDE descriptors.  T <= 8: column weights in registers; T = 12 (bins of near-full-image ROIs on a 64-wide map):
    // read from the descriptor (smem) inside the loop, 84 registers would not fit
    constexpr int MAXT = DescL<true>::MT, WYP = DescL<true>::WYP;
    constexpr bool WREG = T <= 8;
    float wx[PW][WREG ? T : 1];
    int xo[PW];
    const float *dwx = reinterpret_cast<const float *>(d + DescL<true>::WX);
    const float *dwy = reinterpret_cast<const float *>(d + D_WY);
    const unsigned char *phr = reinterpret_cast<const unsigned char *>(d + D_PHR);
    {
        int4 a = *reinterpret_cast<const int4 *>(d + D_XLO), b = *reinterpret_cast<const int4 *>(d + D_XLO + 4);
        xo[0] = a.x * xs; xo[1] = a.y * xs; xo[2] = a.z * xs; xo[3] = a.w * xs;
        xo[4] = b.x * xs; xo[5] = b.y * xs; xo[6] = b.z * xs;
    }
    if (WREG) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
            float4 a = *reinterpret_cast<const float4 *>(dwx + pw * MAXT);
            float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
            if (T > 4) b = *reinterpret_cast<const float4 *>(dwx + pw * MAXT + 4);
            float t8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int l = 0; l < (WREG ? T : 1); ++l) wx[pw][l] = t8[l];
        }
    }
    const int pb = d[D_Y0] >> 1, p1 = (d[D_Y1] + 1) >> 1;
#pragma unroll 1
    for (int p = pb; p < p1; ++p) {
        float2 r[PW];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) r[pw] = make_float2(0.f, 0.f);
        const int code = phr[p - pb];
        const int ph_end = (code & 15) + (code >> 4);
#pragma unroll 1
        for (int ph = code & 15; ph < ph_end; ++ph) {
            const int dd = 2 * p - d[D_YLO + ph];
            const float2 w = make_float2(dwy[ph * WYP + dd + 1], dwy[ph * WYP + dd + 2]);
            const float *gp = g + ph * PW;
#pragma unroll
            for (int pw = 0; pw < PW; ++pw) {
                float gv = gp[pw];
                if (FUSED) gv = fmaf(gp[STAGE_FLOATS + pw], __ldg(m + ph * PW + pw), gv);
                r[pw] = __ffma2_rn(bcast2(gv), w, r[pw]);
            }
        }
        float2 *row = base2 + (size_t)p * W * xs;
#pragma unroll
        for (int pw = 0; pw < PW; ++pw)
#pragma unroll
            for (int l = 0; l < T; ++l) {
                const float wv = WREG ? wx[pw][WREG ? l : 0] : dwx[pw * MAXT + l];
                red_add2(row + xo[pw] + l * xs, make_float2(wv * r[pw].x, wv * r[pw].y));
            }
    }
}

constexpr int BWG_MAX_WARPS = 11;

template <bool FUSED>
__global__ void __launch_bounds__(BWG_MAX_WARPS * 32, 1)
roi_align_bwd_glob_kernel(const float *__restrict__ grad_out, const int *__restrict__ hdr,
                          const int *__restrict__ img_start, const int *__restrict__ descs,
                          const float *__restrict__ mask7, float *__restrict__ gradP, int B, int C, int H, int W) {
    constexpr int GST = FUSED ? 2 * STAGE_FLOATS : STAGE_FLOATS;     // gradient floats per (roi, chunk)
    constexpr int DESC_WORDS = DescL<true>::WORDS;                   // WIDE descriptors
    extern __shared__ __align__(128) float smem[];
    const int nw = blockDim.x >> 5;
    float *stages = smem;                                             // [nw][2][GST]
    int *dslots = reinterpret_cast<int *>(stages + (size_t)nw * 2 * GST);   // [nw][2][DESC_WORDS]
    if (__ldg(hdr) != 0) return;              // rois not grouped by image: the generic kernel does it all
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = C / CH, Cg = FUSED ? 2 * C : C;
    const int s0 = __ldg(img_start), sB = __ldg(img_start + B);
    const long long U = (long long)nchunks * (sB - s0);
    long long u = U * blockIdx.x / gridDim.x;
    const long long u_end = U * (blockIdx.x + 1) / gridDim.x;
    float *my_stage = stages + (size_t)warp * 2 * GST;
    int *my_slots = dslots + warp * 2 * DESC_WORDS;
    const int hp2 = (H + 1) >> 1;

    auto prefetch = [&](int roi, int c0, int slot) {
        const int *src = descs + (size_t)roi * DESC_WORDS;
        int *dst = my_slots + slot * DESC_WORDS;
        cp_async16(dst + lane * 4, src + lane * 4);
        if (lane < DESC_WORDS / 4 - 32) cp_async16(dst + (32 + lane) * 4, src + (32 + lane) * 4);
        const float *gs = grad_out + ((size_t)roi * Cg + c0) * NBIN;
        float *gd = my_stage + slot * GST;
        for (int i = lane; i < STAGE_FLOATS / 4; i += 32) {
            cp_async16(gd + i * 4, gs + i * 4);
            if (FUSED) cp_async16(gd + STAGE_FLOATS + i * 4, gs + (size_t)C * NBIN + i * 4);
        }
        cp_async_commit();
    };

    int b = 0;
    while (u < u_end) {
        while (b < B && (long long)nchunks * (__ldg(img_start + b + 1) - s0) <= u) ++b;
        const int is = __ldg(img_start + b), nroi = __ldg(img_start + b + 1) - is;
        const long long base = (long long)nchunks * (is - s0);
        const int ch = (int)((u - base) / nroi);
        const int r0 = (int)((u - base) - (long long)ch * nroi);
        const int r1 = (int)min((long long)nroi, r0 + (u_end - u));
        const int c0 = ch * CH;
        float2 *base2 = reinterpret_cast<float2 *>(gradP) + ((size_t)b * hp2 * W) * C + c0 + lane;

        int r = r0 + warp, slot = 0;
        if (r < r1) prefetch(is + r, c0, 0);
        while (r < r1) {
            const int rn = r + nw;
            if (rn < r1) { prefetch(is + rn, c0, slot ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
            __syncwarp();
            const int *d = my_slots + slot * DESC_WORDS;
            if ((d[D_FLAGY] | d[D_FLAGX]) == 0) {
                const float *g = my_stage + slot * GST + lane * NBIN;
                const float *m = FUSED ? mask7 + (size_t)(is + r) * NBIN : nullptr;
                switch (d[D_TX]) {
                    case 2: bwd_pairs_glob<2, FUSED>(base2, W, C, d, g, m); break;
                    case 3: bwd_pairs_glob<3, FUSED>(base2, W, C, d, g, m); break;
                    case 4: bwd_pairs_glob<4, FUSED>(base2, W, C, d, g, m); break;
                    case 6: bwd_pairs_glob<6, FUSED>(base2, W, C, d, g, m); break;
                    case 8: bwd_pairs_glob<8, FUSED>(base2, W, C, d, g, m); break;
                    default: bwd_pairs_glob<12, FUSED>(base2, W, C, d, g, m); break;
                }
            }
            __syncwarp();
            slot ^= 1;
            r = rn;
        }
        u += r1 - r0;
    }
}

// ------------------------------------------------------------------------------- generic path
struct Geom {
    int b, gh, gw;
    float ys, xs, bh, bw, count;
};
__device__ __forceinline__ Geom roi_geom(const float *__restrict__ r, float scale, int oh, int ow,
                                         int sr, int aligned) {
    Geom g;
    const float off = aligned ? .5f : 0.f;
    g.b = (int)r[0];
    float x1 = __fsub_rn(__fmul_rn(r[1], scale), off), y1 = __fsub_rn(__fmul_rn(r[2], scale), off);
    float x2 = __fsub_rn(__fmul_rn(r[3], scale), off), y2 = __fsub_rn(__fmul_rn(r[4], scale), off);
    float rw = __fsub_rn(x2, x1), rh = __fsub_rn(y2, y1);
    if (!aligned) { rw = fmaxf(rw, 1.f); rh = fmaxf(rh, 1.f); }
    g.xs = x1; g.ys = y1;
    g.bh = __fdiv_rn(rh, (float)oh);
    g.bw = __fdiv_rn(rw, (float)ow);
    g.gh = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rh, (float)oh));
    g.gw = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rw, (float)ow));
    float cnt = fmaxf((float)(g.gh * g.gw), 1.f);
    g.count = cnt;
    return g;
}
__device__ __forceinline__ bool corners(int H, int W, float y, float x, int &y0, int &y1, int &x0,
                                        int &x1, float &w00, float &w01, float &w10, float &w11) {
    if (y < -1.f || y > (float)H || x < -1.f || x > (float)W) return false;
    if (y <= 0.f) y = 0.f;
    if (x <= 0.f) x = 0.f;
    y0 = (int)y; x0 = (int)x;
    if (y0 >= H - 1) { y1 = y0 = H - 1; y = (float)y0; } else { y1 = y0 + 1; }
    if (x0 >= W - 1) { x1 = x0 = W - 1; x = (float)x0; } else { x1 = x0 + 1; }
    float ly = y - (float)y0, lx = x - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    w00 = hy * hx; w01 = hy * lx; w10 = ly * hx; w11 = ly * lx;
    return true;
}

// mode: 0 = every ROI; 1 = only ROIs the tile kernel skipped (flagged, or all if ungrouped)
// mask7 != null: the fused MaskFuse layout -- the ROI-side tensor is [K][2C][oh][ow] (second half = first half
// times the ROI's oh x ow mask)
template <bool BWD>
__global__ void roi_align_generic_kernel(const float *__restrict__ in, const float *__restrict__ rois,
                                         float *__restrict__ outp, const int *__restrict__ hdr,
                                         const int *__restrict__ descs, const float *__restrict__ mask7,
                                         const int *__restrict__ feat_hw, int mode, int B, int C, int H, int W, int K,
                                         int oh, int ow, float scale, int sr, int aligned,
                                         int desc_words = DESC_WORDS) {
    // mode 0: one CTA column per ROI.  mode 1 (leftover pass): 8 ROIs per CTA -- warp w checks ROI 8 blockIdx.x + w
    // (almost every one was done by the tile kernel: 8x fewer CTAs scheduled for nothing), then the WHOLE CTA works
    // through the ROIs that are left, one after the other (a VGG-size ROI with bins wider than 8 taps is 25 000
    // outputs x up to 100 samples: far too much for a single warp)
    __shared__ int s_todo;
    int todo = 1, kbase = blockIdx.x;
    if (mode == 1) {
        if (threadIdx.x == 0) s_todo = 0;
        __syncthreads();
        const int kw = blockIdx.x * 8 + (threadIdx.x >> 5);
        if ((threadIdx.x & 31) == 0 && kw < K) {
            bool left = true;
            if (__ldg(hdr) == 0) {
                const int *d = descs + (size_t)kw * desc_words;
                left = (__ldg(d + D_FLAGY) | __ldg(d + D_FLAGX)) != 0;
            }
            if (left) atomicOr(&s_todo, 1 << (threadIdx.x >> 5));
        }
        __syncthreads();
        todo = s_todo;
        kbase = blockIdx.x * 8;
    }
    for (; todo; todo &= todo - 1) {
    const int k = kbase + (mode == 1 ? __ffs(todo) - 1 : 0);
    const Geom g = roi_geom(rois + 5 * (size_t)k, scale, oh, ow, sr, aligned);
    const int per_roi = C * oh * ow;
    const bool valid_b = g.b >= 0 && g.b < B;
    // the border rule sees the image's extent (H_b, W_b); planes and rows are addressed on the canvas (H, W)
    const int Hb = valid_b ? img_extent(feat_hw, g.b, 0, H) : H, Wb = valid_b ? img_extent(feat_hw, g.b, 1, W) : W;
    const int e0 = mode == 1 ? threadIdx.x : blockIdx.y * blockDim.x + threadIdx.x;
    const int estep = mode == 1 ? blockDim.x : gridDim.y * blockDim.x;
    for (int e = e0; e < per_roi; e += estep) {
        const int pw = e % ow, ph = (e / ow) % oh, c = e / (ow * oh);
        const size_t oidx = mask7 ? (size_t)k * 2 * per_roi + e : (size_t)k * per_roi + e;
        const float mk = mask7 ? __ldg(mask7 + (size_t)k * oh * ow + ph * ow + pw) : 0.f;
        if (!valid_b) {
            if (!BWD) { outp[oidx] = 0.f; if (mask7) outp[oidx + per_roi] = 0.f; }
            continue;
        }
        const size_t plane = ((size_t)g.b * C + c) * H * W;
        float acc = 0.f;
        float top = BWD ? in[oidx] : 0.f;
        if (BWD && mask7) top = fmaf(in[oidx + per_roi], mk, top);
        for (int iy = 0; iy < g.gh; ++iy) {
            const float y = sample_coord(g.ys, g.bh, ph, iy, g.gh);
            for (int ix = 0; ix < g.gw; ++ix) {
                const float x = sample_coord(g.xs, g.bw, pw, ix, g.gw);
                int y0, y1, x0, x1; float a, b2, c2, d2;
                if (!corners(Hb, Wb, y, x, y0, y1, x0, x1, a, b2, c2, d2)) continue;
                if (BWD) {
                    float *p = outp + plane;
                    atomicAdd(p + y0 * W + x0, top * a / g.count);
                    atomicAdd(p + y0 * W + x1, top * b2 / g.count);
                    atomicAdd(p + y1 * W + x0, top * c2 / g.count);
                    atomicAdd(p + y1 * W + x1, top * d2 / g.count);
                } else {
                    const float *p = in + plane;
                    acc += a * __ldg(p + y0 * W + x0) + b2 * __ldg(p + y0 * W + x1) +
                           c2 * __ldg(p + y1 * W + x0) + d2 * __ldg(p + y1 * W + x1);
                }
            }
        }
        if (!BWD) {
            const float v = acc / g.count;
            outp[oidx] = v;
            if (mask7) outp[oidx + per_roi] = v * mk;
        }
    }
    }
}

// masks [K][n] -> [K][MASK_PAD] (zero padded) for the fused backward's bulk copies
__global__ void roi_mask_pad_kernel(const float *__restrict__ m, float *__restrict__ out, int K, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * MASK_PAD) return;
    const int k = i / MASK_PAD, j = i - k * MASK_PAD;
    out[i] = j < n ? m[(size_t)k * n + j] : 0.f;
}

// ------------------------------------------------------------------------------------- host
struct Plan {
    bool tile, glob;                 // glob: map too large for shared memory -> channel-last global copy
    bool win;                        // map too large for shared memory -> window tiles (roi_window.cuh), the default
    WinGeom wg;
    int win_pitch, win_wyd_floats, win_fwd_warps, win_seg_cap;     // win_seg_cap: sub-ROIs per ROI the workspace holds
    size_t smem_fwd_win;
    bool bwd_tm;                     // backward tile kernel keeps its gradient tile in tensor memory
    size_t smem_bwd_tm, smem_bwd_fused_tm;
    int pitch, fwd_warps, wyd_floats, glob_bwd_warps, glob_bwd_warps_fused;
    size_t smem_fwd, smem_bwd, smem_bwd_fused, smem_fwd_glob, smem_bwd_glob, smem_bwd_glob_fused;
};
static Plan make_plan(int C, int H, int W, int oh, int ow) {
    Plan p{};
    const int Hp = (H + 1) & ~1, words = Hp * W;       // rows padded to whole pairs
    p.pitch = ((words >> 1) & 1) ? words : words + 2;  // pitch / 2 odd: conflict-free 64-bit accesses, lane = channel
    p.wyd_floats = (Hp / 2) * 16;                      // dense y-weight table of one warp (forward)
    const size_t cap = (size_t)cim_max_smem_optin();
    // forward: as many warps (11 ... 4) as fit next to the tile: per warp one output stage, two
    // descriptor slots and the y-weight table
    const size_t per_warp = (size_t)STAGE_FLOATS * 4 + 2 * DESC_WORDS * 4 + (size_t)p.wyd_floats * 4;
    const size_t per_warp_wide = per_warp + 2 * (DESC_WORDS_MAX - DESC_WORDS) * 4;
    p.fwd_warps = FWD_MAX_WARPS;
    while (p.fwd_warps > 4 && (size_t)CH * p.pitch * 4 + p.fwd_warps * per_warp > cap) --p.fwd_warps;
    p.smem_fwd = (size_t)CH * p.pitch * 4 + p.fwd_warps * per_warp;
    p.smem_bwd = (size_t)CH * p.pitch * 4 + (size_t)NS * SLOT_FLOATS * 4 + 2 * NS * 8;
    p.smem_bwd_fused = (size_t)CH * p.pitch * 4 + (size_t)NS_F * SLOT_FLOATS_F * 4 + 2 * NS_F * 8;
    p.tile = oh == PH && ow == PW && (C % CH) == 0 && W >= MAXT && p.smem_fwd <= cap &&
             p.smem_bwd <= cap && p.smem_bwd_fused <= cap && (((size_t)CH * p.pitch * 4) % 16 == 0);
    // tensor-memory variant of the backward: 4 warps of a lane quarter x their row pairs x 2 W columns <= 512
    p.bwd_tm = p.tile && 4 * ((((H + 1) >> 1) + NWB_DEFAULT - 1) / NWB_DEFAULT) * W * 2 <= 512;
    p.smem_bwd_tm = (size_t)(NS + NS_TM_EXTRA) * NBR_TM_MUL * SLOT_FLOATS * 4 + 2 * (NS + NS_TM_EXTRA) * 8;
    p.smem_bwd_fused_tm = (size_t)(NS_F + NS_TM_EXTRA) * NBR_TM_MUL * SLOT_FLOATS_F * 4 + 2 * (NS_F + NS_TM_EXTRA) * 8;
    // large maps (VGG-16: 64 x 64): same sweeps over a channel-last copy in global memory
    p.smem_fwd_glob = FWD_GLOB_WARPS * per_warp_wide;
    const size_t bw = (size_t)2 * STAGE_FLOATS * 4 + 2 * DESC_WORDS_MAX * 4, bwf = bw + (size_t)2 * STAGE_FLOATS * 4;
    p.glob_bwd_warps = BWG_MAX_WARPS;
    p.glob_bwd_warps_fused = (int)std::min<size_t>(BWG_MAX_WARPS, cap / bwf);
    p.smem_bwd_glob = p.glob_bwd_warps * bw;
    p.smem_bwd_glob_fused = p.glob_bwd_warps_fused * bwf;
    p.glob = !p.tile && oh == PH && ow == PW && (C % CH) == 0 && W >= MAXT && H <= 512 && p.smem_fwd_glob <= cap &&
             p.smem_bwd_glob <= cap && p.glob_bwd_warps_fused >= 4;
    // window tiles: a WIN_DIM x WIN_DIM window of the map in the same smem tile, ROIs cut into sub-ROIs per window
    p.wg = win_geom(H, W);
    const int wwords = p.wg.wh * p.wg.ww;
    p.win_pitch = ((wwords >> 1) & 1) ? wwords : wwords + 2;
    p.win_wyd_floats = (p.wg.wh / 2) * 16;
    const size_t per_warp_win = (size_t)STAGE_FLOATS * 4 + 2 * DESC_WORDS * 4 + (size_t)p.win_wyd_floats * 4;
    p.win_fwd_warps = FWD_MAX_WARPS;
    while (p.win_fwd_warps > 4 && (size_t)CH * p.win_pitch * 4 + p.win_fwd_warps * per_warp_win > cap) --p.win_fwd_warps;
    p.smem_fwd_win = (size_t)CH * p.win_pitch * 4 + p.win_fwd_warps * per_warp_win;
    auto seg_max = [](int L, int wl) {           // most segments a ROI can need along an axis of L cells
        if (L <= wl) return 1;
        const int emax = L / 7 + 3, per = std::max(1, (wl - (WIN_G - 1)) / emax);
        return std::min(7, (7 + per - 1) / per);
    };
    p.win_seg_cap = std::min(16, seg_max(H, p.wg.wh) * seg_max(W, p.wg.ww));
    p.win = !p.tile && oh == PH && ow == PW && (C % CH) == 0 && W >= MAXT && H >= 2 && p.wg.nwy < (1 << WIN_KEYBITS) &&
            p.wg.nwx < (1 << WIN_KEYBITS) && p.smem_fwd_win <= cap && (((size_t)CH * p.win_pitch * 4) % 16 == 0) &&
            4 * (((p.wg.wh >> 1) + NWB_DEFAULT - 1) / NWB_DEFAULT) * (p.wg.ww + WIN_TM_PAD) * 2 <= 512;
    return p;
}

static int check_args(const void *a, const void *rois, const void *c, int B, int C, int H, int W, int K,
                      int oh, int ow, const void *ws, size_t ws_bytes) {
    if (!a || !c || (K > 0 && !rois)) return CIM_ERR_ARG;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || K < 0 || oh <= 0 || ow <= 0) return CIM_ERR_ARG;
    if ((long long)H * W > (1 << 24) || (long long)C * oh * ow > (1LL << 30)) return CIM_ERR_SHAPE;
    if (!ws || ws_bytes < cim_roi_align_workspace_bytes(K)) return CIM_ERR_WORKSPACE;
    if (!cim_aligned(ws, 16) || !cim_aligned(a, 16) || !cim_aligned(c, 16)) return CIM_ERR_ALIGN;
    return CIM_OK;
}

static RoiWs carve(void *ws, int B, int K) {
    RoiWs w;
    char *p = (char *)ws;
    w.hdr = (int *)p;
    w.img_start = (int *)(p + ws_img_off());
    w.desc = (int *)(p + ws_desc_off(B));
    w.maskpad = (float *)(p + ws_desc_off(4096) + (size_t)(K > 0 ? K : 0) * DESC_WORDS_MAX * 4);
    return w;
}

static int run_prep(const float *rois, const int *feat_hw, int B, int H, int W, int K, int oh, int ow, float scale,
                    int sr, int aligned, const RoiWs &w, bool wide, cudaStream_t st) {
    cudaMemsetAsync(w.hdr, 0, WS_HDR_BYTES + sizeof(int) * (size_t)(B + 1), st);
    if (K > 0) {
        int threads = 128, blocks = (2 * K + threads - 1) / threads;
        if (wide)
            roi_prep_kernel<true><<<blocks, threads, 0, st>>>(rois, feat_hw, K, B, H, W, oh, ow, scale, sr, aligned,
                                                              w.hdr, w.img_start, w.desc);
        else
            roi_prep_kernel<false><<<blocks, threads, 0, st>>>(rois, feat_hw, K, B, H, W, oh, ow, scale, sr, aligned,
                                                               w.hdr, w.img_start, w.desc);
    }
    return cim_launch_status();
}

}  // namespace

static size_t glob_copy_bytes(int B, int C, int H, int W) { return sizeof(float) * (size_t)B * C * ((H + 1) & ~1) * W; }
static size_t ws_glob_off(int K) { return (cim_roi_align_workspace_bytes(K) + 255) & ~(size_t)255; }

// window path: records, keys, bucket table and the sorted sub-ROI descriptors, at ws_glob_off(K)
static size_t a256(size_t n) { return (n + 255) & ~(size_t)255; }
static size_t win_ws_bytes(const Plan &p, int B, int K) {
    const size_t cap = (size_t)std::max(K, 1) * p.win_seg_cap, nb = (size_t)B * p.wg.nwy * p.wg.nwx;
    return a256((size_t)K * 8 * 4) + a256(((size_t)K + 1) * 4) + a256((size_t)K * 4 * 4) + 2 * a256(cap * 4) +
           a256((nb + 2) * 4) + a256(cap * DESC_WORDS * 4);
}
static WinWs carve_win(void *ws, const Plan &p, int B, int K) {
    const size_t cap = (size_t)std::max(K, 1) * p.win_seg_cap, nb = (size_t)B * p.wg.nwy * p.wg.nwx;
    char *q = (char *)ws + ws_glob_off(K);
    WinWs w;
    w.rec = (int *)q;        q += a256((size_t)K * 8 * 4);
    w.item_base = (int *)q;  q += a256(((size_t)K + 1) * 4);
    w.flags = (int *)q;      q += a256((size_t)K * 4 * 4);
    w.keys = (int *)q;       q += a256(cap * 4);
    w.slot = (int *)q;       q += a256(cap * 4);
    w.bucket = (int *)q;     q += a256((nb + 2) * 4);
    w.desc = (int *)q;
    w.cap = (int)std::min<size_t>(cap, 0x7fffffff);
    return w;
}
static bool use_win(const Plan &p, int B, int K, size_t ws_bytes) {
    return p.win && K > 0 && !(cim_get_debug_flags() & CIM_DBG_ROI_NO_WINDOWS) &&
           ws_bytes >= ws_glob_off(K) + win_ws_bytes(p, B, K);
}
static int run_prep_win(const float *rois, const int *feat_hw, int B, int H, int W, int K, float scale, int sr,
                        int aligned, const RoiWs &w, const WinWs &ww, const Plan &p, cudaStream_t st) {
    const int nb = B * p.wg.nwy * p.wg.nwx;
    cudaMemsetAsync(w.hdr, 0, WS_HDR_BYTES, st);
    cudaMemsetAsync(ww.bucket, 0, sizeof(int) * ((size_t)nb + 2), st);
    roi_win_plan_kernel<<<(2 * K + 127) / 128, 128, 0, st>>>(rois, feat_hw, K, B, H, W, scale, sr, aligned, ww);
    roi_win_scan_kernel<<<1, 1024, 0, st>>>(K, ww);
    roi_win_keys_kernel<<<(K + 127) / 128, 128, 0, st>>>(rois, K, p.wg.nwy * p.wg.nwx, p.wg.nwx, ww);
    roi_win_bucket_kernel<<<1, 1024, 0, st>>>(nb, ww);
    roi_win_place_kernel<<<nb, 256, 0, st>>>(K, ww);
    roi_win_emit_kernel<<<(2 * K + 127) / 128, 128, 0, st>>>(rois, feat_hw, K, H, W, scale, sr, aligned, ww);
    return cim_launch_status();
}

CIM_API size_t cim_roi_align_workspace_bytes_ex(int B, int C, int H, int W, int K, int oh, int ow) {
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || oh <= 0 || ow <= 0) return cim_roi_align_workspace_bytes(K);
    const Plan p = make_plan(C, H, W, oh, ow);
    size_t extra = 0;
    if (p.glob) extra = glob_copy_bytes(B, C, H, W);
    if (p.win) extra = std::max(extra, win_ws_bytes(p, B, K));
    return extra ? ws_glob_off(K) + extra : cim_roi_align_workspace_bytes(K);
}

CIM_API size_t cim_roi_align_workspace_bytes(int K) {
    // header + image ranges (up to 4096 images) + descriptors
    return WS_HDR_BYTES + 4097 * sizeof(int) + 64 + (size_t)(K > 0 ? K : 0) * (DESC_WORDS_MAX + MASK_PAD) * 4;
}

static int roi_fwd_impl(const float *feat, const float *rois, const int *feat_hw, const float *mask7, float *out, int B,
                        int C, int H, int W, int K, int oh, int ow, float scale, int sr, int aligned, void *ws,
                        size_t ws_bytes, cim_stream_t stream, bool prepared = false) {
    if (B > 4096) return CIM_ERR_SHAPE;
    if (!cim_aligned(feat_hw, 4)) return CIM_ERR_ALIGN;
    if (K == 0 && feat && B > 0 && C > 0 && H > 0 && W > 0 && oh > 0 && ow > 0) return CIM_OK;   // empty output
    int rc = check_args(feat, rois, out, B, C, H, W, K, oh, ow, ws, ws_bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const Plan p = make_plan(C, H, W, oh, ow);
    const RoiWs w = carve(ws, B, K);
    const int per_roi = C * oh * ow;
    dim3 ggrid((unsigned)K, (unsigned)min(64, (per_roi + 255) / 256));
    if (!p.tile && use_win(p, B, K, ws_bytes)) {
        const WinWs ww = carve_win(ws, p, B, K);
        if (!prepared && (rc = run_prep_win(rois, feat_hw, B, H, W, K, scale, sr, aligned, w, ww, p, st))) return rc;
        cudaFuncSetAttribute(roi_align_fwd_win_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_fwd_win);
        roi_align_fwd_win_kernel<<<cim_num_sms(), p.win_fwd_warps * 32, p.smem_fwd_win, st>>>(
            feat, ww.bucket, ww.desc, mask7, out, B, C, H, W, p.wg, p.win_pitch, p.win_wyd_floats);
        if ((rc = cim_launch_status())) return rc;
        // leftover pass: ROIs the window plan could not take (bins wider than WIN_MTB taps, batch index out of range)
        roi_align_generic_kernel<false><<<dim3((unsigned)((K + 7) / 8), 1), 256, 0, st>>>(
            feat, rois, out, w.hdr, ww.flags, mask7, feat_hw, 1, B, C, H, W, K, oh, ow, scale, sr, aligned, 4);
        return cim_launch_status();
    }
    const bool glob = !p.tile && p.glob && ws_bytes >= ws_glob_off(K) + glob_copy_bytes(B, C, H, W);
    if (!p.tile && !glob) {
        roi_align_generic_kernel<false><<<ggrid, 256, 0, st>>>(feat, rois, out, nullptr, nullptr, mask7, feat_hw, 0, B, C, H, W,
                                                               K, oh, ow, scale, sr, aligned);
        return cim_launch_status();
    }
    if (!prepared && (rc = run_prep(rois, feat_hw, B, H, W, K, oh, ow, scale, sr, aligned, w, glob, st))) return rc;
    const long long units = (long long)(C / CH) * K;
    const int grid = (int)min((long long)cim_num_sms(), units);
    if (glob) {
        float *featP = reinterpret_cast<float *>((char *)ws + ws_glob_off(K));
        dim3 cg((unsigned)((W + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)(B * ((H + 1) >> 1)));
        nchw_to_pairs_kernel<<<cg, 256, 0, st>>>(feat, reinterpret_cast<float2 *>(featP), C, H, W);
        if ((rc = cim_launch_status())) return rc;
        cudaFuncSetAttribute(roi_align_fwd_tile_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)p.smem_fwd_glob);
        roi_align_fwd_tile_kernel<true><<<grid, FWD_GLOB_WARPS * 32, p.smem_fwd_glob, st>>>(
            featP, w.hdr, w.img_start, w.desc, mask7, out, B, C, H, W, p.pitch, p.wyd_floats);
    } else {
        cudaFuncSetAttribute(roi_align_fwd_tile_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)p.smem_fwd);
        roi_align_fwd_tile_kernel<false><<<grid, p.fwd_warps * 32, p.smem_fwd, st>>>(
            feat, w.hdr, w.img_start, w.desc, mask7, out, B, C, H, W, p.pitch, p.wyd_floats);
    }
    if ((rc = cim_launch_status())) return rc;
    // leftover pass: one CTA per ROI, which exits at once unless the tile kernel skipped that ROI
    roi_align_generic_kernel<false><<<dim3((unsigned)((K + 7) / 8), 1), 256, 0, st>>>(
        feat, rois, out, w.hdr, w.desc, mask7, feat_hw, 1, B, C, H, W, K, oh, ow, scale, sr, aligned,
        glob ? DESC_WORDS_MAX : DESC_WORDS);
    return cim_launch_status();
}

static int roi_bwd_impl(const float *grad_out, const float *rois, const int *feat_hw, const float *mask7,
                        float *grad_feat, int B, int C, int H, int W, int K, int oh, int ow, float scale, int sr,
                        int aligned, void *ws, size_t ws_bytes, cim_stream_t stream, bool prepared = false) {
    if (B > 4096) return CIM_ERR_SHAPE;
    if (!cim_aligned(feat_hw, 4)) return CIM_ERR_ALIGN;
    if (K == 0 && grad_feat && B > 0 && C > 0 && H > 0 && W > 0) {                // no ROI: zero gradient
        cudaMemsetAsync(grad_feat, 0, sizeof(float) * (size_t)B * C * H * W, (cudaStream_t)stream);
        return cim_launch_status();
    }
    int rc = check_args(grad_out, rois, grad_feat, B, C, H, W, K, oh, ow, ws, ws_bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const Plan p = make_plan(C, H, W, oh, ow);
    const RoiWs w = carve(ws, B, K);
    const int per_roi = C * oh * ow;
    dim3 ggrid((unsigned)max(K, 1), (unsigned)min(64, (per_roi + 255) / 256));
    if (!p.tile && use_win(p, B, K, ws_bytes)) {
        const WinWs ww = carve_win(ws, p, B, K);
        if (!prepared && (rc = run_prep_win(rois, feat_hw, B, H, W, K, scale, sr, aligned, w, ww, p, st))) return rc;
        cudaMemsetAsync(grad_feat, 0, sizeof(float) * (size_t)B * C * H * W, st);
        const int grid = cim_num_sms();
        if (mask7) {
            roi_mask_pad_kernel<<<(K * MASK_PAD + 255) / 256, 256, 0, st>>>(mask7, w.maskpad, K, NBIN);
            if ((rc = cim_launch_status())) return rc;
            auto kern = roi_align_bwd_tile_kernel<true, NWB_DEFAULT, true, true>;
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bwd_fused_tm);
            kern<<<grid, NWB_DEFAULT * 32, p.smem_bwd_fused_tm, st>>>(grad_out, w.hdr, ww.bucket, ww.desc, w.maskpad,
                                                                       grad_feat, B, C, H, W, p.win_pitch, p.wg);
        } else {
            auto kern = roi_align_bwd_tile_kernel<false, NWB_DEFAULT, true, true>;
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bwd_tm);
            kern<<<grid, NWB_DEFAULT * 32, p.smem_bwd_tm, st>>>(grad_out, w.hdr, ww.bucket, ww.desc, nullptr, grad_feat, B,
                                                                C, H, W, p.win_pitch, p.wg);
        }
        if ((rc = cim_launch_status())) return rc;
        roi_align_generic_kernel<true><<<dim3((unsigned)((K + 7) / 8), 1), 256, 0, st>>>(
            grad_out, rois, grad_feat, w.hdr, ww.flags, mask7, feat_hw, 1, B, C, H, W, K, oh, ow, scale, sr, aligned, 4);
        return cim_launch_status();
    }
    const bool glob = !p.tile && p.glob && K > 0 && ws_bytes >= ws_glob_off(K) + glob_copy_bytes(B, C, H, W);
    if ((!p.tile && !glob) || K == 0) {
        cudaMemsetAsync(grad_feat, 0, sizeof(float) * (size_t)B * C * H * W, st);
        if (K > 0)
            roi_align_generic_kernel<true><<<ggrid, 256, 0, st>>>(grad_out, rois, grad_feat, nullptr, nullptr, mask7, feat_hw, 0,
                                                                  B, C, H, W, K, oh, ow, scale, sr, aligned);
        return cim_launch_status();
    }
    if (!prepared && (rc = run_prep(rois, feat_hw, B, H, W, K, oh, ow, scale, sr, aligned, w, glob, st))) return rc;
    // two chunks per CTA (see the kernel): tensor-memory variant, an even number of chunks, no fused mask, and maps of
    // at most 8 row pairs, where it is what keeps all 16 warps busy (HRNet 16 x 16 x 2048: 2.36 -> 1.74 ms).  On 16
    // row pairs it only rebalances the centre-heavy load and loses more to its smaller batches (8 ROIs per barrier
    // round): 2.54 against 2.36 ms for 16 images x 2000 proposals at 32 x 32 x 1024.
    const bool tm_on = p.bwd_tm && !(cim_get_debug_flags() & CIM_DBG_ROI_BWD_SMEM_TILE);
    const bool two_chunks = tm_on && !glob && !mask7 && (C % (2 * CH)) == 0 && H <= 16 && 16 * W <= 512 &&
                            !(cim_get_debug_flags() & CIM_DBG_ROI_BWD_ONE_CHUNK);
    const long long units = (long long)(C / (two_chunks ? 2 * CH : CH)) * K;
    const int grid = (int)min((long long)cim_num_sms(), units);
    if (glob) {
        // gradients accumulate (red.global.add) in the channel-last pairs copy, which is then written out as NCHW
        float *gradP = reinterpret_cast<float *>((char *)ws + ws_glob_off(K));
        cudaMemsetAsync(gradP, 0, glob_copy_bytes(B, C, H, W), st);
        if (mask7) {
            cudaFuncSetAttribute(roi_align_bwd_glob_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)p.smem_bwd_glob_fused);
            roi_align_bwd_glob_kernel<true><<<grid, p.glob_bwd_warps_fused * 32, p.smem_bwd_glob_fused, st>>>(
                grad_out, w.hdr, w.img_start, w.desc, mask7, gradP, B, C, H, W);
        } else {
            cudaFuncSetAttribute(roi_align_bwd_glob_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)p.smem_bwd_glob);
            roi_align_bwd_glob_kernel<false><<<grid, p.glob_bwd_warps * 32, p.smem_bwd_glob, st>>>(
                grad_out, w.hdr, w.img_start, w.desc, nullptr, gradP, B, C, H, W);
        }
        if ((rc = cim_launch_status())) return rc;
        dim3 cg((unsigned)((W + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)(B * ((H + 1) >> 1)));
        pairs_to_nchw_kernel<<<cg, 256, 0, st>>>(reinterpret_cast<const float2 *>(gradP), grad_feat, C, H, W);
        if ((rc = cim_launch_status())) return rc;
        roi_align_generic_kernel<true><<<dim3((unsigned)((K + 7) / 8), 1), 256, 0, st>>>(
            grad_out, rois, grad_feat, w.hdr, w.desc, mask7, feat_hw, 1, B, C, H, W, K, oh, ow, scale, sr, aligned,
            DESC_WORDS_MAX);
        return cim_launch_status();
    }
    cudaMemsetAsync(grad_feat, 0, sizeof(float) * (size_t)B * C * H * W, st);
    // 16 consumer warps, one row pair each.  (8 warps owning two pairs half a map apart balance the centre-heavy
    // row load better -- max / mean 1.06 instead of 1.21 on the synthetic proposals -- but lose more to the halved
    // thread-level parallelism: 2.10 ms against 1.81 ms at cfg2.)
    auto go = [&](auto kern, int nw, size_t smem, const float *mk) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<grid, nw * 32, smem, st>>>(grad_out, w.hdr, w.img_start, w.desc, mk, grad_feat, B, C, H, W, p.pitch,
                                          WinGeom());
    };
    // CIM_DBG_ROI_BWD_SMEM_TILE keeps the gradient tile in shared memory (A/B timing, tests)
    const bool tm = p.bwd_tm && !(cim_get_debug_flags() & CIM_DBG_ROI_BWD_SMEM_TILE);
    if (mask7) {
        roi_mask_pad_kernel<<<(K * MASK_PAD + 255) / 256, 256, 0, st>>>(mask7, w.maskpad, K, NBIN);
        if ((rc = cim_launch_status())) return rc;
        if (tm) go(roi_align_bwd_tile_kernel<true, NWB_DEFAULT, true>, NWB_DEFAULT, p.smem_bwd_fused_tm, w.maskpad);
        else go(roi_align_bwd_tile_kernel<true, NWB_DEFAULT, false>, NWB_DEFAULT, p.smem_bwd_fused, w.maskpad);
    } else {
        if (two_chunks) go(roi_align_bwd_tile_kernel<false, NWB_DEFAULT, true, false, 2>, NWB_DEFAULT, p.smem_bwd_tm, nullptr);
        else if (tm) go(roi_align_bwd_tile_kernel<false, NWB_DEFAULT, true>, NWB_DEFAULT, p.smem_bwd_tm, nullptr);
        else go(roi_align_bwd_tile_kernel<false, NWB_DEFAULT, false>, NWB_DEFAULT, p.smem_bwd, nullptr);
    }
    if ((rc = cim_launch_status())) return rc;
    roi_align_generic_kernel<true><<<dim3((unsigned)((K + 7) / 8), 1), 256, 0, st>>>(grad_out, rois, grad_feat, w.hdr, w.desc,
                                                                         mask7, feat_hw, 1, B, C, H, W, K, oh, ow, scale, sr,
                                                                         aligned);
    return cim_launch_status();
}

// Descriptors once for several calls on the same rois (forward + backward of one step share them): the same plan /
// layout decision as the _impl functions, which then skip their own prep launch.
CIM_API int cim_roi_align_prepare_ex(const float *rois, const int32_t *feat_hw, int B, int C, int H, int W, int K, int oh,
                                     int ow, float scale, int sr, int aligned, void *ws, size_t ws_bytes,
                                     cim_stream_t stream) {
    if (B > 4096) return CIM_ERR_SHAPE;
    if (K == 0) return CIM_OK;
    if (!rois || B <= 0 || C <= 0 || H <= 0 || W <= 0 || K < 0 || oh <= 0 || ow <= 0) return CIM_ERR_ARG;
    if ((long long)H * W > (1 << 24) || (long long)C * oh * ow > (1LL << 30)) return CIM_ERR_SHAPE;
    if (!ws || ws_bytes < cim_roi_align_workspace_bytes(K)) return CIM_ERR_WORKSPACE;
    if (!cim_aligned(ws, 16) || !cim_aligned(feat_hw, 4)) return CIM_ERR_ALIGN;
    const Plan p = make_plan(C, H, W, oh, ow);
    if (!p.tile && use_win(p, B, K, ws_bytes))
        return run_prep_win(rois, feat_hw, B, H, W, K, scale, sr, aligned, carve(ws, B, K), carve_win(ws, p, B, K), p,
                            (cudaStream_t)stream);
    const bool glob = !p.tile && p.glob && ws_bytes >= ws_glob_off(K) + glob_copy_bytes(B, C, H, W);
    if (!p.tile && !glob) return CIM_OK;                   // generic kernels: no descriptors
    return run_prep(rois, feat_hw, B, H, W, K, oh, ow, scale, sr, aligned, carve(ws, B, K), glob, (cudaStream_t)stream);
}

CIM_API int cim_roi_align_fwd_prepared_ex(const float *feat, const float *rois, const int32_t *feat_hw,
                                          const float *masks7, float *out, int B, int C, int H, int W, int K, int oh,
                                          int ow, float scale, int sr, int aligned, void *ws, size_t ws_bytes,
                                          cim_stream_t stream) {
    return roi_fwd_impl(feat, rois, feat_hw, masks7, out, B, C, H, W, K, oh, ow, scale, sr, aligned, ws, ws_bytes,
                        stream, true);
}

CIM_API int cim_roi_align_bwd_prepared_ex(const float *grad_out, const float *rois, const int32_t *feat_hw,
                                          const float *masks7, float *grad_feat, int B, int C, int H, int W, int K,
                                          int oh, int ow, float scale, int sr, int aligned, void *ws, size_t ws_bytes,
                                          cim_stream_t stream) {
    return roi_bwd_impl(grad_out, rois, feat_hw, masks7, grad_feat, B, C, H, W, K, oh, ow, scale, sr, aligned, ws,
                        ws_bytes, stream, true);
}

CIM_API int cim_roi_align_prepare(const float *rois, int B, int C, int H, int W, int K, int oh, int ow, float scale,
                                  int sr, int aligned, void *ws, size_t ws_bytes, cim_stream_t stream) {
    return cim_roi_align_prepare_ex(rois, nullptr, B, C, H, W, K, oh, ow, scale, sr, aligned, ws, ws_bytes, stream);
}

CIM_API int cim_roi_align_fwd_prepared(const float *feat, const float *rois, const float *masks7, float *out, int B,
                                       int C, int H, int W, int K, int oh, int ow, float scale, int sr, int aligned,
                                       void *ws, size_t ws_bytes, cim_stream_t stream) {
    return roi_fwd_impl(feat, rois, nullptr, masks7, out, B, C, H, W, K, oh, ow, scale, sr, aligned, ws, ws_bytes,
                        stream, true);
}

CIM_API int cim_roi_align_bwd_prepared(const float *grad_out, const float *rois, const float *masks7,
                                       float *grad_feat, int B, int C, int H, int W, int K, int oh, int ow,
                                       float scale, int sr, int aligned, void *ws, size_t ws_bytes,
                                       cim_stream_t stream) {
    return roi_bwd_impl(grad_out, rois, nullptr, masks7, grad_feat, B, C, H, W, K, oh, ow, scale, sr, aligned, ws,
                        ws_bytes, stream, true);
}

CIM_API int cim_roi_align_fwd(const float *feat, const float *rois, float *out, int B, int C, int H, int W,
                              int K, int oh, int ow, float scale, int sr, int aligned, void *ws,
                              size_t ws_bytes, cim_stream_t stream) {
    return roi_fwd_impl(feat, rois, nullptr, nullptr, out, B, C, H, W, K, oh, ow, scale, sr, aligned, ws, ws_bytes,
                        stream);
}

CIM_API int cim_roi_align_bwd(const float *grad_out, const float *rois, float *grad_feat, int B, int C, int H,
                              int W, int K, int oh, int ow, float scale, int sr, int aligned, void *ws,
                              size_t ws_bytes, cim_stream_t stream) {
    return roi_bwd_impl(grad_out, rois, nullptr, nullptr, grad_feat, B, C, H, W, K, oh, ow, scale, sr, aligned, ws,
                        ws_bytes, stream);
}

CIM_API int cim_roi_align_maskfuse_fwd(const float *feat, const float *rois, const float *masks7, float *out, int B,
                                       int C, int H, int W, int K, int oh, int ow, float scale, int sr, int aligned,
                                       void *ws, size_t ws_bytes, cim_stream_t stream) {
    if (!masks7 && K > 0) return CIM_ERR_ARG;
    return roi_fwd_impl(feat, rois, nullptr, masks7, out, B, C, H, W, K, oh, ow, scale, sr, aligned, ws, ws_bytes,
                        stream);
}

CIM_API int cim_roi_align_maskfuse_bwd(const float *grad_out, const float *rois, const float *masks7,
                                       float *grad_feat, int B, int C, int H, int W, int K, int oh, int ow,
                                       float scale, int sr, int aligned, void *ws, size_t ws_bytes,
                                       cim_stream_t stream) {
    if (!masks7 && K > 0) return CIM_ERR_ARG;
    return roi_bwd_impl(grad_out, rois, nullptr, masks7, grad_feat, B, C, H, W, K, oh, ow, scale, sr, aligned, ws,
                        ws_bytes, stream);
}

// Test hook (host only, no GPU): the window plan of roi_window.cuh evaluated on the CPU with the same
// __host__ __device__ code the prep kernels run.  All pointers are HOST memory.  Sub-ROI descriptors come out in ROI
// order (the device sorts them by window afterwards); key_out = window index wy * nwx + wx of each sub-ROI, flag_out[k]
// = 1 for ROIs the window path leaves to the generic kernel, geom_out = {Hp, wh, ww, nwy, nwx, WIN_G}.  feat_hw: host
// [B][2] image extents, clamped like the device's (NULL: the canvas).
// Returns the number of sub-ROIs, or a negative CIM_ERR_* code (CIM_ERR_WORKSPACE: more than `cap`).
CIM_API int cim_debug_roi_window_plan_ex(const float *rois, const int32_t *feat_hw, int K, int B, int H, int W,
                                         float scale, int sr, int aligned, int *desc_out, int *key_out, int cap,
                                         int *flag_out, int *geom_out) {
    if (!rois || !desc_out || !key_out || !flag_out || !geom_out || K < 0 || B <= 0 || H <= 0 || W < MAXT)
        return CIM_ERR_ARG;
    if (!cim_aligned(feat_hw, 4)) return CIM_ERR_ALIGN;
    const WinGeom g = win_geom(H, W);
    geom_out[0] = g.Hp; geom_out[1] = g.wh; geom_out[2] = g.ww; geom_out[3] = g.nwy; geom_out[4] = g.nwx;
    geom_out[5] = WIN_G;
    int n = 0;
    for (int k = 0; k < K; ++k) {
        const float *r = rois + 5 * (size_t)k;
        const int b = (int)r[0];
        flag_out[k] = 1;
        if (b < 0 || b >= B) continue;
        const AxisGeom ay = win_axis_geom(r, 0, 7, scale, sr, aligned), ax = win_axis_geom(r, 1, 7, scale, sr, aligned);
        const int Hb = img_extent(feat_hw, b, 0, H), Wb = img_extent(feat_hw, b, 1, W);
        AxisPlan py, px;
        win_axis_plan(ay, Hb, g.Hp, g.wh, g.nwy, py);
        win_axis_plan(ax, Wb, W, g.ww, g.nwx, px);
        flag_out[k] = (py.nseg == 0 || px.nseg == 0) ? 1 : 0;
        if (flag_out[k]) continue;
        const bool simple = py.nseg == 1 && px.nseg == 1 && py.nslots[0] == 7 && px.nslots[0] == 7;
        for (int sy = 0; sy < py.nseg; ++sy)
            for (int sx = 0; sx < px.nseg; ++sx) {
                if (n >= cap) return CIM_ERR_WORKSPACE;
                int *d = desc_out + (size_t)n * DESC_WORDS;
                for (int i = 0; i < DESC_WORDS; ++i) d[i] = 0;
                win_axis_emit(ay, py, sy, 0, Hb, g.Hp, g.wh, k, simple, d);
                win_axis_emit(ax, px, sx, 1, Wb, W, g.ww, k, simple, d);
                key_out[n] = py.wcoord[sy] * g.nwx + px.wcoord[sx];
                ++n;
            }
    }
    return n;
}

CIM_API int cim_debug_roi_window_plan(const float *rois, int K, int B, int H, int W, float scale, int sr, int aligned,
                                      int *desc_out, int *key_out, int cap, int *flag_out, int *geom_out) {
    return cim_debug_roi_window_plan_ex(rois, nullptr, K, B, H, W, scale, sr, aligned, desc_out, key_out, cap, flag_out,
                                        geom_out);
}
