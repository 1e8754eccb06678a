/*
 * cimhead.h -- C ABI of libcimhead.so: the B200 (sm_100a) implementation of the CIM
 * proposal-level hot path (ZechengLi19/CIM).
 *
 * Every entry point takes plain device pointers, sizes and scalars plus the CUDA stream to
 * launch on.  Contract (SURVEY.md section 8b):
 *   - the caller owns all memory (inputs, outputs, workspaces); the library never allocates,
 *     frees, retains or synchronises; it only enqueues kernels on `stream`;
 *   - re-entrant, no global mutable state (the reference calls its ops from one Python thread
 *     per device, lib/nn/parallel/parallel_apply.py:37-59);
 *   - return value: 0 on success, a negative CIM_ERR_* for bad arguments, or the positive
 *     cudaError_t of a failed launch.  Nothing is printed, nothing calls exit() (the legacy
 *     launchers do: lib/modeling/roi_xfrom/roi_align/src/roi_align_kernel.cu:135-139);
 *   - there is no CPU path.
 *
 * Each declaration cites the reference interface it replaces.
 *
 * Ragged batches (the _ex entry points of the scoring heads, mining, assignment and PCL_loss).  The images of a batch
 * may have different proposal counts.  Tensors keep their shapes: R is a capacity, and image b owns rows [0, n_b) of
 * its R rows, 0 < n_b <= R.  n_props is a device int32 [n_img] array of the n_b; NULL means n_b = R for every image,
 * and each entry point without _ex is its NULL case.  The library cannot validate device-side counts: the kernels
 * clamp every n_b to [1, R], so a count outside that range is well defined but not meaningful.  Contract:
 *   - no result of image b depends on its padding rows r >= n_b: not on x there (which must still be finite: the
 *     grad_weight product multiplies it by a zero dz, and 0 * NaN = NaN), not on the iou / asy map rows and columns
 *     >= n_b (anything, NaN included), not on mat there, not on scores or grad_scores there;
 *   - padding rows of the outputs are defined: every one of the 2+2K score heads is 0 (so cim_test_scores gives 0 and
 *     the test-time NMS, score > 1e-5, never takes a padding row), pseudo labels / pseudo IoU / loss weights are 0
 *     (the ignore row), asy_flag is 0, grad_x and the PCL gradient are exactly 0; cim_head_losses, fed those zeros,
 *     writes exactly 0 into grad_scores there;
 *   - every per-image quantity is computed for n_b, as running that image alone at R = n_b would: the detector
 *     softmax over its n_b proposals, keep_count = int(ceil(p_seed * n_b)) and big_thr = float32(0.9 * n_b)
 *     (cim_mine_image_constants), the containment counts over its n_b columns.
 * RoIAlign and the mask overlap maps have no _ex form: their padding rows are computed and nobody reads them.  Give
 * padding rois their own image index and finite coordinates, and grad_out rows of 0 at padding (what the scoring
 * backward's zero grad_x rows produce through a per-ROI head).  Zero padding masks let the overlap kernel skip them.
 */
#ifndef CIMHEAD_H
#define CIMHEAD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *cim_stream_t;   /* == cudaStream_t */

#define CIM_ABI_VERSION 4

enum {
    CIM_OK = 0,
    CIM_ERR_ARG = -1,          /* null pointer / negative size / bad enum            */
    CIM_ERR_SHAPE = -2,        /* shape outside what the kernels support             */
    CIM_ERR_WORKSPACE = -3,    /* workspace missing or too small                     */
    CIM_ERR_ALIGN = -4         /* pointer not aligned as documented                  */
};

int cim_abi_version(void);
/* Static string for a return code of this library (negative: CIM_ERR_*, positive: CUDA). */
const char *cim_error_string(int code);

/* Diagnostic kernel selection (A/B timing, the bit-identity tests of alternative kernels).  The library reads NOTHING
 * from the process environment; these flags are the only process-wide state it has, they default to 0 (every op
 * takes its production kernel), and a launch samples them once on entry.  Not meant for production code. */
enum {
    CIM_DBG_ROI_BWD_SMEM_TILE = 1u,   /* RoIAlign backward: gradient tile in shared memory, not tensor memory       */
    CIM_DBG_OVERLAP_LOADER_WARP = 2u, /* no effect any more (it selected the loader-warp pipeline of the int8 overlap kernel); kept so that callers still build */
    CIM_DBG_SCORE_FFMA = 4u,          /* scoring GEMMs fwd / bwd: plain fp32 FFMA kernels, not 3xTF32 tcgen05       */
    CIM_DBG_ROI_NO_WINDOWS = 8u,      /* RoIAlign on maps larger than the smem tile: global-pairs kernels           */
    CIM_DBG_ROI_BWD_ONE_CHUNK = 16u,  /* RoIAlign backward: one 32-channel chunk per CTA instead of two             */
    CIM_DBG_ROI_POOL_SIMPLE = 32u     /* RoIPool fwd / bwd: thread-per-output kernels, not the shared-memory tile   */
};
void cim_set_debug_flags(unsigned flags);
unsigned cim_get_debug_flags(void);
/* Test hook, HOST memory only, no GPU needed: the window plan of the RoIAlign window-tile path (maps larger than the
 * shared-memory tile, csrc/roi_window.cuh) evaluated on the CPU with the same code the prep kernels run.  desc_out
 * [cap][168] ints: one tile descriptor per sub-ROI, ROI order; key_out [cap]: its window index; flag_out [K]: 1 = the
 * ROI is left to the generic kernel; geom_out [6] = {Hp, wh, ww, nwy, nwx, origin granularity}.  Returns the number of
 * sub-ROIs or a negative CIM_ERR_* code. */
int cim_debug_roi_window_plan(const float *rois, int K, int B, int H, int W, float scale, int sampling_ratio,
                              int aligned, int *desc_out, int *key_out, int cap, int *flag_out, int *geom_out);

/* ------------------------------------------------------------------ ROI operators
 * Replace mmcv.ops.RoIAlign / RoIPool as imported by lib/ops/__init__.py:6 and called at
 * lib/modeling/model_builder.py:227-231 (`RoIAlign(resolution, spatial_scale,
 * sampling_ratio)(feat, rois)`); arithmetic = lib/modeling/roi_xfrom/roi_align/src/
 * roi_align_kernel.cu:16-121 (fwd) / :150-270 (bwd) plus mmcv's `aligned` half-pixel shift.
 *   feat      [B,C,H,W] fp32 contiguous        rois [K,5] fp32 (batch_idx,x1,y1,x2,y2)
 *   out       [K,C,oh,ow] fp32                 grad_feat [B,C,H,W] fp32 (fully overwritten)
 * sampling_ratio <= 0 means adaptive: ceil(roi_extent / bins) samples per bin and axis.
 * workspace: cim_roi_align_workspace_bytes(K) bytes, 16-byte aligned; contents are private.
 * The forward and the backward of one autograd node may share the workspace. */
size_t cim_roi_align_workspace_bytes(int K);
/* Feature maps too large for the shared-memory tile (32 channels x H x W fp32 > ~130 KB, e.g. VGG-16's 64 x 64 at
 * stride 8) are swept through a channel-last copy of the map kept in the workspace; that needs
 * cim_roi_align_workspace_bytes_ex() bytes (>= cim_roi_align_workspace_bytes(K); equal for maps that fit).  With
 * the smaller workspace such maps fall back to the generic one-thread-per-element kernels.  On this path the
 * backward accumulates with red.global.add, so its summation order is not fixed (the reference's atomicAdd
 * backward is not either). */
size_t cim_roi_align_workspace_bytes_ex(int B, int C, int H, int W, int K, int oh, int ow);
int cim_roi_align_fwd(const float *feat, const float *rois, float *out,
                      int B, int C, int H, int W, int K, int oh, int ow,
                      float spatial_scale, int sampling_ratio, int aligned,
                      void *workspace, size_t workspace_bytes, cim_stream_t stream);
int cim_roi_align_bwd(const float *grad_out, const float *rois, float *grad_feat,
                      int B, int C, int H, int W, int K, int oh, int ow,
                      float spatial_scale, int sampling_ratio, int aligned,
                      void *workspace, size_t workspace_bytes, cim_stream_t stream);

/* RoIAlign fused with the MaskFuse prologue (lib/modeling/resnet50.py:121-134, vgg16.py:172-175, HRNet.py:625-628:
 * `mask_x = box_x * masks.expand(...)`, `torch.concat((box_x, mask_x), dim=1)`): the pooled features and their
 * product with the ROI's oh x ow mask leave the kernel side by side, so the [K,C,oh,ow] tensor is never re-read
 * and the concat never materialised separately.
 *   masks7 [K, oh, ow] fp32 (the 7x7 proposal masks of tools/pre/generate_7_7_voc.py; no gradient, the
 *   reference passes masks.detach());  out / grad_out [K, 2C, oh, ow] fp32: channels [0,C) = RoIAlign,
 *   [C,2C) = RoIAlign * mask.  The backward feeds grad_out[:, :C] + grad_out[:, C:] * mask into the RoIAlign
 *   backward.  Same workspace as cim_roi_align_fwd / _bwd. */
int cim_roi_align_maskfuse_fwd(const float *feat, const float *rois, const float *masks7, float *out,
                               int B, int C, int H, int W, int K, int oh, int ow,
                               float spatial_scale, int sampling_ratio, int aligned,
                               void *workspace, size_t workspace_bytes, cim_stream_t stream);
int cim_roi_align_maskfuse_bwd(const float *grad_out, const float *rois, const float *masks7, float *grad_feat,
                               int B, int C, int H, int W, int K, int oh, int ow,
                               float spatial_scale, int sampling_ratio, int aligned,
                               void *workspace, size_t workspace_bytes, cim_stream_t stream);

/* The ROI descriptors (collapsed bilinear taps per bin) depend on the rois and the geometry only.  Every call above
 * builds them itself (one small kernel); when several calls see the SAME rois -- the forward and the backward of one
 * training step -- cim_roi_align_prepare() builds them once into the workspace and the _prepared entry points skip
 * their own pass.  The caller guarantees that rois, B, C, H, W, K, oh, ow, spatial_scale, sampling_ratio, aligned,
 * workspace and workspace_bytes are those of the prepare call and that the workspace was not used with other rois
 * in between.  masks7 == NULL: plain RoIAlign, else the MaskFuse variants. */
int cim_roi_align_prepare(const float *rois, int B, int C, int H, int W, int K, int oh, int ow,
                          float spatial_scale, int sampling_ratio, int aligned,
                          void *workspace, size_t workspace_bytes, cim_stream_t stream);
int cim_roi_align_fwd_prepared(const float *feat, const float *rois, const float *masks7, float *out,
                               int B, int C, int H, int W, int K, int oh, int ow,
                               float spatial_scale, int sampling_ratio, int aligned,
                               void *workspace, size_t workspace_bytes, cim_stream_t stream);
int cim_roi_align_bwd_prepared(const float *grad_out, const float *rois, const float *masks7, float *grad_feat,
                               int B, int C, int H, int W, int K, int oh, int ow,
                               float spatial_scale, int sampling_ratio, int aligned,
                               void *workspace, size_t workspace_bytes, cim_stream_t stream);

/* RoIPool: lib/model/roi_pooling/src/roi_pooling_kernel.cu:24-93 (fwd), :128-203 (bwd).
 * argmax [K,C,oh,ow] int32 = index inside the H*W plane, -1 for an empty bin. */
int cim_roi_pool_fwd(const float *feat, const float *rois, float *out, int32_t *argmax,
                     int B, int C, int H, int W, int K, int oh, int ow,
                     float spatial_scale, cim_stream_t stream);
/* variant: CIM_ROI_POOL_LEGACY = the bins of the reference's vendored kernel (== torchvision.ops.roi_pool; what
 * cim_roi_pool_fwd computes), CIM_ROI_POOL_MMCV = the bins of mmcv 1.x's RoIPool, which is what lib/ops/__init__.py:6
 * imports (float corners x1*s .. (x2+1)*s, floor / ceil of p*bin + start, degenerate ROIs pool nothing; restated from
 * mmcv's published kernel -- mmcv is an un-vendored, un-pinned dependency: parity unpinned).  The backward is the same
 * for both (it only reads argmax). */
enum { CIM_ROI_POOL_LEGACY = 0, CIM_ROI_POOL_MMCV = 1 };
int cim_roi_pool_fwd_ex(const float *feat, const float *rois, float *out, int32_t *argmax,
                        int B, int C, int H, int W, int K, int oh, int ow,
                        float spatial_scale, int variant, cim_stream_t stream);
int cim_roi_pool_bwd(const float *grad_out, const int32_t *argmax, const float *rois,
                     float *grad_feat, int B, int C, int H, int W, int K, int oh, int ow,
                     cim_stream_t stream);

/* ------------------------------------------------------------------ mask overlap maps
 * Replace lib/utils/mask_utils.py:6-18 (mask_iou) and :20-32 (mask_asymmetric_iou) as driven
 * column by column and cast to float16 by tools/pre/create_cob_iou.py:43-48 and
 * create_cob_asy_iou.py:43-51, and the per-step pickle loads that consume them
 * (lib/modeling/model_builder.py:148-156).
 *
 * cim_mask_pack: byte masks [n_masks, hw] (any non-zero = inside) -> bit masks
 *   [n_masks, words] uint32, bit (p & 31) of word (p >> 5) = pixel p; words >= ceil(hw/32),
 *   padding bits are written as 0.
 * cim_mask_overlap: for each of n_img images with n masks each (packed [n_img, n, words]):
 *   inter [n_img,n,n] int32 (optional, may be NULL), area [n_img,n] int32 (optional),
 *   iou  [n_img,n,n] fp16: inter / (area_i + area_j - inter)
 *   asy  [n_img,n,n] fp16: inter / area_j                       (0/0 -> NaN, as the reference)
 *   both computed as fp32 round-to-nearest division then fp32->fp16 round-to-nearest.
 *   workspace: cim_mask_overlap_workspace_bytes(n_img, n, words, inter != NULL) bytes, 256-byte
 *   aligned (the tensor-core path sorts the masks by position, works in sorted order and un-permutes
 *   the maps at the end; it needs two temporary maps).  n <= 16384.  After a tensor-path call the first
 *   8 bytes of the workspace hold, as uint64, the number of 128-pixel K-blocks the tiles visited
 *   (diagnostic: executed MMA work = that x 2*128*256*128).
 * Pixel order.  Counts do not depend on the order of the pixels inside the bit rows, only on all masks of
 *   a call using the same one.  cim_mask_pack / cim_mask_unpack_crops write the flat row-major order
 *   (p = y*W + x).  cim_mask_pack_tiled / cim_mask_unpack_crops_tiled (H % 8 == 0, W % 16 == 0, else
 *   CIM_ERR_SHAPE) write 8 x 16 pixel patches: q = ((y>>3)*(W>>4) + (x>>4))*128 + (y&7)*16 + (x&15);
 *   the 4 words of a patch are one K-block of the tensor-core kernel, which skips every K-block where one
 *   of the two operand blocks is empty -- with patches that follows the masks' 2-D footprint.  Pass
 *   kb_per_row = W/16 to cim_mask_overlap_ex for tiled input (it only steers the locality sort; 0 = flat). */
int cim_mask_pack(const uint8_t *masks, uint32_t *packed, int64_t n_masks, int64_t hw,
                  int64_t words, cim_stream_t stream);
int cim_mask_pack_tiled(const uint8_t *masks, uint32_t *packed, int64_t n_masks, int H, int W,
                        int64_t words, cim_stream_t stream);
/* cim_mask_unpack_crops: the compact host->device wire format.  Proposal masks are sent as their
 *   bounding-box crops (the reference cuts the same box out of every COB mask,
 *   tools/pre/generate_7_7_voc.py:36-38): crop_meta [n_masks,4] int32 = (wx0, y0, ww, h) -- the crop
 *   starts at pixel column 32*wx0, row y0 and is ww words wide, h rows high; crop_off [n_masks] int64
 *   = offset (in words) of the crop inside crop_words; crop row r, word k, bit j = pixel
 *   (y0 + r, 32*(wx0 + k) + j).  Output: the full bit masks [n_masks, words] cim_mask_overlap reads
 *   (zero outside the crops).  H, W = mask height / width in pixels, words >= ceil(H*W/32). */
int cim_mask_unpack_crops(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                          uint32_t *packed, int64_t n_masks, int H, int W, int64_t words,
                          cim_stream_t stream);
int cim_mask_unpack_crops_tiled(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                uint32_t *packed, int64_t n_masks, int H, int W, int64_t words,
                                cim_stream_t stream);
size_t cim_mask_overlap_workspace_bytes(int n_img, int n, int64_t words, int want_inter);
int cim_mask_overlap(const uint32_t *packed, int n_img, int n, int64_t words,
                     int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16,
                     void *workspace, size_t workspace_bytes, cim_stream_t stream);
/* Same with an explicit kernel choice.  AUTO = tensor cores (tcgen05.mma.kind::i8 over bytes
 * expanded from the bit masks in shared memory, exact S32 accumulation) for n >= 256 and
 * words >= 128 with words % 4 == 0 and a 16-byte aligned `packed`, else the popcount kernel.
 * TENSOR returns CIM_ERR_SHAPE when the problem cannot take that path. */
enum { CIM_OVERLAP_AUTO = 0, CIM_OVERLAP_POPC = 1, CIM_OVERLAP_TENSOR = 2 };
int cim_mask_overlap_algo(const uint32_t *packed, int n_img, int n, int64_t words,
                          int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16,
                          void *workspace, size_t workspace_bytes, int algo, cim_stream_t stream);
/* Same, for input in the tiled pixel order: kb_per_row = W / 16 (K-blocks per row of patches). */
int cim_mask_overlap_ex(const uint32_t *packed, int n_img, int n, int64_t words, int kb_per_row,
                        int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16,
                        void *workspace, size_t workspace_bytes, int algo, cim_stream_t stream);
/* Mask metadata produced WITH the masks instead of inside every overlap call: per mask its area, the occupancy bitmap
 * over 128-pixel K-blocks and the locality-sort key (what cim_mask_overlap's first pass over the packed masks
 * computes -- 0.1 ms at HBM speed for 8 x 2000 masks of 512 x 512).  A producer that packs or unpacks the masks
 * (cim_mask_pack_tiled at data-set preparation, cim_mask_unpack_crops_tiled on the copy stream of the input prefetch)
 * calls cim_mask_meta once on its own stream; cim_mask_overlap_meta then starts with the sort.  meta: opaque,
 * cim_mask_meta_bytes() bytes, 256-byte aligned, tied to (packed, n_img, n, words, kb_per_row); words % 4 == 0 and a
 * 16-byte aligned `packed` (CIM_ERR_ALIGN otherwise).  meta == NULL: identical to cim_mask_overlap_ex. */
size_t cim_mask_meta_bytes(int n_img, int n, int64_t words);
/* cim_mask_unpack_crops_tiled and cim_mask_meta in one pass over the crops: every packed word is written exactly once
 * (zeros outside the crop, so no memset of `packed` beforehand) and the metadata falls out of the same registers.
 * words * 32 == H * W, H % 8 == 0, W % 16 == 0; crops must lie inside the image. */
int cim_mask_unpack_crops_tiled_meta(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                     uint32_t *packed, void *meta, size_t meta_bytes, int n_img, int n, int H, int W,
                                     int64_t words, cim_stream_t stream);
/* The same as a SPARSE UPDATE of a `packed` buffer that already holds an earlier batch of crops: prev_rects [n_img * n][4]
 * int32 (16-byte aligned) = the crop rectangle (wx0, y0, ww, h) of the mask currently stored in each row, all zero for a
 * row of zeros.  Only the patches of the old and the new rectangle are visited (the old ones are cleared), prev_rects is
 * updated in place.  First use: a zero-filled `packed` and zero-filled prev_rects.  The input-prefetch path of a training
 * loop re-writes ~10 % of the buffer per step this way instead of all of it. */
int cim_mask_unpack_crops_tiled_meta_sparse(const uint32_t *crop_words, const int32_t *crop_meta, const int64_t *crop_off,
                                            uint32_t *packed, int32_t *prev_rects, void *meta, size_t meta_bytes, int n_img,
                                            int n, int H, int W, int64_t words, cim_stream_t stream);
int cim_mask_meta(const uint32_t *packed, int n_img, int n, int64_t words, int kb_per_row, void *meta,
                  size_t meta_bytes, cim_stream_t stream);
int cim_mask_overlap_meta(const uint32_t *packed, const void *meta, int n_img, int n, int64_t words, int kb_per_row,
                          int32_t *inter, int32_t *area, void *iou_f16, void *asy_f16,
                          void *workspace, size_t workspace_bytes, int algo, cim_stream_t stream);

/* Rectangular ratios between two mask sets: the offline callers of lib/utils/mask_utils.py
 * (tools/pre/AGPL_label_assign.py:84,165, tools/pre/point_level_label_assign.py:79,
 * tools/generate_mask_for_MaskRCNN.py, tools/pre/create_cob_iou.py:45, create_cob_asy_iou.py:46).
 *   packed_a [na, words], packed_b [nb, words]: bit masks in the same pixel order (cim_mask_pack);
 *   mode 0 mask_iou (mask_utils.py:6-18), 1 mask_asymmetric_iou (I / mask_b.sum() over ALL of b, :20-32),
 *        2 mask_inside (I / |b_k|, :35-47), 3 mask_outside (I / |a_n|, :50-62);
 *   ratio [na, nb] fp32 (the reference's float32 result array; 0/0 -> NaN), inter [na, nb] int32 (optional),
 *   area_a [na], area_b [nb] int32 (outputs: the row popcounts).  words * 32 <= 2^24. */
int cim_mask_pair_ratio(const uint32_t *packed_a, const uint32_t *packed_b, int na, int nb, int64_t words, int mode,
                        float *ratio, int32_t *inter, int32_t *area_a, int32_t *area_b, cim_stream_t stream);

/* ------------------------------------------------------------------ scoring heads
 * Replace heads.cls_iou_model.forward (lib/modeling/heads.py:194-219): n_heads = 2 + 2*K
 * linear layers over the same features, ordered [classifier, detector, refine_cls.0..K-1,
 * refine_iou.0..K-1], followed by softmax over classes (classifier, refine_cls), softmax over
 * the PROPOSALS of each image (detector, heads.py:203) and sigmoid (refine_iou).
 *   x [n_img*R, D] fp32; weight [n_heads, C1, D]; bias [n_heads, C1];
 *   scores [n_heads, n_img*R, C1] fp32.  workspace: cim_score_heads_workspace_bytes() bytes; with
 *   it (and D % 32 == 0, C1 <= 96, n_img*R >= 128) the GEMM runs on the tensor cores as three TF32
 *   products of hi/lo-split operands (fp32-accurate), otherwise as fp32 FFMA. */
size_t cim_score_heads_workspace_bytes(int n_img, int R, int D, int C1, int K);
int cim_score_heads(const float *x, const float *weight, const float *bias, float *scores,
                    int n_img, int R, int D, int C1, int K,
                    void *workspace, size_t workspace_bytes, cim_stream_t stream);
/* Ragged form (see the top of this file): the detector softmax runs over the n_b rows of each image and every head is
 * 0 on its padding rows.  n_props 4-byte aligned. */
int cim_score_heads_ex(const float *x, const float *weight, const float *bias, float *scores, const int32_t *n_props,
                       int n_img, int R, int D, int C1, int K,
                       void *workspace, size_t workspace_bytes, cim_stream_t stream);

/* Backward of cim_score_heads = autograd of heads.cls_iou_model.forward (lib/modeling/heads.py:194-219; the
 * reference gets it from eight nn.Linear backward calls + softmax / sigmoid backward, run by loss.backward(),
 * tools/train.py:436).  grad_weight / grad_bias are the head gradients a data-parallel run all-reduces
 * (reference: comm.reduce_add_coalesced, lib/nn/parallel/_functions.py:39).
 *   scores       [n_heads, n_img*R, C1] fp32: the OUTPUT of cim_score_heads for the same x / weight / bias
 *   grad_scores  [n_heads, n_img*R, C1] fp32: dL/dscores
 *   grad_x       [n_img*R, D]      (may be NULL)     grad_weight [n_heads, C1, D] (may be NULL)
 *   grad_bias    [n_heads, C1]     (may be NULL)     all fully overwritten.
 * Activation backward: y (g - sum_classes g y) for classifier / refine_cls, y (g - sum over the proposals of
 * the image of g y) for the detector, g y (1 - y) for refine_iou.  The two GEMMs run as 3xTF32 on the tensor
 * cores (fp32-accurate) when n_img*R >= 128 and D % 4 == 0, as plain fp32 otherwise.  Deterministic (the
 * split-M partial sums of grad_weight are added in a fixed order).  C1 <= 1700 (one proposal row block of dz is
 * staged in shared memory), CIM_ERR_SHAPE above.
 * workspace: cim_score_heads_bwd_workspace_bytes() bytes, required. */
size_t cim_score_heads_bwd_workspace_bytes(int n_img, int R, int D, int C1, int K);
int cim_score_heads_bwd(const float *x, const float *weight, const float *scores, const float *grad_scores,
                        float *grad_x, float *grad_weight, float *grad_bias,
                        int n_img, int R, int D, int C1, int K,
                        void *workspace, size_t workspace_bytes, cim_stream_t stream);
/* Ragged form: the detector's sum runs over the n_b rows of each image, and dz = 0 on padding rows whatever
 * grad_scores holds there, so grad_x rows there are 0 and padding adds nothing to grad_weight / grad_bias. */
int cim_score_heads_bwd_ex(const float *x, const float *weight, const float *scores, const float *grad_scores,
                           const int32_t *n_props, float *grad_x, float *grad_weight, float *grad_bias,
                           int n_img, int R, int D, int C1, int K,
                           void *workspace, size_t workspace_bytes, cim_stream_t stream);

/* ------------------------------------------------------------------ CIM mining + assignment
 * Replace heads.CIM_layer (lib/modeling/heads.py:222-503) for n_img images x n_layers
 * refinement layers in one go.  Layer l reads cls[l] / det[l] (device pointers, each
 * [n_img, R, C1 or C]); the background column is dropped when C1 == C + 1 (heads.py:327-328).
 * All float16 threshold tests are made in float16 against float16(thr), as torch does.
 *
 * Limits: R <= 10240, keep_count <= 1024, n_layers <= 4.  Scores are assumed finite and >= 0
 * (they are softmax / sigmoid outputs).
 *
 * Phase 1 (cim_mine): seeds = top keep_count by class score, greedy mask NMS on iou_map,
 *   containment mining on asy_map (mode 0 = CIM_label heads.py:318-407, mode 1 = MIST_label
 *   heads.py:260-316), per-proposal arbitration between classes.  Outputs, per (layer, image):
 *     gt_count [L, n_img] int32; gt_rows / gt_class / gt_weight [L, n_img, gt_cap]
 *     (ascending proposal index, the order boolean-mask indexing gives at heads.py:405);
 *     asy_flag [n_img, R] uint8 (asy_iou_flag, heads.py:338).
 * Between the phases the host may drop pseudo GTs (anti-noise sampling, heads.py:440-473,
 *   which draws from numpy's global RNG) by writing gt_keep [L, n_img, gt_cap] uint8.
 * Phase 2 (cim_assign): heads.py:475-501 -> pseudo_labels [L, n_img, R, C+1] fp32,
 *   pseudo_iou [L, n_img, R] fp16, loss_weights [L, n_img, R] fp32, valid [L, n_img] uint8
 *   (0 where the reference returns (None, None, None), heads.py:429-430). */
typedef struct {
    int n_img, R, C, C1, n_layers;   /* C foreground classes; C1 = row length of cls/det   */
    int det_cols;                    /* row length of det[l]: C1, C or 1 (class-agnostic)  */
    int gt_cap;                      /* capacity of the gt_* lists per (layer, image)      */
    int mode;                        /* 0 = CIM_label, 1 = MIST_label                      */
    int keep_count;                  /* int(ceil(p_seed * R)), heads.py:332, host-evaluated */
    float big_thr;                   /* float32(0.9 * R), heads.py:338, host-evaluated      */
    float con_thr;
    float cls_thr[4], iou_thr[4];    /* per layer; nms_thr == cls_thr (heads.py:227)       */
} cim_mine_params;

size_t cim_sizeof_mine_params(void);   /* lets a binding verify its struct layout */
size_t cim_mine_workspace_bytes(const cim_mine_params *p);
int cim_mine(const cim_mine_params *p, const float *const *cls, const float *const *det,
             const float *labels /* [n_img, C] */, const void *iou_f16, const void *asy_f16,
             int32_t *gt_count, int32_t *gt_rows, int32_t *gt_class, float *gt_weight,
             uint8_t *asy_flag, void *workspace, size_t workspace_bytes, cim_stream_t stream);
/* Ragged form: n_props == NULL is cim_mine (p->keep_count and p->big_thr are used, p_seed is ignored).  Otherwise
 * every image gets keep_count and big_thr from its n_b and p_seed (0 < p_seed <= 1) as cim_mine_image_constants()
 * computes them, p->big_thr is ignored, and p->keep_count is the capacity the workspace is sized for: it must be at
 * least the keep_count of n_b = R (CIM_ERR_ARG otherwise). */
int cim_mine_ex(const cim_mine_params *p, const int32_t *n_props, double p_seed, const float *const *cls,
                const float *const *det, const float *labels, const void *iou_f16, const void *asy_f16,
                int32_t *gt_count, int32_t *gt_rows, int32_t *gt_class, float *gt_weight, uint8_t *asy_flag,
                void *workspace, size_t workspace_bytes, cim_stream_t stream);
/* Host memory only, no GPU needed: the per-image constants of cim_mine_ex for an image of n proposals, computed by the
 * same code the kernels run.  keep_count = int(ceil(p_seed * n)) (heads.py:332), big_thr = float32(0.9 * n)
 * (heads.py:338), both from one float64 product rounded to nearest.  n >= 1, 0 < p_seed <= 1, else CIM_ERR_ARG. */
int cim_mine_image_constants(double p_seed, int n, int *keep_count, float *big_thr);
/* Anti-noise sampling between the phases ON THE DEVICE (heads.py:440-473): per (layer, image) list and present class,
 * np.random.choice(class_idx, size=n, replace=True, p=w / w.sum()) with numpy's arithmetic restated bit for bit
 * (float32 pairwise sum, float32 p, float64 cumsum normalised by its last element, searchsorted side='right'); the
 * drawn pseudo GTs keep gt_keep = 1, the other pseudo GTs of the class get 0.  `uniforms` are the doubles the host
 * drew from numpy's GLOBAL RandomState with ONE np.random.random_sample(T) call, T = sum of gt_count: the call
 * consumes the same stream as the reference's per-class calls, in the reference's order (image, then layer, then
 * ascending class, then position), which is the order the kernel reads them in.  So the host hop shrinks to: read
 * gt_count (n_layers * n_img ints), draw T doubles, copy them over -- the lists themselves never leave the device.
 * gt_keep [L, n_img, gt_cap] is fully written.  (choice()'s argument checks -- negative / NaN p -- are not
 * reproduced: the weights are products of softmax outputs.) */
size_t cim_anti_noise_uniform_count_max(const cim_mine_params *p);   /* L * n_img * gt_cap */
int cim_anti_noise(const cim_mine_params *p, const float *labels /* [n_img, C] */, const int32_t *gt_count,
                   const int32_t *gt_class, const float *gt_weight, const double *uniforms, uint8_t *gt_keep,
                   cim_stream_t stream);
/* The same sampling WITHOUT the host hop: `ring` [ring_len doubles, ring_len >= L * n_img * gt_cap] holds a stretch
 * of the host's random stream drawn AHEAD of time (position q of the stream lives in ring[q % ring_len]); the step's
 * first double is at absolute position *cursor_in, and the kernel leaves *cursor_in + T (T = the doubles this step
 * consumed = sum of gt_count) in *cursor_out for the next step (cursor_in != cursor_out: callers alternate two
 * words).  The host never waits for gt_count inside the step: it learns T from a lagged read-back, keeps the ring
 * filled past every position a step in flight can reach, and advances numpy's RandomState by the consumed total at
 * its next synchronisation point (cim_b200.heads.UniformStream; CIMHeadStep(rng="stream")).  Same draws, same
 * gt_keep as cim_anti_noise given the same stream. */
int cim_anti_noise_stream(const cim_mine_params *p, const float *labels, const int32_t *gt_count,
                          const int32_t *gt_class, const float *gt_weight, const double *ring, int64_t ring_len,
                          const int64_t *cursor_in, int64_t *cursor_out, uint8_t *gt_keep, cim_stream_t stream);
int cim_assign(const cim_mine_params *p, const void *iou_f16,
               const int32_t *gt_count, const int32_t *gt_rows, const int32_t *gt_class,
               const float *gt_weight, const uint8_t *gt_keep /* may be NULL = keep all */,
               float *pseudo_labels, void *pseudo_iou_f16, float *loss_weights, uint8_t *valid,
               cim_stream_t stream);
/* Ragged form: padding rows get the ignore row (pseudo labels, pseudo IoU and loss weight 0). */
int cim_assign_ex(const cim_mine_params *p, const int32_t *n_props, const void *iou_f16,
                  const int32_t *gt_count, const int32_t *gt_rows, const int32_t *gt_class,
                  const float *gt_weight, const uint8_t *gt_keep, float *pseudo_labels, void *pseudo_iou_f16,
                  float *loss_weights, uint8_t *valid, cim_stream_t stream);

/* ------------------------------------------------------------------ loss block (forward + backward)
 * cim_head_losses: per image b and refinement layer l < n_layers with valid[l][b] != 0 (the reference skips a
 *   layer whose CIM_layer returned None, lib/modeling/model_builder.py:189-190):
 *   heads.cls_iou_loss(ref_cls[l], ref_iou[l], pseudo_labels, pseudo_iou_labels, lmda * loss_weights, labels)
 *   (lib/modeling/heads.py:78-138, class-specific IoU branch, with loss_weight_bag_loss heads.py:43-74), and
 *   once per image heads.mil_bag_loss(predict_cls, predict_det, labels) (heads.py:149-166).
 *   scores        [2+2K, n_img*R, C+1] fp32 as written by cim_score_heads
 *   pseudo_labels [n_layers, n_img, R, C+1] fp32, pseudo_iou [n_layers, n_img, R] fp16,
 *   loss_weights  [n_layers, n_img, R] fp32, valid [n_layers, n_img] uint8 (outputs of cim_assign),
 *   labels        [n_img, C] fp32 image labels;  lmda0 / lmda_rest: multiplier of loss_weights for layer 0 / the
 *   others (3 / 1, model_builder.py:172,194).
 *   losses      [n_img, K+1, 3] fp32: (cls_loss, iou_loss, bag_loss) per layer slot (zeros for skipped layers);
 *               slot K holds (0, 0, mil_bag_loss).  The reference's totals are sum_l cls, iou_weight * sum_l iou
 *               (iou_weight = 3, model_builder.py:199) and sum_l bag + mil_bag.
 *   grad_scores [2+2K, n_img*R, C+1] fp32 (may be NULL): grad_scale * d(sum_l cls + iou_weight * sum_l iou +
 *               sum_l bag + mil_bag of the row's image) / d scores, every element written.
 * PCL_loss (heads.py:10-41) needs the dataset's cluster matrix and is not covered.  R <= 10240, C + 1 <= 1024. */
int cim_head_losses(const float *scores, const float *pseudo_labels, const void *pseudo_iou_f16,
                    const float *loss_weights, const uint8_t *valid, const float *labels, float *losses,
                    float *grad_scores, int n_img, int R, int C, int K, int n_layers, float lmda0,
                    float lmda_rest, float iou_weight, float grad_scale, cim_stream_t stream);

/* cim_pcl_loss: heads.PCL_loss (lib/modeling/heads.py:10-41; called at lib/modeling/model_builder.py:203) forward and
 *   backward for n_img images.  predict_cls [n_img*R, C1] fp32 (head 0 of the score tensor); mat [n_img, R, C1] fp32
 *   cluster ids as tools/pre/AGPL_label_assign.py writes them (integers in [0, max_id], 0 = none; the background
 *   cluster's id lives in column 0).  loss [n_img] fp32 = 12 * loss / (1e-6 + sum of cluster sizes) per image (NaN for
 *   ids that are not integers in range, or two different ids in column 0 -- the reference asserts there).
 *   grad_cls [n_img*R, C1] (may be NULL) = grad_scale * d loss / d predict_cls, overwritten, or added to when
 *   accumulate != 0 (so it can land on top of cim_head_losses' gradient of the same head).  Deterministic.
 *   C1 <= 128, max_id <= 255, R <= 16384. */
int cim_pcl_loss(const float *predict_cls, const float *mat, float *loss, float *grad_cls, int n_img, int R, int C1,
                 int max_id, float grad_scale, int accumulate, cim_stream_t stream);
/* Ragged form: mat reads as 0 on padding rows, which join no cluster and get gradient 0 (added 0 with accumulate). */
int cim_pcl_loss_ex(const float *predict_cls, const float *mat, const int32_t *n_props, float *loss, float *grad_cls,
                    int n_img, int R, int C1, int max_id, float grad_scale, int accumulate, cim_stream_t stream);

/* ------------------------------------------------------------------ test-time post-processing
 * cim_test_scores: lib/core/test.py:130-133 over lib/modeling/model_builder.py:60-68 -- the K refinement
 *   heads' (cls * iou)[:, 1:] summed in head order and divided by K.
 *   scores [2+2K, M, C1] fp32 as written by cim_score_heads -> out [M, C1-1] fp32.
 * cim_box_nms: the per-class body of lib/utils/mask_eval_utils.py:57-79 -- candidates scores[i][c] >
 *   score_thresh, then the greedy NMS of lib/utils/cython_nms.pyx:37-87 ("+1" areas, float32 arithmetic,
 *   suppression when overlap >= nms_thresh, boxes visited by descending score; equal scores by descending
 *   index).  boxes [n,4] fp32 (x1,y1,x2,y2), 16-byte aligned; scores [n, score_stride] fp32, class c in
 *   column c; keep [n_classes, n] uint8 = 1 where proposal i survives for class c (np.where(suppressed == 0)
 *   + the candidate filter; ascending i is the reference's output order).  n <= 8192. */
int cim_test_scores(const float *scores, float *out, int64_t M, int C1, int K, cim_stream_t stream);
int cim_box_nms(const float *boxes, const float *scores, int n, int n_classes, int score_stride,
                float score_thresh, float nms_thresh, uint8_t *keep, cim_stream_t stream);
/* The same for n_img images in one launch: boxes [n_img, n, 4], scores [n_img, n, score_stride],
 * keep [n_img, n_classes, n] (one CTA per (class, image): 80 CTAs of one image leave half a B200 idle). */
int cim_box_nms_batched(const float *boxes, const float *scores, int n_img, int n, int n_classes, int score_stride,
                        float score_thresh, float nms_thresh, uint8_t *keep, cim_stream_t stream);
/* cim_test_scores_tta: pass t of T of the test-time-augmentation score mean of lib/core/test.py:149-226
 *   (TEST.BBOX_AUG, SCORE_HEUR 'AVG': np.mean(scores_ts, axis=0)).  s = the cim_test_scores result of this pass's
 *   scores [2+2K, M, C1]; acc [M, C1-1] = s when t == 0, fl(acc + s) otherwise, and on the last pass (t == T-1,
 *   T > 1) fl(acc / T).  The passes are summed in call order.  cim_test_scores is the t = 0, T = 1 case. */
int cim_test_scores_tta(const float *scores, float *acc, int64_t M, int C1, int K, int t, int T, cim_stream_t stream);
/* cim_box_detections: the DETECTIONS_PER_IM limit and the per-class detection lists of
 *   lib/utils/mask_eval_utils.py:80-110 for the keep mask of cim_box_nms_batched (same boxes, scores, n_img, n,
 *   n_classes, score_stride).  Per image: total = kept entries over all classes; when detections_per_im > 0 and
 *   total > detections_per_im, thresh = the detections_per_im-th largest kept score (with multiplicity) and an entry
 *   survives iff it is kept and score >= thresh (float32; ties at thresh all survive), otherwise every kept entry
 *   survives.  count [n_img] int32 = survivors (also when > cap); the first min(count, cap) survivors, ordered by
 *   class then proposal index, are written to det_cls / det_idx [n_img, cap] int32, det_score [n_img, cap] fp32
 *   (= scores[i][c]) and det_box [n_img, cap, 4] fp32 (= boxes[i]; may be NULL); the rest of a row is not written.
 *   keep_out [n_img, n_classes, n] uint8 (may be NULL) = the keep mask after the limit.  det_* may be NULL when
 *   cap == 0.  No workspace.  n <= 8192. */
int cim_box_detections(const float *boxes, const float *scores, const uint8_t *keep, int n_img, int n, int n_classes,
                       int score_stride, int detections_per_im, int cap, uint8_t *keep_out, int32_t *count,
                       int32_t *det_cls, int32_t *det_idx, float *det_score, float *det_box, cim_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CIMHEAD_H */
