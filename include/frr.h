/*
 * frr.h -- C ABI of libfrr.so: the B200-native (sm_100a) Faster R-CNN region stage.
 *
 * Drop-in boundary for the region stage of csm-kr/faster_rcnn_pytorch (SURVEY.md §8b).
 * The reference has no FFI layer; its boundary is the Python call sites in
 * models/model.py:6-9,288-298 (torchvision.ops.nms / RoIPool, FRCNNAnchorMaker, the
 * utils.util box helpers and the RegionProposal / *TargetMaker modules).  Every entry
 * point below cites the reference lines it replaces.  The Python mirror of those call
 * sites lives in faster_rcnn_pytorch_b200/ and binds this header with ctypes
 * (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer on the current CUDA device unless named *_host;
 *  - the library never allocates, frees or synchronises: the caller owns outputs and
 *    workspaces and passes the stream (cudaStream_t as void*); all calls are
 *    graph-capturable;
 *  - ragged results use fixed-capacity buffers + int32 counts on the device;
 *  - boxes are fp32 (x1,y1,x2,y2); box arrays must be 16-byte aligned;
 *  - return value: 0 = ok, negative = error (FRR_E_*); frr_last_error() returns a
 *    thread-local message.  No C++ exception crosses the boundary.
 */
#ifndef FRR_H_
#define FRR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#pragma GCC visibility push(default)
#endif

#define FRR_ABI_VERSION 3

#define FRR_OK 0
#define FRR_E_INVALID (-1)   /* bad argument (shape, alignment, range)        */
#define FRR_E_LAUNCH (-2)    /* CUDA launch / runtime error                   */
#define FRR_E_WORKSPACE (-3) /* workspace too small                           */
#define FRR_E_UNSUPPORTED (-4)

typedef void* frr_stream_t; /* cudaStream_t */

int frr_abi_version(void);
const char* frr_last_error(void);
/* Number of kernels this library has launched in the calling process (bench "gpu_launches"). */
uint64_t frr_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * A1/A2  anchors -- anchor.py:15-32 (generate_anchor_base), :34-55 (_enumerate_shifted_anchor)
 * ------------------------------------------------------------------------------------- */
/* Host helper: the reference's 9x4 base table (ratio-major, float64 math stored to fp32). */
int frr_anchor_base_host(float* table_host /* [9*4] */, int base_size);
/* anchors[(y*fw+x)*A+a] = fl32(base[a] + stride*(x,y,x,y)) / (W,H,W,H);  fh=H/stride, fw=W/stride.
 * base_table_host: [A*4] host floats or NULL for the reference table (A=9).  A <= 16. */
int frr_anchors(float* anchors /* [fh*fw*A,4] */, int img_h, int img_w, int stride,
                const float* base_table_host, int A, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A2 (FPN variant)  torchvision.models.detection.rpn.AnchorGenerator(sizes=((32,),(64,),(128,),(256,),(512,)),
 *     aspect_ratios=((0.5,1.0,2.0),)*5) as built at models/new_model.py:23-25 and called at :43-44, followed by
 *     `anchor /= (w, h, w, h)`.  frr_tv_anchor_base_host = generate_anchors of one level (fp32 math, round half to
 *     even) -> [n_ratios,4] on the host; frr_anchors_pyramid = grid_anchors over L <= 8 levels (level_hw_host
 *     [L,2] = (fh, fw) per level, strides img // grid like torchvision, base_tables_host [L,A,4], A <= 8) written
 *     normalised to anchors [sum_l fh_l fw_l A, 4] on the device, levels concatenated, cell-major / anchor-minor.
 * ------------------------------------------------------------------------------------- */
int frr_tv_anchor_base_host(float size, const float* aspect_ratios, int n_ratios, float* table_host);
int frr_anchors_pyramid(float* anchors, int L, const int32_t* level_hw_host, const float* base_tables_host, int A,
                        int img_h, int img_w, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * P1-P3  fused RPN decode -- models/model.py:20 (softmax fg), :31-34 (decode, clamp),
 *        :37-41 (min-size filter); utils/util.py:15-26,46-50.  Anchors are generated in
 *        registers (A2) unless `anchors` is given.
 * ------------------------------------------------------------------------------------- */
int frr_rpn_decode(const float* reg /* [B,N,4] */, const float* cls /* [B,N,2] logits or [B,N] scores */,
                   int cls_is_logits, const float* anchors /* [N,4] or NULL */,
                   const float* base_table_host /* [A*4] or NULL */, int A, int img_h, int img_w,
                   int stride, float min_size /* reference: 0.001f */, float* boxes /* [B,N,4] */,
                   float* scores /* [B,N] */, uint8_t* valid /* [B,N] */, int B, int N,
                   frr_stream_t stream);

/* Mixed-size batches -- the reference builds anchors from each image's own size (models/model.py:310-312,352-354) and
 *     scales rois by each image's own feature grid (:104-110).  A batch of differently sized images is padded to one grid
 *     of grid_h x grid_w cells (N = grid_h * grid_w * A anchors per image, cell-major / anchor-minor over the PADDED grid);
 *     image_hw int32 [B,2] (device, 8-byte aligned) holds each image's (H_b, W_b) in pixels.  Image b covers the cells
 *     y < fh_b = H_b / stride, x < fw_b = W_b / stride; the rest of the grid is padding.  Every entry point that takes
 *     image_hw gives, when it is set, image b exactly what it gives with image_hw == NULL for image b alone at (H_b, W_b)
 *     on the cropped inputs, with indices mapped by (y * grid_w + x) * A + a <-> (y * fw_b + x) * A + a; its size
 *     parameters then describe the padded batch, anchors must be NULL (generated) and stride > 0.  The sizes are read on
 *     the device at run time (one CUDA graph serves every mix of sizes that fits the grid), so the host cannot check
 *     them: fh_b / fw_b are clamped to [0, grid_h] / [0, grid_w], and an image with an empty grid has no valid anchor, no
 *     proposal (count 0) and no rois.
 * frr_rpn_decode_sized: anchors divided by each image's own (W_b, H_b) (the __fdiv_rn recipe of frr_rpn_decode);
 *     padding cells get box 0, score 0, valid 0 whatever reg / cls hold there (NaN included).                        */
int frr_rpn_decode_sized(const float* reg /* [B,N,4] */, const float* cls /* [B,N,2] logits or [B,N] scores */,
                         int cls_is_logits, const float* base_table_host /* [A*4] or NULL */, int A,
                         const int32_t* image_hw /* [B,2] device */, int grid_h, int grid_w, int stride, float min_size,
                         float* boxes /* [B,N,4] */, float* scores /* [B,N] */, uint8_t* valid /* [B,N] */, int B, int N,
                         frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * P4  pre-NMS top-k, sorted descending -- models/model.py:44-49.  One CTA per image, in shared
 *     memory: monotone bucketing of the scores + exact ranking inside the buckets (radix select + radix
 *     sort for inputs that do not bucket).  Ties: lower index first.  Entries past count[b] are padded
 *     (idx -1, score -inf, box 0).  out_cidx = index into the min-size-compacted array (what
 *     the reference's sort returns), out_idx = index into the full N.  k <= 16384.
 * ------------------------------------------------------------------------------------- */
/* ctas_per_image: 0 = automatic (a 2-CTA cluster per image when B * 2 CTAs fit the SMs: lowest latency), 1 = one CTA per
 * image (least SM time: several batches in flight).  Identical results.                                                */
int frr_topk_desc_opt(const float* scores /* [B,N] */, const uint8_t* valid /* [B,N] or NULL */,
                  const float* boxes /* [B,N,4] or NULL */, int B, int N, int k,
                  float* out_scores /* [B,k] or NULL */, int32_t* out_idx /* [B,k] */,
                  int32_t* out_cidx /* [B,k] or NULL */, float* out_boxes /* [B,k,4] or NULL */,
                  int32_t* out_count /* [B] */, int ctas_per_image, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * N1  greedy NMS on score-sorted boxes -- torchvision.ops.nms at models/model.py:53-55
 *     (IoU 0.7, keep[:2000|300]) with torchvision's CPU semantics: fp32 IoU, suppress when
 *     (double)iou > iou_thr.  Keep-list algorithm on a thread-block cluster per image,
 *     stops at max_keep.  keep = positions in the sorted list, ascending, -1 padded.
 *     cluster_size: 0 = auto, else 1,2,4,8,16.
 * ------------------------------------------------------------------------------------- */
/* threads per CTA (0 = auto, 256, 512 or 1024); the settings of the bucketed variant (3 in frr_nms_variant), each
 * 0 = automatic: first_chunk / max_chunk = candidates in the first / the largest chunk (multiples of 256 in [256, 2048];
 * automatic 1024 / 2048), lanes_screen / lanes_pairs = lanes per candidate of its screen / pair phases (powers of two
 * <= 32; automatic: lanes_screen 2 with 1-2 CTAs per image, else 4; lanes_pairs 4); unit_boxes != 0 = the caller
 * guarantees every coordinate lies in [0,1] (true for the clamped RPN / detection boxes of models/model.py:34,378),
 * which enables a cheaper screening test.  Results are identical for every setting.                                    */
int frr_nms_sorted(const float* boxes /* [B,n,4] */, const int32_t* counts /* [B] or NULL (=n) */, int B,
                   int n, double iou_thr, int max_keep, int32_t* keep /* [B,max_keep] */,
                   int32_t* keep_count /* [B] */, float* out_boxes /* [B,max_keep,4] or NULL */,
                   int cluster_size, int threads, int first_chunk, int max_chunk, int lanes_screen, int lanes_pairs,
                   int unit_boxes, frr_stream_t stream);

/* Which kernel variant and launch geometry the NMS entry points pick for a problem (host only, launches nothing;
 * tests and bench.py assert through it that the variant they mean to exercise is the one that runs):
 * out4[0] = CTAs per image, out4[1] = threads per CTA, out4[2] = variant (0 exact test only, 1 screened,
 * 2 screened + unit range, 3 unit range + area-class / x-bin bucketed lists), out4[3] = dynamic shared memory.   */
int frr_nms_variant(int B, int n, double iou_thr, int max_keep, int cluster_size, int threads, int unit_boxes,
                    int32_t* out4);

/* Same, with the score order given as indices into an unsorted array: candidate i of image b is
 * boxes_src[b][order[b][i]] (boxes_src [B,src_n,4]; order int32 [B,n] = out_idx of frr_topk_desc_opt).  Only the
 * candidates NMS visits are gathered; the top-k kernel then need not write sorted boxes at all.          */
int frr_nms_sorted_indirect(const float* boxes_src, int src_n, const int32_t* order, const int32_t* counts, int B,
                            int n, double iou_thr, int max_keep, int32_t* keep, int32_t* keep_count,
                            float* out_boxes, int cluster_size, int unit_boxes, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * RegionProposal.forward for a batch in one call -- models/model.py:17-58 (P1-P4 + N1 chained: the three
 * kernels above on `stream`, intermediates in `workspace`).  k = min(pre_nms_top_k, N) (:46-47).
 * rois [B,post_nms_top_k,4] zero padded, roi_count [B].  Reference constants: 12000/2000 (train),
 * 6000/300 (test), iou_thr 0.7, min_size 0.001f.  workspace: 256-byte aligned, size from
 * frr_rpn_proposals_workspace_bytes.
 * ------------------------------------------------------------------------------------- */
size_t frr_rpn_proposals_workspace_bytes(int B, int N, int pre_nms_top_k, int post_nms_top_k);
/* Byte offsets of the intermediates inside that workspace (for callers / tests that inspect them after a call):
 * offsets[0..5] = decoded boxes [B,N,4] f32, scores [B,N] f32, valid [B,N] u8, top-k order [B,k] i32 (indices into
 * N), top-k count [B] i32, NMS keep list [B,post] i32 (positions in the top-k order, -1 padded).                */
int frr_rpn_proposals_workspace_layout(int B, int N, int pre_nms_top_k, int post_nms_top_k, size_t* offsets6);
/* nms_cluster_size = CTAs per image of the NMS (1, 2, 4, 8, 16; 0 = automatic, the lowest latency of ONE call: 2 at 64
 * images, 8-16 for a single image).  1 spends the least SM time per image (9.4 k vs 15.5 k SM-microseconds per 64
 * images): the setting for several batches in flight on different streams (region.ProposalPipeline), where the other
 * batches' kernels fill the SMs a single CTA per image leaves idle.  Results are identical for every setting.
 * image_hw set: a mixed-size batch padded to (img_h / stride) x (img_w / stride) cells (see frr_rpn_decode_sized); the
 * decode is frr_rpn_decode_sized, top-k and NMS are unchanged (padding cells are invalid; the row-major order of the
 * padded grid keeps each image's relative anchor order, so ties break as for the image alone).  The workspace and the
 * top-k order are those of the padded N.                                                                           */
int frr_rpn_proposals(const float* reg /* [B,N,4] */, const float* cls /* [B,N,2] logits or [B,N] scores */,
                      int cls_is_logits, const float* anchors /* [N,4] or NULL */, const float* base_table_host, int A,
                      int img_h, int img_w, const int32_t* image_hw /* [B,2] device, or NULL */, int stride,
                      float min_size, int B, int N, int pre_nms_top_k, int post_nms_top_k, double iou_thr, float* rois,
                      int32_t* roi_count, void* workspace, size_t workspace_bytes, int nms_cluster_size,
                      frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * R1-R3  RoIPool -- torchvision.ops.RoIPool((7,7), 1.0) at models/model.py:97,113 and its autograd
 *        backward (train.py:36).  Schemas replaced: torchvision::roi_pool(input, rois, spatial_scale,
 *        ph, pw) -> (out, argmax); torchvision::_roi_pool_backward(grad, rois, argmax, ...).
 *        feat [B,C,H,W] fp32, NCHW (channels_last=0) or NHWC memory (channels_last=1);
 *        rois [K,5] = (batch index, x1,y1,x2,y2) fp32; out/argmax [K,C,PH,PW] contiguous
 *        (argmax int32 = h*W+w, -1 for empty bins; may be NULL in inference).
 *        Forward max/argmax bit-exact vs torchvision CPU; backward within 1e-5 (fp32 sum order), or bit-exact through
 *        frr_roi_pool_bwd_deterministic below.
 *        Exception: with argmax == NULL, a 7x7 bin whose maximum is zero may hold +0.0 where torchvision
 *        (first strict maximum) holds -0.0; the values compare equal and every other bit matches.
 * ------------------------------------------------------------------------------------- */
/* R1 glue -- models/model.py:104-110 (roi * [fw,fh,fw,fh]) + TV ops/_utils.py:18-25 (list of per-image rois ->
 * Tensor[K,5] with the batch index): rois [B,R,4] normalised (e.g. the output of frr_rpn_proposals), count [B] or
 * NULL -> rois5 [B*R,5] scaled by the feature grid (fw, fh) = (grid_w, grid_h); rows r >= count[b] get batch index
 * -1 = masked: the RoI kernels skip masked rois (their output rows are not written) and rois whose index is >= B.
 * image_hw set (mixed-size batch, see frr_rpn_decode_sized; grid_h x grid_w = the padded grid): image b's rois are
 * scaled by its own grid (fw_b, fh_b), and the rows of an image with an empty grid are masked. */
int frr_rois5(const float* rois, const int32_t* count, int B, int R, int grid_h, int grid_w,
              const int32_t* image_hw /* [B,2] device, or NULL */, int stride, float* rois5, frr_stream_t stream);
/* image_hw set (mixed-size batch, see frr_rpn_decode_sized; features padded to H x W cells): every bin window of a roi
 * of image b is clipped to [0, fh_b) x [0, fw_b) instead of the padded map, as torchvision does on that image alone: a
 * roi clamped to the image edge has round(x2 * fw_b) == fw_b and loses its last window column there, while the padded
 * map holds padding values in that column.  argmax stays h * W + w, an index into the padded plane, and never points
 * at padding.  fh_b = image_hw[b,0] / stride and fw_b = image_hw[b,1] / stride, clamped to [0, H] / [0, W] (stride 1:
 * image_hw holds the feature extents themselves).  The kernel choice (frr_roi_variant) does not depend on image_hw.
 * frr_roi_pool_bwd needs no extent: it follows argmax, so the padding region of grad_in comes out zero. */
int frr_roi_pool_fwd(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                     float spatial_scale, int channels_last, const int32_t* image_hw /* [B,2] device, or NULL */,
                     int stride, float* out, int32_t* argmax, frr_stream_t stream);
/* grad_in [B,C,H,W] (same memory format as feat) is fully written (no pre-zeroing needed).  Rois of at least 6 feature
 * pixels per side are accumulated in shared memory in a fixed order (bit-reproducible); smaller rois, and every roi on maps
 * whose 8 planes do not fit twice per SM, are added with global fp32 atomics (same sums, order not fixed).  argmax must be
 * the forward's output for the same rois / map shape (torchvision's contract); indices outside [0, H*W) are ignored. */
int frr_roi_pool_bwd(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C, int H,
                     int W, int PH, int PW, float spatial_scale, int channels_last, float* grad_in,
                     frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * R4  RoIAlign -- MultiScaleRoIAlign(7, sampling_ratio=2) at models/new_model.py:127,143
 *     (torchvision::roi_align / _roi_align_backward, aligned=False on the reference path).
 * ------------------------------------------------------------------------------------- */
int frr_roi_align_fwd(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                      float spatial_scale, int sampling_ratio, int aligned, int channels_last, float* out,
                      frr_stream_t stream);
int frr_roi_align_bwd(const float* grad_out, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                      float spatial_scale, int sampling_ratio, int aligned, int channels_last, float* grad_in,
                      frr_stream_t stream);

/* Deterministic backward, bit-exact with torchvision's CPU kernels (torchvision::_roi_pool_backward /
 * _roi_align_backward on CPU): the arguments of frr_roi_pool_bwd (plus image_hw, stride) / frr_roi_align_bwd, for callers
 * that need the same gradient bits on every run (torch.use_deterministic_algorithms).
 * grad_in[b,c,p] is the fp32 sum, starting at +0.0, of the following terms, added in this order.  Only rois with
 * 0 <= (int)rois[k,0] < B count, taken in ascending k.
 *  - RoIPool: for each k, then ph, then pw (row-major): grad_out[k,c,ph,pw] if argmax[k,c,ph,pw] == p and p lies inside
 *    that bin's clipped window.  The forward only produces argmax values of that kind; a value that is -1, out of range
 *    or outside the window contributes nothing.
 *  - RoIAlign: for each k, then ph, pw, iy, ix, then tap 1, 2, 3, 4 of a valid sample: (go * w_t) / count whenever tap
 *    t lands on p (torchvision's bilinear_interpolate_gradient arithmetic).  At the last row or column the snapped taps
 *    land on the same pixel and are added separately, in tap order.  The division is IEEE round-to-nearest (exact for
 *    counts below 2^27 samples per bin).
 * The result is a pure function of the inputs: the same on any stream, inside or outside a CUDA graph, whatever else
 * runs; no atomic touches a value.  NaN / Inf in grad_out reach the same elements as in the CPU loop.  grad_in is fully
 * written (no pre-zeroing needed), NCHW or channels_last like the entry points above.  grad_out / argmax must be
 * 4-byte aligned; PH and PW up to about 70 (a one-channel ring of four rois must fit shared memory). */
/* image_hw set (mixed-size batch): "p lies inside that bin's clipped window" uses image b's extent, exactly as
 * frr_roi_pool_fwd clips with the same image_hw and stride; the padding region of grad_in is written as +0.0. */
int frr_roi_pool_bwd_deterministic(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C,
                                   int H, int W, int PH, int PW, float spatial_scale, int channels_last,
                                   const int32_t* image_hw /* [B,2] device, or NULL */, int stride, float* grad_in,
                                   frr_stream_t stream);
int frr_roi_align_bwd_deterministic(const float* grad_out, const float* rois, int K, int B, int C, int H, int W, int PH,
                                    int PW, float spatial_scale, int sampling_ratio, int aligned, int channels_last,
                                    float* grad_in, frr_stream_t stream);

/* MultiScaleRoIAlign level assignment -- TV ops/poolers.py LevelMapper as used by models/new_model.py:127,143:
 * level = clamp(floor(canonical_level + log2(sqrt(area)/canonical_scale) + 1e-6), k_min, k_max) - k_min, rois in image
 * coordinates.  Writes levels int32 [K] and rois_per_level [L,K,5]: copy l keeps the batch index of the rois of level l
 * and sets it to -1 for the others; frr_roi_align_fwd/bwd skip rois with a negative batch index, so the L per-level
 * launches fill one [K,C,PH,PW] output without gathers or host synchronisation.  L = k_max - k_min + 1. */
int frr_fpn_level_rois(const float* rois5, int K, int k_min, int k_max, int canonical_level, float canonical_scale, int L,
                       int32_t* levels, float* rois_per_level, frr_stream_t stream);

/* Which kernel the RoI entry points pick (host only, launches nothing; tests assert through it that the kernel they mean
 * to exercise is the one that runs).  op: 0 frr_roi_pool_fwd, 1 frr_roi_pool_bwd, 2 frr_roi_align_fwd,
 * 3 frr_roi_align_bwd; want_argmax: the forward's argmax != NULL (same kernel either way).  Assumes 4-byte aligned
 * grad_out / argmax.  out4 = (kernel id, channels per CTA (0: the kernel walks output elements or rois), CTAs per
 * (image, channel group), dynamic shared memory bytes).  Kernel ids:
 * -1 nothing launched (no rois), 0 RoIPool forward flat, 1 RoIAlign forward fast, 2 forward planes, 3 forward direct,
 * 4 RoIPool backward colour classes + tail, 5 RoIPool backward tail only, 6 RoIAlign backward fast,
 * 7 RoIAlign backward stream, 8 backward planes, 9 backward direct. */
int frr_roi_variant(int op, int K, int B, int C, int H, int W, int PH, int PW, int sampling_ratio, int want_argmax,
                    int32_t* out4);

/* ---------------------------------------------------------------------------------------
 * T1  RPN target maker -- RPNTargetMaker.forward, models/model.py:186-266 (IoU: utils/util.py:66-102).
 *     Two kernels around one small D2H copy, because the reference samples with torch.randperm on
 *     the host generator (:228,:235):
 *       assign   -> iou_max/argmax [B,N], label8 [B,N] (1 pos, 0 neg, -1 ignore, -2 outside image),
 *                   order-preserving pos_list/neg_list [B,N] and counts [B,2] = (n_pos, n_neg);
 *       finalize -> applies `disable` (positions inside pos_list / neg_list to turn into -1; per image
 *                   disable_off[3b..3b+2] = (start of pos part, start of neg part, end)), encodes
 *                   (utils/util.py:39-43) and writes labels int64 [B,N], reg fp32 [B,N,4].
 *     gt [B,Gmax,4] + gt_count [B] (NULL = Gmax each); anchors [N,4] or NULL (generated, A2).
 *     Thresholds are fp32 compares (reference 0.3f / 0.7f).
 *     Variant knobs: (iou_eps, inside_only, tie_inclusive) = (1e-5f, 1, 0) is models/model.py (VGG);
 *     (0, 0, 1) is RPNTargetMaker of the FPN variant, models/new_model.py:299-349 (box_iou without eps,
 *     util/box_ops.py:24-37; no inside-image filter; every anchor tied at a GT's best IoU becomes positive, :316-318).
 * ------------------------------------------------------------------------------------- */
/* image_hw set: a mixed-size batch (see frr_rpn_decode_sized) padded to img_h x img_w pixels, anchors generated: image
 * b's anchors are divided by its own (W_b, H_b) and the inside-image test is its own; its padding cells behave like
 * anchors outside the image (label8 -2, then label -1 and a zero target).  pos_list / neg_list hold padded indices in
 * the same order as the image's own lists, and counts are the image's own, so the host randperm path and
 * frr_sample_targets draw the same numbers as for the image alone.  iou_max / argmax / label8 / lists / labels / reg
 * are [B,N] of the padded N.  Pass the same image_hw to both calls. */
int frr_rpn_targets_assign(const float* gt, const int32_t* gt_count, int B, int Gmax, const float* anchors,
                           const float* base_table_host, int A, int img_h, int img_w,
                           const int32_t* image_hw /* [B,2] device, or NULL */, int stride, int N,
                           float neg_thr, float pos_thr, float iou_eps, int inside_only, int tie_inclusive,
                           float* iou_max, int32_t* argmax, int8_t* label8,
                           int32_t* pos_list, int32_t* neg_list, int32_t* counts, frr_stream_t stream);
int frr_rpn_targets_finalize(const float* gt, int B, int Gmax, const float* anchors, const float* base_table_host,
                             int A, int img_h, int img_w, const int32_t* image_hw /* [B,2] device, or NULL */, int stride,
                             int N, const int32_t* argmax, int8_t* label8, const int32_t* pos_list,
                             const int32_t* neg_list, const int32_t* disable, const int32_t* disable_off, int64_t* labels,
                             float* reg, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * T3  Fast R-CNN target maker -- FastRcnnTargetMaker.forward, models/model.py:127-179.
 *     assign: boxes = cat(rois[:roi_count], gt[:gt_count]) (M = Rmax+Gmax slots per image), IoU row
 *     max/argmax, pos (IoU >= fg_thr) / neg ordered lists + counts [B,2].
 *     finalize: sel [B,S] = positions in pos_list (first n_pos) then neg_list; sel_n [B,2] =
 *     (n_pos, n_total); writes cls int64 [B,S] (label+1 / 0 / -1 pad), reg [B,S,4] = encode / std,
 *     sample_rois [B,S,4], keep_index int32 [B,S] (index into the concatenated boxes).
 * ------------------------------------------------------------------------------------- */
/* iou_eps: 1e-5f = models/model.py (find_jaccard_overlap), 0 = FRCNNTargetMaker of models/new_model.py:153-206 (box_iou;
 * that variant samples 512 RoIs with <= 128 positives on the host side). */
int frr_frcnn_targets_assign(const float* rois, const int32_t* roi_count, int B, int Rmax, const float* gt,
                             const int32_t* gt_count, int Gmax, float fg_thr, float iou_eps, float* iou_max,
                             int32_t* argmax, int8_t* label8, int32_t* pos_list, int32_t* neg_list, int32_t* counts,
                             frr_stream_t stream);
int frr_frcnn_targets_finalize(const float* rois, const int32_t* roi_count, int B, int Rmax, const float* gt,
                               const int64_t* gt_label, int Gmax, const int32_t* argmax, const int32_t* pos_list,
                               const int32_t* neg_list, const int32_t* sel, const int32_t* sel_n, int S,
                               const float* std4_host, int label_offset /* 1: models/model.py:141, 0: new_model.py:166 */,
                               int64_t* cls, float* reg, float* sample_rois, int32_t* keep_index, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * T1/T3 sampling without the host round trip -- the torch.randperm draws of models/model.py:149,155,228,235
 *     (models/new_model.py:169-177,328-343) replayed on the device from a device-resident copy of torch's CPU
 *     mt19937 state: mt_state uint32 [626] = the 624 state words, [624] = index of the next unread word (624 =
 *     exhausted), [625] reserved; read and advanced in place exactly as the reference's draws would advance it
 *     (per image: RPN positives if n_pos > rpn_max_pos, RPN negatives if n_neg > rpn_batch - n_pos, then both
 *     Fast R-CNN permutations, always).  rpn_counts / frcnn_counts = the counts [B,2] of the assign kernels (either may
 *     be NULL: that maker is not sampled).  RPN: label8 [B,N] is edited in place (then call frr_rpn_targets_finalize
 *     with disable = NULL); Fast R-CNN: writes sel int32 [B,sel_stride] and sel_n [B,2] for frr_frcnn_targets_finalize.
 *     Workspace: jobs int32 [B,4,4] (16-byte aligned), draws uint32 [B,4,draws_stride], draws_stride >= the batch sizes
 *     (<= 512).  Two launches, no synchronisation, no host memory.
 * ------------------------------------------------------------------------------------- */
int frr_sample_targets(const int32_t* rpn_counts, const int32_t* frcnn_counts, int B, int rpn_batch, int rpn_max_pos,
                       int frcnn_batch, int frcnn_max_pos, uint32_t* mt_state, int N, int8_t* rpn_label8,
                       const int32_t* rpn_pos_list, const int32_t* rpn_neg_list, int32_t* sel, int32_t* sel_n,
                       int sel_stride, int32_t* jobs, uint32_t* draws, int draws_stride, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Loss side (SURVEY 8f) -- losses/loss.py:5-59 (SmoothL1Loss, RPNLoss, FastRCNNLoss) fused with the class-row gather of
 *     models/model.py:340-341, per image: rpn_cls [B,N,2], rpn_reg [B,N,4], rpn_target_cls int64 [B,N] in {-1,0,1},
 *     rpn_target_reg [B,N,4]; frcnn_cls [B,S,C], frcnn_reg [B,S,frcnn_reg_rows,4] (frcnn_reg_rows = C: the head output,
 *     the row of the target class is picked here; 1: already gathered like the reference's loss input),
 *     frcnn_target_cls int64 [B,S] (negative = padding of a short sample), frcnn_target_reg [B,S,4].
 *     loss [B,5] = (total, rpn_cls, rpn_reg, frcnn_cls, frcnn_reg).  The grad_* tensors (same shapes as the predictions,
 *     any may be NULL) receive d loss_component / d prediction for a unit upstream gradient.  Either half may be NULL.
 *     An image with no sampled anchor (or no non-padding row) gets NaN for that half's two losses, like the
 *     reference's 0 / 0, and zero gradients.  A Fast R-CNN class >= C is not checked (a host-side check would
 *     synchronise a captured or compiled step): the row counts in the normaliser and adds no loss term and no
 *     gradient, where the reference raises.  Non-finite logits give what the reference's fp32 cross entropy gives:
 *     NaN for a row with +inf or with every logit -inf, +inf for -inf in the target class only.
 * ------------------------------------------------------------------------------------- */
int frr_region_loss(const float* rpn_cls, const float* rpn_reg, const int64_t* rpn_target_cls, const float* rpn_target_reg,
                    int B, int N, const float* frcnn_cls, const float* frcnn_reg, const int64_t* frcnn_target_cls,
                    const float* frcnn_target_reg, int S, int C, int frcnn_reg_rows, float rpn_beta, float frcnn_beta,
                    float* loss, float* grad_rpn_cls, float* grad_rpn_reg, float* grad_frcnn_cls, float* grad_frcnn_reg,
                    frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * D1  predict tail -- models/model.py:369-378: prob = softmax(cls); boxes = clamp(cxcy_to_xy(
 *     decode(reg*std, xy_to_cxcy(roi))), 0, 1) per class.  cls [rows,C], reg [rows,C,4],
 *     rois [rows,4] -> prob [rows,C], boxes [rows,C,4].
 * D2  FRCNN._suppress -- models/model.py:382-402 for a batch: per class l>=1, prob > score_thres,
 *     NMS at iou_thr (double compare), class-major output.  prob [B,R,C], boxes [B,R,C,4] ->
 *     det_boxes [B,cap,4], det_labels int32 [B,cap] (= l-1, -1 pad), det_scores [B,cap],
 *     det_count [B].  Workspace from frr_class_nms_workspace_bytes, 256-byte aligned.
 * ------------------------------------------------------------------------------------- */
int frr_decode_classwise(const float* cls_logits, const float* reg, const float* rois, int rows, int C,
                         const float* std4_host, float* prob, float* boxes, frr_stream_t stream);
size_t frr_class_nms_workspace_bytes(int B, int R, int C);
int frr_class_nms(const float* prob, const float* boxes, const int32_t* roi_count, int B, int R, int C,
                  float score_thres, double iou_thr, int cap, float* det_boxes, int32_t* det_labels,
                  float* det_scores, int32_t* det_count, void* workspace, size_t workspace_bytes,
                  frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Evaluation hand-off -- test.py:68-88 (boxes * (w,h,w,h)), evaluation/coco_eval.py:70-92,156-158 (convert_to_xywh).
 *     Packs the first max_det detections of every image into fixed-shape rows (x, y, x2|w, y2|h, score, label)
 *     [B,max_det,6] (zero padded) + int32 counts, ready for one tensor all-gather instead of the pickled
 *     all_gather of util/misc.py:89-129.  image_wh [B,2] device floats (w, h) or NULL (keep normalised).
 * ------------------------------------------------------------------------------------- */
int frr_pack_detections(const float* det_boxes /* [B,cap,4] */, const int32_t* det_labels /* [B,cap] */,
                        const float* det_scores /* [B,cap] */, const int32_t* det_count /* [B] */, int B, int cap,
                        int max_det, const float* image_wh, int xywh, float* out /* [B,max_det,6] */,
                        int32_t* out_count /* [B] */, frr_stream_t stream);
/* The same rows for each image's max_det HIGHEST-SCORING detections, the selection evaluators make (torchvision /
 * Detectron keep the top 100 per image by score; COCOeval keeps the top maxDets per (image, category) by score),
 * where frr_pack_detections keeps the first max_det in class order.  Of image b's det_count[b] class-major rows
 * (frr_class_nms's output), per_class_max > 0 first drops every row at position >= per_class_max inside its class;
 * the rest are ordered by score, descending, lower class-major position first on equal scores, and the first max_det
 * are packed exactly as frr_pack_detections packs a row (same scaling, same xywh, zero padding past out_count[b]).
 * Only the rows frr_class_nms kept are ranked: leave its cap at R*(C-1) for a complete ranking.
 * min(max_det, cap) <= 16384, and the top-k's shared-memory limit on cap applies (cap <= 65536 always fits).
 * Workspace from frr_pack_detections_ranked_workspace_bytes, 256-byte aligned.  Three launches: eligibility mask,
 * the top-k of frr_topk_desc_opt over the masked scores, gather into the packed rows. */
size_t frr_pack_detections_ranked_workspace_bytes(int B, int cap, int max_det);
int frr_pack_detections_ranked(const float* det_boxes /* [B,cap,4] */, const int32_t* det_labels /* [B,cap] */,
                               const float* det_scores /* [B,cap] */, const int32_t* det_count /* [B] */, int B,
                               int cap, int max_det, int per_class_max, const float* image_wh, int xywh,
                               float* out /* [B,max_det,6] */, int32_t* out_count /* [B] */, void* workspace,
                               size_t workspace_bytes, frr_stream_t stream);

#ifdef __cplusplus
#pragma GCC visibility pop
}
#endif
#endif /* FRR_H_ */
