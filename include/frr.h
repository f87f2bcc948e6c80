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

#define FRR_ABI_VERSION 1

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

/* ---------------------------------------------------------------------------------------
 * P4  pre-NMS top-k, sorted descending -- models/model.py:44-49.  One CTA per image, in shared
 *     memory: monotone bucketing of the scores + exact ranking inside the buckets (radix select + radix
 *     sort for inputs that do not bucket).  Ties: lower index first.  Entries past count[b] are padded
 *     (idx -1, score -inf, box 0).  out_cidx = index into the min-size-compacted array (what
 *     the reference's sort returns), out_idx = index into the full N.  k <= 16384.
 * ------------------------------------------------------------------------------------- */
int frr_topk_desc(const float* scores /* [B,N] */, const uint8_t* valid /* [B,N] or NULL */,
                  const float* boxes /* [B,N,4] or NULL */, int B, int N, int k,
                  float* out_scores /* [B,k] or NULL */, int32_t* out_idx /* [B,k] */,
                  int32_t* out_cidx /* [B,k] or NULL */, float* out_boxes /* [B,k,4] or NULL */,
                  int32_t* out_count /* [B] */, frr_stream_t stream);
/* The same with the CTAs per image chosen by the caller: 0 = automatic (a 2-CTA cluster per image when B * 2 CTAs fit the
 * SMs: lowest latency), 1 = one CTA per image (least SM time: several batches in flight).  Identical results.        */
int frr_topk_desc_opt(const float* scores /* [B,N] */, const uint8_t* valid /* [B,N] or NULL */,
                  const float* boxes /* [B,N,4] or NULL */, int B, int N, int k,
                  float* out_scores /* [B,k] or NULL */, int32_t* out_idx /* [B,k] */,
                  int32_t* out_cidx /* [B,k] or NULL */, float* out_boxes /* [B,k,4] or NULL */,
                  int32_t* out_count /* [B] */, int ctas_per_image, frr_stream_t stream);
/* Profiling variant: dbg_cycles = int64[16] accumulating clock64() cycles of CTA 0 per phase: [0..4] radix kernel
 * (load+validity, select, compaction, sort, write-out; only when image 0 was handed over), [8..13] bucket kernel
 * (load + min/max, histogram, scan, scatter, -, rank + write-out). */
int frr_topk_desc_profile(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k,
                          float* out_scores, int32_t* out_idx, int32_t* out_cidx, float* out_boxes,
                          int32_t* out_count, int64_t* dbg_cycles, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * N1  greedy NMS on score-sorted boxes -- torchvision.ops.nms at models/model.py:53-55
 *     (IoU 0.7, keep[:2000|300]) with torchvision's CPU semantics: fp32 IoU, suppress when
 *     (double)iou > iou_thr.  Keep-list algorithm on a thread-block cluster per image,
 *     stops at max_keep.  keep = positions in the sorted list, ascending, -1 padded.
 *     cluster_size: 0 = auto, else 1,2,4,8,16.
 * ------------------------------------------------------------------------------------- */
int frr_nms_sorted(const float* boxes /* [B,n,4] */, const int32_t* counts /* [B] or NULL (=n) */, int B,
                   int n, double iou_thr, int max_keep, int32_t* keep /* [B,max_keep] */,
                   int32_t* keep_count /* [B] */, float* out_boxes /* [B,max_keep,4] or NULL */,
                   int cluster_size, frr_stream_t stream);
/* Same, with tuning / profiling knobs: threads per CTA (0 = auto, 256, 512 or 1024); dbg_cycles = NULL
 * or int64[16] accumulating per-phase clock64() cycles of CTA 0 (slots: chunks, load, phase1, cluster
 * sync, phase2..5, survivors, fix-point rounds); unit_boxes != 0 = the caller guarantees every coordinate
 * lies in [0,1] (true for the clamped RPN / detection boxes of models/model.py:34,378), which enables a
 * cheaper screening test; results are identical.                                                    */
int frr_nms_sorted_tuned(const float* boxes, const int32_t* counts, int B, int n, double iou_thr, int max_keep,
                         int32_t* keep, int32_t* keep_count, float* out_boxes, int cluster_size, int threads,
                         int64_t* dbg_cycles, int unit_boxes, frr_stream_t stream);

/* Which kernel variant and launch geometry the NMS entry points pick for a problem (host only, launches nothing;
 * tests and bench.py assert through it that the variant they mean to exercise is the one that runs):
 * out4[0] = CTAs per image, out4[1] = threads per CTA, out4[2] = variant (0 exact test only, 1 screened,
 * 2 screened + unit range, 3 unit range + area-class / x-bin bucketed lists), out4[3] = dynamic shared memory.   */
int frr_nms_variant(int B, int n, double iou_thr, int max_keep, int cluster_size, int threads, int unit_boxes,
                    int32_t* out4);

/* Developer knob for the profiling tools: sizes of the first and of the largest chunk of the bucketed variant
 * (multiples of 256 in [256, 2048]) and the lanes per candidate of its screen / pair phases (powers of two <= 32;
 * lanes_screen 0 = automatic: 2 with 1-2 CTAs per image, else 4; lanes_pairs 0 = unchanged).  Process-wide; results
 * never depend on them. */
int frr_nms_bucket_tune(int first_chunk, int max_chunk, int lanes_screen, int lanes_pairs);

/* Same, with the score order given as indices into an unsorted array: candidate i of image b is
 * boxes_src[b][order[b][i]] (boxes_src [B,src_n,4]; order int32 [B,n] = out_idx of frr_topk_desc).  Only the
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
int frr_rpn_proposals(const float* reg /* [B,N,4] */, const float* cls /* [B,N,2] logits or [B,N] scores */,
                      int cls_is_logits, const float* anchors /* [N,4] or NULL */, const float* base_table_host, int A,
                      int img_h, int img_w, int stride, float min_size, int B, int N, int pre_nms_top_k,
                      int post_nms_top_k, double iou_thr, float* rois, int32_t* roi_count, void* workspace,
                      size_t workspace_bytes, frr_stream_t stream);
/* The same call with the NMS launch geometry chosen by the caller: nms_cluster_size = CTAs per image (1, 2, 4, 8, 16;
 * 0 = automatic, the lowest latency of ONE call: 2 at 64 images, 8-16 for a single image).  1 spends the least SM time
 * per image (9.4 k vs 15.5 k SM-microseconds per 64 images): the setting for several batches in flight on different
 * streams (region.ProposalPipeline), where the other batches' kernels fill the SMs a single CTA per image leaves idle.
 * Results are identical for every setting.                                                                        */
int frr_rpn_proposals_opt(const float* reg, const float* cls, int cls_is_logits, const float* anchors,
                          const float* base_table_host, int A, int img_h, int img_w, int stride, float min_size, int B,
                          int N, int pre_nms_top_k, int post_nms_top_k, double iou_thr, float* rois, int32_t* roi_count,
                          void* workspace, size_t workspace_bytes, int nms_cluster_size, frr_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * R1-R3  RoIPool -- torchvision.ops.RoIPool((7,7), 1.0) at models/model.py:97,113 and its autograd
 *        backward (train.py:36).  Schemas replaced: torchvision::roi_pool(input, rois, spatial_scale,
 *        ph, pw) -> (out, argmax); torchvision::_roi_pool_backward(grad, rois, argmax, ...).
 *        feat [B,C,H,W] fp32, NCHW (channels_last=0) or NHWC memory (channels_last=1);
 *        rois [K,5] = (batch index, x1,y1,x2,y2) fp32; out/argmax [K,C,PH,PW] contiguous
 *        (argmax int32 = h*W+w, -1 for empty bins; may be NULL in inference).
 *        Forward max/argmax bit-exact vs torchvision CPU; backward within 1e-5 (fp32 sum order).
 *        Exception: with argmax == NULL, a 7x7 bin whose maximum is zero may hold +0.0 where torchvision
 *        (first strict maximum) holds -0.0; the values compare equal and every other bit matches.
 * ------------------------------------------------------------------------------------- */
/* R1 glue -- models/model.py:104-110 (roi * [fw,fh,fw,fh]) + TV ops/_utils.py:18-25 (list of per-image rois ->
 * Tensor[K,5] with the batch index): rois [B,R,4] normalised (e.g. the output of frr_rpn_proposals), count [B] or
 * NULL -> rois5 [B*R,5]; rows r >= count[b] get batch index -1 = masked: the RoI kernels skip masked rois (their
 * output rows are not written) and rois whose index is >= B. */
int frr_rois5(const float* rois, const int32_t* count, int B, int R, float fw, float fh, float* rois5,
              frr_stream_t stream);
int frr_roi_pool_fwd(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                     float spatial_scale, int channels_last, float* out, int32_t* argmax, frr_stream_t stream);
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
 * grad_out / argmax and reads FRR_ROI_POOL_BWD like the launchers.  out4 = (kernel id, channels per CTA (0: the kernel
 * walks output elements or rois), CTAs per (image, channel group), dynamic shared memory bytes).  Kernel ids:
 * -1 nothing launched (no rois), 0 RoIPool forward flat, 1 RoIAlign forward fast, 2 forward planes, 3 forward direct,
 * 4 RoIPool backward colour classes + tail, 5 RoIPool backward tail only, 6 RoIAlign backward fast,
 * 7 RoIAlign backward stream, 8 backward planes, 9 backward direct. */
int frr_roi_variant(int op, int K, int B, int C, int H, int W, int PH, int PW, int sampling_ratio, int want_argmax,
                    int32_t* out4);

/* Developer hook: per-phase clock64() cycles of CTA (0,0) of the 7x7 fast kernels, accumulated since the last call
 * (16 slots, see roi_fast.cu); copies to host_out16 and clears.  Synchronises the device. */
int frr_roi_debug_cycles(int64_t* host_out16);

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
int frr_rpn_targets_assign(const float* gt, const int32_t* gt_count, int B, int Gmax, const float* anchors,
                           const float* base_table_host, int A, int img_h, int img_w, int stride, int N,
                           float neg_thr, float pos_thr, float iou_eps, int inside_only, int tie_inclusive,
                           float* iou_max, int32_t* argmax, int8_t* label8,
                           int32_t* pos_list, int32_t* neg_list, int32_t* counts, frr_stream_t stream);
int frr_rpn_targets_finalize(const float* gt, int B, int Gmax, const float* anchors, const float* base_table_host,
                             int A, int img_h, int img_w, int stride, int N, const int32_t* argmax, int8_t* label8,
                             const int32_t* pos_list, const int32_t* neg_list, const int32_t* disable,
                             const int32_t* disable_off, int64_t* labels, float* reg, frr_stream_t stream);

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

#ifdef __cplusplus
#pragma GCC visibility pop
}
#endif
#endif /* FRR_H_ */
