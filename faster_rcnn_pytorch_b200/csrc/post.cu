// D1/D2: detection post-processing of FRCNN.predict (models/model.py:369-402).
//
//   frr_decode_classwise : softmax over the class logits, reg * (0.1,0.1,0.2,0.2), per-class decode
//                          against the roi, corner form, clamp to [0,1]   (:369-378)
//   frr_class_nms        : FRCNN._suppress (:382-402) for a whole batch in three launches and no host
//                          sync (the reference does 2 D2H copies per class):
//       1. one CTA per (image, class): select prob > thres, stable descending sort (bitonic on
//          (~score bits, row) keys in shared memory), gather the class boxes;
//       2. the cluster keep-list NMS kernel of nms.cu over the B*(C-1) sorted lists at IoU 0.3
//          (double-threshold compare: IoU == 0.3f is suppressed, as torchvision's CPU kernel);
//       3. one CTA per image: class-major compaction into [B, cap, 4] boxes / labels (l-1) / scores.
//   frr_pack_detections        : the evaluation hand-off, the first max_det class-major rows of every image;
//   frr_pack_detections_ranked : the same rows for the max_det highest-scoring detections (optionally at most
//                                per_class_max per class first): an eligibility mask, the top-k of topk_radix.cu over
//                                the masked scores, and a gather into the packed rows.
#include "nms_common.cuh"

namespace frr {

int topk_desc_impl(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k, float* out_scores,
                   int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count, int cluster_hint,
                   frr_stream_t stream);

// ------------------------------------------------------------------------------------------------ D1
// torch's clamp(0, 1): NaN stays NaN (fmaxf alone would turn it into 0), every other value as fminf(fmaxf(.))
__device__ __forceinline__ float clamp01(float v) { return v != v ? v : fminf(fmaxf(v, 0.f), 1.f); }

// one warp per roi row
__global__ void __launch_bounds__(256)
    decode_classwise_kernel(const float* __restrict__ cls, const float4* __restrict__ reg, const float4* __restrict__ rois,
                            int rows, int C, float4 stdv, float* __restrict__ prob, float4* __restrict__ boxes) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* x = cls + (size_t)row * C;
    float m = -INFINITY;
    for (int c = lane; c < C; c += 32) m = fmaxf(m, x[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = __fadd_rn(s, expf(__fsub_rn(x[c], m)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    const float4 r = rois[row];
    // xy_to_cxcy(roi)
    const float rcx = __fmul_rn(__fadd_rn(r.z, r.x), 0.5f), rcy = __fmul_rn(__fadd_rn(r.w, r.y), 0.5f);
    const float rw = __fsub_rn(r.z, r.x), rh = __fsub_rn(r.w, r.y);
    for (int c = lane; c < C; c += 32) {
        prob[(size_t)row * C + c] = __fdiv_rn(expf(__fsub_rn(x[c], m)), s);
        float4 t = reg[(size_t)row * C + c];
        t.x = __fmul_rn(t.x, stdv.x); t.y = __fmul_rn(t.y, stdv.y); t.z = __fmul_rn(t.z, stdv.z); t.w = __fmul_rn(t.w, stdv.w);
        const float cx = __fadd_rn(__fmul_rn(t.x, rw), rcx), cy = __fadd_rn(__fmul_rn(t.y, rh), rcy);
        const float w = __fmul_rn(expf(t.z), rw), h = __fmul_rn(expf(t.w), rh);
        const float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);
        float4 b;
        b.x = clamp01(__fsub_rn(cx, hw));
        b.y = clamp01(__fsub_rn(cy, hh));
        b.z = clamp01(__fadd_rn(cx, hw));
        b.w = clamp01(__fadd_rn(cy, hh));
        boxes[(size_t)row * C + c] = b;
    }
}

// ------------------------------------------------------------------------------------------------ D2
// problem p = image * (C-1) + (l-1).  prob [B,R,C], boxes [B,R,C,4].  Output lists have stride R.
__global__ void __launch_bounds__(256)
    class_sort_kernel(const float* __restrict__ prob, const float4* __restrict__ boxes, const int32_t* __restrict__ roi_count,
                      int R, int C, int P2 /* pow2 >= R */, float thres, float4* __restrict__ sboxes,
                      float* __restrict__ sscores, int32_t* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
    __shared__ int s_n;
    const int p = blockIdx.x;
    const int img = p / (C - 1), l = p % (C - 1) + 1;
    const int Rn = roi_count ? min(roi_count[img], R) : R;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    int mine = 0;
    for (int r = threadIdx.x; r < P2; r += blockDim.x) {
        unsigned long long k = ~0ull;
        if (r < Rn) {
            const float s = prob[((size_t)img * R + r) * C + l];
            if (s > thres) {  // fp32 compare (:388)
                k = ((unsigned long long)(~float_to_ordered(s)) << 32) | (unsigned int)r;
                ++mine;
            }
        }
        keys[r] = k;
    }
    if (mine) atomicAdd(&s_n, mine);
    __syncthreads();
    for (int size = 2; size <= P2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int q = threadIdx.x; q < (P2 >> 1); q += blockDim.x) {
                const int lo = 2 * q - (q & (stride - 1)), hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long a = keys[lo], c2 = keys[hi];
                if ((a > c2) == up) { keys[lo] = c2; keys[hi] = a; }
            }
            __syncthreads();
        }
    const int n = s_n;
    for (int j = threadIdx.x; j < R; j += blockDim.x) {
        const size_t o = (size_t)p * R + j;
        if (j < n) {
            const unsigned long long e = keys[j];
            const int r = (int)(unsigned int)(e & 0xffffffffu);
            sscores[o] = ordered_to_float(~(unsigned int)(e >> 32));
            sboxes[o] = boxes[((size_t)img * R + r) * C + l];
        } else {
            sscores[o] = 0.f;
            sboxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    if (threadIdx.x == 0) counts[p] = n;
}

__global__ void __launch_bounds__(256)
    det_compact_kernel(const float4* __restrict__ kept_boxes, const float* __restrict__ sscores,
                       const int32_t* __restrict__ keep, const int32_t* __restrict__ keep_count, int R, int C, int cap,
                       float4* __restrict__ det_boxes, int32_t* __restrict__ det_labels, float* __restrict__ det_scores,
                       int32_t* __restrict__ det_count) {
    __shared__ int s_off[1024];
    const int img = blockIdx.x;
    const int nc = C - 1;
    if (threadIdx.x == 0) {
        int run = 0;
        for (int l = 0; l < nc; ++l) {
            s_off[l] = run;
            run += keep_count[img * nc + l];
        }
        s_off[nc] = run;
        det_count[img] = min(run, cap);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int l = warp; l < nc; l += nwarps) {
        const int p = img * nc + l;
        const int n = keep_count[p], off = s_off[l];
        for (int j = lane; j < n; j += 32) {
            const int d = off + j;
            if (d < cap) {
                const size_t o = (size_t)img * cap + d;
                det_boxes[o] = kept_boxes[(size_t)p * R + j];
                det_scores[o] = sscores[(size_t)p * R + keep[(size_t)p * R + j]];
                det_labels[o] = l;  // class l+1 -> label l (:397)
            }
        }
    }
    const int total = min(s_off[nc], cap);
    for (int d = total + threadIdx.x; d < cap; d += blockDim.x) {
        const size_t o = (size_t)img * cap + d;
        det_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        det_scores[o] = 0.f;
        det_labels[o] = -1;
    }
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Evaluation hand-off (test.py:68-88 + evaluation/coco_eval.py:70-92,156-158): scale the normalised boxes to pixels,
// optionally convert xyxy -> xywh, and pack detections into fixed-shape rows (x, y, x2|w, y2|h, score, label) for ONE
// tensor all-gather instead of a pickled one.  Both packers write a row through this helper, so a detection gets the
// same bits whichever selection picked it.
__device__ __forceinline__ void pack_row(float* __restrict__ o, float4 bx, float score, int32_t label, float2 wh,
                                         int xywh) {
    const float x1 = __fmul_rn(bx.x, wh.x), y1 = __fmul_rn(bx.y, wh.y);
    const float x2 = __fmul_rn(bx.z, wh.x), y2 = __fmul_rn(bx.w, wh.y);
    o[0] = x1;
    o[1] = y1;
    o[2] = xywh ? __fsub_rn(x2, x1) : x2;
    o[3] = xywh ? __fsub_rn(y2, y1) : y2;
    o[4] = score;
    o[5] = (float)label;
}

// The first max_det class-major rows of every image.
__global__ void __launch_bounds__(128)
    pack_detections_kernel(const float4* __restrict__ det_boxes, const int32_t* __restrict__ det_labels,
                           const float* __restrict__ det_scores, const int32_t* __restrict__ det_count, int cap,
                           int max_det, const float2* __restrict__ image_wh, int xywh, float* __restrict__ out,
                           int32_t* __restrict__ out_count) {
    const int b = blockIdx.x;
    const int n = min(min(det_count[b], cap), max_det);
    const float2 wh = image_wh ? image_wh[b] : make_float2(1.f, 1.f);
    for (int j = threadIdx.x; j < max_det; j += blockDim.x) {
        float* o = out + ((size_t)b * max_det + j) * 6;
        if (j < n) {
            const size_t s = (size_t)b * cap + j;
            pack_row(o, det_boxes[s], det_scores[s], det_labels[s], wh, xywh);
        } else {
#pragma unroll
            for (int q = 0; q < 6; ++q) o[q] = 0.f;
        }
    }
    if (threadIdx.x == 0) out_count[b] = n;
}

// Ranked selection, step 1: valid[b][j] = row j of image b takes part in the ranking.  It must be one of the image's
// det_count[b] rows and, with per_class_max = m > 0, among the first m rows of its class.  The rows are class-major, so
// row j is past its class's cap exactly when row j - m has the same label: no scan over the class is needed.
__global__ void __launch_bounds__(256)
    rank_eligible_kernel(const int32_t* __restrict__ det_labels, const int32_t* __restrict__ det_count, int cap,
                         int per_class_max, uint8_t* __restrict__ valid) {
    const int b = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cap) return;
    const size_t o = (size_t)b * cap + j;
    bool ok = j < det_count[b];
    if (ok && per_class_max > 0 && j >= per_class_max) ok = det_labels[o - per_class_max] != det_labels[o];
    valid[o] = ok ? 1 : 0;
}

// Ranked selection, step 3: packed row i of image b is detection order[b][i] (order [B,k] from the top-k, order_count
// [B] rows valid; both NULL when nothing is ranked).
__global__ void __launch_bounds__(128)
    pack_ranked_kernel(const float4* __restrict__ det_boxes, const int32_t* __restrict__ det_labels,
                       const float* __restrict__ det_scores, int cap, const int32_t* __restrict__ order,
                       const int32_t* __restrict__ order_count, int k, int max_det, const float2* __restrict__ image_wh,
                       int xywh, float* __restrict__ out, int32_t* __restrict__ out_count) {
    const int b = blockIdx.x;
    const int n = order_count ? min(order_count[b], max_det) : 0;
    const float2 wh = image_wh ? image_wh[b] : make_float2(1.f, 1.f);
    for (int i = threadIdx.x; i < max_det; i += blockDim.x) {
        float* o = out + ((size_t)b * max_det + i) * 6;
        if (i < n) {
            const size_t s = (size_t)b * cap + order[(size_t)b * k + i];
            pack_row(o, det_boxes[s], det_scores[s], det_labels[s], wh, xywh);
        } else {
#pragma unroll
            for (int q = 0; q < 6; ++q) o[q] = 0.f;
        }
    }
    if (threadIdx.x == 0) out_count[b] = n;
}

}  // namespace frr

extern "C" {

int frr_decode_classwise(const float* cls_logits, const float* reg, const float* rois, int rows, int C,
                         const float* std4_host, float* prob, float* boxes, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(rows >= 0 && C >= 1, "frr_decode_classwise: bad sizes");
    if (rows == 0) return FRR_OK;
    FRR_CHECK_ARG(cls_logits && reg && rois && prob && boxes && std4_host, "frr_decode_classwise: null pointer");
    FRR_CHECK_ARG(aligned16(reg) && aligned16(rois) && aligned16(boxes), "frr_decode_classwise: box arrays must be 16-byte aligned");
    const float4 stdv = make_float4(std4_host[0], std4_host[1], std4_host[2], std4_host[3]);
    decode_classwise_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(cls_logits, (const float4*)reg,
                                                                               (const float4*)rois, rows, C, stdv, prob,
                                                                               (float4*)boxes);
    count_launch();
    FRR_CHECK_LAUNCH("decode_classwise_kernel");
    return FRR_OK;
}

int frr_pack_detections(const float* det_boxes, const int32_t* det_labels, const float* det_scores, const int32_t* det_count,
                        int B, int cap, int max_det, const float* image_wh, int xywh, float* out, int32_t* out_count,
                        frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(B >= 0 && cap >= 0 && max_det >= 1, "frr_pack_detections: bad sizes");
    if (B == 0) return FRR_OK;
    // with cap == 0 there are no rows to read (class_nms(cap=0) hands over empty, unallocated arrays)
    FRR_CHECK_ARG((cap == 0 || (det_boxes && det_labels && det_scores)) && det_count && out && out_count,
                  "frr_pack_detections: null pointer");
    FRR_CHECK_ARG(aligned16(det_boxes) && (image_wh == nullptr || (reinterpret_cast<uintptr_t>(image_wh) & 7u) == 0),
                  "frr_pack_detections: det_boxes must be 16-byte aligned, image_wh 8-byte aligned");
    pack_detections_kernel<<<B, 128, 0, (cudaStream_t)stream>>>((const float4*)det_boxes, det_labels, det_scores, det_count,
                                                                cap, max_det, (const float2*)image_wh, xywh, out, out_count);
    count_launch();
    FRR_CHECK_LAUNCH("pack_detections_kernel");
    return FRR_OK;
}

// The top-k never needs more than the cap rows an image has.
static int ranked_k(int cap, int max_det) { return cap < max_det ? cap : max_det; }

size_t frr_pack_detections_ranked_workspace_bytes(int B, int cap, int max_det) {
    using namespace frr;
    if (B < 0 || cap < 0 || max_det < 1) return 0;
    const size_t k = (size_t)ranked_k(cap, max_det);
    return align256((size_t)B * cap) + align256((size_t)B * k * 4) + align256((size_t)B * 4);
}

int frr_pack_detections_ranked(const float* det_boxes, const int32_t* det_labels, const float* det_scores,
                               const int32_t* det_count, int B, int cap, int max_det, int per_class_max,
                               const float* image_wh, int xywh, float* out, int32_t* out_count, void* workspace,
                               size_t workspace_bytes, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(B >= 0 && B <= 65535 && cap >= 0 && max_det >= 1 && per_class_max >= 0,
                  "frr_pack_detections_ranked: bad sizes");
    const int k = ranked_k(cap, max_det);
    FRR_CHECK_ARG(k <= 16384, "frr_pack_detections_ranked: min(max_det, cap) = %d exceeds the top-k capacity 16384", k);
    if (B == 0) return FRR_OK;
    FRR_CHECK_ARG((cap == 0 || (det_boxes && det_labels && det_scores)) && det_count && out && out_count && workspace,
                  "frr_pack_detections_ranked: null pointer");
    FRR_CHECK_ARG(aligned16(det_boxes) && (image_wh == nullptr || aligned8(image_wh)) &&
                      (reinterpret_cast<uintptr_t>(workspace) & 255u) == 0,
                  "frr_pack_detections_ranked: det_boxes must be 16-byte aligned, image_wh 8-byte aligned, workspace "
                  "256-byte aligned");
    const size_t need = frr_pack_detections_ranked_workspace_bytes(B, cap, max_det);
    if (workspace_bytes < need) {
        set_error("frr_pack_detections_ranked: workspace too small (%zu < %zu)", workspace_bytes, need);
        return FRR_E_WORKSPACE;
    }
    char* w = (char*)workspace;
    uint8_t* valid = (uint8_t*)w;     w += align256((size_t)B * cap);
    int32_t* order = (int32_t*)w;     w += align256((size_t)B * k * 4);
    int32_t* order_count = (int32_t*)w;
    cudaStream_t st = (cudaStream_t)stream;
    if (k > 0) {
        rank_eligible_kernel<<<dim3((unsigned)((cap + 255) / 256), (unsigned)B), 256, 0, st>>>(det_labels, det_count, cap,
                                                                                            per_class_max, valid);
        count_launch();
        FRR_CHECK_LAUNCH("rank_eligible_kernel");
        // score descending, lower class-major position first on equal scores
        const int rc = topk_desc_impl(det_scores, valid, nullptr, B, cap, k, nullptr, order, nullptr, nullptr, order_count,
                                      0, stream);
        if (rc) return rc;
    }
    pack_ranked_kernel<<<B, 128, 0, st>>>((const float4*)det_boxes, det_labels, det_scores, cap, k > 0 ? order : nullptr,
                                          k > 0 ? order_count : nullptr, k, max_det, (const float2*)image_wh, xywh, out,
                                          out_count);
    count_launch();
    FRR_CHECK_LAUNCH("pack_ranked_kernel");
    return FRR_OK;
}

size_t frr_class_nms_workspace_bytes(int B, int R, int C) {
    using namespace frr;
    const size_t P = (size_t)B * (size_t)(C > 1 ? C - 1 : 0);
    return align256(P * R * 16) * 2 + align256(P * R * 4) * 2 + align256(P * 4) * 2 + 256;
}

int frr_class_nms(const float* prob, const float* boxes, const int32_t* roi_count, int B, int R, int C, float score_thres,
                  double iou_thr, int cap, float* det_boxes, int32_t* det_labels, float* det_scores, int32_t* det_count,
                  void* workspace, size_t workspace_bytes, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(B >= 0 && R >= 0 && C >= 2 && cap >= 0, "frr_class_nms: bad sizes");
    FRR_CHECK_ARG(R <= 4096 && C <= 1024, "frr_class_nms: R <= 4096 and C <= 1024 supported");
    if (B == 0) return FRR_OK;
    // cap == 0 asks for the counts only: the detection arrays are empty and may be null
    FRR_CHECK_ARG(prob && boxes && det_count && workspace && (cap == 0 || (det_boxes && det_labels && det_scores)),
                  "frr_class_nms: null pointer");
    FRR_CHECK_ARG(aligned16(boxes) && aligned16(det_boxes) && (reinterpret_cast<uintptr_t>(workspace) & 255u) == 0,
                  "frr_class_nms: boxes must be 16-byte aligned, workspace 256-byte aligned");
    if (workspace_bytes < frr_class_nms_workspace_bytes(B, R, C)) {
        set_error("frr_class_nms: workspace too small (%zu < %zu)", workspace_bytes, frr_class_nms_workspace_bytes(B, R, C));
        return FRR_E_WORKSPACE;
    }
    const size_t P = (size_t)B * (C - 1);
    char* w = (char*)workspace;
    float4* sboxes = (float4*)w;          w += align256(P * R * 16);
    float4* kboxes = (float4*)w;          w += align256(P * R * 16);
    float* sscores = (float*)w;           w += align256(P * R * 4);
    int32_t* keep = (int32_t*)w;          w += align256(P * R * 4);
    int32_t* counts = (int32_t*)w;        w += align256(P * 4);
    int32_t* keep_count = (int32_t*)w;
    cudaStream_t st = (cudaStream_t)stream;
    if (R > 0) {
        int P2 = 32;
        while (P2 < R) P2 <<= 1;
        class_sort_kernel<<<(unsigned)P, 256, (size_t)P2 * 8, st>>>(prob, (const float4*)boxes, roi_count, R, C, P2,
                                                                    score_thres, sboxes, sscores, counts);
        count_launch();
        FRR_CHECK_LAUNCH("class_sort_kernel");
        int rc = nms_launch((const float*)sboxes, counts, (int)P, R, iou_thr, R, keep, keep_count, (float*)kboxes, 1, 256,
                            NmsTune{}, 0, stream);
        if (rc) return rc;
    } else {
        FRR_CUDA(cudaMemsetAsync(keep_count, 0, P * 4, st));
    }
    det_compact_kernel<<<B, 256, 0, st>>>(kboxes, sscores, keep, keep_count, R, C, cap, (float4*)det_boxes, det_labels,
                                          det_scores, det_count);
    count_launch();
    FRR_CHECK_LAUNCH("det_compact_kernel");
    return FRR_OK;
}

}  // extern "C"
