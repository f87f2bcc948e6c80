// RegionProposal.forward for a batch in ONE C-ABI call (models/model.py:17-58): decode + clip + min-size
// -> top-k -> NMS -> first post_nms_top_k boxes.  Three kernel launches on the caller's stream, every
// intermediate lives in the caller-provided workspace; no allocation, no synchronisation, graph-capturable.
#include "nms_common.cuh"

namespace frr {

int topk_desc_impl(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k, float* out_scores,
                   int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count, int cluster_hint,
                   frr_stream_t stream);

struct ProposalWs {
    size_t boxes, scores, valid, top_idx, top_count, keep, total;
};

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

static ProposalWs proposal_ws(int B, int N, int k, int post) {
    ProposalWs w;
    size_t o = 0;
    w.boxes = o;     o += al256((size_t)B * N * 16);
    w.scores = o;    o += al256((size_t)B * N * 4);
    w.valid = o;     o += al256((size_t)B * N);
    w.top_idx = o;   o += al256((size_t)B * k * 4);
    w.top_count = o; o += al256((size_t)B * 4);
    w.keep = o;      o += al256((size_t)B * post * 4);
    w.total = o;
    return w;
}

}  // namespace frr

extern "C" {

size_t frr_rpn_proposals_workspace_bytes(int B, int N, int pre_nms_top_k, int post_nms_top_k) {
    if (B < 0 || N < 0 || pre_nms_top_k < 0 || post_nms_top_k < 0) return 0;
    const int k = pre_nms_top_k < N ? pre_nms_top_k : N;
    return frr::proposal_ws(B, N, k, post_nms_top_k).total;
}

int frr_rpn_proposals_workspace_layout(int B, int N, int pre_nms_top_k, int post_nms_top_k, size_t* offsets6) {
    using namespace frr;
    FRR_CHECK_ARG(offsets6 && B >= 0 && N >= 0 && pre_nms_top_k >= 0 && post_nms_top_k >= 0,
                  "frr_rpn_proposals_workspace_layout: bad arguments");
    const int k = pre_nms_top_k < N ? pre_nms_top_k : N;
    const ProposalWs w = proposal_ws(B, N, k, post_nms_top_k);
    offsets6[0] = w.boxes;
    offsets6[1] = w.scores;
    offsets6[2] = w.valid;
    offsets6[3] = w.top_idx;
    offsets6[4] = w.top_count;
    offsets6[5] = w.keep;
    return FRR_OK;
}

// image_hw == nullptr: one size (img_h, img_w) for the batch; else a batch padded to (img_h / stride) x (img_w / stride)
// cells with per-image sizes.  Top-k and NMS are the same for both: padding cells are invalid after the decode, and the
// row-major order of the padded grid keeps the relative order of every image's cells.
int frr_rpn_proposals(const float* reg, const float* cls, int cls_is_logits, const float* anchors,
                      const float* base_table_host, int A, int img_h, int img_w, const int32_t* image_hw, int stride,
                      float min_size, int B, int N, int pre_nms_top_k, int post_nms_top_k, double iou_thr, float* rois,
                      int32_t* roi_count, void* workspace, size_t workspace_bytes, int nms_cluster_size,
                      frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(nms_cluster_size == 0 || nms_cluster_size == 1 || nms_cluster_size == 2 || nms_cluster_size == 4 ||
                      nms_cluster_size == 8 || nms_cluster_size == 16,
                  "frr_rpn_proposals: nms_cluster_size must be 0 (automatic), 1, 2, 4, 8 or 16");
    FRR_CHECK_ARG(B >= 0 && N >= 0 && pre_nms_top_k >= 1 && post_nms_top_k >= 1, "frr_rpn_proposals: bad sizes");
    FRR_CHECK_ARG(rois && roi_count && aligned16(rois), "frr_rpn_proposals: rois must be non-null and 16-byte aligned");
    FRR_CHECK_ARG(image_hw == nullptr || (anchors == nullptr && stride > 0),
                  "frr_rpn_proposals: with image_hw, anchors must be NULL and stride > 0");
    if (B == 0) return FRR_OK;
    const int k = pre_nms_top_k < N ? pre_nms_top_k : N;  // models/model.py:46-47
    const ProposalWs w = proposal_ws(B, N, k, post_nms_top_k);
    FRR_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 255u) == 0,
                  "frr_rpn_proposals: workspace must be non-null and 256-byte aligned");
    if (workspace_bytes < w.total) {
        set_error("frr_rpn_proposals: workspace too small (%zu < %zu)", workspace_bytes, w.total);
        return FRR_E_WORKSPACE;
    }
    char* p = static_cast<char*>(workspace);
    float* boxes = reinterpret_cast<float*>(p + w.boxes);
    float* scores = reinterpret_cast<float*>(p + w.scores);
    uint8_t* valid = reinterpret_cast<uint8_t*>(p + w.valid);
    int32_t* top_idx = reinterpret_cast<int32_t*>(p + w.top_idx);
    int32_t* top_count = reinterpret_cast<int32_t*>(p + w.top_count);
    int32_t* keep = reinterpret_cast<int32_t*>(p + w.keep);
    int rc = image_hw ? frr_rpn_decode_sized(reg, cls, cls_is_logits, base_table_host, A, image_hw, img_h / stride,
                                             img_w / stride, stride, min_size, boxes, scores, valid, B, N, stream)
                      : frr_rpn_decode(reg, cls, cls_is_logits, anchors, base_table_host, A, img_h, img_w, stride, min_size,
                                       boxes, scores, valid, B, N, stream);
    if (rc) return rc;
    if (k == 0) {
        FRR_CUDA(cudaMemsetAsync(roi_count, 0, (size_t)B * 4, (cudaStream_t)stream));
        FRR_CUDA(cudaMemsetAsync(rois, 0, (size_t)B * post_nms_top_k * 16, (cudaStream_t)stream));
        return FRR_OK;
    }
    // top-k writes only the sorted indices; NMS gathers the candidates it visits straight from the decoded boxes
    // (nms_cluster_size = 1 is the caller's throughput setting: one CTA per image in the top-k as well)
    rc = topk_desc_impl(scores, valid, nullptr, B, N, k, nullptr, top_idx, nullptr, nullptr, top_count,
                        nms_cluster_size == 1 ? 1 : 0, stream);
    if (rc) return rc;
    // the decoded boxes are clamped to [0,1] (models/model.py:34): unit-range screening
    return nms_launch(boxes, top_count, B, k, iou_thr, post_nms_top_k, keep, roi_count, rois, nms_cluster_size, 0, NmsTune{}, 1,
                      stream, top_idx, N);
}

}  // extern "C"
