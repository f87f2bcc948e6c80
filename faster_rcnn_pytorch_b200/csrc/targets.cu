// T1-T4: RPN / Fast R-CNN target makers (models/model.py:123-266, utils/util.py:39-43,66-102).
//
// Each maker is two kernels around ONE small device->host copy, because the reference draws its
// samples with torch.randperm on the host mt19937 generator (models/model.py:149,155,228,235) and
// bit-exact sampled indices need that stream:
//   assign   : one CTA per image.  IoU (find_jaccard_overlap, eps in the union) of every
//              anchor / roi against the image's GT boxes staged in shared memory, row max + first
//              argmax, per-GT best anchor (shared-memory atomicMax on (iou bits, ~index)), the
//              pre-sampling label, and ORDER-PRESERVING lists of the positive and negative
//              candidates (block scans) + their counts.
//   (host)   : reads counts[B,*], draws the permutations exactly as the reference does, uploads
//              the positions to disable / to select.
//   finalize : applies the sampling, encodes the box targets and writes the padded outputs
//              (labels int64 [B,N] in {-1,0,1}, reg fp32 [B,N,4]; cls int64 [B,128], ...).
// IoU and labels are bit-exact (fp32 IEEE ops, no FMA contraction, fp32 threshold compares);
// encode() carries a logf and is within 1e-5.
#include <cooperative_groups.h>

#include "frr_common.cuh"

namespace frr {

constexpr int kTgtThreads = 1024;
constexpr int kTgtWarps = kTgtThreads / 32;

// utils/util.py:66-102
// eps = 1e-5f: find_jaccard_overlap (utils/util.py:66-102, VGG variant); eps = 0: box_iou (util/box_ops.py:24-37, FPN
// variant: union = (a1 + a2) - inter, and x + 0.0f == x bit for bit)
__device__ __forceinline__ float iou_eps(const float4& a, float area_a, const float4& b, float area_b, float eps) {
    const float w = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.f);
    const float h = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.f);
    const float inter = __fmul_rn(w, h);
    const float uni = __fadd_rn(__fsub_rn(__fadd_rn(area_a, area_b), inter), eps);
    return __fdiv_rn(inter, uni);
}
__device__ __forceinline__ float area_of(const float4& b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

// utils/util.py:22-26 + :39-43: encode(xy_to_cxcy(gt), xy_to_cxcy(anchor))
__device__ __forceinline__ float4 encode_box(const float4& g, const float4& a) {
    const float gcx = __fmul_rn(__fadd_rn(g.z, g.x), 0.5f), gcy = __fmul_rn(__fadd_rn(g.w, g.y), 0.5f);
    const float gw = __fsub_rn(g.z, g.x), gh = __fsub_rn(g.w, g.y);
    const float acx = __fmul_rn(__fadd_rn(a.z, a.x), 0.5f), acy = __fmul_rn(__fadd_rn(a.w, a.y), 0.5f);
    const float aw = __fsub_rn(a.z, a.x), ah = __fsub_rn(a.w, a.y);
    float4 t;
    t.x = __fdiv_rn(__fsub_rn(gcx, acx), aw);
    t.y = __fdiv_rn(__fsub_rn(gcy, acy), ah);
    t.z = logf(__fdiv_rn(gw, aw));
    t.w = logf(__fdiv_rn(gh, ah));
    return t;
}

__device__ __forceinline__ float4 anchor_at(const float4* __restrict__ anchors, const AnchorTable& tab, int i, int fw,
                                            float stride, float W, float H) {
    if (anchors) return anchors[i];
    const int cell = i / tab.A, a = i - cell * tab.A;
    const int y = cell / fw, x = cell - y * fw;
    const float sx = (float)x * stride, sy = (float)y * stride;
    float4 r;
    r.x = __fdiv_rn(__fadd_rn(tab.v[4 * a + 0], sx), W);
    r.y = __fdiv_rn(__fadd_rn(tab.v[4 * a + 1], sy), H);
    r.z = __fdiv_rn(__fadd_rn(tab.v[4 * a + 2], sx), W);
    r.w = __fdiv_rn(__fadd_rn(tab.v[4 * a + 3], sy), H);
    return r;
}

// anchor i of a padded batch (cell-major over a grid fw cells wide) lies inside the image extent ext = (fh, fw)
__device__ __forceinline__ bool in_grid(const AnchorTable& tab, int i, int fw, int2 ext) {
    const int cell = i / tab.A;
    const int y = cell / fw, x = cell - y * fw;
    return y < ext.x && x < ext.y;
}

struct TgtSmem {
    unsigned int warp_tmp[32];
    unsigned int total[2];
};

// Ordered compaction of two flag classes (label == 1 -> list A, label == 0 -> list B) over n items of lab8[], one
// CTA, in two steps so that a cluster can exchange the totals in between: ordered_counts leaves the exclusive prefix of
// every 32-item chunk in cnt_a / cnt_b (shared memory, [nchunks] each) and returns the totals; ordered_write stores
// idx_base + i at out_base + prefix for every flagged item i.
__device__ void ordered_counts(const int8_t* __restrict__ lab8, int n, unsigned int* cnt_a, unsigned int* cnt_b, TgtSmem* ts,
                               unsigned int* total_a, unsigned int* total_b) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = (n + 31) >> 5;
    for (int c = warp; c < nchunks; c += kTgtWarps) {
        const int i = c * 32 + lane;
        const int l = (i < n) ? (int)lab8[i] : -1;
        const unsigned int ma = __ballot_sync(0xffffffffu, l == 1), mb = __ballot_sync(0xffffffffu, l == 0);
        if (lane == 0) { cnt_a[c] = __popc(ma); cnt_b[c] = __popc(mb); }
    }
    __syncthreads();
    unsigned int run_a = 0, run_b = 0;
    for (int base = 0; base < nchunks; base += kTgtThreads) {
        const int c = base + tid;
        const unsigned int va = (c < nchunks) ? cnt_a[c] : 0u, vb = (c < nchunks) ? cnt_b[c] : 0u;
        unsigned int ta, tb;
        const unsigned int ea = block_exclusive_scan(va, ts->warp_tmp, &ta);
        const unsigned int eb = block_exclusive_scan(vb, ts->warp_tmp, &tb);
        __syncthreads();
        if (c < nchunks) { cnt_a[c] = run_a + ea; cnt_b[c] = run_b + eb; }
        run_a += ta;
        run_b += tb;
    }
    __syncthreads();
    *total_a = run_a;
    *total_b = run_b;
}

__device__ void ordered_write(const int8_t* __restrict__ lab8, int n, int idx_base, int32_t* __restrict__ list_a,
                              int32_t* __restrict__ list_b, const unsigned int* cnt_a, const unsigned int* cnt_b) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = (n + 31) >> 5;
    for (int c = warp; c < nchunks; c += kTgtWarps) {
        const int i = c * 32 + lane;
        const int l = (i < n) ? (int)lab8[i] : -1;
        const unsigned int ma = __ballot_sync(0xffffffffu, l == 1), mb = __ballot_sync(0xffffffffu, l == 0);
        const unsigned int lt = (1u << lane) - 1u;
        if (l == 1) list_a[cnt_a[c] + __popc(ma & lt)] = idx_base + i;
        if (l == 0) list_b[cnt_b[c] + __popc(mb & lt)] = idx_base + i;
    }
}

__device__ void ordered_lists(const int8_t* __restrict__ lab8, int n, int32_t* __restrict__ list_a,
                              int32_t* __restrict__ list_b, unsigned int* cnt_a, unsigned int* cnt_b, TgtSmem* ts,
                              int32_t* __restrict__ counts_out) {
    unsigned int ta, tb;
    ordered_counts(lab8, n, cnt_a, cnt_b, ts, &ta, &tb);
    ordered_write(lab8, n, 0, list_a, list_b, cnt_a, cnt_b);
    if (threadIdx.x == 0) { counts_out[0] = (int)ta; counts_out[1] = (int)tb; }
}

// ------------------------------------------------------------------------------------------------
// RPN targets  (models/model.py:186-266)
// ------------------------------------------------------------------------------------------------
// One thread-block CLUSTER per image: the anchors are cut into S contiguous slabs (multiples of 32), one per CTA.  The
// per-GT best anchor is reduced across the cluster by storing every slab's best keys into every CTA's copy through
// distributed shared memory, and the ordered positive / negative lists of the slabs are stitched together by exchanging the slab
// totals the same way: two cluster barriers, no global-memory round trip.  (One CTA per image left 132 of 148 SMs idle
// at 16 images per batch: 87 us for 165 k IoUs.)
constexpr int kTgtMaxCluster = 8;

// kSized: a batch padded to grid_h x fw cells; image b's anchors are divided by its own (W_b, H_b) = image_hw[b] and the
// cells outside its own grid are labelled like anchors outside the image (-2)
template <bool kSized>
__device__ __forceinline__ void rpn_assign_body(const float4* __restrict__ gt, const int32_t* __restrict__ gt_count, int Gmax,
                                                const float4* __restrict__ anchors, AnchorTable tab, int N, int fw,
                                                float stride, float W, float H, float neg_thr, float pos_thr, float eps,
                                                int inside_only, int tie_inclusive, float* __restrict__ iou_max,
                                                int32_t* __restrict__ argmax, int8_t* __restrict__ lab8,
                                                int32_t* __restrict__ pos_list, int32_t* __restrict__ neg_list,
                                                int32_t* __restrict__ counts /* [B,2] */,
                                                const int32_t* __restrict__ image_hw, int grid_h) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TgtSmem* ts = reinterpret_cast<TgtSmem*>(smem_raw);
    unsigned int* xch = reinterpret_cast<unsigned int*>(smem_raw + 160);  // [2][kTgtMaxCluster] slab totals of every rank
    float4* sgt = reinterpret_cast<float4*>(smem_raw + 256);
    float* sga = reinterpret_cast<float*>(sgt + Gmax);
    unsigned long long* best = reinterpret_cast<unsigned long long*>(sga + ((Gmax + 1) & ~1));  // this slab
    unsigned long long* gbest = best + Gmax;                                                      // whole image
    const int nchunks = (N + 31) >> 5;
    const int cpc = (nchunks + S - 1) / S;  // chunks per CTA
    unsigned long long* xbest = gbest + Gmax;                                                     // [S][Gmax] slab bests
    unsigned int* cnt_a = reinterpret_cast<unsigned int*>(xbest + (size_t)kTgtMaxCluster * Gmax);
    unsigned int* cnt_b = cnt_a + cpc;

    const int b = blockIdx.x / S, tid = threadIdx.x;
    const int i0 = min(rank * cpc * 32, N), i1 = min((rank + 1) * cpc * 32, N);  // this CTA's anchors
    int2 ext = make_int2(0, 0);
    if (kSized) {
        ext = image_cells(image_hw, b, (int)stride, grid_h, fw);
        const int2 hw = __ldg(reinterpret_cast<const int2*>(image_hw) + b);
        H = (float)hw.x;
        W = (float)hw.y;
    }
    const int G = min(gt_count ? gt_count[b] : Gmax, Gmax);
    for (int g = tid; g < G; g += kTgtThreads) {
        const float4 v = gt[(size_t)b * Gmax + g];
        sgt[g] = v;
        sga[g] = area_of(v);
        best[g] = 0ull;
        gbest[g] = 0ull;
    }
    __syncthreads();
    float* im = iou_max + (size_t)b * N;
    int32_t* am = argmax + (size_t)b * N;
    int8_t* lb = lab8 + (size_t)b * N;

    // pass 1: row max / first argmax, per-GT best inside anchor (iou bits, then lowest index)
    for (int i = i0 + tid; i < i1; i += kTgtThreads) {
        const float4 a = anchor_at(anchors, tab, i, fw, stride, W, H);
        const bool inside = (!kSized || in_grid(tab, i, fw, ext)) &&
                            (!inside_only || ((a.x >= 0.f) && (a.y >= 0.f) && (a.z <= 1.f) && (a.w <= 1.f)));
        float mx = 0.f;
        int arg = 0;
        int8_t l = -2;  // outside the image
        if (inside) {
            const float aa = area_of(a);
            mx = -1.f;
            for (int g = 0; g < G; ++g) {
                const float v = iou_eps(a, aa, sgt[g], sga[g], eps);
                if (v > mx) { mx = v; arg = g; }
                // key on v + 0: a GT inverted in one axis has IoU -0.0 with the anchors smaller than its |area| (0 over
                // a negative union), whose sign bit would outrank every positive IoU; the reference's argmax takes
                // -0.0 == 0.0 and the first anchor
                const unsigned long long key =
                    ((unsigned long long)__float_as_uint(__fadd_rn(v, 0.f)) << 32) | (unsigned int)(~(unsigned int)i);
                if (key > best[g]) atomicMax(&best[g], key);
            }
            l = (mx < neg_thr) ? 0 : -1;
            if (mx >= pos_thr) l = 1;
        }
        im[i] = mx;
        am[i] = arg;
        lb[i] = l;
    }
    __syncthreads();
    if (S > 1) {
        // every CTA stores its slab's best keys into slot `rank` of every CTA's xbest (plain remote stores), then takes
        // the maximum over the slots locally.  (64-bit atomicMax on a remote shared-memory address gave wrong maxima.)
        cluster.sync();  // all CTAs of the cluster have started: their shared memory may be written
        for (int e = tid; e < G * S; e += kTgtThreads) {
            const int g = e / S, r = e - g * S;
            cluster.map_shared_rank(xbest, r)[(size_t)rank * Gmax + g] = best[g];
        }
        cluster.sync();
        for (int g = tid; g < G; g += kTgtThreads) {
            unsigned long long k = 0ull;
            for (int r = 0; r < S; ++r) k = max(k, xbest[(size_t)r * Gmax + g]);
            gbest[g] = k;
        }
        __syncthreads();
    } else {
        for (int g = tid; g < G; g += kTgtThreads) gbest[g] = best[g];
        __syncthreads();
    }
    if (!tie_inclusive) {
        // label[argmax over anchors per GT (first index on tie)] = 1  (models/model.py:206-213); overrides the negative label
        for (int g = tid; g < G; g += kTgtThreads) {
            const unsigned long long k = gbest[g];
            const int idx = (int)(~(unsigned int)(k & 0xffffffffull));
            if (k != 0ull && idx >= i0 && idx < i1) lb[idx] = 1;
        }
    } else {
        // FPN variant (models/new_model.py:316-318): EVERY anchor whose IoU equals the per-GT maximum becomes positive
        // (torch.where(iou == max)), including the degenerate "max == 0" case
        for (int i = i0 + tid; i < i1; i += kTgtThreads) {
            if (lb[i] == -2) continue;
            const float4 a = anchor_at(anchors, tab, i, fw, stride, W, H);
            const float aa = area_of(a);
            bool hit = false;
            for (int g = 0; g < G; ++g) {
                const unsigned long long k = gbest[g];
                if (k != 0ull && iou_eps(a, aa, sgt[g], sga[g], eps) == __uint_as_float((unsigned int)(k >> 32))) hit = true;
            }
            if (hit) lb[i] = 1;
        }
    }
    __syncthreads();
    // ordered lists: slab counts, totals exchanged through distributed shared memory, slab written at its offset
    unsigned int ta, tb;
    ordered_counts(lb + i0, i1 - i0, cnt_a, cnt_b, ts, &ta, &tb);
    unsigned int base_a = 0, base_b = 0, tot_a = ta, tot_b = tb;
    if (S > 1) {
        if (tid < S) {
            unsigned int* dst = cluster.map_shared_rank(xch, tid);
            dst[rank] = ta;
            dst[kTgtMaxCluster + rank] = tb;
        }
        cluster.sync();
        tot_a = tot_b = 0;
        for (int r = 0; r < S; ++r) {
            const unsigned int va = xch[r], vb = xch[kTgtMaxCluster + r];
            if (r < rank) { base_a += va; base_b += vb; }
            tot_a += va;
            tot_b += vb;
        }
    }
    ordered_write(lb + i0, i1 - i0, i0, pos_list + (size_t)b * N + base_a, neg_list + (size_t)b * N + base_b, cnt_a, cnt_b);
    if (rank == 0 && tid == 0) { counts[2 * b] = (int)tot_a; counts[2 * b + 1] = (int)tot_b; }
}
__global__ void __launch_bounds__(kTgtThreads)
    rpn_assign_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_count, int Gmax,
                      const float4* __restrict__ anchors, AnchorTable tab, int N, int fw, float stride, float W, float H,
                      float neg_thr, float pos_thr, float eps, int inside_only, int tie_inclusive,
                      float* __restrict__ iou_max, int32_t* __restrict__ argmax,
                      int8_t* __restrict__ lab8, int32_t* __restrict__ pos_list, int32_t* __restrict__ neg_list,
                      int32_t* __restrict__ counts /* [B,2] */) {
    rpn_assign_body<false>(gt, gt_count, Gmax, anchors, tab, N, fw, stride, W, H, neg_thr, pos_thr, eps, inside_only,
                           tie_inclusive, iou_max, argmax, lab8, pos_list, neg_list, counts, nullptr, 0);
}
__global__ void __launch_bounds__(kTgtThreads)
    rpn_assign_sized_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_count, int Gmax, AnchorTable tab,
                            int N, int grid_h, int grid_w, float stride, const int32_t* __restrict__ image_hw, float neg_thr,
                            float pos_thr, float eps, int inside_only, int tie_inclusive, float* __restrict__ iou_max,
                            int32_t* __restrict__ argmax, int8_t* __restrict__ lab8, int32_t* __restrict__ pos_list,
                            int32_t* __restrict__ neg_list, int32_t* __restrict__ counts /* [B,2] */) {
    rpn_assign_body<true>(gt, gt_count, Gmax, nullptr, tab, N, grid_w, stride, 0.f, 0.f, neg_thr, pos_thr, eps, inside_only,
                          tie_inclusive, iou_max, argmax, lab8, pos_list, neg_list, counts, image_hw, grid_h);
}

// kSized: image b's anchors divided by its own (W_b, H_b); its padding cells carry label -2 from the assign kernel
template <bool kSized>
__device__ __forceinline__ void rpn_finalize_body(const float4* __restrict__ gt, int Gmax, const float4* __restrict__ anchors,
                                                  AnchorTable tab, int N, int fw, float stride, float W, float H,
                                                  const int32_t* __restrict__ argmax, int8_t* __restrict__ lab8,
                                                  const int32_t* __restrict__ pos_list, const int32_t* __restrict__ neg_list,
                                                  const int32_t* __restrict__ disable, const int32_t* __restrict__ disable_off,
                                                  int64_t* __restrict__ labels, float4* __restrict__ reg,
                                                  const int32_t* __restrict__ image_hw) {
    // grid = (anchor slabs, images): every CTA finalises a contiguous slab of one image's anchors
    const int b = blockIdx.y, tid = threadIdx.x;
    if (kSized) {
        const int2 hw = __ldg(reinterpret_cast<const int2*>(image_hw) + b);
        H = (float)hw.x;
        W = (float)hw.y;
    }
    const int per = (((N + (int)gridDim.x - 1) / (int)gridDim.x) + 31) & ~31;
    const int i0 = min((int)blockIdx.x * per, N), i1 = min(i0 + per, N);
    int8_t* lb = lab8 + (size_t)b * N;
    if (disable) {  // host-drawn sample: the entries that fall into this slab
        const int s0 = disable_off[3 * b], s1 = disable_off[3 * b + 1], s2 = disable_off[3 * b + 2];
        for (int p = s0 + tid; p < s2; p += kTgtThreads) {
            const int idx = (p < s1 ? pos_list : neg_list)[(size_t)b * N + disable[p]];
            if (idx >= i0 && idx < i1) lb[idx] = -1;
        }
    }
    __syncthreads();
    for (int i = i0 + tid; i < i1; i += kTgtThreads) {
        const int l = (int)lb[i];
        const size_t o = (size_t)b * N + i;
        if (l == -2) {  // outside the image: label -1, zero target (:256-263)
            labels[o] = -1;
            reg[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            labels[o] = (int64_t)l;
            const float4 a = anchor_at(anchors, tab, i, fw, stride, W, H);
            reg[o] = encode_box(gt[(size_t)b * Gmax + argmax[o]], a);  // :253, for ALL inside anchors
        }
    }
}
__global__ void __launch_bounds__(kTgtThreads)
    rpn_finalize_kernel(const float4* __restrict__ gt, int Gmax, const float4* __restrict__ anchors, AnchorTable tab,
                        int N, int fw, float stride, float W, float H, const int32_t* __restrict__ argmax,
                        int8_t* __restrict__ lab8, const int32_t* __restrict__ pos_list,
                        const int32_t* __restrict__ neg_list, const int32_t* __restrict__ disable /* positions */,
                        const int32_t* __restrict__ disable_off /* [B,3]: start_pos, start_neg, end */,
                        int64_t* __restrict__ labels, float4* __restrict__ reg) {
    rpn_finalize_body<false>(gt, Gmax, anchors, tab, N, fw, stride, W, H, argmax, lab8, pos_list, neg_list, disable,
                             disable_off, labels, reg, nullptr);
}
__global__ void __launch_bounds__(kTgtThreads)
    rpn_finalize_sized_kernel(const float4* __restrict__ gt, int Gmax, AnchorTable tab, int N, int grid_w, float stride,
                              const int32_t* __restrict__ image_hw, const int32_t* __restrict__ argmax,
                              int8_t* __restrict__ lab8, const int32_t* __restrict__ pos_list,
                              const int32_t* __restrict__ neg_list, const int32_t* __restrict__ disable,
                              const int32_t* __restrict__ disable_off, int64_t* __restrict__ labels, float4* __restrict__ reg) {
    rpn_finalize_body<true>(gt, Gmax, nullptr, tab, N, grid_w, stride, 0.f, 0.f, argmax, lab8, pos_list, neg_list, disable,
                            disable_off, labels, reg, image_hw);
}

// ------------------------------------------------------------------------------------------------
// Fast R-CNN targets  (models/model.py:127-179)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTgtThreads)
    frcnn_assign_kernel(const float4* __restrict__ rois, const int32_t* __restrict__ roi_count, int Rmax,
                        const float4* __restrict__ gt, const int32_t* __restrict__ gt_count, int Gmax, float fg_thr, float eps,
                        float* __restrict__ iou_max, int32_t* __restrict__ argmax, int8_t* __restrict__ lab8,
                        int32_t* __restrict__ pos_list, int32_t* __restrict__ neg_list, int32_t* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TgtSmem* ts = reinterpret_cast<TgtSmem*>(smem_raw);
    float4* sgt = reinterpret_cast<float4*>(smem_raw + 256);
    float* sga = reinterpret_cast<float*>(sgt + Gmax);
    const int M = Rmax + Gmax;
    const int nchunks = (M + 31) >> 5;
    unsigned int* cnt_a = reinterpret_cast<unsigned int*>(sga + ((Gmax + 3) & ~3));
    unsigned int* cnt_b = cnt_a + nchunks;

    const int b = blockIdx.x, tid = threadIdx.x;
    const int G = min(gt_count ? gt_count[b] : Gmax, Gmax);
    const int R = min(roi_count ? roi_count[b] : Rmax, Rmax);
    for (int g = tid; g < G; g += kTgtThreads) {
        const float4 v = gt[(size_t)b * Gmax + g];
        sgt[g] = v;
        sga[g] = area_of(v);
    }
    __syncthreads();
    const int m = R + G;  // rois <- cat(rois, gt)  (:135)
    float* im = iou_max + (size_t)b * M;
    int32_t* am = argmax + (size_t)b * M;
    int8_t* lb = lab8 + (size_t)b * M;
    for (int i = tid; i < M; i += kTgtThreads) {
        float mx = 0.f;
        int arg = 0;
        int8_t l = -1;
        if (i < m) {
            const float4 a = (i < R) ? rois[(size_t)b * Rmax + i] : sgt[i - R];
            const float aa = area_of(a);
            mx = -1.f;
            for (int g = 0; g < G; ++g) {
                const float v = iou_eps(a, aa, sgt[g], sga[g], eps);
                if (v > mx) { mx = v; arg = g; }
            }
            if (mx >= fg_thr) l = 1;               // :147
            else if (mx < fg_thr && mx >= 0.f) l = 0;  // :153
        }
        im[i] = mx;
        am[i] = arg;
        lb[i] = l;
    }
    __syncthreads();
    ordered_lists(lb, M, pos_list + (size_t)b * M, neg_list + (size_t)b * M, cnt_a, cnt_b, ts, counts + 2 * b);
}

__global__ void __launch_bounds__(128)
    frcnn_finalize_kernel(const float4* __restrict__ rois, const int32_t* __restrict__ roi_count, int Rmax,
                          const float4* __restrict__ gt, const int64_t* __restrict__ gt_label, int Gmax,
                          const int32_t* __restrict__ argmax, const int32_t* __restrict__ pos_list,
                          const int32_t* __restrict__ neg_list, const int32_t* __restrict__ sel /* [B,S] positions */,
                          const int32_t* __restrict__ sel_n /* [B,2]: n_pos, n_total */, int S, float4 stdv, int label_offset,
                          int64_t* __restrict__ cls, float4* __restrict__ reg, float4* __restrict__ sample_rois,
                          int32_t* __restrict__ keep_index) {
    const int b = blockIdx.x;
    const int M = Rmax + Gmax;
    const int R = min(roi_count ? roi_count[b] : Rmax, Rmax);
    const int n_pos = sel_n[2 * b], n_tot = sel_n[2 * b + 1];
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
        const size_t o = (size_t)b * S + j;
        if (j < n_tot) {
            const int p = sel[o];
            const int idx = (j < n_pos) ? pos_list[(size_t)b * M + p] : neg_list[(size_t)b * M + p];
            const float4 box = (idx < R) ? rois[(size_t)b * Rmax + idx] : gt[(size_t)b * Gmax + (idx - R)];
            const int g = argmax[(size_t)b * M + idx];
            cls[o] = (j < n_pos) ? gt_label[(size_t)b * Gmax + g] + label_offset : 0;  // :141,:165 (+1) / new_model.py:166 (+0)
            float4 t = encode_box(gt[(size_t)b * Gmax + g], box);           // :171
            t.x = __fdiv_rn(t.x, stdv.x);                                   // :174-177 (mean is 0)
            t.y = __fdiv_rn(t.y, stdv.y);
            t.z = __fdiv_rn(t.z, stdv.z);
            t.w = __fdiv_rn(t.w, stdv.w);
            reg[o] = t;
            sample_rois[o] = box;
            keep_index[o] = idx;
        } else {
            cls[o] = -1;
            reg[o] = make_float4(0.f, 0.f, 0.f, 0.f);
            sample_rois[o] = make_float4(0.f, 0.f, 0.f, 0.f);
            keep_index[o] = -1;
        }
    }
}

static size_t rpn_assign_smem(int Gmax, int N, int S) {
    const size_t cpc = (size_t)(((N + 31) / 32 + S - 1) / S);
    return 256 + (size_t)Gmax * 16 + (size_t)((Gmax + 1) & ~1) * 4 + (2 + (size_t)kTgtMaxCluster) * Gmax * 8 + 2 * cpc * 4 + 16;
}
static size_t frcnn_assign_smem(int Gmax, int M) {
    return 256 + (size_t)Gmax * 16 + (size_t)((Gmax + 3) & ~3) * 4 + 2 * (size_t)((M + 31) / 32) * 4 + 16;
}

// anchors given, or generated for the (img_h / stride) x (img_w / stride) grid (with image_hw: the padded grid)
static int anchor_args(AnchorTable* tab, int* fw, const float* anchors, const float* base_table_host, int A, int img_h,
                       int img_w, const int32_t* image_hw, int stride, int N) {
    tab->A = 1;
    *fw = 1;
    FRR_CHECK_ARG(image_hw == nullptr || (anchors == nullptr && aligned8(image_hw)),
                  "rpn targets: with image_hw, anchors must be NULL and image_hw 8-byte aligned");
    if (anchors == nullptr) {
        FRR_CHECK_ARG(img_h > 0 && img_w > 0 && stride > 0, "rpn targets: bad image size");
        int rc = fill_anchor_table(tab, base_table_host, A, stride);
        if (rc) return rc;
        *fw = img_w / stride;
        FRR_CHECK_ARG((long long)(img_h / stride) * (*fw) * tab->A == N, "rpn targets: N=%d does not match the image size", N);
    } else {
        FRR_CHECK_ARG(aligned16(anchors), "rpn targets: anchors must be 16-byte aligned");
    }
    return FRR_OK;
}

// One cluster of S CTAs per image: one CTA per ~2048 anchors, at most 8, and no more CTAs than ~2 per SM for the batch
template <typename... KArgs, typename... Args>
static int launch_rpn_assign(void (*kern)(KArgs...), int B, int N, int Gmax, frr_stream_t stream, Args... args) {
    int S = 1;
    while (S < kTgtMaxCluster && N >= 2048 * (S * 2) && (long)B * (S * 2) <= 2L * num_sms()) S *= 2;
    const size_t smem = rpn_assign_smem(Gmax, N, S);
    FRR_CHECK_ARG(smem <= 227 * 1024, "frr_rpn_targets_assign: Gmax=%d N=%d needs %zu B shared memory", Gmax, N, smem);
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * S), 1, 1);
    cfg.blockDim = dim3((unsigned)kTgtThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FRR_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
    count_launch();
    FRR_CHECK_LAUNCH("rpn_assign_kernel");
    return FRR_OK;
}

// finalize: ~2048 anchors per CTA, about two CTAs per SM for the batch at most
static int finalize_slabs(int B, int N) {
    int slabs = 1;
    while (slabs < 16 && N >= 2048 * (slabs * 2) && (long)B * (slabs * 2) <= 2L * num_sms()) slabs *= 2;
    return slabs;
}

}  // namespace frr

extern "C" {

int frr_rpn_targets_assign(const float* gt, const int32_t* gt_count, int B, int Gmax, const float* anchors,
                           const float* base_table_host, int A, int img_h, int img_w, const int32_t* image_hw, int stride,
                           int N, float neg_thr, float pos_thr, float iou_eps_, int inside_only, int tie_inclusive,
                           float* iou_max, int32_t* argmax, int8_t* label8, int32_t* pos_list, int32_t* neg_list,
                           int32_t* counts, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(gt && iou_max && argmax && label8 && pos_list && neg_list && counts, "frr_rpn_targets_assign: null pointer");
    FRR_CHECK_ARG(B >= 0 && Gmax >= 1 && N >= 1, "frr_rpn_targets_assign: bad sizes (G = 0 is an error in the reference too)");
    FRR_CHECK_ARG(aligned16(gt), "frr_rpn_targets_assign: gt must be 16-byte aligned");
    AnchorTable tab;
    int fw;
    int rc = anchor_args(&tab, &fw, anchors, base_table_host, A, img_h, img_w, image_hw, stride, N);
    if (rc) return rc;
    if (B == 0) return FRR_OK;
    if (image_hw)
        return launch_rpn_assign(rpn_assign_sized_kernel, B, N, Gmax, stream, (const float4*)gt, gt_count, Gmax, tab, N,
                                 img_h / stride, fw, (float)stride, image_hw, neg_thr, pos_thr, iou_eps_, inside_only,
                                 tie_inclusive, iou_max, argmax, label8, pos_list, neg_list, counts);
    return launch_rpn_assign(rpn_assign_kernel, B, N, Gmax, stream, (const float4*)gt, gt_count, Gmax, (const float4*)anchors,
                             tab, N, fw, (float)stride, (float)img_w, (float)img_h, neg_thr, pos_thr, iou_eps_, inside_only,
                             tie_inclusive, iou_max, argmax, label8, pos_list, neg_list, counts);
}

int frr_rpn_targets_finalize(const float* gt, int B, int Gmax, const float* anchors, const float* base_table_host, int A,
                             int img_h, int img_w, const int32_t* image_hw, int stride, int N, const int32_t* argmax,
                             int8_t* label8, const int32_t* pos_list, const int32_t* neg_list, const int32_t* disable,
                             const int32_t* disable_off, int64_t* labels, float* reg, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(gt && argmax && label8 && pos_list && neg_list && labels && reg, "frr_rpn_targets_finalize: null pointer");
    FRR_CHECK_ARG((disable == nullptr) == (disable_off == nullptr), "frr_rpn_targets_finalize: disable/disable_off mismatch");
    FRR_CHECK_ARG(aligned16(gt) && aligned16(reg), "frr_rpn_targets_finalize: gt/reg must be 16-byte aligned");
    AnchorTable tab;
    int fw;
    int rc = anchor_args(&tab, &fw, anchors, base_table_host, A, img_h, img_w, image_hw, stride, N);
    if (rc) return rc;
    if (B == 0) return FRR_OK;
    FRR_CHECK_ARG(B <= 65535, "frr_rpn_targets_finalize: B=%d exceeds the grid limit", B);
    const dim3 grid((unsigned)finalize_slabs(B, N), (unsigned)B);
    if (image_hw)
        rpn_finalize_sized_kernel<<<grid, kTgtThreads, 0, (cudaStream_t)stream>>>(
            (const float4*)gt, Gmax, tab, N, fw, (float)stride, image_hw, argmax, label8, pos_list, neg_list, disable,
            disable_off, labels, (float4*)reg);
    else
        rpn_finalize_kernel<<<grid, kTgtThreads, 0, (cudaStream_t)stream>>>(
            (const float4*)gt, Gmax, (const float4*)anchors, tab, N, fw, (float)stride, (float)img_w, (float)img_h, argmax,
            label8, pos_list, neg_list, disable, disable_off, labels, (float4*)reg);
    count_launch();
    FRR_CHECK_LAUNCH(image_hw ? "rpn_finalize_sized_kernel" : "rpn_finalize_kernel");
    return FRR_OK;
}

int frr_frcnn_targets_assign(const float* rois, const int32_t* roi_count, int B, int Rmax, const float* gt,
                             const int32_t* gt_count, int Gmax, float fg_thr, float iou_eps_, float* iou_max,
                             int32_t* argmax, int8_t* label8, int32_t* pos_list, int32_t* neg_list, int32_t* counts,
                             frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG((rois || Rmax == 0) && gt && iou_max && argmax && label8 && pos_list && neg_list && counts,
                  "frr_frcnn_targets_assign: null pointer");
    FRR_CHECK_ARG(B >= 0 && Rmax >= 0 && Gmax >= 1, "frr_frcnn_targets_assign: bad sizes");
    FRR_CHECK_ARG(aligned16(rois) && aligned16(gt), "frr_frcnn_targets_assign: rois/gt must be 16-byte aligned");
    if (B == 0) return FRR_OK;
    const size_t smem = frcnn_assign_smem(Gmax, Rmax + Gmax);
    FRR_CHECK_ARG(smem <= 227 * 1024, "frr_frcnn_targets_assign: needs %zu B shared memory", smem);
    FRR_CUDA(cudaFuncSetAttribute(frcnn_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    frcnn_assign_kernel<<<B, kTgtThreads, smem, (cudaStream_t)stream>>>((const float4*)rois, roi_count, Rmax,
                                                                         (const float4*)gt, gt_count, Gmax, fg_thr, iou_eps_,
                                                                         iou_max, argmax, label8, pos_list, neg_list, counts);
    count_launch();
    FRR_CHECK_LAUNCH("frcnn_assign_kernel");
    return FRR_OK;
}

int frr_frcnn_targets_finalize(const float* rois, const int32_t* roi_count, int B, int Rmax, const float* gt,
                               const int64_t* gt_label, int Gmax, const int32_t* argmax, const int32_t* pos_list,
                               const int32_t* neg_list, const int32_t* sel, const int32_t* sel_n, int S,
                               const float* std4_host, int label_offset, int64_t* cls, float* reg, float* sample_rois,
                               int32_t* keep_index, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG((rois || Rmax == 0) && gt && gt_label && argmax && pos_list && neg_list && sel && sel_n && cls && reg && sample_rois &&
                      keep_index && std4_host,
                  "frr_frcnn_targets_finalize: null pointer");
    FRR_CHECK_ARG(B >= 0 && S >= 1, "frr_frcnn_targets_finalize: bad sizes");
    FRR_CHECK_ARG(aligned16(rois) && aligned16(gt) && aligned16(reg) && aligned16(sample_rois),
                  "frr_frcnn_targets_finalize: box arrays must be 16-byte aligned");
    if (B == 0) return FRR_OK;
    const float4 stdv = make_float4(std4_host[0], std4_host[1], std4_host[2], std4_host[3]);
    frcnn_finalize_kernel<<<B, 128, 0, (cudaStream_t)stream>>>((const float4*)rois, roi_count, Rmax, (const float4*)gt,
                                                               gt_label, Gmax, argmax, pos_list, neg_list, sel, sel_n, S,
                                                               stdv, label_offset, cls, (float4*)reg, (float4*)sample_rois,
                                                               keep_index);
    count_launch();
    FRR_CHECK_LAUNCH("frcnn_finalize_kernel");
    return FRR_OK;
}

}  // extern "C"
