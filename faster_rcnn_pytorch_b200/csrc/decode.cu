// A2 + P1 + P2 + P3: anchors, fg softmax, box decode, clamp and min-size test in one pass.
//
// Reference: anchor.py:34-55, models/model.py:20,31-41, utils/util.py:15-26,46-50.
// HBM-bound streaming kernel: per anchor it reads reg (16 B) + logits (8 B) and writes the box
// (16 B), the score (4 B) and a validity byte -> 44 B/anchor algorithmic (SURVEY §8d).  Anchors
// are rebuilt in registers from the 9x4 table (kernel parameter) so no anchor tensor is read.
// Parity-critical arithmetic uses explicit round-to-nearest intrinsics (no FMA contraction).
#include "frr_common.cuh"

namespace frr {

__device__ __forceinline__ float4 make_anchor(const AnchorTable& tab, int cell, int a, int fw, float stride, float W,
                                              float H) {
    const int y = cell / fw, x = cell - y * fw;
    const float sx = (float)x * stride, sy = (float)y * stride;  // exact: small integers
    float4 r;
    r.x = __fdiv_rn(__fadd_rn(tab.v[4 * a + 0], sx), W);
    r.y = __fdiv_rn(__fadd_rn(tab.v[4 * a + 1], sy), H);
    r.z = __fdiv_rn(__fadd_rn(tab.v[4 * a + 2], sx), W);
    r.w = __fdiv_rn(__fadd_rn(tab.v[4 * a + 3], sy), H);
    return r;
}

__global__ void __launch_bounds__(256) anchors_kernel(float4* __restrict__ out, AnchorTable tab, int n, int fw,
                                                      float stride, float W, float H) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int cell = i / tab.A, a = i - cell * tab.A;
    out[i] = make_anchor(tab, cell, a, fw, stride, W, H);
}

// Multi-level anchors of the FPN variant (torchvision AnchorGenerator.grid_anchors as called at models/new_model.py:43-44,
// then `anchor /= (w, h, w, h)`): level l has fh_l x fw_l cells with strides (img_h // fh_l, img_w // fw_l) and its own
// A base boxes; anchors are cell-major, anchor-minor inside a level, levels concatenated.
constexpr int kPyrLevels = 8, kPyrA = 8;
struct PyramidParams {
    int L, A;
    int off[kPyrLevels + 1];  // first anchor of level l
    int fw[kPyrLevels];
    float sx[kPyrLevels], sy[kPyrLevels];
    float tab[kPyrLevels][kPyrA * 4];
};

__global__ void __launch_bounds__(256) anchors_pyramid_kernel(float4* __restrict__ out, PyramidParams p, int n, float W, float H) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int l = 0;
#pragma unroll
    for (int q = 1; q < kPyrLevels; ++q) l += (q < p.L && i >= p.off[q]) ? 1 : 0;
    const int j = i - p.off[l];
    const int cell = j / p.A, a = j - cell * p.A;
    const int y = cell / p.fw[l], x = cell - y * p.fw[l];
    const float shx = (float)x * p.sx[l], shy = (float)y * p.sy[l];  // exact: small integers
    float4 r;
    r.x = __fdiv_rn(__fadd_rn(p.tab[l][4 * a + 0], shx), W);
    r.y = __fdiv_rn(__fadd_rn(p.tab[l][4 * a + 1], shy), H);
    r.z = __fdiv_rn(__fadd_rn(p.tab[l][4 * a + 2], shx), W);
    r.w = __fdiv_rn(__fadd_rn(p.tab[l][4 * a + 3], shy), H);
    out[i] = r;
}

// One image's box, score and validity from its regression t and logits l (l.y alone: a score) and the anchor in centre
// form, for the mixed-size decode.  The same operations, in the same order, as the body of rpn_decode_kernel below (which
// keeps them inline: moving them into this function changes that kernel's register allocation).
template <bool kLogits>
__device__ __forceinline__ void decode_one(const float4& t, const float2& l, float acx, float acy, float aw, float ah,
                                           float min_size, float4* boxes, float* scores, uint8_t* valid, size_t g) {
    float s = l.y;
    if (kLogits) s = __frcp_rn(__fadd_rn(1.0f, expf(__fsub_rn(l.x, l.y))));
    // decode: c = t_xy * a_wh + a_c ; wh/2 = exp(t_wh) * a_wh / 2 ; cxcy_to_xy ; clamp(0,1)
    const float cx = __fadd_rn(__fmul_rn(t.x, aw), acx), cy = __fadd_rn(__fmul_rn(t.y, ah), acy);
    const float hw = __fmul_rn(__fmul_rn(expf(t.z), aw), 0.5f);
    const float hh = __fmul_rn(__fmul_rn(expf(t.w), ah), 0.5f);
    const float r0 = __fsub_rn(cx, hw), r1 = __fsub_rn(cy, hh), r2 = __fadd_rn(cx, hw), r3 = __fadd_rn(cy, hh);
    float4 bx;
    bx.x = __saturatef(r0);
    bx.y = __saturatef(r1);
    bx.z = __saturatef(r2);
    bx.w = __saturatef(r3);
    const bool finite = (r0 == r0) && (r1 == r1) && (r2 == r2) && (r3 == r3);
    const bool ok = finite && (__fsub_rn(bx.w, bx.y) >= min_size) && (__fsub_rn(bx.z, bx.x) >= min_size);
    st_stream(boxes + g, bx);
    scores[g] = s;
    valid[g] = ok ? 1 : 0;
}

// One thread per anchor and kImgs images (grid.y = image group): the anchor (4 IEEE divisions) and its
// centre form are built once and reused for every image of the group; the 2*kImgs loads of a thread are
// issued back to back (memory-level parallelism) before any arithmetic.
//   score = 1 / (1 + exp(l0 - l1))           (== softmax(l)[1]; one ex2 + one reciprocal)
//   box   = sat(c -/+ exp(t_wh) * a_wh / 2)  (add.sat == clamp(0,1) of the rounded sum)
// exp() is CUDA's accurate expf (<= 1 ulp; the kernel is HBM-bound, the extra instructions are free), well inside the
// 1e-5 contract for decoded boxes and scores; every index-valued stage downstream is evaluated on the fp32 values
// written here.  A NaN regression output stays out of the proposals exactly as in the reference: torch.clamp
// propagates NaN and `NaN - y1 >= min_size` is false (models/model.py:34,39), whereas add.sat maps NaN to 0 -- so the
// box is marked invalid when any pre-clamp coordinate is NaN.
template <bool kLogits, bool kGenAnchors, int kImgs>
__global__ void __launch_bounds__(256)
    rpn_decode_kernel(const float4* __restrict__ reg, const float* __restrict__ cls, const float4* __restrict__ anchors,
                      AnchorTable tab, int B, int N, int fw, float stride, float W, float H, float min_size,
                      float4* __restrict__ boxes, float* __restrict__ scores, uint8_t* __restrict__ valid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int b0 = blockIdx.y * kImgs;

    float4 t[kImgs];
    float2 l[kImgs];
#pragma unroll
    for (int j = 0; j < kImgs; ++j) {
        if (b0 + j < B) {
            const size_t g = (size_t)(b0 + j) * N + i;
            t[j] = ld_stream(reg + g);
            if (kLogits) l[j] = __ldg(reinterpret_cast<const float2*>(cls) + g);
            else l[j].y = __ldg(cls + g);
        }
    }

    float4 an;
    if (kGenAnchors) {
        const int cell = i / tab.A, a = i - cell * tab.A;
        an = make_anchor(tab, cell, a, fw, stride, W, H);
    } else {
        an = anchors[i];
    }
    // xy_to_cxcy(anchor): c = (hi + lo)/2, wh = hi - lo
    const float acx = __fmul_rn(__fadd_rn(an.z, an.x), 0.5f), acy = __fmul_rn(__fadd_rn(an.w, an.y), 0.5f);
    const float aw = __fsub_rn(an.z, an.x), ah = __fsub_rn(an.w, an.y);

#pragma unroll
    for (int j = 0; j < kImgs; ++j) {
        if (b0 + j < B) {
            const size_t g = (size_t)(b0 + j) * N + i;
            float s = l[j].y;
            if (kLogits) s = __frcp_rn(__fadd_rn(1.0f, expf(__fsub_rn(l[j].x, l[j].y))));
            // decode: c = t_xy * a_wh + a_c ; wh/2 = exp(t_wh) * a_wh / 2 ; cxcy_to_xy ; clamp(0,1)
            const float cx = __fadd_rn(__fmul_rn(t[j].x, aw), acx), cy = __fadd_rn(__fmul_rn(t[j].y, ah), acy);
            const float hw = __fmul_rn(__fmul_rn(expf(t[j].z), aw), 0.5f);
            const float hh = __fmul_rn(__fmul_rn(expf(t[j].w), ah), 0.5f);
            const float r0 = __fsub_rn(cx, hw), r1 = __fsub_rn(cy, hh), r2 = __fadd_rn(cx, hw), r3 = __fadd_rn(cy, hh);
            float4 bx;
            bx.x = __saturatef(r0);
            bx.y = __saturatef(r1);
            bx.z = __saturatef(r2);
            bx.w = __saturatef(r3);
            const bool finite = (r0 == r0) && (r1 == r1) && (r2 == r2) && (r3 == r3);
            const bool ok = finite && (__fsub_rn(bx.w, bx.y) >= min_size) && (__fsub_rn(bx.z, bx.x) >= min_size);
            st_stream(boxes + g, bx);
            scores[g] = s;
            valid[g] = ok ? 1 : 0;
        }
    }
}

// The same for a batch padded to grid_h x grid_w cells (N = grid_h * grid_w * A): only the cell shift is shared by the
// images of a group; every image divides the anchor by its own (W_b, H_b), exactly as frr_rpn_decode does for that image
// alone, and cells outside its own grid get box 0, score 0, valid 0 whatever the head outputs hold there.
template <bool kLogits, int kImgs>
__global__ void __launch_bounds__(256)
    rpn_decode_sized_kernel(const float4* __restrict__ reg, const float* __restrict__ cls, AnchorTable tab, int B, int N,
                            int grid_h, int grid_w, int stride, const int32_t* __restrict__ image_hw, float min_size,
                            float4* __restrict__ boxes, float* __restrict__ scores, uint8_t* __restrict__ valid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int b0 = blockIdx.y * kImgs;

    float4 t[kImgs];
    float2 l[kImgs];
#pragma unroll
    for (int j = 0; j < kImgs; ++j) {
        if (b0 + j < B) {
            const size_t g = (size_t)(b0 + j) * N + i;
            t[j] = ld_stream(reg + g);
            if (kLogits) l[j] = __ldg(reinterpret_cast<const float2*>(cls) + g);
            else l[j].y = __ldg(cls + g);
        }
    }

    const int cell = i / tab.A, a = i - cell * tab.A;
    const int y = cell / grid_w, x = cell - y * grid_w;
    const float sx = (float)x * (float)stride, sy = (float)y * (float)stride;  // exact: small integers
    const float bx1 = __fadd_rn(tab.v[4 * a + 0], sx), by1 = __fadd_rn(tab.v[4 * a + 1], sy);
    const float bx2 = __fadd_rn(tab.v[4 * a + 2], sx), by2 = __fadd_rn(tab.v[4 * a + 3], sy);

#pragma unroll
    for (int j = 0; j < kImgs; ++j) {
        if (b0 + j < B) {
            const size_t g = (size_t)(b0 + j) * N + i;
            const int2 ext = image_cells(image_hw, b0 + j, stride, grid_h, grid_w);
            if (y < ext.x && x < ext.y) {
                const int2 hw = __ldg(reinterpret_cast<const int2*>(image_hw) + b0 + j);
                const float W = (float)hw.y, H = (float)hw.x;
                const float4 an = make_float4(__fdiv_rn(bx1, W), __fdiv_rn(by1, H), __fdiv_rn(bx2, W), __fdiv_rn(by2, H));
                const float acx = __fmul_rn(__fadd_rn(an.z, an.x), 0.5f), acy = __fmul_rn(__fadd_rn(an.w, an.y), 0.5f);
                const float aw = __fsub_rn(an.z, an.x), ah = __fsub_rn(an.w, an.y);
                decode_one<kLogits>(t[j], l[j], acx, acy, aw, ah, min_size, boxes, scores, valid, g);
            } else {  // padding cell of this image
                st_stream(boxes + g, make_float4(0.f, 0.f, 0.f, 0.f));
                scores[g] = 0.f;
                valid[g] = 0;
            }
        }
    }
}

}  // namespace frr

extern "C" {

int frr_anchors(float* anchors, int img_h, int img_w, int stride, const float* base_table_host, int A,
                frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(anchors && img_h > 0 && img_w > 0 && stride > 0, "frr_anchors: bad arguments");
    FRR_CHECK_ARG(aligned16(anchors), "frr_anchors: output must be 16-byte aligned");
    AnchorTable tab;
    int rc = fill_anchor_table(&tab, base_table_host, A, stride);
    if (rc) return rc;
    const int fh = img_h / stride, fw = img_w / stride;
    const int n = fh * fw * tab.A;
    if (n == 0) return FRR_OK;
    anchors_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>((float4*)anchors, tab, n, fw, (float)stride,
                                                                       (float)img_w, (float)img_h);
    count_launch();
    FRR_CHECK_LAUNCH("anchors_kernel");
    return FRR_OK;
}

int frr_anchors_pyramid(float* anchors, int L, const int32_t* level_hw_host, const float* base_tables_host, int A, int img_h,
                        int img_w, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(anchors && level_hw_host && base_tables_host, "frr_anchors_pyramid: null pointer");
    FRR_CHECK_ARG(L >= 1 && L <= kPyrLevels && A >= 1 && A <= kPyrA && img_h > 0 && img_w > 0,
                  "frr_anchors_pyramid: L must be in [1,%d], A in [1,%d]", kPyrLevels, kPyrA);
    FRR_CHECK_ARG(aligned16(anchors), "frr_anchors_pyramid: output must be 16-byte aligned");
    PyramidParams p;
    p.L = L;
    p.A = A;
    long long n = 0;
    for (int l = 0; l < kPyrLevels; ++l) {
        p.off[l] = (int)n;
        p.fw[l] = 1; p.sx[l] = 0.f; p.sy[l] = 0.f;
        if (l < L) {
            const int fh = level_hw_host[2 * l], fw = level_hw_host[2 * l + 1];
            FRR_CHECK_ARG(fh > 0 && fw > 0, "frr_anchors_pyramid: level %d has an empty grid", l);
            p.fw[l] = fw;
            p.sy[l] = (float)(img_h / fh);  // integer strides, like torchvision (image_size // grid_size)
            p.sx[l] = (float)(img_w / fw);
            for (int q = 0; q < 4 * A; ++q) p.tab[l][q] = base_tables_host[(size_t)l * A * 4 + q];
            n += (long long)fh * fw * A;
        }
    }
    p.off[kPyrLevels] = (int)n;
    FRR_CHECK_ARG(n > 0 && n < (1ll << 30), "frr_anchors_pyramid: bad total size");
    anchors_pyramid_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((float4*)anchors, p, (int)n, (float)img_w,
                                                                                         (float)img_h);
    count_launch();
    FRR_CHECK_LAUNCH("anchors_pyramid_kernel");
    return FRR_OK;
}

int frr_rpn_decode(const float* reg, const float* cls, int cls_is_logits, const float* anchors,
                   const float* base_table_host, int A, int img_h, int img_w, int stride, float min_size, float* boxes,
                   float* scores, uint8_t* valid, int B, int N, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(reg && cls && boxes && scores && valid, "frr_rpn_decode: null pointer");
    FRR_CHECK_ARG(B >= 0 && N >= 0 && B <= 65535, "frr_rpn_decode: bad B=%d N=%d", B, N);
    FRR_CHECK_ARG(aligned16(reg) && aligned16(boxes) && (anchors == nullptr || aligned16(anchors)),
                  "frr_rpn_decode: reg/boxes/anchors must be 16-byte aligned");
    FRR_CHECK_ARG((reinterpret_cast<uintptr_t>(cls) & 7u) == 0, "frr_rpn_decode: cls must be 8-byte aligned");
    AnchorTable tab;
    tab.A = 1;
    int fw = 1;
    if (anchors == nullptr) {
        FRR_CHECK_ARG(img_h > 0 && img_w > 0 && stride > 0, "frr_rpn_decode: bad image size");
        int rc = fill_anchor_table(&tab, base_table_host, A, stride);
        if (rc) return rc;
        fw = img_w / stride;
        FRR_CHECK_ARG((img_h / stride) * fw * tab.A == N, "frr_rpn_decode: N=%d does not match %dx%d/%d x A=%d", N,
                      img_h, img_w, stride, tab.A);
    }
    if (B == 0 || N == 0) return FRR_OK;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(L, G, I)                                                                                               \
    rpn_decode_kernel<L, G, I><<<dim3((N + 255) / 256, (B + I - 1) / I), 256, 0, st>>>(                              \
        (const float4*)reg, cls, (const float4*)anchors, tab, B, N, fw, (float)stride, (float)img_w, (float)img_h,   \
        min_size, (float4*)boxes, scores, valid)
#define LAUNCH_I(L, G)                        \
    do {                                      \
        if (B >= 4) LAUNCH(L, G, 4);          \
        else LAUNCH(L, G, 1);                 \
    } while (0)
    if (cls_is_logits) {
        if (anchors) LAUNCH_I(true, false); else LAUNCH_I(true, true);
    } else {
        if (anchors) LAUNCH_I(false, false); else LAUNCH_I(false, true);
    }
#undef LAUNCH_I
#undef LAUNCH
    count_launch();
    FRR_CHECK_LAUNCH("rpn_decode_kernel");
    return FRR_OK;
}

int frr_rpn_decode_sized(const float* reg, const float* cls, int cls_is_logits, const float* base_table_host, int A,
                         const int32_t* image_hw, int grid_h, int grid_w, int stride, float min_size, float* boxes,
                         float* scores, uint8_t* valid, int B, int N, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(reg && cls && boxes && scores && valid && image_hw, "frr_rpn_decode_sized: null pointer");
    FRR_CHECK_ARG(B >= 0 && N >= 0 && B <= 65535, "frr_rpn_decode_sized: bad B=%d N=%d", B, N);
    FRR_CHECK_ARG(aligned16(reg) && aligned16(boxes), "frr_rpn_decode_sized: reg/boxes must be 16-byte aligned");
    FRR_CHECK_ARG((reinterpret_cast<uintptr_t>(cls) & 7u) == 0 && aligned8(image_hw),
                  "frr_rpn_decode_sized: cls and image_hw must be 8-byte aligned");
    FRR_CHECK_ARG(grid_h >= 0 && grid_w >= 0 && stride > 0, "frr_rpn_decode_sized: bad grid %dx%d / stride %d", grid_h,
                  grid_w, stride);
    AnchorTable tab;
    int rc = fill_anchor_table(&tab, base_table_host, A, stride);
    if (rc) return rc;
    FRR_CHECK_ARG((long long)grid_h * grid_w * tab.A == N, "frr_rpn_decode_sized: N=%d does not match a %dx%d grid x A=%d",
                  N, grid_h, grid_w, tab.A);
    if (B == 0 || N == 0) return FRR_OK;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(L, I)                                                                                                   \
    rpn_decode_sized_kernel<L, I><<<dim3((N + 255) / 256, (B + I - 1) / I), 256, 0, st>>>(                           \
        (const float4*)reg, cls, tab, B, N, grid_h, grid_w, stride, image_hw, min_size, (float4*)boxes, scores, valid)
    if (cls_is_logits) {
        if (B >= 4) LAUNCH(true, 4); else LAUNCH(true, 1);
    } else {
        if (B >= 4) LAUNCH(false, 4); else LAUNCH(false, 1);
    }
#undef LAUNCH
    count_launch();
    FRR_CHECK_LAUNCH("rpn_decode_sized_kernel");
    return FRR_OK;
}

}  // extern "C"
