// Shared by the NMS kernels (nms.cu: keep-list kernel; nms_bucket.cu: bucketed large-chunk kernel): the decision
// arithmetic of torchvision's CPU kernel, the division-free screen, and the (x bin, y bin, area class) bucket keys.
#pragma once
#include <math.h>

#include "frr_common.cuh"

namespace frr {

constexpr int kMaxCluster = 16;
constexpr int kBkChunk = 2048;  // most candidates per chunk of the bucketed kernel (1024 below 1024 threads: bk_chunk_cap)

// Per-call settings of the bucketed kernel (frr_nms_sorted); 0 = automatic.  Results never depend on them.
struct NmsTune {
    int first_chunk, max_chunk;      // candidates in the first / the largest chunk: multiples of 256 in [256, kBkChunk],
                                     // clamped to the chunk capacity of the launch's thread count
    int lanes_screen, lanes_pairs;   // lanes per candidate of the screen / pair phases: powers of two <= 32
};

struct NmsThr {
    float up;  // smallest fp32 with (double)up > thr
    float c2;  // up/(1+up) * (1 - 2^-19): screening constant
    float alo, ahi;  // a box of area A can only be suppressed by boxes with area in [alo * A, ahi * A] (IoU <= min/max area)
    float fx;        // ... and only by boxes whose x-centre is within fx * (its width) of its own, y-centre likewise
    int fast;  // screening usable (1e-6 <= thr, finite)
};

__device__ __forceinline__ float box_area(const float4& b) {
    return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}
// c2-scaled area used by the screen: NaN for boxes that are not well formed or tiny (forces the exact path)
__device__ __forceinline__ float screen_area(const float4& b, float c2) {
    const float a = box_area(b);
    const bool ok = (b.z >= b.x) && (b.w >= b.y) && (a <= 3.0e38f) && (a >= 1.0e-30f);
    return ok ? __fmul_rn(c2, a) : __int_as_float(0x7fc00000);
}

// The exact torchvision CPU decision for one pair (a = earlier box).  Rare path.
static __device__ __noinline__ bool suppress_exact(float4 a, float4 b, float up) {
    const float w = fmaxf(0.f, __fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)));
    const float h = fmaxf(0.f, __fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)));
    const float inter = __fmul_rn(w, h);
    const float uni = __fsub_rn(__fadd_rn(box_area(a), box_area(b)), inter);
    const float ovr = __fdiv_rn(inter, uni);
    return ovr >= up;  // false for NaN, as (double)NaN > thr
}

// Screen: returns false only when the pair is certainly NOT suppressed.
//   exact:  ovr = RN(I / U),  U = RN(RN(Aa+Ab) - I) = (Aa+Ab-I)(1+e), |e| <= 2^-22 (I <= (Aa+Ab)/2)
//   ovr < up  <=  I/U < up(1-2^-23)  <=  I < u'(Aa+Ab-I), u' = up(1-2^-21)  <=>  I < u'/(1+u') (Aa+Ab)
//   screen:  T = RN(RN(c2 Aa) + RN(c2 Ab)) <= c2 (Aa+Ab)(1+2^-22), and c2 (1+2^-22) < u'/(1+u').
// Only one of w/h is clamped: if w < 0 then I <= 0 < T (the true intersection is 0: not suppressed).
// sa/sb are the c2-scaled areas (NaN if degenerate -> T is NaN -> the screen reports "maybe").
// kUnit: all coordinates lie in [0,1] (RPN / detection boxes are clamped there), so |h| <= 1 and the clamp of h at 0
// is the free .sat modifier of the subtraction (FMA pipe) instead of an FMNMX on the half-rate ALU pipe.
template <bool kUnit>
__device__ __forceinline__ bool suppress_screen(const float4& a, float sa, const float4& b, float sb) {
    const float w = __fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x));
    const float hd = __fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y));
    const float h = kUnit ? __saturatef(hd) : fmaxf(0.f, hd);
    return !(__fmul_rn(w, h) < __fadd_rn(sa, sb));
}

// Bucket key of a box = (x bin, y bin, area class) of the bucketed kernel, area class minor: the admissible area classes
// of one cell are ONE contiguous run of a bucketed array, so a walk is one range per admissible cell.
// Area class: the top bits of the fp32 area (exponent + 2 mantissa bits = 4 classes per octave), an exactly monotone
// integer function of the area, clamped to [2^-15, 1) (clamping keeps it monotone, so the admissible classes of a box
// still contain every class that can suppress it).  IoU <= min(area) / max(area) (in fp32 as well: w <= both widths and
// RN is monotone, so inter <= both areas), hence only kept boxes whose area lies within [thr, 1/thr] of the
// candidate's can suppress it: for RPN proposals (three anchor scales, a factor 4 apart in area) that alone removes 3/4
// of the pairs.
// Cell: kX x kY equal bins of the x- and y-centre; IoU >= thr also needs |cx_a - cx_b| <= fx * w and, the same rule
// with the axes swapped, |cy_a - cy_b| <= fx * h of either box, which is sharp exactly where the area cut is not -- the
// many small boxes of the most populated classes.  kY = 1 is the x-only key (nms_bucket.cu: bk_ybins).
// Boxes without a usable screening area (degenerate / malformed, NaN sa) get the extra key kKeys and are tested
// against everything.
template <int kYBins>
struct BkGrid {
    static constexpr int kX = 8, kY = kYBins;
    static constexpr int kClasses = 60;                   // 4 per octave, 2^-15 .. 1
    static constexpr int kKeys = kX * kY * kClasses;      // key kKeys: boxes that must always be tested
    static __device__ __forceinline__ int cls(float a) {
        return min(kClasses - 1, max(0, (__float_as_int(a) >> 21) - ((127 - 15) << 2)));
    }
    static __device__ __forceinline__ int xbin(float cx) { return min(kX - 1, max(0, (int)(cx * (float)kX))); }
    static __device__ __forceinline__ int ybin(float cy) { return min(kY - 1, max(0, (int)(cy * (float)kY))); }
    static __device__ __forceinline__ int key(const float4& b, float sa) {
        return (sa != sa) ? kKeys
                          : (xbin(0.5f * (b.x + b.z)) * kY + ybin(0.5f * (b.y + b.w))) * kClasses + cls(box_area(b));
    }
};

inline NmsThr make_thr(double thr) {
    NmsThr t;
    float f = (float)thr;
    if (isnan(thr)) {
        t.up = NAN;  // nothing is ever > NaN
    } else {
        if (!((double)f > thr)) f = nextafterf(f, INFINITY);
        t.up = f;
    }
    t.fast = (thr >= 1.0e-6) && isfinite(thr) && (t.up < 1.0e30f) ? 1 : 0;
    const double u = (double)t.up;
    t.c2 = t.fast ? (float)(u / (1.0 + u) * (1.0 - 1.9073486328125e-06)) : 0.f;
    // IoU >= thr needs min(area) / max(area) >= thr; thr is lowered by 2^-17 relative to cover the fp32 roundings of the
    // exact IoU (<= 2^-20) and of the two products below
    const double tl = thr * (1.0 - 7.62939453125e-06);
    // ... and |cx_a - cx_b| <= max(1 - thr, (1 - thr) / (2 thr)) * w of EITHER box, |cy_a - cy_b| the same with h
    // (DESIGN.md)
    t.fx = t.fast ? (float)(fmax(1.0 - tl, (1.0 - tl) / (2.0 * tl)) * (1.0 + 1.0e-6)) : 0.f;
    t.alo = t.fast ? (float)(tl * (1.0 - 1.0e-6)) : 0.f;
    t.ahi = t.fast ? (float)(1.0 / tl * (1.0 + 1.0e-6)) : 0.f;
    return t;
}


int nms_launch(const float* boxes, const int32_t* counts, int B, int n, double iou_thr, int max_keep, int32_t* keep,
               int32_t* keep_count, float* out_boxes, int cluster_size, int threads, const NmsTune& tune, int unit_boxes,
               frr_stream_t stream, const int32_t* gather_idx = nullptr, int src_n = 0);

// nms_bucket.cu: eligibility + launch of the bucketed kernel (unit-range boxes, screenable threshold, kept list <= 2047)
bool nms_bucket_eligible(int n, int max_keep, const NmsThr& thr, int unit_boxes);
size_t nms_bucket_smem_bytes(int threads, int S);  // dynamic shared memory of a launch: threads per CTA, CTAs per image
int nms_bucket_launch(const float* boxes, const int32_t* counts, int B, int n, const NmsThr& thr, int max_keep, int32_t* keep,
                      int32_t* keep_count, float* out_boxes, int S, int threads, const NmsTune& tune, frr_stream_t stream,
                      const int32_t* gather_idx, int src_n);

}  // namespace frr
