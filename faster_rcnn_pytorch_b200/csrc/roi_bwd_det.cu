// Deterministic RoIPool / RoIAlign backward, bit-exact with torchvision's CPU kernels
// (frr_roi_pool_bwd_deterministic / frr_roi_align_bwd_deterministic; contract in include/frr.h).
//
// torchvision's CPU loop adds every contribution into grad_in in one fixed order: roi k ascending, then channel, ph, pw
// and, for RoIAlign, iy, ix and bilinear taps 1-4.  The other backward kernels scatter, and a scatter cannot keep that
// order without sorting.  These kernels gather instead (owner computes):
//
//   * a CTA owns a spatial tile of one image (256 pixels, one per thread) for CG <= 16 channels and keeps the CG sums of
//     its pixel in registers: no two threads ever add into the same element, and no value is touched by an atomic;
//   * the CTA scans the rois once (kDetIdCap per round, in k order) and keeps the rois of its image whose footprint meets
//     the tile -- the union of the clipped windows for RoIPool, a bounding box of the bilinear taps for RoIAlign;
//   * per listed roi, in k order, the CTA builds the roi's geometry once into shared memory (RoIPool: the bin windows
//     of pool_window; RoIAlign: one (low, high, l, h) record per y-sample (ph, iy) and per x-sample (pw, ix), taken from
//     bilinear_taps) and streams the roi's grad_out (and argmax) rows of its channels through a cp.async ring that runs
//     kDetDepth - 1 rois ahead; one barrier per roi;
//   * each thread then walks, in canonical order, the bins / samples whose window / taps reach its pixel and adds their
//     terms with the fp32 arithmetic of the CPU loop (*_rn intrinsics, no contraction).  Every element is therefore the
//     same sequence of roundings as torchvision's CPU sum, whatever the grid, stream or concurrent work.
//
// HBM traffic: grad_in written once (no memset pass); grad_out (+ argmax) rows are read by every tile a roi meets, which
// the L2 absorbs (the tiles of one (image, channel group) are neighbouring CTAs).
#include "roi_common.cuh"

namespace frr {

constexpr int kDetThreads = 256;  // pixels per tile
constexpr int kDetCG = 16;        // channel sums per thread (registers)
constexpr int kDetDepth = 4;      // ring slots: rois in flight
constexpr int kDetIdCap = 1024;   // rois scanned per round
constexpr int kDetPer = kDetIdCap / kDetThreads;

struct DetHdr {
    unsigned int scan[32];
    int id[kDetIdCap];
};
constexpr int kDetHdrBytes = (sizeof(DetHdr) + 127) & ~127;

// RoIAlign sample record of one y-sample (low/high rows, ly, hy) or x-sample (low/high columns, lx, hx); lo = hi = -1
// for a sample bilinear_taps rejects (it then matches no pixel)
struct SampleRec {
    int lo, hi;
    float l, h;
};

struct DetRoi {  // per-slot header
    AlignGeom g;
    int r0, r1, q0, q1;  // footprint rows r0..r1, columns q0..q1 (inclusive; empty when r1 < r0 or q1 < q0)
    int big;             // RoIAlign grid larger than the record capacity: records are computed where they are used
};
static_assert(sizeof(DetRoi) <= 64, "slot header");

// Byte offsets inside one ring slot (host and device agree through this one function)
struct DetLayout {
    int go, arg, geo, ycap, xcap, bytes;
};
__host__ __device__ inline DetLayout det_layout(bool align, int CG, int PH, int PW) {
    DetLayout L;
    const int rows = ((CG * PH * PW * 4) + 15) & ~15;
    L.go = 64;
    L.arg = L.go + rows;
    L.geo = align ? L.arg : L.arg + rows;
    L.ycap = align ? 16 * PH : 0;  // sampling grids up to 16 x 16 per bin keep their records in shared memory
    L.xcap = align ? 16 * PW : 0;
    const int geo = align ? (L.ycap + L.xcap) * (int)sizeof(SampleRec) : 2 * (PH + PW) * 4;
    L.bytes = (L.geo + geo + 127) & ~127;
    return L;
}

// Rows lo..hi of [0, n) that the taps of samples spread between s and s + P * bin can reach (conservative: rounding
// of the sample positions is covered by the margin; non-finite geometry covers the whole map).
__device__ __forceinline__ void align_span(float s, float bin, int P, int n, int& lo, int& hi) {
    const float e = __fadd_rn(s, __fmul_rn((float)P, bin));
    if (isnan(s) || isnan(e)) { lo = 0; hi = n - 1; return; }
    const float m = __fadd_rn(2.f, __fmul_rn(1e-6f, __fadd_rn(fabsf(s), fabsf(e))));
    const float a = fminf(fmaxf(__fsub_rn(fminf(s, e), m), -4.f), (float)n + 4.f);
    const float z = fminf(fmaxf(__fadd_rn(fmaxf(s, e), m), -4.f), (float)n + 4.f);
    lo = max((int)floorf(a), 0);
    hi = min((int)floorf(z) + 1, n - 1);
}

template <bool kAlign>
__device__ __forceinline__ void det_footprint(const float* r, float scale, int H, int W, int PH, int PW, int sampling,
                                              bool aligned, int& r0, int& r1, int& q0, int& q1) {
    if (!kAlign) {
        const PoolGeom g = pool_geom(r, scale);
        int hs, he, ws, we;
        pool_window(g, 0, 0, PH, PW, H, W, r0, he, q0, we);
        pool_window(g, PH - 1, PW - 1, PH, PW, H, W, hs, he, ws, we);
        r1 = he - 1;
        q1 = we - 1;
    } else {
        const AlignGeom g = align_geom(r, scale, PH, PW, sampling, aligned);
        align_span(g.sh, g.bin_h, PH, H, r0, r1);
        align_span(g.sw, g.bin_w, PW, W, q0, q1);
    }
}

__device__ __forceinline__ SampleRec y_record(const AlignGeom& g, int j, int H, int W) {
    const int ph = j / g.gh, iy = j - ph * g.gh;
    Taps t;
    if (!bilinear_taps(sample_y(g, ph, iy), 0.f, H, W, t)) return SampleRec{-1, -1, 0.f, 0.f};
    return SampleRec{t.p1 / W, t.p3 / W, t.w3, t.w1};  // x = 0: hx = 1, lx = 0, so w1 = hy and w3 = ly exactly
}
__device__ __forceinline__ SampleRec x_record(const AlignGeom& g, int j, int H, int W) {
    const int pw = j / g.gw, ix = j - pw * g.gw;
    Taps t;
    if (!bilinear_taps(0.f, sample_x(g, pw, ix), H, W, t)) return SampleRec{-1, -1, 0.f, 0.f};
    return SampleRec{t.p1, t.p2, t.w2, t.w1};  // y = 0: hy = 1, ly = 0, so w1 = hx and w2 = lx exactly
}

// t / c rounded to fp32 exactly as __fdiv_rn does, without its out-of-line slow path (a call inside the accumulate loop
// makes ptxas spill the channel sums).  The quotient is formed in fp64 with one Markstein correction (error < 2^-52
// relative); for an integer c < 2^27 that is not a power of two, t / c lies at least 2^-24 / c (relative) away from
// every fp32 rounding boundary, so rounding the fp64 value to fp32 gives the correctly rounded quotient, subnormal
// results included.  inv = det_rcp(c).
__device__ __forceinline__ double det_rcp(double c) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(c));
    r = __fma_rn(r, __fma_rn(-c, r, 1.0), r);
    return __fma_rn(r, __fma_rn(-c, r, 1.0), r);
}
__device__ __forceinline__ float det_div(float t, double c, double inv) {
    if (!isfinite(t)) return t;  // +-inf / c = +-inf, NaN stays NaN (c >= 1)
    const double q = __dmul_rn((double)t, inv);
    return __double2float_rn(__fma_rn(__fma_rn(-q, c, (double)t), inv, q));
}

// kCG: channels per CTA = channel sums per thread, 16 unless a ring of 16-channel slots does not fit shared memory
// kSized (RoIPool only): the bin windows are clipped to image b's own extent (image_cells), as in the sized forward
template <bool kAlign, int kCG, bool kSized>
__device__ __forceinline__ void roi_bwd_det_body(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                                                 const float* __restrict__ rois, int K, int C, int H, int W, int PH, int PW,
                                                 float scale, int sampling, int aligned, int nhwc, int TW, int tiles_w,
                                                 float* __restrict__ grad_in, const int32_t* __restrict__ image_hw,
                                                 int stride) {
    constexpr int CG = kCG;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    DetHdr* hd = reinterpret_cast<DetHdr*>(smem_raw);
    unsigned char* ring = smem_raw + kDetHdrBytes;
    const DetLayout L = det_layout(kAlign, CG, PH, PW);
    const int tid = threadIdx.x;
    const int TH = kDetThreads / TW;
    const int ty = blockIdx.x / tiles_w, tx = blockIdx.x - ty * tiles_w;
    const int ty0 = ty * TH, tx0 = tx * TW;
    const int ty1 = min(ty0 + TH, H) - 1, tx1 = min(tx0 + TW, W) - 1;
    const int c0 = blockIdx.y * CG, b = blockIdx.z;
    const int cg = min(CG, C - c0);
    const int h = ty0 + tid / TW, w = tx0 + tid % TW;
    const bool mine = h < H && w < W;
    const int bins = PH * PW, rows = cg * bins;
    const bool al = aligned != 0;
    const int2 ext = kSized ? image_cells(image_hw, b, stride, H, W) : make_int2(H, W);  // RoIPool window clip

    float acc[CG];
#pragma unroll
    for (int c = 0; c < CG; ++c) acc[c] = 0.f;

    for (int k0 = 0; k0 < K; k0 += kDetIdCap) {
        // the rois of image b in rois[k0, k0 + kDetIdCap) whose footprint meets the tile, in k order
        const int lo = k0 + tid * kDetPer;
        unsigned int keep = 0;
#pragma unroll
        for (int j = 0; j < kDetPer; ++j) {
            const int k = lo + j;
            if (k >= K) break;
            const float* r = rois + 5 * (size_t)k;
            if ((int)__ldg(r) != b) continue;
            int r0, r1, q0, q1;
            det_footprint<kAlign>(r, scale, ext.x, ext.y, PH, PW, sampling, al, r0, r1, q0, q1);
            if (r0 <= r1 && q0 <= q1 && r0 <= ty1 && r1 >= ty0 && q0 <= tx1 && q1 >= tx0) keep |= 1u << j;
        }
        unsigned int n;
        unsigned int pos = block_exclusive_scan(__popc(keep), hd->scan, &n);
        while (keep) {
            const int j = __ffs(keep) - 1;
            keep &= keep - 1u;
            hd->id[pos++] = lo + j;
        }
        __syncthreads();

        // roi r of the list -> ring slot r % kDetDepth: copies of its rows + its geometry (always commits a group)
        auto issue = [&](int r) {
            if (r < (int)n) {
                unsigned char* slot = ring + (size_t)(r % kDetDepth) * L.bytes;
                const int k = hd->id[r];
                const size_t src = ((size_t)k * C + c0) * bins;
                const uint32_t s_go = smem_u32(slot + L.go), s_arg = smem_u32(slot + L.arg);
                for (int i = tid; i < CG * bins; i += kDetThreads) {
                    const bool live = i < rows;
                    const size_t o = src + (live ? i : 0);
                    cp_async4_zfill(s_go + 4u * i, grad_out + o, live ? 4u : 0u);
                    if (!kAlign) cp_async4_zfill(s_arg + 4u * i, argmax + o, live ? 4u : 0u);
                }
                const float* rr = rois + 5 * (size_t)k;
                DetRoi* dr = reinterpret_cast<DetRoi*>(slot);
                if (!kAlign) {
                    const PoolGeom g = pool_geom(rr, scale);
                    int* win = reinterpret_cast<int*>(slot + L.geo);  // hs[PH], he[PH], ws[PW], we[PW]
                    for (int i = tid; i < PH + PW; i += kDetThreads) {
                        int hs, he, ws, we;
                        if (i < PH) {
                            pool_window(g, i, 0, PH, PW, ext.x, ext.y, hs, he, ws, we);
                            win[i] = hs;
                            win[PH + i] = he;
                        } else {
                            pool_window(g, 0, i - PH, PH, PW, ext.x, ext.y, hs, he, ws, we);
                            win[2 * PH + i - PH] = ws;
                            win[2 * PH + PW + i - PH] = we;
                        }
                    }
                } else {
                    const AlignGeom g = align_geom(rr, scale, PH, PW, sampling, al);
                    const int ny = max(PH * g.gh, 0), nx = max(PW * g.gw, 0);
                    if (ny <= L.ycap && nx <= L.xcap) {
                        SampleRec* yr = reinterpret_cast<SampleRec*>(slot + L.geo);
                        SampleRec* xr = yr + L.ycap;
                        for (int i = tid; i < ny + nx; i += kDetThreads) {
                            if (i < ny) yr[i] = y_record(g, i, H, W);
                            else xr[i - ny] = x_record(g, i - ny, H, W);
                        }
                    }
                    if (tid == 0) {
                        dr->g = g;
                        dr->big = ny > L.ycap || nx > L.xcap;
                    }
                }
                if (tid == 0) det_footprint<kAlign>(rr, scale, ext.x, ext.y, PH, PW, sampling, al, dr->r0, dr->r1, dr->q0, dr->q1);
            }
            cp_async_commit();
        };

        for (int r = 0; r < kDetDepth - 1; ++r) issue(r);
        for (int r = 0; r < (int)n; ++r) {
            cp_async_wait<kDetDepth - 2>();  // this thread's copies of roi r have landed ...
            __syncthreads();                 // ... everyone's, with the geometry; slot (r - 1) % D is free again
            issue(r + kDetDepth - 1);
            const unsigned char* slot = ring + (size_t)(r % kDetDepth) * L.bytes;
            const DetRoi* dr = reinterpret_cast<const DetRoi*>(slot);
            if (!mine || h < dr->r0 || h > dr->r1 || w < dr->q0 || w > dr->q1) continue;
            const float* go = reinterpret_cast<const float*>(slot + L.go);
            if (!kAlign) {
                const int32_t* am = reinterpret_cast<const int32_t*>(slot + L.arg);
                const int* hs = reinterpret_cast<const int*>(slot + L.geo);
                const int *he = hs + PH, *ws = he + PH, *we = ws + PW;
                const int p = h * W + w;
                int pa = PH, pb = -1, qa = PW, qb = -1;
                for (int ph = 0; ph < PH; ++ph)
                    if (hs[ph] <= h && h < he[ph]) { pa = min(pa, ph); pb = ph; }
                for (int pw = 0; pw < PW; ++pw)
                    if (ws[pw] <= w && w < we[pw]) { qa = min(qa, pw); qb = pw; }
                for (int ph = pa; ph <= pb; ++ph) {
                    if (!(hs[ph] <= h && h < he[ph])) continue;
                    for (int pw = qa; pw <= qb; ++pw) {
                        if (!(ws[pw] <= w && w < we[pw])) continue;
                        const int bin = ph * PW + pw;
#pragma unroll
                        for (int c = 0; c < CG; ++c)
                            if (am[c * bins + bin] == p) acc[c] = __fadd_rn(acc[c], go[c * bins + bin]);
                    }
                }
            } else {
                const AlignGeom g = dr->g;
                const bool big = dr->big != 0;
                const SampleRec* yr = reinterpret_cast<const SampleRec*>(slot + L.geo);
                const SampleRec* xr = yr + L.ycap;
                auto yrec = [&](int j) { return big ? y_record(g, j, H, W) : yr[j]; };
                auto xrec = [&](int j) { return big ? x_record(g, j, H, W) : xr[j]; };
                const int ny = max(PH * g.gh, 0), nx = max(PW * g.gw, 0);
                int ja = ny, jb = -1, xa = nx, xb = -1;
                for (int j = 0; j < ny; ++j) {
                    const SampleRec s = yrec(j);
                    if (s.lo == h || s.hi == h) { ja = min(ja, j); jb = j; }
                }
                if (jb < 0) continue;
                for (int j = 0; j < nx; ++j) {
                    const SampleRec s = xrec(j);
                    if (s.lo == w || s.hi == w) { xa = min(xa, j); xb = j; }
                }
                if (xb < 0) continue;
                // / count == * (1 / count) bit for bit when count is a power of two (both round the same exact value)
                const int cnt = (int)g.count;
                const bool pow2 = (cnt & (cnt - 1)) == 0;
                const float inv = __int_as_float((127 - (__ffs(cnt) - 1)) << 23);
                const double cd = (double)g.count, invd = det_rcp(cd);
                for (int ph = ja / g.gh; ph <= jb / g.gh; ++ph) {
                    for (int pw = xa / g.gw; pw <= xb / g.gw; ++pw) {
                        const float* gb = go + ph * PW + pw;
                        auto add = [&](float wt) {
#pragma unroll
                            for (int c = 0; c < CG; ++c) {
                                const float t = __fmul_rn(gb[c * bins], wt);
                                acc[c] = __fadd_rn(acc[c], pow2 ? __fmul_rn(t, inv) : det_div(t, cd, invd));
                            }
                        };
                        for (int iy = 0; iy < g.gh; ++iy) {
                            const int jy = ph * g.gh + iy;
                            if (jy < ja || jy > jb) continue;
                            const SampleRec sy = yrec(jy);
                            const bool yl = sy.lo == h, yh = sy.hi == h;
                            if (!(yl || yh)) continue;
                            for (int ix = 0; ix < g.gw; ++ix) {
                                const int jx = pw * g.gw + ix;
                                if (jx < xa || jx > xb) continue;
                                const SampleRec sx = xrec(jx);
                                const bool xl = sx.lo == w, xh = sx.hi == w;
                                if (!(xl || xh)) continue;
                                // taps 1-4 of bilinear_taps: (yl,xl), (yl,xh), (yh,xl), (yh,xh), weights as it rounds them
                                if (yl && xl) add(__fmul_rn(sy.h, sx.h));
                                if (yl && xh) add(__fmul_rn(sy.h, sx.l));
                                if (yh && xl) add(__fmul_rn(sy.l, sx.h));
                                if (yh && xh) add(__fmul_rn(sy.l, sx.l));
                            }
                        }
                    }
                }
            }
        }
        cp_async_wait<0>();
        __syncthreads();  // the id list and the ring are rewritten by the next round
    }
    if (!mine) return;
    const int p = h * W + w;
    if (nhwc) {
        float* dst = grad_in + ((size_t)b * H * W + p) * C + c0;
#pragma unroll
        for (int c = 0; c < CG; ++c)
            if (c < cg) dst[c] = acc[c];
    } else {
        float* dst = grad_in + ((size_t)b * C + c0) * H * W + p;
#pragma unroll
        for (int c = 0; c < CG; ++c)
            if (c < cg) dst[(size_t)c * H * W] = acc[c];
    }
}
template <bool kAlign, int kCG>
__global__ void __launch_bounds__(kDetThreads)
    roi_bwd_det_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                       const float* __restrict__ rois, int K, int C, int H, int W, int PH, int PW, float scale,
                       int sampling, int aligned, int nhwc, int TW, int tiles_w, float* __restrict__ grad_in) {
    roi_bwd_det_body<kAlign, kCG, false>(grad_out, argmax, rois, K, C, H, W, PH, PW, scale, sampling, aligned, nhwc, TW,
                                         tiles_w, grad_in, nullptr, 0);
}
template <int kCG>
__global__ void __launch_bounds__(kDetThreads)
    roi_pool_bwd_det_sized_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                                  const float* __restrict__ rois, int K, int C, int H, int W, int PH, int PW, float scale,
                                  int nhwc, int TW, int tiles_w, float* __restrict__ grad_in,
                                  const int32_t* __restrict__ image_hw, int stride) {
    roi_bwd_det_body<false, kCG, true>(grad_out, argmax, rois, K, C, H, W, PH, PW, scale, 0, 0, nhwc, TW, tiles_w, grad_in,
                                       image_hw, stride);
}

static const size_t kDetSmemLimit = 227 * 1024;

template <bool kAlign>
static int roi_backward_det(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C, int H,
                            int W, int PH, int PW, float scale, int sampling, int aligned, int nhwc, float* grad_in,
                            frr_stream_t stream, const int32_t* image_hw = nullptr, int stride = 0) {
    FRR_CHECK_ARG(K >= 0 && B > 0 && C > 0 && H > 0 && W > 0 && PH > 0 && PW > 0 && B <= 65535,
                  "roi deterministic backward: bad sizes");
    FRR_CHECK_ARG(grad_in && (K == 0 || (grad_out && rois && (kAlign || argmax))),
                  "roi deterministic backward: null pointer");
    FRR_CHECK_ARG(!(reinterpret_cast<uintptr_t>(grad_out) & 3u) && !(reinterpret_cast<uintptr_t>(argmax) & 3u),
                  "roi deterministic backward: grad_out / argmax must be 4-byte aligned");
    FRR_CHECK_ARG((size_t)H * W <= (size_t)INT32_MAX && (size_t)K * 5 <= (size_t)INT32_MAX,
                  "roi deterministic backward: map or roi list too large");
    // channels per CTA: fewer when one ring of kDetDepth rois of 16 channels does not fit shared memory (large PH x PW)
    // (no 4-channel instantiation: ptxas spills in the RoIAlign one; 2 channels take those shapes)
    int CG = kDetCG;
    while (CG > 1 && kDetHdrBytes + (size_t)kDetDepth * det_layout(kAlign, CG, PH, PW).bytes > kDetSmemLimit)
        CG = CG == 8 ? 2 : CG >> 1;
    const size_t smem = kDetHdrBytes + (size_t)kDetDepth * det_layout(kAlign, CG, PH, PW).bytes;
    FRR_CHECK_ARG(smem <= kDetSmemLimit, "roi deterministic backward: %d x %d bins do not fit shared memory", PH, PW);
    FRR_CHECK_ARG((C + CG - 1) / CG <= 65535, "roi deterministic backward: too many channels");
    const int TW = W >= 32 ? 32 : W >= 16 ? 16 : 8;
    const int TH = kDetThreads / TW;
    const int tiles_w = (W + TW - 1) / TW;
    const long tiles = (long)tiles_w * ((H + TH - 1) / TH);
    FRR_CHECK_ARG(tiles <= INT32_MAX, "roi deterministic backward: map too large");
    const dim3 grid((unsigned)tiles, (unsigned)((C + CG - 1) / CG), (unsigned)B);
    if (!kAlign && image_hw) {
        auto kern = CG == 16 ? roi_pool_bwd_det_sized_kernel<16>
                  : CG == 8  ? roi_pool_bwd_det_sized_kernel<8>
                  : CG == 2  ? roi_pool_bwd_det_sized_kernel<2>
                             : roi_pool_bwd_det_sized_kernel<1>;
        FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDetSmemLimit));
        kern<<<grid, kDetThreads, smem, (cudaStream_t)stream>>>(grad_out, argmax, rois, K, C, H, W, PH, PW, scale, nhwc, TW,
                                                                tiles_w, grad_in, image_hw, stride);
    } else {
        auto kern = CG == 16 ? roi_bwd_det_kernel<kAlign, 16>
                  : CG == 8  ? roi_bwd_det_kernel<kAlign, 8>
                  : CG == 2  ? roi_bwd_det_kernel<kAlign, 2>
                             : roi_bwd_det_kernel<kAlign, 1>;
        FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDetSmemLimit));
        kern<<<grid, kDetThreads, smem, (cudaStream_t)stream>>>(grad_out, argmax, rois, K, C, H, W, PH, PW, scale, sampling,
                                                                aligned, nhwc, TW, tiles_w, grad_in);
    }
    count_launch();
    FRR_CHECK_LAUNCH(kAlign ? "roi_bwd_det_kernel<align>" : "roi_bwd_det_kernel<pool>");
    return FRR_OK;
}

}  // namespace frr

extern "C" {

int frr_roi_pool_bwd_deterministic(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C,
                                   int H, int W, int PH, int PW, float spatial_scale, int channels_last,
                                   const int32_t* image_hw, int stride, float* grad_in, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(image_hw == nullptr || (aligned8(image_hw) && stride > 0),
                  "frr_roi_pool_bwd_deterministic: image_hw must be 8-byte aligned, stride > 0");
    return roi_backward_det<false>(grad_out, argmax, rois, K, B, C, H, W, PH, PW, spatial_scale, 0, 0, channels_last,
                                   grad_in, stream, image_hw, stride);
}
int frr_roi_align_bwd_deterministic(const float* grad_out, const float* rois, int K, int B, int C, int H, int W, int PH,
                                    int PW, float spatial_scale, int sampling_ratio, int aligned, int channels_last,
                                    float* grad_in, frr_stream_t stream) {
    return frr::roi_backward_det<true>(grad_out, nullptr, rois, K, B, C, H, W, PH, PW, spatial_scale, sampling_ratio,
                                       aligned, channels_last, grad_in, stream);
}

}  // extern "C"
