// R1-R4: RoIPool / RoIAlign 7x7 forward + backward (torchvision semantics; reference call sites
// models/model.py:97,113 and models/new_model.py:127,143).
//
// Design (B200: 227 KB shared memory per CTA, TMA bulk copies):
//   a CTA owns CB whole channel planes of ONE image.  Forward: the planes are brought into shared
//   memory once (NCHW: one contiguous chunk -> cp.async.bulk / TMA with an mbarrier; channels_last:
//   64-byte granules), then every (roi, channel, bin) output of that image is produced by scanning its
//   window out of shared memory and stored straight to the [K,C,7,7] output, where the CB*49 values of
//   a roi are contiguous (coalesced).  Each feature element is read from HBM exactly once and nothing
//   is transposed, so HBM traffic equals the algorithmic bytes (features + out + argmax).
//   Backward: the CTA owns the CB gradient planes in shared memory, accumulates every roi of its
//   image with shared-memory atomics (no global atomics, no memset pass) and writes each plane once.
//   Planes that do not fit shared memory (large FPN levels) take the direct global-memory kernels.
//
// Numerics: RoIPool max/argmax bit-exact (first strict maximum in h-then-w order, -FLT_MAX start,
// empty bin -> 0/-1); RoIAlign sums w1*v1+w2*v2+w3*v3+w4*v4 left to right without FMA contraction.
#include <stdlib.h>
#include <string.h>

#include "roi_common.cuh"

namespace frr {


// Stage the rois of image b found in rois[tile .. tile+kRoiTile) into smem (ids + 5 floats each).
__device__ __forceinline__ int stage_rois(const float* __restrict__ rois, int K, int tile, int b, int* s_id, float* s_roi,
                                          int* s_n) {
    if (threadIdx.x == 0) *s_n = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < kRoiTile; t += blockDim.x) {
        const int k = tile + t;
        if (k < K && (int)rois[5 * (size_t)k] == b) {
            const int slot = atomicAdd(s_n, 1);
            s_id[slot] = k;
#pragma unroll
            for (int q = 0; q < 5; ++q) s_roi[5 * slot + q] = rois[5 * (size_t)k + q];
        }
    }
    __syncthreads();
    return *s_n;
}

struct RoiSmemHdr {
    uint64_t bar;
    int n;
    int pad;
    int id[kRoiTile];
    float roi[kRoiTile * 5];
};

// ---------------------------------------------------------------------------------------------
// forward (planes in shared memory)
// ---------------------------------------------------------------------------------------------
template <bool kAlign>
__global__ void __launch_bounds__(kRoiThreads)
    roi_fwd_planes_kernel(const float* __restrict__ feat, const float* __restrict__ rois, int K, int C, int H, int W,
                          int CB, int PH, int PW, float scale, int sampling, int aligned, int nhwc,
                          float* __restrict__ out, int32_t* __restrict__ argmax) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RoiSmemHdr* hd = reinterpret_cast<RoiSmemHdr*>(smem_raw);
    float* planes = reinterpret_cast<float*>(smem_raw + ((sizeof(RoiSmemHdr) + 127) & ~(size_t)127));
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int HW = H * W, bins = PH * PW;
    const int cb = min(CB, C - c0);
    load_planes(planes, feat, b, c0, cb, C, HW, nhwc != 0, &hd->bar);

    for (int tile = 0; tile < K; tile += kRoiTile) {
        const int ns = stage_rois(rois, K, tile, b, hd->id, hd->roi, &hd->n);
        const int items = ns * cb * bins;
        for (int it = threadIdx.x; it < items; it += blockDim.x) {
            const int slot = it / (cb * bins);
            const int rem = it - slot * (cb * bins);
            const int cl = rem / bins, bin = rem - cl * bins;
            const int ph = bin / PW, pw = bin - ph * PW;
            const float* pl = planes + (size_t)cl * HW;
            const size_t o = ((size_t)hd->id[slot] * C + c0 + cl) * bins + bin;
            if (!kAlign) {
                const PoolGeom g = pool_geom(hd->roi + 5 * slot, scale);
                int hs, he, ws, we;
                pool_window(g, ph, pw, PH, PW, H, W, hs, he, ws, we);
                const bool empty = (he <= hs) || (we <= ws);
                float best = empty ? 0.f : -FLT_MAX;
                int bi = -1;
                for (int h = hs; h < he; ++h)
                    for (int w = ws; w < we; ++w) {
                        const float v = pl[h * W + w];
                        if (v > best) { best = v; bi = h * W + w; }
                    }
                out[o] = best;
                if (argmax) argmax[o] = bi;
            } else {
                const AlignGeom g = align_geom(hd->roi + 5 * slot, scale, PH, PW, sampling, aligned != 0);
                float acc = 0.f;
                for (int iy = 0; iy < g.gh; ++iy) {
                    const float y = sample_y(g, ph, iy);
                    for (int ix = 0; ix < g.gw; ++ix) {
                        const float x = sample_x(g, pw, ix);
                        Taps t;
                        if (bilinear_taps(y, x, H, W, t)) {
                            const float v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t.w1, pl[t.p1]), __fmul_rn(t.w2, pl[t.p2])),
                                                                __fmul_rn(t.w3, pl[t.p3])),
                                                      __fmul_rn(t.w4, pl[t.p4]));
                            acc = __fadd_rn(acc, v);
                        }
                    }
                }
                out[o] = __fdiv_rn(acc, g.count);
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// backward (gradient planes accumulated in shared memory, written once)
// ---------------------------------------------------------------------------------------------
template <bool kAlign>
__global__ void __launch_bounds__(kRoiThreads)
    roi_bwd_planes_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                          const float* __restrict__ rois, int K, int C, int H, int W, int CB, int PH, int PW, float scale,
                          int sampling, int aligned, int nhwc, float* __restrict__ grad_in) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RoiSmemHdr* hd = reinterpret_cast<RoiSmemHdr*>(smem_raw);
    float* planes = reinterpret_cast<float*>(smem_raw + ((sizeof(RoiSmemHdr) + 127) & ~(size_t)127));
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int HW = H * W, bins = PH * PW;
    const int cb = min(CB, C - c0);
    for (int i = threadIdx.x; i < cb * HW; i += blockDim.x) planes[i] = 0.f;
    __syncthreads();

    for (int tile = 0; tile < K; tile += kRoiTile) {
        const int ns = stage_rois(rois, K, tile, b, hd->id, hd->roi, &hd->n);
        const int items = ns * cb * bins;
        for (int it = threadIdx.x; it < items; it += blockDim.x) {
            const int slot = it / (cb * bins);
            const int rem = it - slot * (cb * bins);
            const int cl = rem / bins, bin = rem - cl * bins;
            float* pl = planes + (size_t)cl * HW;
            const size_t o = ((size_t)hd->id[slot] * C + c0 + cl) * bins + bin;
            const float go = grad_out[o];
            if (!kAlign) {
                const int a = argmax[o];
                if (a >= 0) atomicAdd(pl + a, go);
            } else {
                const int ph = bin / PW, pw = bin - ph * PW;
                const AlignGeom g = align_geom(hd->roi + 5 * slot, scale, PH, PW, sampling, aligned != 0);
                for (int iy = 0; iy < g.gh; ++iy) {
                    const float y = sample_y(g, ph, iy);
                    for (int ix = 0; ix < g.gw; ++ix) {
                        const float x = sample_x(g, pw, ix);
                        Taps t;
                        if (bilinear_taps(y, x, H, W, t)) {
                            atomicAdd(pl + t.p1, __fdiv_rn(__fmul_rn(go, t.w1), g.count));
                            atomicAdd(pl + t.p2, __fdiv_rn(__fmul_rn(go, t.w2), g.count));
                            atomicAdd(pl + t.p3, __fdiv_rn(__fmul_rn(go, t.w3), g.count));
                            atomicAdd(pl + t.p4, __fdiv_rn(__fmul_rn(go, t.w4), g.count));
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    store_planes(planes, grad_in, b, c0, cb, C, HW, nhwc != 0);
}

// ---------------------------------------------------------------------------------------------
// direct global-memory kernels for planes too large for shared memory (NCHW or NHWC)
// ---------------------------------------------------------------------------------------------
template <bool kAlign>
__global__ void __launch_bounds__(256)
    roi_fwd_direct_kernel(const float* __restrict__ feat, const float* __restrict__ rois, size_t total, int B, int C, int H, int W,
                          int PH, int PW, float scale, int sampling, int aligned, int nhwc, float* __restrict__ out,
                          int32_t* __restrict__ argmax) {
    const int bins = PH * PW;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (size_t)gridDim.x * blockDim.x) {
        const int bin = (int)(o % bins);
        const int c = (int)((o / bins) % C);
        const size_t k = o / ((size_t)bins * C);
        const int ph = bin / PW, pw = bin - ph * PW;
        const float* r = rois + 5 * k;
        const int b = (int)r[0];
        // masked roi (index -1: belongs to another pyramid level / padding row, its output row is written elsewhere);
        // an index >= B is malformed input and is skipped the same way instead of reading out of bounds
        if (b < 0 || b >= B) continue;
        const float* base = nhwc ? feat + (size_t)b * H * W * C + c : feat + ((size_t)b * C + c) * H * W;
        const size_t ps = nhwc ? (size_t)C : 1;  // pixel stride
        if (!kAlign) {
            const PoolGeom g = pool_geom(r, scale);
            int hs, he, ws, we;
            pool_window(g, ph, pw, PH, PW, H, W, hs, he, ws, we);
            const bool empty = (he <= hs) || (we <= ws);
            float best = empty ? 0.f : -FLT_MAX;
            int bi = -1;
            for (int h = hs; h < he; ++h)
                for (int w = ws; w < we; ++w) {
                    const float v = base[(size_t)(h * W + w) * ps];
                    if (v > best) { best = v; bi = h * W + w; }
                }
            out[o] = best;
            if (argmax) argmax[o] = bi;
        } else {
            const AlignGeom g = align_geom(r, scale, PH, PW, sampling, aligned != 0);
            float acc = 0.f;
            for (int iy = 0; iy < g.gh; ++iy) {
                const float y = sample_y(g, ph, iy);
                for (int ix = 0; ix < g.gw; ++ix) {
                    const float x = sample_x(g, pw, ix);
                    Taps t;
                    if (bilinear_taps(y, x, H, W, t)) {
                        const float v = __fadd_rn(
                            __fadd_rn(__fadd_rn(__fmul_rn(t.w1, base[t.p1 * ps]), __fmul_rn(t.w2, base[t.p2 * ps])),
                                      __fmul_rn(t.w3, base[t.p3 * ps])),
                            __fmul_rn(t.w4, base[t.p4 * ps]));
                        acc = __fadd_rn(acc, v);
                    }
                }
            }
            out[o] = __fdiv_rn(acc, g.count);
        }
    }
}

template <bool kAlign>
__global__ void __launch_bounds__(256)
    roi_bwd_direct_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                          const float* __restrict__ rois, size_t total, int B, int C, int H, int W, int PH, int PW, float scale,
                          int sampling, int aligned, int nhwc, float* __restrict__ grad_in /* zeroed */) {
    const int bins = PH * PW;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (size_t)gridDim.x * blockDim.x) {
        const int bin = (int)(o % bins);
        const int c = (int)((o / bins) % C);
        const size_t k = o / ((size_t)bins * C);
        const float* r = rois + 5 * k;
        const int b = (int)r[0];
        if (b < 0 || b >= B) continue;  // masked / malformed roi: contributes nothing
        float* base = nhwc ? grad_in + (size_t)b * H * W * C + c : grad_in + ((size_t)b * C + c) * H * W;
        const size_t ps = nhwc ? (size_t)C : 1;
        const float go = grad_out[o];
        if (!kAlign) {
            const int a = argmax[o];
            if (a >= 0) atomicAdd(base + (size_t)a * ps, go);
        } else {
            const int ph = bin / PW, pw = bin - ph * PW;
            const AlignGeom g = align_geom(r, scale, PH, PW, sampling, aligned != 0);
            for (int iy = 0; iy < g.gh; ++iy) {
                const float y = sample_y(g, ph, iy);
                for (int ix = 0; ix < g.gw; ++ix) {
                    const float x = sample_x(g, pw, ix);
                    Taps t;
                    if (bilinear_taps(y, x, H, W, t)) {
                        atomicAdd(base + t.p1 * ps, __fdiv_rn(__fmul_rn(go, t.w1), g.count));
                        atomicAdd(base + t.p2 * ps, __fdiv_rn(__fmul_rn(go, t.w2), g.count));
                        atomicAdd(base + t.p3 * ps, __fdiv_rn(__fmul_rn(go, t.w3), g.count));
                        atomicAdd(base + t.p4 * ps, __fdiv_rn(__fmul_rn(go, t.w4), g.count));
                    }
                }
            }
        }
    }
}

// RoIAlign backward for maps on which the separable plane kernel (roi_fast.cu) is left with 8 or fewer planes per SM
// (50 x 83: latency bound, 2.7 ms): one CTA per roi.  The <= 16 bilinear taps of every bin (2 x 2 samples x 4 taps,
// channel independent) are built once per roi, weights divided by the sample count and taps on the same pixel merged
// (neighbouring samples share pixel rows / columns: ~9 distinct pixels per bin instead of 16), then the roi's C * 49
// contiguous gradients are streamed and scattered with RED.ADD.F32.  A thread keeps ONE bin for every element it visits
// (490 = 10 x 49 threads, element t + 490 j has bin t % 49), so the bin's taps live in registers for the whole roi and an
// element costs one load + one multiply and one atomic per tap: 1.10-1.49 ms on that map (torchvision, which recomputes
// the geometry per element and issues all 16 atomics: 1.82-1.90 ms); 0.84-1.30 ms at 37 x 62 (plane kernel 1.21-1.25 ms).
struct AlignTapTable {
    int n[49];
    int idx[49][16];
    float w[49][16];
};

constexpr int kAlignStreamThreads = 490;  // 10 x 49: thread t keeps bin t % 49 for every element t + 490 j it visits

__global__ void __launch_bounds__(kAlignStreamThreads)
    roi_align_bwd_stream_kernel(const float* __restrict__ grad_out, const float* __restrict__ rois, int B, int C, int H, int W,
                                float scale, int aligned, int nhwc, float* __restrict__ grad_in /* zeroed */) {
    __shared__ AlignTapTable tb;
    const int k = blockIdx.x;
    const float* r = rois + 5 * (size_t)k;
    const int b = (int)__ldg(r);
    if (b < 0 || b >= B) return;
    if (threadIdx.x < 49) {
        const int bin = threadIdx.x, ph = bin / 7, pw = bin - ph * 7;
        const AlignGeom g = align_geom(r, scale, 7, 7, 2, aligned != 0);
        int n = 0;
        for (int iy = 0; iy < 2; ++iy) {
            const float y = sample_y(g, ph, iy);
            for (int ix = 0; ix < 2; ++ix) {
                const float x = sample_x(g, pw, ix);
                Taps t;
                if (!bilinear_taps(y, x, H, W, t)) continue;
                const int pi[4] = {t.p1, t.p2, t.p3, t.p4};
                const float wi[4] = {t.w1, t.w2, t.w3, t.w4};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float wq = __fmul_rn(wi[q], 0.25f);
                    int j = 0;
                    while (j < n && tb.idx[bin][j] != pi[q]) ++j;
                    if (j < n) {
                        tb.w[bin][j] = __fadd_rn(tb.w[bin][j], wq);
                    } else {
                        tb.idx[bin][n] = pi[q];
                        tb.w[bin][n] = wq;
                        ++n;
                    }
                }
            }
        }
        for (int j = n; j < 16; ++j) { tb.idx[bin][j] = 0; tb.w[bin][j] = 0.f; }
        tb.n[bin] = n;
    }
    __syncthreads();
    // the taps of this thread's bin, in registers for the whole roi (pixel offsets pre-multiplied by the pixel stride)
    const int bin = threadIdx.x % 49;
    const int HW = H * W;
    const size_t ps = nhwc ? (size_t)C : 1;
    const int n = tb.n[bin];
    int ti[16];
    float tw[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { ti[j] = tb.idx[bin][j] * (int)ps; tw[j] = tb.w[bin][j]; }
    const int total = C * 49;
    const size_t src0 = (size_t)k * total, img = (size_t)b * C * HW;
    const size_t cstep = nhwc ? (size_t)1 : (size_t)HW;  // channel stride
    constexpr int U = 4;
    for (int e0 = threadIdx.x; e0 < total; e0 += U * kAlignStreamThreads) {
        float gv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * kAlignStreamThreads;
            gv[u] = e < total ? __ldg(grad_out + src0 + e) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * kAlignStreamThreads;
            if (e >= total) break;
            float* base = grad_in + img + (size_t)(e / 49) * cstep;
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (j < n) atomicAdd(base + ti[j], __fmul_rn(gv[u], tw[j]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// 7x7 fast paths (roi_fast.cu, roi_pool_bwd.cu): *_pick fills the choice (false = shape outside the fast path),
// *_launch runs it (0 = launched, < 0 = error)
bool roi_fwd_fast_pick(bool align, int B, int C, int H, int W, int PH, int PW, int sampling, RoiPick* pk);
int roi_fwd_fast_launch(const RoiPick& pk, const float* feat, const float* rois, int K, int B, int C, int H, int W,
                        float scale, int aligned, int nhwc, float* out, int32_t* argmax, frr_stream_t stream);
bool roi_align_bwd_fast_pick(int B, int C, int H, int W, int PH, int PW, int sampling, RoiPick* pk);
int roi_align_bwd_fast_launch(const RoiPick& pk, const float* grad_out, const float* rois, int K, int B, int C, int H, int W,
                              float scale, int aligned, int nhwc, float* grad_in, frr_stream_t stream);
bool roi_pool_bwd_fast_pick(int K, int H, int W, int PH, int PW, bool ptrs_aligned, bool force_tail, RoiPick* pk);
int roi_pool_bwd_fast_launch(const RoiPick& pk, const float* grad_out, const int32_t* argmax, const float* rois, int K, int B,
                             int C, int H, int W, float scale, int nhwc, float* grad_in, frr_stream_t stream);

// developer knob (A/B measurements only): FRR_ROI_POOL_BWD=tail sends every roi through the streaming atomic kernel
static int pool_bwd_force_tail() {
    static const int v = [] {
        const char* e = getenv("FRR_ROI_POOL_BWD");
        return (e && !strcmp(e, "tail")) ? 1 : 0;
    }();
    return v;
}

static size_t roi_smem_bytes(int CB, int HW) {
    return ((sizeof(RoiSmemHdr) + 127) & ~(size_t)127) + (size_t)CB * HW * sizeof(float);
}

// channels per CTA: the largest of {16,8,4,2,1} that fits shared memory while keeping >= one wave of CTAs
static int pick_cb(int B, int C, int HW) {
    const size_t limit = 200 * 1024;
    int best = 0;
    for (int cb = 16; cb >= 1; cb >>= 1) {
        if (roi_smem_bytes(cb, HW) > limit) continue;
        if (best == 0) best = cb;
        const long ctas = (long)B * ((C + cb - 1) / cb);
        if (ctas >= (long)num_sms()) return cb;
        best = cb;
    }
    return best;  // 0 -> does not fit at all
}

// The kernel an RoI entry point runs (host only, launches nothing): shared by the launchers below and frr_roi_variant.
// op: 0 roi_pool fwd, 1 roi_pool bwd, 2 roi_align fwd, 3 roi_align bwd.  ptrs_aligned: grad_out and argmax are 4-byte
// aligned (the colour-class RoIPool backward copies them word by word with cp.async).
static int roi_pick(int op, int K, int B, int C, int H, int W, int PH, int PW, int sampling, bool ptrs_aligned, RoiPick* pk) {
    FRR_CHECK_ARG(op >= 0 && op <= 3, "roi variant: op %d not in 0..3", op);
    FRR_CHECK_ARG(K >= 0 && B > 0 && C > 0 && H > 0 && W > 0 && PH > 0 && PW > 0 && B <= 65535, "roi %s: bad sizes",
                  (op & 1) ? "backward" : "forward");
    const bool align = op >= 2, bwd = (op & 1) != 0;
    const int HW = H * W;
    if (!bwd) {
        if (K == 0) { *pk = RoiPick{kRoiNone, 0, 0, 0, 0}; return FRR_OK; }
        if (roi_fwd_fast_pick(align, B, C, H, W, PH, PW, sampling, pk)) return FRR_OK;
    } else if (K > 0) {
        if (align ? roi_align_bwd_fast_pick(B, C, H, W, PH, PW, sampling, pk)
                  : roi_pool_bwd_fast_pick(K, H, W, PH, PW, ptrs_aligned, pool_bwd_force_tail() != 0, pk))
            return FRR_OK;
    }
    const int cb = pick_cb(B, C, HW);
    if (cb > 0) *pk = RoiPick{bwd ? kBwdPlanes : kFwdPlanes, cb, 1, 0, roi_smem_bytes(cb, HW)};
    else *pk = RoiPick{(bwd && K == 0) ? kRoiNone : bwd ? kBwdDirect : kFwdDirect, 0, 1, 0, 0};
    return FRR_OK;
}

static int direct_blocks(size_t total) {
    return (int)((total + 255) / 256 < (size_t)num_sms() * 16 ? (total + 255) / 256 : (size_t)num_sms() * 16);
}

template <bool kAlign>
static int roi_forward(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW, float scale,
                       int sampling, int aligned, int nhwc, float* out, int32_t* argmax, frr_stream_t stream) {
    FRR_CHECK_ARG(K == 0 || (feat && out && rois), "roi forward: null pointer");
    RoiPick pk;
    {
        const int rc = roi_pick(kAlign ? 2 : 0, K, B, C, H, W, PH, PW, sampling, true, &pk);
        if (rc) return rc;
    }
    if (pk.kernel == kRoiNone) return FRR_OK;
    if (pk.kernel == kPoolFwdFlat || pk.kernel == kAlignFwdFast)
        return roi_fwd_fast_launch(pk, feat, rois, K, B, C, H, W, scale, aligned, nhwc, out, kAlign ? nullptr : argmax, stream);
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.kernel == kFwdPlanes) {
        auto kern = roi_fwd_planes_kernel<kAlign>;
        FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        dim3 grid((C + pk.cb - 1) / pk.cb, B);
        kern<<<grid, kRoiThreads, pk.smem, st>>>(feat, rois, K, C, H, W, pk.cb, PH, PW, scale, sampling, aligned, nhwc, out,
                                                 argmax);
    } else {
        const size_t total = (size_t)K * C * PH * PW;
        roi_fwd_direct_kernel<kAlign><<<direct_blocks(total), 256, 0, st>>>(feat, rois, total, B, C, H, W, PH, PW, scale,
                                                                            sampling, aligned, nhwc, out, argmax);
    }
    count_launch();
    FRR_CHECK_LAUNCH("roi forward kernel");
    return FRR_OK;
}

template <bool kAlign>
static int roi_backward(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C, int H, int W,
                        int PH, int PW, float scale, int sampling, int aligned, int nhwc, float* grad_in,
                        frr_stream_t stream) {
    FRR_CHECK_ARG(grad_in && (K == 0 || (grad_out && rois)), "roi backward: null pointer");
    FRR_CHECK_ARG(kAlign || K == 0 || argmax, "roi_pool backward: argmax is required");
    const bool ptrs_aligned =
        !(reinterpret_cast<uintptr_t>(grad_out) & 3u) && !(reinterpret_cast<uintptr_t>(argmax) & 3u);
    RoiPick pk;
    {
        const int rc = roi_pick(kAlign ? 3 : 1, K, B, C, H, W, PH, PW, sampling, ptrs_aligned, &pk);
        if (rc) return rc;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = H * W;
    switch (pk.kernel) {
        case kPoolBwdColorTail:
        case kPoolBwdTail:
            return roi_pool_bwd_fast_launch(pk, grad_out, argmax, rois, K, B, C, H, W, scale, nhwc, grad_in, stream);
        case kAlignBwdFast:
            return roi_align_bwd_fast_launch(pk, grad_out, rois, K, B, C, H, W, scale, aligned, nhwc, grad_in, stream);
        case kAlignBwdStream:
            FRR_CUDA(cudaMemsetAsync(grad_in, 0, (size_t)B * C * HW * sizeof(float), st));
            roi_align_bwd_stream_kernel<<<K, kAlignStreamThreads, 0, st>>>(grad_out, rois, B, C, H, W, scale, aligned, nhwc,
                                                                           grad_in);
            count_launch();
            FRR_CHECK_LAUNCH("roi_align_bwd_stream_kernel");
            return FRR_OK;
        case kBwdPlanes: {
            auto kern = roi_bwd_planes_kernel<kAlign>;
            FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            dim3 grid((C + pk.cb - 1) / pk.cb, B);
            kern<<<grid, kRoiThreads, pk.smem, st>>>(grad_out, argmax, rois, K, C, H, W, pk.cb, PH, PW, scale, sampling, aligned,
                                                     nhwc, grad_in);
            count_launch();
            break;
        }
        default:  // kBwdDirect, or kRoiNone (no rois): the zeroed gradient
            FRR_CUDA(cudaMemsetAsync(grad_in, 0, (size_t)B * C * HW * sizeof(float), st));
            if (pk.kernel == kBwdDirect) {
                const size_t total = (size_t)K * C * PH * PW;
                roi_bwd_direct_kernel<kAlign><<<direct_blocks(total), 256, 0, st>>>(grad_out, argmax, rois, total, B, C, H, W, PH,
                                                                                    PW, scale, sampling, aligned, nhwc, grad_in);
                count_launch();
            }
    }
    FRR_CHECK_LAUNCH("roi backward kernel");
    return FRR_OK;
}

// MultiScaleRoIAlign level assignment (TV ops/poolers.py LevelMapper, used by models/new_model.py:127,143):
//   lvl = clamp(floor(lvl0 + log2(sqrt(area) / s0) + 1e-6), k_min, k_max) - k_min
// and, for every level l, a copy of the rois whose batch index is kept for rois of that level and -1 otherwise: the
// per-level RoIAlign launches then skip foreign rois and all write into ONE [K,C,7,7] output, no index gathers.
__global__ void __launch_bounds__(256)
    fpn_level_rois_kernel(const float* __restrict__ rois, int K, int k_min, int k_max, float lvl0, float s0, int L,
                          int32_t* __restrict__ levels, float* __restrict__ rois_lvl) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const float* r = rois + 5 * (size_t)k;
    const float area = __fmul_rn(__fsub_rn(r[3], r[1]), __fsub_rn(r[4], r[2]));
    const float s = sqrtf(area);
    float t = floorf(__fadd_rn(__fadd_rn(lvl0, log2f(__fdiv_rn(s, s0))), 1e-6f));
    t = fminf(fmaxf(t, (float)k_min), (float)k_max);  // NaN (negative area) -> k_min, like torch.clamp + to(int64) is not defined
    const int lvl = (int)t - k_min;
    levels[k] = lvl;
    for (int l = 0; l < L; ++l) {
        float* o = rois_lvl + ((size_t)l * K + k) * 5;
        o[0] = (l == lvl) ? r[0] : -1.0f;
        o[1] = r[1]; o[2] = r[2]; o[3] = r[3]; o[4] = r[4];
    }
}

// R1 glue (models/model.py:104-110 + TV ops/_utils.py:18-25): normalised rois [B,R,4] -> feature-map rois [B*R,5] with
// the batch index in column 0; rows past count[b] get index -1 (masked: the RoI kernels skip them).
__global__ void __launch_bounds__(256)
    rois5_kernel(const float4* __restrict__ rois, const int32_t* __restrict__ count, int B, int R, float fw, float fh,
                 float* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= B * R) return;
    const int b = k / R, r = k - b * R;
    const float4 v = rois[k];
    float* o = out + 5 * (size_t)k;
    o[0] = (count == nullptr || r < count[b]) ? (float)b : -1.0f;
    o[1] = __fmul_rn(v.x, fw);
    o[2] = __fmul_rn(v.y, fh);
    o[3] = __fmul_rn(v.z, fw);
    o[4] = __fmul_rn(v.w, fh);
}

}  // namespace frr

extern "C" {

int frr_rois5(const float* rois, const int32_t* count, int B, int R, float fw, float fh, float* rois5, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(B >= 0 && R >= 0, "frr_rois5: bad sizes");
    if (B == 0 || R == 0) return FRR_OK;
    FRR_CHECK_ARG(rois && rois5 && aligned16(rois), "frr_rois5: rois must be non-null and 16-byte aligned");
    rois5_kernel<<<(B * R + 255) / 256, 256, 0, (cudaStream_t)stream>>>((const float4*)rois, count, B, R, fw, fh, rois5);
    count_launch();
    FRR_CHECK_LAUNCH("rois5_kernel");
    return FRR_OK;
}

int frr_fpn_level_rois(const float* rois5, int K, int k_min, int k_max, int canonical_level, float canonical_scale, int L,
                       int32_t* levels, float* rois_per_level, frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(K >= 0 && L >= 1 && k_max >= k_min && k_max - k_min + 1 == L && canonical_scale > 0.f,
                  "frr_fpn_level_rois: bad arguments (L must equal k_max - k_min + 1)");
    if (K == 0) return FRR_OK;
    FRR_CHECK_ARG(rois5 && levels && rois_per_level, "frr_fpn_level_rois: null pointer");
    fpn_level_rois_kernel<<<(K + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rois5, K, k_min, k_max, (float)canonical_level,
                                                                            canonical_scale, L, levels, rois_per_level);
    count_launch();
    FRR_CHECK_LAUNCH("fpn_level_rois_kernel");
    return FRR_OK;
}

int frr_roi_pool_fwd(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                     float spatial_scale, int channels_last, float* out, int32_t* argmax, frr_stream_t stream) {
    return frr::roi_forward<false>(feat, rois, K, B, C, H, W, PH, PW, spatial_scale, 0, 0, channels_last, out, argmax, stream);
}
int frr_roi_pool_bwd(const float* grad_out, const int32_t* argmax, const float* rois, int K, int B, int C, int H, int W,
                     int PH, int PW, float spatial_scale, int channels_last, float* grad_in, frr_stream_t stream) {
    return frr::roi_backward<false>(grad_out, argmax, rois, K, B, C, H, W, PH, PW, spatial_scale, 0, 0, channels_last, grad_in,
                                    stream);
}
int frr_roi_align_fwd(const float* feat, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                      float spatial_scale, int sampling_ratio, int aligned, int channels_last, float* out,
                      frr_stream_t stream) {
    return frr::roi_forward<true>(feat, rois, K, B, C, H, W, PH, PW, spatial_scale, sampling_ratio, aligned, channels_last, out,
                                  nullptr, stream);
}
int frr_roi_align_bwd(const float* grad_out, const float* rois, int K, int B, int C, int H, int W, int PH, int PW,
                      float spatial_scale, int sampling_ratio, int aligned, int channels_last, float* grad_in,
                      frr_stream_t stream) {
    return frr::roi_backward<true>(grad_out, nullptr, rois, K, B, C, H, W, PH, PW, spatial_scale, sampling_ratio, aligned,
                                   channels_last, grad_in, stream);
}

int frr_roi_variant(int op, int K, int B, int C, int H, int W, int PH, int PW, int sampling_ratio, int want_argmax,
                    int32_t* out4) {
    using namespace frr;
    FRR_CHECK_ARG(out4 != nullptr, "frr_roi_variant: null output");
    (void)want_argmax;  // selects the kArg instantiation of the same kernel, never another kernel
    RoiPick pk;
    const int rc = roi_pick(op, K, B, C, H, W, PH, PW, sampling_ratio, true, &pk);
    if (rc) return rc;
    out4[0] = pk.kernel;
    out4[1] = pk.cb;
    out4[2] = pk.nz;
    out4[3] = (int32_t)pk.smem;
    return FRR_OK;
}

}  // extern "C"
