// Shared helpers of the RoIPool / RoIAlign kernels (roi.cu: generic + direct kernels and host dispatch;
// roi_fast.cu: the 7x7 fast paths): TMA 1-D bulk copies, plane load / store, torchvision geometry.
#pragma once
#include <float.h>

#include "frr_common.cuh"

namespace frr {

constexpr int kRoiThreads = 512;
constexpr int kRoiTile = 256;  // rois staged per pass

// ---------------------------------------------------------------------------------------------
// host dispatch: which kernel an RoI entry point runs (ids as reported by frr_roi_variant)
// ---------------------------------------------------------------------------------------------
enum RoiKernel {
    kRoiNone = -1,          // nothing is launched (forward without rois; backward without rois on planes too large for smem)
    kPoolFwdFlat = 0,       // roi_pool_fwd_flat_kernel<cb, argmax>
    kAlignFwdFast = 1,      // roi_align_fwd_fast_kernel<cb>
    kFwdPlanes = 2,         // roi_fwd_planes_kernel<align>
    kFwdDirect = 3,         // roi_fwd_direct_kernel<align>
    kPoolBwdColorTail = 4,  // roi_pool_bwd_color_kernel<8> + roi_pool_bwd_tail_kernel (small rois)
    kPoolBwdTail = 5,       // roi_pool_bwd_tail_kernel for every roi
    kAlignBwdFast = 6,      // roi_align_bwd_fast_kernel<cb>
    kAlignBwdStream = 7,    // roi_align_bwd_stream_kernel
    kBwdPlanes = 8,         // roi_bwd_planes_kernel<align>
    kBwdDirect = 9,         // roi_bwd_direct_kernel<align>
};
struct RoiPick {
    int kernel;   // RoiKernel
    int cb;       // channels per CTA (0: the kernel walks output elements or rois)
    int nz;       // CTAs per (image, channel group)
    int rp;       // roi_align_fwd_fast_kernel: rois per pass
    size_t smem;  // dynamic shared memory bytes
};

// ---------------------------------------------------------------------------------------------
// TMA 1-D bulk copy helpers (global -> shared with mbarrier completion; shared -> global)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(phase)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_wait() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 4-byte cp.async global -> shared (src_bytes 0: zero fill, nothing is read) and its group bookkeeping
__device__ __forceinline__ void cp_async4_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Load CB planes of image b into smem planes[CB][HW].  NCHW: contiguous chunk (TMA when 16-B aligned),
// NHWC: gather CB consecutive channels per pixel.
__device__ __forceinline__ void load_planes(float* planes, const float* __restrict__ feat, int b, int c0, int CB, int C,
                                            int HW, bool nhwc, uint64_t* bar) {
    const int tid = threadIdx.x;
    if (!nhwc) {
        const float* src = feat + ((size_t)b * C + c0) * HW;
        const size_t bytes = (size_t)CB * HW * sizeof(float);
        const bool tma_ok = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && ((bytes & 15u) == 0);
        if (tma_ok) {
            if (tid == 0) {
                mbar_init(bar, 1);
                mbar_expect_tx(bar, (uint32_t)bytes);
                const uint32_t kMax = 32768;
                for (size_t off = 0; off < bytes; off += kMax) {
                    const uint32_t nb = (uint32_t)((bytes - off) < kMax ? (bytes - off) : kMax);
                    bulk_g2s(reinterpret_cast<char*>(planes) + off, reinterpret_cast<const char*>(src) + off, nb, bar);
                }
            }
            __syncthreads();  // barrier init visible to the waiters
            mbar_wait(bar, 0);
        } else {
            for (int i = tid; i < CB * HW; i += blockDim.x) planes[i] = src[i];
        }
    } else {
        const float* src = feat + (size_t)b * HW * C + c0;
        for (int i = tid; i < CB * HW; i += blockDim.x) {
            const int pix = i / CB, cl = i - pix * CB;
            planes[(size_t)cl * HW + pix] = src[(size_t)pix * C + cl];
        }
    }
    __syncthreads();
}

// Store CB planes from smem to image b (zero-copy layout choice as above).
__device__ __forceinline__ void store_planes(const float* planes, float* __restrict__ out, int b, int c0, int CB, int C,
                                             int HW, bool nhwc) {
    const int tid = threadIdx.x;
    __syncthreads();
    if (!nhwc) {
        float* dst = out + ((size_t)b * C + c0) * HW;
        const size_t bytes = (size_t)CB * HW * sizeof(float);
        const bool tma_ok = ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) && ((bytes & 15u) == 0);
        if (tma_ok) {
            fence_async_smem();  // generic-proxy smem writes -> visible to the async proxy
            __syncthreads();
            if (tid == 0) {
                const uint32_t kMax = 32768;
                for (size_t off = 0; off < bytes; off += kMax) {
                    const uint32_t nb = (uint32_t)((bytes - off) < kMax ? (bytes - off) : kMax);
                    bulk_s2g(reinterpret_cast<char*>(dst) + off, reinterpret_cast<const char*>(planes) + off, nb);
                }
                bulk_commit_wait();
            }
        } else {
            for (int i = tid; i < CB * HW; i += blockDim.x) dst[i] = planes[i];
        }
    } else {
        float* dst = out + (size_t)b * HW * C + c0;
        for (int i = tid; i < CB * HW; i += blockDim.x) {
            const int pix = i / CB, cl = i - pix * CB;
            dst[(size_t)pix * C + cl] = planes[(size_t)cl * HW + pix];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------------------------
struct PoolGeom {  // torchvision roi_pool: rounded roi, integer bins
    int sw, sh, rw, rh;
};
__device__ __forceinline__ PoolGeom pool_geom(const float* r, float scale) {
    PoolGeom g;
    g.sw = (int)roundf(__fmul_rn(r[1], scale));
    g.sh = (int)roundf(__fmul_rn(r[2], scale));
    const int ew = (int)roundf(__fmul_rn(r[3], scale));
    const int eh = (int)roundf(__fmul_rn(r[4], scale));
    g.rw = max(ew - g.sw + 1, 1);
    g.rh = max(eh - g.sh + 1, 1);
    return g;
}
__device__ __forceinline__ void pool_window(const PoolGeom& g, int ph, int pw, int PH, int PW, int H, int W, int& hs,
                                            int& he, int& ws, int& we) {
    const float bin_h = __fdiv_rn((float)g.rh, (float)PH);
    const float bin_w = __fdiv_rn((float)g.rw, (float)PW);
    hs = (int)floorf(__fmul_rn((float)ph, bin_h)) + g.sh;
    ws = (int)floorf(__fmul_rn((float)pw, bin_w)) + g.sw;
    he = (int)ceilf(__fmul_rn((float)(ph + 1), bin_h)) + g.sh;
    we = (int)ceilf(__fmul_rn((float)(pw + 1), bin_w)) + g.sw;
    hs = min(max(hs, 0), H);
    he = min(max(he, 0), H);
    ws = min(max(ws, 0), W);
    we = min(max(we, 0), W);
}

struct AlignGeom {  // torchvision roi_align
    float sw, sh, bin_h, bin_w, count;
    int gh, gw;
};
__device__ __forceinline__ AlignGeom align_geom(const float* r, float scale, int PH, int PW, int sampling, bool aligned) {
    AlignGeom g;
    const float off = aligned ? 0.5f : 0.0f;
    g.sw = __fsub_rn(__fmul_rn(r[1], scale), off);
    g.sh = __fsub_rn(__fmul_rn(r[2], scale), off);
    const float ew = __fsub_rn(__fmul_rn(r[3], scale), off);
    const float eh = __fsub_rn(__fmul_rn(r[4], scale), off);
    float rw = __fsub_rn(ew, g.sw), rh = __fsub_rn(eh, g.sh);
    if (!aligned) {
        rw = fmaxf(rw, 1.0f);
        rh = fmaxf(rh, 1.0f);
    }
    g.bin_h = __fdiv_rn(rh, (float)PH);
    g.bin_w = __fdiv_rn(rw, (float)PW);
    g.gh = sampling > 0 ? sampling : (int)ceilf(__fdiv_rn(rh, (float)PH));
    g.gw = sampling > 0 ? sampling : (int)ceilf(__fdiv_rn(rw, (float)PW));
    g.count = (float)max(g.gh * g.gw, 1);
    return g;
}
struct Taps {
    int p1, p2, p3, p4;
    float w1, w2, w3, w4;
};
__device__ __forceinline__ bool bilinear_taps(float y, float x, int H, int W, Taps& t) {
    if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) return false;
    if (y <= 0.f) y = 0.f;
    if (x <= 0.f) x = 0.f;
    int yl = (int)y, xl = (int)x, yh, xh;
    if (yl >= H - 1) { yh = yl = H - 1; y = (float)yl; } else { yh = yl + 1; }
    if (xl >= W - 1) { xh = xl = W - 1; x = (float)xl; } else { xh = xl + 1; }
    const float ly = __fsub_rn(y, (float)yl), lx = __fsub_rn(x, (float)xl);
    const float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
    t.w1 = __fmul_rn(hy, hx); t.w2 = __fmul_rn(hy, lx); t.w3 = __fmul_rn(ly, hx); t.w4 = __fmul_rn(ly, lx);
    t.p1 = yl * W + xl; t.p2 = yl * W + xh; t.p3 = yh * W + xl; t.p4 = yh * W + xh;
    return true;
}
__device__ __forceinline__ float sample_y(const AlignGeom& g, int ph, int iy) {
    // roi_start_h + ph*bin_h + (iy + .5f)*bin_h/grid_h   (left to right)
    return __fadd_rn(__fadd_rn(g.sh, __fmul_rn((float)ph, g.bin_h)),
                     __fdiv_rn(__fmul_rn((float)iy + .5f, g.bin_h), (float)g.gh));
}
__device__ __forceinline__ float sample_x(const AlignGeom& g, int pw, int ix) {
    return __fadd_rn(__fadd_rn(g.sw, __fmul_rn((float)pw, g.bin_w)),
                     __fdiv_rn(__fmul_rn((float)ix + .5f, g.bin_w), (float)g.gw));
}

}  // namespace frr
