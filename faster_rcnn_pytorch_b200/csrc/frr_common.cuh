// Shared helpers for libfrr.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "frr.h"

namespace frr {

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

#define FRR_CHECK_ARG(cond, ...)            \
    do {                                    \
        if (!(cond)) {                      \
            ::frr::set_error(__VA_ARGS__);  \
            return FRR_E_INVALID;           \
        }                                   \
    } while (0)

#define FRR_CHECK_LAUNCH(what)                                                          \
    do {                                                                                \
        cudaError_t e__ = cudaGetLastError();                                           \
        if (e__ != cudaSuccess) {                                                       \
            ::frr::set_error("%s: %s", what, cudaGetErrorString(e__));                  \
            return FRR_E_LAUNCH;                                                        \
        }                                                                               \
    } while (0)

#define FRR_CUDA(call)                                                                  \
    do {                                                                                \
        cudaError_t e__ = (call);                                                       \
        if (e__ != cudaSuccess) {                                                       \
            ::frr::set_error("%s: %s", #call, cudaGetErrorString(e__));                 \
            return FRR_E_LAUNCH;                                                        \
        }                                                                               \
    } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline int num_sms() {  // of the CURRENT device (cached per device id: a process may drive several GPUs)
    static std::atomic<int> cache[64];
    int dev = 0;
    cudaGetDevice(&dev);
    const int slot = (dev >= 0 && dev < 64) ? dev : 0;
    int n = cache[slot].load(std::memory_order_relaxed);
    if (n == 0) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
        cache[slot].store(n, std::memory_order_relaxed);
    }
    return n;
}

// streaming 128-bit load / store (read-once inputs, write-once outputs)
__device__ __forceinline__ float4 ld_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream(float4* p, const float4& v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// fp32 <-> order-preserving uint32 (ascending uint == ascending float; -0 < +0)
__device__ __forceinline__ uint32_t float_to_ordered(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// block-wide exclusive scan of one value per thread for a 1024-thread CTA; returns the exclusive prefix,
// the block total in *total.  warp_tmp: 32 words of shared memory.  Must be called by all threads.
__device__ __forceinline__ unsigned int block_exclusive_scan(unsigned int v, unsigned int* warp_tmp,
                                                             unsigned int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (blockDim.x + 31) >> 5;
    unsigned int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();  // warp_tmp reuse
    if (lane == 31) warp_tmp[warp] = inc;
    __syncthreads();
    unsigned int wsum = (lane < nwarps) ? warp_tmp[lane] : 0u;
    unsigned int winc = wsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned int t = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += t;
    }
    const unsigned int wexc = __shfl_sync(0xffffffffu, winc - wsum, warp);
    *total = __shfl_sync(0xffffffffu, winc, 31);
    return wexc + inc - v;
}

struct AnchorTable {
    float v[16 * 4];
    int A;
};

int fill_anchor_table(AnchorTable* t, const float* base_table_host, int A, int stride);

// Mixed-size batches (the entry points given image_hw): image b of a batch padded to a grid of grid_h x grid_w cells has
// image_hw[b] = (H_b, W_b) pixels and covers cells y < H_b / stride, x < W_b / stride.  The sizes live in device memory,
// where the host cannot check them, so the extent is clamped to [0, grid] here: an out-of-range size never reads or
// writes outside the padded grid, and an image with an empty extent has no cells.  image_hw must be 8-byte aligned.
__device__ __forceinline__ int2 image_cells(const int32_t* __restrict__ image_hw, int b, int stride, int grid_h,
                                            int grid_w) {
    const int2 hw = __ldg(reinterpret_cast<const int2*>(image_hw) + b);
    return make_int2(min(max(hw.x / stride, 0), grid_h), min(max(hw.y / stride, 0), grid_w));
}
inline bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

}  // namespace frr
