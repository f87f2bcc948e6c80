// R1-R4 fast paths: RoIPool / RoIAlign 7x7 on feature planes that fit shared memory (the VGG16 stride-16 map of
// models/model.py:97,113 and the coarse FPN levels of models/new_model.py:127,143).
//
// A CTA owns CB channel planes of ONE image; every feature element is read from HBM once and every output
// element written once (HBM traffic = the algorithmic bytes), for NCHW and channels_last inputs alike.
//
// Forward (CB = 8 or 4): the features are staged in shared memory PIXEL-MAJOR ([pixel][CB], chunk-rotated so that the
//   8 lanes of a quarter-warp hit 8 different bank groups unless their pixels agree mod 8): a thread owns one bin and
//   ALL CB channels, so CB/4 LDS.128 feed CB running maxima and every loop / bounds / index instruction is shared by
//   CB channels (one channel per thread cost 131 warp instructions per bin and channel, this layout ~25).  The
//   per-roi geometry (bin boundaries for RoIPool, 1-D bilinear sample records for RoIAlign) is computed once per roi
//   into shared memory, not once per output element.
//   RoIPool (roi_pool_fwd_flat_kernel): a warp owns a share of the image's rois (ordered by window size) and walks
//   their flattened bins 32 at a time, storing straight to the [K,C,7,7] output (lanes = consecutive bins =
//   consecutive addresses): no per-pass barriers, no staging tile, every lane busy.
//   RoIAlign (roi_align_fwd_fast_kernel): 9 rois x 49 bins per pass, results staged in a [roi][channel][49] tile (= the
//   output layout) and written with coalesced 16-byte streaming stores.
// Backward: RoIPool in roi_pool_bwd.cu (colour classes, no atomics on the plane path); RoIAlign below (separable).
//
// Numerics: RoIPool max/argmax bit-exact vs torchvision CPU (same scan order, strict >); RoIAlign keeps
// torchvision's operation order (w1*v1+w2*v2+w3*v3+w4*v4, samples iy-major, / count), no FMA contraction.
#include "roi_common.cuh"

namespace frr {

constexpr int kFastFwdThreads = 448;
constexpr int kIdCap = 512;  // rois scanned per tile (one per thread, blockDim <= 512)

// developer instrumentation: clock64() cycles of CTA (0,0) per phase, accumulated over launches
__device__ long long g_roi_dbg[16];
#define ROI_TICK(slot)                          \
    if (prof) {                                 \
        const long long t1_ = clock64();        \
        g_roi_dbg[slot] += t1_ - t0_;           \
        t0_ = t1_;                              \
    }

struct FastHdr {
    int cnt[16];
    int id[kIdCap];
    int id2[kIdCap];              // forward RoIPool: the same rois ordered by window size
    unsigned short key[kIdCap];
};
constexpr int kHdrBytes = 5376;
static_assert(sizeof(FastHdr) <= kHdrBytes, "header does not fit");

struct AlignRec {  // 1-D half of torchvision's bilinear_interpolate for one sample coordinate
    int lo, hi;    // lo < 0: the sample is outside [-1, size] and contributes nothing
    float l, h;    // weights of hi / lo
};

__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Ordered list of the rois of image b inside rois[tile, tile + blockDim): ids ascending.  Called by all threads
// (blockDim a multiple of 32, <= 512).  Returns the count.
__device__ __forceinline__ int stage_ids(const float* __restrict__ rois, int K, int tile, int b, FastHdr* hd) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = blockDim.x >> 5;
    const int k = tile + tid;
    const bool ok = (k < K) && ((int)__ldg(rois + 5 * (size_t)k) == b);
    const unsigned int m = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) hd->cnt[warp] = __popc(m);
    __syncthreads();
    int pre = 0, tot = 0;
    for (int w = 0; w < nwarps; ++w) {
        const int c = hd->cnt[w];
        if (w < warp) pre += c;
        tot += c;
    }
    if (ok) hd->id[pre + __popc(m & ((1u << lane) - 1u))] = k;
    __syncthreads();
    return tot;
}

// The same list for a WIDE window: every thread looks at PER consecutive rois of rois[k0, k0 + PER * blockDim) with all
// its loads in flight, so a batch of a few thousand rois is scanned once per CTA instead of once per 448 rois (the scan
// is a chain of global-load and barrier latencies: ~5 K cycles a round, 30 % of a CTA's life when every 448-roi tile
// paid it).  Returns the number of matches; *mine (bit j = roi k0 + tid * PER + j matches) and *pos (list position of
// the thread's first match) stay in registers and ids_emit() writes the list out 'cap' entries at a time.
template <int PER>
__device__ __forceinline__ int ids_scan(const float* __restrict__ rois, int K, int k0, int b, FastHdr* hd, unsigned int* mine,
                                        int* pos) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int lo = k0 + tid * PER;
    float bi[PER];
#pragma unroll
    for (int j = 0; j < PER; ++j) bi[j] = __ldg(rois + 5 * (size_t)min(lo + j, K - 1));
    unsigned int m = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j)
        if (lo + j < K && (int)bi[j] == b) m |= 1u << j;
    const int v = __popc(m);
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();  // cnt reuse
    if (lane == 31) hd->cnt[warp] = inc;
    __syncthreads();
    int pre = 0, tot = 0;
    for (int w = 0; w < nwarps; ++w) {
        const int c = hd->cnt[w];
        if (w < warp) pre += c;
        tot += c;
    }
    *mine = m;
    *pos = pre + inc - v;
    return tot;
}
// entries [r0, r0 + cap) of the list go to hd->id[0, cap) (ids ascending).  Called by all threads.
template <int PER>
__device__ __forceinline__ void ids_emit(int k0, unsigned int mine, int pos, int r0, int cap, FastHdr* hd) {
    const int lo = k0 + (int)threadIdx.x * PER;
    while (mine) {
        const int j = __ffs(mine) - 1;
        mine &= mine - 1u;
        if (pos >= r0 && pos < r0 + cap) hd->id[pos - r0] = lo + j;
        ++pos;
    }
    __syncthreads();
}

// RoIPool forward processes RS rois per pass with a barrier per pass, so a pass costs as much as its LARGEST window:
// order the image's rois by their per-bin window size (descending rank sort, ns <= 512 keys in shared memory) so that
// every pass works on rois of similar cost.  The output position of a roi is its id, so the order is free.
__device__ __forceinline__ void order_ids_by_window(const float* __restrict__ rois, float scale, int ns, FastHdr* hd) {
    const int tid = threadIdx.x;
    if (tid < ns) {
        const PoolGeom gm = pool_geom(rois + 5 * (size_t)hd->id[tid], scale);
        const int kh = min(gm.rh, 4096) / 7 + 2, kw = min(gm.rw, 4096) / 7 + 2;
        hd->key[tid] = (unsigned short)min(kh * kw, 65535);
    }
    __syncthreads();
    if (tid < ns) {
        const unsigned int my = hd->key[tid];
        int rank = 0;
        for (int j = 0; j < ns; ++j) {
            const unsigned int kj = hd->key[j];
            rank += (kj > my || (kj == my && j < tid)) ? 1 : 0;
        }
        hd->id2[rank] = hd->id[tid];
    }
    __syncthreads();
    if (tid < ns) hd->id[tid] = hd->id2[tid];
    __syncthreads();
}

__device__ __forceinline__ AlignRec align_rec(float v, int size) {
    AlignRec r;
    if (v < -1.0f || v > (float)size) {
        r.lo = -1; r.hi = -1; r.l = 0.f; r.h = 0.f;
        return r;
    }
    if (v <= 0.f) v = 0.f;
    int lo = (int)v, hi;
    if (lo >= size - 1) { hi = lo = size - 1; v = (float)lo; } else { hi = lo + 1; }
    r.lo = lo; r.hi = hi;
    r.l = __fsub_rn(v, (float)lo);
    r.h = __fsub_rn(1.f, r.l);
    return r;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// Shared-memory feature layout: px[p][CB] -- the CB channels of pixel p are contiguous (CB/4 float4 chunks); chunk k of
// pixel p is stored at chunk slot (k + p) % NCH so that lanes reading neighbouring pixels hit different bank groups.
// A quarter-warp (8 lanes x 16 bytes) is conflict-free when its 8 chunks fall into 8 different 4-bank groups; the group
// of (p, k) is ((p * NCH + slot) mod 8), so the rotation must depend on p / (8 / NCH): then pixels that differ mod 8 never
// collide (with the rotation (k + p) pixels that agree mod 4 always collided: 8 lanes into 4 groups).
// Element index of chunk k of pixel p in the staged array, two forms.  kPlanar: chunk-major ([chunk][pixel] of 16-byte
// elements): RoIPool's lanes (neighbouring bins) read pixels 2-3 apart, i.e. elements 2-3 apart -> mostly different bank
// groups (247 vs 260 us on RPN rois).  Pixel-major ([pixel][chunk], chunks rotated, below): RoIAlign's four taps per sample
// are neighbouring pixels, and both chunks of a pixel share a 32-byte segment (305 vs 330 us).
template <int CB, bool kPlanar>
__device__ __forceinline__ size_t chunk_at(int p, int k, int HW);
template <int CB>
__device__ __forceinline__ int chunk_slot(int p, int k) {
    constexpr int NCH = CB / 4;
    constexpr int SH = NCH >= 8 ? 0 : NCH == 4 ? 1 : NCH == 2 ? 2 : 3;
    return (k + (p >> SH)) & (NCH - 1);
}

template <int CB, bool kPlanar>
__device__ __forceinline__ size_t chunk_at(int p, int k, int HW) {
    return kPlanar ? (size_t)k * HW + p : (size_t)p * (CB / 4) + chunk_slot<CB>(p, k);
}

// NCHW: consecutive threads read consecutive pixels of 4 planes (coalesced), 2 trips (8 loads) in flight; channels_last:
// consecutive threads read consecutive 16-byte channel chunks of a pixel, 4 trips in flight.  No runtime divisions.
template <int CB, bool kPlanar>
__device__ __forceinline__ void load_pixels(float4* px, const float* __restrict__ feat, int b, int c0, int C, int HW,
                                            bool nhwc) {
    constexpr int NCH = CB / 4;
    const int nt = blockDim.x;
    if (!nhwc) {
#pragma unroll 1
        for (int k = 0; k < NCH; ++k) {
            const int c = c0 + 4 * k;
            const float* src = feat + ((size_t)b * C + c) * HW;
            const bool h0 = c + 0 < C, h1 = c + 1 < C, h2 = c + 2 < C, h3 = c + 3 < C;
            for (int p0 = threadIdx.x; p0 < HW; p0 += 2 * nt) {
                float4 v[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int p = p0 + u * nt;
                    v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p < HW) {
                        if (h0) v[u].x = __ldg(src + p);
                        if (h1) v[u].y = __ldg(src + HW + p);
                        if (h2) v[u].z = __ldg(src + 2 * (size_t)HW + p);
                        if (h3) v[u].w = __ldg(src + 3 * (size_t)HW + p);
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int p = p0 + u * nt;
                    if (p < HW) px[chunk_at<CB, kPlanar>(p, k, HW)] = v[u];
                }
            }
        }
    } else {
        const int n = NCH * HW;
        const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(feat) & 15u) == 0);
        for (int i0 = threadIdx.x; i0 < n; i0 += 4 * nt) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * nt;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (i < n) {
                    const int p = i / NCH, k = i - p * NCH;  // NCH is a compile-time power of two
                    const int c = c0 + 4 * k;
                    const float* src = feat + ((size_t)b * HW + p) * C + c;
                    if (vec && c + 3 < C) {
                        v[u] = __ldg(reinterpret_cast<const float4*>(src));
                    } else {
                        if (c + 0 < C) v[u].x = __ldg(src);
                        if (c + 1 < C) v[u].y = __ldg(src + 1);
                        if (c + 2 < C) v[u].z = __ldg(src + 2);
                        if (c + 3 < C) v[u].w = __ldg(src + 3);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * nt;
                if (i < n) {
                    const int p = i / NCH, k = i - p * NCH;
                    px[chunk_at<CB, kPlanar>(p, k, HW)] = v[u];
                }
            }
        }
    }
    __syncthreads();
}

// RoIAlign forward (R4): 441 threads = 9 rois x 49 bins per pass, results staged as [roi][channel][49] tiles.
template <int CB>
__global__ void __launch_bounds__(kFastFwdThreads, (CB <= 8) ? 2 : 1)
    roi_align_fwd_fast_kernel(const float* __restrict__ feat, const float* __restrict__ rois, int K, int C, int H, int W,
                              int RP, float scale, int aligned, int nhwc, float* __restrict__ out) {
    constexpr int NCH = CB / 4;               // float4 chunks per pixel
    constexpr int RS = kFastFwdThreads / 49;  // rois worked on at the same time (9)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FastHdr* hd = reinterpret_cast<FastHdr*>(smem_raw);
    AlignRec* geo = reinterpret_cast<AlignRec*>(smem_raw + kHdrBytes);  // [RP][28] 1-D sample records
    const int stage = RP * CB * 49;                                     // values in the staging tile: [roi][channel][49]
    float* s_out = reinterpret_cast<float*>(smem_raw + kHdrBytes + ((RP * 28 * 16 + 127) & ~127));
    float4* px = reinterpret_cast<float4*>(s_out + stage);

    const int tid = threadIdx.x;
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int HW = H * W;
    const int cb = min(CB, C - c0);
    const bool prof = (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0);
    long long t0_ = clock64();
    load_pixels<CB, false>(px, feat, b, c0, C, HW, nhwc != 0);
    ROI_TICK(0);

    // thread -> (roi slot rs, bin): the 49 bins of a roi sit in consecutive lanes
    const int rs = tid / 49;
    const int bin = tid - rs * 49;
    const int ph = bin / 7, pw = bin - ph * 7;
    const bool worker = rs < RS;
    // vector copy-out needs 16-byte aligned runs of cb*49 values
    const bool vec_ok = ((cb * 196) % 16 == 0) && (((size_t)C * 196) % 16 == 0) && (((size_t)c0 * 196) % 16 == 0) &&
                        ((reinterpret_cast<uintptr_t>(out) & 15u) == 0);

    for (int tile = 0; tile < K; tile += kFastFwdThreads) {
        const int ns = stage_ids(rois, K, tile, b, hd);
        ROI_TICK(1);
        for (int p0 = 0; p0 < ns; p0 += RP) {
            const int nr = min(RP, ns - p0);
            // ---- 14 y-sample and 14 x-sample records per roi, once per roi ---------------------------------
            for (int t = tid; t < nr * 28; t += kFastFwdThreads) {
                const int s = t / 28, j = t - s * 28;
                const AlignGeom gm = align_geom(rois + 5 * (size_t)hd->id[p0 + s], scale, 7, 7, 2, aligned != 0);
                geo[t] = (j < 14) ? align_rec(sample_y(gm, j >> 1, j & 1), H)
                                  : align_rec(sample_x(gm, (j - 14) >> 1, (j - 14) & 1), W);
            }
            __syncthreads();
            ROI_TICK(2);
            if (worker) {
#pragma unroll 1
                for (int s = rs; s < nr; s += RS) {
                    float* so = s_out + s * CB * 49 + bin;
                    const AlignRec* rec = geo + s * 28;
                    float acc[CB];
#pragma unroll
                    for (int c = 0; c < CB; ++c) acc[c] = 0.f;
#pragma unroll 1
                    for (int s4 = 0; s4 < 4; ++s4) {
                        const AlignRec yy = rec[2 * ph + (s4 >> 1)];
                        const AlignRec xx = rec[14 + 2 * pw + (s4 & 1)];
                        if (yy.lo >= 0 && xx.lo >= 0) {
                            const float w1 = __fmul_rn(yy.h, xx.h), w2 = __fmul_rn(yy.h, xx.l);
                            const float w3 = __fmul_rn(yy.l, xx.h), w4 = __fmul_rn(yy.l, xx.l);
                            const int i1 = yy.lo * W + xx.lo, i2 = yy.lo * W + xx.hi;
                            const int i3 = yy.hi * W + xx.lo, i4 = yy.hi * W + xx.hi;
#pragma unroll
                            for (int k = 0; k < NCH; ++k) {
                                const float4 v1 = px[chunk_at<CB, false>(i1, k, HW)];
                                const float4 v2 = px[chunk_at<CB, false>(i2, k, HW)];
                                const float4 v3 = px[chunk_at<CB, false>(i3, k, HW)];
                                const float4 v4 = px[chunk_at<CB, false>(i4, k, HW)];
#define FRR_BIL(e, c)                                                                                                   \
    acc[4 * k + e] = __fadd_rn(acc[4 * k + e],                                                                          \
                               __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, v1.c), __fmul_rn(w2, v2.c)), __fmul_rn(w3, v3.c)), \
                                         __fmul_rn(w4, v4.c)))
                                FRR_BIL(0, x); FRR_BIL(1, y); FRR_BIL(2, z); FRR_BIL(3, w);
#undef FRR_BIL
                            }
                        }
                    }
#pragma unroll
                    for (int c = 0; c < CB; ++c) so[c * 49] = __fdiv_rn(acc[c], 4.0f);
                }
            }
            __syncthreads();
            ROI_TICK(3);
            // ---- copy-out: the cb*49 values of a roi are contiguous in the output -> coalesced 16-byte stores;
            //      warp w takes rois w, w + 14, ...: no index divisions
            {
                const int warp = tid >> 5, lane = tid & 31;
                for (int s = warp; s < nr; s += kFastFwdThreads / 32) {
                    const size_t o = ((size_t)hd->id[p0 + s] * C + c0) * 49;
                    if (vec_ok) {
                        const float4* so4 = reinterpret_cast<const float4*>(s_out + s * CB * 49);
                        for (int e = lane; e < cb * 49 / 4; e += 32) st_stream(reinterpret_cast<float4*>(out + o) + e, so4[e]);
                    } else {
                        for (int e = lane; e < cb * 49; e += 32) out[o + e] = s_out[s * CB * 49 + e];
                    }
                }
            }
            __syncthreads();  // the staging tile and the sample records are rewritten next
            ROI_TICK(4);
        }
    }
    ROI_TICK(5);
}

// NCHW planes -> the planar staging layout ([chunk][pixel] of float4 = 4 channels) with 4-byte cp.async: no registers
// between the load and the shared-memory write, so ALL of a thread's ~40 words are in flight at once (the register
// version above pays six dependent load round trips, ~10 K cycles per CTA) and the roi scan / ordering / bin geometry
// of the CTA run while they land.  Channels past C are zero-filled.  The caller waits (cp_async_wait_all) before the
// barrier that precedes the first read.
__device__ __forceinline__ void cp_async4_zfill(uint32_t dst, const void* src, bool ok) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(ok ? 4 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int CB>
__device__ __forceinline__ void load_planes_async(float4* px, const float* __restrict__ feat, int b, int c0, int C, int HW) {
    const uint32_t base = smem_u32(px);
#pragma unroll
    for (int ce = 0; ce < CB; ++ce) {
        const int c = c0 + ce;
        const bool ok = c < C;
        const float* src = feat + ((size_t)b * C + (ok ? c : c0)) * HW;
        const uint32_t dst = base + (uint32_t)(((ce >> 2) * HW) * 16 + (ce & 3) * 4);
        for (int p = threadIdx.x; p < HW; p += blockDim.x) cp_async4_zfill(dst + (uint32_t)p * 16u, src + p, ok);
    }
    cp_async_commit_group();
}

// ---------------------------------------------------------------------------------------------
// RoIPool forward without per-pass barriers (R1/R2)
// ---------------------------------------------------------------------------------------------
// The staged version above spends more issue slots waiting at its per-pass barriers (compute -> copy-out -> next 9
// rois) than in any other stall (ncu: 3.7 of 12 stall cycles per issued instruction).  Here the WARPS of a CTA take
// 32-bin slices of the flattened (roi, bin) sequence of the image's rois (ordered by window size), from a shared counter
// or as fixed shares: every lane always has a bin (49 bins per roi do not leave 15 of 64 lanes idle), neighbouring lanes work on the same
// or a similarly sized roi, and the only barriers left are the ones around the per-image roi list.  Results are stored directly: the lanes of a warp hold consecutive
// bins of one (roi, channel) row, i.e. consecutive addresses of the [K,C,7,7] output -- no staging tile, which also
// frees ~28 KB of shared memory per CTA.
constexpr int kFlatThreads = 448;
constexpr int kFlatGeoCap = 252;  // rois whose bin boundaries are held at once (56 bytes each)

template <int CB, bool kArg>
__global__ void __launch_bounds__(kFlatThreads, (CB <= 8) ? 2 : 1)
    roi_pool_fwd_flat_kernel(const float* __restrict__ feat, const float* __restrict__ rois, int K, int C, int H, int W,
                             float scale, int nhwc, float* __restrict__ out, int32_t* __restrict__ argmax) {
    constexpr int NCH = CB / 4;
    constexpr int kWarps = kFlatThreads / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FastHdr* hd = reinterpret_cast<FastHdr*>(smem_raw);
    short* geo = reinterpret_cast<short*>(smem_raw + kHdrBytes);  // [kFlatGeoCap][28]: hs[7] he[7] ws[7] we[7]
    float4* px = reinterpret_cast<float4*>(smem_raw + kHdrBytes + ((kFlatGeoCap * 56 + 127) & ~127));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int HW = H * W;
    const int cb = min(CB, C - c0);
    const bool prof = (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0);
    long long t0_ = clock64();
    if (nhwc)
        load_pixels<CB, true>(px, feat, b, c0, C, HW, true);
    else
        load_planes_async<CB>(px, feat, b, c0, C, HW);  // lands behind the roi scan and the bin geometry
    ROI_TICK(0);

    constexpr int kScanPer = 6;  // 448 x 6 = 2688 rois per scan round
    for (int k0 = 0; k0 < K; k0 += kScanPer * kFlatThreads) {
    unsigned int match_bits;
    int match_pos;
    const int nmatch = ids_scan<kScanPer>(rois, K, k0, b, hd, &match_bits, &match_pos);
    for (int r0 = 0; r0 < nmatch; r0 += kFlatThreads) {  // block-uniform trip count
        int ns = min(kFlatThreads, nmatch - r0);
        ids_emit<kScanPer>(k0, match_bits, match_pos, r0, kFlatThreads, hd);
        if (ns > kWarps) order_ids_by_window(rois, scale, ns, hd);
        if (gridDim.z > 1) {
            // thin grids (one image): the rois of the image are dealt to gridDim.z CTAs that hold the same planes, every
            // gridDim.z-th entry of the list ordered by window size each
            const int nz = gridDim.z, z = blockIdx.z;
            const int mine = (ns - z + nz - 1) / nz;
            const int v = (tid < mine) ? hd->id[tid * nz + z] : 0;
            __syncthreads();
            if (tid < mine) hd->id[tid] = v;
            __syncthreads();
            ns = mine;
            if (ns <= 0) continue;  // block-uniform
        }
        ROI_TICK(1);
        for (int g0 = 0; g0 < ns; g0 += kFlatGeoCap) {
            const int ng = min(kFlatGeoCap, ns - g0);
            // one thread per (roi, dimension): the rounded roi once, then the 7 window starts and 7 window ends
            for (int t = tid; t < ng * 2; t += kFlatThreads) {
                const int s = t >> 1, isw = t & 1;
                const PoolGeom gm = pool_geom(rois + 5 * (size_t)hd->id[g0 + s], scale);
                const int len = isw ? gm.rw : gm.rh, start = isw ? gm.sw : gm.sh, lim = isw ? W : H;
                const float bsz = __fdiv_rn((float)len, 7.0f);
                short* o = geo + s * 28 + isw * 14;
#pragma unroll
                for (int p = 0; p < 7; ++p) {
                    const int lo = (int)floorf(__fmul_rn((float)p, bsz)) + start;
                    const int hi = (int)ceilf(__fmul_rn((float)(p + 1), bsz)) + start;
                    o[p] = (short)min(max(lo, 0), lim);
                    o[7 + p] = (short)min(max(hi, 0), lim);
                }
            }
            if (tid == 0) hd->cnt[15] = 0;  // slice counter of this group
            cp_async_wait_all();    // this thread's share of the planes (first group only; nothing pending afterwards)
            __syncthreads();
            ROI_TICK(2);
            // With argmax (training): the (roi, bin) sequence of the group -- rois in descending window size -- is cut into
            // slices of 32 consecutive bins and the warps take the next slice from a shared counter as they finish (largest
            // first: the warps of a CTA end within one small slice of each other; fixed shares of ~9 rois per warp left them
            // 12 % and more apart: 176 -> 145 us, 226 -> 216 us at 128 rois per image, no change at 300).  The counter is
            // read one slice ahead, so the shared-memory atomic of the NEXT slice is in flight during the body.
            // Without argmax (inference) the body is a third shorter and the counter costs more than the balance gains
            // (109 -> 113 us, 181 -> 190 us): every warp walks a fixed share instead, one roi of each group of 14
            // consecutive ranks in boustrophedon order (rank 14 g + warp for even g, 14 g + 13 - warp for odd g).
            // Either way the lanes of a trip hold bins of one roi or of two rois of similar window size.
            constexpr bool kDealt = kArg;
            const int total = kDealt ? ng * 49 : ((ng + kWarps - 1) / kWarps) * 49;
            int ahead = 0, trip = 0;
            if (kDealt) {
                if (lane == 0) ahead = atomicAdd(&hd->cnt[15], 1);
                trip = __shfl_sync(0xffffffffu, ahead, 0);
            }
#pragma unroll 1
            for (; trip * 32 < total; trip = kDealt ? __shfl_sync(0xffffffffu, ahead, 0) : trip + 1) {
                if (kDealt && lane == 0) ahead = atomicAdd(&hd->cnt[15], 1);
                const int f = trip * 32 + lane;
                const int li = f / 49, bin = f - li * 49;
                const int s = kDealt ? li : li * kWarps + ((li & 1) ? kWarps - 1 - warp : warp);
                if (f >= total || s >= ng) continue;  // last, partial trip / group
                const int ph = bin / 7, pw = bin - ph * 7;
                const short* bnd = geo + s * 28;
                const int hs = bnd[ph], he = bnd[7 + ph], ws = bnd[14 + pw], we = bnd[21 + pw];
                const float init = ((he <= hs) || (we <= ws)) ? 0.f : -FLT_MAX;
                float best[CB];
                int bidx[CB];
#pragma unroll
                for (int c = 0; c < CB; ++c) { best[c] = init; bidx[c] = -1; }
#pragma unroll 1
                for (int h = hs; h < he; ++h) {
                    const int end = h * W + we;
                    // two pixels per trip: four 16-byte reads in flight before the first compare (the loop is bound by the
                    // latency of its shared-memory reads, not by an execution pipe); an odd tail pixel is fed as -FLT_MAX,
                    // which never passes the strict compare
#pragma unroll 1
                    for (int idx = h * W + ws; idx < end; idx += 2) {
                        const bool two = idx + 1 < end;
                        float4 va[NCH], vb[NCH];
#pragma unroll
                        for (int k = 0; k < NCH; ++k) {
                            va[k] = px[chunk_at<CB, true>(idx, k, HW)];
                            vb[k] = make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX);
                            if (two) vb[k] = px[chunk_at<CB, true>(idx + 1, k, HW)];
                        }
#pragma unroll
                        for (int k = 0; k < NCH; ++k) {
                            if (kArg) {
                                // first strict maximum in scan order (torchvision).  Compare + index select on the ALU
                                // pipe, the conditional move of the maximum as a predicated FFMA (x * 1 - 0, exact) on
                                // the FMA pipe
#define FRR_UPD(val, c, ix)                                                                                               \
    asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %2, %0;\n\t@p fma.rn.f32 %0, %2, 0f3F800000, 0f80000000;\n\tselp.b32 %1, %3, %1, p;\n\t}" \
        : "+f"(best[c]), "+r"(bidx[c])                                                                                     \
        : "f"(val), "r"(ix))
                                FRR_UPD(va[k].x, 4 * k + 0, idx); FRR_UPD(va[k].y, 4 * k + 1, idx);
                                FRR_UPD(va[k].z, 4 * k + 2, idx); FRR_UPD(va[k].w, 4 * k + 3, idx);
                                FRR_UPD(vb[k].x, 4 * k + 0, idx + 1); FRR_UPD(vb[k].y, 4 * k + 1, idx + 1);
                                FRR_UPD(vb[k].z, 4 * k + 2, idx + 1); FRR_UPD(vb[k].w, 4 * k + 3, idx + 1);
#undef FRR_UPD
                            } else {
                                // fmaxf orders -0.0 below +0.0: a window whose maximum is zero and that holds both
                                // signs stores +0.0 where torchvision (first strict maximum) may store -0.0 -- the only
                                // difference from the argmax path.  A strict compare here (setp + predicated move)
                                // costs 10 % of the inference workload on a B200 (27.7k -> 25.0k images/s)
                                best[4 * k + 0] = fmaxf(best[4 * k + 0], fmaxf(va[k].x, vb[k].x));
                                best[4 * k + 1] = fmaxf(best[4 * k + 1], fmaxf(va[k].y, vb[k].y));
                                best[4 * k + 2] = fmaxf(best[4 * k + 2], fmaxf(va[k].z, vb[k].z));
                                best[4 * k + 3] = fmaxf(best[4 * k + 3], fmaxf(va[k].w, vb[k].w));
                            }
                        }
                    }
                }
                // lanes = consecutive bins of a (roi, channel) row = consecutive addresses; write-once -> streaming stores
                const size_t o = ((size_t)hd->id[g0 + s] * C + c0) * 49 + bin;
#pragma unroll
                for (int c = 0; c < CB; ++c)
                    if (c < cb) __stcs(out + o + c * 49, best[c]);
                if (kArg) {
#pragma unroll
                    for (int c = 0; c < CB; ++c)
                        if (c < cb) __stcs(argmax + o + c * 49, bidx[c]);
                }
            }
            ROI_TICK(3);
            __syncthreads();  // the boundaries (and, after the last group, the id list) are rewritten next
            ROI_TICK(4);
        }
    }
    }
    cp_async_wait_all();  // (a CTA without rois leaves with nothing in flight)
    ROI_TICK(5);
}

// ---------------------------------------------------------------------------------------------
// RoIAlign backward (sampling_ratio = 2)
// ---------------------------------------------------------------------------------------------
// The bilinear weights are separable and channel independent.  Per roi the CTA builds, once, the 14 y-sample records
// and the dense 7 x Wt matrix Ax[pw][w] = total x-weight of bin column pw on pixel column w; then every warp (= one
// channel plane, owned exclusively) computes for ITS channel
//     T[ph][w]      = sum_pw grad_out[ph][pw] * Ax[pw][w]              (lanes = pixel columns, <= 3 bins per column)
//     plane[y][w]  += 0.25 * wy * T[ph(s)][w]   for the 2 taps (y, wy) of each of the 14 y samples
// Lanes own distinct columns and the samples are walked in order, so the adds are plain LDS / FFMA / STS: no atomics,
// no tickets.  torchvision scatters 16 atomicAdd per output element instead (822 M atomics at the config-3 shape).
constexpr int kAbRois = 8;    // rois per geometry group
constexpr int kAbCols = 128;  // widest feature map of the fast path (a roi touches at most W pixel columns)

struct AlignBwdGeo {
    AlignRec y[14];
    AlignRec x[14];
    float ax[7][kAbCols];
    unsigned char pw_lo[kAbCols];
    int x0, wt, span, pad;
};

template <int CB>
__global__ void __launch_bounds__(CB * 32, 1)
    roi_align_bwd_fast_kernel(const float* __restrict__ grad_out, const float* __restrict__ rois, int K, int C, int H,
                              int W, float scale, int aligned, int nhwc, float* __restrict__ grad_in) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FastHdr* hd = reinterpret_cast<FastHdr*>(smem_raw);
    AlignBwdGeo* geo = reinterpret_cast<AlignBwdGeo*>(smem_raw + kHdrBytes);                 // [kAbRois]
    float* sgo = reinterpret_cast<float*>(geo + kAbRois);                                     // [CB][64]
    float* planes = sgo + CB * 64;
    const int HW = H * W;

    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;  // warp c owns plane c
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int cb = min(CB, C - c0);
    for (int i = tid; i < CB * HW; i += CB * 32) planes[i] = 0.f;
    float* pl = planes + (size_t)c * HW;
    float* mygo = sgo + c * 64;
    const size_t chan = (size_t)(c0 + c) * 49;
    if (tid < kAbRois) geo[tid].span = 0;
    __syncthreads();

    for (int tile = 0; tile < K; tile += CB * 32) {
        const int ns = stage_ids(rois, K, tile, b, hd);
        for (int r0 = 0; r0 < ns; r0 += kAbRois) {
            const int nr = min(kAbRois, ns - r0);
            // ---- geometry of the group, built once for all channels -----------------------------------
            // (a) sample records: thread (roi, j < 28)
            for (int t = tid; t < nr * 28; t += CB * 32) {
                const int s = t / 28, j = t - s * 28;
                const AlignGeom gm = align_geom(rois + 5 * (size_t)hd->id[r0 + s], scale, 7, 7, 2, aligned != 0);
                if (j < 14) geo[s].y[j] = align_rec(sample_y(gm, j >> 1, j & 1), H);
                else geo[s].x[j - 14] = align_rec(sample_x(gm, (j - 14) >> 1, (j - 14) & 1), W);
            }
            __syncthreads();
            // (b) column extent of every roi
            if (tid < nr) {
                int lo = W, hi = -1;
                for (int j = 0; j < 14; ++j) {
                    const AlignRec r = geo[tid].x[j];
                    if (r.lo >= 0) { lo = min(lo, r.lo); hi = max(hi, r.hi); }
                }
                geo[tid].x0 = lo;
                geo[tid].wt = hi >= lo ? hi - lo + 1 : 0;
            }
            __syncthreads();
            // (c) Ax[pw][w] and the first bin column of every pixel column
            for (int t = tid; t < nr * kAbCols; t += CB * 32) {
                const int s = t / kAbCols, w = t - s * kAbCols;
                const int col = geo[s].x0 + w;
                int first = 7, last = -1;
#pragma unroll
                for (int pw = 0; pw < 7; ++pw) {
                    float a = 0.f;
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const AlignRec r = geo[s].x[2 * pw + i];
                        if (r.lo >= 0) {
                            if (r.lo == col) a = __fadd_rn(a, r.h);
                            if (r.hi == col) a = __fadd_rn(a, r.l);
                        }
                    }
                    geo[s].ax[pw][w] = a;
                    if (a != 0.f) { first = min(first, pw); last = pw; }
                }
                geo[s].pw_lo[w] = (unsigned char)(first == 7 ? 0 : first);
                if (w < geo[s].wt && last >= first) atomicMax(&geo[s].span, last - first + 1);
            }
            __syncthreads();

            if (c < cb) {
                for (int s = 0; s < nr; ++s) {
                    const AlignBwdGeo& gg = geo[s];
                    // stage this channel's 49 output gradients (coalesced) for broadcast reads
                    const size_t base = (size_t)hd->id[r0 + s] * C * 49 + chan;
                    mygo[lane] = __ldg(grad_out + base + lane);
                    if (lane + 32 < 49) mygo[lane + 32] = __ldg(grad_out + base + lane + 32);
                    __syncwarp();
                    const int span = gg.span;
                    for (int w0 = 0; w0 < gg.wt; w0 += 32) {
                        const int w = w0 + lane;
                        const bool on = w < gg.wt;
                        float T[7];
#pragma unroll
                        for (int ph = 0; ph < 7; ++ph) T[ph] = 0.f;
                        const int plo = on ? (int)gg.pw_lo[w] : 0;
                        for (int i = 0; i < span; ++i) {
                            const int pw = min(plo + i, 6);
                            const float a = (on && plo + i < 7) ? gg.ax[pw][w] : 0.f;
#pragma unroll
                            for (int ph = 0; ph < 7; ++ph) T[ph] = __fmaf_rn(a, mygo[ph * 7 + pw], T[ph]);
                        }
                        float* colp = pl + gg.x0 + w;
#pragma unroll
                        for (int sy = 0; sy < 14; ++sy) {
                            const AlignRec yr = gg.y[sy];
                            if (on && yr.lo >= 0) {
                                const float t = __fmul_rn(0.25f, T[sy >> 1]);
                                float* p0 = colp + yr.lo * W;
                                *p0 = __fmaf_rn(yr.h, t, *p0);
                                float* p1 = colp + yr.hi * W;
                                *p1 = __fmaf_rn(yr.l, t, *p1);
                            }
                        }
                    }
                    __syncwarp();
                }
            }
            __syncthreads();  // geometry is rewritten by the next group
            if (tid < kAbRois) geo[tid].span = 0;
        }
        __syncthreads();  // ids are rewritten by the next tile
    }
    store_planes(planes, grad_in, b, c0, cb, C, HW, nhwc != 0);
}

// ---------------------------------------------------------------------------------------------
// host side: 0 = launched, 1 = shape outside the fast path (caller falls back), < 0 = error
// ---------------------------------------------------------------------------------------------
static const size_t kSmemLimit = 227 * 1024;

// RoIAlign: rois per pass for a shared-memory budget: as many as fit beside the pixels, a multiple of 9 (9 rois are
// worked on at the same time: 448 threads / 49 bins), capped; 0 = no fit
static int align_fwd_rp(int CB, int HW, size_t budget) {
    const size_t fixed = kHdrBytes + 128 + (size_t)CB * HW * 4;
    if (fixed >= budget) return 0;
    const size_t per_roi = (size_t)CB * 49 * 4 + 28 * 16;
    int rp = (int)((budget - fixed) / per_roi);
    if (rp > 36) rp = 36;
    return rp / 9 * 9;
}
static size_t align_fwd_smem(int CB, int HW, int rp) {
    return kHdrBytes + (((size_t)rp * 28 * 16 + 127) & ~(size_t)127) + (size_t)rp * CB * 49 * 4 + (size_t)CB * HW * 4;
}
// CB <= 8 kernels are built for two CTAs per SM (28 warps hide the shared-memory latency of the window loops)
static size_t fwd_budget(int CB) { return CB <= 8 ? (kSmemLimit - 2048) / 2 : kSmemLimit; }

template <int CB>
static int launch_align_fwd(const RoiPick& pk, const float* feat, const float* rois, int K, int B, int C, int H, int W,
                            float scale, int aligned, int nhwc, float* out, cudaStream_t st) {
    auto kern = roi_align_fwd_fast_kernel<CB>;
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    kern<<<dim3((C + CB - 1) / CB, B), kFastFwdThreads, pk.smem, st>>>(feat, rois, K, C, H, W, pk.rp, scale, aligned, nhwc,
                                                                        out);
    return FRR_OK;
}

static size_t flat_smem(int CB, int HW) {
    return kHdrBytes + ((kFlatGeoCap * 56 + 127) & ~(size_t)127) + (size_t)CB * HW * 4;
}
template <bool kArg, int CB>
static int launch_flat(const RoiPick& pk, const float* feat, const float* rois, int K, int B, int C, int H, int W, float scale,
                       int nhwc, float* out, int32_t* argmax, cudaStream_t st) {
    auto kern = roi_pool_fwd_flat_kernel<CB, kArg>;
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    kern<<<dim3((C + CB - 1) / CB, B, pk.nz), kFlatThreads, pk.smem, st>>>(feat, rois, K, C, H, W, scale, nhwc, out, argmax);
    return FRR_OK;
}

// 7x7 forward fast paths: false = shape outside them (the caller takes the generic kernels)
bool roi_fwd_fast_pick(bool align, int B, int C, int H, int W, int PH, int PW, int sampling, RoiPick* pk) {
    if (PH != 7 || PW != 7 || (align && sampling != 2) || H > 32767 || W > 32767) return false;
    const int HW = H * W;
    if (!align) {
        // CB = 8 (else 4) when two CTAs fit an SM, else 8 or 4 at one CTA per SM (16 planes would need HW <= 3326, where
        // 4 planes already fit twice)
        int cbk = 0;
        if (flat_smem(8, HW) <= fwd_budget(8)) cbk = 8;
        else if (flat_smem(4, HW) <= fwd_budget(4)) cbk = 4;
        // a single image (or a thin batch) with 8 channels per CTA leaves SMs without a CTA (1 x 512 / 8 = 64 CTAs on 148
        // SMs): 4 channels per CTA then
        if (cbk == 8 && (long)B * ((C + 7) / 8) < (long)num_sms()) cbk = 4;
        for (int t = 8; t >= 4 && cbk == 0; t >>= 1)
            if (flat_smem(t, HW) <= kSmemLimit) cbk = t;
        if (cbk == 0) return false;
        // fewer CTAs than resident slots (two per SM): split the rois of an image over 2 or 4 CTAs with the same planes
        const long ctas = (long)B * ((C + cbk - 1) / cbk), slots = 2L * num_sms();
        const int nz = ctas * 4 <= slots ? 4 : ctas * 2 <= slots ? 2 : 1;
        *pk = RoiPick{kPoolFwdFlat, cbk, nz, 0, flat_smem(cbk, HW)};
        return true;
    }
    // 8 (else 4) channels at two CTAs per SM, else at one (16 would need HW <= 3042, where 4 already fit twice)
    int cbk = 0, rp = 0;
    for (int t = 8; t >= 4 && cbk == 0; t >>= 1)
        if ((rp = align_fwd_rp(t, HW, fwd_budget(t))) > 0) cbk = t;
    for (int t = 8; t >= 4 && cbk == 0; t >>= 1)
        if ((rp = align_fwd_rp(t, HW, kSmemLimit)) > 0) cbk = t;
    if (cbk == 0) return false;
    *pk = RoiPick{kAlignFwdFast, cbk, 1, rp, align_fwd_smem(cbk, HW, rp)};
    return true;
}

int roi_fwd_fast_launch(const RoiPick& pk, const float* feat, const float* rois, int K, int B, int C, int H, int W,
                        float scale, int aligned, int nhwc, float* out, int32_t* argmax, frr_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (pk.kernel == kPoolFwdFlat) {
        const bool arg = argmax != nullptr;
#define FRR_FLAT(CBK)                                                                                   \
    (arg ? launch_flat<true, CBK>(pk, feat, rois, K, B, C, H, W, scale, nhwc, out, argmax, st)          \
         : launch_flat<false, CBK>(pk, feat, rois, K, B, C, H, W, scale, nhwc, out, argmax, st))
        rc = pk.cb == 8 ? FRR_FLAT(8) : FRR_FLAT(4);
#undef FRR_FLAT
        if (rc) return rc;
        count_launch();
        FRR_CHECK_LAUNCH("roi_pool_fwd_flat_kernel");
        return FRR_OK;
    }
    rc = pk.cb == 8 ? launch_align_fwd<8>(pk, feat, rois, K, B, C, H, W, scale, aligned, nhwc, out, st)
                    : launch_align_fwd<4>(pk, feat, rois, K, B, C, H, W, scale, aligned, nhwc, out, st);
    if (rc) return rc;
    count_launch();
    FRR_CHECK_LAUNCH("roi_align_fwd_fast_kernel");
    return FRR_OK;
}

static size_t align_bwd_smem(int CB, int HW) {
    return kHdrBytes + sizeof(AlignBwdGeo) * kAbRois + (size_t)CB * 64 * 4 + (size_t)CB * HW * 4;
}

template <int CB>
static int launch_align_bwd(const RoiPick& pk, const float* go, const float* rois, int K, int B, int C, int H, int W,
                            float scale, int aligned, int nhwc, float* gin, cudaStream_t st) {
    auto kern = roi_align_bwd_fast_kernel<CB>;
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    kern<<<dim3((C + CB - 1) / CB, B), CB * 32, pk.smem, st>>>(go, rois, K, C, H, W, scale, aligned, nhwc, gin);
    return FRR_OK;
}

// 7x7 RoIAlign backward (sampling_ratio 2): the separable plane kernel or the streaming atomic kernel (roi.cu);
// false = shape outside both (the caller takes the generic kernels)
bool roi_align_bwd_fast_pick(int B, int C, int H, int W, int PH, int PW, int sampling, RoiPick* pk) {
    // every roi may touch at most kAbCols pixel columns: guaranteed when the map is no wider than that
    if (PH != 7 || PW != 7 || sampling != 2 || W > kAbCols) return false;
    const int HW = H * W;
    int cbk = 0;
    for (int t = 16; t >= 4; t >>= 1) {
        if (align_bwd_smem(t, HW) > kSmemLimit) continue;
        cbk = t;
        if ((long)B * ((C + t - 1) / t) >= (long)num_sms()) break;
    }
    if (cbk == 0) return false;
    // when 16 planes do not fit (maps above ~3400 pixels: 50 x 83) this kernel is left with 8 warps per SM and is latency
    // bound (2.7 ms on the config-4 shape): the streaming atomic kernel instead (1.9-2.3 ms)
    if (align_bwd_smem(16, HW) > kSmemLimit) *pk = RoiPick{kAlignBwdStream, 0, 1, 0, 0};
    else *pk = RoiPick{kAlignBwdFast, cbk, 1, 0, align_bwd_smem(cbk, HW)};
    return true;
}

int roi_align_bwd_fast_launch(const RoiPick& pk, const float* grad_out, const float* rois, int K, int B, int C, int H, int W,
                              float scale, int aligned, int nhwc, float* grad_in, frr_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = pk.cb == 16 ? launch_align_bwd<16>(pk, grad_out, rois, K, B, C, H, W, scale, aligned, nhwc, grad_in, st)
                 : pk.cb == 8  ? launch_align_bwd<8>(pk, grad_out, rois, K, B, C, H, W, scale, aligned, nhwc, grad_in, st)
                               : launch_align_bwd<4>(pk, grad_out, rois, K, B, C, H, W, scale, aligned, nhwc, grad_in, st);
    if (rc) return rc;
    count_launch();
    FRR_CHECK_LAUNCH("roi_align_bwd_fast_kernel");
    return FRR_OK;
}

}  // namespace frr

// Developer hook: copies the 16 phase counters (cycles of CTA (0,0): forward 0 plane load, 1 roi scan, 2 geometry +
// buffer wait, 3 compute, 4 store issue, 5 drain; backward 8 zero, 9 roi scan, 10 accumulate, 11 tile syncs,
// 12 plane store) to the host and clears them.  Synchronises the device.
namespace frr { void pool_bwd_debug_fetch(long long* host_out8); }
extern "C" int frr_roi_debug_cycles(int64_t* host_out16) {
    FRR_CHECK_ARG(host_out16 != nullptr, "frr_roi_debug_cycles: null pointer");
    long long z[16] = {0};
    FRR_CUDA(cudaMemcpyFromSymbol(host_out16, frr::g_roi_dbg, sizeof(z)));
    FRR_CUDA(cudaMemcpyToSymbol(frr::g_roi_dbg, z, sizeof(z)));
    // slots 8-15 when the colour-class RoIPool backward ran (roi_pool_bwd.cu): 8 wait full, 9 ring loads + adds, 10 release,
    // 11 producer wait empty, 12 producer issue, 13 roi scan, 14 zero, 15 store
    long long pb[8];
    frr::pool_bwd_debug_fetch(pb);
    bool any = false;
    for (int i = 0; i < 8; ++i) any = any || pb[i] != 0;
    if (any)
        for (int i = 0; i < 8; ++i) host_out16[8 + i] = pb[i];
    return FRR_OK;
}
