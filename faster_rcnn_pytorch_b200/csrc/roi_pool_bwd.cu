// R3: RoIPool 7x7 backward, conflict-free by construction (autograd of models/model.py:113 <- train.py:36;
// torchvision::_roi_pool_backward: grad_in[b, c, argmax[k, c, bin]] += grad_out[k, c, bin] for argmax != -1).
//
// torchvision scatters one global atomic per output element (K*C*49 RED.ADD.F32, at the L2 atomic floor); shared-memory
// float atomics are a CAS loop on sm_100.  This kernel needs neither:
//
//   * a CTA keeps CB channel planes of one image in shared memory (zeroed once, written once with a TMA bulk store);
//     a WARP owns two planes exclusively (lanes = 2 planes x 16 bins), so no two warps ever touch the same word and
//     the warps never synchronise with each other while they accumulate;
//   * the bins of a roi are processed in four COLOUR classes (ph mod 2, pw mod 2).  For a roi of at least 6 feature
//     pixels per side the pooling windows of two bins that are two apart in a dimension are disjoint
//         floor((p + 2) * b) >= ceil((p + 1) * b)      (checked per roi with the forward's own fp32 arithmetic),
//     clipping to the map only shrinks windows, and an argmax lies inside its bin's window -- so within one colour
//     class all <= 16 argmax pixels of the plane are distinct and the adds are plain LDS / FADD / STS in a fixed
//     order (deterministic, unlike atomics);
//   * smaller rois (a side under 6 pixels: bin size < 1, windows two apart may coincide) would need s_h x s_w > 4 classes
//     (s = smallest stride with disjoint windows) -- more shared-memory steps than one global atomic per element costs
//     (measured: strided classes 313 us, MATCH.ANY merging 640-970 us, atomics 180-200 us on rois of 1-7 pixels).  The plane
//     kernel leaves them out and roi_pool_bwd_tail_kernel adds them afterwards: one CTA per roi streams the roi's C * 49
//     contiguous values, sums the gradients of consecutive lanes that hit the same (channel, pixel) in registers and issues
//     one RED.ADD.F32 per run onto the stored planes (faster than torchvision's kernel of the same atomics: coalesced
//     reads, no per-element index arithmetic, fewer atomics);
//   * every warp streams the grad_out / argmax rows of its two planes (2 x 98 contiguous words per roi) into its own
//     shared-memory ring with cp.async, kPbDepth rois ahead of the adds, each word to a class-major position so that
//     an adding lane fetches its four class values with one 16-byte read: HBM latency is covered without registers,
//     without a producer warp and without barriers.
//
// HBM traffic = the algorithmic bytes: grad_out + argmax read once, grad_in written once (no memset pass).
// The contract on argmax is torchvision's: it comes from the forward call on the same rois and map shape (an index
// outside [0, H*W) is ignored instead of written out of bounds).
#include <stddef.h>

#include "roi_common.cuh"

namespace frr {

constexpr int kPbDepth = 8;     // rois in flight per warp (ring slots)
constexpr int kPbSlotBytes = 1024;  // ring slot: [32 lanes][4 classes] argmax words, then the same for grad_out
constexpr int kPbIdCap = 512;    // input rois scanned per round

struct PoolBwdHdr {
    int cnt[32];
    int id[kPbIdCap];  // roi index (24 bits) | class stride in h << 24 | class stride in w << 27 (both 2 for every listed roi)
};
constexpr int kPbHdrBytes = (sizeof(PoolBwdHdr) + 127) & ~127;
constexpr int kPbIdMask = (1 << 24) - 1;

// Word position of (plane half, bin) inside the argmax block of a ring slot: the four colour-class values of RMW lane
// (half, i) are adjacent (one 16-byte read), i = index of the bin inside its class (rows of 4 for even pw, of 3 for odd)
__host__ __device__ constexpr int ring_pos(int half, int bin) {
    const int ph = bin / 7, pw = bin - ph * 7;
    const int q = (ph & 1) * 2 + (pw & 1);
    const int i = (ph >> 1) * ((pw & 1) ? 3 : 4) + (pw >> 1);
    return (half * 16 + i) * 4 + q;
}

// shared memory through 32-bit shared-window addresses (no generic -> shared conversion inside the loops); volatile +
// "memory": the read-modify-write steps of a warp stay in program order
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ int lds_s32(uint32_t a) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}

// Smallest s in 2..7 such that the (unclipped) windows of bins p and p + s never overlap: floor((p+s)*b) >= ceil((p+1)*b)
// for all p, evaluated with the forward's own fp32 arithmetic.  r >= 6 gives 2; 7 puts every bin of the dimension into
// its own class.
__device__ __forceinline__ int class_stride(int r) {
    if (r >= 7) return 2;
    const float bsz = __fdiv_rn((float)r, 7.0f);
    int lo[8], hi[7];
#pragma unroll
    for (int p = 0; p < 7; ++p) {
        lo[p] = (int)floorf(__fmul_rn((float)p, bsz));
        hi[p] = (int)ceilf(__fmul_rn((float)(p + 1), bsz));
    }
    int s = 2;
#pragma unroll
    for (int t = 2; t <= 6; ++t) {
        bool ok = true;
#pragma unroll
        for (int p = 0; p + t < 7; ++p) ok = ok && (lo[p + t] >= hi[p]);
        if (s == t && !ok) s = t + 1;
    }
    return s;
}

// rois that need more than the four (mod 2, mod 2) classes (a side below ~6 pixels) -> roi_pool_bwd_tail_kernel
__device__ __forceinline__ bool pb_small(int sh, int sw) { return sh * sw > 4; }

// block-wide exclusive prefix sum of one int per thread (blockDim a multiple of 32, <= 1024); *total = block sum
__device__ __forceinline__ int pb_block_scan(int v, int* warp_cnt, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();  // warp_cnt reuse
    if (lane == 31) warp_cnt[warp] = inc;
    __syncthreads();
    int pre = 0, tot = 0;
    for (int w = 0; w < nwarps; ++w) {
        const int c = warp_cnt[w];
        if (w < warp) pre += c;
        tot += c;
    }
    *total = tot;
    return pre + inc - v;
}

// One round of the roi scan over rois[k0, k0 + kPbIdCap): the rois of image b that take the shared-memory paths go to
// hd->id with their class strides (pb_small rois are left to roi_pool_bwd_tail_kernel).  The order of the list is a fixed function of the input (determinism of the sums).
// PER = kPbIdCap / blockDim.  Returns the length of hd->id.  Called by all threads.
template <int PER>
__device__ __forceinline__ int collect_rois(const float* __restrict__ rois, int K, int k0, int b, float scale, PoolBwdHdr* hd) {
    const int tid = threadIdx.x, nt = blockDim.x;
    // pass 1: batch indices of a contiguous run per thread (all loads in flight), compaction of the matching rois
    const int lo = k0 + tid * PER;
    float bi[PER];
#pragma unroll
    for (int j = 0; j < PER; ++j) bi[j] = __ldg(rois + 5 * (size_t)min(lo + j, K - 1));
    unsigned int mine = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j)
        if (lo + j < K && (int)bi[j] == b) mine |= 1u << j;
    int n = 0;
    int pos = pb_block_scan(__popc(mine), hd->cnt, &n);
    while (mine) {
        const int j = __ffs(mine) - 1;
        mine &= mine - 1u;
        hd->id[pos++] = lo + j;
    }
    __syncthreads();
    if (n == 0) return 0;  // block-uniform
    // pass 2: geometry of list entries tid, tid + blockDim, ... (balanced over the threads), split into the two lists
    int ent[PER];
    int nb = 0, ns = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int e = tid + j * nt;
        ent[j] = -1;
        if (e < n) {
            const int k = hd->id[e];
            const PoolGeom gm = pool_geom(rois + 5 * (size_t)k, scale);
            const int sh = class_stride(gm.rh), sw = class_stride(gm.rw);
            const bool small = pb_small(sh, sw);
            ent[j] = k | (sh << 24) | (sw << 27) | (small ? (1 << 30) : 0);
            nb += small ? 0 : 1;
            ns += small ? 1 : 0;
        }
    }
    int tot = 0;
    const int packed = pb_block_scan(nb | (ns << 16), hd->cnt, &tot);  // (its barriers: every entry of id has been read)
    int pb = packed & 0xffff;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        if (ent[j] < 0) continue;
        if (!(ent[j] & (1 << 30))) hd->id[pb++] = ent[j];
    }
    __syncthreads();
    return tot & 0xffff;
}

// One accumulate step of the colour path, split in two so that independent work can be placed between the load and the
// add (the warp stalls only at the first use of `t`): both halves are predicated on a valid pixel index, no branches.
__device__ __forceinline__ void rmw_load(float& t, int a, uint32_t hw, uint32_t addr) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p ld.shared.f32 %0, [%3];\n\t}" : "+f"(t) : "r"(a), "r"(hw), "r"(addr) : "memory");
}
__device__ __forceinline__ void rmw_store(float v, int a, uint32_t hw, uint32_t addr) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p st.shared.f32 [%3], %0;\n\t}" ::"f"(v), "r"(a), "r"(hw), "r"(addr) : "memory");
}

struct PbVals {  // the four colour-class values of one lane for one roi
    int a0, a1, a2, a3;
    float g0, g1, g2, g3;
    int entry;
};

template <int CB>
__global__ void __launch_bounds__(CB * 16)
    roi_pool_bwd_color_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                              const float* __restrict__ rois, int K, int C, int H, int W, float scale, int nhwc,
                              float* __restrict__ grad_in) {
    constexpr int kWarps = CB / 2;  // a warp owns two planes
    constexpr int D = kPbDepth;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PoolBwdHdr* hd = reinterpret_cast<PoolBwdHdr*>(smem_raw);
    int* ring = reinterpret_cast<int*>(smem_raw + kPbHdrBytes);  // [kWarps][D][256 words]
    float* planes = reinterpret_cast<float*>(smem_raw + kPbHdrBytes + kWarps * D * kPbSlotBytes);  // [CB][HW]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y, c0 = blockIdx.x * CB;
    const int HW = H * W;
    const int cb = min(CB, C - c0);

    {
        float4* p4 = reinterpret_cast<float4*>(planes);
        const int n4 = CB * HW / 4;
        for (int i = tid; i < n4; i += blockDim.x) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = n4 * 4 + tid; i < CB * HW; i += blockDim.x) planes[i] = 0.f;
        // argmax positions of bins that do not exist (classes with fewer than 16 bins) stay -1 for good
        for (int i = tid; i < kWarps * D * (kPbSlotBytes / 4); i += blockDim.x) ring[i] = -1;
    }

    // the shared-window base, converted once inside a volatile asm (the compiler would otherwise rematerialise the
    // conversion -- an S2R -- inside the loop)
    uint32_t sbase;
    {
        uint64_t t;
        asm volatile("cvta.to.shared.u64 %0, %1;" : "=l"(t) : "l"(smem_raw));
        sbase = (uint32_t)t;
    }
    const uint32_t id0 = sbase + (uint32_t)offsetof(PoolBwdHdr, id);
    const uint32_t ring0 = sbase + kPbHdrBytes + (uint32_t)warp * (D * kPbSlotBytes);
    const uint32_t planes0 = sbase + kPbHdrBytes + kWarps * D * kPbSlotBytes;
    const int half = lane >> 4;
    const int my_pl = 2 * warp + half;
    const bool pl_ok = my_pl < cb;
    const uint32_t pl0 = planes0 + (uint32_t)(pl_ok ? my_pl : 0) * (uint32_t)HW * 4u;
    const int npl = min(2, cb - 2 * warp);  // planes of this warp that exist (<= 0: idle warp)
    // copy roles: lane l moves words l, l + 32, l + 64, l + 96 of the 49 * npl contiguous words of a roi's row pair to
    // their class-major positions
    uint32_t dpos[4];
    bool cpy[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int w = lane + 32 * j;
        cpy[j] = w < 49 * npl;
        dpos[j] = ring0 + (cpy[j] ? 4u * (uint32_t)ring_pos(w / 49, w % 49) : 0u);
    }
    const int32_t* src_a = argmax + (size_t)(c0 + 2 * warp) * 49 + lane;
    const float* src_g = grad_out + (size_t)(c0 + 2 * warp) * 49 + lane;
    const uint32_t row_pitch = (uint32_t)C * 49u;  // words between consecutive rois
    const uint32_t myq = ring0 + 16u * (uint32_t)lane;  // this lane's 4 class values inside slot 0
    const uint32_t uHW = (uint32_t)HW;

    for (int k0 = 0; k0 < K; k0 += kPbIdCap) {
        // (the barriers of the scan also order the initialisation above)
        const int n = collect_rois<kPbIdCap / (CB * 16)>(rois, K, k0, b, scale, hd);
        if (npl > 0 && n > 0) {
            // copies of roi r into the ring slot at byte offset `so` (always commits a group; past the end of the list
            // nothing is read)
            auto issue = [&](int r, uint32_t so) {
                const uint32_t live = r < n ? 4u : 0u;
                const int idn = lds_s32(id0 + 4u * (uint32_t)min(r, n - 1)) & kPbIdMask;
                const size_t off = (size_t)(uint32_t)idn * row_pitch;
                const int32_t* sa = src_a + off;
                const float* sg = src_g + off;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (cpy[j]) {
                        cp_async4_zfill(dpos[j] + so, sa + 32 * j, live);
                        cp_async4_zfill(dpos[j] + so + 512u, sg + 32 * j, live);
                    }
                }
                cp_async_commit();
            };
            // this lane's class values of the roi in slot `so`; rois that take another path (or a missing plane) get -1
            auto fetch = [&](int r, uint32_t so, PbVals& v) {
                v.entry = lds_s32(id0 + 4u * (uint32_t)min(r, n - 1));
                asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.a0), "=r"(v.a1), "=r"(v.a2), "=r"(v.a3) : "r"(myq + so) : "memory");
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.g0), "=f"(v.g1), "=f"(v.g2), "=f"(v.g3) : "r"(myq + so + 512u) : "memory");
            };
            auto mask = [&](PbVals& v) {
                if (!pl_ok || ((v.entry >> 24) & 63) != (2 | (2 << 3))) v.a0 = v.a1 = v.a2 = v.a3 = -1;
            };
            // One roi: `cur` (already in registers) is accumulated while its ring slot is refilled with roi r + D and the
            // values of roi r + 1 are fetched into `nxt` -- three independent instruction streams, interleaved in source
            // order so that each one's shared-memory latency is covered by the other two.
            auto body = [&](int r, uint32_t so, uint32_t so_next, PbVals& cur, PbVals& nxt) {
                __syncwarp();  // every lane is done with slot `so`
                float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
                const uint32_t p0 = pl0 + 4u * (uint32_t)cur.a0, p1 = pl0 + 4u * (uint32_t)cur.a1;
                const uint32_t p2 = pl0 + 4u * (uint32_t)cur.a2, p3 = pl0 + 4u * (uint32_t)cur.a3;
                rmw_load(t0, cur.a0, uHW, p0);
                issue(r + D, so);
                rmw_store(__fadd_rn(t0, cur.g0), cur.a0, uHW, p0);
                rmw_load(t1, cur.a1, uHW, p1);
                cp_async_wait<D - 1>();  // this lane's copies of roi r + 1 have landed ...
                __syncwarp();            // ... and so have the other lanes'
                fetch(r + 1, so_next, nxt);
                rmw_store(__fadd_rn(t1, cur.g1), cur.a1, uHW, p1);
                rmw_load(t2, cur.a2, uHW, p2);
                mask(nxt);
                rmw_store(__fadd_rn(t2, cur.g2), cur.a2, uHW, p2);
                rmw_load(t3, cur.a3, uHW, p3);
                rmw_store(__fadd_rn(t3, cur.g3), cur.a3, uHW, p3);
            };
            for (int r = 0; r < D; ++r) issue(r, (uint32_t)r * kPbSlotBytes);
            cp_async_wait<D - 1>();
            __syncwarp();
            PbVals va, vb;
            fetch(0, 0u, va);
            mask(va);
            uint32_t so = 0;
#pragma unroll 1
            for (int r = 0; r < n; r += 2) {
                const uint32_t so1 = so + kPbSlotBytes == D * kPbSlotBytes ? 0u : so + kPbSlotBytes;
                body(r, so, so1, va, vb);
                if (r + 1 >= n) break;
                const uint32_t so2 = so1 + kPbSlotBytes == D * kPbSlotBytes ? 0u : so1 + kPbSlotBytes;
                body(r + 1, so1, so2, vb, va);
                so = so2;
            }
            cp_async_wait<0>();
        }
        __syncthreads();  // the id list is rewritten by the next round
    }
    store_planes(planes, grad_in, b, c0, cb, C, HW, nhwc != 0);
}

// The rois the plane kernel skipped (pb_small): one CTA per roi, which leaves at once unless the roi is small; a small
// roi streams its C * 49 contiguous grad_out / argmax values (8 independent elements per thread in flight) and adds
// them with RED.ADD.F32 onto the planes the first kernel has already written (stream order).
__global__ void __launch_bounds__(256)
    roi_pool_bwd_tail_kernel(const float* __restrict__ grad_out, const int32_t* __restrict__ argmax,
                             const float* __restrict__ rois, int B, int C, int H, int W, float scale, int nhwc, int all,
                             float* __restrict__ grad_in) {
    const int k = blockIdx.x;
    const float* r = rois + 5 * (size_t)k;
    const int b = (int)__ldg(r);
    if (b < 0 || b >= B) return;
    if (!all) {
        const PoolGeom gm = pool_geom(r, scale);
        if (!pb_small(class_stride(gm.rh), class_stride(gm.rw))) return;
    }
    const int HW = H * W;
    const uint32_t uHW = (uint32_t)HW;
    const int total = C * 49;
    const size_t src0 = (size_t)k * total, img = (size_t)b * C * HW;
    constexpr int U = 8;
    for (int e0 = threadIdx.x; e0 < total; e0 += U * 256) {
        int av[U];
        float gv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * 256;
            av[u] = -1;
            if (e < total) {
                av[u] = __ldg(argmax + src0 + e);
                gv[u] = __ldg(grad_out + src0 + e);
            }
        }
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            // neighbouring bins of a small roi often share their argmax pixel (windows coincide): consecutive lanes with the
            // same (channel, pixel) are summed in registers (segmented sum over runs: 5 shuffle steps) and only the first
            // lane of a run issues the atomic -- the kernel is bound by the L2 atomic rate, not by instructions
            const int c = (e0 + u * 256) / 49;
            const bool ok = (uint32_t)av[u] < uHW;
            const int key = ok ? av[u] : (-1 - lane);   // (an invalid element is a run of its own)
            const int prev = __shfl_up_sync(0xffffffffu, key, 1);
            const int prev_c = __shfl_up_sync(0xffffffffu, c, 1);
            const bool head = lane == 0 || prev != key || prev_c != c;
            const unsigned int heads = __ballot_sync(0xffffffffu, head);
            // end of this lane's run: the next head above it
            const unsigned int above = heads & ~((2u << lane) - 1u);
            const int run_end = above ? __ffs(above) - 1 : 32;   // first lane of the next run
            float sum = gv[u];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float v = __shfl_down_sync(0xffffffffu, sum, d);
                if (lane + d < run_end) sum = __fadd_rn(sum, v);
            }
            if (ok && head) {
                const size_t o = nhwc ? img + (size_t)av[u] * C + c : img + (size_t)c * HW + av[u];
                atomicAdd(grad_in + o, sum);
            }
        }
    }
}

static const size_t kPbSmemLimit = 227 * 1024;
static size_t pool_bwd_color_smem(int CB, int HW) {
    return kPbHdrBytes + (size_t)(CB / 2) * kPbDepth * kPbSlotBytes + (size_t)CB * HW * 4;
}

template <int CB>
static int launch_pool_bwd_color(const RoiPick& pk, const float* go, const int32_t* argmax, const float* rois, int K, int B,
                                 int C, int H, int W, float scale, int nhwc, float* gin, cudaStream_t st) {
    auto kern = roi_pool_bwd_color_kernel<CB>;
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPbSmemLimit));
    kern<<<dim3((C + CB - 1) / CB, B), CB * 16, pk.smem, st>>>(go, argmax, rois, K, C, H, W, scale, nhwc, gin);
    return FRR_OK;
}

// 7x7 RoIPool backward: colour classes + tail, or the tail kernel for every roi.
// false = outside this path (the caller takes the generic kernels)
bool roi_pool_bwd_fast_pick(int K, int H, int W, int PH, int PW, bool ptrs_aligned, RoiPick* pk) {
    if (PH != 7 || PW != 7 || K > kPbIdMask || !ptrs_aligned) return false;
    const int HW = H * W;
    // Two co-resident CTAs of 8 planes (one zeroes / scans / stores while the other accumulates) when they fit: the
    // 37 x 62 map of a 600 x 1000 image.  Larger maps (50 x 83 of an 800 x 1333 image: 4 accumulating warps per SM)
    // are faster with every roi through the streaming atomic kernel (measured 216-300 us against 287-330 us, torchvision
    // 320-341 us).
    if (2 * (pool_bwd_color_smem(8, HW) + 1024) <= kPbSmemLimit)
        *pk = RoiPick{kPoolBwdColorTail, 8, 1, 0, pool_bwd_color_smem(8, HW)};
    else
        *pk = RoiPick{kPoolBwdTail, 0, 1, 0, 0};
    return true;
}

int roi_pool_bwd_fast_launch(const RoiPick& pk, const float* grad_out, const int32_t* argmax, const float* rois, int K, int B,
                             int C, int H, int W, float scale, int nhwc, float* grad_in, frr_stream_t stream) {
    const int HW = H * W;
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.kernel == kPoolBwdTail) {
        FRR_CUDA(cudaMemsetAsync(grad_in, 0, (size_t)B * C * HW * sizeof(float), st));
        roi_pool_bwd_tail_kernel<<<K, 256, 0, st>>>(grad_out, argmax, rois, B, C, H, W, scale, nhwc, 1, grad_in);
        count_launch();
        FRR_CHECK_LAUNCH("roi_pool_bwd_tail_kernel");
        return FRR_OK;
    }
    const int rc = launch_pool_bwd_color<8>(pk, grad_out, argmax, rois, K, B, C, H, W, scale, nhwc, grad_in, st);
    if (rc) return rc;
    count_launch();
    FRR_CHECK_LAUNCH("roi_pool_bwd_color_kernel");
    roi_pool_bwd_tail_kernel<<<K, 256, 0, st>>>(grad_out, argmax, rois, B, C, H, W, scale, nhwc, 0, grad_in);
    count_launch();
    FRR_CHECK_LAUNCH("roi_pool_bwd_tail_kernel");
    return FRR_OK;
}

}  // namespace frr
