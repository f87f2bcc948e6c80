// N1: greedy NMS over score-sorted boxes (torchvision.ops.nms semantics, models/model.py:53-55).
//
// Keep-list algorithm on one thread-block cluster per image (no n x n mask in HBM):
//   the cluster walks the sorted candidates in chunks of 256; each CTA owns a round-robin slice
//   of the boxes kept so far (shared memory) and tests the chunk against its slice; the
//   per-CTA suppression words are exchanged through distributed shared memory (one
//   cluster barrier per chunk); every CTA then resolves the chunk's survivors among
//   themselves (warp-ballot predecessor masks + a parallel fix-point) and appends the newly
//   kept boxes to its slice.  The walk stops at max_keep, so with the RPN's 12000 -> 2000
//   only the first ~5-6k candidates are ever touched and each is tested against kept boxes
//   only (~5 M pair tests instead of the 72 M of the full upper triangle).
//
// Phase 1 is register tiled: a thread holds 4 candidates and streams kept boxes from shared
// memory (one broadcast LDS.128 feeds 128 pair tests), because the un-tiled version was bound
// by shared-memory wavefronts, not by the FP32/ALU pipes.
//
// Bit-exactness vs the CPU kernel: IoU = inter / ((area_i + area_j) - inter) in fp32 with IEEE
// division and no FMA contraction; suppress when (double)iou > thr  <=>  iou >= up, where up is
// the smallest fp32 strictly above thr.  Almost every pair is rejected without the division by
// a conservative 10-instruction screen:  inter/union < up  <=  inter < c2*(area_a + area_b) with
// c2 = up/(1+up)*(1 - 2^-19)  (the 2^-19 margin covers every fp32 rounding in the screen and in
// the exact formula, see suppress_screen<kUnit>()); the ~0.3 % of pairs that pass the screen take the exact
// division.  Degenerate / tiny boxes carry a NaN screening area, which always fails the screen.
#include <cooperative_groups.h>
#include <math.h>

#include "nms_common.cuh"

namespace cg = cooperative_groups;

namespace frr {

constexpr int kChunk = 256;  // candidates per chunk
constexpr int kChunkWords = kChunk / 32;
constexpr int kTile = 4;                // candidates per thread in phase 1
constexpr int kGroup = kChunk / kTile;  // threads that together cover one chunk (64)

struct NmsSmem {
    unsigned int supp[2][kMaxCluster][kChunkWords];  // [parity][src rank][word]: suppressed-by-slice words
    unsigned int acc[2][kChunkWords];                // [parity][word]: this CTA's words (OR over its parts)
    unsigned int warp_cnt[kChunkWords];
    unsigned int kept_w[2][kChunkWords];  // fix-point state, double buffered
    unsigned int removed_w[2][kChunkWords];
    unsigned int pred[kChunk][kChunkWords];  // pred[i][q]: bit j set if survivor 32q+j (< i) suppresses survivor i
    float4 cbox[kChunk];                     // the chunk's candidates
    float carea[kChunk];
    float4 sbox[kChunk];  // survivor boxes (compacted)
    float sarea[kChunk];
    short ssrc[kChunk];  // survivor -> position inside the chunk
};

// barrier over the first `n` threads of the CTA with an OR reduction of `pred`
__device__ __forceinline__ bool bar_or(int id, int n, bool pred) {
    int r;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
        : "=r"(r)
        : "r"((int)pred), "r"(id), "r"(n)
        : "memory");
    return r != 0;
}

template <int kThreads, bool kFast, bool kUnit>
__global__ void __launch_bounds__(kThreads)
    nms_keeplist_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ counts, int n, int max_keep,
                        int slice_cap, NmsThr thr, int32_t* __restrict__ keep, int32_t* __restrict__ keep_count,
                        float4* __restrict__ out_boxes, const int32_t* __restrict__ gather_idx, int src_n) {
    static_assert(kThreads >= kChunk && kThreads % kGroup == 0, "bad thread count");
    constexpr int kWarps = kThreads / 32;
    constexpr int kParts = kThreads / kGroup;  // interleaved parts of the kept slice
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int img = blockIdx.x / S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int part = tid / kGroup;  // which interleaved part of the kept slice this thread scans
    const int u = tid % kGroup;     // candidates u, u+64, u+128, u+192 of the chunk

    extern __shared__ __align__(16) unsigned char smem_raw[];
    NmsSmem* sm = reinterpret_cast<NmsSmem*>(smem_raw);
    float4* kbox = reinterpret_cast<float4*>(smem_raw + ((sizeof(NmsSmem) + 15) & ~(size_t)15));  // [slice_cap]
    float* karea = reinterpret_cast<float*>(kbox + slice_cap);                                      // [slice_cap]

    const int cnt = counts ? min(counts[img], n) : n;
    // candidate i of the image: boxes[img][i], or boxes[img][gather_idx[img][i]] when the sorted order is given as
    // indices into an unsorted [B, src_n, 4] array (the top-k kernel then never writes the 12 000 gathered boxes, and
    // only the ~5 000 candidates NMS really visits are ever gathered)
    const float4* ib = boxes + (size_t)img * (gather_idx ? src_n : n);
    const int32_t* gi = gather_idx ? gather_idx + (size_t)img * n : nullptr;
    auto cand = [&](int i) -> float4 { return gi ? ib[gi[i]] : ib[i]; };
    int32_t* ikeep = keep + (size_t)img * max_keep;
    float4* iout = out_boxes ? out_boxes + (size_t)img * max_keep : nullptr;
    int nk = 0;  // kept so far (identical in every CTA of the cluster)
    int par = 0;
    float4 nbx = make_float4(0.f, 0.f, 0.f, 0.f);  // prefetched candidate of the next chunk (first kChunk threads)
    if (tid < kChunk && tid < cnt) nbx = cand(tid);
    if (tid < 2 * kChunkWords) (&sm->acc[0][0])[tid] = 0u;
    for (int base = 0; base < cnt && nk < max_keep; base += kChunk, par ^= 1) {
        // ---- phase 0: stage the chunk's candidates in shared memory, prefetch the next chunk ----------
        if (tid < kChunk) {
            sm->cbox[tid] = nbx;
            sm->carea[tid] = screen_area(nbx, thr.c2);
            const int nx = base + kChunk + tid;
            if (nx < cnt) nbx = cand(nx);
        }
        __syncthreads();

        const int ns = (nk - rank + S - 1) / S;  // kept ordinals o with o % S == rank
        // ---- phase 1: 4 candidates per thread vs this CTA's slice of the kept list ----------------------
        {
            float4 cb[kTile];
            float ca[kTile];
            bool has[kTile], sup[kTile];
#pragma unroll
            for (int j = 0; j < kTile; ++j) {
                cb[j] = sm->cbox[u + j * kGroup];
                ca[j] = sm->carea[u + j * kGroup];
                has[j] = base + u + j * kGroup < cnt;
                sup[j] = !has[j];
            }
            if (kFast) {
                // Screen every kept box of the slice; remember only the FIRST one that passes the screen and
                // evaluate it exactly after the loop (all lanes together).  The screen is tight (2^-19), so a
                // pass is almost always a true suppression; the rare lane whose exact test fails rescans.
                // The slice part is walked from its END so that the plain conditional move below leaves the SMALLEST
                // passing k (one ALU op less per pair than "first hit wins").
                int pk[kTile];
#pragma unroll
                for (int j = 0; j < kTile; ++j) pk[j] = -1;
                const int cntp = (ns > part) ? (ns - part + kParts - 1) / kParts : 0;
#pragma unroll 2
                for (int k = part + (cntp - 1) * kParts; k >= part; k -= kParts) {
                    const float4 kb = kbox[k];
                    const float ka = karea[k];
#pragma unroll
                    for (int j = 0; j < kTile; ++j)
                        if (suppress_screen<kUnit>(kb, ka, cb[j], ca[j])) pk[j] = k;
                }
#pragma unroll
                for (int j = 0; j < kTile; ++j) {
                    if (has[j] && pk[j] >= 0) {
                        sup[j] = suppress_exact(kbox[pk[j]], cb[j], thr.up);
                        for (int k2 = pk[j] + kParts; k2 < ns && !sup[j]; k2 += kParts)
                            if (suppress_screen<kUnit>(kbox[k2], karea[k2], cb[j], ca[j]))
                                sup[j] = suppress_exact(kbox[k2], cb[j], thr.up);
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < kTile; ++j)
                    for (int k = part; k < ns && !sup[j]; k += kParts) sup[j] = suppress_exact(kbox[k], cb[j], thr.up);
            }
            // warp covers candidates u in [32 * (warp % kGW), +32) + kGroup j  ->  word (warp % kGW) + kGW j
            constexpr int kGW = kGroup / 32;
#pragma unroll
            for (int j = 0; j < kTile; ++j) {
                const unsigned int wj = __ballot_sync(0xffffffffu, sup[j]);
                if (lane == 0 && wj != 0u) atomicOr(&sm->acc[par][(warp % kGW) + kGW * j], wj);
            }
        }
        __syncthreads();
        // publish this CTA's 8 words to every CTA of the cluster (distributed shared memory)
        if (tid < kChunkWords * S) {
            const int wd = tid % kChunkWords, dstr = tid / kChunkWords;
            unsigned int* dst = cluster.map_shared_rank(&sm->supp[par][rank][wd], dstr);
            *dst = sm->acc[par][wd];
        }
        cluster.sync();

        // ---- phase 2: combine the S words per 32 candidates, compact survivors (first kChunk threads) ---
        bool alive = false;
        unsigned int am = 0;
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        float fa = 0.f;
        if (tid < kChunk) {
            const unsigned int v = (lane < S) ? sm->supp[par][lane][warp] : 0u;
            const unsigned int all = __reduce_or_sync(0xffffffffu, v);
            alive = !((all >> lane) & 1u);
            am = __ballot_sync(0xffffffffu, alive);
            if (lane == 0) sm->warp_cnt[warp] = __popc(am);
            if (tid < kChunkWords) {
                sm->kept_w[0][tid] = 0;
                sm->removed_w[0][tid] = 0;
                sm->acc[par ^ 1][tid] = 0;  // for the next chunk
            }
            bx = sm->cbox[tid];
            fa = sm->carea[tid];
        }
        __syncthreads();
        int s = 0;
        {
            int soff = 0;
#pragma unroll
            for (int w2 = 0; w2 < kChunkWords; ++w2) {
                const int cc = (int)sm->warp_cnt[w2];
                if (w2 < warp) soff += cc;
                s += cc;
            }
            if (alive) {
                const int si = soff + __popc(am & ((1u << lane) - 1u));
                sm->sbox[si] = bx;
                sm->sarea[si] = fa;
                sm->ssrc[si] = (short)tid;
            }
        }
        __syncthreads();

        // ---- phase 3: predecessor masks among survivors.  3a: warp item = (row, 32-column word), screen only (two
        //      words per trip for ILP); 3b: the few set bits are refined with the exact test, one (row, word) entry
        //      per thread, so the exact path never diverges a busy warp ----------------------------------------
        for (int row = warp; row < s; row += kWarps) {
            const float4 rb = sm->sbox[row];
            const float ra = sm->sarea[row];
            for (int q = 0; q * 32 < row; q += 2) {
                const int j0 = q * 32 + lane, j1 = j0 + 32;  // j1 <= 255
                bool h0 = false, h1 = false;
                if (kFast) {
                    h0 = (j0 < row) && suppress_screen<kUnit>(sm->sbox[j0], sm->sarea[j0], rb, ra);
                    h1 = (j1 < row) && suppress_screen<kUnit>(sm->sbox[j1], sm->sarea[j1], rb, ra);
                } else {
                    if (j0 < row) h0 = suppress_exact(sm->sbox[j0], rb, thr.up);
                    if (j1 < row) h1 = suppress_exact(sm->sbox[j1], rb, thr.up);
                }
                const unsigned int b0 = __ballot_sync(0xffffffffu, h0);
                const unsigned int b1 = __ballot_sync(0xffffffffu, h1);
                if (lane == 0) {
                    sm->pred[row][q] = b0;
                    sm->pred[row][q + 1] = b1;
                }
            }
        }
        if (kFast) {
            __syncthreads();
            for (int e = tid; e < s * kChunkWords; e += kThreads) {
                const int row = e / kChunkWords, q = e - row * kChunkWords;
                if (q * 32 < row) {
                    unsigned int m = sm->pred[row][q], keepm = m;
                    while (m) {
                        const int bit = __ffs(m) - 1;
                        m &= m - 1;
                        if (!suppress_exact(sm->sbox[q * 32 + bit], sm->sbox[row], thr.up)) keepm &= ~(1u << bit);
                    }
                    sm->pred[row][q] = keepm;
                }
            }
        }
        __syncthreads();

        // ---- phase 4: parallel fix-point over the survivors (first kChunk threads, named barrier 1).
        //      survivor i is kept once every predecessor that suppresses it is removed; removed as soon
        //      as one such predecessor is kept.  State words are double buffered: one barrier / round. ----
        int fin = 0;
        if (tid < kChunk) {
            int state = (tid < s) ? 0 : 3;  // 0 undecided, 1 kept, 2 removed, 3 n/a
            unsigned int p[kChunkWords];
#pragma unroll
            for (int q = 0; q < kChunkWords; ++q) p[q] = (state == 0 && q * 32 < tid) ? sm->pred[tid][q] : 0u;
            int cur = 0;
            for (;;) {
                if (state == 0) {
                    bool hit_kept = false, pending = false;
#pragma unroll
                    for (int q = 0; q < kChunkWords; ++q) {
                        const unsigned int kw = sm->kept_w[cur][q], rw = sm->removed_w[cur][q];
                        hit_kept |= (p[q] & kw) != 0u;
                        pending |= (p[q] & ~(kw | rw)) != 0u;
                    }
                    if (hit_kept) state = 2;
                    else if (!pending) state = 1;
                }
                const unsigned int km = __ballot_sync(0xffffffffu, state == 1);
                const unsigned int rm = __ballot_sync(0xffffffffu, state == 2);
                if (lane == 0) {
                    sm->kept_w[cur ^ 1][warp] = km;
                    sm->removed_w[cur ^ 1][warp] = rm;
                }
                cur ^= 1;
                if (!bar_or(1, kChunk, state == 0)) break;
            }
            fin = cur;
        }
        // every thread needs the final buffer index: it is uniform over the first kChunk threads
        fin = __syncthreads_or(fin);

        // ---- phase 5: append kept survivors --------------------------------------------------------------
        {
            int koff = 0, ktot = 0;
#pragma unroll
            for (int w2 = 0; w2 < kChunkWords; ++w2) {
                const int cc = __popc(sm->kept_w[fin][w2]);
                if (w2 < warp) koff += cc;
                ktot += cc;
            }
            if (tid < kChunk) {
                const unsigned int kw = sm->kept_w[fin][warp];
                if ((kw >> lane) & 1u) {
                    const int o = nk + koff + __popc(kw & ((1u << lane) - 1u));
                    if (o < max_keep) {
                        const float4 kb = sm->sbox[tid];
                        if (o % S == rank) {
                            kbox[o / S] = kb;
                            karea[o / S] = sm->sarea[tid];
                        }
                        if (rank == 0) {
                            ikeep[o] = base + (int)sm->ssrc[tid];
                            if (iout) iout[o] = kb;
                        }
                    }
                }
            }
            nk = min(nk + ktot, max_keep);
        }
        __syncthreads();
    }

    if (rank == 0) {
        for (int o = nk + tid; o < max_keep; o += kThreads) {
            ikeep[o] = -1;
            if (iout) iout[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (tid == 0) keep_count[img] = nk;
    }
}

static size_t nms_smem_bytes(int slice_cap) {
    return ((sizeof(NmsSmem) + 15) & ~(size_t)15) + (size_t)slice_cap * (sizeof(float4) + sizeof(float));
}

// Launch geometry and kernel variant for a problem: shared by nms_launch and frr_nms_variant (tests / bench assert
// through the latter that the variant they mean to exercise is the one that runs).
struct NmsPick {
    int S, threads, slice_cap, bucketed;
    size_t smem;
    NmsThr thr;
};

static int nms_pick(int B, int n, double iou_thr, int max_keep, int cluster_size, int threads, int unit_boxes, NmsPick* out) {
    FRR_CHECK_ARG(B >= 0 && n >= 0 && max_keep >= 0, "frr_nms_sorted: bad sizes B=%d n=%d max_keep=%d", B, n, max_keep);
    FRR_CHECK_ARG(threads == 0 || threads == 256 || threads == 512 || threads == 1024,
                  "frr_nms_sorted: threads %d not in {0,256,512,1024}", threads);
    const int kcap = max_keep < n ? max_keep : n;  // most boxes that can ever be kept
    int S = cluster_size;
    if (S == 0) {
        // auto: fill the machine.  148 SMs / B images, rounded down to a power of two, capped at 16.
        int per = num_sms() / (B > 0 ? B : 1);
        S = 1;
        while (S * 2 <= per && S < 16) S *= 2;
    }
    FRR_CHECK_ARG(S == 1 || S == 2 || S == 4 || S == 8 || S == 16, "frr_nms_sorted: cluster_size %d not in {1,2,4,8,16}", S);
    const NmsThr thr = make_thr(iou_thr);
    out->thr = thr;
    // Unit-range boxes with a screenable threshold (the RPN proposal layer, models/model.py:53): the bucketed
    // large-chunk kernel of nms_bucket.cu, every CTA of the cluster holds the whole kept list.  1024 threads by default,
    // also for one CTA per image: the 512-thread form fits twice per SM, but a CTA of it alone takes 173 instead of
    // 135 us per 148 images and two per SM only 2 % less SM time (250 vs 256 us per 296 images), so with several
    // batches in flight the 1024-thread form is faster (B200).
    if (nms_bucket_eligible(n, max_keep, thr, unit_boxes)) {
        out->S = S;
        out->threads = threads != 0 ? threads : 1024;
        out->slice_cap = 0;
        out->bucketed = 1;
        out->smem = nms_bucket_smem_bytes(out->threads, S);
        return FRR_OK;
    }
    // a CTA whose slice of the kept list is short (one image spread over 16 CTAs) is bound by its per-chunk barriers:
    // 16 warps resolve them faster than 32 (130 vs 134 us for 12000 -> 2000 boxes)
    if (threads == 0) threads = (kcap / S < 192) ? 512 : 1024;
    if (threads < kChunk) threads = kChunk;  // the first kChunk threads own one candidate each
    // grow the cluster until a slice of the kept list fits in shared memory
    const size_t limit = 227 * 1024;
    while (nms_smem_bytes((kcap + S - 1) / S + 1) > limit && S < 16) S *= 2;
    const int slice_cap = (kcap + S - 1) / S + 1;
    const size_t smem = nms_smem_bytes(slice_cap);
    FRR_CHECK_ARG(smem <= limit, "frr_nms_sorted: max_keep=%d does not fit the kept list in shared memory", max_keep);
    out->S = S;
    out->threads = threads;
    out->slice_cap = slice_cap;
    out->bucketed = 0;
    out->smem = smem;
    return FRR_OK;
}

int nms_launch(const float* boxes, const int32_t* counts, int B, int n, double iou_thr, int max_keep,
                      int32_t* keep, int32_t* keep_count, float* out_boxes, int cluster_size, int threads,
                      const NmsTune& tune, int unit_boxes, frr_stream_t stream, const int32_t* gather_idx, int src_n) {
    FRR_CHECK_ARG(keep && keep_count, "frr_nms_sorted: null output");
    FRR_CHECK_ARG(n == 0 || (boxes && aligned16(boxes)), "frr_nms_sorted: boxes must be non-null, 16-byte aligned");
    FRR_CHECK_ARG(out_boxes == nullptr || aligned16(out_boxes), "frr_nms_sorted: out_boxes must be 16-byte aligned");
    NmsPick pk;
    {
        const int rc = nms_pick(B, n, iou_thr, max_keep, cluster_size, threads, unit_boxes, &pk);
        if (rc) return rc;
    }
    if (B == 0) return FRR_OK;
    if (pk.bucketed)
        return nms_bucket_launch(boxes, counts, B, n, pk.thr, max_keep, keep, keep_count, out_boxes, pk.S, pk.threads, tune,
                                 stream, gather_idx, src_n);
    const int S = pk.S, slice_cap = pk.slice_cap;
    threads = pk.threads;
    const size_t smem = pk.smem, limit = 227 * 1024;
    const NmsThr thr = pk.thr;

    using kern_t = void (*)(const float4*, const int32_t*, int, int, int, NmsThr, int32_t*, int32_t*, float4*, const int32_t*,
                            int);
    kern_t kern = nullptr;
#define FRR_NMS_PICK(F, U)                                                                      \
    (threads < kChunk * 2 ? nms_keeplist_kernel<kChunk, F, U>                                            \
                    : threads == 512 ? nms_keeplist_kernel<512, F, U> : nms_keeplist_kernel<1024, F, U>)
    if (thr.fast && unit_boxes) kern = FRR_NMS_PICK(true, true);
    else if (thr.fast) kern = FRR_NMS_PICK(true, false);
    else kern = FRR_NMS_PICK(false, false);
#undef FRR_NMS_PICK
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    if (S > 8) FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));

    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * S), 1, 1);
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FRR_CUDA(cudaLaunchKernelEx(&cfg, kern, (const float4*)boxes, counts, n, max_keep, slice_cap, thr, keep, keep_count,
                                (float4*)out_boxes, gather_idx, src_n));
    count_launch();
    FRR_CHECK_LAUNCH("nms_keeplist_kernel");
    return FRR_OK;
}

}  // namespace frr

extern "C" int frr_nms_sorted(const float* boxes, const int32_t* counts, int B, int n, double iou_thr, int max_keep,
                              int32_t* keep, int32_t* keep_count, float* out_boxes, int cluster_size, int threads,
                              int first_chunk, int max_chunk, int lanes_screen, int lanes_pairs, int unit_boxes,
                              frr_stream_t stream) {
    using frr::kBkChunk;
    auto chunk_ok = [](int v) { return v == 0 || (v >= 256 && v <= kBkChunk); };
    auto lanes_ok = [](int v) { return v == 0 || (v >= 1 && v <= 32 && (v & (v - 1)) == 0); };
    FRR_CHECK_ARG(chunk_ok(first_chunk) && chunk_ok(max_chunk),
                  "frr_nms_sorted: chunk sizes must be 0 or lie in [256, %d]", kBkChunk);
    FRR_CHECK_ARG(lanes_ok(lanes_screen) && lanes_ok(lanes_pairs),
                  "frr_nms_sorted: lanes per candidate must be 0 or a power of two <= 32");
    return frr::nms_launch(boxes, counts, B, n, iou_thr, max_keep, keep, keep_count, out_boxes, cluster_size, threads,
                           frr::NmsTune{first_chunk, max_chunk, lanes_screen, lanes_pairs}, unit_boxes, stream, nullptr, 0);
}

// Which kernel variant / launch geometry frr_nms_sorted* picks for a problem (host only, launches nothing):
// out[0] = CTAs per image (cluster size), out[1] = threads per CTA, out[2] = variant (0 exact only, 1 screened,
// 2 screened + unit range, 3 unit range + class / x-bin bucketed kept slice), out[3] = dynamic shared memory bytes.
extern "C" int frr_nms_variant(int B, int n, double iou_thr, int max_keep, int cluster_size, int threads, int unit_boxes,
                               int32_t* out4) {
    FRR_CHECK_ARG(out4 != nullptr, "frr_nms_variant: null output");
    frr::NmsPick pk;
    const int rc = frr::nms_pick(B, n, iou_thr, max_keep, cluster_size, threads, unit_boxes, &pk);
    if (rc) return rc;
    out4[0] = pk.S;
    out4[1] = pk.threads;
    out4[2] = pk.bucketed ? 3 : (pk.thr.fast ? (unit_boxes ? 2 : 1) : 0);
    out4[3] = (int32_t)pk.smem;
    return FRR_OK;
}

// Same as frr_nms_sorted, but the score order is given as indices: candidate i of image b is
// boxes_src[b][order[b][i]] (boxes_src [B,src_n,4], order int32 [B,n], e.g. the out_idx of frr_topk_desc_opt).
extern "C" int frr_nms_sorted_indirect(const float* boxes_src, int src_n, const int32_t* order, const int32_t* counts, int B,
                                       int n, double iou_thr, int max_keep, int32_t* keep, int32_t* keep_count,
                                       float* out_boxes, int cluster_size, int unit_boxes, frr_stream_t stream) {
    FRR_CHECK_ARG(order != nullptr && src_n >= 0, "frr_nms_sorted_indirect: order must be given");
    return frr::nms_launch(boxes_src, counts, B, n, iou_thr, max_keep, keep, keep_count, out_boxes, cluster_size, 0, frr::NmsTune{},
                           unit_boxes, stream, order, src_n);
}
