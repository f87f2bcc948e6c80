// P4 (general path): pre-NMS top-k of the RPN objectness scores, sorted descending (models/model.py:44-49).
// The fast path for N <= 65536 is the shared-memory bucket top-k of topk_radix.cu; this kernel covers larger N.
//
// One CTA (1024 threads) per image:
//   1. MSB-first radix select (4 x 8-bit digits) over order-preserving uint32 keys finds the
//      k-th largest key T and how many keys are strictly greater;
//   2. every key > T plus the lowest-index keys == T (ties: lower index first) are packed as
//      u64 (~key << 32 | index) into shared memory; per-32-anchor validity words and their
//      exclusive prefix give the index into the min-size-compacted array (what the reference's
//      sort returns) without a separate compaction pass;
//   3. an in-place bitonic sort of the <=16384 packed words in shared memory (ascending packed
//      == descending score, ascending index);
//   4. scores / indices / compacted indices / gathered boxes are written out, padded past count.
// Traffic: N*4 B of scores are re-read from L2 for the 4 select passes (<=150 KB per image),
// HBM algorithmic bytes = 4N + 40k per image (SURVEY §8d).
#include "frr_common.cuh"

namespace frr {

constexpr int kTopkThreads = 1024;
constexpr int kTopkWarps = kTopkThreads / 32;

struct TopkSmemHeader {
    unsigned int hist[256];
    unsigned int warp_tmp[kTopkWarps];
    unsigned int sel_count;   // packed entries written so far (for key > T)
    unsigned int prefix_key;  // selected high digits of T so far
    unsigned int remaining;   // how many still to take within the current digit bucket
    unsigned int nvalid;
};

__global__ void __launch_bounds__(kTopkThreads, 1)
    topk_bitonic_kernel(const float* __restrict__ scores, const uint8_t* __restrict__ valid,
                     const float4* __restrict__ boxes, int N, int k, int P /* pow2 >= k */, int nchunks /* ceil(N/32) */,
                     float* __restrict__ out_scores, int32_t* __restrict__ out_idx, int32_t* __restrict__ out_cidx,
                     float4* __restrict__ out_boxes, int32_t* __restrict__ out_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TopkSmemHeader* hd = reinterpret_cast<TopkSmemHeader*>(smem_raw);
    unsigned int* vbits = reinterpret_cast<unsigned int*>(smem_raw + sizeof(TopkSmemHeader));  // [nchunks]
    unsigned int* vpre = vbits + nchunks;                                                        // [nchunks]
    unsigned int* tpre = vpre + nchunks;                                                         // [nchunks] tie prefix
    unsigned long long* packed = reinterpret_cast<unsigned long long*>(
        smem_raw + ((sizeof(TopkSmemHeader) + 3 * sizeof(unsigned int) * (size_t)nchunks + 15) & ~(size_t)15));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x;
    const float* sc = scores + (size_t)b * N;
    const uint8_t* va = valid ? valid + (size_t)b * N : nullptr;

    // ---- validity words + count ------------------------------------------------------------
    unsigned int my_valid = 0;
    for (int c = warp; c < nchunks; c += kTopkWarps) {
        const int i = c * 32 + lane;
        const bool ok = (i < N) && (va ? (va[i] != 0) : true);
        const unsigned int w = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) vbits[c] = w;
        my_valid += ok ? 1u : 0u;
    }
    if (tid < 256) hd->hist[tid] = 0;
    if (tid == 0) { hd->sel_count = 0; hd->prefix_key = 0; }
    __syncthreads();
    {
        // exclusive prefix of popc(vbits) over chunks -> vpre ; total -> nvalid
        unsigned int run = 0;  // chunks are scanned in tiles of 1024
        for (int base = 0; base < nchunks; base += kTopkThreads) {
            const int c = base + tid;
            const unsigned int v = (c < nchunks) ? __popc(vbits[c]) : 0u;
            unsigned int tot;
            const unsigned int ex = block_exclusive_scan(v, hd->warp_tmp, &tot);
            if (c < nchunks) vpre[c] = run + ex;
            run += tot;
        }
        if (tid == 0) hd->nvalid = run;
    }
    __syncthreads();
    const int nvalid = (int)hd->nvalid;
    const int keff = min(k, nvalid);
    if (tid == 0) {
        out_count[b] = keff;
        hd->remaining = (unsigned int)keff;
    }
    __syncthreads();

    // ---- radix select: find T = keff-th largest key among valid ------------------------------
    if (keff > 0) {
        unsigned int prefix = 0, pmask = 0;
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int c = warp; c < nchunks; c += kTopkWarps) {
                const int i = c * 32 + lane;
                const bool ok = (vbits[c] >> lane) & 1u;
                if (ok) {
                    const unsigned int key = float_to_ordered(sc[i]);
                    if ((key & pmask) == prefix) atomicAdd(&hd->hist[(key >> shift) & 255u], 1u);
                }
            }
            __syncthreads();
            // warp 0: walk digits from 255 down, find bucket where cumulative >= remaining
            if (warp == 0) {
                const unsigned int need = hd->remaining;
                // lane handles 8 digits: d = 255 - (lane*8 + j)
                unsigned int cnt[8], s = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) { cnt[j] = hd->hist[255 - (lane * 8 + j)]; s += cnt[j]; }
                unsigned int inc = s;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                unsigned int before = inc - s;  // keys in strictly higher digits handled by lower lanes
                const bool here = (before < need) && (inc >= need);
                if (here) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (before < need && before + cnt[j] >= need) {
                            hd->prefix_key = prefix | ((unsigned int)(255 - (lane * 8 + j)) << shift);
                            hd->remaining = need - before;  // to take from inside this bucket
                            before = need;                  // stop
                        } else {
                            before += cnt[j];
                        }
                    }
                }
            }
            __syncthreads();
            prefix = hd->prefix_key;
            pmask |= (255u << shift);
            if (tid < 256) hd->hist[tid] = 0;
            __syncthreads();
        }
        // now prefix == T, hd->remaining == number of keys == T to take (lowest index first)
        const unsigned int T = prefix;
        const unsigned int take_ties = hd->remaining;

        // ---- tie prefix per chunk (ordered) --------------------------------------------------
        {
            unsigned int run = 0;
            for (int base = 0; base < nchunks; base += kTopkThreads) {
                const int c = base + tid;
                unsigned int v = 0;
                if (c < nchunks) {
                    unsigned int w = vbits[c];
                    while (w) {
                        const int l = __ffs(w) - 1;
                        w &= w - 1;
                        v += (float_to_ordered(sc[c * 32 + l]) == T) ? 1u : 0u;
                    }
                }
                unsigned int tot;
                const unsigned int ex = block_exclusive_scan(v, hd->warp_tmp, &tot);
                if (c < nchunks) tpre[c] = run + ex;
                run += tot;
            }
        }
        __syncthreads();

        // ---- pack selected entries into smem ---------------------------------------------------
        for (int c = warp; c < nchunks; c += kTopkWarps) {
            const int i = c * 32 + lane;
            const bool ok = (vbits[c] >> lane) & 1u;
            unsigned int key = 0;
            if (ok) key = float_to_ordered(sc[i]);
            const bool gt = ok && key > T;
            const bool eq = ok && key == T;
            const unsigned int eqm = __ballot_sync(0xffffffffu, eq);
            const bool take_eq = eq && (tpre[c] + __popc(eqm & ((1u << lane) - 1u)) < take_ties);
            const bool take = gt || take_eq;
            const unsigned int tm = __ballot_sync(0xffffffffu, take);
            if (tm) {
                unsigned int basepos = 0;
                if (lane == 0) basepos = atomicAdd(&hd->sel_count, (unsigned int)__popc(tm));
                basepos = __shfl_sync(0xffffffffu, basepos, 0);
                if (take) {
                    const unsigned int pos = basepos + __popc(tm & ((1u << lane) - 1u));
                    packed[pos] = ((unsigned long long)(~key) << 32) | (unsigned int)i;
                }
            }
        }
    }
    // pad to P with sentinels (sort last)
    for (int p = keff + tid; p < P; p += kTopkThreads) packed[p] = ~0ull;
    __syncthreads();

    // ---- bitonic sort ascending over P packed words ----------------------------------------------
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int p = tid; p < (P >> 1); p += kTopkThreads) {
                const int lo = 2 * p - (p & (stride - 1));  // index with bit `stride` clear
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long a = packed[lo], c2 = packed[hi];
                if ((a > c2) == up) { packed[lo] = c2; packed[hi] = a; }
            }
            __syncthreads();
        }
    }

    // ---- write-out ---------------------------------------------------------------------------------
    for (int j = tid; j < k; j += kTopkThreads) {
        const size_t o = (size_t)b * k + j;
        if (j < keff) {
            const unsigned long long e = packed[j];
            const unsigned int key = ~(unsigned int)(e >> 32);
            const int i = (int)(unsigned int)(e & 0xffffffffu);
            if (out_scores) out_scores[o] = ordered_to_float(key);
            out_idx[o] = i;
            if (out_cidx) out_cidx[o] = (int)(vpre[i >> 5] + __popc(vbits[i >> 5] & ((1u << (i & 31)) - 1u)));
            if (out_boxes) out_boxes[o] = boxes[(size_t)b * N + i];
        } else {
            if (out_scores) out_scores[o] = __uint_as_float(0xff800000u);  // -inf
            out_idx[o] = -1;
            if (out_cidx) out_cidx[o] = -1;
            if (out_boxes) out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

static size_t topk_smem_bytes(int nchunks, int P) {
    size_t s = sizeof(TopkSmemHeader) + 3 * sizeof(unsigned int) * (size_t)nchunks;
    s = (s + 15) & ~(size_t)15;
    return s + sizeof(unsigned long long) * (size_t)P;
}

int topk_radix_launch(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k,
                      float* out_scores, int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count,
                      frr_stream_t stream, int cluster_hint);

int topk_desc_impl(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k, float* out_scores,
                   int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count, int cluster_hint,
                   frr_stream_t stream);

}  // namespace frr

extern "C" int frr_topk_desc_opt(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k,
                                 float* out_scores, int32_t* out_idx, int32_t* out_cidx, float* out_boxes,
                                 int32_t* out_count, int ctas_per_image, frr_stream_t stream) {
    FRR_CHECK_ARG(ctas_per_image == 0 || ctas_per_image == 1, "frr_topk_desc_opt: ctas_per_image must be 0 (automatic) or 1");
    return frr::topk_desc_impl(scores, valid, boxes, B, N, k, out_scores, out_idx, out_cidx, out_boxes, out_count,
                               ctas_per_image, stream);
}

// cluster_hint: 0 = CTAs per image chosen for the lowest latency of this call, 1 = one CTA per image
int frr::topk_desc_impl(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k, float* out_scores,
                        int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count, int cluster_hint,
                        frr_stream_t stream) {
    using namespace frr;
    FRR_CHECK_ARG(scores && out_idx && out_count, "frr_topk_desc_opt: null pointer");
    FRR_CHECK_ARG(B >= 0 && N >= 0 && k >= 0, "frr_topk_desc_opt: bad sizes B=%d N=%d k=%d", B, N, k);
    FRR_CHECK_ARG((out_boxes == nullptr) || (boxes != nullptr && aligned16(boxes) && aligned16(out_boxes)),
                  "frr_topk_desc_opt: boxes must be given and 16-byte aligned when out_boxes is requested");
    if (B == 0 || k == 0) return FRR_OK;
    FRR_CHECK_ARG(k <= 16384, "frr_topk_desc_opt: k=%d exceeds the in-smem sort capacity 16384", k);
    {   // fast path: shared-memory bucket top-k (topk_radix.cu); shapes outside it take the bitonic kernel below
        const int rc = topk_radix_launch(scores, valid, boxes, B, N, k, out_scores, out_idx, out_cidx, out_boxes, out_count,
                                         stream, cluster_hint);
        if (rc <= 0) return rc;
    }
    int P = 32;
    while (P < k) P <<= 1;
    const int nchunks = (N + 31) / 32;
    const size_t smem = topk_smem_bytes(nchunks, P);
    FRR_CHECK_ARG(smem <= 227 * 1024, "frr_topk_desc_opt: N=%d k=%d needs %zu B shared memory (> 227 KB)", N, k, smem);
    // per device attribute: set before every launch (a process may drive several GPUs)
    FRR_CUDA(cudaFuncSetAttribute(topk_bitonic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    topk_bitonic_kernel<<<B, kTopkThreads, smem, (cudaStream_t)stream>>>(scores, valid, (const float4*)boxes, N, k, P,
                                                                       nchunks, out_scores, out_idx, out_cidx,
                                                                       (float4*)out_boxes, out_count);
    count_launch();
    FRR_CHECK_LAUNCH("topk_bitonic_kernel");
    return FRR_OK;
}
