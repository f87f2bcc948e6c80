// P4 (fast path): pre-NMS top-k, sorted descending, ties lower-index-first (models/model.py:44-49).
// Two algorithms in one launch: topk_bucket_kernel (below, the default: one or two CTAs per image) and the radix path
// described here, which it falls into for inputs that do not bucket.  The bucket kernel's shared memory fits for every
// shape the fast path takes (static_assert after bkc_layout), so the radix path never runs as a kernel of its own.
//
// Radix path: one CTA (1024 threads) per image, everything after the first read of the scores stays in shared memory:
//   0. validity words (ballot) + the order-preserving uint32 keys of all N scores staged in shared memory;
//   1. MSB-first radix select (4 x 8-bit digits, warp-aggregated histogram atomics) -> T = k-th largest key
//      and how many keys == T to take;
//   2. ORDER-PRESERVING compaction of the selected (key, index) pairs (two block scans: #greater and #equal
//      before every 32-anchor chunk), so that a STABLE sort by key alone yields "ties: lower index first";
//   3. stable LSD radix sort of the <= 16384 selected pairs, 4 passes of 8 bits: every warp owns a contiguous
//      run of rows, ranks its keys with ballot-built peer masks, keeps a private 256-bin histogram (u16), the digit-major /
//      warp-minor exclusive scan turns the 32 x 256 counts into scatter offsets;
//   4. scores / indices / compacted indices / gathered boxes are written out (padded past count).
// Compared with the bitonic version (105 compare-exchange stages with a barrier each, contended histogram
// atomics) this is ~10x fewer shared-memory wavefronts and barriers.  HBM bytes: 5N in, 40k out per image.
#include <cooperative_groups.h>

#include "frr_common.cuh"

namespace frr {

constexpr int kRsThreads = 1024;
constexpr int kRsWarps = kRsThreads / 32;

struct RsHdr {
    unsigned int hist[256];
    unsigned int warp_tmp[kRsWarps];
    unsigned int prefix_key;
    unsigned int remaining;
    unsigned int nvalid;
    unsigned int bsize;    // keys in the bucket chosen by the last select pass
    unsigned int lcount;   // candidate list fill
    unsigned int pad[3];
};

struct RsLayout {
    size_t vbits, gpre, epre, vpre, whist, keyA, idxA, area2, total;
    int staged;
    int db;  // digit bits of the sort passes (5 when the 2^db x 1024 u16 counters fit, else 4)
};

__host__ __device__ constexpr size_t up16(size_t x) { return (x + 15) & ~(size_t)15; }

static RsLayout rs_layout(int N, int kcap, int nchunks, bool want_stage, int db) {
    RsLayout L;
    size_t o = up16(sizeof(RsHdr));
    L.vbits = o; o += 4 * (size_t)nchunks;
    L.gpre = o;  o += 4 * (size_t)nchunks;
    L.epre = o;  o += 4 * (size_t)nchunks;
    L.vpre = o;  o += 4 * (size_t)nchunks;
    o = up16(o);
    L.whist = o; o += ((size_t)1 << db) * kRsThreads * 2;  // counters [digit][thread] u16
    L.db = db;
    L.keyA = o;  o += 4 * (size_t)kcap;
    L.idxA = o;  o += 2 * (size_t)kcap;
    o = up16(o);
    L.area2 = o;
    const size_t sortB = 6 * (size_t)kcap;
    const size_t stage = 4 * (size_t)N;
    L.staged = want_stage ? 1 : 0;
    L.total = o + up16(want_stage && stage > sortB ? stage : sortB);
    return L;
}

// Lanes of the warp that are active and hold the same 8-bit digit (9 ballots).  match.any is not used: its
// throughput on sm_100 is ~1 warp instruction per ~50 cycles per SM (measured: 1.6k cycles per row with 32 warps).
__device__ __forceinline__ unsigned int match_digit8(unsigned int d, bool act) {
    unsigned int m = __ballot_sync(0xffffffffu, act);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const bool bit = (d >> b) & 1u;
        const unsigned int v = __ballot_sync(0xffffffffu, bit);
        m &= bit ? v : ~v;
    }
    return m;
}

// The whole radix top-k of image blockIdx.x (or img) in the CTA's dynamic shared memory: the path the bucket kernels fall
// into for inputs that do not bucket.
template <bool kStaged>
__device__ __forceinline__ void topk_radix_body(unsigned char* smem, const float* __restrict__ scores,
                                                const uint8_t* __restrict__ valid, const float4* __restrict__ boxes, int N,
                                                int k, int kcap, int nchunks, const RsLayout& L,
                                                float* __restrict__ out_scores, int32_t* __restrict__ out_idx,
                                                int32_t* __restrict__ out_cidx, float4* __restrict__ out_boxes,
                                                int32_t* __restrict__ out_count, int img = -1) {
    RsHdr* hd = reinterpret_cast<RsHdr*>(smem);
    unsigned int* vbits = reinterpret_cast<unsigned int*>(smem + L.vbits);
    unsigned int* gpre = reinterpret_cast<unsigned int*>(smem + L.gpre);
    unsigned int* epre = reinterpret_cast<unsigned int*>(smem + L.epre);
    unsigned int* vpre = reinterpret_cast<unsigned int*>(smem + L.vpre);
    unsigned short* whist = reinterpret_cast<unsigned short*>(smem + L.whist);  // [warp][256]
    unsigned int* keyA = reinterpret_cast<unsigned int*>(smem + L.keyA);
    unsigned short* idxA = reinterpret_cast<unsigned short*>(smem + L.idxA);
    unsigned int* keyB = reinterpret_cast<unsigned int*>(smem + L.area2);
    unsigned short* idxB = reinterpret_cast<unsigned short*>(smem + L.area2 + 4 * (size_t)kcap);
    unsigned int* skey = reinterpret_cast<unsigned int*>(smem + L.area2);  // [N] staged keys (dead before the sort)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int lt = (1u << lane) - 1u;
    const int b = img >= 0 ? img : (int)blockIdx.x;
    const float* sc = scores + (size_t)b * N;
    const uint8_t* va = valid ? valid + (size_t)b * N : nullptr;

    // ---- 0. validity words, staged keys ---------------------------------------------------------------
    for (int c0 = warp; c0 < nchunks; c0 += 4 * kRsWarps) {  // 4 chunks per trip: 8 independent loads in flight
        uint8_t v4[4];
        float s4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = (c0 + j * kRsWarps) * 32 + lane;
            v4[j] = (i < N && va) ? va[i] : (uint8_t)1;
            s4[j] = (kStaged && i < N) ? sc[i] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = c0 + j * kRsWarps;
            const int i = c * 32 + lane;
            const unsigned int w = __ballot_sync(0xffffffffu, (i < N) && (v4[j] != 0));
            if (c < nchunks) {
                if (lane == 0) vbits[c] = w;
                if (kStaged && i < N) skey[i] = float_to_ordered(s4[j]);
            }
        }
    }
    if (tid < 256) hd->hist[tid] = 0;
    if (tid == 0) hd->prefix_key = 0;
    __syncthreads();
    auto key_at = [&](int i) -> unsigned int { return kStaged ? skey[i] : float_to_ordered(sc[i]); };
    {
        unsigned int run = 0;
        for (int base = 0; base < nchunks; base += kRsThreads) {
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
    const int keff = min(k, (int)hd->nvalid);
    if (tid == 0) {
        out_count[b] = keff;
        hd->remaining = (unsigned int)keff;
    }
    __syncthreads();

    if (keff > 0) {
        // ---- 1. radix select ----------------------------------------------------------------------------
        // After the first pass only the keys of the threshold bucket matter: they are collected once into a
        // candidate list (scratch in keyA, unordered) and the remaining passes walk the list instead of all N keys.
        unsigned int prefix = 0, pmask = 0;
        unsigned int* lst = keyA;
        int ln = -1;  // < 0: walk all keys
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (ln < 0) {
                for (int c = warp; c < nchunks; c += kRsWarps) {
                    const bool ok = (vbits[c] >> lane) & 1u;
                    const unsigned int key = ok ? key_at(c * 32 + lane) : 0u;
                    const bool in = ok && ((key & pmask) == prefix);
                    const unsigned int d = (key >> shift) & 255u;
                    const unsigned int m = match_digit8(d, in);
                    if (in && lane == __ffs(m) - 1) atomicAdd(&hd->hist[d], (unsigned int)__popc(m));
                }
            } else {
                for (int i0 = warp * 32; i0 < ln; i0 += kRsThreads) {
                    const int i = i0 + lane;
                    const unsigned int key = (i < ln) ? lst[i] : 0u;
                    const bool in = (i < ln) && ((key & pmask) == prefix);
                    const unsigned int d = (key >> shift) & 255u;
                    const unsigned int m = match_digit8(d, in);
                    if (in && lane == __ffs(m) - 1) atomicAdd(&hd->hist[d], (unsigned int)__popc(m));
                }
            }
            __syncthreads();
            if (warp == 0) {  // walk digits from 255 down: the bucket where the cumulative count reaches `remaining`
                const unsigned int need = hd->remaining;
                unsigned int cnt[8], s = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) { cnt[j] = hd->hist[255 - (lane * 8 + j)]; s += cnt[j]; }
                unsigned int inc = s;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                unsigned int before = inc - s;
                if (before < need && inc >= need) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (before < need && before + cnt[j] >= need) {
                            hd->prefix_key = prefix | ((unsigned int)(255 - (lane * 8 + j)) << shift);
                            hd->remaining = need - before;
                            hd->bsize = cnt[j];
                            before = need;
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
            if (tid == 0) hd->lcount = 0u;
            __syncthreads();
            if (ln < 0 && shift > 0 && (int)hd->bsize <= kcap) {  // collect the threshold bucket (uniform branch)
                for (int c = warp; c < nchunks; c += kRsWarps) {
                    const bool ok = (vbits[c] >> lane) & 1u;
                    const unsigned int key = ok ? key_at(c * 32 + lane) : 0u;
                    const bool in = ok && ((key & pmask) == prefix);
                    const unsigned int m = __ballot_sync(0xffffffffu, in);
                    unsigned int basepos = 0;
                    if (lane == 0 && m) basepos = atomicAdd(&hd->lcount, (unsigned int)__popc(m));
                    basepos = __shfl_sync(0xffffffffu, basepos, 0);
                    if (in) lst[basepos + __popc(m & lt)] = key;
                }
                __syncthreads();
                ln = (int)hd->lcount;
            }
        }
        __syncthreads();  // the list (keyA) is dead from here on
        const unsigned int T = prefix;
        const unsigned int take_ties = hd->remaining;

        // ---- 2. order-preserving compaction ---------------------------------------------------------------
        for (int c = warp; c < nchunks; c += kRsWarps) {
            const bool ok = (vbits[c] >> lane) & 1u;
            const unsigned int key = ok ? key_at(c * 32 + lane) : 0u;
            const unsigned int mg = __ballot_sync(0xffffffffu, ok && key > T);
            const unsigned int me = __ballot_sync(0xffffffffu, ok && key == T);
            if (lane == 0) { gpre[c] = __popc(mg); epre[c] = __popc(me); }
        }
        __syncthreads();
        {
            unsigned int run_g = 0, run_e = 0;
            for (int base = 0; base < nchunks; base += kRsThreads) {
                const int c = base + tid;
                const unsigned int vg = (c < nchunks) ? gpre[c] : 0u, ve = (c < nchunks) ? epre[c] : 0u;
                unsigned int tg, te;
                const unsigned int eg = block_exclusive_scan(vg, hd->warp_tmp, &tg);
                const unsigned int ee = block_exclusive_scan(ve, hd->warp_tmp, &te);
                if (c < nchunks) { gpre[c] = run_g + eg; epre[c] = run_e + ee; }
                run_g += tg;
                run_e += te;
            }
        }
        __syncthreads();
        for (int c = warp; c < nchunks; c += kRsWarps) {
            const int i = c * 32 + lane;
            const bool ok = (vbits[c] >> lane) & 1u;
            const unsigned int key = ok ? key_at(i) : 0u;
            const bool gt = ok && key > T, eq = ok && key == T;
            const unsigned int mg = __ballot_sync(0xffffffffu, gt), me = __ballot_sync(0xffffffffu, eq);
            const unsigned int gb = gpre[c] + __popc(mg & lt), eb = epre[c] + __popc(me & lt);
            if (gt || (eq && eb < take_ties)) {
                const unsigned int pos = gb + min(eb, take_ties);
                keyA[pos] = ~key;  // ascending ~key == descending score
                idxA[pos] = (unsigned short)i;
            }
        }
        __syncthreads();

        // ---- 3. stable LSD radix sort of keyA/idxA[0..keff) --------------------------------------------------
        // Thread t owns the `ipt` consecutive pairs [t*ipt, (t+1)*ipt) (ipt odd: conflict-free strided LDS) and a PRIVATE
        // u16 counter per digit, cnt[d][t]: counting and ranking are plain LDS / STS (no ballots, no atomics; the
        // ballot-ranked version spent 60 ALU-pipe instructions per 32 keys and pass).  The exclusive scan over
        // cnt in (digit, thread) order gives every thread its scatter cursor per digit; walking the pairs in order
        // keeps the sort stable.  Only the bits that differ between the selected keys are sorted.
        unsigned int* cnt32 = reinterpret_cast<unsigned int*>(whist);
        const int DB = L.db, ND = 1 << DB;
        const int ipt = ((keff + kRsThreads - 1) / kRsThreads) | 1;
        const int i0 = tid * ipt, i1 = min(i0 + ipt, keff);
        unsigned int orv = 0u, andv = 0xffffffffu;
        for (int i = i0; i < i1; ++i) { const unsigned int kk = keyA[i]; orv |= kk; andv &= kk; }
        orv = __reduce_or_sync(0xffffffffu, orv);
        andv = __reduce_and_sync(0xffffffffu, andv);
        if (lane == 0) { hd->warp_tmp[warp] = orv; hd->hist[warp] = andv; }
        __syncthreads();
        orv = hd->warp_tmp[lane]; andv = hd->hist[lane];
        orv = __reduce_or_sync(0xffffffffu, orv);
        andv = __reduce_and_sync(0xffffffffu, andv);
        __syncthreads();
        const unsigned int vary = orv ^ andv;
        const int lowbit = vary ? (__ffs(vary) - 1) : 0;
        const int nbits = vary ? (32 - __clz(vary) - lowbit) : 0;
        const int npass = (nbits + DB - 1) / DB;
        unsigned int* srcK = keyA;
        unsigned short* srcI = idxA;
        unsigned int* dstK = keyB;
        unsigned short* dstI = idxB;
        unsigned short* mycnt = whist + tid;  // cnt[d][tid] = mycnt[d * kRsThreads]
        for (int pass = 0; pass < npass; ++pass) {
            const int shift = lowbit + pass * DB;
            for (int i = tid; i < ND * kRsThreads / 2; i += kRsThreads) cnt32[i] = 0u;
            __syncthreads();
            for (int i = i0; i < i1; ++i) {
                const unsigned int d = (srcK[i] >> shift) & (unsigned int)(ND - 1);
                mycnt[d * kRsThreads] = (unsigned short)(mycnt[d * kRsThreads] + 1);
            }
            __syncthreads();
            // scan in (digit, thread) order: warp d walks row d of cnt (1024 threads) in 32 coalesced steps with a
            // running warp scan (conflict-free, unlike a per-thread walk of 2^DB strided counters); then the digit bases
            if (warp < ND) {
                unsigned short* row = whist + warp * kRsThreads;
                unsigned int run = 0;
                for (int st = 0; st < kRsThreads / 32; ++st) {
                    const unsigned int v = row[st * 32 + lane];
                    unsigned int inc = v;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
                        if (lane >= o) inc += t;
                    }
                    row[st * 32 + lane] = (unsigned short)(run + inc - v);
                    run += __shfl_sync(0xffffffffu, inc, 31);
                }
                if (lane == 0) hd->hist[warp] = run;  // digit total
            }
            __syncthreads();
            if (warp == 0) {  // exclusive scan of the ND digit totals -> hist[64 + d]
                const unsigned int v = (lane < ND) ? hd->hist[lane] : 0u;
                unsigned int inc = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                hd->hist[64 + lane] = inc - v;
            }
            __syncthreads();
            for (int i = i0; i < i1; ++i) {
                const unsigned int key = srcK[i];
                const unsigned int d = (key >> shift) & (unsigned int)(ND - 1);
                const unsigned int within = mycnt[d * kRsThreads];
                mycnt[d * kRsThreads] = (unsigned short)(within + 1);
                const unsigned int pos = hd->hist[64 + d] + within;
                dstK[pos] = key;
                dstI[pos] = srcI[i];
            }
            __syncthreads();
            unsigned int* tk = srcK; srcK = dstK; dstK = tk;
            unsigned short* ti = srcI; srcI = dstI; dstI = ti;
        }
        if (srcK != keyA) {  // odd number of passes: bring the result back to keyA / idxA
            for (int i = tid; i < keff; i += kRsThreads) { keyA[i] = srcK[i]; idxA[i] = srcI[i]; }
            __syncthreads();
        }
    }

    // ---- 4. write-out (4 independent gathers in flight per thread) ------------------------------------------
    for (int j0 = tid; j0 < k; j0 += 4 * kRsThreads) {
        int ii[4];
        unsigned int kk[4];
        float4 bx[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u * kRsThreads;
            ii[u] = -1;
            kk[u] = 0u;
            if (j < keff) { kk[u] = ~keyA[j]; ii[u] = (int)idxA[j]; }
        }
        if (out_boxes) {
#pragma unroll
            for (int u = 0; u < 4; ++u)
                bx[u] = ii[u] >= 0 ? boxes[(size_t)b * N + ii[u]] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u * kRsThreads;
            if (j >= k) continue;
            const size_t o = (size_t)b * k + j;
            const int i = ii[u];
            if (out_scores) out_scores[o] = i >= 0 ? ordered_to_float(kk[u]) : __uint_as_float(0xff800000u);  // -inf pad
            out_idx[o] = i;
            if (out_cidx) out_cidx[o] = i >= 0 ? (int)(vpre[i >> 5] + __popc(vbits[i >> 5] & ((1u << (i & 31)) - 1u))) : -1;
            if (out_boxes) out_boxes[o] = bx[u];
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// Bucket version (default): ONE histogram pass replaces both the 4-pass radix select and the 6-pass LSD sort.
//   The valid scores are mapped monotonically onto 8192 buckets, bucket(s) = floor((smax - s) * 8192 / (smax - smin))
//   (float arithmetic is monotone under rounding, so a higher score never lands in a later bucket; RPN scores are
//   sigmoid outputs, nearly uniform in value, ~2.6 per bucket).  A shared-memory histogram + one block scan give the
//   bucket b* in which the k-th largest score lies; the (key, index) pairs of buckets <= b* are scattered to their
//   bucket ranges (unordered, atomic cursors) and every pair is ranked inside its bucket on the EXACT total order
//   (ordered key descending, index ascending) -- the same order the radix path produces, so ties and the cut inside b*
//   are bit-identical.  Inputs that do not bucket well (non-finite range, a bucket of > kBucketMax, more than `cap`
//   stored pairs: e.g. all scores equal) are redone on the radix path by CTA 0 of the image alone.
//
// An image runs on a thread-block CLUSTER of S = 1 or 2 CTAs (small batches: one CTA per image leaves most SMs idle -- a
// single image ran on ONE SM).  CTA r of the S CTAs owns a contiguous range of the 32-anchor chunks: it loads / stages /
// histograms its own scores; the S histograms are merged through distributed shared memory (every CTA reads the peers'
// counts and derives the same bucket starts, plus how many pairs the lower-ranked CTAs put in every bucket: its first
// scatter cursors); pairs are scattered straight into the shared memory of the CTA that OWNS their bucket (buckets are
// dealt to the CTAs by their start position, whole buckets only), which ranks them and writes its contiguous piece of
// the output row.  Same buckets, same exact total order for every S: identical results.
constexpr int kBuckets = 8192;
constexpr int kBucketMax = 192;
constexpr int kBucketSlack = 1024;  // pairs stored beyond k (the rest of bucket b*)

struct BkXch {
    float mn, mx;
    unsigned int nvalid, bad;
};
constexpr int kBkMaxCluster = 8;

struct BkcHdr {
    unsigned int warp_tmp[kRsWarps];
    unsigned int red[kRsWarps];
    unsigned int bstar, stored, bad;
    unsigned int obase[kBkMaxCluster + 1];  // first output position owned by CTA o (0xffffffff: none)
    BkXch xch[kBkMaxCluster];
};

struct BkcLayout {
    size_t vbits, vpre, hist, start, sval, keyA, idxA, total;
    int cper, capS;
};
constexpr BkcLayout bkc_layout(int cap, int nchunks, int S, bool staged) {
    BkcLayout L{};
    L.cper = (nchunks + S - 1) / S;
    // pairs a CTA may own: a single CTA owns all `stored <= cap`; with S > 1 an owner may take up to one bucket
    // (<= kBucketMax pairs) beyond cap / S
    L.capS = S == 1 ? cap : (cap + S - 1) / S + 256;
    size_t o = up16(sizeof(BkcHdr));
    L.vbits = o; o += 4 * (size_t)L.cper;
    L.vpre = o;  o = up16(o + 4 * (size_t)L.cper);
    L.hist = o;  o += 4 * (size_t)kBuckets;
    L.start = o; o = up16(o + 2 * (size_t)(kBuckets + 1));
    L.sval = o;  o = up16(o + (staged ? 4 * 32 * (size_t)L.cper : 0));
    L.keyA = o;  o += 4 * (size_t)L.capS;
    L.idxA = o;  o = up16(o + 2 * (size_t)L.capS);
    L.total = o;
    return L;
}

// kStaged: scores staged in shared memory, or re-read from global / L2 in the two passes.  kCluster: launched with S > 1;
// without it (S = 1) the cluster barriers and distributed-shared-memory mappings below are plain CTA barriers and shared
// accesses -- a cluster barrier carries a memory fence and an L1 invalidate, and a mapped access is a generic one, which
// cost one CTA per image 22-32 % of its time (tools/topk_latency.py, B200 at 1000 W)
template <bool kStaged, bool kCluster>
__global__ void __launch_bounds__(kRsThreads, 1)
    topk_bucket_kernel(const float* __restrict__ scores, const uint8_t* __restrict__ valid,
                       const float4* __restrict__ boxes, int N, int k, int cap, int nchunks,
                       float* __restrict__ out_scores, int32_t* __restrict__ out_idx, int32_t* __restrict__ out_cidx,
                       float4* __restrict__ out_boxes, int32_t* __restrict__ out_count, RsLayout L, int kcap,
                       BkcLayout Lc) {
    namespace cg = cooperative_groups;
    extern __shared__ __align__(16) unsigned char smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int S = kCluster ? (int)cluster.num_blocks() : 1, rank = kCluster ? (int)cluster.block_rank() : 0;
    auto csync = [&] { if (kCluster) cluster.sync(); else __syncthreads(); };
    auto peer = [&](auto* p, int r) { return kCluster ? cluster.map_shared_rank(p, r) : p; };
    const int b = (int)blockIdx.x / S;
    BkcHdr* hd = reinterpret_cast<BkcHdr*>(smem);
    unsigned int* vbits = reinterpret_cast<unsigned int*>(smem + Lc.vbits);
    unsigned int* vpre = reinterpret_cast<unsigned int*>(smem + Lc.vpre);
    unsigned int* hist = reinterpret_cast<unsigned int*>(smem + Lc.hist);
    unsigned short* start = reinterpret_cast<unsigned short*>(smem + Lc.start);
    float* sval = reinterpret_cast<float*>(smem + Lc.sval);
    unsigned int* keyA = reinterpret_cast<unsigned int*>(smem + Lc.keyA);
    unsigned short* idxA = reinterpret_cast<unsigned short*>(smem + Lc.idxA);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* sc = scores + (size_t)b * N;
    const uint8_t* va = valid ? valid + (size_t)b * N : nullptr;
    const int c_lo = min(nchunks, rank * Lc.cper), c_hi = min(nchunks, c_lo + Lc.cper);

    // ---- 0. own chunks: validity words, staged scores, min / max; zeroed histogram ---------------------------------
    float lmin = 3.0e38f, lmax = -3.0e38f;
    bool lbad = false;
    constexpr int kLd = 4;
    for (int c0 = c_lo + warp; c0 < c_hi; c0 += kLd * kRsWarps) {
        uint8_t v4[kLd];
        float s4[kLd];
#pragma unroll
        for (int j = 0; j < kLd; ++j) {
            const int c = c0 + j * kRsWarps;
            const int i = c * 32 + lane;
            const bool in = c < c_hi && i < N;
            v4[j] = (in && va) ? va[i] : (uint8_t)(in ? 1 : 0);
            s4[j] = in ? sc[i] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < kLd; ++j) {
            const int c = c0 + j * kRsWarps;
            const int i = c * 32 + lane;
            const bool ok = (c < c_hi) && (i < N) && (v4[j] != 0);
            const unsigned int w = __ballot_sync(0xffffffffu, ok);
            if (c < c_hi) {
                if (lane == 0) vbits[c - c_lo] = w;
                if (kStaged) sval[(c - c_lo) * 32 + lane] = s4[j];
                if (ok) {
                    lbad |= !(fabsf(s4[j]) <= 3.0e38f);
                    lmin = fminf(lmin, s4[j]);
                    lmax = fmaxf(lmax, s4[j]);
                }
            }
        }
    }
    for (int i = tid; i < kBuckets; i += kRsThreads) hist[i] = 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    const bool wbad = __any_sync(0xffffffffu, lbad);   // (lmin / lmax: the warp's values, in every lane)
    if (tid == 0) hd->bad = 0u;
    __syncthreads();
    if (wbad && lane == 0) hd->bad = 1u;
    unsigned int nvalid_local = 0;
    {   // exclusive prefix of the valid counts of the own chunks
        unsigned int run = 0;
        for (int base = 0; base < c_hi - c_lo; base += kRsThreads) {
            const int c = base + tid;
            const unsigned int v = (c < c_hi - c_lo) ? __popc(vbits[c]) : 0u;
            unsigned int tot;
            const unsigned int ex = block_exclusive_scan(v, hd->warp_tmp, &tot);
            if (c < c_hi - c_lo) vpre[c] = run + ex;
            run += tot;
        }
        nvalid_local = run;
    }
    __syncthreads();
    {   // block min / max (after the scan: it uses warp_tmp), then this CTA's summary into every CTA of the cluster
        float a = lmin, z = lmax;
        if (lane == 0) { hd->warp_tmp[warp] = __float_as_uint(a); hd->red[warp] = __float_as_uint(z); }
        __syncthreads();
        if (warp == 0) {
            a = __uint_as_float(hd->warp_tmp[lane]);
            z = __uint_as_float(hd->red[lane]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                a = fminf(a, __shfl_xor_sync(0xffffffffu, a, o));
                z = fmaxf(z, __shfl_xor_sync(0xffffffffu, z, o));
            }
            if (lane < S) {  // this CTA's summary into every CTA's exchange array
                BkXch x;
                x.mn = a; x.mx = z; x.nvalid = nvalid_local; x.bad = hd->bad;
                *peer(&hd->xch[rank], lane) = x;
            }
        }
    }
    csync();
    float smin = 3.0e38f, smax = -3.0e38f;
    unsigned int nvalid = 0, anybad = 0;
    for (int r = 0; r < S; ++r) {
        const BkXch x = hd->xch[r];
        smin = fminf(smin, x.mn);
        smax = fmaxf(smax, x.mx);
        nvalid += x.nvalid;
        anybad |= x.bad;
    }
    const int keff = min(k, (int)nvalid);
    const float scale = (float)kBuckets / (smax - smin);
    bool handover = anybad != 0u || (keff > 0 && !(scale <= 3.0e38f));
    auto bucket_of = [&](float s) { return min(kBuckets - 1, (int)((smax - s) * scale)); };
    auto score_at = [&](int i) -> float { return kStaged ? sval[i - c_lo * 32] : sc[i]; };

    if (keff > 0 && !handover) {
        // ---- 1. histogram of the own valid scores ----------------------------------------------------------------
        for (int c = c_lo + warp; c < c_hi; c += kRsWarps) {
            const int i = c * 32 + lane;
            if ((vbits[c - c_lo] >> lane) & 1u) atomicAdd(&hist[bucket_of(score_at(i))], 1u);
        }
        csync();  // every CTA's counts are complete
        // ---- 2. merged counts -> bucket starts (same in every CTA), pairs of the lower-ranked CTAs in every bucket ----
        constexpr int kPerT = kBuckets / kRsThreads;
        unsigned int o4[kPerT];
        {
            unsigned int h4[kPerT], t4 = 0;
#pragma unroll
            for (int q = 0; q < kPerT; ++q) { h4[q] = 0; o4[q] = 0; }
            for (int r = 0; r < S; ++r) {
                const uint4* ph = reinterpret_cast<const uint4*>(peer(hist, r) + kPerT * tid);
#pragma unroll
                for (int q4 = 0; q4 < kPerT / 4; ++q4) {
                    const uint4 v = ph[q4];
                    h4[4 * q4 + 0] += v.x; h4[4 * q4 + 1] += v.y; h4[4 * q4 + 2] += v.z; h4[4 * q4 + 3] += v.w;
                    if (r < rank) { o4[4 * q4 + 0] += v.x; o4[4 * q4 + 1] += v.y; o4[4 * q4 + 2] += v.z; o4[4 * q4 + 3] += v.w; }
                }
            }
#pragma unroll
            for (int q = 0; q < kPerT; ++q) t4 += h4[q];
            unsigned int tot;
            unsigned int run = block_exclusive_scan(t4, hd->warp_tmp, &tot);
            unsigned int big = 0;
#pragma unroll
            for (int q = 0; q < kPerT; ++q) {
                start[kPerT * tid + q] = (unsigned short)min(run, 65535u);
                if (run < (unsigned int)keff) {
                    big = max(big, h4[q]);
                    if (run + h4[q] >= (unsigned int)keff) { hd->bstar = kPerT * tid + q; hd->stored = run + h4[q]; }
                }
                run += h4[q];
            }
            if (tid == kRsThreads - 1) start[kBuckets] = (unsigned short)min(run, 65535u);
            big = __reduce_max_sync(0xffffffffu, big);
            __syncthreads();
            if (lane == 0) hd->red[warp] = big;
            if (tid <= kBkMaxCluster) hd->obase[tid] = 0xffffffffu;
            __syncthreads();
            if (warp == 0) {
                big = __reduce_max_sync(0xffffffffu, hd->red[lane]);
                if (lane == 0 && (big > kBucketMax || hd->stored > (unsigned int)cap)) hd->bad = 1u;
            }
            __syncthreads();
            handover = hd->bad != 0u;
        }
        csync();  // every CTA has read the counts: they become the scatter cursors, past the lower ranks' pairs
        uint4* cur = reinterpret_cast<uint4*>(hist + kPerT * tid);
#pragma unroll
        for (int q4 = 0; q4 < kPerT / 4; ++q4)
            cur[q4] = make_uint4(o4[4 * q4 + 0], o4[4 * q4 + 1], o4[4 * q4 + 2], o4[4 * q4 + 3]);
    }
    if (handover) {  // cluster-uniform: CTA 0 redoes the image alone on the radix path
        csync();
        if (rank != 0) return;
        if (L.staged) topk_radix_body<true>(smem, scores, valid, boxes, N, k, kcap, nchunks, L, out_scores, out_idx, out_cidx,
                                            out_boxes, out_count, b);
        else topk_radix_body<false>(smem, scores, valid, boxes, N, k, kcap, nchunks, L, out_scores, out_idx, out_cidx,
                                    out_boxes, out_count, b);
        return;
    }
    if (rank == 0 && tid == 0) out_count[b] = keff;
    if (keff > 0) {
        const int bstar = (int)hd->bstar;
        const unsigned int stored = hd->stored;
        const unsigned int per = (stored + (unsigned int)S - 1u) / (unsigned int)S;  // output positions per owner
        auto owner_of = [&](unsigned int pos) { return min((unsigned int)S - 1u, pos / per); };
        // first position of every owner (whole buckets: a bucket belongs to the owner of its start)
        for (int bk = tid; bk <= bstar; bk += kRsThreads) {
            const unsigned int o = owner_of(start[bk]);
            if (bk == 0 || owner_of(start[bk - 1]) != o) hd->obase[o] = start[bk];
        }
        __syncthreads();
        // ---- 3. scatter the own pairs of buckets <= b* into their owners' arrays ------------------------------------
        for (int c = c_lo + warp; c < c_hi; c += kRsWarps) {
            const int i = c * 32 + lane;
            if ((vbits[c - c_lo] >> lane) & 1u) {
                const float sv = score_at(i);
                const int bk = bucket_of(sv);
                if (bk <= bstar) {
                    const unsigned int s0 = start[bk];
                    const unsigned int pos = s0 + atomicAdd(&hist[bk], 1u);
                    const unsigned int o = owner_of(s0);
                    const unsigned int li = pos - hd->obase[o];
                    peer(keyA, o)[li] = float_to_ordered(sv);
                    peer(idxA, o)[li] = (unsigned short)i;
                }
            }
        }
        csync();
        // ---- 4. rank the own range and write its piece of the output row: every stored pair counts the pairs of ITS
        //         bucket that precede it in the exact total order (ordered key descending, index ascending); start[bucket]
        //         + that count is its final rank -- no sorted copy in shared memory, no separate write-out pass.  One
        //         thread per pair: ~2.6 pairs per bucket, so the loops are a few iterations long and every lane is busy (a
        //         thread sorting whole buckets left the warp waiting for its largest bucket: 19 k of 59 k cycles).
        const unsigned int my0 = hd->obase[rank];
        unsigned int my1 = stored;
        for (int o = rank + 1; o < S; ++o)
            if (hd->obase[o] != 0xffffffffu) { my1 = hd->obase[o]; break; }
        const int cnt = my0 == 0xffffffffu ? 0 : (int)(my1 - my0);
        // the scatter cursors are dead: their 32 KB stage the output piece (u16 anchor index per rank, keff <= 16384), so
        // that the global writes of the index row are coalesced instead of one sector per pair
        unsigned short* orow = reinterpret_cast<unsigned short*>(hist);
        __syncthreads();
        for (int p2 = tid; p2 < cnt; p2 += kRsThreads) {
            const unsigned int ku = keyA[p2];
            const unsigned int ki = idxA[p2];
            const int bk = bucket_of(ordered_to_float(ku));
            const int s0 = (int)start[bk] - (int)my0, s1 = (int)start[bk + 1] - (int)my0;
            int r = s0;
            for (int a = s0; a < s1; ++a) {
                const unsigned int ka = keyA[a];
                r += (ka > ku || (ka == ku && (unsigned int)idxA[a] < ki)) ? 1 : 0;
            }
            const int g = r + (int)my0;  // final rank
            if (g < keff) {
                const size_t oo = (size_t)b * k + g;
                const int i = (int)ki;
                orow[r] = (unsigned short)ki;
                if (out_scores) out_scores[oo] = ordered_to_float(ku);
                if (out_cidx) {
                    const int hc = i >> 5, hr = min(S - 1, hc / Lc.cper);   // the anchor's home CTA holds its validity words
                    const unsigned int hb = peer(vbits, hr)[hc - hr * Lc.cper];
                    const unsigned int hp = peer(vpre, hr)[hc - hr * Lc.cper];
                    unsigned int base_r = 0;
                    for (int q = 0; q < hr; ++q) base_r += hd->xch[q].nvalid;
                    out_cidx[oo] = (int)(base_r + hp + __popc(hb & ((1u << (i & 31)) - 1u)));
                }
                if (out_boxes) out_boxes[oo] = boxes[(size_t)b * N + i];
            }
        }
        __syncthreads();
        {
            int32_t* orow_g = out_idx + (size_t)b * k + my0;
            const int lim = min(cnt, keff - (int)my0);
            for (int j2 = tid; j2 < lim; j2 += kRsThreads) orow_g[j2] = (int32_t)orow[j2];
        }
    }
    // ---- 5. padding past the count (dealt over the cluster) ---------------------------------------------------------
    for (int j2 = keff + rank * kRsThreads + tid; j2 < k; j2 += S * kRsThreads) {
        const size_t oo = (size_t)b * k + j2;
        out_idx[oo] = -1;
        if (out_scores) out_scores[oo] = __uint_as_float(0xff800000u);
        if (out_cidx) out_cidx[oo] = -1;
        if (out_boxes) out_boxes[oo] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    csync();  // nobody leaves while a peer may still read its shared memory
}

constexpr size_t kSmemLimit = 227 * 1024;
// The largest shape topk_radix_launch takes (N 65536, k 16384) fits the bucket kernel unstaged at one CTA per image (two
// CTAs per image need less), so every shape that has a radix layout runs the bucket kernel, with the radix path as its
// hand-over.
static_assert(bkc_layout(16384 + kBucketSlack, 65536 / 32, 1, false).total <= kSmemLimit,
              "the bucket kernel must fit every shape of the fast path");

// Returns FRR_OK when the launch was done, 1 when the shape is outside the fast path (caller falls back).
int topk_radix_launch(const float* scores, const uint8_t* valid, const float* boxes, int B, int N, int k,
                      float* out_scores, int32_t* out_idx, int32_t* out_cidx, float* out_boxes, int32_t* out_count,
                      frr_stream_t stream, int cluster_hint) {
    if (N > 65536 || k > 16384) return 1;
    const size_t limit = kSmemLimit;
    const int kcap = (k + 31) & ~31;
    const int nchunks = (N + 31) / 32;
    RsLayout L = rs_layout(N, kcap, nchunks, true, 5);
    if (L.total > limit) L = rs_layout(N, kcap, nchunks, true, 4);
    if (L.total > limit) L = rs_layout(N, kcap, nchunks, false, 5);
    if (L.total > limit) L = rs_layout(N, kcap, nchunks, false, 4);
    if (L.total > limit) return 1;
    // bucket kernel, with the radix path compiled in as its hand-over
    const int cap = kcap + kBucketSlack;
    // CTAs per image: small batches (B * S <= SMs) spread an image over a cluster; cluster_hint = 1 keeps one CTA per
    // image (the least SM time: several batches in flight).  Two CTAs per image when they fit: 26-27 us against 29-39 us;
    // more do not pay (measured: 4 CTAs equal 2, 8 CTAs take 37-44 us -- five cluster barriers and an S-fold histogram
    // merge against ~25 us of divisible work)
    const int S = cluster_hint != 1 && (long)B * 2 <= num_sms() ? 2 : 1;
    BkcLayout Lc = bkc_layout(cap, nchunks, S, true);
    const bool staged = Lc.total <= limit;
    if (!staged) Lc = bkc_layout(cap, nchunks, S, false);
    auto kern = S > 1 ? (staged ? topk_bucket_kernel<true, true> : topk_bucket_kernel<false, true>)
                      : (staged ? topk_bucket_kernel<true, false> : topk_bucket_kernel<false, false>);
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * S), 1, 1);
    cfg.blockDim = dim3((unsigned)kRsThreads, 1, 1);
    cfg.dynamicSmemBytes = Lc.total > L.total ? Lc.total : L.total;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = S > 1 ? 1 : 0;  // one CTA per image: a plain launch
    FRR_CUDA(cudaLaunchKernelEx(&cfg, kern, scores, valid, (const float4*)boxes, N, k, cap, nchunks, out_scores, out_idx,
                                out_cidx, (float4*)out_boxes, out_count, L, kcap, Lc));
    count_launch();
    FRR_CHECK_LAUNCH("topk_bucket_kernel");
    return FRR_OK;
}

}  // namespace frr
