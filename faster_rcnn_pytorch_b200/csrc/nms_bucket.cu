// N1 for the RPN proposal layer (models/model.py:53-55: nms(roi, softmax, 0.7), keep[:2000|300]) on boxes clamped to
// [0,1] (models/model.py:34): greedy NMS in LARGE chunks with every pair test restricted to admissible buckets.
//
// One thread-block cluster per image; every CTA holds the WHOLE kept list in shared memory, the candidates of a chunk
// (up to 2048 at 1024 threads, 1024 below, in score order) are dealt round-robin to the CTAs.  Per chunk:
//   A-C  the kept list is re-bucketed (counting sort by key = (x bin, y bin, area class), see nms_common.cuh) and
//        every CTA orders its own candidates by key, so the lanes of a warp walk ranges of similar length;
//   D    screen: a candidate walks only the kept boxes whose keys are admissible for it -- IoU >= thr needs an area
//        ratio in [thr, 1/thr], an x-centre distance <= fx * width and a y-centre distance <= fx * height, all exact
//        necessary conditions -- with the division-free screen; one screen hit is confirmed with the exact
//        torchvision arithmetic.  Dead candidates are flagged in every CTA through distributed shared memory (one
//        cluster barrier);
//   E-G  the chunk's survivors are bucketed the same way, in a DETERMINISTIC order (key, then score position: an
//        unordered counting-sort scatter followed by a rank inside the bucket), so every CTA builds the same array;
//   H    suppression pairs among the survivors: the survivor at bucketed position p walks only the admissible
//        positions ABOVE p (both pruning rules are symmetric in the pair, so every pair that can suppress is met
//        exactly once, from its lower position; positions are dealt round-robin to the CTAs).  Screen hits are parked
//        in a per-thread ring and confirmed with the exact test after the walk; a confirmed pair becomes an EDGE
//        (later, earlier in score order), appended to the CTA's edge region and mirrored into every CTA (second
//        cluster barrier).  A survivor whose edges do not fit is flagged and decided by a walk of its own instead;
//   I    fix-point over the edges (every CTA, redundantly): a survivor is removed as soon as one predecessor is kept
//        and kept once all its predecessors are removed -- edge pass + node pass per round, 3-6 rounds on RPN boxes;
//   J    the kept survivors are appended in score order (block scan), the walk stops at max_keep.
// Against the keep-list kernel of nms.cu (chunks of 256, ~10 barriers each): 3-4 chunks instead of 18-25, i.e. 3-4
// latency chains per image, and 0.1-0.2 M pair tests per image instead of 4.6 M.  The keep list is the one of
// torchvision's CPU kernel bit for bit: every decision is taken by suppress_exact(); screen and buckets only skip
// pairs that provably cannot suppress.  tests/nms_model.py restates this algorithm on the CPU, tests/nms_cell_model.py
// its keys and walk order.
#include <cooperative_groups.h>

#include "nms_common.cuh"

namespace cg = cooperative_groups;

namespace frr {

constexpr int kBkListCap = 2048;   // kept-list capacity (max_keep <= 2047)
constexpr int kBkBins = 3;         // cells of a walk whose bounds are prefetched (more: tail loop)
constexpr int kBkUpBins = 2;       // same for the upward walk (cells after the own one)
constexpr int kBkHits = 4;         // screen hits a thread parks per walk before it falls back to the slow walk

// Largest chunk of a CTA of `threads` threads.  Below 1024 threads the chunk arrays are sized for 1024 candidates, which
// brings the layout of the 512-thread form under half an SM's shared memory: two CTAs (two images) share an SM and
// one's barrier-bound phases overlap the other's pair tests.  Results never depend on the chunk size.
__host__ __device__ constexpr int bk_chunk_cap(int threads) { return threads >= 1024 ? kBkChunk : kBkChunk / 2; }

// y bins of the bucket key of a launch: 8 x 4 (x, y) cells at 1024 threads with one or two CTAs per image.  8 x 8 cells
// test 2.7x fewer pairs than 8 x bins but walk 7.4 instead of 2.3 cells per candidate and measured slower; 8 x 4 (4.8
// cells, 2.1x fewer pairs) is the fastest grid there (DESIGN.md 4.3).  The clusters of 4-16 CTAs of the single-image form,
// whose CTAs walk a few hundred candidates each, measured slower with cells and key by x bin only, and so does the
// 512-thread layout, which has no room for the larger per-key arrays next to its two-per-SM budget.  Results never
// depend on the grid.
__host__ __device__ constexpr int bk_ybins(int threads, int S) { return threads >= 1024 && S <= 2 ? 4 : 1; }

template <int kThreads, int kYBins>
struct BkSmem {
    using G = BkGrid<kYBins>;
    static constexpr int kCap = bk_chunk_cap(kThreads);
    static constexpr int kEdgeCap = 2 * kCap;  // edges per chunk over the whole cluster (each CTA owns kEdgeCap / S)
    static constexpr int kKeyPer = (G::kKeys + 2 + kThreads - 1) / kThreads;  // keys per thread of a block scan
    static constexpr int kKeyCap = kKeyPer * kThreads;  // padded length of the per-key arrays ([kKeys + 1]: length)
    float4 lbox[kBkListCap];  // kept list: bucketed by key in phase C, new keeps appended in score order in phase J
    float la[kBkListCap];     // its c2-scaled screening areas
    float4 sbox[kCap];        // the chunk's survivors, bucketed (phase G)
    float ssa[kCap];
    float4 cbox[kCap];  // the chunk's candidates, score order
    float csa[kCap];    // c2-scaled screening areas (NaN = always take the exact path)
    unsigned int hist[kKeyCap];   // phases A-C: key histogram, then scatter cursors, of the kept list (low 16 bits) and
                                  // of this CTA's candidates (high 16 bits): both counts are <= kBkChunk
    unsigned int shist[kKeyCap];  // phases E-G: the same for the survivors
    unsigned short lstart[kKeyCap];  // first list position of key s; [kKeys + 1] = list length
    unsigned short sstart[kKeyCap];  // same for the bucketed survivors
    unsigned int edges[kEdgeCap];    // (later << 16) | earlier, chunk-local positions; region r belongs to CTA r
    unsigned int ecount[kMaxCluster];
    unsigned int ecursor;
    unsigned int work[2];  // dynamic dealing of the items of phases D and H
    unsigned int warp_tmp[32];
    unsigned short ckey[kCap];
    unsigned short cord[kCap];  // this CTA's candidates ordered by key
    unsigned short sidx[kCap];  // bucketed survivor -> chunk position
    unsigned short hitbuf[kThreads * kBkHits];  // per-thread ring of screen hits (phase H): bucketed survivor positions
    unsigned char cstate[2][kCap];  // [chunk parity]: 0 undecided, 1 kept, 2 removed
    unsigned char pend[kCap];
    unsigned char ovf[kCap];
};

// Whole block: in-place exclusive scan of hist[0 .. kPer * kThreads) (kPer consecutive entries per thread), the low
// 16 bits of the result also written as start offsets.  Entries past kKeys + 1 are zero.
template <int kThreads, int kPer>
__device__ __forceinline__ void bk_scan_keys(unsigned int* hist, unsigned short* start, unsigned int* warp_tmp) {
    const int e0 = threadIdx.x * kPer;
    unsigned int h[kPer], t = 0;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        h[q] = hist[e0 + q];
        t += h[q];
    }
    unsigned int total;
    unsigned int run = block_exclusive_scan(t, warp_tmp, &total);
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        hist[e0 + q] = run;
        start[e0 + q] = (unsigned short)run;
        run += h[q];
    }
}

struct BkAdm {
    int c_lo, c_hi, x_lo, x_hi, y_lo, y_hi;
};
// Admissible keys of a box: area classes of [alo * A, ahi * A] (IoU <= min / max area), x bins of cx -+ fx * w and
// y bins of cy -+ fx * h.
template <class G>
__device__ __forceinline__ BkAdm bk_admissible(const float4& cbx, const NmsThr& thr) {
    BkAdm r;
    const float a = box_area(cbx);
    r.c_lo = G::cls(a * thr.alo);
    r.c_hi = G::cls(a * thr.ahi);
    const float cx = 0.5f * (cbx.x + cbx.z);
    const float rx = thr.fx * (cbx.z - cbx.x) * 1.0001f + 2.0e-6f;
    r.x_lo = G::xbin(cx - rx);
    r.x_hi = G::xbin(cx + rx);
    if (G::kY > 1) {
        const float cy = 0.5f * (cbx.y + cbx.w);
        const float ry = thr.fx * (cbx.w - cbx.y) * 1.0001f + 2.0e-6f;
        r.y_lo = G::ybin(cy - ry);
        r.y_hi = G::ybin(cy + ry);
    } else {
        r.y_lo = r.y_hi = 0;
    }
    return r;
}

// The next admissible cell in key order (y minor).
__device__ __forceinline__ void bk_next_cell(const BkAdm& ad, int& xb, int& yb) {
    if (++yb > ad.y_hi) {
        yb = ad.y_lo;
        ++xb;
    }
}

// Calls f(k) for the positions of the admissible area classes of every admissible cell from (xb, yb) on, in key order;
// this thread takes every nsub-th position of each range, starting at sub.  The bounds of the first kPre cells are
// fetched before the first walk (independent loads).
template <class G, int kPre, class F>
__device__ __forceinline__ void bk_walk_cells(const unsigned short* __restrict__ start, const BkAdm& ad, int xb, int yb,
                                              int sub, int nsub, F& f) {
    int lo_b[kPre], hi_b[kPre];
#pragma unroll
    for (int q = 0; q < kPre; ++q) {
        const int c0 = (min(xb, G::kX - 1) * G::kY + yb) * G::kClasses;
        lo_b[q] = start[c0 + ad.c_lo];
        hi_b[q] = (xb <= ad.x_hi) ? (int)start[c0 + ad.c_hi + 1] : 0;
        bk_next_cell(ad, xb, yb);
    }
#pragma unroll
    for (int q = 0; q < kPre; ++q) {
#pragma unroll 2
        for (int k = lo_b[q] + sub; k < hi_b[q]; k += nsub) f(k);
    }
    for (; xb <= ad.x_hi; bk_next_cell(ad, xb, yb)) {  // wide boxes / low thresholds: more cells
        const int c0 = (xb * G::kY + yb) * G::kClasses;
        const int lo = start[c0 + ad.c_lo], hi = start[c0 + ad.c_hi + 1];
        for (int k = lo + sub; k < hi; k += nsub) f(k);
    }
}

// Calls f(k) for every position k of a bucketed array (start offsets `start`) whose key is admissible for the box
// (cbx, screening area ca); this thread takes every nsub-th position of each range, starting at sub.
template <class G, class F>
__device__ __forceinline__ void bk_walk(const unsigned short* __restrict__ start, const float4& cbx, float ca,
                                        const NmsThr& thr, int sub, int nsub, F&& f) {
    if (ca == ca) {
        const BkAdm ad = bk_admissible<G>(cbx, thr);
        const int lo2 = start[G::kKeys], hi2 = start[G::kKeys + 1];  // boxes that must always be tested
        bk_walk_cells<G, kBkBins>(start, ad, ad.x_lo, ad.y_lo, sub, nsub, f);
        for (int k = lo2 + sub; k < hi2; k += nsub) f(k);
    } else {  // no usable screening area: everything
        const int hi = start[G::kKeys + 1];
        for (int k = sub; k < hi; k += nsub) f(k);
    }
}

// Upward half of bk_walk for the element at position p of the bucketed array (its key: own_key): positions above p
// only -- the rest of the own cell's classes up to c_hi, then the admissible cells after the own one in key order
// (the later y bins of the own x bin, then every admissible cell of the higher x bins), then the always-tested
// bucket.  Both pruning rules are symmetric in a pair, so a pair that can suppress is found from its lower position.
template <class G, class F>
__device__ __forceinline__ void bk_walk_up(const unsigned short* __restrict__ start, int p, int own_key, const float4& cbx,
                                           float ca, const NmsThr& thr, int sub, int nsub, F&& f) {
    const int total = start[G::kKeys + 1];
    if (ca == ca) {
        const BkAdm ad = bk_admissible<G>(cbx, thr);
        const int cell = own_key / G::kClasses;
        const int hi0 = start[cell * G::kClasses + ad.c_hi + 1];
        const int lo2 = start[G::kKeys];
#pragma unroll 2
        for (int k = p + 1 + sub; k < hi0; k += nsub) f(k);
        int xb = cell / G::kY, yb = cell % G::kY;
        bk_next_cell(ad, xb, yb);
        bk_walk_cells<G, kBkUpBins>(start, ad, xb, yb, sub, nsub, f);
        for (int k = lo2 + sub; k < total; k += nsub) f(k);
    } else {  // the always-tested bucket is the last one
        for (int k = p + 1 + sub; k < total; k += nsub) f(k);
    }
}

// Same positions and the same dealing to the sub-threads as bk_walk, one compact copy of the code (rare paths: kept
// out of the hot loops' footprint).  f returns true to stop.
template <class G, class F>
__device__ __noinline__ void bk_walk_slow(const unsigned short* __restrict__ start, float4 cbx, float ca, NmsThr thr,
                                          int sub, int nsub, F f) {
    int lo2 = 0;
    const int hi2 = start[G::kKeys + 1];
    if (ca == ca) {
        const BkAdm ad = bk_admissible<G>(cbx, thr);
        for (int xb = ad.x_lo; xb <= ad.x_hi; ++xb)
            for (int yb = ad.y_lo; yb <= ad.y_hi; ++yb) {
                const int c0 = (xb * G::kY + yb) * G::kClasses;
                const int lo = start[c0 + ad.c_lo], hi = start[c0 + ad.c_hi + 1];
                for (int k = lo + sub; k < hi; k += nsub)
                    if (f(k)) return;
            }
        lo2 = start[G::kKeys];
    }
    for (int k = lo2 + sub; k < hi2; k += nsub)
        if (f(k)) return;
}

// bk_walk_up's positions with the same dealing to the sub-threads, one compact copy (a thread whose hit ring
// overflowed re-walks exactly ITS share).
template <class G, class F>
__device__ __noinline__ void bk_walk_up_slow(const unsigned short* __restrict__ start, int p, int own_key, float4 cbx,
                                             float ca, NmsThr thr, int sub, int nsub, F f) {
    const int total = start[G::kKeys + 1];
    if (ca == ca) {
        const BkAdm ad = bk_admissible<G>(cbx, thr);
        const int cell = own_key / G::kClasses;
        const int hi0 = start[cell * G::kClasses + ad.c_hi + 1];
        for (int k = p + 1 + sub; k < hi0; k += nsub) f(k);
        int xb = cell / G::kY, yb = cell % G::kY;
        for (bk_next_cell(ad, xb, yb); xb <= ad.x_hi; bk_next_cell(ad, xb, yb)) {
            const int c0 = (xb * G::kY + yb) * G::kClasses;
            const int lo = start[c0 + ad.c_lo], hi = start[c0 + ad.c_hi + 1];
            for (int k = lo + sub; k < hi; k += nsub) f(k);
        }
        for (int k = start[G::kKeys] + sub; k < total; k += nsub) f(k);
    } else {
        for (int k = p + 1 + sub; k < total; k += nsub) f(k);
    }
}

// A confirmed suppression pair of the chunk: the later box (chunk position i) has the earlier one (j) as predecessor.
// Appended to this CTA's edge region (mirrored into the other CTAs after the phase); if the region is full the later
// box is flagged and decides from a walk of its own in the fix-point.
template <class Smem>
__device__ __forceinline__ void bk_push_edge(Smem* sm, int i, int j, int rank, int ecap) {
    const unsigned int e = atomicAdd(&sm->ecursor, 1u);
    if (e < (unsigned int)ecap) sm->edges[rank * ecap + e] = ((unsigned int)i << 16) | (unsigned int)j;
    else sm->ovf[i] = 1;
}

// A warp takes the next 32 / nsub items of a phase (dynamic dealing: walks differ in length by more than 10x).
__device__ __forceinline__ int bk_grab(unsigned int* cursor, int per_warp, int lane) {
    int q0 = 0;
    if (lane == 0) q0 = (int)atomicAdd(cursor, (unsigned int)per_warp);
    return __shfl_sync(0xffffffffu, q0, 0);
}

template <int kThreads, int kYBins>
__global__ void __launch_bounds__(kThreads, kThreads <= 512 ? 2 : 1)
    nms_bucket_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ counts, int n, int max_keep, NmsThr thr,
                      int32_t* __restrict__ keep, int32_t* __restrict__ keep_count, float4* __restrict__ out_boxes,
                      const int32_t* __restrict__ gather_idx, int src_n, int kc0, int kc_max, int nsub1, int nsub2) {
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int img = blockIdx.x / S;
    const int tid = threadIdx.x, lane = tid & 31;

    using Smem = BkSmem<kThreads, kYBins>;
    using G = typename Smem::G;
    constexpr int kCap = Smem::kCap;
    constexpr int kKeyCap = Smem::kKeyCap;
    constexpr int kRegList = kBkListCap - kCap;     // phase C: list entries held in registers ...
    constexpr int kListPer = kRegList / kThreads;   // ... per thread
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem* sm = reinterpret_cast<Smem*>(smem_raw);

    const int cnt = counts ? min(counts[img], n) : n;
    const float4* ib = boxes + (size_t)img * (gather_idx ? src_n : n);
    const int32_t* gi = gather_idx ? gather_idx + (size_t)img * n : nullptr;
    int32_t* ikeep = keep + (size_t)img * max_keep;
    float4* iout = out_boxes ? out_boxes + (size_t)img * max_keep : nullptr;
    const int ecap = Smem::kEdgeCap / S;

    for (int e = tid; e < kKeyCap; e += kThreads) sm->hist[e] = 0u;
    for (int i = tid; i < kCap; i += kThreads) sm->cstate[0][i] = 0;
    if (tid == 0) {
        sm->ecursor = 0u;
        sm->work[0] = 0u;
        sm->work[1] = 0u;
    }
    // (one CTA per image: a block barrier does; the hardware cluster barrier costs ~1 us even for a cluster of one)
    auto cluster_sync = [&]() { if (S == 1) __syncthreads(); else cluster.sync(); };
    cluster_sync();  // every CTA's shared memory is initialised before a peer writes into it

    int nk = 0;   // kept so far (identical in every CTA of the cluster)
    int par = 0;  // chunk parity (cstate double buffer)
    int kc = kc0;
    for (int base = 0; base < cnt && nk < max_keep; par ^= 1) {
        const int m = min(kc, cnt - base);
        unsigned char* st = sm->cstate[par];
        // ---- A: stage the chunk (screening areas, keys), histograms of the list keys and of the own candidates' keys
        //      (a thread's gather indices are all loaded before the first box: one memory latency, not two per box)
        constexpr int kPerA = kCap / kThreads;
        int src[kPerA];
#pragma unroll
        for (int q = 0; q < kPerA; ++q) {
            const int i = tid + q * kThreads;
            src[q] = i < m ? (gi ? gi[base + i] : base + i) : 0;
        }
#pragma unroll
        for (int q = 0; q < kPerA; ++q) {
            const int i = tid + q * kThreads;
            if (i >= m) break;
            const float4 b = ib[src[q]];
            const float sa = screen_area(b, thr.c2);
            const int key = G::key(b, sa);
            sm->cbox[i] = b;
            sm->csa[i] = sa;
            sm->ckey[i] = (unsigned short)key;
            sm->pend[i] = 0;
            sm->ovf[i] = 0;
            if (i % S == rank) atomicAdd(&sm->hist[key], 0x10000u);
        }
        for (int k = tid; k < nk; k += kThreads) atomicAdd(&sm->hist[G::key(sm->lbox[k], sm->la[k])], 1u);
        __syncthreads();
        // ---- B: exclusive scan of both histograms at once (the block; the list's half gives its start offsets)
        bk_scan_keys<kThreads, Smem::kKeyPer>(sm->hist, sm->lstart, sm->warp_tmp);
        __syncthreads();
        // ---- C: scatter the list in place (order inside a bucket does not matter to any decision), the own
        //      candidates into cord.  Every entry is read before any is written: list entries below kRegList wait in
        //      registers (their screening area is recomputed, it is screen_area() of the box), the others in the
        //      survivors' arrays, which are free until phase G.
        {
            float4 lb_r[kListPer > 0 ? kListPer : 1];
            unsigned int pos[kListPer > 0 ? (kListPer + 1) / 2 : 1];  // two 16-bit list positions per register
#pragma unroll
            for (int q = 0; q < kListPer; ++q) {
                const int k = tid + q * kThreads;
                if (k < nk) {
                    lb_r[q] = sm->lbox[k];
                    const unsigned int p = atomicAdd(&sm->hist[G::key(lb_r[q], sm->la[k])], 1u) & 0xffffu;
                    pos[q / 2] = (q & 1) ? (pos[q / 2] | (p << 16)) : p;
                }
            }
            for (int k = kRegList + tid; k < nk; k += kThreads) {
                const float4 b = sm->lbox[k];
                const float a = sm->la[k];
                sm->sidx[k - kRegList] = (unsigned short)atomicAdd(&sm->hist[G::key(b, a)], 1u);
                sm->sbox[k - kRegList] = b;
                sm->ssa[k - kRegList] = a;
            }
            for (int i = tid; i < m; i += kThreads)
                if (i % S == rank) sm->cord[atomicAdd(&sm->hist[sm->ckey[i]], 0x10000u) >> 16] = (unsigned short)i;
            __syncthreads();
#pragma unroll
            for (int q = 0; q < kListPer; ++q) {
                if (tid + q * kThreads < nk) {
                    const unsigned int p = (pos[q / 2] >> (16 * (q & 1))) & 0xffffu;
                    sm->lbox[p] = lb_r[q];
                    sm->la[p] = screen_area(lb_r[q], thr.c2);
                }
            }
            for (int k = kRegList + tid; k < nk; k += kThreads) {
                const int p = sm->sidx[k - kRegList];
                sm->lbox[p] = sm->sbox[k - kRegList];
                sm->la[p] = sm->ssa[k - kRegList];
            }
        }
        __syncthreads();
        const float4* lb = sm->lbox;
        const float* la = sm->la;
        // ---- D: screen the own candidates against the admissible part of the kept list: nsub1 lanes per candidate,
        //      a warp takes 32 / nsub1 candidates (adjacent in key order: walks of similar length) at a time
        const int n_own = (m - rank + S - 1) / S;
        for (int e = tid; e < kKeyCap; e += kThreads) {  // the next chunk's histograms, the survivors' of phase E
            sm->hist[e] = 0u;
            sm->shist[e] = 0u;
        }
        if (nk > 0) {
            const int per_warp = 32 / nsub1, sub = lane % nsub1;
            for (;;) {
                const int q = bk_grab(&sm->work[0], per_warp, lane) + lane / nsub1;
                if (q - lane / nsub1 >= n_own) break;
                if (q >= n_own) continue;
                const int i = sm->cord[q];
                const float4 cbx = sm->cbox[i];
                const float ca = sm->csa[i];
                int pk = -1;
                bk_walk<G>(sm->lstart, cbx, ca, thr, sub, nsub1, [&](int k) {
                    if (suppress_screen<true>(lb[k], la[k], cbx, ca)) pk = k;
                });
                if (pk >= 0) {
                    bool r = suppress_exact(lb[pk], cbx, thr.up);
                    if (!r) {  // the screen hit was not confirmed by the exact test (rare): exact walk of the own share
                        const float up = thr.up;
                        bool* rp = &r;
                        bk_walk_slow<G>(sm->lstart, cbx, ca, thr, sub, nsub1, [=](int k) {
                            if (suppress_screen<true>(lb[k], la[k], cbx, ca) && suppress_exact(lb[k], cbx, up)) *rp = true;
                            return *rp;
                        });
                    }
                    if (r) {
                        st[i] = 2;
                        for (int d = 1; d < S; ++d) *cluster.map_shared_rank(&st[i], (rank + d) % S) = 2;
                    }
                }
            }
        }
        cluster_sync();
        // ---- E: histogram of the survivors' keys; reset the next chunk's states
        unsigned int* shist = sm->shist;
        for (int i = tid; i < kCap; i += kThreads) sm->cstate[par ^ 1][i] = 0;
        for (int i = tid; i < m; i += kThreads)
            if (st[i] == 0) atomicAdd(&shist[sm->ckey[i]], 1u);
        __syncthreads();
        // ---- F: scan
        bk_scan_keys<kThreads, Smem::kKeyPer>(shist, sm->sstart, sm->warp_tmp);
        __syncthreads();
        // ---- G: bucket the survivors, ordered by (key, chunk position): an unordered scatter of the positions, then
        //      every entry ranks itself inside its bucket -- the array is the same in every CTA of the cluster, which
        //      phase H relies on to deal the pairs out
        float4* sb = sm->sbox;
        float* sa_ = sm->ssa;
        unsigned short* tmp = sm->cord;  // the own-candidate order is not needed any more
        for (int i = tid; i < m; i += kThreads)
            if (st[i] == 0) tmp[atomicAdd(&shist[sm->ckey[i]], 1u)] = (unsigned short)i;
        __syncthreads();
        const int ns = sm->sstart[G::kKeys + 1];
        for (int t = tid; t < ns; t += kThreads) {
            const int i = tmp[t];
            const int key = sm->ckey[i];
            const int lo = sm->sstart[key], hi = sm->sstart[key + 1];
            int r = 0;
            for (int u = lo; u < hi; ++u) r += (tmp[u] < i) ? 1 : 0;
            const int p = lo + r;
            sb[p] = sm->cbox[i];
            sa_[p] = sm->csa[i];
            sm->sidx[p] = (unsigned short)i;
        }
        __syncthreads();
        // ---- H: suppression pairs among the survivors, every pair from its lower bucketed position (nsub2 lanes per
        //      survivor, dealt like phase D)
        {
            const int ns_own = (ns - rank + S - 1) / S;
            const int per_warp = 32 / nsub2, sub = lane % nsub2;
            unsigned short* hb = sm->hitbuf + tid * kBkHits;
            for (;;) {
                const int q = bk_grab(&sm->work[1], per_warp, lane) + lane / nsub2;
                if (q - lane / nsub2 >= ns_own) break;
                if (q >= ns_own) continue;
                const int p = q * S + rank;
                const int i = sm->sidx[p];
                const float4 cbx = sb[p];
                const float ca = sa_[p];
                int nh = 0;
                bk_walk_up<G>(sm->sstart, p, sm->ckey[i], cbx, ca, thr, sub, nsub2, [&](int k) {
                    if (suppress_screen<true>(sb[k], sa_[k], cbx, ca)) {
                        hb[nh & (kBkHits - 1)] = (unsigned short)k;
                        ++nh;
                    }
                });
                if (nh > kBkHits) {  // more screen hits than the ring holds: walk the share again, confirming as they come
                    const float up = thr.up;
                    const unsigned short* sidx = sm->sidx;
                    Smem* smp = sm;
                    bk_walk_up_slow<G>(sm->sstart, p, sm->ckey[i], cbx, ca, thr, sub, nsub2, [=](int k) {
                        if (suppress_screen<true>(sb[k], sa_[k], cbx, ca) && suppress_exact(sb[k], cbx, up)) {
                            const int j = sidx[k];
                            bk_push_edge(smp, max(i, j), min(i, j), rank, ecap);
                        }
                    });
                } else {
                    for (int h = 0; h < nh; ++h) {
                        const int k = (int)hb[h];
                        if (suppress_exact(sb[k], cbx, thr.up)) {
                            const int j = sm->sidx[k];
                            bk_push_edge(sm, max(i, j), min(i, j), rank, ecap);
                        }
                    }
                }
            }
        }
        __syncthreads();
        {   // mirror this CTA's edges (and, if its region overflowed, the flags) into the other CTAs of the cluster
            const unsigned int raw = sm->ecursor;
            const int ne = (int)min(raw, (unsigned int)ecap);
            for (int d = 1; d < S; ++d) {
                const int dst = (rank + d) % S;
                unsigned int* re = cluster.map_shared_rank(&sm->edges[rank * ecap], dst);
                for (int e = tid; e < ne; e += kThreads) re[e] = sm->edges[rank * ecap + e];
                if (raw > (unsigned int)ecap) {
                    unsigned char* ro = cluster.map_shared_rank(&sm->ovf[0], dst);
                    for (int i = tid; i < m; i += kThreads)
                        if (sm->ovf[i]) ro[i] = 1;
                }
            }
            if (tid < S) *cluster.map_shared_rank(&sm->ecount[rank], tid) = (unsigned int)ne;
        }
        cluster_sync();
        // ---- I: fix-point (every CTA on all survivors and all edges)
        for (;;) {
            {   // a thread works on one region: regions fill evenly (positions are dealt round-robin)
                const int r = tid % S;
                const int ne = (int)sm->ecount[r];
                for (int e = tid / S; e < ne; e += kThreads / S) {
                    const unsigned int v = sm->edges[r * ecap + e];
                    const int i = (int)(v >> 16), j = (int)(v & 0xffffu);
                    if (st[i] == 0) {
                        const int sj = st[j];
                        if (sj == 1) st[i] = 2;
                        else if (sj == 0) sm->pend[i] = 1;
                    }
                }
            }
            __syncthreads();
            bool any = false;
            for (int i = tid; i < m; i += kThreads) {
                if (st[i] != 0) continue;
                if (sm->ovf[i]) {  // edges incomplete: decide from a walk over all admissible predecessors
                    bool hit_kept = false, pending = false;
                    bool* hk = &hit_kept;
                    bool* pd = &pending;
                    const float4 cbx = sm->cbox[i];
                    const float ca = sm->csa[i];
                    const float up = thr.up;
                    const unsigned short* sidx = sm->sidx;
                    const unsigned char* stc = st;
                    bk_walk_slow<G>(sm->sstart, cbx, ca, thr, 0, 1, [=](int p) {
                        const int j = sidx[p];
                        if (j < i) {
                            const int sj = stc[j];
                            if (sj != 2 && suppress_screen<true>(sb[p], sa_[p], cbx, ca) && suppress_exact(sb[p], cbx, up)) {
                                if (sj == 1) *hk = true;
                                else *pd = true;
                            }
                        }
                        return *hk;
                    });
                    sm->pend[i] = 0;
                    if (hit_kept) st[i] = 2;
                    else if (!pending) st[i] = 1;
                    else any = true;
                } else if (sm->pend[i]) {
                    sm->pend[i] = 0;
                    any = true;
                } else {
                    st[i] = 1;
                }
            }
            if (!__syncthreads_or(any)) break;
        }
        // ---- J: append the kept survivors in score order
        int kept_chunk;
        {
            constexpr int kPer = kCap / kThreads;  // consecutive candidates per thread
            const int i0 = tid * kPer;
            unsigned int c = 0;
#pragma unroll
            for (int q = 0; q < kPer; ++q) c += (i0 + q < m && st[i0 + q] == 1) ? 1u : 0u;
            unsigned int total;
            int o = nk + (int)block_exclusive_scan(c, sm->warp_tmp, &total);
#pragma unroll
            for (int q = 0; q < kPer; ++q) {
                const int i = i0 + q;
                if (i < m && st[i] == 1) {
                    if (o < max_keep) {
                        const float4 kb = sm->cbox[i];
                        sm->lbox[o] = kb;
                        sm->la[o] = sm->csa[i];
                        if (rank == 0) {
                            ikeep[o] = base + i;
                            if (iout) iout[o] = kb;
                        }
                    }
                    ++o;
                }
            }
            kept_chunk = (int)total;
            nk = min(nk + kept_chunk, max_keep);
        }
        if (tid == 0) {
            sm->ecursor = 0u;
            sm->work[0] = 0u;
            sm->work[1] = 0u;
        }
        base += m;
        // next chunk: enough candidates for the missing keeps at the rate of this chunk, plus half
        {
            const long long need = max_keep - nk;
            long long next = (need * m * 3) / (2 * (long long)max(kept_chunk, 1)) + 1;
            next = (next + 255) & ~255LL;
            kc = (int)min((long long)kc_max, max(256LL, next));
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

bool nms_bucket_eligible(int n, int max_keep, const NmsThr& thr, int unit_boxes) {
    const int kcap = max_keep < n ? max_keep : n;
    return thr.fast && unit_boxes && kcap < kBkListCap && n >= 1;
}

size_t nms_bucket_smem_bytes(int threads, int S) {
    return threads <= 256              ? sizeof(BkSmem<256, 1>)
           : threads == 512            ? sizeof(BkSmem<512, 1>)
           : bk_ybins(1024, S) == 4    ? sizeof(BkSmem<1024, 4>)
                                       : sizeof(BkSmem<1024, 1>);
}
// two CTAs of the throughput form per SM: 228 KB of shared memory per SM, 1 KB of it reserved per CTA
static_assert(sizeof(BkSmem<512, 1>) <= 115712, "the 512-thread layout must fit twice per SM");

int nms_bucket_launch(const float* boxes, const int32_t* counts, int B, int n, const NmsThr& thr, int max_keep, int32_t* keep,
                      int32_t* keep_count, float* out_boxes, int S, int threads, const NmsTune& tune, frr_stream_t stream,
                      const int32_t* gather_idx, int src_n) {
    using kern_t = void (*)(const float4*, const int32_t*, int, int, NmsThr, int32_t*, int32_t*, float4*, const int32_t*,
                            int, int, int, int, int);
    kern_t kern = threads <= 256          ? nms_bucket_kernel<256, 1>
                  : threads == 512        ? nms_bucket_kernel<512, 1>
                  : bk_ybins(1024, S) == 4 ? nms_bucket_kernel<1024, 4>
                                          : nms_bucket_kernel<1024, 1>;
    if (threads < 256) threads = 256;
    const size_t smem = nms_bucket_smem_bytes(threads, S);
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // (otherwise the driver may pick an L1 / shared split that holds one CTA of the 512-thread form per SM)
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (S > 8) FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    // chunk sizes (frr_nms_sorted has checked them to lie in [256, kBkChunk]; clamped to what the thread count's
    // layout holds): the first chunk is small when few boxes are wanted (test mode: 300), at most first_chunk
    // (automatic: 512 with one CTA per image -- the first chunk is screened against an empty list, and the rate at which
    // it keeps sizes the next ones: 128 against 138 us per 64 images with the cell keys -- and 1024 in the clusters, whose
    // single-image latency grows with 512: 79 / 86 against 72 / 77 us at 8 / 16 CTAs)
    const int cap = bk_chunk_cap(threads);
    const int kc_max = tune.max_chunk ? min(tune.max_chunk & ~255, cap) : cap;
    int want = ((max_keep + max_keep / 2) + 255) & ~255;
    if (want < 256) want = 256;
    int kc0 = tune.first_chunk ? tune.first_chunk & ~255 : (S == 1 ? 512 : 1024);
    if (kc0 > want) kc0 = want;
    if (kc0 > kc_max) kc0 = kc_max;
    // lanes per candidate, automatic: in the screen 1 with one CTA per image (B = 64: 126 vs 129 us with 2), 2 with two
    // CTAs (tools/nms_s1_sweep.py), 4 in the large clusters of the single-image form (81 vs 85 us)
    const int nsub1 = tune.lanes_screen ? tune.lanes_screen : (S == 1 ? 1 : S == 2 ? 2 : 4);
    const int nsub2 = tune.lanes_pairs ? tune.lanes_pairs : 4;

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
    FRR_CUDA(cudaLaunchKernelEx(&cfg, kern, (const float4*)boxes, counts, n, max_keep, thr, keep, keep_count,
                                (float4*)out_boxes, gather_idx, src_n, kc0, kc_max, nsub1, nsub2));
    count_launch();
    FRR_CHECK_LAUNCH("nms_bucket_kernel");
    return FRR_OK;
}

}  // namespace frr
