// Hand-written sm_100a kernels for the map hot path of `pandora map` that drprg launches at
// /root/reference/src/lib.rs:580-642 (argv :594-609, src/predict.rs:288-294); stage semantics follow pandora's
// add_read_hits, define_clusters, filter_clusters(2), add_clusters_to_pangraph and
// pangenome::Graph::add_hits_to_kmergraphs (SURVEY.md §8a rows a4, a5).
//
// This file: S3 - S5 (hit grouping, clustering + filters, k-mer coverage) with no library sort and no host round trip.
//
// The lookup kernels append hits in no particular order and count them per read as they go.  pandora orders the hits
// (read, prg, strand, read_start, k-mer node) and everything downstream is per read, so nothing here sorts globally:
//   assign_kernel         one pass over the per-read hit counters: every read with hits ("active", ~1.4 % of whole-genome
//                         reads) gets a contiguous slice of the grouped-hit array (block scan, one slice allocation per
//                         CTA; the order of the slices is immaterial, all later results are sums) and a class:
//                         <= 64 hits -> a warp, more -> a CTA
//   scatter_kernel        hits move into their read's slice as ONE 64-bit key prg | strand | read_start | k-mer node whose
//                         integer order is pandora's MinimizerHit order within a read; the per-read counters count back
//                         down to zero, so they never need a memset
//   cluster_warp_kernel   one warp per read: register bitonic sort of its <= 64 keys by shuffles, cluster boundaries by
//                         ballot (define_clusters), size thresholds, then filter_clusters / filter_clusters2 on the
//                         surviving clusters (usually one)
//   cluster_cta_kernel    one CTA per long read: the same with a shared-memory (or, beyond 8 k hits, in-place global)
//                         bitonic sort and a block scan for the cluster boundaries
//   both write, next to every grouped hit, its coverage key 2 * k-mer node + strand (or "none" when the hit is dropped),
//   and per read the keys 2N + locus of its kept clusters: no allocation, no atomics
//   cov_count_kernel      S5: a job = (range of 56 k counters, stretch of key slots); its CTA counts the keys of the
//                         stretch that fall into the range in ONE copy of the range's 32-bit counters in shared memory,
//                         with shared-memory atomic adds, and stores the copy as the job's partial
//   cov_merge_kernel      column sum of the partials into the sample's accumulator — or, on a read-sharded run, straight
//                         into the ROOT GPU's accumulator over NVLink with red.global.add (integers: bit-exact for any
//                         number of GPUs), which is the whole "allreduce" of the path; also counts the kept hits
// Overflowing buffers are detected at the end of the batch (the kernels skip their work when a counter exceeds its
// capacity, the accumulators stay untouched) and the batch is redone with larger buffers.
#include <algorithm>
#include <cfloat>
#include <cstdlib>

#include "kernels_common.cuh"

namespace drprg {

// ---- grouped-hit key: prg 16 | reverse 1 | read_start 25 | k-mer node rank 22 ---------------------------------
__device__ __forceinline__ unsigned long long group_key(unsigned long long hi, unsigned long long lo) {
    const unsigned long long prg = (hi >> 16) & 0xffffull, rev = (hi >> 15) & 1ull;
    return (prg << 48) | (rev << 47) | ((lo >> 32) << GKEY_KNODE_BITS) | (lo & ((1ull << GKEY_KNODE_BITS) - 1ull));
}
__device__ __forceinline__ uint32_t gk_pf(unsigned long long k) { return (uint32_t)(k >> 47); }                // prg << 1 | reverse
__device__ __forceinline__ uint32_t gk_prg(unsigned long long k) { return (uint32_t)(k >> 48); }
__device__ __forceinline__ uint32_t gk_rev(unsigned long long k) { return (uint32_t)(k >> 47) & 1u; }
__device__ __forceinline__ uint32_t gk_start(unsigned long long k) { return (uint32_t)(k >> GKEY_KNODE_BITS) & ((1u << GKEY_START_BITS) - 1u); }
__device__ __forceinline__ uint32_t gk_knode(unsigned long long k) { return (uint32_t)k & ((1u << GKEY_KNODE_BITS) - 1u); }

// counters (unsigned long long): the layout is shared with sketch.cu / capi.cu through kernels.cuh (CTR_*)
__device__ __forceinline__ bool batch_overflowed(const unsigned long long* __restrict__ ctr, PostCaps C) {
    return ctr[CTR_HITS] > C.hit_cap || ctr[CTR_QUEUE_NEED] > C.queue_cap;
}

// ============================================================================================
// grouping by read
// ============================================================================================
constexpr int AS_THREADS = 256, AS_PER = 4;  // a CTA step covers 1024 reads: four consecutive counters per thread (one 16-byte load)
__global__ void __launch_bounds__(AS_THREADS) assign_kernel(unsigned long long* __restrict__ ctr, PostCaps C, unsigned long long n_reads,
                                                            const int32_t* __restrict__ read_count, uint32_t* __restrict__ act_read,
                                                            uint32_t* __restrict__ act_base, uint32_t* __restrict__ act_count,
                                                            uint32_t* __restrict__ read_base, uint32_t* __restrict__ big_list) {
    __shared__ unsigned long long s_warp[AS_THREADS / 32];
    __shared__ unsigned long long s_base[3];
    if (batch_overflowed(ctr, C)) return;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned long long step = (unsigned long long)AS_THREADS * AS_PER;
    for (unsigned long long r0 = (unsigned long long)blockIdx.x * step; r0 < n_reads; r0 += (unsigned long long)gridDim.x * step) {
        const unsigned long long r = r0 + (unsigned long long)tid * AS_PER;
        uint32_t c[AS_PER] = {0u, 0u, 0u, 0u};
        if (r + AS_PER <= n_reads) {  // read_count comes from cudaMalloc and r is a multiple of 4: the 16-byte load is aligned
            const int4 v = __ldg(reinterpret_cast<const int4*>(read_count + r));
            c[0] = (uint32_t)v.x; c[1] = (uint32_t)v.y; c[2] = (uint32_t)v.z; c[3] = (uint32_t)v.w;
        } else {
#pragma unroll
            for (int q = 0; q < AS_PER; ++q)
                if (r + q < n_reads) c[q] = (uint32_t)read_count[r + q];
        }
        // one scan for three running sums: hits (bits 0..39), active reads (40..51), long reads (52..63)
        unsigned long long pre[AS_PER + 1];
        pre[0] = 0;
#pragma unroll
        for (int q = 0; q < AS_PER; ++q)
            pre[q + 1] = pre[q] + ((unsigned long long)c[q] | (c[q] ? 1ull << 40 : 0ull) | (c[q] > CLUSTER_WARP_MAX ? 1ull << 52 : 0ull));
        const unsigned long long mine = pre[AS_PER];
        unsigned long long incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = ((unsigned long long)__shfl_up_sync(FULL, (uint32_t)(incl >> 32), d) << 32) | __shfl_up_sync(FULL, (uint32_t)incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            const unsigned long long v = lane < AS_THREADS / 32 ? s_warp[lane] : 0ull;
            unsigned long long w = v;
#pragma unroll
            for (int d = 1; d < AS_THREADS / 32; d <<= 1) {
                const unsigned long long t = ((unsigned long long)__shfl_up_sync(FULL, (uint32_t)(w >> 32), d) << 32) | __shfl_up_sync(FULL, (uint32_t)w, d);
                if (lane >= d) w += t;
            }
            if (lane < AS_THREADS / 32) s_warp[lane] = w - v;  // exclusive warp offsets
            if (lane == AS_THREADS / 32 - 1 && w) {          // one allocation per CTA step for the three lists
                s_base[0] = atomicAdd(ctr + CTR_CURSOR, w & ((1ull << 40) - 1ull));
                s_base[1] = atomicAdd(ctr + CTR_ACTIVE, (w >> 40) & 0xfffull);
                s_base[2] = ((w >> 52) & 0xfffull) ? atomicAdd(ctr + CTR_BIG, (w >> 52) & 0xfffull) : 0ull;
            }
        }
        __syncthreads();
        if (mine) {
            const unsigned long long excl0 = s_warp[wid] + incl - mine;
#pragma unroll
            for (int q = 0; q < AS_PER; ++q) {
                if (!c[q]) continue;
                const unsigned long long excl = excl0 + pre[q];
                const uint32_t base = (uint32_t)(s_base[0] + (excl & ((1ull << 40) - 1ull)));
                const uint32_t a = (uint32_t)(s_base[1] + ((excl >> 40) & 0xfffull));
                act_read[a] = (uint32_t)(r + q);
                act_base[a] = base;
                act_count[a] = c[q];
                read_base[r + q] = base;
                if (c[q] > CLUSTER_WARP_MAX) big_list[s_base[2] + ((excl >> 52) & 0xfffull)] = a;
            }
        }
        __syncthreads();
    }
}

// The lookup kernels emit a read's hits next to each other, so the lanes of a warp mostly share a read: its lanes are
// grouped by read and one atomic per group takes the group's slots (their order within the slice does not matter, the
// cluster kernels sort it)
constexpr int SC_UNROLL = 4;  // warp chunks of 32 hits in flight per warp: their loads, then their atomics, are issued together
__global__ void scatter_kernel(const unsigned long long* __restrict__ hi, const unsigned long long* __restrict__ lo,
                               const unsigned long long* __restrict__ ctr, PostCaps C, uint32_t read_id_base,
                               int32_t* __restrict__ read_count, const uint32_t* __restrict__ read_base,
                               unsigned long long* __restrict__ gkey) {
    if (batch_overflowed(ctr, C)) return;
    const unsigned long long n = ctr[CTR_HITS];
    const int lane = threadIdx.x & 31;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x * SC_UNROLL;
    for (unsigned long long i0 = ((unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) * SC_UNROLL; i0 < n; i0 += stride) {  // warp-uniform
        unsigned long long h[SC_UNROLL];
        uint32_t r[SC_UNROLL], peers[SC_UNROLL];
        int32_t old[SC_UNROLL];
#pragma unroll
        for (int u = 0; u < SC_UNROLL; ++u) {
            const unsigned long long i = i0 + 32 * u + lane;
            h[u] = i < n ? hi[i] : 0ull;
            r[u] = i < n ? (uint32_t)(h[u] >> 32) - read_id_base : 0xffffffffu;  // a read index is below 2^32 - 1
        }
#pragma unroll
        for (int u = 0; u < SC_UNROLL; ++u) {
            peers[u] = __match_any_sync(FULL, r[u]);
            old[u] = 0;
            if (r[u] != 0xffffffffu && lane == __ffs(peers[u]) - 1) old[u] = atomicSub(read_count + r[u], __popc(peers[u]));  // ends at 0 again
        }
#pragma unroll
        for (int u = 0; u < SC_UNROLL; ++u) {
            old[u] = __shfl_sync(FULL, old[u], __ffs(peers[u]) - 1);
            const unsigned long long i = i0 + 32 * u + lane;
            if (i < n) gkey[read_base[r[u]] + (uint32_t)(old[u] - 1) - (uint32_t)__popc(peers[u] & ((1u << lane) - 1u))] = group_key(h[u], lo[i]);
        }
    }
}

// ============================================================================================
// S3 + S4 on one read's clusters that passed the size threshold (pandora filter_clusters, filter_clusters2), run by
// ONE WARP.  Cluster t: first / last = read_start of its first / last hit, size, pf = prg << 1 | reverse.
//   filter_clusters : clusters in the order (first, size desc, prg, strand forward-first); adjacent-pair sweep: two
//                     clusters of the same prg on opposite strands, or one ending no later than its predecessor, lose
//                     the smaller one (ties: the later one);
//   filter_clusters2: survivors by decreasing size; a cluster whose read span is already covered by the spans of the
//                     bigger survivors is dropped.
// The orders are total (two clusters of one read cannot agree on prg, strand and first start), so they are built by
// rank counting across the lanes; the sweep is sequential like pandora's.
// ============================================================================================
struct ClusterArrays {
    uint32_t *first, *last, *size, *pf;  // per cluster
    uint32_t *ord, *ord2;                // work: the two orders
    uint32_t* alive;                     // in: 1 for every cluster; out: survivors
};

__device__ void filter_clusters_warp(uint32_t ncl, const ClusterArrays& A, int lane) {
    // ---- filter_clusters
    for (uint32_t c = lane; c < ncl; c += 32) {
        const uint32_t f = A.first[c], s = A.size[c], p = A.pf[c];
        uint32_t rank = 0;
        for (uint32_t d = 0; d < ncl; ++d) {
            const uint32_t fd = A.first[d], sd = A.size[d], pd = A.pf[d];
            const bool before = fd != f ? fd < f : (sd != s ? sd > s : (pd != p ? pd < p : d < c));
            rank += before ? 1u : 0u;
        }
        A.ord[rank] = c;
    }
    __syncwarp();
    if (lane == 0) {
        uint32_t prev = A.ord[0];
        for (uint32_t t = 1; t < ncl; ++t) {
            const uint32_t cur = A.ord[t];
            const uint32_t pc = A.pf[cur], pp = A.pf[prev];
            const bool cond = ((pc >> 1) == (pp >> 1) && (pc & 1u) != (pp & 1u)) || (A.last[cur] <= A.last[prev]);
            if (cond) {
                if (A.size[prev] >= A.size[cur]) {
                    A.alive[cur] = 0;
                    continue;
                }
                A.alive[prev] = 0;
            }
            prev = cur;
        }
    }
    __syncwarp();
    // ---- filter_clusters2: order (size desc, first, prg, strand) among the survivors
    uint32_t n2 = 0;
    for (uint32_t c0 = 0; c0 < ncl; c0 += 32) {
        const uint32_t c = c0 + lane;
        const bool live = c < ncl && A.alive[c];
        if (live) {
            const uint32_t f = A.first[c], s = A.size[c], p = A.pf[c];
            uint32_t rank = 0;
            for (uint32_t d = 0; d < ncl; ++d) {
                if (!A.alive[d]) continue;
                const uint32_t fd = A.first[d], sd = A.size[d], pd = A.pf[d];
                const bool before = sd != s ? sd > s : (fd != f ? fd < f : (pd != p ? pd < p : d < c));
                rank += before ? 1u : 0u;
            }
            A.ord2[rank] = c;
        }
        n2 += __popc(__ballot_sync(FULL, live));
    }
    __syncwarp();
    for (uint32_t t = 1; t < n2; ++t) {
        const uint32_t c = A.ord2[t];
        const uint32_t z = A.last[c];
        uint32_t cur = A.first[c];
        bool contained = true;
        while (cur < z) {
            uint32_t best = cur;
            for (uint32_t u = lane; u < t; u += 32) {
                const uint32_t pc = A.ord2[u];
                if (!A.alive[pc]) continue;  // erased clusters never marked the read
                if (A.first[pc] <= cur && cur < A.last[pc]) best = max(best, A.last[pc]);
            }
            best = __reduce_max_sync(FULL, best);
            if (best == cur) {
                contained = false;
                break;
            }
            cur = best;
        }
        if (contained && lane == 0) A.alive[c] = 0;
        __syncwarp();
    }
}

// ============================================================================================
// one warp per read with <= 64 hits
// ============================================================================================
constexpr int CW_WARPS = 8;

__device__ __forceinline__ unsigned long long shfl_xor64(unsigned long long v, int m) {
    return ((unsigned long long)__shfl_xor_sync(FULL, (uint32_t)(v >> 32), m) << 32) | __shfl_xor_sync(FULL, (uint32_t)v, m);
}
__device__ __forceinline__ unsigned long long shfl_up64(unsigned long long v, int d) {
    return ((unsigned long long)__shfl_up_sync(FULL, (uint32_t)(v >> 32), d) << 32) | __shfl_up_sync(FULL, (uint32_t)v, d);
}
__device__ __forceinline__ unsigned long long shfl64(unsigned long long v, int src) {
    return ((unsigned long long)__shfl_sync(FULL, (uint32_t)(v >> 32), src) << 32) | __shfl_sync(FULL, (uint32_t)v, src);
}

// bitonic network over the 32 * NREG keys of a warp, fully unrolled (every shuffle distance and direction is static)
template <int NREG>
__device__ __forceinline__ void warp_sort64(unsigned long long& x0, unsigned long long& x1, int lane) {
#pragma unroll
    for (int k = 2; k <= 32 * NREG; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j == 32) {  // k == 64: the last merge is ascending over all 64 elements
                const unsigned long long lo = x0 < x1 ? x0 : x1, hi = x0 < x1 ? x1 : x0;
                x0 = lo;
                x1 = hi;
            } else {
                const bool lower = (lane & j) == 0;
                {
                    const unsigned long long y = shfl_xor64(x0, j);
                    const bool take_min = lower == ((lane & k) == 0);
                    x0 = ((x0 < y) == take_min) ? x0 : y;
                }
                if (NREG == 2) {
                    const unsigned long long y = shfl_xor64(x1, j);
                    const bool take_min = lower == (((lane + 32) & k) == 0);
                    x1 = ((x1 < y) == take_min) ? x1 : y;
                }
            }
        }
    }
}

// the keys of read slice [base, base + c) a warp sorts (element i in lane i & 31, register i >> 5; padding sorts to the
// end), loaded only for a read this kernel clusters
struct WarpRead {
    uint32_t c, base;
    unsigned long long x0, x1;
};
__device__ __forceinline__ void load_warp_read_keys(WarpRead& R, const unsigned long long* __restrict__ gkey, uint32_t min_thresh, int lane) {
    const bool mine = R.c > min_thresh && R.c <= CLUSTER_WARP_MAX;
    R.x0 = mine && (uint32_t)lane < R.c ? gkey[R.base + lane] : ~0ull;
    R.x1 = mine && (uint32_t)lane + 32u < R.c ? gkey[R.base + 32 + lane] : ~0ull;
}

__device__ __forceinline__ void cluster_warp_read(
    unsigned long long a, WarpRead R, unsigned long long* __restrict__ ctr, unsigned long long* __restrict__ gkey, uint8_t* __restrict__ gkept,
    uint32_t max_diff, uint32_t min_thresh, const uint32_t* __restrict__ thresh, const uint32_t* __restrict__ knode_base, uint32_t locus_key_base,
    uint32_t* __restrict__ cov_keys, uint32_t* __restrict__ act_lk, uint32_t* __restrict__ lk_ovf, uint32_t (*s_u32)[64], uint32_t* s_alive, int lane) {
    const uint32_t c = R.c, base = R.base;
    if (c > CLUSTER_WARP_MAX) return;  // the CTA kernel's read
    if (c <= min_thresh) {  // no cluster of this read can exceed any locus's size threshold (stray hits): nothing is kept
        if ((uint32_t)lane < c) {
            gkept[base + lane] = 0;
            cov_keys[base + lane] = COV_KEY_NONE;
        }
        if ((uint32_t)lane + 32u < c) {
            gkept[base + 32 + lane] = 0;
            cov_keys[base + 32 + lane] = COV_KEY_NONE;
        }
        if (lane < 2) act_lk[2 * a + lane] = COV_KEY_NONE;
        return;
    }
    unsigned long long x0 = R.x0, x1 = R.x1;
    if (c > 32u) warp_sort64<2>(x0, x1, lane);  // warp-uniform
    else warp_sort64<1>(x0, x1, lane);
    if ((uint32_t)lane < c) gkey[base + lane] = x0;  // the slice stays sorted for the hooks / later consumers
    if ((uint32_t)lane + 32u < c) gkey[base + 32 + lane] = x1;
    // ---- define_clusters: a hit opens a cluster when prg or strand change or the gap exceeds max_diff
    const unsigned long long p0 = shfl_up64(x0, 1), x0_31 = shfl64(x0, 31);
    unsigned long long p1 = shfl_up64(x1, 1);
    if (lane == 0) p1 = x0_31;
    auto opens = [&](unsigned long long cur, unsigned long long prev, uint32_t i) {
        if (i == 0u || i == c) return true;  // i == c: the first padding element closes the last cluster
        if (i > c) return false;
        return gk_pf(cur) != gk_pf(prev) || gk_start(cur) - gk_start(prev) > max_diff;
    };
    const uint32_t m0 = __ballot_sync(FULL, opens(x0, p0, (uint32_t)lane));
    const uint32_t m1 = __ballot_sync(FULL, opens(x1, p1, (uint32_t)lane + 32u));
    const unsigned long long S = (unsigned long long)m0 | ((unsigned long long)m1 << 32);
    uint32_t cb[2], ce[2];
    bool pass[2], begin_pass[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const uint32_t i = (uint32_t)lane + 32u * r;
        const unsigned long long le = i == 63u ? ~0ull : ((2ull << i) - 1ull);
        cb[r] = 63u - (uint32_t)__clzll((long long)(S & le));
        const unsigned long long gt = S & ~le;
        ce[r] = gt ? (uint32_t)__ffsll((long long)gt) - 1u : c;
        const unsigned long long xr = r ? x1 : x0;
        pass[r] = i < c && (ce[r] - cb[r]) > thresh[gk_prg(xr)];
        begin_pass[r] = pass[r] && cb[r] == i;
    }
    const uint32_t b0 = __ballot_sync(FULL, begin_pass[0]), b1 = __ballot_sync(FULL, begin_pass[1]);
    const unsigned long long BP = (unsigned long long)b0 | ((unsigned long long)b1 << 32);
    const uint32_t ncl = (uint32_t)__popcll(BP);
    if (ncl == 0u) {
        if ((uint32_t)lane < c) {
            gkept[base + lane] = 0;
            cov_keys[base + lane] = COV_KEY_NONE;
        }
        if ((uint32_t)lane + 32u < c) {
            gkept[base + 32 + lane] = 0;
            cov_keys[base + 32 + lane] = COV_KEY_NONE;
        }
        if (lane < 2) act_lk[2 * a + lane] = COV_KEY_NONE;
        return;
    }
    bool alive[2] = {pass[0], pass[1]};
    if (ncl > 1u) {
        uint32_t* first = s_u32[0];
        uint32_t* last = s_u32[1];
        uint32_t* size = s_u32[2];
        uint32_t* pf = s_u32[3];
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const unsigned long long xr = r ? x1 : x0;
            const uint32_t i = (uint32_t)lane + 32u * r;
            if (begin_pass[r]) {
                const uint32_t t = (uint32_t)__popcll(BP & ((1ull << i) - 1ull));
                first[t] = gk_start(xr);
                size[t] = ce[r] - cb[r];
                pf[t] = gk_pf(xr);
                s_alive[t] = 1u;
            }
            if (pass[r] && i + 1u == ce[r]) last[(uint32_t)__popcll(BP & ((1ull << cb[r]) - 1ull))] = gk_start(xr);
        }
        __syncwarp();
        ClusterArrays A{first, last, size, pf, s_u32[4], s_u32[5], s_alive};
        filter_clusters_warp(ncl, A, lane);
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (pass[r]) alive[r] = s_alive[(uint32_t)__popcll(BP & ((1ull << cb[r]) - 1ull))] != 0u;
    }
    // ---- add_clusters_to_pangraph: kept flags, one coverage key per kept hit, one locus key per kept cluster
    const uint32_t k0m = __ballot_sync(FULL, alive[0] && begin_pass[0]), k1m = __ballot_sync(FULL, alive[1] && begin_pass[1]);
    const unsigned long long KB = (unsigned long long)k0m | ((unsigned long long)k1m << 32);  // begins of the kept clusters
    if (lane < 2 && (uint32_t)__popcll(KB) <= (uint32_t)lane) act_lk[2 * a + lane] = COV_KEY_NONE;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const uint32_t i = (uint32_t)lane + 32u * r;
        if (i >= c) continue;
        const unsigned long long xr = r ? x1 : x0;
        gkept[base + i] = alive[r] ? 1 : 0;
        cov_keys[base + i] = alive[r] ? 2u * (knode_base[gk_prg(xr)] + gk_knode(xr)) + gk_rev(xr) : COV_KEY_NONE;
        if (alive[r] && begin_pass[r]) {
            const uint32_t t = (uint32_t)__popcll(KB & ((1ull << i) - 1ull));
            if (t < 2u) act_lk[2 * a + t] = locus_key_base + gk_prg(xr);
            else lk_ovf[atomicAdd(ctr + CTR_LKOVF, 1ull)] = locus_key_base + gk_prg(xr);  // a third kept cluster on one short read: rare
        }
    }
}

// One warp per read, the next read's keys and the one after's count and slice base in flight while the current read is
// clustered: each read is a chain of dependent loads (count, base -> keys -> thresholds), which the pipeline overlaps
__global__ void __launch_bounds__(CW_WARPS * 32) cluster_warp_kernel(
    unsigned long long* __restrict__ ctr, PostCaps C, const uint32_t* __restrict__ act_base, const uint32_t* __restrict__ act_count,
    unsigned long long* __restrict__ gkey, uint8_t* __restrict__ gkept, uint32_t max_diff, uint32_t min_thresh, const uint32_t* __restrict__ thresh,
    const uint32_t* __restrict__ knode_base, uint32_t locus_key_base, uint32_t* __restrict__ cov_keys, uint32_t* __restrict__ act_lk,
    uint32_t* __restrict__ lk_ovf) {
    __shared__ uint32_t s_u32[CW_WARPS][6][64];  // first, last, size, pf, ord, ord2
    __shared__ uint32_t s_alive[CW_WARPS][64];
    if (batch_overflowed(ctr, C)) return;
    const unsigned long long n_active = ctr[CTR_ACTIVE];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned long long stride = (unsigned long long)gridDim.x * CW_WARPS;
    auto head = [&](unsigned long long a) {
        WarpRead R{0u, 0u, ~0ull, ~0ull};
        if (a < n_active) {
            R.c = act_count[a];
            R.base = act_base[a];
        }
        return R;
    };
    unsigned long long a = (unsigned long long)blockIdx.x * CW_WARPS + wid;
    WarpRead cur = head(a);
    load_warp_read_keys(cur, gkey, min_thresh, lane);
    WarpRead nxt = head(a + stride);
    for (; a < n_active; a += stride) {
        load_warp_read_keys(nxt, gkey, min_thresh, lane);
        const WarpRead after = head(a + 2 * stride);
        cluster_warp_read(a, cur, ctr, gkey, gkept, max_diff, min_thresh, thresh, knode_base, locus_key_base, cov_keys, act_lk, lk_ovf,
                          s_u32[wid], s_alive[wid], lane);
        cur = nxt;
        nxt = after;
    }
}

// ============================================================================================
// one CTA per read with more than 64 hits (long reads)
// ============================================================================================
constexpr int CC_THREADS = 256;
constexpr uint32_t CC_SMEM_KEYS = 8192;  // 64 KB of keys sorted in shared memory; longer slices are sorted in place in global memory

// ascending-only bitonic network (first step of every merge compares i with i ^ (k-1), the rest i ^ j): elements past n
// act as +infinity and never move, so n need not be a power of two
template <class T>
__device__ void block_bitonic(T* a, uint32_t n, int tid, int nthreads) {
    uint32_t P = 2;
    while (P < n) P <<= 1;
    for (uint32_t k = 2; k <= P; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            const uint32_t mask = (j == (k >> 1)) ? (k - 1u) : j;
            for (uint32_t i = tid; i < n; i += nthreads) {
                const uint32_t l = i ^ mask;
                if (l > i && l < n) {
                    const T x = a[i], y = a[l];
                    if (x > y) {
                        a[i] = y;
                        a[l] = x;
                    }
                }
            }
            __syncthreads();
        }
}

struct BigScratch {  // per-hit scratch, indexed like the grouped-hit array
    uint32_t *cbeg, *cend;                      // cluster begin of every hit; end, stored at the begin
    uint32_t *first, *last, *size, *pf, *ord, *ord2, *alive;  // per cluster that passed the threshold, at [slice base + t]
    uint32_t* slot;                             // cluster number of a begin, stored at the begin
};

__global__ void __launch_bounds__(CC_THREADS) cluster_cta_kernel(
    unsigned long long* __restrict__ ctr, PostCaps C, const uint32_t* __restrict__ big_list, const uint32_t* __restrict__ act_base,
    const uint32_t* __restrict__ act_count, unsigned long long* __restrict__ gkey, uint8_t* __restrict__ gkept, uint32_t max_diff,
    const uint32_t* __restrict__ thresh, const uint32_t* __restrict__ knode_base, uint32_t locus_key_base,
    uint32_t* __restrict__ cov_keys, uint32_t* __restrict__ act_lk, uint32_t* __restrict__ lk_ovf, BigScratch B) {
    extern __shared__ unsigned long long s_keys[];
    __shared__ uint32_t s_carry, s_ncl, s_nlk, s_warp_max[CC_THREADS / 32];
    if (batch_overflowed(ctr, C)) return;
    const unsigned long long n_big = ctr[CTR_BIG];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (unsigned long long bi = blockIdx.x; bi < n_big; bi += gridDim.x) {
        const uint32_t a = big_list[bi];
        const uint32_t c = act_count[a], base = act_base[a];
        unsigned long long* K = gkey + base;
        // ---- sort the slice
        if (c <= CC_SMEM_KEYS) {
            for (uint32_t i = tid; i < c; i += CC_THREADS) s_keys[i] = K[i];
            __syncthreads();
            block_bitonic(s_keys, c, tid, CC_THREADS);
            for (uint32_t i = tid; i < c; i += CC_THREADS) K[i] = s_keys[i];
        } else {
            block_bitonic(K, c, tid, CC_THREADS);
        }
        if (tid == 0) {
            s_carry = 0;
            s_ncl = 0;
            s_nlk = 0;
        }
        if (tid < 2) act_lk[2 * a + tid] = COV_KEY_NONE;
        __syncthreads();
        // ---- define_clusters: cbeg[i] = index of the last hit <= i that opens a cluster (running maximum)
        for (uint32_t i0 = 0; i0 < c; i0 += CC_THREADS) {
            const uint32_t i = i0 + tid;
            uint32_t v = 0;
            if (i < c && i > 0) {
                const unsigned long long cur = K[i], prev = K[i - 1];
                if (gk_pf(cur) != gk_pf(prev) || gk_start(cur) - gk_start(prev) > max_diff) v = i;
            }
            uint32_t m = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) m = max(m, __shfl_up_sync(FULL, m, d) * (lane >= d ? 1u : 0u));
            if (lane == 31) s_warp_max[wid] = m;
            __syncthreads();
            uint32_t pre = s_carry;
            for (int w = 0; w < wid; ++w) pre = max(pre, s_warp_max[w]);
            m = max(m, pre);
            if (i < c) B.cbeg[base + i] = m;
            __syncthreads();
            if (tid == CC_THREADS - 1) s_carry = m;
            __syncthreads();
        }
        // a hit that is the last of its cluster knows the end
        for (uint32_t i = tid; i < c; i += CC_THREADS) {
            const uint32_t b = B.cbeg[base + i];
            if (i + 1 == c || B.cbeg[base + i + 1] != b) B.cend[base + b] = i + 1;
        }
        __syncthreads();
        // ---- size threshold: the passing clusters form the list the filters work on
        for (uint32_t i = tid; i < c; i += CC_THREADS) {
            uint32_t sl = 0xffffffffu;
            if (B.cbeg[base + i] == i) {
                const uint32_t e = B.cend[base + i];
                const unsigned long long k0 = K[i];
                if (e - i > thresh[gk_prg(k0)]) {
                    sl = atomicAdd(&s_ncl, 1u);
                    B.first[base + sl] = gk_start(k0);
                    B.last[base + sl] = gk_start(K[e - 1]);
                    B.size[base + sl] = e - i;
                    B.pf[base + sl] = gk_pf(k0);
                    B.alive[base + sl] = 1u;
                }
                B.slot[base + i] = sl;
            }
        }
        __syncthreads();
        const uint32_t ncl = s_ncl;
        if (ncl > 1u && wid == 0) {
            ClusterArrays A{B.first + base, B.last + base, B.size + base, B.pf + base, B.ord + base, B.ord2 + base, B.alive + base};
            __threadfence_block();
            filter_clusters_warp(ncl, A, lane);
        }
        __syncthreads();
        // ---- kept flags + coverage keys
        for (uint32_t i = tid; i < c; i += CC_THREADS) {
            const uint32_t b = B.cbeg[base + i];
            const uint32_t sl = B.slot[base + b];
            const bool keep = sl != 0xffffffffu && B.alive[base + sl] != 0u;
            const unsigned long long k0 = K[i];
            gkept[base + i] = keep ? 1 : 0;
            cov_keys[base + i] = keep ? 2u * (knode_base[gk_prg(k0)] + gk_knode(k0)) + gk_rev(k0) : COV_KEY_NONE;
            if (keep && b == i) {  // one locus key per kept cluster: the first two next to the read, the rest in the overflow list
                const uint32_t t = atomicAdd(&s_nlk, 1u);
                if (t < 2u) act_lk[2 * a + t] = locus_key_base + gk_prg(k0);
                else lk_ovf[atomicAdd(ctr + CTR_LKOVF, 1ull)] = locus_key_base + gk_prg(k0);
            }
        }
        __syncthreads();
    }
}

// ============================================================================================
// S5 : coverage counted in shared memory.
// The key slots of a batch ([one per grouped hit | two per active read | overflow list], "none" where nothing is
// counted) are cut into STRETCHES and the key space into RANGES of 56 k counters, as many 32-bit counters as one CTA's
// shared memory holds (224 KB: the Mtb-scale panel's 76 k keys are two ranges).  A job = (range, stretch): its CTA zeroes
// one copy of the range's counters, every thread counts the keys of its share of the stretch that fall into the range
// with shared-memory atomic adds (integers: the order of the adds does not matter), and the copy is STORED (not added) to
// the job's own piece of partial[stretch][range]; cov_merge_kernel sums over the stretches.  A slot is read once per range.
// ============================================================================================
constexpr int CV_THREADS = 1024;
constexpr uint32_t CV_RANGE = 56 * 1024;                 // counters per range: 224 KB of shared memory
constexpr uint32_t CV_STRETCH_MIN = 32768;               // a job's fixed cost is zeroing and storing 224 KB: a small batch
                                                         // gets fewer, longer stretches rather than more jobs
constexpr unsigned long long CV_STRETCH_MAX = 1ull << 28;  // the per-stretch partials are int32: far below 2^31 slots
constexpr int CV_UNROLL = 4;                             // 16-byte slot loads in flight per thread

// slots per stretch for n slots on a grid of `grid` CTAs and n_range key ranges: the (range, stretch) jobs fill the grid in
// whole waves (one wave while a stretch stays below CV_STRETCH_MAX); a multiple of 1024
__host__ __device__ __forceinline__ unsigned long long cov_stretch_len(unsigned long long n, uint32_t grid, uint32_t n_range) {
    const unsigned long long min_stretches = (n + CV_STRETCH_MAX - 1) / CV_STRETCH_MAX;
    const unsigned long long waves = (min_stretches * n_range + grid - 1) / grid;          // at least this many waves
    unsigned long long stretches = (waves < 1 ? 1 : waves) * grid / n_range;               // stretches that fill them
    if (stretches < 1) stretches = 1;
    unsigned long long len = (n + stretches - 1) / stretches;
    len = (len + 1023ull) & ~1023ull;
    return len < CV_STRETCH_MIN ? CV_STRETCH_MIN : (len > CV_STRETCH_MAX ? CV_STRETCH_MAX : len);
}

// counts the keys of p[lo, hi) that fall into [k_lo, k_lo + k_n): whole 16-byte groups by vector loads, the ends singly
__device__ __forceinline__ void cov_count_segment(const uint32_t* __restrict__ p, unsigned long long lo, unsigned long long hi,
                                                  uint32_t k_lo, uint32_t k_n, uint32_t* cnt, int tid) {
    if (lo >= hi) return;
    auto count = [&](uint32_t key) {
        const uint32_t rel = key - k_lo;  // "none" is far above every range
        if (rel < k_n) atomicAdd(cnt + rel, 1u);
    };
    const unsigned long long v_lo = (lo + 3) & ~3ull, v_hi = hi & ~3ull;
    if (v_lo >= v_hi) {
        for (unsigned long long i = lo + tid; i < hi; i += CV_THREADS) count(__ldg(p + i));
        return;
    }
    if (lo + tid < v_lo) count(__ldg(p + lo + tid));
    if (v_hi + tid < hi) count(__ldg(p + v_hi + tid));
    const uint4* v = reinterpret_cast<const uint4*>(p);  // the slot arrays come from cudaMalloc: 16-byte aligned
    const unsigned long long g_lo = v_lo / 4, g_hi = v_hi / 4;
    for (unsigned long long g0 = g_lo + tid; g0 < g_hi; g0 += (unsigned long long)CV_UNROLL * CV_THREADS) {
        uint4 x[CV_UNROLL];
#pragma unroll
        for (int u = 0; u < CV_UNROLL; ++u) {
            const unsigned long long g = g0 + (unsigned long long)u * CV_THREADS;
            x[u] = g < g_hi ? __ldg(v + g) : make_uint4(COV_KEY_NONE, COV_KEY_NONE, COV_KEY_NONE, COV_KEY_NONE);
        }
#pragma unroll
        for (int u = 0; u < CV_UNROLL; ++u) {
            count(x[u].x);
            count(x[u].y);
            count(x[u].z);
            count(x[u].w);
        }
    }
}

__global__ void __launch_bounds__(CV_THREADS, 1) cov_count_kernel(const unsigned long long* __restrict__ ctr, PostCaps C,
                                                                 const uint32_t* __restrict__ cov_keys, const uint32_t* __restrict__ act_lk,
                                                                 const uint32_t* __restrict__ lk_ovf, int32_t* __restrict__ partials,
                                                                 uint32_t max_stretches, uint32_t n_accum, uint32_t n_keys) {
    extern __shared__ uint32_t s_cnt[];  // [CV_RANGE] counters
    if (batch_overflowed(ctr, C)) return;
    // the slots, concatenated: [per grouped hit | two per active read | overflow list]
    const unsigned long long n0 = ctr[CTR_HITS], n1 = 2ull * ctr[CTR_ACTIVE], n = n0 + n1 + ctr[CTR_LKOVF];
    const uint32_t n_range = (n_keys + CV_RANGE - 1) / CV_RANGE;
    const unsigned long long stretch_len = cov_stretch_len(n, gridDim.x, n_range);
    const uint32_t n_stretch = (uint32_t)min((unsigned long long)max_stretches, (n + stretch_len - 1) / stretch_len);
    const int tid = threadIdx.x;
    for (uint32_t job = blockIdx.x; job < n_stretch * n_range; job += gridDim.x) {
        const uint32_t stretch = job / n_range, k_lo = (job % n_range) * CV_RANGE;
        const uint32_t k_n = min(CV_RANGE, n_keys - k_lo);
        for (uint32_t i = tid; i < CV_RANGE / 4; i += CV_THREADS) reinterpret_cast<uint4*>(s_cnt)[i] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        const unsigned long long s_lo = (unsigned long long)stretch * stretch_len, s_hi = min(n, s_lo + stretch_len);
        auto segment = [&](const uint32_t* p, unsigned long long b, unsigned long long e) {  // the stretch's part of slots [b, e)
            cov_count_segment(p, min(max(s_lo, b), e) - b, min(max(s_hi, b), e) - b, k_lo, k_n, s_cnt, tid);
        };
        segment(cov_keys, 0, n0);
        segment(act_lk, n0, n0 + n1);
        segment(lk_ovf, n0 + n1, n);
        __syncthreads();
        // the job's piece of the partial is this job's alone: a store, not an add
        int32_t* out = partials + (size_t)stretch * n_accum + k_lo;
        for (uint32_t k = tid; k < k_n; k += CV_THREADS) out[k] = (int32_t)s_cnt[k];
        __syncthreads();
    }
}

// Column sum over the stretches into `dst`.  dst is the sample's accumulator on this GPU, or — remote != 0 — the ROOT
// GPU's accumulator mapped over NVLink, which receives one fire-and-forget red.global.add per non-zero counter: the
// fused form of the path's only collective.  The coverage counters (keys below 2N) also add up to the number of kept hits.
__global__ void cov_merge_kernel(unsigned long long* __restrict__ ctr, PostCaps C, const int32_t* __restrict__ partials,
                                 uint32_t max_stretches, uint32_t count_grid, uint32_t n_accum, uint32_t n_keys, uint32_t n_cov_keys,
                                 int32_t* __restrict__ dst, int remote) {
    if (batch_overflowed(ctr, C)) return;
    const unsigned long long n = ctr[CTR_HITS] + 2ull * ctr[CTR_ACTIVE] + ctr[CTR_LKOVF];
    const unsigned long long stretch_len = cov_stretch_len(n, count_grid, (n_keys + CV_RANGE - 1) / CV_RANGE);
    const uint32_t used = (uint32_t)min((unsigned long long)max_stretches, (n + stretch_len - 1) / stretch_len);
    unsigned long long kept = 0;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_keys; k += gridDim.x * blockDim.x) {
        int32_t sum = 0;
#pragma unroll 8
        for (uint32_t g = 0; g < used; ++g) sum += partials[(size_t)g * n_accum + k];  // a row per stretch: eight loads in flight
        if (!sum) continue;
        if (k < n_cov_keys) kept += (unsigned long long)sum;
        if (remote) asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(dst + k), "r"(sum) : "memory");
        else dst[k] += sum;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) kept += ((unsigned long long)__shfl_xor_sync(FULL, (uint32_t)(kept >> 32), d) << 32) | __shfl_xor_sync(FULL, (uint32_t)kept, d);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(ctr + CTR_KEPT, kept);
}

// stretches a hit capacity can produce: [hit_cap | 2 per active read <= 2 hit_cap | overflow <= hit_cap] slots
uint32_t cov_max_stretches(uint64_t hit_cap, int sm_count) {
    // whole waves of the grid: at most (minimum stretches + one wave's worth) stretches
    return (uint32_t)((4 * hit_cap + CV_STRETCH_MAX - 1) / CV_STRETCH_MAX + (uint64_t)sm_count) + 1;
}

// ---- cross-GPU signalling of a read-sharded run (flags live behind the root GPU's accumulator) ------------------
__global__ void flag_wait_kernel(const uint32_t* flag, uint32_t want) {  // spins until *flag >= want (system scope)
    uint32_t v;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v < want) __nanosleep(200);
    } while (v < want);
}
__global__ void flag_publish_kernel(uint32_t* flag, uint32_t value) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
// a shard is finished: its four scalars (bases / reads, lo24 | hi) join the root's, then the arrival counter goes up
__global__ void shard_done_kernel(int32_t* root_tail, int4 scalars, uint32_t* arrivals) {
    asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(root_tail + 0), "r"(scalars.x) : "memory");
    asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(root_tail + 1), "r"(scalars.y) : "memory");
    asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(root_tail + 2), "r"(scalars.z) : "memory");
    asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(root_tail + 3), "r"(scalars.w) : "memory");
    __threadfence_system();
    asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(arrivals), "r"(1u) : "memory");
}
__global__ void add_scalars_kernel(int32_t* tail, int4 scalars) {
    tail[0] += scalars.x;
    tail[1] += scalars.y;
    tail[2] += scalars.z;
    tail[3] += scalars.w;
}
void launch_flag_wait(const uint32_t* flag, uint32_t want, cudaStream_t st) {
    flag_wait_kernel<<<1, 1, 0, st>>>(flag, want);
    ++g_launches;
}
void launch_flag_publish(uint32_t* flag, uint32_t value, cudaStream_t st) {
    flag_publish_kernel<<<1, 1, 0, st>>>(flag, value);
    ++g_launches;
}
void launch_shard_done(int32_t* root_tail, const int32_t scalars[4], uint32_t* arrivals, cudaStream_t st) {
    shard_done_kernel<<<1, 1, 0, st>>>(root_tail, make_int4(scalars[0], scalars[1], scalars[2], scalars[3]), arrivals);
    ++g_launches;
}
void launch_add_scalars(int32_t* tail, const int32_t scalars[4], cudaStream_t st) {
    add_scalars_kernel<<<1, 1, 0, st>>>(tail, make_int4(scalars[0], scalars[1], scalars[2], scalars[3]));
    ++g_launches;
}

void launch_postprocess(const PostBuffers& P, PostCaps C, uint32_t read_id_base, uint64_t n_reads, uint32_t max_diff,
                        uint32_t min_thresh, const uint32_t* d_thresh_per_prg, const uint32_t* d_knode_base, uint32_t total_knodes, uint32_t n_loci,
                        int32_t* d_accum_dst, int remote_dst, int sm_count, cudaStream_t st, cudaEvent_t ev_grouped,
                        cudaEvent_t ev_clustered) {
    const unsigned sm = (unsigned)sm_count;
    const uint64_t as_step = (uint64_t)AS_THREADS * AS_PER;
    const unsigned as_grid = (unsigned)std::min<uint64_t>((n_reads + as_step - 1) / as_step, (uint64_t)sm * 8);
    if (as_grid) assign_kernel<<<as_grid, AS_THREADS, 0, st>>>(P.ctr, C, n_reads, P.read_count, P.act_read, P.act_base, P.act_count, P.read_base, P.big_list);
    scatter_kernel<<<sm * 16, 256, 0, st>>>(P.hi, P.lo, P.ctr, C, read_id_base, P.read_count, P.read_base, P.gkey);
    if (ev_grouped) cudaEventRecord(ev_grouped, st);
    const uint32_t locus_key_base = 2u * total_knodes;
    static const int cw_per_sm = [] {
        int n = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, cluster_warp_kernel, CW_WARPS * 32, 0);
        return std::max(n, 1);
    }();
    cluster_warp_kernel<<<sm * cw_per_sm, CW_WARPS * 32, 0, st>>>(P.ctr, C, P.act_base, P.act_count, P.gkey, P.gkept, max_diff, min_thresh, d_thresh_per_prg,
                                                                  d_knode_base, locus_key_base, P.cov_keys, P.act_lk, P.lk_ovf);
    ensure_dyn_smem(cluster_cta_kernel, (size_t)CC_SMEM_KEYS * 8);
    BigScratch B{P.scratch[0], P.scratch[1], P.scratch[2], P.scratch[3], P.scratch[4], P.scratch[5], P.scratch[6], P.scratch[7],
                 P.scratch[8], P.scratch[9]};
    cluster_cta_kernel<<<sm * 2, CC_THREADS, (size_t)CC_SMEM_KEYS * 8, st>>>(P.ctr, C, P.big_list, P.act_base, P.act_count, P.gkey,
                                                                            P.gkept, max_diff, d_thresh_per_prg, d_knode_base,
                                                                            locus_key_base, P.cov_keys, P.act_lk, P.lk_ovf, B);
    if (ev_clustered) cudaEventRecord(ev_clustered, st);
    const uint32_t n_accum = 2u * total_knodes + n_loci + 4u, n_keys = 2u * total_knodes + n_loci;
    const size_t cv_smem = (size_t)CV_RANGE * sizeof(uint32_t);
    ensure_dyn_smem(cov_count_kernel, cv_smem);
    cov_count_kernel<<<sm, CV_THREADS, cv_smem, st>>>(P.ctr, C, P.cov_keys, P.act_lk, P.lk_ovf, P.partials, P.n_partials, n_accum, n_keys);
    cov_merge_kernel<<<(n_keys + 255) / 256, 256, 0, st>>>(P.ctr, C, P.partials, P.n_partials, sm, n_accum, n_keys, 2u * total_knodes, d_accum_dst,
                                                          remote_dst);
    g_launches += 6;
}

}  // namespace drprg
