// Hand-written sm_100a kernels for the map hot path: read sketching + index lookup (S1+S2), hit
// clustering (S3/S4), k-mer coverage (S5), ML path (S7) and genotyping (S8).  These replace the
// per-read and per-locus loops of `pandora map` that drprg launches at
// /root/reference/src/lib.rs:580-642 (argv :594-609, src/predict.rs:288-294); stage semantics
// follow pandora's Seq::minimizer_sketch, add_read_hits, define_clusters, filter_clusters(2),
// add_hits_to_kmergraphs, KmerGraphWithCoverage::find_max_path and SampleInfo (SURVEY.md §8a).
// This file: S6 device halves (node scores, histograms, threshold) and S7 (max-likelihood path).
#include <algorithm>
#include <cfloat>
#include <cstdlib>

#include "kernels_common.cuh"

namespace drprg {

// ============================================================================================
// S7 : node log-probabilities and the max-likelihood path
// ============================================================================================

__device__ double node_log_prob(const ModelParams& P, uint32_t f, uint32_t r, bool terminal) {
    if (P.bin) {
        if (terminal) return 0.0;
        const uint32_t s = f + r;
        const double n = (double)(s > P.exp_depth ? s : P.exp_depth);
        const double lnck2 = lgamma(n + 1.0) - lgamma((double)f + 1.0) - lgamma((double)r + 1.0) - lgamma(n - (double)f - (double)r + 1.0);
        if (s > P.exp_depth) return lnck2 + (double)s * log(P.bin_p / 2);
        return lnck2 + (double)s * log(P.bin_p / 2) + (double)(P.exp_depth - s) * log(1 - P.bin_p);
    }
    const double c = (double)f + (double)r;
    const double v = lgamma(c + P.nb_r) - lgamma(P.nb_r) - lgamma(c + 1.0) + P.nb_r * log(P.nb_p) + c * log(1.0 - P.nb_p);
    const double FLOOR = -(double)FLT_MAX / 1000.0;
    return v > FLOOR ? v : FLOOR;
}

__global__ void node_prob_kernel(const int32_t* __restrict__ cov, uint32_t total, const uint8_t* __restrict__ is_terminal,
                                 ModelParams P, double* __restrict__ prob) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    prob[g] = node_log_prob(P, cov_sat(cov[2 * g]), cov_sat(cov[2 * g + 1]), is_terminal[g] != 0);
}

void launch_node_prob(const int32_t* d_cov, uint32_t total_knodes, const uint8_t* d_is_terminal, ModelParams P,
                      double* d_prob, cudaStream_t st) {
    if (!total_knodes) return;
    node_prob_kernel<<<(total_knodes + 255) / 256, 256, 0, st>>>(d_cov, total_knodes, d_is_terminal, P, d_prob);
    ++g_launches;
}

// histogram of floor(log-prob + 200) over the inner k-mer nodes of the loci present in the sample: the
// data-parallel half of pandora's estimate_parameters (the valley search itself is a 200-bin host scan)
__global__ void prob_hist_kernel(const double* __restrict__ prob, uint32_t total, const uint8_t* __restrict__ is_terminal,
                                 const uint32_t* __restrict__ knode_locus, const int32_t* __restrict__ locus_reads,
                                 uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[200];
    for (int i = threadIdx.x; i < 200; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < total && !is_terminal[g] && locus_reads[knode_locus[g]] > 0) {
        const double p = prob[g];
        if (p >= -200.0 && p < 0.0) {
            const int j = (int)floor(p + 200.0);
            if (j >= 0 && j < 200) atomicAdd(&sh[j], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 200; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// histogram of the per-node total coverage (0..999) over the inner k-mer nodes of the loci present in the sample:
// the data-parallel half of pandora's estimate_parameters moments / peak search (the 1000-bin scans stay on the host)
__global__ void cov_hist_kernel(const int32_t* __restrict__ cov, uint32_t total, const uint8_t* __restrict__ is_terminal,
                                const uint32_t* __restrict__ knode_locus, const int32_t* __restrict__ locus_reads,
                                uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[1000];
    for (int i = threadIdx.x; i < 1000; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x)
        if (!is_terminal[g] && locus_reads[knode_locus[g]] > 0) {
            const uint32_t c = cov_sat(max(cov[2 * g], 0)) + cov_sat(max(cov[2 * g + 1], 0));
            if (c < 1000u) atomicAdd(&sh[c], 1u);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 1000; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

void launch_cov_hist(const int32_t* d_cov, uint32_t total, const uint8_t* d_is_terminal, const uint32_t* d_knode_locus,
                     const int32_t* d_locus_reads, uint32_t* d_hist1000, cudaStream_t st) {
    cudaMemsetAsync(d_hist1000, 0, 1000 * sizeof(uint32_t), st);
    if (!total) return;
    const unsigned grid = std::min<unsigned>((total + 1023) / 1024, 64u);
    cov_hist_kernel<<<grid, 1024, 0, st>>>(d_cov, total, d_is_terminal, d_knode_locus, d_locus_reads, d_hist1000);
    ++g_launches;
}

void launch_prob_hist(const double* d_prob, uint32_t total, const uint8_t* d_is_terminal, const uint32_t* d_knode_locus,
                      const int32_t* d_locus_reads, uint32_t* d_hist, cudaStream_t st) {
    cudaMemsetAsync(d_hist, 0, 200 * sizeof(uint32_t), st);
    if (!total) return;
    prob_hist_kernel<<<(total + 255) / 256, 256, 0, st>>>(d_prob, total, d_is_terminal, d_knode_locus, d_locus_reads, d_hist);
    ++g_launches;
}

// pandora's find_prob_thresh on the 200-bin histogram (same scan as prob_threshold() on the host): the valley between
// the error peak and the signal peak.  One thread; lets the ML-path kernel start without a host round trip.
__global__ void prob_thresh_kernel(const uint32_t* __restrict__ hist, int any_present, int fallback, double* __restrict__ out_f64,
                                   int* __restrict__ out_i32) {
    __shared__ uint32_t ph[200];  // three scans by one thread: from shared memory they cost ~1 us, from global ~20 us
    for (int i = threadIdx.x; i < 200; i += blockDim.x) ph[i] = hist[i];
    __syncthreads();
    if (threadIdx.x) return;
    int t = fallback;
    if (any_present) {
        int p1 = 0, p2 = -1;
        for (int i = 1; i < 200; ++i)
            if (ph[i] > ph[p1]) p1 = i;  // first maximum
        for (int i = 0; i < 200; ++i) {
            const int d = i > p1 ? i - p1 : p1 - i;
            if (d <= 10 || ph[i] == 0) continue;
            if (p2 < 0 || ph[i] > ph[p2]) p2 = i;
        }
        if (p2 < 0) {
            t = p1 - 200 - 10 > -200 ? p1 - 200 - 10 : -200;
        } else {
            const int a = p1 < p2 ? p1 : p2, b = p1 < p2 ? p2 : p1;
            int m = a;
            for (int i = a + 1; i <= b; ++i)
                if (ph[i] < ph[m]) m = i;  // first minimum
            t = m - 200;
        }
    }
    *out_i32 = t;
    *out_f64 = (double)t;
}

void launch_prob_thresh(const uint32_t* d_hist200, bool any_present, int fallback, double* d_thresh_f64, int* d_thresh_i32,
                        cudaStream_t st) {
    prob_thresh_kernel<<<1, 256, 0, st>>>(d_hist200, any_present ? 1 : 0, fallback, d_thresh_f64, d_thresh_i32);
    ++g_launches;
}

// One warp per locus.  The recurrence is a chain (node j needs its successors), and the choice
// among successors is order dependent (1e-6 tolerance, longer path wins ties), so lane 0 walks the
// nodes in reverse rank order; the windowed mean needs the node `window` steps down the chosen
// path, found in O(log window) with binary-lifting pointers instead of pandora's linear walk.
template <bool IN_SMEM, int LVT>
__device__ __forceinline__ void mlpath_chain(uint32_t n, double* __restrict__ M, double* __restrict__ mean,
                                             const double* __restrict__ prb, uint32_t* __restrict__ len,
                                             uint32_t* __restrict__ up, uint32_t up_stride,
                                             const uint32_t* __restrict__ eo, const uint32_t* __restrict__ ed,
                                             const ModelParams& P) {
    const double tol = 0.000001;
    const uint32_t term = n - 1;
    const uint32_t steps = P.window - 1;  // the node `window` steps down the chosen path = window-1 steps after v
    M[term] = 0.0;
    len[term] = 0;
    if (IN_SMEM) mean[term] = 0.0;  // never read: the terminus competes with the threshold instead
#pragma unroll
    for (int v = 0; v < LVT; ++v) up[v * up_stride + term] = term;
    for (uint32_t j = term; j-- > 0;) {
        double max_mean = -(double)FLT_MAX;
        uint32_t max_len = 0;
        double Mj = 0.0;
        uint32_t lenj = 0, prevj = term;
        const double pj = prb[j];
        const uint32_t e1 = eo[j + 1];
        for (uint32_t e = eo[j]; e < e1; ++e) {
            const uint32_t v = ed[e];
            const bool is_term = (v == term);
            const uint32_t lv = len[v];
            double mean_v = 0.0;
            if (!is_term) mean_v = IN_SMEM ? mean[v] : M[v] / (double)lv;
            const bool take = is_term ? (P.thresh > max_mean + tol)
                                      : ((mean_v > max_mean + tol) || (max_mean - mean_v <= tol && lv > max_len));
            if (!take) continue;
            Mj = pj + M[v];
            lenj = 1 + lv;
            prevj = v;
            if (lenj > P.window) {
                uint32_t pn = v;
#pragma unroll
                for (int b = 0; b < LVT; ++b)
                    if ((steps >> b) & 1u) pn = up[b * up_stride + pn];
                Mj -= prb[pn];
                lenj -= 1;
            }
            max_mean = is_term ? P.thresh : mean_v;
            if (!is_term) max_len = lv;
        }
        M[j] = Mj;
        len[j] = lenj;
        if (IN_SMEM) mean[j] = Mj / (double)lenj;  // 0/0 = NaN for a dead end: never chosen, like pandora
        up[j] = prevj;
        uint32_t a = prevj;
#pragma unroll
        for (int v = 1; v < LVT; ++v) {
            a = up[(v - 1) * up_stride + a];
            up[v * up_stride + j] = a;
        }
    }
}

template <int LVT>
__global__ void mlpath_kernel(uint32_t n_loci, const uint32_t* __restrict__ knode_base, const uint32_t* __restrict__ edge_off,
                              const uint32_t* __restrict__ edges, const double* __restrict__ prob,
                              const int32_t* __restrict__ locus_reads, ModelParams P, double* __restrict__ gM,
                              uint32_t* __restrict__ glen, uint32_t* __restrict__ gup, uint32_t total,
                              uint32_t* __restrict__ path, uint32_t* __restrict__ path_len, uint32_t smem_nodes,
                              uint32_t smem_edges) {
    extern __shared__ double s_dyn[];
    const uint32_t l = blockIdx.x;
    if (l >= n_loci) return;
    const uint32_t base = knode_base[l], n = knode_base[l + 1] - base;
    if (locus_reads[l] <= 0 || n < 2) {
        if (threadIdx.x == 0) path_len[l] = 0xffffffffu;
        return;
    }
    // The chain's whole working set lives in shared memory when the locus fits: running sum, cached mean
    // (sum / length: one fp64 division per node instead of one per edge visit), node score, length, the
    // binary-lifting pointers and the locus's CSR edges.  Every step of the serial dependency is then an
    // LDS with 32-bit addressing instead of an L2 round trip.
    const uint32_t e_base = edge_off[base], n_edges = edge_off[base + n] - e_base;
    const bool in_smem = n <= smem_nodes && n_edges <= smem_edges;
    const uint32_t term = n - 1;
    uint32_t cnt = 0;
    if (in_smem) {
        double* M = s_dyn;
        double* mean = s_dyn + smem_nodes;
        double* pr = s_dyn + 2 * (size_t)smem_nodes;
        uint32_t* len = (uint32_t*)(s_dyn + 3 * (size_t)smem_nodes);
        uint32_t* up = len + smem_nodes;
        uint32_t* s_eoff = up + (size_t)LVT * smem_nodes;
        uint32_t* s_edges = s_eoff + smem_nodes + 2;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) pr[i] = prob[base + i];
        for (uint32_t i = threadIdx.x; i <= n; i += blockDim.x) s_eoff[i] = edge_off[base + i] - e_base;
        for (uint32_t i = threadIdx.x; i < n_edges; i += blockDim.x) s_edges[i] = edges[e_base + i];
        __syncwarp();
        if (threadIdx.x != 0) return;
        mlpath_chain<true, LVT>(n, M, mean, pr, len, up, smem_nodes, s_eoff, s_edges, P);
        uint32_t p = up[0];
        while (p < term && cnt < n) {
            path[base + cnt++] = p;
            p = up[p];
        }
    } else {
        if (threadIdx.x != 0) return;
        uint32_t* up = gup + base;
        mlpath_chain<false, LVT>(n, gM + base, nullptr, prob + base, glen + base, up, total, edge_off + base, edges, P);
        uint32_t p = up[0];
        while (p < term && cnt < n) {
            path[base + cnt++] = p;
            p = up[p];
        }
    }
    path_len[l] = cnt;
}

// ---- level-parallel kernel ---------------------------------------------------------------------------------
// A node only needs its successors' finished records, so all nodes at the same distance-to-sink ("level": 1 + the
// largest level among the successors) are independent: the alleles of a bubble advance side by side.  The host
// sorts every locus by level, single-successor nodes first within a level.  A locus gets a CTA of four warps: warps
// 0-1 take the level's single-successor nodes, warps 2-3 the nodes with a choice, one node per lane, so the two code
// paths run on different schedulers instead of serialising inside one warp (a lone warp issues one instruction every
// ~6 cycles here: the kernel is bound by its own instruction latency, not by shared memory).  Each node runs the
// per-node step of the generic kernel's chain (successors still visited in rank order, so pandora's order-dependent
// tie-breaking is unchanged); the CTA synchronises between levels.  The serial chain shrinks from the number of nodes
// to the number of levels (benchmark panel: 38 251 nodes -> 15 128 levels, widest level 22 nodes).
//
// Node records are 64 bytes of shared memory, and every pointer the DP follows (successor, lifting pointers, window
// tail, edge targets, level lists) is stored as the 32-bit shared-memory ADDRESS of the target's record, so one hop is
// a single LDS with an immediate offset.  The generic kernel above spends ~160 instructions and ~1000 cycles per node,
// two thirds of it address arithmetic and dependent-issue waits (ncu: stall_wait 2.4, stall_short_scoreboard 2.6 per
// issued instruction).
constexpr uint32_t REC = 64;
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ double lds64(uint32_t a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v)); }
__device__ __forceinline__ void sts64(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v)); }

// sum / length on the level kernel's critical path.  The length is an integer <= 128, so the correctly rounded quotient
// comes from a table of correctly rounded reciprocals and two Markstein corrections (q += fma(-q, n, a) * y): five
// dependent FP64 operations instead of the ~15 of the generic division sequence.  The first correction makes q
// faithful, the second one makes it RN(a / n) because y = RN(1 / n) (Markstein's theorem; also checked against the
// hardware division on 7.7e8 random and adversarial operands, tools/divtest.c).  n == 0 gives NaN like 0.0 / 0.
__constant__ double c_rcp_small[129];
static void upload_rcp_table() {
    static std::mutex m;
    static uint64_t done_mask[4] = {0, 0, 0, 0};  // __constant__ memory is per device: one upload per device of the process
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> g(m);
    if (dev >= 0 && dev < 256 && (done_mask[dev >> 6] >> (dev & 63)) & 1ull) return;
    double h[129];
    h[0] = 0.0;
    for (int n = 1; n <= 128; ++n) h[n] = 1.0 / (double)n;
    if (cudaMemcpyToSymbol(c_rcp_small, h, sizeof h) != cudaSuccess) throw std::runtime_error("reciprocal table upload failed");
    if (dev >= 0 && dev < 256) done_mask[dev >> 6] |= 1ull << (dev & 63);
}
__device__ __forceinline__ double div_small(double a, uint32_t n) {
    if (n == 0u) return __longlong_as_double(0x7ff8000000000000ll);  // what 0.0 / 0 gives: never compares true
    const double y = c_rcp_small[n], b = (double)n;
    double q = a * y;
    q = fma(fma(-q, b, a), y, q);
    q = fma(fma(-q, b, a), y, q);
    return q;
}

// The record layout (64 B), arranged for vector shared-memory accesses: a lone warp per scheduler
// pays ~6 cycles per instruction, so fewer, wider accesses matter more than anything else here.
//   0 sum f64 | 8 mean f64 | 16 score f64 | 24 len u32 | 28 T u32 | 32 edge-list address u32 | 36 up[0..6] u32
// sum+mean come with one LDS.128, len+T with one LDS.64; up[1..6] sit at 40/48/56 and are stored as three STS.64.
constexpr uint32_t L_M = 0, L_MEAN = 8, L_PR = 16, L_LEN = 24, L_T = 28, L_EOFF = 32, L_UP = 36;
static_assert(L_MEAN == L_M + 8 && L_T == L_LEN + 4 && (L_UP + 4) % 8 == 0 && L_UP + 28 == REC, "vector accesses rely on this layout");
__device__ __forceinline__ void lds_sum_mean(uint32_t a, double& m, double& mean) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(m), "=d"(mean) : "r"(a + L_M));
}
__device__ __forceinline__ void lds_len_t(uint32_t a, uint32_t& len, uint32_t& t) {
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(len), "=r"(t) : "r"(a + L_LEN));
}
__device__ __forceinline__ void sts_pair32(uint32_t addr, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y));
}
// After the successor v of node a is known, two pointer chases remain, both through the records of finished nodes only
// and therefore independent of each other and of the fp chain: the lifting pointers of a (level l of a = level l-1 of the
// node 2^(l-1) steps down) and T(a) = succ^(window-2)(v).  Their loads are issued interleaved so the two chains overlap
// instead of adding up.  The stores are batched: up[0] | (up[1],up[2]) | (up[3],up[4]) | (up[5],up[6]); T is returned.
__device__ __forceinline__ uint32_t level_link(uint32_t a, uint32_t v, uint32_t steps2) {
    uint32_t up[7];
    up[0] = v;
    uint32_t x = v, t = v;
#pragma unroll
    for (int l = 0; l < 7; ++l) {
        const uint32_t xn = (l < 6) ? lds32(x + L_UP + 4 * l) : 0u;              // level l+1 of a
        const uint32_t tn = ((steps2 >> l) & 1u) ? lds32(t + L_UP + 4 * l) : t;  // walk window-2 steps from v
        if (l < 6) {
            up[l + 1] = xn;
            x = xn;
        }
        t = tn;
    }
    sts32(a + L_UP, up[0]);
    sts_pair32(a + L_UP + 4, up[1], up[2]);
    sts_pair32(a + L_UP + 12, up[3], up[4]);
    sts_pair32(a + L_UP + 20, up[5], up[6]);
    return t;
}

// The level order built at index load: the levels of locus l are locus_level_off[l] .. locus_level_off[l + 1] - 1, and
// level u holds the nodes level_nodes[level_start[u] .. level_start[u + 1]), single-successor nodes first.
struct MlLevelsDev {
    const uint32_t* locus_level_off;  // n_loci + 1 -> levels
    const uint32_t* level_start;      // n_levels + 1 -> level_nodes
    const uint32_t* level_nodes;      // ranks within the locus
};

constexpr int ML_LEVEL_THREADS = 128;
constexpr uint32_t ML_FAN = 4;  // successors whose records are fetched side by side (nodes with more take the serial loop)
__global__ void __launch_bounds__(ML_LEVEL_THREADS) mlpath_level_kernel(
    uint32_t n_loci, const uint32_t* __restrict__ knode_base, const uint32_t* __restrict__ edge_off,
    const uint32_t* __restrict__ edges, const double* __restrict__ prob, const int32_t* __restrict__ locus_reads,
    const uint8_t* __restrict__ needs_mean, MlLevelsDev L, const uint32_t* __restrict__ level_singles, ModelParams P,
    uint32_t* __restrict__ path, uint32_t* __restrict__ path_len, uint32_t max_nodes, uint32_t max_edges,
    volatile uint32_t* done,     // done != nullptr: path / path_len are host-mapped and done[l] tells the host that locus l is there
    const double* d_thresh) {    // != nullptr: the probability threshold is read from device memory (computed by prob_thresh_kernel)
    extern __shared__ double s_dyn[];
    const uint32_t l = blockIdx.x;
    if (l >= n_loci) return;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t base = knode_base[l], n = knode_base[l + 1] - base;
    if (locus_reads[l] <= 0 || n < 2) {
        if (tid == 0) {
            path_len[l] = 0xffffffffu;
            if (done) {
                __threadfence_system();
                done[l] = 1u;
            }
        }
        return;
    }
    const uint32_t e_base = edge_off[base], n_edges = edge_off[base + n] - e_base;
    const uint32_t recs = (uint32_t)__cvta_generic_to_shared(s_dyn);
    const uint32_t edg = recs + (max_nodes + 1) * REC;
    const uint32_t lvn = edg + (max_edges + 1) * 4u;  // record addresses in level order
    const uint32_t lvs = (lvn + max_nodes * 4u + 7u) & ~7u;  // per level: first index into lvn, number of single-successor nodes (8-byte aligned pairs)
    // The locus moves into shared memory in batches of four independent global loads per thread and array: one load per
    // iteration made the setup a chain of L2 round trips (25 us for the largest locus, measured)
    constexpr uint32_t UNR = 4, STEP = UNR * ML_LEVEL_THREADS;
    for (uint32_t i0 = tid; i0 <= n; i0 += STEP) {
        double pr[UNR];
        uint32_t eo[UNR], nm[UNR];
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) {
            const uint32_t i = i0 + u * ML_LEVEL_THREADS;
            pr[u] = i < n ? prob[base + i] : 0.0;
            eo[u] = i <= n ? edge_off[base + i] : 0u;
            nm[u] = i < n ? (uint32_t)needs_mean[base + i] : 0u;
        }
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) {
            const uint32_t i = i0 + u * ML_LEVEL_THREADS;
            const uint32_t a = recs + i * REC;
            if (i < n) sts64(a + L_PR, pr[u]);
            if (i <= n) sts32(a + L_EOFF, (edg + (eo[u] - e_base) * 4u) | nm[u]);
        }
    }
    for (uint32_t i0 = tid; i0 < n_edges; i0 += STEP) {
        uint32_t e[UNR];
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) e[u] = i0 + u * ML_LEVEL_THREADS < n_edges ? edges[e_base + i0 + u * ML_LEVEL_THREADS] : 0u;
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u)
            if (i0 + u * ML_LEVEL_THREADS < n_edges) sts32(edg + (i0 + u * ML_LEVEL_THREADS) * 4u, recs + e[u] * REC);
    }
    const uint32_t u0 = L.locus_level_off[l], n_levels = L.locus_level_off[l + 1] - u0;
    const uint32_t s00 = L.level_start[u0];
    for (uint32_t i0 = tid; i0 <= n_levels; i0 += STEP) {
        uint32_t us[UNR], ls[UNR];
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) {
            const uint32_t i = i0 + u * ML_LEVEL_THREADS;
            us[u] = i <= n_levels ? L.level_start[u0 + i] : 0u;
            ls[u] = i < n_levels ? level_singles[u0 + i] : 0u;
        }
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) {
            const uint32_t i = i0 + u * ML_LEVEL_THREADS;
            if (i <= n_levels) sts_pair32(lvs + 8u * i, us[u] - s00, ls[u]);
        }
    }
    for (uint32_t i0 = tid; i0 + 1 < n; i0 += STEP) {
        uint32_t un[UNR];
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u) un[u] = i0 + u * ML_LEVEL_THREADS + 1 < n ? L.level_nodes[s00 + i0 + u * ML_LEVEL_THREADS] : 0u;
#pragma unroll
        for (uint32_t u = 0; u < UNR; ++u)
            if (i0 + u * ML_LEVEL_THREADS + 1 < n) sts32(lvn + 4u * (i0 + u * ML_LEVEL_THREADS), recs + un[u] * REC);
    }
    const double tol = 0.000001;
    const double thresh = d_thresh ? *d_thresh : P.thresh;
    const uint32_t term = recs + (n - 1) * REC;
    const uint32_t steps2 = P.window - 2;
    if (tid == 0) {
        sts64(term + L_M, 0.0);
        sts_pair32(term + L_LEN, 0u, term);
#pragma unroll
        for (int v = 0; v < 7; ++v) sts32(term + L_UP + 4 * v, term);
    }
    __syncthreads();
    const bool single_warp = warp < 2;
    uint32_t sub = (warp & 1u) + 2u * lane;  // this lane's slot among the level's nodes of its kind (64 per pass)
    asm volatile("" : "+r"(sub));            // keep it in a register: recomputing it every level costs issue slots
    // level bounds: one LDS.64 per level ({first index, number of single-successor nodes} of the NEXT level; the
    // current pair is carried in registers)
    uint32_t s0, ns;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(s0), "=r"(ns) : "r"(lvs));
    for (uint32_t u = 0; u < n_levels; ++u) {
        uint32_t s1, ns1;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(s1), "=r"(ns1) : "r"(lvs + 8u * (u + 1)));
        const uint32_t lo = single_warp ? s0 : s0 + ns, hi = single_warp ? s0 + ns : s1;
        s0 = s1;
        ns = ns1;
        for (uint32_t idx = lo + sub; idx < hi; idx += 64) {
            const uint32_t a = lds32(lvn + 4u * idx);
            double Mj = 0.0;
            uint32_t lenj = 0, prevj = term;
            const double pj = lds64(a + L_PR);
            const uint32_t e0w = lds32(a + L_EOFF);
            const uint32_t e0 = e0w & ~3u;
            uint32_t Tj = term;
            if (single_warp) {
                // single successor: pandora's comparison against the initial -FLT_MAX accepts any successor that is
                // not a dead end
                const uint32_t v = lds32(e0);
                uint32_t lv, tv;
                lds_len_t(v, lv, tv);
                const double Mv = lds64(v + L_M);
                if (v == term || lv > 0u) {
                    Tj = level_link(a, v, steps2);  // independent of the sums below: overlaps them
                    prevj = v;
                    lenj = 1 + lv;
                    Mj = pj + Mv;
                    if (lenj > P.window) {
                        Mj -= lds64(tv + L_PR);
                        lenj -= 1;
                    }
                }
            } else {
                const uint32_t e1 = lds32(a + REC + L_EOFF) & ~3u;
                double max_mean = -(double)FLT_MAX;
                uint32_t max_len = 0;
                const uint32_t deg = (e1 - e0) >> 2;
                if (deg <= ML_FAN) {
                    // Up to ML_FAN successors (almost every node): everything the ordered comparison needs is fetched
                    // for ALL successors first — successor, its (length, window tail), (sum, mean) and the score that would
                    // leave the window — so the shared-memory latencies of the edges overlap instead of adding up
                    // (one edge after the other cost ~135-165 cycles each, measured); the comparison itself is pandora's
                    // sequential rule on registers, the arithmetic and its order are unchanged.
                    uint32_t vv[ML_FAN], lvv[ML_FAN], tvv[ML_FAN];
                    double Mvv[ML_FAN], meanv[ML_FAN], pT[ML_FAN];
#pragma unroll
                    for (uint32_t k = 0; k < ML_FAN; ++k) vv[k] = k < deg ? lds32(e0 + 4u * k) : term;
#pragma unroll
                    for (uint32_t k = 0; k < ML_FAN; ++k) {
                        lds_len_t(vv[k], lvv[k], tvv[k]);
                        lds_sum_mean(vv[k], Mvv[k], meanv[k]);
                    }
#pragma unroll
                    for (uint32_t k = 0; k < ML_FAN; ++k) pT[k] = lds64(tvv[k] + L_PR);
#pragma unroll
                    for (uint32_t k = 0; k < ML_FAN; ++k) {
                        if (k < deg) {
                            const bool is_term = (vv[k] == term);
                            const bool take = is_term ? (thresh > max_mean + tol)
                                                      : ((meanv[k] > max_mean + tol) || (max_mean - meanv[k] <= tol && lvv[k] > max_len));
                            if (take) {
                                Mj = pj + Mvv[k];
                                lenj = 1 + lvv[k];
                                prevj = vv[k];
                                if (lenj > P.window) {
                                    Mj -= pT[k];
                                    lenj -= 1;
                                }
                                max_mean = is_term ? thresh : meanv[k];
                                if (!is_term) max_len = lvv[k];
                            }
                        }
                    }
                } else
                for (uint32_t e = e0; e < e1; e += 4u) {
                    const uint32_t v = lds32(e);
                    const bool is_term = (v == term);
                    uint32_t lv, tv;
                    lds_len_t(v, lv, tv);
                    double Mv, mean_v;
                    lds_sum_mean(v, Mv, mean_v);
                    const bool take = is_term ? (thresh > max_mean + tol)
                                              : ((mean_v > max_mean + tol) || (max_mean - mean_v <= tol && lv > max_len));
                    if (!take) continue;
                    Mj = pj + Mv;
                    lenj = 1 + lv;
                    prevj = v;
                    if (lenj > P.window) {
                        Mj -= lds64(tv + L_PR);
                        lenj -= 1;
                    }
                    max_mean = is_term ? thresh : mean_v;
                    if (!is_term) max_len = lv;
                }
                if (lenj) Tj = level_link(a, prevj, steps2);
            }
            if (!lenj) {  // dead end (or no acceptable successor): points at the terminus like pandora's default
#pragma unroll
                for (int v = 0; v < 7; ++v) sts32(a + L_UP + 4 * v, term);
            }
            sts_pair32(a + L_LEN, lenj, Tj);
            if (e0w & 1u) {  // 0/0 = NaN for a dead end: never chosen, like pandora
                const double mean_j = div_small(Mj, lenj);
                asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a + L_M), "d"(Mj), "d"(mean_j));
            } else {
                sts64(a + L_M, Mj);
            }
        }
        __syncthreads();
    }
    // The chosen path, element i = the node i + 1 steps below the source: every thread walks to its own elements through
    // the lifting pointers (64-step hops, then the low bits) instead of one thread following 700 successor pointers one
    // after the other (18 us on the largest locus, measured).  The terminus points at itself on every level, so a walk
    // that overshoots stays there; the path ends at the first element that is the terminus.
    __shared__ uint32_t s_cnt;
    if (tid == 0) s_cnt = n;
    __syncthreads();
    for (uint32_t i0 = 0; i0 < n; i0 += ML_LEVEL_THREADS) {
        const uint32_t i = i0 + tid;
        uint32_t x = term;
        if (i < n) {
            x = recs;
            const uint32_t steps = i + 1;
            for (uint32_t q = steps >> 6; q; --q) x = lds32(x + L_UP + 4u * 6u);
#pragma unroll
            for (int b = 5; b >= 0; --b)
                if ((steps >> b) & 1u) x = lds32(x + L_UP + 4u * b);
            if (x != term) path[base + i] = (x - recs) / REC;
            else atomicMin(&s_cnt, i);
        }
        if (__syncthreads_or(x == term)) break;
    }
    if (done) __threadfence_system();  // this thread's part of the path, before the flag below
    __syncthreads();
    if (tid == 0) {
        path_len[l] = s_cnt;
        if (done) {  // the loci finish at different times (170 .. 860 levels): the host verifies each one as it lands
            __threadfence_system();
            done[l] = 1u;
        }
    }
}

bool launch_mlpath(uint32_t n_loci, const uint32_t* d_knode_base, const uint32_t* d_edge_off, const uint32_t* d_edges,
                   const double* d_prob, const int32_t* d_locus_reads, ModelParams P, double* d_M, uint32_t* d_len,
                   uint32_t* d_up, uint32_t total_knodes, uint32_t* d_path, uint32_t* d_path_len,
                   uint32_t max_locus_knodes, uint32_t max_locus_edges, const uint8_t* d_needs_mean, cudaStream_t st,
                   const uint32_t* d_locus_level_off, const uint32_t* d_level_start, const uint32_t* d_level_nodes,
                   const uint32_t* d_level_singles, uint32_t* h_path, uint32_t* h_path_len, uint32_t* h_done,
                   const double* d_thresh) {
    if (!n_loci) return false;
    // the level-parallel kernel when the largest locus fits in shared memory; otherwise the generic kernel below, which
    // DRPRG_MLPATH_GENERIC also forces
    static const bool force_generic = getenv("DRPRG_MLPATH_GENERIC") != nullptr;
    const size_t lvl_smem = ((size_t)max_locus_knodes + 1) * REC + (size_t)(max_locus_edges + 1) * 4 + (size_t)max_locus_knodes * 12 + 32;
    if (!force_generic && d_level_nodes && d_level_singles && d_needs_mean && P.window >= 2 && P.window <= 128 && lvl_smem <= 220u * 1024u) {
        ensure_dyn_smem(mlpath_level_kernel, lvl_smem);
        MlLevelsDev L{d_locus_level_off, d_level_start, d_level_nodes};
        upload_rcp_table();
        const bool streamed = h_path && h_path_len && h_done;  // results straight into host-mapped memory, locus by locus
        mlpath_level_kernel<<<n_loci, ML_LEVEL_THREADS, lvl_smem, st>>>(
            n_loci, d_knode_base, d_edge_off, d_edges, d_prob, d_locus_reads, d_needs_mean, L, d_level_singles, P,
            streamed ? h_path : d_path, streamed ? h_path_len : d_path_len, max_locus_knodes, max_locus_edges,
            streamed ? h_done : nullptr, d_thresh);
        ++g_launches;
        return streamed;
    }
    if (d_thresh) {  // the generic kernel takes the threshold by value: one small read-back
        double t = P.thresh;
        cudaMemcpyAsync(&t, d_thresh, sizeof t, cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        P.thresh = t;
    }
    // shared memory: per k-mer node sum, mean, score (f64), length, LV lifting pointers, edge offset (u32);
    // per edge one u32.  Up to the 227 KB a CTA may own; larger loci fall back to global memory.
    int LV = 1;
    while ((1u << LV) <= P.window && LV < LV_MAX) ++LV;
    LV = LV <= 7 ? 7 : LV_MAX;  // the two instantiated level counts
    const size_t per_node = 24 + 4 + 4 * (size_t)LV + 4;
    const size_t budget = 220u * 1024u;
    uint32_t smem_nodes = (max_locus_knodes + 3) & ~1u, smem_edges = max_locus_edges + 2;
    if ((size_t)smem_nodes * per_node + 16 + 4 * (size_t)smem_edges > budget) {  // biggest locus does not fit: size for the rest
        smem_nodes = (uint32_t)((budget / 2) / per_node) & ~1u;
        smem_edges = (uint32_t)((budget / 2) / 4);
    }
    const size_t smem = (size_t)smem_nodes * per_node + 16 + 4 * (size_t)smem_edges;
    auto go = [&](auto kernel) {
        ensure_dyn_smem(kernel, smem);
        kernel<<<n_loci, 32, smem, st>>>(n_loci, d_knode_base, d_edge_off, d_edges, d_prob, d_locus_reads, P, d_M, d_len, d_up,
                                         total_knodes, d_path, d_path_len, smem_nodes, smem_edges);
    };
    switch (LV) {  // levels needed for the window (pandora's default 100 -> 7)
        case 7: go(mlpath_kernel<7>); break;
        case 1: case 2: case 3: case 4: case 5: case 6: go(mlpath_kernel<7>); break;
        default: go(mlpath_kernel<LV_MAX>); break;
    }
    ++g_launches;
    return false;
}

}  // namespace drprg
