// Hand-written sm_100a kernels for the map hot path: read sketching + index lookup (S1+S2), hit
// clustering (S3/S4), k-mer coverage (S5), ML path (S7) and genotyping (S8).  These replace the
// per-read and per-locus loops of `pandora map` that drprg launches at
// /root/reference/src/lib.rs:580-642 (argv :594-609, src/predict.rs:288-294); stage semantics
// follow pandora's Seq::minimizer_sketch, add_read_hits, define_clusters, filter_clusters(2),
// add_hits_to_kmergraphs, KmerGraphWithCoverage::find_max_path and SampleInfo (SURVEY.md §8a).
// This file: S1 + S2 (read sketch, k-mer screen, index lookup).
#include <algorithm>
#include <cfloat>
#include <cstdlib>

#include "kernels_common.cuh"

namespace drprg {

std::atomic<uint64_t>& launch_counter() {
    static std::atomic<uint64_t> n{0};
    return n;
}
uint64_t launch_count() { return launch_counter().load(std::memory_order_relaxed); }

// ============================================================================================
// S1 + S2 : sketch + lookup.  One warp per read; lanes own consecutive k-mer positions.
//   * bases are 2-bit packed, first base in the top bits, so the forward k-mer at position p is a
//     funnel shift of two words and the reverse complement is brev + pair swap of its complement;
//   * k-mers are kept LEFT-ALIGNED in 32 bits (value << (32-2k)): every "& mask" of pandora's
//     hash64 becomes the natural 2^32 wrap, the three shift-add steps become single IMADs
//     (x2097151, x265, x21) and hash order is preserved, so the canonical min works in place;
//   * window minima with all ties (pandora keeps every k-mer attaining a window minimum) are a
//     sliding min followed by a sliding max of the minima, both by doubling in shared memory:
//     position i is a minimizer  <=>  h[i] == max over windows s containing i of min(h[s..s+w)).
// ============================================================================================
constexpr int WARPS = 8;
constexpr int EXT_MAX = CHUNK + 2 * (W_MAX - 1);
constexpr int BUF_N = EXT_MAX + W_MAX + 2;
constexpr int SW_N = (EXT_MAX + K_MAX + 15) / 16 + 3;

__device__ __forceinline__ uint32_t hash_left_aligned(uint32_t K, uint32_t S, uint32_t hm) {
    K = K * 2097151u - (1u << S);  // (~key + (key << 21)) & mask
    K ^= (K >> 24) & hm;           // key ^= key >> 24
    K *= 265u;                     // (key + (key << 3) + (key << 8)) & mask
    K ^= (K >> 14) & hm;
    K *= 21u;                      // (key + (key << 2) + (key << 4)) & mask
    K ^= (K >> 28) & hm;
    K += K << 31;                  // (key + (key << 31)) & mask : only bit 31 can change (k = 16)
    return K;
}

// hash of the k-mer held RIGHT-aligned (possibly with garbage above bit 2k): the left alignment (<< S) is folded
// into the first multiply
template <uint32_t S>
__device__ __forceinline__ uint32_t hash_right_aligned(uint32_t F) {
    constexpr uint32_t hm = ~((1u << S) - 1u);
    uint32_t K = F * (2097151u << S) - (1u << S);
    K ^= (K >> 24) & hm;
    K *= 265u;
    K ^= (K >> 14) & hm;
    K *= 21u;
    K ^= (K >> 28) & hm;
    return K;  // S >= 1: the final (key + (key << 31)) & mask step cannot change a kept bit
}

__device__ __forceinline__ uint32_t table_slot(uint32_t h, uint32_t bits) { return (h * 0x9E3779B1u) >> (32 - bits); }

// A slot's second word is rec_begin | rec_count << 24.  A minimizer that occurs in 255 or more k-mer nodes (repetitive
// or heavily nested PRGs; pandora has no limit) stores 255 there and its real count in a header pseudo-record
// {count, 0xffffffff} in front of its records.
constexpr uint32_t REC_COUNT_ESCAPE = 255u;
__device__ __forceinline__ void rec_span(const uint2* __restrict__ recs, uint32_t y, uint32_t& begin, uint32_t& n) {
    begin = y & 0xffffffu;
    n = y >> 24;
    if (n == REC_COUNT_ESCAPE) {
        n = __ldg(recs + begin).x;
        ++begin;
    }
}

template <bool LOOKUP>
__global__ void __launch_bounds__(WARPS * 32) sketch_kernel(DevReads R, DevTable T, uint32_t w, uint32_t k,
                                                           unsigned long long* __restrict__ out_a,
                                                           unsigned long long* __restrict__ out_b,
                                                           unsigned long long* __restrict__ out_count,
                                                           unsigned long long cap) {
    __shared__ uint32_t s_words[WARPS][SW_N];
    __shared__ uint32_t s_h[WARPS][BUF_N];
    __shared__ uint32_t s_a[WARPS][BUF_N];
    __shared__ uint32_t s_b[WARPS][BUF_N];
    __shared__ uint32_t s_strand[WARPS][(EXT_MAX + 31) / 32 + 1];

    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t* sw = s_words[wid];
    uint32_t* H = s_h[wid];
    uint32_t* A = s_a[wid];
    uint32_t* B = s_b[wid];
    uint32_t* SS = s_strand[wid];
    const uint32_t S = 32 - 2 * k;
    const uint32_t hm = (S == 0) ? 0xffffffffu : ~((1u << S) - 1u);
    const unsigned long long nwarps = (unsigned long long)gridDim.x * WARPS;

    for (unsigned long long r = (unsigned long long)blockIdx.x * WARPS + wid; r < R.n_reads; r += nwarps) {
        const uint32_t len = R.lens[r];
        if (len + 1 < w + k) continue;  // too short, or flagged 0 (non-ACGT): contributes nothing
        const uint32_t nk = len - k + 1;
        const unsigned long long wbase = R.stride_words ? r * R.stride_words : R.word_off[r];
        const uint32_t nwords_read = (len + 15) >> 4;

        for (uint32_t c0 = 0; c0 < nk; c0 += CHUNK) {
            const uint32_t ext_lo = (c0 >= w - 1) ? c0 - (w - 1) : 0;
            const uint32_t ext_hi = min(c0 + CHUNK + (w - 1), nk);
            const uint32_t n_ext = ext_hi - ext_lo;
            const uint32_t w0 = ext_lo >> 4;
            const uint32_t nw = ((ext_hi + k - 2) >> 4) - w0 + 1;
            __syncwarp();
            for (uint32_t i = lane; i < nw + 1; i += 32) {
                uint32_t wi = w0 + i;
                sw[i] = (wi < nwords_read) ? __ldg(R.words + wbase + wi) : 0u;
            }
            __syncwarp();
            // ---- canonical hashes of positions [ext_lo, ext_hi)
            for (uint32_t e0 = 0; e0 < n_ext; e0 += 32) {
                const uint32_t e = e0 + lane;
                const uint32_t b = 2u * (ext_lo + e - (w0 << 4));
                const uint32_t wi = min(b >> 5, nw - 1);
                const uint32_t v = __funnelshift_l(sw[wi + 1], sw[wi], b & 31u);
                const uint32_t F = v & hm;
                uint32_t y = __brev(~v & hm);
                y = ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
                const uint32_t Rc = y << S;
                const uint32_t hf = hash_left_aligned(F, S, hm), hr = hash_left_aligned(Rc, S, hm);
                const bool valid = e < n_ext;
                if (valid) H[e] = min(hf, hr);
                const uint32_t bal = __ballot_sync(FULL, valid && hf <= hr);
                if (lane == 0) SS[e0 >> 5] = bal;
            }
            __syncwarp();
            // ---- sliding minimum over w consecutive hashes: wm[e] = min(H[e .. e+w-1])
            uint32_t span = 1;
            const uint32_t* src = H;
            uint32_t* dst = A;
            while (span * 2 <= w) {
                const uint32_t cnt = n_ext - (2 * span - 1);
                for (uint32_t e = lane; e < cnt; e += 32) dst[e] = min(src[e], src[e + span]);
                __syncwarp();
                src = dst;
                dst = (dst == A) ? B : A;
                span *= 2;
            }
            // padded array P[t], t in [0, n_ext + w - 1): windows start at ext_lo - (w-1) + t
            const uint32_t n_win = n_ext - w + 1;
            const uint32_t n_pad = n_ext + w - 1;
            for (uint32_t t = lane; t < n_pad; t += 32) {
                uint32_t val = 0;
                if (t >= w - 1 && t - (w - 1) < n_win) {
                    const uint32_t e = t - (w - 1);
                    val = min(src[e], src[e + w - span]);
                }
                dst[t] = val;
            }
            __syncwarp();
            // ---- sliding maximum of the window minima: X[e] = max(P[e .. e+w-1])
            src = dst;
            dst = (dst == A) ? B : A;
            span = 1;
            while (span * 2 <= w) {
                const uint32_t cnt = n_pad - (2 * span - 1);
                for (uint32_t t = lane; t < cnt; t += 32) dst[t] = max(src[t], src[t + span]);
                __syncwarp();
                src = dst;
                dst = (dst == A) ? B : A;
                span *= 2;
            }
            // ---- minimizers of this chunk
            const uint32_t chunk_hi = min(c0 + CHUNK, nk);
            for (uint32_t p0 = c0; p0 < chunk_hi; p0 += 32) {
                const uint32_t p = p0 + lane;
                const uint32_t e = p - ext_lo;
                bool is_min = false;
                uint32_t hv = 0;
                if (p < chunk_hi) {
                    const uint32_t x = max(src[e], src[e + w - span]);
                    hv = H[e];
                    is_min = (hv == x);
                    hv >>= S;
                }
                const uint32_t read_strand = (SS[e >> 5] >> (e & 31)) & 1u;
                if (!LOOKUP) {
                    const uint32_t bal = __ballot_sync(FULL, is_min);
                    if (bal) {
                        unsigned long long base = 0;
                        if (lane == 0) base = atomicAdd(out_count, (unsigned long long)__popc(bal));
                        base = __shfl_sync(FULL, base, 0);
                        if (is_min) {
                            const unsigned long long o = base + __popc(bal & ((1u << lane) - 1u));
                            if (o < cap) {
                                out_a[o] = ((unsigned long long)(R.read_id_base + (uint32_t)r) << 32) | p;
                                out_b[o] = ((unsigned long long)hv << 1) | read_strand;
                            }
                        }
                    }
                } else {
                    bool pass = false;
                    if (is_min) {
                        const uint32_t fw = __ldg(T.filter + (hv & ((1u << T.filter_bits) - 1u)));
                        const uint32_t m = (1u << ((hv >> T.filter_bits) & 31u)) | (1u << ((hv >> (T.filter_bits + 5)) & 31u));
                        pass = (fw & m) == m;
                    }
                    if (__any_sync(FULL, pass)) {
                        uint32_t rec_begin = 0, rec_n = 0;
                        if (pass) {
                            uint32_t slot = table_slot(hv, T.slot_bits);
                            const uint32_t smask = (1u << T.slot_bits) - 1u;
                            while (true) {
                                const uint2 ent = __ldg(T.slots + slot);
                                if (ent.y == 0u) break;
                                if (ent.x == hv) {
                                    rec_span(T.recs, ent.y, rec_begin, rec_n);
                                    break;
                                }
                                slot = (slot + 1) & smask;
                            }
                        }
                        // warp-aggregated append
                        uint32_t incl = rec_n;
#pragma unroll
                        for (int d = 1; d < 32; d <<= 1) {
                            const uint32_t t = __shfl_up_sync(FULL, incl, d);
                            if (lane >= d) incl += t;
                        }
                        const uint32_t total = __shfl_sync(FULL, incl, 31);
                        if (total) {
                            unsigned long long base = 0;
                            if (lane == 0) {
                                base = atomicAdd(out_count, (unsigned long long)total);
                                if (R.hit_count) atomicAdd(R.hit_count + r, (int32_t)total);
                            }
                            base = __shfl_sync(FULL, base, 0) + (incl - rec_n);
                            for (uint32_t j = 0; j < rec_n; ++j) {
                                const uint2 rc = __ldg(T.recs + rec_begin + j);
                                const uint32_t fwd = ((rc.y & 1u) == read_strand) ? 1u : 0u;
                                if (base + j < cap) {
                                    out_a[base + j] = ((unsigned long long)(R.read_id_base + (uint32_t)r) << 32) |
                                                      ((unsigned long long)(rc.y >> 1) << 16) | ((unsigned long long)(fwd ^ 1u) << 15);
                                    out_b[base + j] = ((unsigned long long)p << 32) | rc.x;
                                }
                            }
                        }
                    }
                }
            }
        }
    }
}

// ============================================================================================
// S1 + S2, short reads (Illumina): ONE THREAD PER READ, W and K compile-time.
// The warp-per-read kernel above spends ~90 % of its issue slots on the shared-memory min/max passes
// and partial rounds (ncu: 1236 warp instructions per 150 bp read, hashing only 8 % of them).  Here all
// 32 lanes of a warp walk 32 different reads in lockstep, everything lives in registers and the
// per-position cost is ~50 instructions:
//   * rolling k-mers: forward by one funnel shift taking the next base from the top of the current
//     word, reverse complement by one funnel shift taking the complemented base from a rotating copy;
//   * window minima with ties by the van Herk / Gil-Werman block decomposition with block = W and the
//     loop unrolled by W so every array index is static: prefix/suffix minima give the minimum of each
//     window, prefix/suffix maxima of those give, per position, the largest window minimum among the
//     windows containing it; position i is a minimizer iff h[i] equals that value;
//   * positions past the read end (and windows before its start) carry hash 0 == "-infinity": a window
//     touching them has minimum 0 and so can never certify a real minimizer (a real hash of 0 is the
//     minimum of its valid windows anyway), which removes every boundary branch;
//   * the block's hashes are parked in shared memory ([slot][thread], conflict free) only so that the
//     rare flagged positions can be fetched with a dynamic index when they probe the index.
// ============================================================================================
constexpr int SHORT_THREADS = 512;
constexpr uint32_t SMEM_FILTER_BITS = 14;  // a pre-filter of <= 2^14 words (64 KB) is copied into shared memory
#ifndef DRPRG_DEFAULT_VARIANT
#define DRPRG_DEFAULT_VARIANT 3
#endif

template <int W, int K, bool LOOKUP, int VARIANT, bool SMEM_FILTER, int THREADS>
__global__ void __launch_bounds__(THREADS) sketch_short_kernel(DevReads R, DevTable T,
                                                                     unsigned long long* __restrict__ out_a,
                                                                     unsigned long long* __restrict__ out_b,
                                                                     unsigned long long* __restrict__ out_count,
                                                                     unsigned long long cap) {
    static_assert(K >= 2 && K <= 15, "left-aligned hash with a spare low bit range needs k <= 15");
    constexpr uint32_t S = 32 - 2 * K;
    constexpr uint32_t HM = ~((1u << S) - 1u);
    extern __shared__ uint32_t s_short[];
    uint32_t(*s_h)[W][THREADS] = reinterpret_cast<uint32_t(*)[W][THREADS]>(s_short);
    const uint32_t* s_filter = s_short + 2 * W * THREADS;
    const int tid = threadIdx.x;
    if (LOOKUP && SMEM_FILTER) {  // "hot buckets in shared memory": the whole negative filter, once per persistent CTA
        uint32_t* f = s_short + 2 * W * THREADS;
        const uint32_t nwf = 1u << T.filter_bits;
        for (uint32_t i = tid * 4; i < nwf; i += THREADS * 4)
            *reinterpret_cast<uint4*>(f + i) = __ldg(reinterpret_cast<const uint4*>(T.filter + i));
        __syncthreads();
    }
    // A work item is a whole read, or — for long reads — a SEGMENT of one (R.seg_read != nullptr): seg_len k-mer
    // positions whose minimizer status only depends on the w-1 positions either side, so a thread streams
    // [seg_start-(w-1), seg_end+(w-1)) and reports [seg_start, seg_end).  Padding with hash 0 outside the streamed
    // range is exact at the true read ends and harmless inside the read (it only affects the halo).
    const unsigned long long n_items = R.seg_read ? R.n_segs : R.n_reads;
    const unsigned long long n_tiles = (n_items + THREADS - 1) / THREADS;
    for (unsigned long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const unsigned long long item = tile * THREADS + tid;
    const bool have = item < n_items;
    const unsigned long long r = have ? (R.seg_read ? (unsigned long long)__ldg(R.seg_read + item) : item) : 0ull;
    uint32_t len = have ? __ldg(R.lens + r) : 0u;
    if (len + 1 < (uint32_t)(W + K)) len = 0;  // too short or dropped: no k-mer position is valid
    const uint32_t nk_read = len ? len - K + 1 : 0;
    const uint32_t seg_s = (have && R.seg_read) ? __ldg(R.seg_start + item) : 0u;
    const uint32_t seg_e = R.seg_read ? min(seg_s + R.seg_len, nk_read) : nk_read;   // report [seg_s, seg_e)
    const uint32_t str_lo = seg_s >= (uint32_t)(W - 1) ? seg_s - (W - 1) : 0u;        // stream [str_lo, str_lo + nk)
    const uint32_t nk = nk_read ? min(nk_read, seg_e + (W - 1)) - str_lo : 0u;
    const uint32_t nk_max = __reduce_max_sync(FULL, nk);
    if (nk_max == 0) continue;
    const uint32_t nk_min = __reduce_min_sync(FULL, nk);
    const uint32_t* wp = R.words + (have ? (R.stride_words ? r * R.stride_words : __ldg(R.word_off + r)) : 0ull) + (str_lo >> 4);
    const uint32_t nwords = ((len + 15) >> 4) - (nk_read ? (str_lo >> 4) : 0u);

    // Bases are served from a 64-bit shift register (hi:lo) holding `avail` bases, top aligned; it is
    // topped up with the next 16-base word once per block of W positions (W <= 16 bases are consumed per
    // block), so the refill test is per block, not per base, and warp-uniform: all lanes are in lockstep.
    static_assert(W <= 16, "one refill per block must cover the block");
    uint32_t hi = 0, lo = 0, avail = 0, widx = 0, F = 0, Rc = 0;
    uint32_t wnext = nwords ? __ldg(wp) : 0u;  // always one word ahead: the load has a whole block to land
    auto refill = [&]() {
        if (avail <= 16u) {
            const uint32_t word = wnext;
            ++widx;
            wnext = (widx < nwords) ? __ldg(wp + widx) : 0u;
            const uint32_t t = 2u * avail;  // 0..32 bits already occupied at the top of hi; lo is empty
            hi |= __funnelshift_rc(word, 0u, t);
            lo = __funnelshift_rc(0u, word, t);
            avail += 16u;
        }
    };
    auto next_base = [&]() {
        const uint32_t c = hi >> 30;
        hi = __funnelshift_l(lo, hi, 2);
        lo <<= 2;
        F = F * 4u + c;                                     // garbage above bit 2K wraps away in the first hash multiply
        Rc = (__funnelshift_r(Rc, c, 2) & HM) ^ 0xC0000000u;  // complemented base enters at the top; bases older than K fall off
    };
    {
        // skip to the first streamed base inside its word, then prime the first K-1 bases
        const uint32_t prime = (str_lo & 15u) + (uint32_t)(K - 1);
#pragma unroll 1
        for (uint32_t i = 0; i < prime; ++i) {
            refill();
            next_base();
            --avail;
        }
    }

    uint32_t hp[W], Sp[W], SXo[W + 1];
#pragma unroll
    for (int j = 0; j < W; ++j) hp[j] = Sp[j] = SXo[j] = 0u;
    SXo[W] = 0u;
    uint32_t strand_prev = 0;
    const uint32_t n_blocks = (nk_max + W - 1) / W + 1;  // one extra all-padding block resolves the last real one
#pragma unroll 1
    for (uint32_t b = 0; b < n_blocks; ++b) {
        uint32_t h[W];
        uint32_t not_strand = 0;  // bit (W-1-j) = !(hf <= hr) of position j
        const uint32_t p0 = b * W;
        uint32_t* sh = &s_h[b & 1][0][tid];
        refill();
        avail -= (uint32_t)W;
        // blocks that lie inside every lane's read (all but the last one or two) may skip the per-position padding select
        auto strand_bit = [&](uint32_t hf, uint32_t hr, int j) {
            if (VARIANT & 1)
                asm("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(not_strand) : "r"(hf), "r"(hr), "r"(1u << (W - 1 - j)));
            else
                not_strand |= (hf > hr ? 1u : 0u) << (W - 1 - j);
        };
        if ((VARIANT & 2) && p0 + W <= nk_min) {
#pragma unroll
            for (int j = 0; j < W; ++j) {
                next_base();
                const uint32_t hf = hash_right_aligned<S>(F), hr = hash_left_aligned(Rc, S, HM);
                const uint32_t hv = min(hf, hr);
                strand_bit(hf, hr, j);
                h[j] = hv;
                sh[j * THREADS] = hv;
            }
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j) {
                next_base();
                const uint32_t hf = hash_right_aligned<S>(F), hr = hash_left_aligned(Rc, S, HM);
                uint32_t hv = min(hf, hr);
                strand_bit(hf, hr, j);
                hv = (p0 + j < nk) ? hv : 0u;
                h[j] = hv;
                sh[j * THREADS] = hv;
            }
        }
        const uint32_t strand_cur = ~not_strand;
        // windows starting in the previous block: offset t covers prev[t..W-1] + cur[0..t-1]
        uint32_t wm[W];
        wm[0] = Sp[0];
        {
            uint32_t pmin = h[0];
#pragma unroll
            for (int t = 1; t < W; ++t) {
                wm[t] = min(Sp[t], pmin);
                pmin = min(pmin, h[t]);
            }
        }
        // previous block's positions: best window minimum among the windows containing them
        uint32_t flags = 0;
        {
            uint32_t pmax = 0;
#pragma unroll
            for (int j = 0; j < W; ++j) {
                pmax = max(pmax, wm[j]);
                const uint32_t best = max(pmax, SXo[j + 1]);
                if (VARIANT & 1)
                    asm("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(flags) : "r"(hp[j]), "r"(best), "r"(1u << j));
                else
                    flags |= (hp[j] == best ? 1u : 0u) << j;
            }
        }
        if (b > 0) {
            const uint32_t prev0 = str_lo + p0 - W;  // read coordinate of the previous block's first position
            // positions to report: prev0 + j in [seg_s, seg_e)
            const uint32_t first = seg_s > prev0 ? min(seg_s - prev0, (uint32_t)W) : 0u;
            const uint32_t last = seg_e > prev0 ? min(seg_e - prev0, (uint32_t)W) : 0u;
            uint32_t fm = flags & ((1u << last) - 1u) & ~((1u << first) - 1u);
            while (fm) {
                const int j = __ffs(fm) - 1;
                fm &= fm - 1;
                const uint32_t hv = s_h[(b - 1) & 1][j][tid] >> S;
                const uint32_t pos = prev0 + j;
                const uint32_t read_strand = (strand_prev >> (W - 1 - j)) & 1u;
                if (!LOOKUP) {
                    const unsigned long long o = atomicAdd(out_count, 1ull);
                    if (o < cap) {
                        out_a[o] = ((unsigned long long)(R.read_id_base + (uint32_t)r) << 32) | pos;
                        out_b[o] = ((unsigned long long)hv << 1) | read_strand;
                    }
                } else {
                    const uint32_t fidx = hv & ((1u << T.filter_bits) - 1u);
                    const uint32_t fw = SMEM_FILTER ? s_filter[fidx] : __ldg(T.filter + fidx);
                    // both filter bits set?  (funnel shifts take the shift amount modulo 32)
                    const uint32_t hb = hv >> T.filter_bits;
                    if (!(__funnelshift_r(fw, 0u, hb) & __funnelshift_r(fw, 0u, hb >> 5) & 1u)) continue;
                    uint32_t slot = table_slot(hv, T.slot_bits);
                    const uint32_t smask = (1u << T.slot_bits) - 1u;
                    uint32_t rec_begin = 0, rec_n = 0;
                    while (true) {
                        const uint2 ent = __ldg(T.slots + slot);
                        if (ent.y == 0u) break;
                        if (ent.x == hv) {
                            rec_span(T.recs, ent.y, rec_begin, rec_n);
                            break;
                        }
                        slot = (slot + 1) & smask;
                    }
                    if (rec_n) {
                        const unsigned long long base = atomicAdd(out_count, (unsigned long long)rec_n);
                        if (R.hit_count) atomicAdd(R.hit_count + r, (int32_t)rec_n);
                        for (uint32_t q = 0; q < rec_n; ++q) {
                            const uint2 rc = __ldg(T.recs + rec_begin + q);
                            const uint32_t fwd = ((rc.y & 1u) == read_strand) ? 1u : 0u;
                            if (base + q < cap) {
                                out_a[base + q] = ((unsigned long long)(R.read_id_base + (uint32_t)r) << 32) |
                                                  ((unsigned long long)(rc.y >> 1) << 16) | ((unsigned long long)(fwd ^ 1u) << 15);
                                out_b[base + q] = ((unsigned long long)pos << 32) | rc.x;
                            }
                        }
                    }
                }
            }
        }
        // roll the block state
        {
            uint32_t smax = 0;
#pragma unroll
            for (int j = W - 1; j >= 0; --j) {
                smax = max(smax, wm[j]);
                SXo[j] = smax;
            }
            uint32_t smin = 0xffffffffu;
#pragma unroll
            for (int j = W - 1; j >= 0; --j) {
                smin = min(smin, h[j]);
                Sp[j] = smin;
                hp[j] = h[j];
            }
        }
        strand_prev = strand_cur;
    }
    }  // persistent tile loop
}

template <int W, int K, bool LOOKUP, int V, bool SF>
static void launch_short_one(const DevReads& R, const DevTable& T, unsigned long long* a, unsigned long long* b,
                             unsigned long long* cnt, uint64_t cap, int sm_count, cudaStream_t st) {
    const size_t smem = (size_t)2 * W * SHORT_THREADS * 4 + (SF ? (size_t)4 << T.filter_bits : 0);
    ensure_dyn_smem(sketch_short_kernel<W, K, LOOKUP, V, SF, SHORT_THREADS>, (size_t)(2 * W * SHORT_THREADS * 4 + (SF ? (4u << SMEM_FILTER_BITS) : 0)));
    // persistent CTAs: two per SM (register file: 2 x 512 threads x 62 registers), each loops over read tiles
    const unsigned long long n_items = R.seg_read ? R.n_segs : R.n_reads;
    const unsigned long long n_tiles = (n_items + SHORT_THREADS - 1) / SHORT_THREADS;
    const unsigned grid = (unsigned)std::min<unsigned long long>(n_tiles, 2ull * (unsigned)sm_count);
    sketch_short_kernel<W, K, LOOKUP, V, SF, SHORT_THREADS><<<grid, SHORT_THREADS, smem, st>>>(R, T, a, b, cnt, cap);
    ++g_launches;
}

template <bool LOOKUP>
static bool launch_short(const DevReads& R, const DevTable& T, uint32_t w, uint32_t k, unsigned long long* a,
                         unsigned long long* b, unsigned long long* cnt, uint64_t cap, int sm_count, cudaStream_t st) {
    // two instantiations per (w,k): the default (predicated-OR flag accumulation + padding-free fast path, the fastest
    // of the four variants measured in round 1) and the plain one as the fallback / second implementation
    // (DRPRG_SKETCH_VARIANT=0, exercised by the parity tests)
    static const bool plain = [] {
        const char* e = getenv("DRPRG_SKETCH_VARIANT");
        return e && atoi(e) == 0;
    }();
    const bool sf = LOOKUP && T.filter_bits <= SMEM_FILTER_BITS;
#define DRPRG_SHORT_V(WW, KK, VV)                                                                             \
    {                                                                                                         \
        if (!LOOKUP) launch_short_one<WW, KK, LOOKUP, VV, false>(R, T, a, b, cnt, cap, sm_count, st);         \
        else if (sf) launch_short_one<WW, KK, LOOKUP, VV, LOOKUP>(R, T, a, b, cnt, cap, sm_count, st);        \
        else launch_short_one<WW, KK, LOOKUP, VV, false>(R, T, a, b, cnt, cap, sm_count, st);                 \
        return true;                                                                                          \
    }
#define DRPRG_SHORT(WW, KK)                                 \
    if (w == WW && k == KK) {                               \
        if (plain && LOOKUP) DRPRG_SHORT_V(WW, KK, 0)       \
        DRPRG_SHORT_V(WW, KK, DRPRG_DEFAULT_VARIANT)        \
    }
    DRPRG_SHORT(11, 15)  // drprg defaults (src/builder.rs:40-41)
    DRPRG_SHORT(14, 15)  // pandora's default w, used by the reference's build tests (src/builder.rs:1181)
#undef DRPRG_SHORT
#undef DRPRG_SHORT_V
    return false;
}

// ============================================================================================
// K-mer screen.  ~99 % of whole-genome reads share no k-mer with the panel, yet the sketch above spends
// ~70 instructions per k-mer position on them (two hashes + window minima).  pandora's hash64 is a
// bijection on 2k-bit values, so "this minimizer is in the index" implies "this FORWARD k-mer of the read is
// one of the indexed k-mers or their reverse complements" — a set-membership test on the raw 2-bit k-mer
// that needs no hash and no window logic.
//   screen_kernel   streams every read once (a warp takes 32 reads at a time from a global ticket counter,
//                   words in registers) and tests each k-mer against a blocked 2-bit Bloom filter held in
//                   shared memory: one multiply, one LDS, two shifts, ~10 instructions per position.  The
//                   flagged positions (~1 % false positives + the real ones) are appended to a queue.
//   resolve_kernel  persistent warps, several queued (read, position) pairs per lane: canonical hash of each k-mer,
//                   index probes side by side (exact, drops the false positives), survivors collected in a per-warp
//                   shared-memory ring and tested 32 at a time — a position is a (w,k)-minimizer with pandora's
//                   "all ties kept" rule iff the run of neighbours whose hash is >= its own covers a whole window —
//                   then the hit records (details above the kernel).
// The hits are the same set the full sketch + lookup kernels emit; only ~2 % of the positions ever get hashed.
// ============================================================================================
constexpr int SCREEN_THREADS = 1024;
constexpr uint32_t SCREEN_MUL = 0x9E3779B1u;

void screen_filter_insert(uint32_t* filter, uint32_t n_words, uint32_t kmer, uint32_t k) {
    const uint32_t p = kmer * (SCREEN_MUL << (32u - 2u * k));  // bits above 2k wrap away
    const uint32_t idx = (uint32_t)(((unsigned long long)p * n_words) >> 32);
    filter[idx] |= (1u << (kmer & 31u)) | (1u << ((p >> 11) & 31u));
}

// V: pipe-balance variants (the ALU pipe — SHF/LOP3/LEA — binds first, the multiplier pipe has room):
//   bit 0: shared-memory address by IMAD with a run-time 4 instead of LEA;  bit 1: the second bit index by
//   multiply-high with a run-time 2^21 instead of a shift;  bit 2: the flag of a position shifted into its word by a
//   multiply-add instead of a compare + predicated OR.  Default 5 (bits 0 and 2): measured 0.152 ms against 0.155 for 1
//   and 0.159 for 0 per million reads; bit 1 never paid.
struct ScreenConsts { uint32_t four, two21, prefetch, two; };
template <int K, int CW, int V>
__global__ void __launch_bounds__(SCREEN_THREADS, 1) screen_kernel(DevReads R, DevTable T, uint32_t wk, ScreenConsts SC,
                                                                   unsigned long long* __restrict__ queue,
                                                                   uint32_t* __restrict__ queue_kmer,
                                                                   unsigned long long* __restrict__ queue_count,
                                                                   unsigned long long queue_cap,
                                                                   unsigned long long* __restrict__ ticket) {
    static_assert(K >= 8 && K <= 15, "the filter bit choice needs >= 16 k-mer bits; 2k < 32");
    constexpr int NF = (CW + 1) / 2;
    extern __shared__ uint32_t s_kf[];
    const int tid = threadIdx.x, lane = tid & 31;
    for (uint32_t i = tid * 4; i < T.kfilter_words; i += SCREEN_THREADS * 4)
        *reinterpret_cast<uint4*>(s_kf + i) = __ldg(reinterpret_cast<const uint4*>(T.kfilter + i));
    __syncthreads();
    const uint32_t n_fw = T.kfilter_words;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(s_kf);
    const unsigned long long n_items = R.seg_read ? R.n_segs : R.n_reads;
    const unsigned long long n_tiles = (n_items + 31) / 32;
    const bool wide = R.stride_words && !(R.stride_words & 1u) && !R.seg_read &&
                      (reinterpret_cast<unsigned long long>(R.words) & 7ull) == 0ull;  // every read starts 8-byte aligned
    // tickets are drawn two tiles ahead: the next tile's id is known when a tile starts, so its words can be
    // prefetched into L2 while this tile is screened (a cold read otherwise costs the full HBM latency per tile)
    unsigned long long tile = 0, next_tile = 0;
    if (lane == 0) {
        tile = atomicAdd(ticket, 1ull);
        next_tile = atomicAdd(ticket, 1ull);
    }
    tile = __shfl_sync(FULL, tile, 0);
    next_tile = __shfl_sync(FULL, next_tile, 0);
    while (tile < n_tiles) {
        unsigned long long after_next = 0;
        if (lane == 0) after_next = atomicAdd(ticket, 1ull);  // lands while this tile is screened
        if (SC.prefetch && !R.seg_read && R.stride_words && next_tile * 32 + lane < n_items) {
            const uint32_t* np = R.words + (next_tile * 32 + lane) * R.stride_words;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(np));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(np + R.stride_words - 1));
            if (lane == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(R.lens + next_tile * 32));
        }
        const unsigned long long item = tile * 32 + lane;
        const bool have = item < n_items;
        const unsigned long long r = have ? (R.seg_read ? (unsigned long long)__ldg(R.seg_read + item) : item) : 0ull;
        uint32_t len = have ? __ldg(R.lens + r) : 0u;
        if (len + 1 < wk) len = 0;  // too short or dropped: the sketch skips it too
        const uint32_t nk_read = len ? len - K + 1 : 0;
        const uint32_t seg_s = (have && R.seg_read) ? __ldg(R.seg_start + item) : 0u;
        const uint32_t seg_e = R.seg_read ? min(seg_s + R.seg_len, nk_read) : nk_read;  // screen positions [seg_s, seg_e)
        const uint32_t q0 = seg_s & ~15u;                                             // streamed from a word boundary
        const uint32_t span = seg_e > seg_s ? seg_e - q0 : 0u;
        const uint32_t span_max = __reduce_max_sync(FULL, span);
        const uint32_t* wp = R.words + (have ? (R.stride_words ? r * R.stride_words : __ldg(R.word_off + r)) : 0ull) + (q0 >> 4);
        const uint32_t nwords = span ? ((len + 15) >> 4) - (q0 >> 4) : 0u;  // words that may be read from wp
#pragma unroll 1
        for (uint32_t c0 = 0; c0 < span_max; c0 += CW * 16) {
            const uint32_t w0 = c0 >> 4;
            uint32_t cw[CW + 2];
            if (wide) {
#pragma unroll
                for (int i = 0; i <= CW; i += 2) {
                    uint2 t = make_uint2(0u, 0u);
                    if (w0 + i < nwords) t = __ldg(reinterpret_cast<const uint2*>(wp + w0 + i));  // nwords bounds the pair: the stride is even
                    cw[i] = t.x;
                    cw[i + 1] = (w0 + i + 1 < nwords) ? t.y : 0u;
                }
            } else {
#pragma unroll
                for (int i = 0; i <= CW; ++i) cw[i] = (w0 + i < nwords) ? __ldg(wp + w0 + i) : 0u;
            }
            uint32_t f[NF];
#pragma unroll
            for (int i = 0; i < NF; ++i) f[i] = 0u;
#pragma unroll
            for (int i = 0; i < CW; ++i) {
                if (c0 + i * 16 < span_max) {  // warp-uniform: skip words past every lane's last position
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        // 32 bits ENDING at the last base of the k-mer that starts at base j of word i; the older
                        // bases above bit 2K are removed by the multiply
                        const int n = 64 - 2 * (j + K);
                        const uint32_t v = (n >= 32) ? (cw[i] >> ((n - 32) & 31)) : __funnelshift_r(cw[i + 1], cw[i], n & 31);
                        const uint32_t p = v * (SCREEN_MUL << (32 - 2 * K));
                        uint32_t word;
                        if (V & 1) {
                            uint32_t addr;
                            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(__umulhi(p, n_fw)), "r"(SC.four), "r"(s_base));
                            asm("ld.shared.u32 %0, [%1];" : "=r"(word) : "r"(addr));
                        } else {
                            word = s_kf[__umulhi(p, n_fw)];
                        }
                        const uint32_t s2 = (V & 2) ? __umulhi(p, SC.two21) : (p >> 11);
                        const uint32_t t = __funnelshift_r(word, 0u, v) & __funnelshift_r(word, 0u, s2);
                        if (V & 4) {
                            // flags shifted in by a multiply-add (the multiplier pipe has room, the shift/logic pipe does not);
                            // the word is bit-reversed once at the end
                            asm("mad.lo.u32 %0, %0, %1, %2;" : "+r"(f[i >> 1]) : "r"(SC.two), "r"(t & 1u));
                        } else {
                            asm("{\n\t.reg .pred q;\n\t.reg .b32 t;\n\tand.b32 t, %1, 1;\n\tsetp.ne.u32 q, t, 0;\n\t@q or.b32 %0, %0, %2;\n\t}"
                                : "+r"(f[i >> 1])
                                : "r"(t), "r"(1u << ((i & 1) * 16 + j)));
                        }
                    }
                } else if (V & 4) {
                    f[i >> 1] <<= 16;  // a skipped word still occupies its sixteen flag positions
                }
            }
            if (V & 4) {
#pragma unroll
                for (int i = 0; i < NF; ++i) f[i] = __brev((CW & 1) && i == NF - 1 ? f[i] << 16 : f[i]);
            }
            // keep the flags of positions inside [seg_s, seg_e), count them, reserve queue space per warp
            uint32_t cnt = 0;
            {
                const uint32_t lo_cut = (c0 == 0) ? (seg_s - q0) : 0u;                          // < 16
                const uint32_t hi_cut = span > c0 ? min(span - c0, (uint32_t)(CW * 16)) : 0u;  // valid positions in this chunk
#pragma unroll
                for (int i = 0; i < NF; ++i) {
                    const uint32_t base = i * 32;
                    const uint32_t hi_n = hi_cut > base ? min(hi_cut - base, 32u) : 0u;
                    uint32_t m = hi_n >= 32u ? 0xffffffffu : ((1u << hi_n) - 1u);
                    if (i == 0) m &= ~((1u << lo_cut) - 1u);
                    f[i] &= m;
                    cnt += __popc(f[i]);
                }
            }
            const uint32_t total = __reduce_add_sync(FULL, cnt);
            if (total) {
                unsigned long long o = 0;
                if (lane == 0) o = atomicAdd(queue_count, (unsigned long long)total);  // in flight during the prefix scan
                uint32_t incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t t = __shfl_up_sync(FULL, incl, d);
                    if (lane >= d) incl += t;
                }
                o = __shfl_sync(FULL, o, 0);
                // a warp whose entries do not all fit writes none of them: the host sees the overflow in the counter and
                // redoes the batch with a larger queue, so one bounds test per warp is enough
                if (o + total <= queue_cap) {
                    unsigned long long* qp = queue + o + (incl - cnt);
                    uint32_t* kp = queue_kmer + o + (incl - cnt);
                    const uint32_t tag = (uint32_t)r, pos0 = q0 + c0;
#pragma unroll
                    for (int i = 0; i < NF; ++i) {
                        uint32_t m = f[i];
                        while (m) {
                            const uint32_t bit = __ffs(m) - 1;
                            m &= m - 1u;
                            *reinterpret_cast<uint2*>(qp++) = make_uint2(pos0 + i * 32 + bit, tag);  // read << 32 | position
                            // the k-mer travels with the entry, so the resolve kernel's index probe needs no access to the read
                            const bool up = bit >= 16u;
                            const uint32_t a = up ? cw[2 * i + 1] : cw[2 * i], b = up ? cw[2 * i + 2] : cw[2 * i + 1];
                            *kp++ = __funnelshift_l(b, a, 2u * (bit & 15u)) >> (32 - 2 * K);
                        }
                    }
                }
            }
        }
        tile = next_tile;
        next_tile = __shfl_sync(FULL, after_next, 0);
    }
}

// Resolve the flagged (read, position) pairs: persistent warps, no CTA barrier.  A warp takes tiles of RESOLVE_PER_LANE
// queue entries per lane (lane-strided, so the queue loads stay coalesced), computes the canonical hash of every queued
// k-mer and issues the index probes of all of them before it uses any result: RESOLVE_PER_LANE independent L2 chains per
// thread.  The probe is exact, so the Bloom filter's false positives (~80 % of the queue) end here.  The survivors are
// appended by ballot to a ring in the warp's own shared memory; whenever it holds 32 of them the warp runs the minimizer
// test restricted to those positions with every lane busy, and after its last tile it tests what is left.
//   W > 0: compile-time window (2W-2+K bases around the position fit three aligned words): the words are fetched once,
//          shifted so that every neighbour sits at a static offset, and all 2W-1 canonical hashes are computed branch-free;
//   W == 0: any window, neighbours fetched one by one with early exit.
constexpr int RESOLVE_WARPS = 8;
constexpr int RESOLVE_PER_LANE = 4;
constexpr uint32_t RESOLVE_TILE = 32 * RESOLVE_PER_LANE;
constexpr int RESOLVE_RING = 31 + RESOLVE_TILE;  // < 32 untested survivors + one tile's
template <int W, int K>
__global__ void __launch_bounds__(RESOLVE_WARPS * 32) resolve_kernel(DevReads R, DevTable T, uint32_t w_rt, uint32_t k_rt,
                                                                     const unsigned long long* __restrict__ queue,
                                                                     const uint32_t* __restrict__ queue_kmer,
                                                                     const unsigned long long* __restrict__ queue_count,
                                                                     unsigned long long queue_cap,
                                                                     unsigned long long* __restrict__ queue_need,
                                                                     unsigned long long* __restrict__ survivors,
                                                                     unsigned long long* __restrict__ out_a,
                                                                     unsigned long long* __restrict__ out_b,
                                                                     unsigned long long* __restrict__ out_count,
                                                                     unsigned long long cap) {
    static_assert(W == 0 || 2 * W - 2 + K <= 48, "window + k-mer must fit three aligned words");
    __shared__ unsigned long long s_q[RESOLVE_WARPS][RESOLVE_RING];
    __shared__ uint32_t s_rec[RESOLVE_WARPS][RESOLVE_RING];
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicMax(queue_need, *queue_count);  // sticky over the chunks of a batch: the host regrows and redoes
    if (*queue_count > queue_cap) return;  // overflow: the queue has unwritten slots and the batch is redone anyway
    const unsigned long long n = *queue_count;
    const uint32_t w = W ? (uint32_t)W : w_rt, k = W ? (uint32_t)K : k_rt;
    const uint32_t S = 32 - 2 * k;
    const uint32_t hm = (S == 0) ? 0xffffffffu : ~((1u << S) - 1u);
    const uint32_t smask = (1u << T.slot_bits) - 1u;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long* ring_q = s_q[wid];
    uint32_t* ring_rec = s_rec[wid];
    auto canon_of = [&](uint32_t v, uint32_t& strand) {  // v: 32 bits starting at the k-mer's first base
        const uint32_t F = v & hm;
        uint32_t y = __brev(~v & hm);
        y = ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
        const uint32_t hf = hash_left_aligned(F, S, hm), hr = hash_left_aligned(y << S, S, hm);
        strand = hf <= hr ? 1u : 0u;
        return min(hf, hr);
    };
    const unsigned long long n_tiles = (n + RESOLVE_TILE - 1) / RESOLVE_TILE;
    const unsigned long long n_warps = (unsigned long long)gridDim.x * RESOLVE_WARPS;
    uint32_t ring_n = 0;              // survivors in the ring (warp-uniform)
    unsigned long long n_surv = 0;    // survivors this warp found (warp-uniform)
    for (unsigned long long tile = (unsigned long long)blockIdx.x * RESOLVE_WARPS + wid;; tile += n_warps) {
        const bool more = tile < n_tiles;  // warp-uniform
        if (more) {
            unsigned long long q[RESOLVE_PER_LANE];
            uint32_t km[RESOLVE_PER_LANE], hv[RESOLVE_PER_LANE], slot[RESOLVE_PER_LANE], rec[RESOLVE_PER_LANE];
            uint32_t pending = 0;  // bit i: entry i still walks its probe chain
#pragma unroll
            for (int i = 0; i < RESOLVE_PER_LANE; ++i) {
                const unsigned long long e = tile * RESOLVE_TILE + i * 32 + lane;
                q[i] = 0;
                km[i] = 0;
                rec[i] = 0;
                if (e < n) {
                    q[i] = queue[e];
                    km[i] = queue_kmer[e];
                    pending |= 1u << i;
                }
            }
#pragma unroll
            for (int i = 0; i < RESOLVE_PER_LANE; ++i) {
                uint32_t strand;
                hv[i] = canon_of(km[i] << S, strand) >> S;  // the queued k-mer, left aligned
                slot[i] = table_slot(hv[i], T.slot_bits);
            }
            // one slot of every unfinished chain per round: the loads of a round are independent of each other
            while (pending) {
                uint2 ent[RESOLVE_PER_LANE];
#pragma unroll
                for (int i = 0; i < RESOLVE_PER_LANE; ++i) ent[i] = (pending >> i & 1u) ? __ldg(T.slots + slot[i]) : make_uint2(0u, 0u);
#pragma unroll
                for (int i = 0; i < RESOLVE_PER_LANE; ++i) {
                    if (!(pending >> i & 1u)) continue;
                    if (ent[i].y == 0u || ent[i].x == hv[i]) {
                        rec[i] = ent[i].y;  // rec_begin | rec_count << 24 (count >= 1), or 0: not indexed
                        pending &= ~(1u << i);
                    } else {
                        slot[i] = (slot[i] + 1) & smask;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < RESOLVE_PER_LANE; ++i) {
                const uint32_t bal = __ballot_sync(FULL, rec[i] != 0u);
                if (rec[i]) {
                    const uint32_t o = ring_n + __popc(bal & ((1u << lane) - 1u));
                    ring_q[o] = q[i];
                    ring_rec[o] = rec[i];
                }
                ring_n += __popc(bal);
                n_surv += __popc(bal);
            }
            __syncwarp();
        }
        // minimizer tests, 32 survivors at a time; after the last tile also the partial batch
        uint32_t done = 0;
        for (; done + 32 <= ring_n || (!more && done < ring_n); done += 32) {
            uint32_t emit_n = 0, rec_begin = 0, read_strand = 0, r = 0, pos = 0;
            if (done + lane < ring_n) {
                const unsigned long long q = ring_q[done + lane];
                const uint32_t rec = ring_rec[done + lane];
                r = (uint32_t)(q >> 32);
                pos = (uint32_t)q;
                uint32_t rec_n;
                rec_span(T.recs, rec, rec_begin, rec_n);
                const uint32_t len = __ldg(R.lens + r);
                const uint32_t nk = len - k + 1;
                const uint32_t* wp = R.words + (R.stride_words ? (unsigned long long)r * R.stride_words : __ldg(R.word_off + r));
                const uint32_t nwords = (len + 15) >> 4;
                uint32_t run = 1, dummy;
                if (W) {
                    // minimizer test: the neighbours with hash >= h on both sides must cover a window of w positions
                    const int start = (int)pos - (W - 1);  // may be negative near the read start: those words read as 0
                    const int sw = start >> 4;
                    const uint32_t sh = 2u * ((uint32_t)start & 15u);
                    uint32_t x[4], y[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) x[i] = (sw + i >= 0 && sw + i < (int)nwords) ? __ldg(wp + sw + i) : 0u;
#pragma unroll
                    for (int i = 0; i < 3; ++i) y[i] = __funnelshift_l(x[i + 1], x[i], sh);  // base `start + j` now sits at base j
                    y[3] = 0u;
                    constexpr int c0 = W - 1;
                    const uint32_t h = canon_of(__funnelshift_l(y[(c0 >> 4) + 1], y[c0 >> 4], 2 * (c0 & 15)), read_strand);
                    bool ok = true;
#pragma unroll
                    for (int d = 1; d < (W ? W : 1); ++d) {
                        const int c = W - 1 - d;
                        const uint32_t hn = canon_of(__funnelshift_l(y[(c >> 4) + 1], y[c >> 4], 2 * (c & 15)), dummy);
                        ok = ok && (uint32_t)d <= pos && hn >= h;
                        run += ok ? 1u : 0u;
                    }
                    ok = true;
#pragma unroll
                    for (int d = 1; d < (W ? W : 1); ++d) {
                        const int c = W - 1 + d;
                        const uint32_t hn = canon_of(__funnelshift_l(y[(c >> 4) + 1], y[c >> 4], 2 * (c & 15)), dummy);
                        ok = ok && pos + d < nk && hn >= h;
                        run += ok ? 1u : 0u;
                    }
                } else {
                    auto canon_at = [&](uint32_t x, uint32_t& strand) {  // fetch the two words of position x
                        const uint32_t wi = x >> 4;
                        const uint32_t a = __ldg(wp + wi), b = (wi + 1 < nwords) ? __ldg(wp + wi + 1) : 0u;
                        return canon_of(__funnelshift_l(b, a, 2u * (x & 15u)), strand);
                    };
                    const uint32_t h = canon_at(pos, read_strand);
                    for (uint32_t d = 1; d < w && d <= pos && run < w; ++d) {
                        if (canon_at(pos - d, dummy) < h) break;
                        ++run;
                    }
                    for (uint32_t d = 1; d < w && pos + d < nk && run < w; ++d) {
                        if (canon_at(pos + d, dummy) < h) break;
                        ++run;
                    }
                }
                if (run >= w) emit_n = rec_n;
                if (emit_n && R.hit_count) atomicAdd(R.hit_count + r, (int32_t)emit_n);
            }
            // one atomic per warp: a single hit counter takes ~1 atomic per clock
            uint32_t incl = emit_n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += t;
            }
            const uint32_t total = __shfl_sync(FULL, incl, 31);
            if (total) {
                unsigned long long ob = 0;
                if (lane == 0) ob = atomicAdd(out_count, (unsigned long long)total);
                ob = __shfl_sync(FULL, ob, 0) + (incl - emit_n);
                for (uint32_t j = 0; j < emit_n; ++j) {
                    const uint2 rc = __ldg(T.recs + rec_begin + j);
                    const uint32_t fwd = ((rc.y & 1u) == read_strand) ? 1u : 0u;
                    if (ob + j < cap) {
                        out_a[ob + j] = ((unsigned long long)(R.read_id_base + r) << 32) | ((unsigned long long)(rc.y >> 1) << 16) |
                                        ((unsigned long long)(fwd ^ 1u) << 15);
                        out_b[ob + j] = ((unsigned long long)pos << 32) | rc.x;
                    }
                }
            }
        }
        if (!more) break;
        // the < 32 untested survivors move to the front of the ring
        if (done) {
            const uint32_t left = ring_n - done;
            unsigned long long q = 0;
            uint32_t rec = 0;
            if ((uint32_t)lane < left) {
                q = ring_q[done + lane];
                rec = ring_rec[done + lane];
            }
            __syncwarp();
            if ((uint32_t)lane < left) {
                ring_q[lane] = q;
                ring_rec[lane] = rec;
            }
            __syncwarp();
            ring_n = left;
        }
    }
    if (lane == 0 && n_surv) atomicAdd(survivors, n_surv);
}

template <int K, int CW, int V>
static void launch_screen_v(const DevReads& R, const DevTable& T, uint32_t wk, unsigned long long* queue, uint32_t* queue_kmer,
                            unsigned long long* counters, uint64_t queue_cap, int sm_count, cudaStream_t st) {
    ensure_dyn_smem(screen_kernel<K, CW, V>, (size_t)SCREEN_MAX_FILTER_WORDS * 4);
    static const uint32_t prefetch = [] {
        const char* e = getenv("DRPRG_SCREEN_PREFETCH");  // L2 prefetch of the next tile: measured neutral (cold == warm L2 time), off
        return e ? (uint32_t)atoi(e) : 0u;
    }();
    const unsigned long long n_items = R.seg_read ? R.n_segs : R.n_reads;
    const unsigned long long n_ctas = (n_items + SCREEN_THREADS - 1) / SCREEN_THREADS;
    const unsigned grid = (unsigned)std::min<unsigned long long>(n_ctas, (unsigned long long)sm_count);  // one persistent CTA per SM
    screen_kernel<K, CW, V><<<grid, SCREEN_THREADS, (size_t)T.kfilter_words * 4, st>>>(R, T, wk, ScreenConsts{4u, 1u << 21, prefetch, 2u}, queue, queue_kmer, counters, queue_cap, counters + 1);
    ++g_launches;
}

#ifndef DRPRG_SCREEN_DEFAULT_VARIANT
#define DRPRG_SCREEN_DEFAULT_VARIANT 5
#endif
template <int K, int CW>
static void launch_screen_one(const DevReads& R, const DevTable& T, uint32_t wk, unsigned long long* queue, uint32_t* queue_kmer,
                              unsigned long long* counters, uint64_t queue_cap, int sm_count, cudaStream_t st) {
    static const int variant = [] {
        const char* e = getenv("DRPRG_SCREEN_VARIANT");
        return e ? atoi(e) & 7 : DRPRG_SCREEN_DEFAULT_VARIANT;
    }();
    switch (variant) {  // the default and the plain kernel (second implementation for the parity tests)
        case 0: return launch_screen_v<K, CW, 0>(R, T, wk, queue, queue_kmer, counters, queue_cap, sm_count, st);
        case 1: return launch_screen_v<K, CW, 1>(R, T, wk, queue, queue_kmer, counters, queue_cap, sm_count, st);
        default: return launch_screen_v<K, CW, 5>(R, T, wk, queue, queue_kmer, counters, queue_cap, sm_count, st);
    }
}

// counters = the CTR_QUEUE.. slots of the batch counters
template <int W, int K>
static void launch_resolve(const DevReads& R, const DevTable& T, uint32_t w, const unsigned long long* queue, const uint32_t* queue_kmer,
                           uint64_t queue_cap, unsigned long long* counters, unsigned long long* a, unsigned long long* b,
                           unsigned long long* cnt, uint64_t cap, int sm_count, uint32_t max_len, cudaStream_t st) {
    static const int per_sm = [] {
        int n = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, resolve_kernel<W, K>, RESOLVE_WARPS * 32, 0);
        return std::max(n, 1);
    }();
    // persistent warps at full occupancy; the queue length is only known on the device, but it cannot exceed the number of
    // k-mer positions, which caps the grid of a small batch
    const unsigned long long positions = (R.seg_read ? R.n_segs * R.seg_len : R.n_reads * max_len) + 1;
    const unsigned long long want = (positions + RESOLVE_TILE * RESOLVE_WARPS - 1) / (RESOLVE_TILE * RESOLVE_WARPS);
    const unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)per_sm * (unsigned)sm_count);
    resolve_kernel<W, K><<<grid, RESOLVE_WARPS * 32, 0, st>>>(R, T, w, K, queue, queue_kmer, counters, queue_cap,
                                                              counters + (CTR_QUEUE_NEED - CTR_QUEUE), counters + (CTR_SURVIVORS - CTR_QUEUE),
                                                              a, b, cnt, cap);
    ++g_launches;
}

// screen + resolve; counters = the CTR_QUEUE.. slots of the batch counters: {queue length, ticket, largest queue length
// wanted, ...} (only the first two are reset here)
template <int K>
static void launch_screened(const DevReads& R, const DevTable& T, uint32_t w, unsigned long long* a, unsigned long long* b,
                            unsigned long long* cnt, uint64_t cap, int sm_count, uint32_t max_len,
                            unsigned long long* queue, uint32_t* queue_kmer, uint64_t queue_cap, unsigned long long* counters,
                            cudaStream_t st) {
    cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), st);
    if (!R.seg_read && max_len >= (uint32_t)K && max_len - K + 1 <= 10 * 16) launch_screen_one<K, 10>(R, T, w + K, queue, queue_kmer, counters, queue_cap, sm_count, st);
    else launch_screen_one<K, 8>(R, T, w + K, queue, queue_kmer, counters, queue_cap, sm_count, st);
    if (w == 11) launch_resolve<11, K>(R, T, w, queue, queue_kmer, queue_cap, counters, a, b, cnt, cap, sm_count, max_len, st);
    else if (w == 14) launch_resolve<14, K>(R, T, w, queue, queue_kmer, queue_cap, counters, a, b, cnt, cap, sm_count, max_len, st);
    else launch_resolve<0, K>(R, T, w, queue, queue_kmer, queue_cap, counters, a, b, cnt, cap, sm_count, max_len, st);
}

static int grid_for(int sm_count, uint64_t n_reads) {
    // persistent-style grid: a multiple of the SM count, capped by the work available
    long long want = (long long)((n_reads + WARPS - 1) / WARPS);
    long long g = (long long)sm_count * 8;
    if (want < g) g = want;
    return (int)(g < 1 ? 1 : g);
}

void launch_sketch_lookup(const DevReads& R, const DevTable& T, uint32_t w, uint32_t k, unsigned long long* d_hi,
                          unsigned long long* d_lo, unsigned long long* d_hit_count, uint64_t hit_cap, int sm_count,
                          uint32_t max_len, cudaStream_t st, unsigned long long* d_queue, uint64_t queue_cap,
                          unsigned long long* d_screen_counters, uint32_t* d_queue_kmer) {
    if (R.n_reads == 0) return;
    static const bool screen_on = [] {
        const char* e = getenv("DRPRG_SCREEN");  // DRPRG_SCREEN=0 sketches every read (A/B measurements, parity tests)
        return !e || atoi(e) != 0;
    }();
    if (screen_on && d_queue && d_queue_kmer && T.kfilter && (max_len <= SHORT_READ_MAX || R.seg_read) && k == 15)
        return launch_screened<15>(R, T, w, d_hi, d_lo, d_hit_count, hit_cap, sm_count, max_len, d_queue, d_queue_kmer, queue_cap, d_screen_counters, st);
    if ((max_len <= SHORT_READ_MAX || R.seg_read) && launch_short<true>(R, T, w, k, d_hi, d_lo, d_hit_count, hit_cap, sm_count, st)) return;
    sketch_kernel<true><<<grid_for(sm_count, R.n_reads), WARPS * 32, 0, st>>>(R, T, w, k, d_hi, d_lo, d_hit_count, hit_cap);
    ++g_launches;
}

// ---- issue-rate yardstick for the roofline of the k-mer screen ------------------------------------------------------
// The screen kernel is bound by instruction issue (multiply-add, shift and logic on 32-bit integers), not by HBM.  This
// kernel issues the same instruction classes from eight independent dependency chains per thread with nothing else in
// the loop, which is what the SM can issue at best for that mix; bench.py reports the screen's warp-instructions per
// second as a fraction of it next to the HBM fraction.
constexpr int ISSUE_OPS_PER_ITER = 32;  // 16 mad.lo + 8 shf + 8 lop3 per loop iteration
__global__ void __launch_bounds__(1024, 1) issue_peak_kernel(uint32_t iters, uint32_t a, uint32_t b, uint32_t* __restrict__ out) {
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = threadIdx.x * 8u + i + b;
#pragma unroll 1
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(a), "r"(b));
            asm volatile("shf.r.wrap.b32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(b), "r"(a));
            asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(b), "r"(a));
            asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(a), "r"(b));
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r ^= x[i];
    if (r == 0x12345678u) out[0] = r;  // never true in practice: keeps the chains alive
}
double measure_issue_peak(int sm_count, cudaStream_t st) {
    uint32_t* d = nullptr;
    if (cudaMalloc(&d, 4) != cudaSuccess) return 0.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const uint32_t iters = 4096;
    issue_peak_kernel<<<sm_count, 1024, 0, st>>>(64, 3u, 5u, d);  // warm-up
    cudaEventRecord(e0, st);
    issue_peak_kernel<<<sm_count, 1024, 0, st>>>(iters, 3u, 5u, d);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    g_launches += 2;
    if (ms <= 0) return 0.0;
    return (double)sm_count * 32.0 /* warps */ * (double)iters * ISSUE_OPS_PER_ITER / (ms * 1e-3);
}

void launch_sketch_only(const DevReads& R, uint32_t w, uint32_t k, unsigned long long* d_key, unsigned long long* d_val,
                        unsigned long long* d_count, uint64_t cap, int sm_count, uint32_t max_len, cudaStream_t st) {
    if (R.n_reads == 0) return;
    DevTable T{};
    if ((max_len <= SHORT_READ_MAX || R.seg_read) && launch_short<false>(R, T, w, k, d_key, d_val, d_count, cap, sm_count, st)) return;
    sketch_kernel<false><<<grid_for(sm_count, R.n_reads), WARPS * 32, 0, st>>>(R, T, w, k, d_key, d_val, d_count, cap);
    ++g_launches;
}

}  // namespace drprg
