// Hand-written sm_100a kernels for the second half of `pandora discover` (drprg src/predict.rs:247-256 -> src/lib.rs:513-578):
// the local assembly of the reads over each candidate region into de-novo alleles.  discover.cpp finds the regions and
// their reads from the map pass; the semantics restated here are tests/denovo_oracle.py's (assemble_region), which pins
// every choice that upstream's GATB-based assembler leaves unpinned.
//   retain_gather_kernel  at the end of a mapped batch (hit retention on): one warp per active read appends the kept hits
//                         of every read that has one to the GPU's retained-hit store (slice order, one cursor atomic per
//                         read) and copies the read's 2-bit words into one buffer, so the bases outlive the batch
//   region_reads_kernel   one warp per retained read: its hits inside each padded candidate region of their locus give
//                         the read's span and strand over the region (discover.cpp's host half finds the regions)
//   assemble_kernel       one CTA per region.  Counting: the warps take the pileup reads in turn, their lanes stride over
//                         the k-mer positions, read each 22-bit k-mer with a funnel shift of two words (reverse complement
//                         for reads on the reverse strand) and count it in an open-addressed table (atomicCAS on the key,
//                         atomicAdd on the count) in shared memory, or for a pileup too large for it in a per-region
//                         table in global scratch (second instantiation).  Walk: warp 0 picks the first solid anchor pair
//                         and walks depth first from an explicit stack in shared memory; the four successor probes of a
//                         step go to lanes 0-3 and come back as one ballot.  It stops at max_paths + 1 complete walks.
#include <algorithm>

#include "kernels_common.cuh"

namespace drprg {

namespace {

constexpr uint32_t KEY_EMPTY = 0xffffffffu;
constexpr uint32_t KMASK = (1u << (2 * DISCOVER_K)) - 1u;

__global__ void __launch_bounds__(256) retain_gather_kernel(DevReads R, const uint32_t* __restrict__ act_read,
                                                            const uint32_t* __restrict__ act_base,
                                                            const uint32_t* __restrict__ act_count,
                                                            const unsigned long long* __restrict__ gkey,
                                                            const uint8_t* __restrict__ gkept, uint32_t n_active,
                                                            RetainStore S, uint64_t row_base, uint4* __restrict__ table,
                                                            uint32_t* __restrict__ out_words, uint64_t word_cap,
                                                            unsigned long long* __restrict__ cursor) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t a = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; a < n_active; a += warps) {
        const uint32_t b = act_base[a], n = act_count[a];
        uint32_t n_kept = 0;
        for (uint32_t j0 = 0; j0 < n; j0 += 32) n_kept += __popc(__ballot_sync(FULL, j0 + lane < n && gkept[b + j0 + lane]));
        if (n_kept == 0) continue;
        const uint32_t r = act_read[a], read = R.read_id_base + r;
        const uint32_t len = R.lens[r];
        const uint32_t nw = (len + 15) / 16;
        // lanes 0-2 take the read's three cursor slots side by side: its words, its hits, its row
        unsigned long long got = 0;
        if (lane < RT_COUNT) got = atomicAdd(cursor + lane, lane == RT_WORDS ? (unsigned long long)nw : lane == RT_HITS ? n_kept : 1ull);
        const unsigned long long woff = __shfl_sync(FULL, got, RT_WORDS), hoff = __shfl_sync(FULL, got, RT_HITS),
                                 row = __shfl_sync(FULL, got, RT_ROWS);
        const bool words_fit = woff + nw <= word_cap;
        if (lane == 0) table[row - row_base] = make_uint4(words_fit ? (uint32_t)woff : 0xffffffffu, len, read, 0u);
        if (lane == 0 && row < S.row_cap) S.rows[row] = make_uint2((uint32_t)hoff, n_kept);
        if (hoff + n_kept <= S.hit_cap) {  // slice order: a kept hit's place is the kept hits before it
            uint32_t before = 0;
            for (uint32_t j0 = 0; j0 < n; j0 += 32) {
                const bool kept = j0 + lane < n && gkept[b + j0 + lane];
                const uint32_t m = __ballot_sync(FULL, kept);
                if (kept) {
                    const uint64_t q = hoff + before + __popc(m & ((1u << lane) - 1u));
                    S.hit_read[q] = read;
                    S.hit_key[q] = gkey[b + j0 + lane];
                }
                before += __popc(m);
            }
        }
        if (!words_fit) continue;
        const uint32_t* src = R.stride_words ? R.words + (uint64_t)r * R.stride_words : R.words + R.word_off[r];
        for (uint32_t w = lane; w < nw; w += 32) out_words[woff + w] = src[w];
    }
}

__global__ void __launch_bounds__(256) region_reads_kernel(RetainStore S, uint32_t n_rows, const uint32_t* __restrict__ knode_base,
                                                           const uint32_t* __restrict__ cons_start,
                                                           const uint32_t* __restrict__ locus_region_off, uint32_t n_loci,
                                                           const uint2* __restrict__ pad, uint32_t k, uint32_t min_hits,
                                                           RegionRead* __restrict__ out, uint64_t out_cap,
                                                           unsigned long long* __restrict__ cursor) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n_rows; row += warps) {
        const uint2 rw = S.rows[row];
        const unsigned long long* key = S.hit_key + rw.x;
        const uint32_t n = rw.y, read = S.hit_read[rw.x];
        for (uint32_t i = 0; i < n;) {
            // a (read, locus) group: the hits are sorted by locus within a read
            const uint32_t l = (uint32_t)(key[i] >> 48);
            uint32_t j = i;
            for (;; j += 32) {
                const uint32_t m = __ballot_sync(FULL, j + lane >= n || (uint32_t)(key[j + lane] >> 48) != l);
                if (m) {
                    j += __ffs(m) - 1;
                    break;
                }
            }
            const uint32_t r0 = l < n_loci ? locus_region_off[l] : 0u, r1 = l < n_loci ? locus_region_off[l + 1] : 0u;
            for (uint32_t rg = r0; rg < r1; ++rg) {
                const uint2 P = pad[rg];
                uint32_t cnt = 0, lo = 0xffffffffu, hi = 0, fwd = 2;
                for (uint32_t c = i; c < j; c += 32) {
                    bool in = false;
                    uint32_t st = 0, f = 0;
                    if (c + lane < j) {
                        const unsigned long long x = key[c + lane];
                        const uint32_t cs = cons_start[knode_base[l] + ((uint32_t)x & ((1u << GKEY_KNODE_BITS) - 1u))];
                        in = cs != 0xffffffffu && cs >= P.x && cs + k <= P.y;
                        st = (uint32_t)(x >> GKEY_KNODE_BITS) & ((1u << GKEY_START_BITS) - 1u);
                        f = (uint32_t)((x >> 47) & 1ull) ^ 1u;
                    }
                    const uint32_t m = __ballot_sync(FULL, in);
                    if (m && fwd == 2) fwd = __shfl_sync(FULL, f, __ffs(m) - 1);
                    cnt += __popc(m);
                    if (in) {
                        lo = min(lo, st);
                        hi = max(hi, st + k);
                    }
                }
                if (cnt < min_hits) continue;
                for (int o = 16; o; o >>= 1) {
                    lo = min(lo, __shfl_xor_sync(FULL, lo, o));
                    hi = max(hi, __shfl_xor_sync(FULL, hi, o));
                }
                if (lane == 0) {
                    const unsigned long long q = atomicAdd(cursor, 1ull);
                    if (q < out_cap) out[q] = RegionRead{rg, read, lo, hi, fwd};
                }
            }
            i = j;
        }
    }
}

__device__ __forceinline__ uint32_t kmer_hash(uint32_t x) { return (x * 0x9E3779B1u) ^ (x >> 15); }

// forward k-mer of the read whose words start at w, at base t (first base in the top bits of a word)
__device__ __forceinline__ uint32_t read_kmer(const uint32_t* __restrict__ w, uint32_t t) {
    const uint32_t q = t >> 4, sh = 2 * (t & 15);
    const uint32_t hi = w[q];
    const uint32_t lo = (t & 15) + DISCOVER_K > 16 ? w[q + 1] : 0u;
    return __funnelshift_l(lo, hi, sh) >> (32 - 2 * DISCOVER_K);
}

__device__ __forceinline__ uint32_t revcomp_kmer(uint32_t x) {
    const uint32_t r = __brev(~x) >> (32 - 2 * DISCOVER_K);  // complemented, bits reversed: 2-bit codes come back swapped
    return ((r & 0x55555555u) << 1) | ((r >> 1) & 0x55555555u);
}

__device__ __forceinline__ void table_add(uint32_t* keys, uint32_t* counts, uint32_t mask, uint32_t x) {
    uint32_t h = kmer_hash(x) & mask;
    for (;;) {  // at most half the slots are ever taken: the probe ends
        uint32_t k = ((volatile uint32_t*)keys)[h];
        if (k == KEY_EMPTY) {
            k = atomicCAS(keys + h, KEY_EMPTY, x);
            if (k == KEY_EMPTY) k = x;
        }
        if (k == x) {
            atomicAdd(counts + h, 1u);
            return;
        }
        h = (h + 1) & mask;
    }
}

__device__ __forceinline__ uint32_t table_count(const uint32_t* keys, const uint32_t* counts, uint32_t mask, uint32_t x) {
    for (uint32_t h = kmer_hash(x) & mask;; h = (h + 1) & mask) {
        const uint32_t k = keys[h];
        if (k == x) return counts[h];
        if (k == KEY_EMPTY) return 0;
    }
}

template <bool GLOBAL_TABLE>
__global__ void __launch_bounds__(128) assemble_kernel(const AsmRegion* __restrict__ regions, const uint32_t* __restrict__ list,
                                                       const uint4* __restrict__ entries, const uint32_t* __restrict__ words,
                                                       uint32_t smem_slots, uint32_t* g_keys, uint32_t* g_counts,
                                                       uint32_t max_walk, AsmParams P, AsmResult* __restrict__ res,
                                                       uint32_t* __restrict__ walk_len, char* __restrict__ out_bases,
                                                       unsigned long long* __restrict__ cursor) {
    extern __shared__ __align__(16) uint32_t sm[];
    const uint32_t r = list[blockIdx.x];
    const AsmRegion& R = regions[r];
    const uint32_t slots = R.slots, mask = slots - 1;
    uint32_t* keys = GLOBAL_TABLE ? g_keys + R.table_off : sm;
    uint32_t* counts = GLOBAL_TABLE ? g_counts + R.table_off : sm + smem_slots;
    uint32_t* kst = GLOBAL_TABLE ? sm : sm + 2 * smem_slots;  // walk stack: k-mer per depth
    uint8_t* succ = reinterpret_cast<uint8_t*>(kst + max_walk);  // successors still to try per depth
    uint8_t* bases = succ + max_walk;                              // the walk's bases
    uint8_t* store = bases + max_walk;                             // complete walks, max_walk bytes each
    uint32_t* store_len = reinterpret_cast<uint32_t*>(store + (size_t)P.max_paths * max_walk);

    for (uint32_t i = threadIdx.x; i < slots; i += blockDim.x) {
        keys[i] = KEY_EMPTY;
        counts[i] = 0;
    }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    for (uint32_t e = warp; e < R.n_entries; e += n_warps) {
        const uint4 E = entries[R.entry_off + e];  // word offset, start, end, fwd
        const uint32_t* w = words + E.x;
        const uint32_t n_pos = E.z - E.y >= DISCOVER_K ? E.z - E.y - DISCOVER_K + 1 : 0;
        for (uint32_t p = lane; p < n_pos; p += 32) {
            // pileup sequences are in consensus orientation: position p of a reverse read is the reverse complement of
            // the forward k-mer that ends p bases before the span's end
            const uint32_t x = E.w ? read_kmer(w, E.y + p) : revcomp_kmer(read_kmer(w, E.z - DISCOVER_K - p));
            table_add(keys, counts, mask, x);
        }
    }
    __syncthreads();
    if (warp != 0) return;

    AsmResult out{ASM_NO_ANCHOR, 0, 0, 0, 0};
    // the first (i, j), i outer, with both anchors solid: the first solid start and the first solid end
    const bool s_ok = lane < R.n_start && table_count(keys, counts, mask, R.start_kmer[lane < KMER_ATTEMPTS ? lane : 0]) >= P.min_dp;
    const bool e_ok = lane < R.n_end && table_count(keys, counts, mask, R.end_kmer[lane < KMER_ATTEMPTS ? lane : 0]) >= P.min_dp;
    const uint32_t sm_ok = __ballot_sync(FULL, s_ok), em_ok = __ballot_sync(FULL, e_ok);
    if (sm_ok && em_ok) {
        const uint32_t ai = __ffs(sm_ok) - 1, aj = __ffs(em_ok) - 1;
        const uint32_t start = R.start_kmer[ai], end = R.end_kmer[aj];
        const uint32_t max_len = R.span - ai - aj + P.max_insertion;
        if (lane < DISCOVER_K) bases[lane] = (start >> (2 * (DISCOVER_K - 1 - lane))) & 3u;
        uint32_t n_walks = 0;
        // entering the node of depth d (spelled length K + d): a walk is complete where it first reaches the end anchor;
        // otherwise its solid successors, A C G T in bit order, as long as one more base keeps it within max_len
        auto enter = [&](uint32_t x, uint32_t d) -> uint32_t {
            const uint32_t L = DISCOVER_K + d;
            if (x == end) {
                if (n_walks < P.max_paths) {
                    __syncwarp();
                    for (uint32_t i = lane; i < L; i += 32) store[(size_t)n_walks * max_walk + i] = bases[i];
                    if (lane == 0) store_len[n_walks] = L;
                }
                ++n_walks;
                return 0u;
            }
            if (L + 1 > max_len) return 0u;
            const bool solid = lane < 4 && table_count(keys, counts, mask, ((x << 2) | lane) & KMASK) >= P.min_dp;
            return __ballot_sync(FULL, solid);
        };
        uint32_t d = 0, cur = start;
        uint32_t m = enter(cur, 0);
        while (n_walks <= P.max_paths) {
            if (m == 0) {  // backtrack
                if (d == 0) break;
                --d;
                __syncwarp();
                cur = kst[d];
                m = succ[d];
                continue;
            }
            const uint32_t b = __ffs(m) - 1;
            __syncwarp();
            if (lane == 0) {
                kst[d] = cur;
                succ[d] = (uint8_t)(m & (m - 1));
                bases[DISCOVER_K + d] = (uint8_t)b;
            }
            __syncwarp();
            cur = ((cur << 2) | b) & KMASK;
            ++d;
            m = enter(cur, d);
        }
        out.anchor_i = ai;
        out.anchor_j = aj;
        out.n_walks = n_walks;
        out.status = n_walks > P.max_paths ? ASM_TOO_MANY_PATHS : n_walks == 0 ? ASM_NO_PATH : ASM_ASSEMBLED;
        if (out.status == ASM_ASSEMBLED) {
            __syncwarp();
            uint32_t total = 0;
            for (uint32_t i = 0; i < n_walks; ++i) total += store_len[i];
            unsigned long long off = 0;
            if (lane == 0) off = atomicAdd(cursor, (unsigned long long)total);
            off = __shfl_sync(FULL, off, 0);
            out.byte_off = off;
            for (uint32_t i = 0; i < n_walks; ++i) {
                const uint32_t L = store_len[i];
                for (uint32_t q = lane; q < L; q += 32) out_bases[off + q] = "ACGT"[store[(size_t)i * max_walk + q]];
                if (lane == 0) walk_len[(size_t)r * P.max_paths + i] = L;
                off += L;
            }
        }
    }
    if (lane == 0) res[r] = out;
}

}  // namespace

void launch_retain_gather(const DevReads& R, const uint32_t* act_read, const uint32_t* act_base, const uint32_t* act_count,
                          const unsigned long long* gkey, const uint8_t* gkept, uint32_t n_active, RetainStore S,
                          uint64_t row_base, uint4* table, uint32_t* out_words, uint64_t word_cap, unsigned long long* d_cursor,
                          cudaStream_t st) {
    if (!n_active) return;
    const uint32_t blocks = (uint32_t)std::min<uint64_t>(4096, ((uint64_t)n_active + 7) / 8);
    retain_gather_kernel<<<blocks, 256, 0, st>>>(R, act_read, act_base, act_count, gkey, gkept, n_active, S, row_base, table,
                                                 out_words, word_cap, d_cursor);
    ++g_launches;
}

void launch_region_reads(RetainStore S, uint32_t n_rows, const uint32_t* knode_base, const uint32_t* cons_start,
                         const uint32_t* locus_region_off, uint32_t n_loci, const uint2* pad, uint32_t k, uint32_t min_hits,
                         RegionRead* out, uint64_t out_cap, unsigned long long* d_cursor, cudaStream_t st) {
    if (!n_rows) return;
    const uint32_t blocks = (uint32_t)std::min<uint64_t>(4096, ((uint64_t)n_rows + 7) / 8);
    region_reads_kernel<<<blocks, 256, 0, st>>>(S, n_rows, knode_base, cons_start, locus_region_off, n_loci, pad, k, min_hits,
                                                out, out_cap, d_cursor);
    ++g_launches;
}

static size_t walk_smem_bytes(uint32_t max_walk, uint32_t max_paths) {
    return (size_t)max_walk * (4 + 1 + 1) + (size_t)max_paths * max_walk + 4 * (size_t)max_paths + 16;
}

void launch_assemble(const AsmRegion* regions, const uint32_t* list, uint32_t n_list, const uint4* entries, const uint32_t* words,
                     uint32_t smem_slots, uint32_t* g_keys, uint32_t* g_counts, uint32_t max_walk, AsmParams P,
                     AsmResult* res, uint32_t* walk_len, char* out_bases, unsigned long long* d_cursor, cudaStream_t st) {
    if (!n_list) return;
    max_walk = (max_walk + 3) & ~3u;  // keeps the byte arrays behind the k-mer stack 4-byte aligned
    if (g_keys) {
        const size_t smem = walk_smem_bytes(max_walk, P.max_paths);
        ensure_dyn_smem(assemble_kernel<true>, smem);
        assemble_kernel<true><<<n_list, 128, smem, st>>>(regions, list, entries, words, 0, g_keys, g_counts, max_walk, P, res,
                                                         walk_len, out_bases, d_cursor);
    } else {
        const size_t smem = 8 * (size_t)smem_slots + walk_smem_bytes(max_walk, P.max_paths);
        ensure_dyn_smem(assemble_kernel<false>, smem);
        assemble_kernel<false><<<n_list, 128, smem, st>>>(regions, list, entries, words, smem_slots, nullptr, nullptr, max_walk,
                                                          P, res, walk_len, out_bases, d_cursor);
    }
    ++g_launches;
}

}  // namespace drprg
