// Device-side interface of the map hot path (SURVEY.md §8a rows a2-a5, a7, a8).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace drprg {

constexpr int W_MAX = 32;    // largest minimizer window supported on the device
constexpr int K_MAX = 16;    // 2k <= 32: k-mers and hashes live in one 32-bit register
constexpr int CHUNK = 192;   // k-mer positions a warp resolves per pass (a 150 bp read is one pass)
constexpr uint32_t SHORT_READ_MAX = 640;  // batches whose reads are all this short take the thread-per-read kernel
constexpr int LV_MAX = 12;   // binary-lifting levels of the windowed ML-path score (window <= 4095)

// packed reads resident in HBM
struct DevReads {
    const uint32_t* words;     // 2-bit bases, 16 per word, first base in the top bits
    const uint64_t* word_off;  // n+1 word offsets, or nullptr when stride_words > 0
    uint32_t stride_words;
    const uint32_t* lens;      // bases per read; 0 = dropped (non-ACGT)
    uint64_t n_reads;
    uint32_t read_id_base;
    // optional segment table for long reads (thread-per-segment sketching): segment i covers k-mer positions
    // [seg_start[i], seg_start[i] + seg_len) of read seg_read[i]
    const uint32_t* seg_read = nullptr;
    const uint32_t* seg_start = nullptr;
    uint64_t n_segs = 0;
    uint32_t seg_len = 0;
    // optional per-read hit counters (index = read within this DevReads): the lookup kernels add the hits they emit, which
    // is what groups the hits by read afterwards (cluster.cu)
    int32_t* hit_count = nullptr;
};

// minimizer index resident in HBM (small: lives in L2)
struct DevTable {
    const uint2* slots;      // {hash, rec_begin | rec_count << 24}; y == 0 => empty
    uint32_t slot_bits;      // table has 1 << slot_bits slots
    const uint2* recs;       // {knode rank within locus, prg << 1 | strand}, grouped by hash
    const uint32_t* filter;  // blocked 2-bit Bloom pre-filter, 1 << filter_bits words
    uint32_t filter_bits;
    // k-mer screen (k = 15): every indexed minimizer k-mer in both orientations.  A read can only produce a hit if
    // one of its forward k-mers is in this set, which is tested WITHOUT hashing (hash64 is a bijection).
    const uint32_t* kfilter = nullptr;  // blocked 2-bit Bloom over those 15-mers, kfilter_words words (multiple of 4)
    uint32_t kfilter_words = 0;
    // the same over both 14-mers of each of them, copied to shared memory: a read's indexed 15-mer at p contains the 14-mer
    // at the even one of p, p + 1, so testing the 14-mers at even positions finds every candidate
    const uint32_t* kfilter14 = nullptr;
    uint32_t kfilter14_words = 0;
};

struct Hit128 {  // sort key: (hi, lo) ascending == pandora MinimizerHit order
    unsigned long long hi;  // read_id << 32 | prg << 16 | (!forward) << 15
    unsigned long long lo;  // read_start << 32 | knode rank
};

struct ModelParams {  // S6 output, computed on the host
    int bin;
    double nb_p, nb_r;
    double bin_p;          // 1 / exp(e_rate * k)
    uint32_t exp_depth;    // E (integer)
    double thresh;
    uint32_t window;       // max_num_kmers_to_average
    uint32_t min_kmer_covg;
    double gt_err, gt_conf;
    float minor_af;        // drprg's --maf for the minor-allele statistic (src/minor.rs:19-33): 1.0, or 0.1 with --illumina
};

uint64_t launch_count();

// S1+S2: sketch every read and probe the index; hits appended (unordered) through *hit_count
// With a screen workspace (d_queue + d_queue_kmer: queue_cap entries each, d_screen_counters: the batch counters from CTR_QUEUE on,
// i.e. {queue length, ticket, largest queue length wanted, ..., probe survivors at CTR_SURVIVORS}) and a screenable index (k = 15),
// a k-mer screen queues the positions whose k-mer may be indexed and only those are hashed, probed and tested for minimizer
// status (identical hits).  The queue overflowed when d_screen_counters[2] > queue_cap (the caller zeroes the counters before a
// batch and redoes the batch with a larger queue).
void launch_sketch_lookup(const DevReads& R, const DevTable& T, uint32_t w, uint32_t k, unsigned long long* d_hi,
                          unsigned long long* d_lo, unsigned long long* d_hit_count, uint64_t hit_cap, int sm_count,
                          uint32_t max_len, cudaStream_t st, unsigned long long* d_queue = nullptr, uint64_t queue_cap = 0,
                          unsigned long long* d_screen_counters = nullptr, uint32_t* d_queue_kmer = nullptr);
// host mirror of the screen's filter addressing (used when the index is uploaded)
void screen_filter_insert(uint32_t* filter, uint32_t n_words, uint32_t kmer, uint32_t k);
constexpr uint32_t SCREEN_MAX_FILTER_WORDS = 54 * 1024;  // 216 KB of shared memory
// warp-instructions per second the GPU issues for a pure 32-bit integer multiply-add / shift / logic mix (the screen
// kernel's instruction classes): the issue-rate ceiling bench.py reports next to the HBM roofline
double measure_issue_peak(int sm_count, cudaStream_t st);
// S1 only (parity hook): emits key = read << 32 | start, val = hash << 1 | strand
void launch_sketch_only(const DevReads& R, uint32_t w, uint32_t k, unsigned long long* d_key, unsigned long long* d_val,
                        unsigned long long* d_count, uint64_t cap, int sm_count, uint32_t max_len, cudaStream_t st);
// ---- S3-S5: hits grouped by read, per-read sort + clustering, coverage by sorted-key reduction (cluster.cu) ------
// device counters of one batch (unsigned long long each)
enum : int {
    CTR_HITS = 0,        // hits appended by the lookup kernels
    CTR_KEPT = 1,        // kept hits
    CTR_QUEUE = 2,       // k-mer screen: queue length of the current chunk
    CTR_TICKET = 3,      // k-mer screen: tile ticket
    CTR_QUEUE_NEED = 4,  // largest queue length any chunk wanted
    CTR_ACTIVE = 5,      // reads with at least one hit
    CTR_CURSOR = 6,      // grouped-hit slices handed out
    CTR_BIG = 7,         // active reads with more than CLUSTER_WARP_MAX hits
    CTR_LKOVF = 8,       // locus keys beyond two kept clusters per read
    CTR_SURVIVORS = 9,   // k-mer screen: queue entries whose k-mer is in the index (summed over the chunks)
    CTR_COUNT = 16
};
constexpr uint32_t CLUSTER_WARP_MAX = 64;  // hits of a read one warp sorts in registers; longer reads get a CTA
// grouped-hit key: prg 16 | reverse 1 | read_start 25 | k-mer node rank 22 (limits checked at index load / upload)
constexpr int GKEY_KNODE_BITS = 22, GKEY_START_BITS = 25;
constexpr uint32_t COV_KEY_NONE = 0xffffffffu;  // "no coverage key in this slot"
struct PostCaps {
    unsigned long long hit_cap, queue_cap;
};
struct PostBuffers {
    const unsigned long long *hi, *lo;  // unordered hits from the lookup kernels
    unsigned long long* ctr;            // CTR_COUNT counters
    int32_t* read_count;                // per read of the batch: filled by the lookup kernels, all zero again after the scatter
    uint32_t* read_base;                // per read
    uint32_t *act_read, *act_base, *act_count;  // active reads (hit_cap entries)
    uint32_t* act_lk;                   // 2 per active read: locus keys of its first two kept clusters
    uint32_t* lk_ovf;                   // locus keys of further kept clusters (hit_cap entries)
    uint32_t* big_list;                 // indices into the active list (hit_cap / 64 + 16 entries)
    unsigned long long* gkey;           // grouped hits (hit_cap), sorted within each read's slice after the cluster kernels
    uint8_t* gkept;                     // kept flag per grouped hit
    uint32_t* cov_keys;                 // per grouped hit: its coverage key, COV_KEY_NONE when the hit is not kept
    uint32_t* scratch[10];              // hit_cap each: long-read clustering
    int32_t* partials;                  // n_partials x n_accum: per-stretch coverage partials (cov_count_kernel)
    uint32_t n_partials;
};
uint32_t cov_max_stretches(uint64_t hit_cap, int sm_count);  // rows of PostBuffers::partials a hit capacity needs
// everything after the lookup kernels for one batch; results are added to d_accum_dst: the sample's accumulator
// [2*total_knodes coverage | n_loci locus reads | 4 scalars] on this GPU, or (remote_dst != 0) the root GPU's accumulator
// mapped over NVLink, updated with red.global.add
// min_thresh = smallest entry of d_thresh_per_prg (a read with no more hits than that keeps nothing)
void launch_postprocess(const PostBuffers& P, PostCaps C, uint32_t read_id_base, uint64_t n_reads, uint32_t max_diff,
                        uint32_t min_thresh, const uint32_t* d_thresh_per_prg, const uint32_t* d_knode_base, uint32_t total_knodes, uint32_t n_loci,
                        int32_t* d_accum_dst, int remote_dst, int sm_count, cudaStream_t st, cudaEvent_t ev_grouped,
                        cudaEvent_t ev_clustered);
// cross-GPU signalling of a read-sharded run: flags behind the root GPU's accumulator (system-scope acquire / release)
void launch_flag_wait(const uint32_t* flag, uint32_t want, cudaStream_t st);      // spins until *flag >= want
void launch_flag_publish(uint32_t* flag, uint32_t value, cudaStream_t st);
void launch_shard_done(int32_t* root_tail, const int32_t scalars[4], uint32_t* arrivals, cudaStream_t st);
void launch_add_scalars(int32_t* tail, const int32_t scalars[4], cudaStream_t st);
// S7: per-node log-probabilities then one warp per locus for the ML-path DP
void launch_node_prob(const int32_t* d_cov, uint32_t total_knodes, const uint8_t* d_is_terminal, ModelParams P,
                      double* d_prob, cudaStream_t st);
// returns true when the results are streamed into the host-mapped h_path / h_path_len with per-locus h_done flags
// (level-parallel kernel); otherwise they are in d_path / d_path_len when the stream has finished
bool launch_mlpath(uint32_t n_loci, const uint32_t* d_knode_base, const uint32_t* d_edge_off, const uint32_t* d_edges,
                   const double* d_prob, const int32_t* d_locus_reads, ModelParams P, double* d_M, uint32_t* d_len,
                   uint32_t* d_up, uint32_t total_knodes, uint32_t* d_path, uint32_t* d_path_len,
                   uint32_t max_locus_knodes, uint32_t max_locus_edges, const uint8_t* d_needs_mean,
                   cudaStream_t st, const uint32_t* d_locus_level_off = nullptr,
                   const uint32_t* d_level_start = nullptr, const uint32_t* d_level_nodes = nullptr,
                   const uint32_t* d_level_singles = nullptr, uint32_t* h_path = nullptr, uint32_t* h_path_len = nullptr,
                   uint32_t* h_done = nullptr, const double* d_thresh = nullptr);
// the probability threshold from the 200-bin histogram, on the device (d_thresh_f64 feeds launch_mlpath)
void launch_prob_thresh(const uint32_t* d_hist200, bool any_present, int fallback, double* d_thresh_f64, int* d_thresh_i32,
                        cudaStream_t st);
void launch_cov_hist(const int32_t* d_cov, uint32_t total, const uint8_t* d_is_terminal, const uint32_t* d_knode_locus,
                     const int32_t* d_locus_reads, uint32_t* d_hist1000, cudaStream_t st);
void launch_prob_hist(const double* d_prob, uint32_t total, const uint8_t* d_is_terminal, const uint32_t* d_knode_locus,
                      const int32_t* d_locus_reads, uint32_t* d_hist, cudaStream_t st);
// S8: per-allele coverage statistics, then per-record likelihoods / GT / GT_CONF
struct DevGenotype {
    uint32_t n_records, n_alleles;
    const uint32_t* rec_off;     // n_records+1 -> alleles
    const uint32_t* allele_off;  // n_alleles+1 -> allele_kn
    const uint32_t* allele_kn;   // global knode ids
    uint32_t *mean_fwd, *mean_rev, *med_fwd, *med_rev, *sum_fwd, *sum_rev;
    double *gaps, *lik, *gt_conf;
    int32_t* gt;
    // optional (nullptr = skip): the per-record statistics drprg's Filterer / MinorAllele derive from the same vectors
    // (src/filter.rs:212-301, src/minor.rs:70-127, VcfExt src/lib.rs:973-1058,1165-1180), in their f32 arithmetic
    int32_t* covg_gt = nullptr;   // depth on the called allele (all alleles when the call is null)
    float* frs = nullptr;         // fraction of read support; NaN = None
    float* sb_ratio = nullptr;    // strand-bias ratio min(fwd, rev) / (fwd + rev); NaN = None
    int32_t* minor_gt = nullptr;  // allele check_for_minor_alternate would switch the call to; -1 = none
    float* pdp = nullptr;         // per allele: proportion of the position's depth; NaN when the depth is 0
};
void launch_genotype(const int32_t* d_cov, const DevGenotype& G, ModelParams P, cudaStream_t st);
// the VCF record lines formatted on the device (genotype.cu): static CHROM..FORMAT columns + the sample column
struct DevVcfText {
    const char* prefix;          // the records' static columns, back to back
    const uint32_t* prefix_off;  // n_records + 1
    const uint32_t* slot_off;    // n_records + 1: upper bounds of the sample columns
    char* slots;                 // scratch for the sample columns
    uint32_t* line_len;          // n_records
    uint32_t* out_off;           // n_records + 1
    char* text;                  // the lines, back to back (host-mapped pinned memory, 16-byte aligned, text_bound + 16 bytes)
    uint32_t text_bound;         // upper bound of the text's length
    uint32_t* total;             // bytes of text written (host-mapped)
    uint32_t* flags;             // bit 0: a value was refused by the device formatter (host-mapped)
};
void launch_vcf_text(const DevGenotype& G, const DevVcfText& V, cudaStream_t st);
void launch_format_g6_batch(const double* d_v, uint32_t n, char* d_out, uint8_t* d_len, uint8_t* d_refused, cudaStream_t st);
// the likelihood / GT / GT_CONF kernel alone, on per-allele rows already in G.mean_fwd / G.mean_rev / G.gaps
void launch_genotype_rows(const DevGenotype& G, ModelParams P, cudaStream_t st);

// ---- discover: retained hits and reads, region reads and the local assembler (assemble.cu) --------------------------
// The kept hits of a sample on one GPU, appended batch after batch (hit retention on): per hit the global read id and the
// grouped-hit key, per read with a kept hit one row {first hit, hit count}.  A read's hits keep their slice order.
struct RetainStore {
    uint32_t* hit_read;
    unsigned long long* hit_key;
    uint64_t hit_cap;
    uint2* rows;
    uint64_t row_cap;
};
enum : int { RT_WORDS = 0, RT_HITS = 1, RT_ROWS = 2, RT_COUNT = 3 };  // cursors of launch_retain_gather
// per active read of the last batch (n_active, lists of PostBuffers), one warp each: a read with at least one kept hit takes
// one row and appends its kept hits to the store, and its 2-bit words are copied to out_words.  table[row - row_base] =
// {word offset (UINT32_MAX when the words did not fit), length in bases, global read id}.  d_cursor[RT_WORDS] (zero) and
// d_cursor[RT_HITS / RT_ROWS] (the store's fill) count on past the capacities: the caller regrows, resets and launches again.
void launch_retain_gather(const DevReads& R, const uint32_t* act_read, const uint32_t* act_base, const uint32_t* act_count,
                          const unsigned long long* gkey, const uint8_t* gkept, uint32_t n_active, RetainStore S,
                          uint64_t row_base, uint4* table, uint32_t* out_words, uint64_t word_cap, unsigned long long* d_cursor,
                          cudaStream_t st);
struct RegionRead {  // a read with at least min_hits kept hits inside a candidate region
    uint32_t region, read, start, end, fwd;
};
// one warp per row of the store: for every (read, locus) group and every region of that locus (regions
// [locus_region_off[l], locus_region_off[l + 1]), padded intervals pad[r]), the hits whose k-mer node has a consensus start
// cs = cons_start[knode_base[l] + node] (UINT32_MAX: off the ML path) with pad.x <= cs and cs + k <= pad.y: their count, the
// smallest start, the largest start + k and the strand of the first.  Groups with count >= min_hits go to out at slots
// taken from *d_cursor (zeroed by the caller), which counts on past out_cap.
void launch_region_reads(RetainStore S, uint32_t n_rows, const uint32_t* knode_base, const uint32_t* cons_start,
                         const uint32_t* locus_region_off, uint32_t n_loci, const uint2* pad, uint32_t k, uint32_t min_hits,
                         RegionRead* out, uint64_t out_cap, unsigned long long* d_cursor, cudaStream_t st);
constexpr uint32_t DISCOVER_K = 11;             // de Bruijn k-mer size: 22-bit k-mers
constexpr uint32_t KMER_ATTEMPTS = 10;          // anchor k-mers tried per flank
constexpr uint32_t ASM_MAX_PATHS_LIMIT = 64;    // largest max_candidate_paths the walk's shared-memory store takes
constexpr uint32_t ASM_SMEM_SLOTS = 16384;      // k-mer table slots one CTA keeps in shared memory (128 KB)
constexpr uint32_t ASM_MAX_WALK = 1024;         // longest walk (consensus span + max insertion) the kernel takes
enum : uint32_t { ASM_ASSEMBLED = 0, ASM_NO_ANCHOR = 1, ASM_TOO_MANY_PATHS = 2, ASM_NO_PATH = 3 };
struct AsmRegion {
    uint32_t entry_off, n_entries;  // pileup reads: entries[entry_off, + n_entries)
    uint32_t slots;                 // k-mer table slots, a power of two >= 2 x the pileup's k-mer positions
    uint32_t span;                  // padded interval length pe - ps
    unsigned long long table_off;   // global-table launch: first slot of the region's table in the scratch
    uint32_t n_start, n_end;        // anchor candidates: C[ps + i, + K) and C[pe - K - j, pe - j), UINT32_MAX if not ACGT
    uint32_t start_kmer[KMER_ATTEMPTS], end_kmer[KMER_ATTEMPTS];
};
struct AsmResult {
    uint32_t status, anchor_i, anchor_j, n_walks;  // n_walks complete walks (the consensus one included) when assembled
    unsigned long long byte_off;                     // their bases, back to back in out_bases
};
struct AsmParams {
    uint32_t min_dp, max_insertion, max_paths;
};
// one CTA per listed region: count the pileup's k-mers (entries: {word offset into words, start, end, fwd}) into an
// open-addressed table, in shared memory (g_keys == nullptr; every region's slots <= smem_slots) or in the global scratch
// g_keys / g_counts at the region's table_off; then one warp picks the anchors and enumerates the walks.  Complete walks of
// an assembled region go to out_bases at an offset taken from *d_cursor, their lengths to walk_len[region * max_paths + w].
void launch_assemble(const AsmRegion* regions, const uint32_t* list, uint32_t n_list, const uint4* entries, const uint32_t* words,
                     uint32_t smem_slots, uint32_t* g_keys, uint32_t* g_counts, uint32_t max_walk, AsmParams P,
                     AsmResult* res, uint32_t* walk_len, char* out_bases, unsigned long long* d_cursor, cudaStream_t st);

}  // namespace drprg
