// C ABI of include/drprg_cuda.h: the drop-in for Pandora::genotype_with
// (/root/reference/src/lib.rs:580-642) plus the staged interface used for multi-GPU read sharding,
// benches and parity tests.  Owns all device memory of an index (cuda_owned.hpp; no torch types).
#include <cuda_runtime.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <cmath>
#include <map>
#include <cstdio>
#include <cstring>
#include <deque>
#include <fstream>
#include <future>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <thread>
#include <unordered_map>

#include "../../include/drprg_cuda.h"
#include "cuda_owned.hpp"
#include "genotype_host.hpp"
#include "fastq_frame.hpp"
#include "ingest.hpp"
#include "kernels.cuh"
#include "prg_graph.hpp"

using namespace drprg;

namespace {
thread_local std::string g_err;

}  // namespace

// one persistent host thread per extra GPU of a multi-GPU handle: launches for the devices are issued side by side
class GpuWorker {
   public:
    GpuWorker() : th_([this] { loop(); }) {}
    ~GpuWorker() {
        {
            std::lock_guard<std::mutex> g(m_);
            stop_ = true;
        }
        cv_.notify_all();
        th_.join();
    }
    void submit(std::function<void()> fn) {
        {
            std::lock_guard<std::mutex> g(m_);
            task_ = std::move(fn);
            busy_ = true;
            error_.clear();
        }
        cv_.notify_all();
    }
    void wait() {  // rethrows what the task threw
        std::unique_lock<std::mutex> g(m_);
        done_.wait(g, [this] { return !busy_; });
        if (!error_.empty()) throw std::runtime_error(error_);
    }

   private:
    void loop() {
        for (;;) {
            std::function<void()> fn;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [this] { return stop_ || (busy_ && task_); });
                if (stop_) return;
                fn = std::move(task_);
                task_ = nullptr;
            }
            std::string err;
            try {
                fn();
            } catch (const std::exception& e) {
                err = e.what();
            } catch (...) {
                err = "unknown error";
            }
            {
                std::lock_guard<std::mutex> g(m_);
                error_ = err;
                busy_ = false;
            }
            done_.notify_all();
        }
    }
    std::mutex m_;
    std::condition_variable cv_, done_;
    std::function<void()> task_;
    std::string error_;
    bool busy_ = false, stop_ = false;
    std::thread th_;
};

struct drprg_batch {
    // multi-GPU handle: one sub-batch per GPU (this object is then only the container)
    std::vector<std::unique_ptr<drprg_batch>> shards;
    DevReads R{};
    PoolBuf<uint32_t> d_words, d_lens, d_seg_read, d_seg_start;  // empty for a batch wrapping the caller's arrays
    PoolBuf<uint64_t> d_off;
    uint64_t total_bases = 0;
    uint32_t max_len = UINT32_MAX;  // longest read (bound); selects the short-read kernel
    // host uploads are split into chunks copied on a separate stream; the sketch kernel of chunk c starts as soon
    // as its bytes have landed, so the H2D copy overlaps the sketch of the previous chunks
    int n_chunks = 1;
    uint64_t chunk_lo[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    Event ev[8];
};

struct drprg_index {
    HostIndex H;
    int device = 0, sm_count = 148;
    // device-resident index
    DevTable T{};
    DBuf<uint2> d_slots, d_recs;
    DBuf<uint32_t> d_kfilter, d_kfilter14;
    DBuf<uint32_t> d_filter, d_knode_base, d_edge_off, d_edges;
    DBuf<uint8_t> d_is_terminal, d_needs_mean;
    DBuf<uint32_t> d_locus_level_off, d_level_start, d_level_nodes, d_level_singles;
    uint32_t table_slots = 0, filter_words = 0;
    uint64_t n_edges = 0, n_ivs = 0;
    // accumulators: [2*N coverage | P locus reads | 4 scalars]; one exact allocation, never from g_pool: other processes
    // open it through cudaIpcGetMemHandle, and the cross-GPU flag words sit behind it
    DBuf<int32_t> d_accum;
    uint64_t n_accum = 0;
    uint64_t total_bases = 0, n_reads = 0;
    bool scalars_in_buffer = false;
    bool hist_on_host = false;  // h_small holds the coverage histogram + locus read counts of the current accumulators
    // sample state
    SampleOpts opts;
    bool sample_open = false;
    uint32_t first_read_len = 0;
    DBuf<uint32_t> d_thresh;
    uint32_t min_thresh = 0;
    std::vector<uint32_t> thresh_on_device;
    // workspace
    DBuf<unsigned long long> hi, lo;  // unordered hits from the lookup kernels
    DBuf<unsigned long long> gkey;    // hits grouped by read (sorted within a read after the cluster kernels)
    DBuf<uint8_t> gkept;
    DBuf<uint32_t> act_read, act_base, act_count, act_lk, lk_ovf, big_list, cov_keys, scratch[10];
    DBuf<int32_t> read_count;         // per read of a batch; all zero between batches
    DBuf<uint32_t> read_base;
    DBuf<int32_t> partials;           // per-stretch coverage partials (cov_count_kernel): n_partials x n_accum
    uint32_t n_partials = 0;
    DBuf<unsigned long long> queue;  // k-mer screen: flagged (read, position) pairs
    DBuf<uint32_t> queue_kmer;       // ... and their k-mers
    DBuf<unsigned long long> d_counters;  // CTR_* of kernels.cuh
    PinnedBuf<unsigned long long> h_counters;
    uint64_t last_n_hits = 0, last_n_active = 0;
    uint32_t last_id_base = 0;
    // read-sharded runs: where this GPU's coverage goes (nullptr = its own accumulator; otherwise the root GPU's
    // accumulator, peer-mapped, updated with red.global.add by cov_merge_kernel)
    int32_t* reduce_dst = nullptr;
    bool accum_shared = false;  // other GPUs add into this accumulator: the histogram taken at the end of map_batch is not final
    // multi-GPU handle (drprg_cuda_index_load_multi): this object is the root; gpus[0] == this
    std::vector<std::unique_ptr<drprg_index>> replicas;
    std::vector<std::unique_ptr<GpuWorker>> workers;
    std::vector<drprg_index*> gpus;
    uint64_t own_bases = 0, own_reads = 0;  // this GPU's share of the sample (total_bases / n_reads hold the sample's)
    // one PROCESS per GPU (torchrun): flags behind the root's accumulator, reached through a CUDA IPC mapping
    int world = 1;               // ranks sharing the root accumulator (1 = not shared across processes)
    uint32_t epoch = 0;          // samples begun
    void* ipc_mapping = nullptr; // non-root: the root's accumulator allocation opened in this process
    uint32_t* flag_ready = nullptr;     // root's "accumulator zeroed for sample e" word
    uint32_t* flag_arrivals = nullptr;  // root's arrival counter (world - 1 per sample)
    Event ev[6];  // batch timeline: start, lookup done, hits grouped, clustered, coverage merged
    float timings[4] = {0, 0, 0, 0};
    // genotype state
    std::string refs_path;
    std::map<std::string, std::string> refs;
    struct LocusSites {  // read-independent site tables of one locus for the current --vcf-refs
        bool ready = false;
        std::vector<uint32_t> ref_path;
        std::vector<SiteRecord> biallelic, merged;
        SiteKeySet known;
    };
    std::vector<LocusSites> sites;
    std::vector<uint32_t> loci_by_name, loci_by_size;
    FitParams fit;
    std::vector<std::vector<uint32_t>> mlpaths;
    std::vector<char> present;
    std::vector<const SiteRecord*> records, csr_records;  // csr_records: what the device CSR was built for
    std::deque<std::vector<SiteRecord>> sample_records;    // per-sample merged lists (ML path added records)
    GenotypeArrays GA;
    DBuf<uint32_t> d_rec_off, d_allele_off, d_allele_kn, d_knode_locus, d_hist;
    DBuf<uint32_t> d_gt_u32;
    DBuf<double> d_gt_f64;
    DBuf<int32_t> d_gt_i32;
    DBuf<float> d_gt_f32;  // frs | strand-bias ratio (per record), depth proportions (per allele)
    float minor_af = -1.0f;  // < 0: drprg's default (1.0, or 0.1 with --illumina)
    // discover's front half from the map pass (SURVEY 8f rank 1): kept hits of the sample, retained on request
    bool retain_hits = false;
    DBuf<uint32_t> d_rt_hit_read;        // the RetainStore of this GPU, filled to rt_hits hits and rt_rows rows
    DBuf<unsigned long long> d_rt_hit_key;
    DBuf<uint2> d_rt_rows;
    uint64_t rt_hits = 0, rt_rows = 0;
    // ... and the 2-bit words of every read with a kept hit (per global read id: word offset and length in bases)
    struct RetainedReads {
        std::vector<uint32_t> read, len;
        std::vector<uint64_t> off;
        std::vector<uint32_t> words;
    } retained_reads;
    DBuf<uint4> d_rt_table;
    DBuf<uint32_t> d_rt_words;
    DBuf<unsigned long long> d_rt_cursor;  // RT_COUNT: the hit and row cursors carry over from batch to batch
    PinnedBuf<uint4> h_rt_table;
    PinnedBuf<uint32_t> h_rt_words;
    PinnedBuf<unsigned long long> h_rt_cursor;
    DiscoverResult discover;
    bool discover_ready = false;  // drprg_cuda_discover_candidates ran for the current sample
    // the local assembler's results (drprg_cuda_discover_assemble)
    std::vector<uint8_t> asm_status;
    std::vector<drprg_denovo_path> asm_paths;
    std::string asm_bases;
    double asm_stats[4] = {0, 0, 0, 0};
    uint32_t max_locus_knodes = 0, max_locus_edges = 0;
    Event ev_ml[2];
    Stream st_ml, st_gt, st_copy, st_acc;
    Event ev_acc[3];  // [2]: node scores + threshold ready on `st`
    DBuf<double> d_thresh_f64;
    DBuf<int> d_thresh_i32;
    PinnedBuf<int> h_thresh;
    DBuf<uint32_t> d_hist1000;
    PinnedBuf<uint32_t> h_small;  // coverage histogram | locus read counts | scalars  // ML-path kernel / genotype kernels run concurrently
    PinnedBuf<uint32_t> h_path, h_plen, h_u32, h_done;
    PinnedBuf<double> h_f64;
    PinnedBuf<int32_t> h_gt, h_acc;
    double gt_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<std::string> contigs;
    // pandora_genotyped.vcf: header written by the host, record lines written by the device kernels straight into this
    // host-mapped pinned buffer (genotype.cu: vcf_*_kernel); vcf_len bytes are valid, NUL-terminated
    PinnedBuf<char> h_vcf;
    size_t vcf_len = 0, vcf_begin = 0;  // the text is h_vcf[vcf_begin, vcf_begin + vcf_len)
    std::string vcf_header, vcf_fallback;
    DBuf<char> d_vcf_prefix;
    DBuf<uint32_t> d_vcf_prefix_off, d_vcf_slot_off, d_vcf_ctl;  // ctl: [0] text bytes, [1] flags
    DBuf<char> d_vcf_slots;
    DBuf<uint32_t> d_vcf_line_len, d_vcf_out_off;
    PinnedBuf<uint32_t> h_vcf_ctl;
    size_t vcf_prefix_bytes = 0, vcf_slot_bytes = 0;
    bool ga_stale = false;  // the per-allele / per-record arrays are in the pinned download buffers, not yet in GA
    bool have_gt = false;
    bool ml_in_flight = false;  // the ML-path kernel of an unfinished drprg_cuda_genotype may still be writing h_path / h_done
    DBuf<double> d_prob, d_M;
    DBuf<uint32_t> d_len, d_up, d_path, d_path_len;

    // the members free the rest, on this device; a host-only handle (device -1) owns nothing and makes no CUDA call
    ~drprg_index() {
        workers.clear();
        replicas.clear();
        if (device < 0) return;
        cudaSetDevice(device);
        if (ipc_mapping) cudaIpcCloseMemHandle(ipc_mapping);
    }
};

namespace {
inline size_t accum_flag_offset(uint64_t n_accum) { return (size_t)((n_accum + 31) & ~31ull); }  // 128-byte aligned flag words

// ~24 filter bits per entry, capped by the shared memory of one SM
std::vector<uint32_t> screen_filter(const std::vector<uint32_t>& kmers, uint32_t k) {
    uint32_t nw = (uint32_t)std::min<uint64_t>(SCREEN_MAX_FILTER_WORDS, std::max<uint64_t>(1024, (kmers.size() * 24 + 31) / 32));
    nw = (nw + 3) & ~3u;
    std::vector<uint32_t> f(nw, 0);
    for (uint32_t x : kmers) screen_filter_insert(f.data(), nw, x, k);
    return f;
}

// k-mer screen filters (k = 15): the k-mers behind the indexed hashes in both orientations (hash64 is invertible), and the
// two 14-mers of each of them, which the screen tests at every other read position
struct ScreenFilters {
    std::vector<uint32_t> kfilter, kfilter14;  // both empty: the index keeps the sketch kernels
};
ScreenFilters build_screen_filters(const HostIndex& H) {
    ScreenFilters F;
    if (H.k != 15 || H.records.empty()) return F;
    const uint64_t mask = (1ull << (2 * H.k)) - 1;
    std::vector<uint32_t> kmers;
    kmers.reserve(H.records.size() * 2);
    for (size_t i = 0; i < H.records.size(); ++i) {
        if (i && H.records[i - 1].hash == H.records[i].hash) continue;
        const uint64_t y = hash64_inverse_host(H.records[i].hash, mask);
        if (hash64_host(y, mask) != H.records[i].hash) throw std::runtime_error("hash64 inversion failed");
        uint64_t rc = 0, t = y;
        for (uint32_t b = 0; b < H.k; ++b) {
            rc = (rc << 2) | (3 - (t & 3));
            t >>= 2;
        }
        kmers.push_back((uint32_t)y);
        kmers.push_back((uint32_t)rc);
    }
    std::sort(kmers.begin(), kmers.end());
    kmers.erase(std::unique(kmers.begin(), kmers.end()), kmers.end());
    std::vector<uint32_t> sub;
    sub.reserve(kmers.size() * 2);
    for (uint32_t x : kmers) {
        sub.push_back(x >> 2);                              // bases 0..13
        sub.push_back(x & ((1u << (2 * (H.k - 1))) - 1u));  // bases 1..14
    }
    std::sort(sub.begin(), sub.end());
    sub.erase(std::unique(sub.begin(), sub.end()), sub.end());
    // The filters are capped by one SM's shared memory (1.77 Mbit).  Beyond ~300 k k-mers (4x the Mtb-scale panel) more
    // than a third of the 15-mer filter's bits are set, over 10 % of all read positions are flagged and resolving them
    // costs as much as sketching every read: such an index keeps the sketch kernels.
    if (kmers.size() > 300000) return F;
    F.kfilter = screen_filter(kmers, H.k);
    F.kfilter14 = screen_filter(sub, H.k - 1);
    return F;
}

void upload_index(drprg_index* X) {
    const HostIndex& H = X->H;
    if (H.k > (uint32_t)K_MAX) throw std::runtime_error("k > 16 is not supported by the device kernels (2k must fit 32 bits)");
    if (H.w > (uint32_t)W_MAX) throw std::runtime_error("w > 32 is not supported by the device kernels");
    if (H.loci.size() > 65535) throw std::runtime_error("more than 65535 loci");
    for (size_t l = 0; l < H.loci.size(); ++l)
        if (H.loci[l].kpath.size() >= (1ull << GKEY_KNODE_BITS)) throw std::runtime_error("a locus has more than 4 M k-mer nodes");
    if (2ull * H.total_knodes() + H.loci.size() >= (1ull << 31)) throw std::runtime_error("too many k-mer nodes for 32-bit coverage keys");
    // ---- hash table + pre-filter
    std::vector<uint2> recs;
    recs.reserve(H.records.size() + 16);
    size_t distinct = 0;
    for (size_t i = 0; i < H.records.size(); ++i)
        if (i == 0 || H.records[i - 1].hash != H.records[i].hash) ++distinct;
    uint32_t sb = 10;
    while ((1ull << sb) < distinct * 2) ++sb;
    uint32_t fb = 8;
    while ((1ull << fb) < (distinct + 3) / 4) ++fb;  // ~4 keys per 32-bit word: 2 % false positives, 64 KB for a 60 k-key panel
    std::vector<uint2> slots(1ull << sb, make_uint2(0, 0));
    std::vector<uint32_t> filter(1ull << fb, 0);
    for (size_t i = 0; i < H.records.size();) {
        size_t j = i;
        while (j < H.records.size() && H.records[j].hash == H.records[i].hash) ++j;
        // a minimizer in 255 or more k-mer nodes (pandora has no limit): count 255 = "the real count is in a header
        // pseudo-record in front of the group" (rec_span in kernels.cu)
        const uint32_t count = (uint32_t)(j - i), begin = (uint32_t)recs.size();
        if (count >= 255u) recs.push_back(make_uint2(count, 0xffffffffu));
        for (size_t q = i; q < j; ++q) recs.push_back(make_uint2(H.records[q].knode, (H.records[q].prg << 1) | H.records[q].strand));
        if (recs.size() >= (1u << 24)) throw std::runtime_error("too many index records");
        const uint32_t h = (uint32_t)H.records[i].hash;
        uint32_t s = (h * 0x9E3779B1u) >> (32 - sb);
        while (slots[s].y != 0) s = (s + 1) & ((1u << sb) - 1);
        slots[s] = make_uint2(h, begin | (std::min(count, 255u) << 24));
        filter[h & ((1u << fb) - 1)] |= (1u << ((h >> fb) & 31)) | (1u << ((h >> (fb + 5)) & 31));
        i = j;
    }
    X->d_slots.assign(slots);
    X->d_recs.assign(recs);
    X->d_filter.assign(filter);
    X->table_slots = 1u << sb;
    X->filter_words = 1u << fb;
    X->T = DevTable{X->d_slots.p, sb, X->d_recs.p, X->d_filter.p, fb};
    const ScreenFilters F = build_screen_filters(H);
    if (!F.kfilter.empty()) {
        X->d_kfilter.assign(F.kfilter);
        X->d_kfilter14.assign(F.kfilter14);
        X->T.kfilter = X->d_kfilter.p;
        X->T.kfilter_words = (uint32_t)F.kfilter.size();
        X->T.kfilter14 = X->d_kfilter14.p;
        X->T.kfilter14_words = (uint32_t)F.kfilter14.size();
    }
    // ---- k-mer graphs
    const uint32_t N = H.total_knodes();
    std::vector<uint32_t> edge_off(N + 1, 0), edges;
    std::vector<uint8_t> term(N, 0);
    uint64_t n_ivs = 0;
    for (size_t l = 0; l < H.loci.size(); ++l) {
        const Locus& L = H.loci[l];
        const uint32_t base = H.knode_base[l];
        for (uint32_t r = 0; r < L.kpath.size(); ++r) {
            edge_off[base + r] = (uint32_t)edges.size();
            for (uint32_t o : L.kout[r]) edges.push_back(o);
            n_ivs += L.kpath[r].size();
        }
        term[base] = 1;
        term[base + (uint32_t)L.kpath.size() - 1] = 1;
    }
    edge_off[N] = (uint32_t)edges.size();
    X->n_edges = edges.size();
    X->n_ivs = n_ivs;
    X->d_knode_base.assign(H.knode_base);
    X->d_edge_off.assign(edge_off);
    X->d_edges.assign(edges);
    X->d_is_terminal.assign(term);
    {   // a node's mean log-prob is only ever compared when one of its predecessors has more than one out-edge
        std::vector<uint8_t> needs(N, 0);
        for (size_t l = 0; l < H.loci.size(); ++l) {
            const Locus& L = H.loci[l];
            const uint32_t base = H.knode_base[l];
            for (uint32_t r = 0; r < L.kpath.size(); ++r)
                if (L.kout[r].size() > 1)
                    for (uint32_t o : L.kout[r]) needs[base + o] = 1;
        }
        X->d_needs_mean.assign(needs);
    }
    {   // level order for the level-parallel ML-path kernel: level = 1 + max level of the successors (terminus = 0)
        std::vector<uint32_t> locus_level_off(1, 0), level_start(1, 0), level_nodes, level_singles;
        for (size_t l = 0; l < H.loci.size(); ++l) {
            const Locus& L = H.loci[l];
            const uint32_t n = (uint32_t)L.kpath.size();
            std::vector<uint32_t> lev(n, 0);
            uint32_t max_lev = 0;
            for (uint32_t r = n >= 2 ? n - 1 : 0; r-- > 0;) {  // successors have higher ranks
                uint32_t m = 0;
                for (uint32_t o : L.kout[r]) m = std::max(m, lev[o]);
                lev[r] = m + 1;
                max_lev = std::max(max_lev, lev[r]);
            }
            std::vector<std::vector<uint32_t>> by(max_lev + 1);
            for (uint32_t r = n >= 2 ? n - 1 : 0; r-- > 0;) by[lev[r]].push_back(r);
            for (uint32_t v = 1; v <= max_lev; ++v) {  // single-successor nodes first: they go to their own warps
                std::stable_partition(by[v].begin(), by[v].end(), [&](uint32_t r) { return L.kout[r].size() == 1; });
                uint32_t ns = 0;
                for (uint32_t r : by[v]) ns += L.kout[r].size() == 1;
                level_nodes.insert(level_nodes.end(), by[v].begin(), by[v].end());
                level_start.push_back((uint32_t)level_nodes.size());
                level_singles.push_back(ns);
            }
            locus_level_off.push_back((uint32_t)level_start.size() - 1);
        }
        X->d_locus_level_off.assign(locus_level_off);
        X->d_level_start.assign(level_start);
        X->d_level_nodes.assign(level_nodes);
        X->d_level_singles.assign(level_singles);
    }
    X->n_accum = 2ull * N + H.loci.size() + 4;
    // 16 extra words behind the accumulator hold the cross-GPU flags of a read-sharded run (ready epoch, arrival counter)
    const size_t accum_words = accum_flag_offset(X->n_accum) + 16;
    X->d_accum.reserve(accum_words, accum_words);
    CK(cudaMemset(X->d_accum.p, 0, accum_words * sizeof(int32_t)));
    X->d_thresh.reserve(std::max<size_t>(1, H.loci.size()), std::max<size_t>(1, H.loci.size()));
    X->d_counters.reserve(CTR_COUNT, CTR_COUNT);
    X->h_counters.reserve(CTR_COUNT, CTR_COUNT);

    for (auto& e : X->ev) e = new_event(cudaEventDefault);
    std::vector<uint32_t> knode_locus(N);
    for (size_t l = 0; l < H.loci.size(); ++l) {
        for (uint32_t g = H.knode_base[l]; g < H.knode_base[l + 1]; ++g) knode_locus[g] = (uint32_t)l;
        X->max_locus_knodes = std::max(X->max_locus_knodes, H.knode_base[l + 1] - H.knode_base[l]);
        X->max_locus_edges = std::max(X->max_locus_edges, edge_off[H.knode_base[l + 1]] - edge_off[H.knode_base[l]]);
    }
    X->d_knode_locus.assign(knode_locus);
    X->d_hist.reserve(200, 200);
    X->d_hist1000.reserve(1000, 1000);
    X->sites.assign(H.loci.size(), drprg_index::LocusSites());
    X->loci_by_name.resize(H.loci.size());
    for (uint32_t l = 0; l < H.loci.size(); ++l) X->loci_by_name[l] = l;
    std::sort(X->loci_by_name.begin(), X->loci_by_name.end(),
              [&](uint32_t a, uint32_t b) { return H.loci[a].name < H.loci[b].name; });
    X->loci_by_size = X->loci_by_name;
    std::stable_sort(X->loci_by_size.begin(), X->loci_by_size.end(),
                     [&](uint32_t a, uint32_t b) { return H.loci[a].kpath.size() > H.loci[b].kpath.size(); });
}

int load_common(const std::string& text, uint32_t w, uint32_t k, int device, drprg_index** out) {
    std::unique_ptr<drprg_index> X(new drprg_index());
    X->device = device;
    if (device == -1) {  // host-only handle: index introspection; every compute entry point refuses it
        X->H = build_host_index(text, w, k);
        *out = X.release();
        return 0;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw std::runtime_error("no CUDA device visible: drprg-cuda has no CPU fallback");
    if (device < 0 || device >= ndev) throw std::runtime_error("bad device ordinal");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    X->sm_count = prop.multiProcessorCount;
    X->H = build_host_index(text, w, k);
    upload_index(X.get());
    *out = X.release();
    return 0;
}

SampleOpts opts_from(const drprg_map_opts* o, uint32_t k) {
    SampleOpts s;
    if (o) {
        s.threads = o->threads ? o->threads : 1;
        s.min_cluster_size = o->min_cluster_size;
        s.illumina = o->illumina != 0;
        if (o->genome_size) s.genome_size = o->genome_size;
        s.gt_conf = o->gt_conf;
        if (o->genotyping_error_rate > 0) s.gt_error_rate = o->genotyping_error_rate;
        if (o->max_diff) s.max_diff = o->max_diff;
        if (o->error_rate > 0) s.e_rate = o->error_rate;
    }
    if (s.illumina) {  // pandora map -I
        if (s.e_rate == 0.11) s.e_rate = 0.001;
        if (s.max_diff > 200) s.max_diff = 2 * k + 1;
    }
    return s;
}

void need_device(drprg_index* X) {
    if (X->device < 0) throw std::runtime_error("host-only index (device = -1): the map path has no CPU fallback");
}

void sample_begin(drprg_index* X, const drprg_map_opts* o, uint32_t first_read_len) {
    need_device(X);
    CK(cudaSetDevice(X->device));
    X->opts = opts_from(o, X->H.k);
    X->first_read_len = first_read_len;
    uint32_t expected = UINT32_MAX;
    if (X->opts.illumina) expected = first_read_len * 2 / (X->H.w + 1);
    const double fraction = 0.5 / std::exp(X->opts.e_rate * X->H.k);
    std::vector<uint32_t> thr(X->H.loci.size());
    for (size_t l = 0; l < thr.size(); ++l) {
        uint32_t lbt = (uint32_t)(std::min(X->H.loci[l].min_path_len, expected) * fraction);
        thr[l] = std::max(lbt, X->opts.min_cluster_size);
    }
    X->min_thresh = thr.empty() ? 0u : *std::min_element(thr.begin(), thr.end());
    if (thr != X->thresh_on_device) {  // unchanged between the samples of a batch: skip the synchronous copy
        if (!thr.empty()) CK(cudaMemcpy(X->d_thresh.p, thr.data(), thr.size() * 4, cudaMemcpyHostToDevice));
        X->thresh_on_device = thr;
    }
    CK(cudaMemset(X->d_accum.p, 0, X->n_accum * sizeof(int32_t)));
    ++X->epoch;
    if (X->world > 1 && X->accum_shared)  // the other ranks may add to this accumulator from here on
        launch_flag_publish(reinterpret_cast<uint32_t*>(X->d_accum.p + accum_flag_offset(X->n_accum)), X->epoch, 0);
    X->total_bases = X->n_reads = 0;
    X->own_bases = X->own_reads = 0;
    X->rt_hits = X->rt_rows = 0;
    X->retained_reads = drprg_index::RetainedReads();
    X->discover_ready = false;
    X->scalars_in_buffer = false;
    X->hist_on_host = false;
    X->sample_open = true;
    X->have_gt = false;
}

void ensure_hit_capacity(drprg_index* X, uint64_t cap) {
    if (cap >= 0xfffffff0ull) throw std::runtime_error("more than 2^32 hits in one batch: split the batch");
    if (cap <= X->hi.cap) return;
    X->hi.ensure(cap);
    const size_t c = X->hi.cap;  // every per-hit buffer follows the hit buffer's capacity
    X->lo.ensure(c); X->gkey.ensure(c); X->gkept.ensure(c);
    X->act_read.ensure(c); X->act_base.ensure(c); X->act_count.ensure(c);
    X->act_lk.ensure(2 * c); X->lk_ovf.ensure(c);
    X->big_list.ensure(c / CLUSTER_WARP_MAX + 16);
    X->cov_keys.ensure(c);
    for (auto& b : X->scratch) b.ensure(c);
    X->n_partials = cov_max_stretches(c, X->sm_count);
    X->partials.ensure((size_t)X->n_partials * X->n_accum);
}

void ensure_read_capacity(drprg_index* X, uint64_t n_reads) {
    if (n_reads <= X->read_count.cap) return;
    X->read_count.ensure(n_reads);
    X->read_base.ensure(X->read_count.cap);
    CK(cudaMemset(X->read_count.p, 0, X->read_count.cap * sizeof(int32_t)));  // the kernels leave it zero after every batch
}

RetainStore retain_store(drprg_index* X) {
    return RetainStore{X->d_rt_hit_read.p, X->d_rt_hit_key.p, std::min(X->d_rt_hit_read.cap, X->d_rt_hit_key.cap), X->d_rt_rows.p,
                       X->d_rt_rows.cap};
}

// grow-only like DBuf::ensure, but the first `used` elements survive the move to the larger buffer
template <class T>
void grow_keep(DBuf<T>& b, size_t used, size_t need, cudaStream_t st) {
    if (need <= b.cap) return;
    DBuf<T> g;
    g.ensure(need);
    if (used) CK(cudaMemcpyAsync(g.p, b.p, used * sizeof(T), cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    b = std::move(g);
}

// The kept hits of the batch into the GPU's retained-hit store, and the words of the reads that kept a hit into the
// sample's host-side store: the assembler needs their bases after the batch (a file's wave) is gone.  What a store lacked
// is counted past its capacity: it regrows, keeping what earlier batches appended, and the append is redone.
void retain_batch(drprg_index* X, drprg_batch* B, cudaStream_t st) {
    const uint64_t na = X->last_n_active;
    if (!na) return;
    X->d_rt_table.ensure(na);
    X->d_rt_cursor.ensure(RT_COUNT);
    if (!X->d_rt_words.cap) X->d_rt_words.ensure(na * 16);
    grow_keep(X->d_rt_rows, X->rt_rows, X->rt_rows + na, st);  // at most one row per active read: never short
    grow_keep(X->d_rt_hit_read, X->rt_hits, X->rt_hits + na, st);  // first guess: one kept hit per active read
    grow_keep(X->d_rt_hit_key, X->rt_hits, X->rt_hits + na, st);
    // a new sample starts its store empty; later batches only restart the per-batch words cursor
    CK(cudaMemsetAsync(X->d_rt_cursor.p, 0, (X->rt_hits || X->rt_rows ? 1 : RT_COUNT) * sizeof(unsigned long long), st));
    X->h_rt_cursor.resize(RT_COUNT);
    const unsigned long long* c = X->h_rt_cursor.data();
    for (;;) {
        const RetainStore S = retain_store(X);
        launch_retain_gather(B->R, X->act_read.p, X->act_base.p, X->act_count.p, X->gkey.p, X->gkept.p, (uint32_t)na, S, X->rt_rows,
                             X->d_rt_table.p, X->d_rt_words.p, X->d_rt_words.cap, X->d_rt_cursor.p, st);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(X->h_rt_cursor.data(), X->d_rt_cursor.p, RT_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (c[RT_WORDS] <= X->d_rt_words.cap && c[RT_HITS] <= S.hit_cap && c[RT_ROWS] <= S.row_cap) break;
        if (c[RT_WORDS] >= 0xffffffffull) throw std::runtime_error("the reads of one batch that kept a hit exceed 2^32 words: split the batch");
        if (c[RT_HITS] >= 0xffffffffull) throw std::runtime_error("the kept hits of one sample exceed 2^32 on one GPU");
        X->d_rt_words.ensure(c[RT_WORDS]);
        grow_keep(X->d_rt_hit_read, X->rt_hits, c[RT_HITS], st);
        grow_keep(X->d_rt_hit_key, X->rt_hits, c[RT_HITS], st);
        grow_keep(X->d_rt_rows, X->rt_rows, c[RT_ROWS], st);
        const unsigned long long again[RT_COUNT] = {0, X->rt_hits, X->rt_rows};  // the batch's append is redone
        CK(cudaMemcpyAsync(X->d_rt_cursor.p, again, sizeof again, cudaMemcpyHostToDevice, st));
    }
    const uint64_t n_rows = c[RT_ROWS] - X->rt_rows, used = c[RT_WORDS];
    X->rt_hits = c[RT_HITS];
    X->rt_rows = c[RT_ROWS];
    X->h_rt_table.resize(n_rows);
    X->h_rt_words.resize(used);
    if (n_rows) CK(cudaMemcpyAsync(X->h_rt_table.data(), X->d_rt_table.p, n_rows * sizeof(uint4), cudaMemcpyDeviceToHost, st));
    if (used) CK(cudaMemcpyAsync(X->h_rt_words.data(), X->d_rt_words.p, used * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    drprg_index::RetainedReads& R = X->retained_reads;
    const uint64_t base = R.words.size();
    R.words.insert(R.words.end(), X->h_rt_words.begin(), X->h_rt_words.end());
    for (const uint4& t : X->h_rt_table) {
        R.read.push_back(t.z);
        R.off.push_back(base + t.x);
        R.len.push_back(t.y);
    }
}

void map_batch(drprg_index* X, drprg_batch* B, cudaStream_t st, uint64_t* n_hits, uint64_t* n_kept) {
    if (!X->sample_open) throw std::runtime_error("drprg_cuda_sample_begin was not called");
    CK(cudaSetDevice(X->device));
    const HostIndex& H = X->H;
    if (B->max_len != UINT32_MAX && B->max_len >= (1u << GKEY_START_BITS)) throw std::runtime_error("reads of 32 Mb or more are not supported");
    // whole-genome reads give ~0.35 hits per 150 bp read; a targeted run overflows once, regrows to the exact count and is redone
    ensure_hit_capacity(X, std::max<uint64_t>(X->hi.cap, std::max<uint64_t>(1u << 20, B->total_bases / 256)));
    ensure_read_capacity(X, B->R.n_reads);
    if (X->T.kfilter) {  // ~0.6 queued candidates per whole-genome 150 bp read; room for ~8x that, reads on the panel queue more
        X->queue.ensure(std::max<uint64_t>(X->queue.cap, B->total_bases / 32 + (1u << 20)));
        X->queue_kmer.ensure(X->queue.cap);
    }
    const uint32_t N = H.total_knodes(), P = (uint32_t)H.loci.size();
    uint64_t nh = 0;
    // The whole batch is enqueued without a host round trip: the kernels after the lookup read their sizes from the
    // device counters.  A buffer that turned out too small is noticed at the end (the kernels downstream of an overflow
    // skip their work, the accumulators are untouched) and the batch is redone with larger buffers.
    for (int attempt = 0;; ++attempt) {
        const uint64_t queue_cap = X->T.kfilter ? std::min(X->queue.cap, X->queue_kmer.cap) : 0;
        if (queue_cap >= (1ull << 31)) throw std::runtime_error("k-mer screen queue beyond 2^31 entries");  // resolve stages 31-bit indices
        CK(cudaMemsetAsync(X->d_counters.p, 0, CTR_COUNT * sizeof(unsigned long long), st));
        CK(cudaEventRecord(X->ev[0].get(), st));
        for (int c = 0; c < B->n_chunks; ++c) {
            DevReads Rc = B->R;
            Rc.hit_count = X->read_count.p;
            if (B->n_chunks > 1) {
                const uint64_t lo = B->chunk_lo[c], hi = B->chunk_lo[c + 1];
                Rc.hit_count = X->read_count.p + lo;
                if (B->ev[c]) CK(cudaStreamWaitEvent(st, B->ev[c].get(), 0));
                Rc.words = B->R.stride_words ? B->R.words + lo * B->R.stride_words : B->R.words;
                Rc.word_off = B->R.word_off ? B->R.word_off + lo : nullptr;
                Rc.lens = B->R.lens + lo;
                Rc.n_reads = hi - lo;
                Rc.read_id_base = B->R.read_id_base + (uint32_t)lo;
            }
            launch_sketch_lookup(Rc, X->T, H.w, H.k, X->hi.p, X->lo.p, X->d_counters.p + CTR_HITS, X->hi.cap, X->sm_count, B->max_len, st,
                                 X->queue.p, queue_cap, X->d_counters.p + CTR_QUEUE, X->queue_kmer.p);
        }
        CK(cudaGetLastError());
        CK(cudaEventRecord(X->ev[1].get(), st));
        PostBuffers PB{};
        PB.hi = X->hi.p; PB.lo = X->lo.p; PB.ctr = X->d_counters.p;
        PB.read_count = X->read_count.p; PB.read_base = X->read_base.p;
        PB.act_read = X->act_read.p; PB.act_base = X->act_base.p; PB.act_count = X->act_count.p;
        PB.act_lk = X->act_lk.p; PB.lk_ovf = X->lk_ovf.p;
        PB.big_list = X->big_list.p; PB.gkey = X->gkey.p; PB.gkept = X->gkept.p; PB.cov_keys = X->cov_keys.p;
        for (int i = 0; i < 10; ++i) PB.scratch[i] = X->scratch[i].p;
        PB.partials = X->partials.p; PB.n_partials = X->n_partials;
        if (X->reduce_dst && X->flag_ready) launch_flag_wait(X->flag_ready, X->epoch, st);  // root has zeroed its accumulator for this sample
        launch_postprocess(PB, PostCaps{X->hi.cap, queue_cap}, B->R.read_id_base, B->R.n_reads, X->opts.max_diff, X->min_thresh, X->d_thresh.p,
                           X->d_knode_base.p, N, P, X->reduce_dst ? X->reduce_dst : X->d_accum.p,
                           (X->reduce_dst || X->accum_shared) ? 1 : 0,  // several GPUs add into one accumulator: every writer uses red
                           X->sm_count, st,
                           X->ev[2].get(), X->ev[3].get());
        CK(cudaEventRecord(X->ev[4].get(), st));
        CK(cudaGetLastError());
        if (!X->reduce_dst && !X->accum_shared) {
            // what the genotype step needs first (coverage histogram, locus read counts: 4 KB) rides on this batch's final
            // synchronisation; it stays valid unless the accumulators change before drprg_cuda_genotype (another batch
            // recomputes it, a reduce from other GPUs invalidates it)
            launch_cov_hist(X->d_accum.p, N, X->d_is_terminal.p, X->d_knode_locus.p, X->d_accum.p + 2ull * N, X->d_hist1000.p, st);
            X->h_small.resize(1000 + (size_t)P + 4);
            CK(cudaMemcpyAsync(X->h_small.data(), X->d_hist1000.p, 1000 * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(X->h_small.data() + 1000, X->d_accum.p + 2ull * N, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaMemcpyAsync(X->h_counters.p, X->d_counters.p, CTR_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nh = X->h_counters.p[CTR_HITS];
        const uint64_t nq = X->h_counters.p[CTR_QUEUE_NEED];  // largest screen queue any chunk wanted
        if (nh <= X->hi.cap && nq <= queue_cap) break;
        if (attempt == 2) throw std::runtime_error("hit buffer overflow");
        // the lookup kernels counted hits per read that were never scattered: the counters must be zero before the redo
        CK(cudaMemsetAsync(X->read_count.p, 0, X->read_count.cap * sizeof(int32_t), st));
        if (nh > X->hi.cap) ensure_hit_capacity(X, nh);
        if (nq > queue_cap) {
            X->queue.ensure(nq);
            X->queue_kmer.ensure(X->queue.cap);
        }
    }
    static const bool timing = getenv("DRPRG_TIMING") != nullptr;
    if (timing)
        fprintf(stderr, "[drprg-cuda] map batch: %llu reads, %d chunks, screen queue %llu (largest chunk), probe survivors %llu, hits %llu, active reads %llu\n",
                (unsigned long long)B->R.n_reads, B->n_chunks, X->h_counters.p[CTR_QUEUE_NEED], X->h_counters.p[CTR_SURVIVORS], (unsigned long long)nh,
                X->h_counters.p[CTR_ACTIVE]);
    X->hist_on_host = !X->reduce_dst && !X->accum_shared;
    CK(cudaEventElapsedTime(&X->timings[0], X->ev[0].get(), X->ev[1].get()));
    CK(cudaEventElapsedTime(&X->timings[1], X->ev[1].get(), X->ev[2].get()));
    CK(cudaEventElapsedTime(&X->timings[2], X->ev[2].get(), X->ev[3].get()));
    CK(cudaEventElapsedTime(&X->timings[3], X->ev[3].get(), X->ev[4].get()));
    X->last_n_hits = nh;
    X->last_n_active = X->h_counters.p[CTR_ACTIVE];
    X->last_id_base = B->R.read_id_base;
    X->total_bases += B->total_bases;
    X->n_reads += B->R.n_reads;
    X->own_bases += B->total_bases;
    X->own_reads += B->R.n_reads;
    if (X->retain_hits && nh) retain_batch(X, B, st);
    if (n_hits) *n_hits = nh;
    if (n_kept) *n_kept = X->h_counters.p[CTR_KEPT];
}

void flush_scalars(drprg_index* X) {
    if (X->scalars_in_buffer) return;
    int32_t s[4] = {(int32_t)(X->total_bases & 0xffffff), (int32_t)(X->total_bases >> 24), (int32_t)(X->n_reads & 0xffffff),
                    (int32_t)(X->n_reads >> 24)};
    if (X->accum_shared && X->world > 1) {  // the other ranks have added their scalars (shard_done): this rank's join them
        launch_add_scalars(X->d_accum.p + X->n_accum - 4, s, 0);
        CK(cudaStreamSynchronize(0));
    } else {
        CK(cudaMemcpy(X->d_accum.p + X->n_accum - 4, s, sizeof s, cudaMemcpyHostToDevice));
    }
    X->scalars_in_buffer = true;
}

// The genotype arrays of the last sample as host vectors (getters, the host text formatter): the step itself leaves them
// in the pinned download buffers, the copies into GA are made on first use.
void ensure_ga(drprg_index* X) {
    if (!X->ga_stale) return;
    GenotypeArrays& G = X->GA;
    const size_t nr = X->records.size(), na = G.allele_off.empty() ? 0 : G.allele_off.size() - 1;
    std::vector<uint32_t>* cols[6] = {&G.mean_fwd, &G.mean_rev, &G.med_fwd, &G.med_rev, &G.sum_fwd, &G.sum_rev};
    for (auto* v : cols) v->resize(na);
    G.gaps.resize(na);
    G.lik.resize(na);
    G.gt_conf.resize(nr);
    G.gt.resize(nr);
    if (nr) {
        std::copy(X->h_gt.begin(), X->h_gt.end(), G.gt.begin());
        for (int c = 0; c < 6; ++c)
            std::copy(X->h_u32.begin() + (size_t)c * na, X->h_u32.begin() + (size_t)(c + 1) * na, cols[c]->begin());
        std::copy(X->h_f64.begin(), X->h_f64.begin() + na, G.gaps.begin());
        std::copy(X->h_f64.begin() + na, X->h_f64.begin() + 2 * (size_t)na, G.lik.begin());
        std::copy(X->h_f64.begin() + 2 * (size_t)na, X->h_f64.end(), G.gt_conf.begin());
    }
    X->ga_stale = false;
}

void genotype(drprg_index* X, const char* vcf_refs, const char* sample) {
    if (!X->sample_open) throw std::runtime_error("drprg_cuda_sample_begin was not called");
    need_device(X);
    CK(cudaSetDevice(X->device));
    const HostIndex& H = X->H;
    const uint32_t N = H.total_knodes(), P = (uint32_t)H.loci.size();
    cudaStream_t st = 0;
    double t0 = now_ms();
    auto lap = [&](int i) {
        const double t = now_ms();
        X->gt_ms[i] = t - t0;
        t0 = t;
    };
    // a previous call that threw after launching the ML-path kernel may have left it running: it writes into the pinned
    // path / flag buffers this call is about to reset
    if (X->ml_in_flight) {
        cudaStreamSynchronize(X->st_ml.get());
        X->ml_in_flight = false;
    }
    // --vcf-refs is loaded before anything is launched (a bad path must not leave kernels behind)
    {
        const std::string rp = vcf_refs ? vcf_refs : "";
        if (rp != X->refs_path) {
            X->refs = rp.empty() ? std::map<std::string, std::string>() : load_fasta(rp);
            X->refs_path = rp;
            for (auto& s : X->sites) s = drprg_index::LocusSites();
            X->csr_records.clear();
        }
    }
    if (X->accum_shared && X->world > 1)  // every other rank has finished adding its shard (shard_done)
        launch_flag_wait(reinterpret_cast<uint32_t*>(X->d_accum.p + accum_flag_offset(X->n_accum)) + 1, X->epoch * (uint32_t)(X->world - 1), 0);
    const bool reuse_hist = X->hist_on_host;  // downloaded at the end of the last map_batch, accumulators untouched since
    if (!reuse_hist) flush_scalars(X);
    if (!X->st_ml) {
        X->st_ml = new_stream();
        X->st_gt = new_stream();
        X->st_acc = new_stream();
        for (auto& e : X->ev_acc) e = new_event(cudaEventDisableTiming);
        X->d_thresh_f64.reserve(1, 1);
        X->d_thresh_i32.reserve(1, 1);
    }
    // On the critical path the host only needs the 1000-bin coverage histogram (built on the device), the locus read
    // counts and the scalars: 4 KB.  The full accumulator (0.3 MB, pinned destination) is needed when the ML paths are
    // verified; it comes down on its own stream, ordered after whatever produced the accumulator on `st` (map_batch, or
    // the caller's allreduce).
    X->h_acc.resize(X->n_accum);
    CK(cudaEventRecord(X->ev_acc[0].get(), st));
    CK(cudaStreamWaitEvent(X->st_acc.get(), X->ev_acc[0].get(), 0));
    CK(cudaMemcpyAsync(X->h_acc.data(), X->d_accum.p, X->n_accum * 4, cudaMemcpyDeviceToHost, X->st_acc.get()));
    CK(cudaEventRecord(X->ev_acc[1].get(), X->st_acc.get()));
    uint64_t total_bases = X->total_bases;  // this process's batches; after an allreduce the summed scalars are read back
    if (!reuse_hist) {
        launch_cov_hist(X->d_accum.p, N, X->d_is_terminal.p, X->d_knode_locus.p, X->d_accum.p + 2ull * N, X->d_hist1000.p, st);
        X->h_small.resize(1000 + (size_t)P + 4);
        CK(cudaMemcpyAsync(X->h_small.data(), X->d_hist1000.p, 1000 * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(X->h_small.data() + 1000, X->d_accum.p + 2ull * N, ((size_t)P + 4) * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int32_t* sc = (const int32_t*)(X->h_small.data() + 1000) + P;
        total_bases = (uint64_t)(uint32_t)sc[0] + ((uint64_t)(uint32_t)sc[1] << 24);
    }
    const int32_t* cov = X->h_acc.data();  // valid after ev_acc[1]
    const int32_t* locus_reads = (const int32_t*)(X->h_small.data() + 1000);
    lap(0);
    // ---- S6: moments / model choice on the host, histograms on the device
    X->fit = fit_parameters_hist(H, X->h_small.data(), locus_reads, total_bases, X->opts);
    ModelParams MP{};
    MP.bin = X->fit.bin;
    MP.nb_p = X->fit.nb_p;
    MP.nb_r = X->fit.nb_r;
    MP.bin_p = 1.0 / std::exp(X->fit.e_rate * H.k);
    MP.exp_depth = X->fit.E;
    MP.window = X->opts.window;
    MP.min_kmer_covg = X->fit.min_kmer_covg;
    MP.gt_err = X->opts.gt_error_rate;
    MP.gt_conf = X->opts.gt_conf;
    MP.minor_af = X->minor_af >= 0.0f ? X->minor_af : (X->opts.illumina ? 0.1f : 1.0f);  // src/minor.rs:11-12,26-33
    X->d_prob.ensure(N); X->d_M.ensure(N); X->d_len.ensure(N);
    X->d_up.ensure((size_t)N * LV_MAX); X->d_path.ensure(N); X->d_path_len.ensure(P);
    launch_node_prob(X->d_accum.p, N, X->d_is_terminal.p, MP, X->d_prob.p, st);
    launch_prob_hist(X->d_prob.p, N, X->d_is_terminal.p, X->d_knode_locus.p, X->d_accum.p + 2ull * N, X->d_hist.p, st);
    bool any_present = false;
    for (uint32_t l = 0; l < P; ++l) any_present = any_present || locus_reads[l] > 0;
    // the threshold (valley of the 200-bin histogram) is found on the device too: the ML-path kernel reads it from
    // device memory and starts without a host round trip; the host picks the value up later
    launch_prob_thresh(X->d_hist.p, any_present, X->fit.thresh, X->d_thresh_f64.p, X->d_thresh_i32.p, st);
    X->h_thresh.resize(1);
    CK(cudaMemcpyAsync(X->h_thresh.data(), X->d_thresh_i32.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(X->ev_acc[2].get(), st));
    MP.thresh = (double)X->fit.thresh;  // placeholder for kernels that do not read it (S8); S7 uses d_thresh_f64
    lap(1);
    // ---- S7 on the device: the ML-path kernel is a latency chain per locus (~0.4 ms).  It only decides which loci
    // are reported and whether the path spells alleles the site tables lack (rare), so it runs on its own stream
    // while S8 (per-allele statistics + likelihoods) and the VCF text are produced SPECULATIVELY for the common
    // outcome "every locus with reads is present, no extra records"; the outcome is verified afterwards and
    // anything that deviates is redone on the slow path.
    if (!X->ev_ml[0])
        for (auto& e : X->ev_ml) e = new_event(cudaEventDefault);
    X->h_path.resize(N);
    X->h_plen.resize(P);
    X->h_done.resize(P);
    std::fill(X->h_done.begin(), X->h_done.end(), 0u);
    CK(cudaStreamWaitEvent(X->st_ml.get(), X->ev_acc[2].get(), 0));  // node scores and threshold are produced on `st`
    CK(cudaMemsetAsync(X->d_path.p, 0, (size_t)N * 4, X->st_ml.get()));  // absent loci leave their slice unwritten
    CK(cudaEventRecord(X->ev_ml[0].get(), X->st_ml.get()));
    // The level-parallel kernel writes every locus's path straight into pinned host memory (UVA: the same pointers
    // are valid on the device) and raises a per-locus flag, so the host can verify the small loci while the big ones
    // are still running; the generic kernel leaves the paths in device memory and they are copied back as a whole.
    const bool ml_streamed = launch_mlpath(
        P, X->d_knode_base.p, X->d_edge_off.p, X->d_edges.p, X->d_prob.p, X->d_accum.p + 2ull * N, MP, X->d_M.p, X->d_len.p, X->d_up.p, N,
        X->d_path.p, X->d_path_len.p, X->max_locus_knodes, X->max_locus_edges, X->d_needs_mean.p, X->st_ml.get(),
        X->d_locus_level_off.p, X->d_level_start.p, X->d_level_nodes.p, X->d_level_singles.p,
        X->h_path.data(), X->h_plen.data(), X->h_done.data(), X->d_thresh_f64.p);
    X->ml_in_flight = true;
    CK(cudaEventRecord(X->ev_ml[1].get(), X->st_ml.get()));
    CK(cudaGetLastError());
    if (!ml_streamed) {
        CK(cudaMemcpyAsync(X->h_path.data(), X->d_path.p, (size_t)N * 4, cudaMemcpyDeviceToHost, X->st_ml.get()));
        CK(cudaMemcpyAsync(X->h_plen.data(), X->d_path_len.p, (size_t)P * 4, cudaMemcpyDeviceToHost, X->st_ml.get()));
    }
    // ---- reference paths / site tables (read independent, cached per --vcf-refs file, loaded above)
    auto ensure_sites = [&](uint32_t l) {
        auto& S = X->sites[l];
        if (S.ready) return;
        const Locus& L = H.loci[l];
        auto it = X->refs.find(L.name);
        if (it != X->refs.end()) S.ref_path = thread_sequence(L, it->second);
        if (S.ref_path.empty()) S.ref_path = top_path(L);
        S.biallelic = enumerate_sites(H, l, S.ref_path);
        for (auto& r : S.biallelic) S.known.insert(std::make_tuple(r.pos, r.ref, r.alts[0]));
        S.merged = merge_records(L, S.ref_path, S.biallelic);
        S.ready = true;
    };
    const std::string sample_name = sample && *sample ? sample : "sample";
    GenotypeArrays& G = X->GA;
    // S8 + text for a given record list (uses the cached device CSR while the list is the cached one)
    auto run_s8_and_format = [&](cudaStream_t s8) {
        const double ts0 = now_ms();
        if (X->records != X->csr_records || G.rec_off.empty() || !X->sample_records.empty()) {
            G.rec_off.assign(1, 0);
            G.allele_off.assign(1, 0);
            G.allele_kn.clear();
            for (const SiteRecord* r : X->records) {
                for (auto& kn : r->allele_kn) {
                    for (uint32_t x : kn) G.allele_kn.push_back(H.knode_base[r->locus] + x);
                    G.allele_off.push_back((uint32_t)G.allele_kn.size());
                }
                G.rec_off.push_back((uint32_t)G.allele_off.size() - 1);
            }
            CK(cudaStreamSynchronize(s8));
            X->d_rec_off.assign(G.rec_off);
            X->d_allele_off.assign(G.allele_off);
            X->d_allele_kn.assign(G.allele_kn);
            {   // the static columns of every record line and the slots of the sample columns (VCF text on the device)
                std::vector<char> prefix;
                std::vector<uint32_t> poff(1, 0), soff(1, 0);
                for (size_t i = 0; i < X->records.size(); ++i) {
                    const std::string& t = vcf_record_prefix(H, *X->records[i]);
                    prefix.insert(prefix.end(), t.begin(), t.end());
                    poff.push_back((uint32_t)prefix.size());
                    soff.push_back(soff.back() + (uint32_t)vcf_sample_column_bound(G.rec_off[i + 1] - G.rec_off[i]));
                }
                X->d_vcf_prefix.assign(prefix);
                X->d_vcf_prefix_off.assign(poff);
                X->d_vcf_slot_off.assign(soff);
                X->vcf_prefix_bytes = prefix.size();
                X->vcf_slot_bytes = soff.back();
                X->d_vcf_ctl.reserve(2, 2);
            }
            X->csr_records = X->sample_records.empty() ? X->records : std::vector<const SiteRecord*>();
        }
        const uint32_t nr = (uint32_t)X->records.size(), na = (uint32_t)G.allele_off.size() - 1;
        format_vcf_header(X->contigs, sample_name, X->vcf_header);
        // the header is padded in front so that the record lines start 16-byte aligned (the device writes them with
        // 128-bit stores); the text handed out begins at vcf_begin
        const size_t hl_raw = X->vcf_header.size(), pad = (16 - hl_raw % 16) % 16, hl = hl_raw + pad;
        X->h_vcf.resize(hl + X->vcf_prefix_bytes + X->vcf_slot_bytes + 32);
        X->vcf_begin = pad;
        memcpy(X->h_vcf.data() + pad, X->vcf_header.data(), hl_raw);
        X->h_vcf_ctl.resize(2);
        X->h_vcf_ctl.data()[0] = X->h_vcf_ctl.data()[1] = 0;
        if (nr) {
            X->d_gt_u32.ensure((size_t)na * 6);
            X->d_gt_f64.ensure((size_t)na * 2 + nr);
            X->d_gt_i32.ensure((size_t)nr * 3);
            X->d_gt_f32.ensure((size_t)nr * 2 + na);
            uint32_t* u = X->d_gt_u32.p;
            double* f = X->d_gt_f64.p;
            DevGenotype DG{nr, na, X->d_rec_off.p, X->d_allele_off.p, X->d_allele_kn.p, u, u + na, u + 2 * (size_t)na, u + 3 * (size_t)na,
                           u + 4 * (size_t)na, u + 5 * (size_t)na, f, f + na, f + 2 * (size_t)na, X->d_gt_i32.p};
            // the statistics drprg's filters derive from the record come out of the same kernel (they stay on the device
            // until drprg_cuda_gt_filter_stats asks for them)
            DG.covg_gt = X->d_gt_i32.p + nr;
            DG.minor_gt = X->d_gt_i32.p + 2 * (size_t)nr;
            DG.frs = X->d_gt_f32.p;
            DG.sb_ratio = X->d_gt_f32.p + nr;
            DG.pdp = X->d_gt_f32.p + 2 * (size_t)nr;
            launch_genotype(X->d_accum.p, DG, MP, s8);
            // the record lines: formatted by the device into the host-mapped text buffer, right behind the header
            X->d_vcf_slots.ensure(X->vcf_slot_bytes + 1);
            X->d_vcf_line_len.ensure(nr);
            X->d_vcf_out_off.ensure((size_t)nr + 1);
            CK(cudaMemsetAsync(X->d_vcf_ctl.p, 0, 2 * sizeof(uint32_t), s8));
            DevVcfText VT{X->d_vcf_prefix.p, X->d_vcf_prefix_off.p, X->d_vcf_slot_off.p, X->d_vcf_slots.p, X->d_vcf_line_len.p,
                          X->d_vcf_out_off.p, X->h_vcf.data() + hl, (uint32_t)(X->vcf_prefix_bytes + X->vcf_slot_bytes), X->d_vcf_ctl.p,
                          X->d_vcf_ctl.p + 1};
            static const bool host_text = getenv("DRPRG_VCF_TEXT") && std::string(getenv("DRPRG_VCF_TEXT")) == "host";
            if (!host_text) launch_vcf_text(DG, VT, s8);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(X->h_vcf_ctl.data(), X->d_vcf_ctl.p, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s8));
            // the arrays themselves (getters, drprg_cuda_gt_*): downloaded into pinned buffers, unpacked on first use
            X->h_u32.resize((size_t)na * 6);
            X->h_f64.resize((size_t)na * 2 + nr);
            CK(cudaMemcpyAsync(X->h_u32.data(), u, X->h_u32.size() * 4, cudaMemcpyDeviceToHost, s8));
            CK(cudaMemcpyAsync(X->h_f64.data(), f, X->h_f64.size() * 8, cudaMemcpyDeviceToHost, s8));
            X->h_gt.resize(nr);
            CK(cudaMemcpyAsync(X->h_gt.data(), X->d_gt_i32.p, (size_t)nr * 4, cudaMemcpyDeviceToHost, s8));
            CK(cudaStreamSynchronize(s8));
            X->ga_stale = true;
            if (host_text) X->h_vcf_ctl.data()[1] = 1u;
        } else {
            X->ga_stale = true;
        }
        const double tf0 = now_ms();
        if (X->h_vcf_ctl.data()[1]) {
            // a value the device formatter refuses (exponent notation, a rounding tie, -0, inf / nan) — or DRPRG_VCF_TEXT=host:
            // the host formatter writes the whole text
            ensure_ga(X);
            format_vcf(H, X->records, G, X->contigs, sample_name, X->vcf_fallback);
            X->h_vcf.resize(X->vcf_fallback.size() + 1);
            memcpy(X->h_vcf.data(), X->vcf_fallback.data(), X->vcf_fallback.size());
            X->vcf_begin = 0;
            X->vcf_len = X->vcf_fallback.size();
        } else {
            X->vcf_len = hl_raw + X->h_vcf_ctl.data()[0];
        }
        X->h_vcf.data()[X->vcf_begin + X->vcf_len] = 0;
        static const bool timing = getenv("DRPRG_TIMING") != nullptr;
        if (timing) fprintf(stderr, "[drprg-cuda] s8 + vcf text kernels + downloads %.3f ms, host text (fallback only) %.3f ms\n", tf0 - ts0, now_ms() - tf0);
    };
    // ---- speculative pass: every locus with reads present, cached merged site tables
    {
        std::vector<uint32_t> todo;
        for (uint32_t l = 0; l < P; ++l)
            if (locus_reads[l] > 0 && !X->sites[l].ready) todo.push_back(l);
        parallel_for(todo.size(), [&](size_t i) { ensure_sites(todo[i]); });
    }
    X->records.clear();
    X->sample_records.clear();
    X->contigs.clear();
    for (uint32_t l : X->loci_by_name) {  // name order == VCF record order
        if (locus_reads[l] <= 0) continue;
        X->contigs.push_back(H.loci[l].name);
        for (auto& r : X->sites[l].merged) X->records.push_back(&r);
    }
    lap(2);
    run_s8_and_format(X->st_gt.get());
    CK(cudaEventSynchronize(X->ev_acc[2].get()));  // long done: the threshold the device chose
    X->fit.thresh = X->h_thresh.data()[0];
    MP.thresh = (double)X->fit.thresh;
    lap(3);
    // ---- verify the speculation against the ML paths
    const double tw0 = now_ms();
    if (!ml_streamed) CK(cudaStreamSynchronize(X->st_ml.get()));
    CK(cudaEventSynchronize(X->ev_acc[1].get()));  // the full accumulator is on the host from here on
    const double tw1 = now_ms();
    const uint32_t* path = X->h_path.data();
    const uint32_t* plen = X->h_plen.data();
    const volatile uint32_t* done = X->h_done.data();
    std::atomic<bool> ml_failed{false};
    auto wait_for_locus = [&](uint32_t l) {  // streamed mode: spin until the kernel has published locus l
        if (!ml_streamed) return true;
        for (uint64_t spin = 0; done[l] == 0u; ++spin) {
            if (ml_failed.load(std::memory_order_relaxed)) return false;
            if ((spin & 0xffffu) == 0xffffu && cudaStreamQuery(X->st_ml.get()) != cudaErrorNotReady && done[l] == 0u) {
                ml_failed = true;  // the stream ended (or failed) without publishing: never spin forever
                return false;
            }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        return true;
    };
    X->mlpaths.assign(P, {});
    X->present.assign(P, 0);
    struct LocusOut {
        bool present = false;
        std::vector<uint32_t> kp;
        std::vector<SiteRecord> sample_merged;  // only when the ML path adds records
        bool use_cached = true;
    };
    std::vector<LocusOut> lout(P);
    parallel_for(P, [&](size_t li) {
        // the pool hands loci out in order: biggest first when all paths are already there; smallest first when they are
        // streamed (small loci finish first, and only the biggest one's check is left when the kernel ends)
        const uint32_t l = ml_streamed ? X->loci_by_size[P - 1 - li] : X->loci_by_size[li];
        if (locus_reads[l] <= 0 || !wait_for_locus(l) || plen[l] == 0xffffffffu || plen[l] == 0) return;
        const Locus& L = H.loci[l];
        LocusOut& O = lout[l];
        static const bool vt = getenv("DRPRG_TIMING_VERIFY") != nullptr;
        const double v0 = vt ? now_ms() : 0;
        O.kp.assign(path + H.knode_base[l], path + H.knode_base[l] + plen[l]);
        std::vector<uint32_t> lp = local_path_of(L, O.kp);
        const double v1 = vt ? now_ms() : 0;
        if (locus_coverage_outlier(H, l, O.kp, lp, cov, X->fit.covg)) return;
        const double v2 = vt ? now_ms() : 0;
        O.present = true;
        auto& S = X->sites[l];
        std::vector<SiteRecord> extra;
        find_ml_path_records(H, l, S.ref_path, lp, S.known, extra);
        if (vt && l == X->loci_by_size[0])
            fprintf(stderr, "[drprg-cuda] verify of the largest locus (%u k-mer nodes on the path): local path %.1f us, outlier %.1f us, records %.1f us; published at %.3f ms after tw1\n",
                    plen[l], (v1 - v0) * 1e3, (v2 - v1) * 1e3, (now_ms() - v2) * 1e3, v0 - tw1);
        if (!extra.empty()) {  // the ML path spells alleles the site table lacks: merge them in for this sample only
            std::vector<SiteRecord> all = S.biallelic;
            for (auto& r : extra) all.push_back(std::move(r));
            O.sample_merged = merge_records(L, S.ref_path, std::move(all));
            O.use_cached = false;
        }
    }, 16);
    {
        const cudaError_t mle = cudaStreamSynchronize(X->st_ml.get());
        X->ml_in_flight = false;
        if (mle != cudaSuccess)
            throw std::runtime_error(std::string("ML-path kernel failed: ") + cudaGetErrorString(mle));
    }
    if (ml_failed.load()) throw std::runtime_error("the ML-path kernel ended without publishing every locus");
    {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, X->ev_ml[0].get(), X->ev_ml[1].get()));
        X->gt_ms[6] = ms;  // device time of the ML-path kernel (overlapped with S8 + VCF text on the host)
    }
    bool speculation_ok = true;
    for (uint32_t l = 0; l < P; ++l) {
        if (lout[l].present) {
            X->present[l] = 1;
            X->mlpaths[l] = std::move(lout[l].kp);
        }
        if ((locus_reads[l] > 0) != lout[l].present || !lout[l].use_cached) speculation_ok = false;
    }
    {
        static const bool timing = getenv("DRPRG_TIMING") != nullptr;
        if (timing) fprintf(stderr, "[drprg-cuda] ml wait %.3f ms, verify %.3f ms\n", tw1 - tw0, now_ms() - tw1);
    }
    lap(4);
    if (!speculation_ok) {  // slow path: rebuild the record list exactly and redo S8 + text
        X->records.clear();
        X->contigs.clear();
        for (uint32_t l : X->loci_by_name) {
            LocusOut& O = lout[l];
            if (!O.present) continue;
            X->contigs.push_back(H.loci[l].name);
            if (O.use_cached) {
                for (auto& r : X->sites[l].merged) X->records.push_back(&r);
            } else {
                X->sample_records.push_back(std::move(O.sample_merged));
                for (auto& r : X->sample_records.back()) X->records.push_back(&r);
            }
        }
        run_s8_and_format(X->st_gt.get());
    }
    lap(5);
    X->have_gt = true;
}

// long reads: cut every read into segments of 40*w k-mer positions so that the thread-per-item kernels get evenly
// sized work (a 10 kb read becomes ~23 items instead of one warp-long loop)
void build_segments(drprg_index* X, drprg_batch* B, const uint32_t* lens, uint64_t n, uint64_t total_bases, cudaStream_t cs) {
    const uint32_t w = X->H.w, k = X->H.k, seg_len = 40 * w;
    std::vector<uint32_t> sr, ss;
    sr.reserve(total_bases / seg_len + n);
    ss.reserve(total_bases / seg_len + n);
    for (uint64_t r = 0; r < n; ++r) {
        const uint32_t len = lens[r];
        if (len + 1 < w + k) continue;
        const uint32_t nk = len - k + 1;
        for (uint32_t s0 = 0; s0 < nk; s0 += seg_len) {
            sr.push_back((uint32_t)r);
            ss.push_back(s0);
        }
    }
    if (sr.empty()) return;
    const size_t bytes = sr.size() * 4;
    B->d_seg_read = pool_get<uint32_t>(bytes, X->device);
    B->d_seg_start = pool_get<uint32_t>(bytes, X->device);
    CK(cudaMemcpyAsync(B->d_seg_read.get(), sr.data(), bytes, cudaMemcpyHostToDevice, cs));
    CK(cudaMemcpyAsync(B->d_seg_start.get(), ss.data(), bytes, cudaMemcpyHostToDevice, cs));
    CK(cudaStreamSynchronize(cs));  // the staging vectors die with this scope
    B->R.seg_read = B->d_seg_read.get();
    B->R.seg_start = B->d_seg_start.get();
    B->R.n_segs = sr.size();
    B->R.seg_len = seg_len;
}

std::unique_ptr<drprg_batch> upload_batch(drprg_index* X, const uint32_t* words, const uint64_t* word_off, uint32_t stride,
                                          const uint32_t* lens, uint64_t n, uint64_t total_bases, uint32_t id_base, cudaStream_t st) {
    need_device(X);
    CK(cudaSetDevice(X->device));
    std::unique_ptr<drprg_batch> B(new drprg_batch());
    const uint64_t nwords = stride ? n * (uint64_t)stride : (n ? word_off[n] : 0);
    B->d_words = pool_get<uint32_t>(std::max<uint64_t>(1, nwords + 2) * 4, X->device);
    B->d_lens = pool_get<uint32_t>(std::max<uint64_t>(1, n) * 4, X->device);
    if (!stride) B->d_off = pool_get<uint64_t>((n + 1) * 8, X->device);
    const bool chunked = (st == nullptr) && nwords * 4 >= (8u << 20) && stride && stride * 16u <= SHORT_READ_MAX;
    cudaStream_t cs = st;
    if (chunked) {
        if (!X->st_copy) X->st_copy = new_stream();
        cs = X->st_copy.get();
        B->n_chunks = 4;
    }
    if (!stride) CK(cudaMemcpyAsync(B->d_off.get(), word_off, (n + 1) * 8, cudaMemcpyHostToDevice, cs));
    uint32_t ml = 0;
    for (int c = 0; c < B->n_chunks; ++c) {
        const uint64_t lo = n * (uint64_t)c / B->n_chunks, hi = n * (uint64_t)(c + 1) / B->n_chunks;
        B->chunk_lo[c] = lo;
        B->chunk_lo[c + 1] = hi;
        const uint64_t w0 = stride ? lo * stride : word_off[lo], w1 = stride ? hi * stride : word_off[hi];
        if (w1 > w0) CK(cudaMemcpyAsync(B->d_words.get() + w0, words + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, cs));
        if (hi > lo) CK(cudaMemcpyAsync(B->d_lens.get() + lo, lens + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, cs));
        if (chunked) {
            B->ev[c] = new_event(cudaEventDisableTiming);
            CK(cudaEventRecord(B->ev[c].get(), cs));
        }
        // the longest read only selects the kernel: a fixed stride that already bounds it needs no scan
        if (!(stride && stride * 16u <= SHORT_READ_MAX))
            for (uint64_t i = lo; i < hi; ++i) ml = std::max(ml, lens[i]);  // overlaps the copy just enqueued
    }
    if (stride && stride * 16u <= SHORT_READ_MAX) ml = stride * 16u;
    B->R = DevReads{B->d_words.get(), B->d_off.get(), stride, B->d_lens.get(), n, id_base};
    B->total_bases = total_bases;
    B->max_len = ml;
    if (ml > SHORT_READ_MAX) build_segments(X, B.get(), lens, n, total_bases, cs);
    return B;
}

// ============================================================================================
// Read-sharded multi-GPU handle (SURVEY 8e): the index is replicated, a batch is cut into one contiguous shard of reads
// per GPU, every GPU runs S1-S5 on its shard — one host thread per GPU issues the launches side by side — and the
// coverage merge kernel of every non-root GPU adds straight into the ROOT GPU's accumulator over NVLink (peer-mapped
// memory, red.global.add): there is no separate collective.  The root then runs S6-S8.
// ============================================================================================
bool is_multi(const drprg_index* X) { return X->gpus.size() > 1; }

void for_each_gpu(drprg_index* root, const std::function<void(size_t, drprg_index*)>& fn) {
    const size_t G = root->gpus.size();
    for (size_t g = 1; g < G; ++g) {
        drprg_index* X = root->gpus[g];
        root->workers[g - 1]->submit([&fn, g, X] {
            CK(cudaSetDevice(X->device));
            fn(g, X);
        });
    }
    std::string err;
    try {
        CK(cudaSetDevice(root->device));
        fn(0, root);
    } catch (const std::exception& e) {
        err = e.what();
    }
    for (size_t g = 1; g < G; ++g) {
        try {
            root->workers[g - 1]->wait();
        } catch (const std::exception& e) {
            if (err.empty()) err = e.what();
        }
    }
    CK(cudaSetDevice(root->device));
    if (!err.empty()) throw std::runtime_error(err);
}

int load_multi(const std::string& text, uint32_t w, uint32_t k, int n_gpus, const int* devices, drprg_index** out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw std::runtime_error("no CUDA device visible: drprg-cuda has no CPU fallback");
    const int G = n_gpus <= 0 ? ndev : n_gpus;
    if (G > ndev && !devices) throw std::runtime_error("more GPUs requested than are visible");
    if (G > 64) throw std::runtime_error("more than 64 shards");
    std::vector<int> devs(G);
    for (int i = 0; i < G; ++i) devs[i] = devices ? devices[i] : i;
    // an explicit list may name a device more than once: its shards then share that GPU (how a one-GPU box exercises
    // the sharded path); n_gpus alone always means distinct devices
    for (int i = 0; i < G; ++i)
        if (devs[i] < 0 || devs[i] >= ndev) throw std::runtime_error("bad device ordinal");
    drprg_index* raw = nullptr;
    load_common(text, w, k, devs[0], &raw);
    std::unique_ptr<drprg_index> root(raw);
    if (G == 1) {
        *out = root.release();
        return 0;
    }
    for (int i = 1; i < G; ++i) {
        if (devs[i] != devs[0]) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, devs[i], devs[0]));
            if (!can) throw std::runtime_error("GPU " + std::to_string(devs[i]) + " cannot reach GPU " + std::to_string(devs[0]) + " over NVLink/PCIe peer access");
        }
        std::unique_ptr<drprg_index> R(new drprg_index());
        R->device = devs[i];
        CK(cudaSetDevice(devs[i]));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, devs[i]));
        R->sm_count = prop.multiProcessorCount;
        R->H = root->H;  // the host index is built once
        upload_index(R.get());
        if (devs[i] != devs[0]) {
            const cudaError_t pe = cudaDeviceEnablePeerAccess(devs[0], 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CK(pe);
            cudaGetLastError();
        }
        R->reduce_dst = root->d_accum.p;  // UVA: the root's pointer is valid on the peer once access is enabled
        root->replicas.push_back(std::move(R));
        root->workers.emplace_back(new GpuWorker());
    }
    CK(cudaSetDevice(devs[0]));
    root->accum_shared = true;
    root->gpus.push_back(root.get());
    for (auto& r : root->replicas) root->gpus.push_back(r.get());
    *out = root.release();
    return 0;
}

void multi_sample_begin(drprg_index* root, const drprg_map_opts* o, uint32_t first_read_len) {
    // the root zeroes its accumulator first: the other GPUs only touch it in map_batch, which the host starts afterwards
    for_each_gpu(root, [&](size_t, drprg_index* X) {
        sample_begin(X, o, first_read_len);
        CK(cudaStreamSynchronize(0));
    });
}

std::unique_ptr<drprg_batch> multi_upload(drprg_index* root, const uint32_t* words, const uint64_t* word_off, uint32_t stride,
                                          const uint32_t* lens, uint64_t n, uint64_t total_bases, uint32_t id_base) {
    const size_t G = root->gpus.size();
    std::unique_ptr<drprg_batch> B(new drprg_batch());
    B->shards.resize(G);
    B->R.n_reads = n;
    B->R.read_id_base = id_base;
    B->total_bases = total_bases;
    for_each_gpu(root, [&](size_t g, drprg_index* X) {
        const uint64_t lo = n * g / G, hi = n * (g + 1) / G;  // rank r maps reads [rN/G, (r+1)N/G)
        uint64_t bases = 0;
        for (uint64_t i = lo; i < hi; ++i) bases += lens[i];
        if (stride) {
            // dropped reads (lens == 0) still occupy bases in total_bases bookkeeping of the single-GPU path: keep the caller's
            // total on the last shard so that the sum over shards equals total_bases
            B->shards[g] = upload_batch(X, words + lo * stride, nullptr, stride, lens + lo, hi - lo, bases, id_base + (uint32_t)lo, 0);
        } else {
            std::vector<uint64_t> off(hi - lo + 1);
            for (uint64_t i = lo; i <= hi; ++i) off[i - lo] = word_off[i] - word_off[lo];
            B->shards[g] = upload_batch(X, words + word_off[lo], off.data(), 0, lens + lo, hi - lo, bases, id_base + (uint32_t)lo, 0);
            CK(cudaStreamSynchronize(0));  // `off` dies with this scope
        }
    });
    // total_bases counts the bases of dropped reads too (their lens are 0): the difference goes to the last shard
    uint64_t sum = 0;
    for (auto& sh : B->shards) sum += sh->total_bases;
    if (total_bases > sum) B->shards[G - 1]->total_bases += total_bases - sum;
    return B;
}

void multi_map_batch(drprg_index* root, drprg_batch* B, uint64_t* n_hits, uint64_t* n_kept) {
    const size_t G = root->gpus.size();
    if (B->shards.size() != G) throw std::runtime_error("the batch was not uploaded through this multi-GPU handle");
    std::vector<uint64_t> nh(G, 0), nk(G, 0);
    for_each_gpu(root, [&](size_t g, drprg_index* X) { map_batch(X, B->shards[g].get(), 0, &nh[g], &nk[g]); });
    // every GPU's stream has been synchronised: all remote adds have landed in the root's accumulator
    uint64_t bases = 0, reads = 0, h = 0, kpt = 0;
    for (size_t g = 0; g < G; ++g) {
        bases += root->gpus[g]->own_bases;
        reads += root->gpus[g]->own_reads;
        h += nh[g];
        kpt += nk[g];
    }
    root->total_bases = bases;
    root->n_reads = reads;
    root->scalars_in_buffer = false;
    root->hist_on_host = false;
    if (n_hits) *n_hits = h;
    if (n_kept) *n_kept = kpt;
}

void sample_begin_any(drprg_index* X, const drprg_map_opts* o, uint32_t first_read_len) {
    if (is_multi(X)) multi_sample_begin(X, o, first_read_len);
    else sample_begin(X, o, first_read_len);
}
void map_batch_any(drprg_index* X, drprg_batch* B, cudaStream_t st, uint64_t* n_hits, uint64_t* n_kept) {
    if (is_multi(X)) multi_map_batch(X, B, n_hits, n_kept);
    else map_batch(X, B, st, n_hits, n_kept);
}

// A reads file as a device-resident batch.  Strict 4-line FASTQ (plain or gzip) is framed on the host and packed on the
// device (ingest.cu); FASTA and anything unusual goes through the host parser and an upload.  DRPRG_HOST_INGEST=1 forces
// the host parser (tests compare the two).
struct FileBatch {
    std::unique_ptr<drprg_batch> B;
    uint64_t n_dropped = 0;
    uint32_t first_read_len = 0;
    bool on_device = false;  // packed on the device (else: host parser)
};
bool host_ingest_forced() {
    static const bool on = getenv("DRPRG_HOST_INGEST") != nullptr && atoi(getenv("DRPRG_HOST_INGEST")) != 0;
    return on;
}
struct Inflated {  // a gzip reads file inflated into host memory (ahead of time in batch mode)
    std::unique_ptr<char, void (*)(void*)> p{nullptr, free};
    size_t n = 0;
    std::string error;
    void inflate(const std::string& path) {
        char* q = nullptr;
        inflate_file(path, &q, &n);
        p.reset(q);
    }
};

// The whole text of a reads file for the framer: a gzip file is inflated into host memory on all host threads
// (gzip_inflate.cpp) unless the batch driver has done that already (`pre`); a plain file is read in place with pread.
struct ReadsText {
    TextSource src;
    Inflated local;
    ReadsText(const char* path, const Inflated* pre) {
        if (!pre && file_is_gzip(path)) {
            local.inflate(path);
            pre = &local;
        }
        if (pre) {
            src.mem = pre->p.get();
            src.size = pre->n;
            return;
        }
        src.fd = open(path, O_RDONLY);
        if (src.fd < 0) throw std::runtime_error(std::string("cannot open ") + path);
        src.size = (size_t)lseek(src.fd, 0, SEEK_END);
    }
    ReadsText(const ReadsText&) = delete;
    ReadsText& operator=(const ReadsText&) = delete;
    ~ReadsText() {
        if (src.fd >= 0) close(src.fd);
    }
    // FASTA, leading blank lines and files too small for one record go to the host parser without being framed
    bool may_be_fastq() const {
        char first = 0;
        return src.size >= 8 && src.read(&first, 0, 1) == 1 && first == '@';
    }
};

// the packed reads an ingest left on the device, as a batch of this index: takes over the buffers of I
std::unique_ptr<drprg_batch> batch_from_ingest(drprg_index* X, IngestResult& I, uint32_t read_id_base) {
    std::unique_ptr<drprg_batch> B(new drprg_batch());
    B->d_words = std::move(I.words);
    B->d_lens = std::move(I.lens);
    B->d_off = std::move(I.word_off);
    B->R = DevReads{B->d_words.get(), B->d_off.get(), I.stride_words, B->d_lens.get(), I.n_reads, read_id_base};
    B->total_bases = I.total_bases;
    B->max_len = I.stride_words ? I.stride_words * 16u : I.max_len;
    if (I.max_len > SHORT_READ_MAX) {  // the segment table is built from the lengths on the host
        std::vector<uint32_t> lens(I.n_reads);
        CK(cudaMemcpy(lens.data(), B->d_lens.get(), I.n_reads * 4, cudaMemcpyDeviceToHost));
        build_segments(X, B.get(), lens.data(), I.n_reads, I.total_bases, 0);
    }
    return B;
}

// the host parser's batch; a multi-GPU handle gets one shard of the reads per GPU
FileBatch host_parsed_batch(drprg_index* X, const char* reads_path, uint32_t threads) {
    need_device(X);
    CK(cudaSetDevice(X->device));
    PackedReads pr;
    load_reads_packed(reads_path, threads, pr);
    const uint64_t n = pr.lens.size();
    if (n > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
    FileBatch F;
    if (is_multi(X)) {
        F.B = multi_upload(X, pr.words.data(), pr.word_off.data(), 0, pr.lens.data(), n, pr.total_bases, 0);
    } else {
        F.B = upload_batch(X, pr.words.data(), pr.word_off.data(), 0, pr.lens.data(), n, pr.total_bases, 0, 0);
        CK(cudaStreamSynchronize(0));  // pr dies with this scope
    }
    F.n_dropped = pr.n_dropped;
    F.first_read_len = pr.first_read_len;
    return F;
}

FileBatch batch_from_file(drprg_index* X, const char* reads_path, uint32_t threads) {
    need_device(X);
    if (!is_multi(X) && !host_ingest_forced()) {
        CK(cudaSetDevice(X->device));
        const ReadsText T(reads_path, nullptr);
        IngestResult I;
        if (T.may_be_fastq() && ingest_fastq_text(T.src, X->device, threads, I, 0)) {
            FileBatch F;
            F.B = batch_from_ingest(X, I, 0);
            F.n_dropped = I.n_dropped;
            F.first_read_len = I.first_read_len;
            F.on_device = true;
            return F;
        }
    }
    return host_parsed_batch(X, reads_path, threads);
}

// A reads file of any size, mapped wave by wave: plain strict FASTQ (or a gzip file inflated into host memory) is cut at
// record starts into waves of ~1 GiB of text; every wave is framed on the host, uploaded (sequence lines only), packed and
// mapped into the sample's accumulators before the next one is read, so a 30 M-read file (9.4 GB of text, BASELINE
// config 3) needs 0.5 GiB of pinned and 1 GiB of device memory instead of the whole text, and files beyond the 8 GB limit
// of one ingest still take the fast path.  false = the host parser must handle the file; a sample that was begun here is
// begun again there.
struct WaveTotals {
    uint64_t n = 0, dropped = 0, bases = 0, hits = 0, kept = 0;
    uint32_t first_len = 0;
    size_t waves = 0;
    double ms_ingest = 0, ms_map = 0;
};
bool map_file_in_waves(drprg_index* X, const char* reads_path, const drprg_map_opts* o, const Inflated* pre, WaveTotals& W) {
    if (host_ingest_forced()) return false;
    // A multi-GPU handle maps the file on its root GPU: a file-fed sample is bound by the host's framing rate (~45 GB/s of
    // text on 16 cores against 1.9 ms of GPU time per 10 M reads), so sharding the waves would leave every GPU idle
    // anyway; read sharding pays for batches that are already packed (drprg_cuda_batch_upload).
    static const size_t wave_bytes = [] {
        const char* e = getenv("DRPRG_WAVE_BYTES");
        return e && atol(e) > 0 ? (size_t)atol(e) : (size_t)(1u << 30);
    }();
    const ReadsText T(reads_path, pre);
    if (!T.may_be_fastq()) return false;
    const TextSource& F = T.src;
    const uint32_t threads = o ? std::max(1u, o->threads) : 1u;
    std::vector<char> scratch;
    size_t lo = 0;
    while (lo < F.size) {
        size_t hi = F.size - lo <= wave_bytes + wave_bytes / 4 ? F.size : F.boundary(lo + wave_bytes, scratch);
        if (hi == SIZE_MAX) throw std::runtime_error(std::string("read error in ") + reads_path);
        if (hi <= lo) hi = F.size;
        TextSource S;
        S.fd = F.fd;
        S.mem = F.mem ? F.mem + lo : nullptr;
        S.size = hi - lo;
        S.origin = lo;
        IngestResult I;
        const double tw0 = now_ms();
        if (!ingest_fastq_text(S, X->device, threads, I, 0)) return false;
        if (W.n + I.n_reads > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
        const std::unique_ptr<drprg_batch> B = batch_from_ingest(X, I, (uint32_t)W.n);
        if (W.waves == 0) {
            W.first_len = I.first_read_len;
            sample_begin_any(X, o, I.first_read_len);
        }
        uint64_t nh = 0, nk = 0;
        const double tw1 = now_ms();
        map_batch(X, B.get(), 0, &nh, &nk);
        W.ms_ingest += tw1 - tw0;
        W.ms_map += now_ms() - tw1;
        W.n += I.n_reads;
        W.dropped += I.n_dropped;
        W.bases += I.total_bases;
        W.hits += nh;
        W.kept += nk;
        ++W.waves;
        lo = hi;
    }
    return W.waves > 0;
}

// discover's candidate regions and the reads over them: the per-locus half on the host (discover.cpp), the reads on every
// GPU from its retained-hit store (region_reads_kernel), sorted by (region, read) here
void find_candidates(drprg_index* X, const DiscoverOpts& o) {
    std::vector<uint32_t> cons_start;
    discover_regions(X->H, X->present, X->mlpaths, X->h_acc.data(), o, X->discover, cons_start);
    DiscoverResult& D = X->discover;
    X->discover_ready = true;
    X->asm_status.clear();
    X->asm_paths.clear();
    X->asm_bases.clear();
    const size_t nR = D.regions.size();
    if (nR >= 0xffffffffull) throw std::runtime_error("more than 2^32 candidate regions");
    const uint32_t P = (uint32_t)X->H.loci.size();
    std::vector<uint32_t> region_off(P + 1, 0);
    std::vector<uint2> pad(nR);
    for (size_t r = 0; r < nR; ++r) {
        ++region_off[D.regions[r].locus + 1];
        pad[r] = make_uint2(D.regions[r].pad_start, D.regions[r].pad_end);
    }
    for (uint32_t l = 0; l < P; ++l) region_off[l + 1] += region_off[l];
    const std::vector<drprg_index*> gpus = X->gpus.empty() ? std::vector<drprg_index*>{X} : X->gpus;
    std::vector<std::vector<RegionRead>> found(gpus.size());
    auto run = [&](size_t g, drprg_index* G) {
        if (!nR || !G->rt_rows) return;
        Stream st = new_stream();
        DBuf<uint32_t> d_cons_start, d_region_off;
        DBuf<uint2> d_pad;
        DBuf<RegionRead> d_out;
        DBuf<unsigned long long> d_cursor;
        d_cons_start.assign(cons_start);
        d_region_off.assign(region_off);
        d_pad.assign(pad);
        d_cursor.ensure(1);
        d_out.ensure(std::max<uint64_t>(1024, G->rt_rows / 8));
        unsigned long long n = 0;
        for (;;) {  // the entries wanted are counted past the capacity: regrow once to the exact need
            CK(cudaMemsetAsync(d_cursor.p, 0, sizeof(unsigned long long), st.get()));
            launch_region_reads(retain_store(G), (uint32_t)G->rt_rows, G->d_knode_base.p, d_cons_start.p, d_region_off.p, P, d_pad.p,
                                G->H.k, o.min_hits, d_out.p, d_out.cap, d_cursor.p, st.get());
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(&n, d_cursor.p, sizeof n, cudaMemcpyDeviceToHost, st.get()));
            CK(cudaStreamSynchronize(st.get()));
            if (n <= d_out.cap) break;
            d_out.ensure(n);
        }
        found[g].resize(n);
        if (n) CK(cudaMemcpyAsync(found[g].data(), d_out.p, n * sizeof(RegionRead), cudaMemcpyDeviceToHost, st.get()));
        CK(cudaStreamSynchronize(st.get()));
    };
    if (is_multi(X)) {
        for_each_gpu(X, run);
    } else {
        CK(cudaSetDevice(X->device));
        run(0, X);
    }
    std::vector<RegionRead> all;
    for (auto& f : found) all.insert(all.end(), f.begin(), f.end());
    std::sort(all.begin(), all.end(), [](const RegionRead& a, const RegionRead& b) {
        return a.region != b.region ? a.region < b.region : a.read < b.read;
    });
    D.reads.resize(all.size());
    for (size_t i = 0; i < all.size(); ++i) D.reads[i] = ReadCoordinate{all[i].read, all[i].start, all[i].end, (uint8_t)all[i].fwd};
    for (size_t r = 0, i = 0; r < nR; ++r) {
        CandidateRegion& c = D.regions[r];
        c.read_off = i;
        while (i < all.size() && all[i].region == r) ++i;
        c.n_reads = (uint32_t)(i - c.read_off);
    }
}

// ============================================================================================
// discover's local assembler (assemble.cu): the pileups of all candidate regions of the sample are uploaded once, one
// CTA per region counts and walks them, and the host reads back the statuses, the walk lengths and the walks' bases.
// The consensus walk is dropped and the rest sorted here.
// ============================================================================================
uint32_t consensus_kmer(const std::string& c, size_t at) {  // UINT32_MAX when a base is not ACGT: never solid
    static const char acgt[] = "ACGT";
    uint32_t x = 0;
    for (size_t i = at; i < at + DISCOVER_K; ++i) {
        const char* q = c[i] ? strchr(acgt, c[i]) : nullptr;
        if (!q) return UINT32_MAX;
        x = (x << 2) | (uint32_t)(q - acgt);
    }
    return x;
}

void assemble_regions(drprg_index* X, const drprg_assemble_opts* o) {
    AsmParams P{2, 15, 25};  // pandora discover: --min-dbg-dp 2, --max-ins 15, --max-num-candidate-paths 25
    if (o && o->min_dbg_dp) P.min_dp = o->min_dbg_dp;
    if (o && o->max_insertion != 0xffffffffu) P.max_insertion = o->max_insertion;
    if (o && o->max_candidate_paths) P.max_paths = o->max_candidate_paths;
    if (P.max_paths > ASM_MAX_PATHS_LIMIT) throw std::runtime_error("max_candidate_paths above " + std::to_string(ASM_MAX_PATHS_LIMIT));
    const DiscoverResult& D = X->discover;
    const size_t nR = D.regions.size();
    // every retained read of the sample, over the GPUs of a multi-GPU handle
    std::unordered_map<uint32_t, std::pair<const drprg_index::RetainedReads*, size_t>> where;
    for (drprg_index* g : (X->gpus.empty() ? std::vector<drprg_index*>{X} : X->gpus))
        for (size_t i = 0; i < g->retained_reads.read.size(); ++i) where[g->retained_reads.read[i]] = {&g->retained_reads, i};
    std::unordered_map<uint32_t, uint32_t> uploaded;  // read -> its words in `words`
    std::vector<uint32_t> words, list;
    std::vector<uint4> entries;
    std::vector<AsmRegion> regs(nR);
    std::vector<uint32_t> global_list;
    uint64_t global_slots = 0, out_cap = 0;
    uint32_t max_walk = DISCOVER_K, smem_slots = 64;
    for (size_t r = 0; r < nR; ++r) {
        const CandidateRegion& c = D.regions[r];
        const std::string& cons = D.consensus[c.locus];
        AsmRegion& A = regs[r];
        memset(&A, 0, sizeof A);
        A.entry_off = (uint32_t)entries.size();
        uint64_t n_pos = 0;
        for (uint64_t q = c.read_off; q < c.read_off + c.n_reads; ++q) {
            const ReadCoordinate& rc = D.reads[q];
            const auto it = where.find(rc.read);
            if (it == where.end()) throw std::runtime_error("the bases of read " + std::to_string(rc.read) + " were not retained");
            const drprg_index::RetainedReads& S = *it->second.first;
            const size_t i = it->second.second;
            if (rc.start > rc.end || rc.end > S.len[i]) throw std::runtime_error("region read span outside its read");
            auto up = uploaded.find(rc.read);
            if (up == uploaded.end()) {
                up = uploaded.emplace(rc.read, (uint32_t)words.size()).first;
                words.insert(words.end(), S.words.begin() + S.off[i], S.words.begin() + S.off[i] + (S.len[i] + 15) / 16);
                if (words.size() >= 0xffffffffull) throw std::runtime_error("region reads exceed 2^32 words");
            }
            entries.push_back(make_uint4(up->second, rc.start, rc.end, rc.fwd));
            if (rc.end - rc.start >= DISCOVER_K) n_pos += rc.end - rc.start - DISCOVER_K + 1;
        }
        if (entries.size() >= 0xffffffffull) throw std::runtime_error("too many region reads");
        A.n_entries = (uint32_t)(entries.size() - A.entry_off);
        uint64_t slots = 64;
        while (slots < 2 * n_pos) slots <<= 1;
        A.slots = (uint32_t)slots;
        A.span = c.pad_end - c.pad_start;
        for (uint32_t i = 0; i < KMER_ATTEMPTS && c.pad_start + i + DISCOVER_K <= c.start; ++i)
            A.start_kmer[A.n_start++] = consensus_kmer(cons, c.pad_start + i);
        for (uint32_t j = 0; j < KMER_ATTEMPTS && c.pad_end >= c.end + DISCOVER_K + j; ++j)
            A.end_kmer[A.n_end++] = consensus_kmer(cons, c.pad_end - DISCOVER_K - j);
        const uint32_t walk = A.span + P.max_insertion;
        if (walk > ASM_MAX_WALK) throw std::runtime_error("a candidate region is wider than the assembler takes (" + std::to_string(ASM_MAX_WALK) + " bases with the insertion)");
        max_walk = std::max(max_walk, walk);
        out_cap += (uint64_t)P.max_paths * walk;
        if (slots <= ASM_SMEM_SLOTS) {
            list.push_back((uint32_t)r);
            smem_slots = std::max(smem_slots, (uint32_t)slots);
        } else {
            A.table_off = global_slots;
            global_slots += slots;
            global_list.push_back((uint32_t)r);
        }
    }
    const uint32_t n_smem = (uint32_t)list.size(), n_global = (uint32_t)global_list.size();
    list.insert(list.end(), global_list.begin(), global_list.end());
    X->asm_status.assign(nR, 0);
    X->asm_paths.clear();
    X->asm_bases.clear();
    X->asm_stats[0] = n_smem;
    X->asm_stats[1] = n_global;
    X->asm_stats[2] = X->asm_stats[3] = 0;
    if (!nR) return;
    CK(cudaSetDevice(X->device));
    Stream st = new_stream();
    Event ev[3] = {new_event(cudaEventDefault), new_event(cudaEventDefault), new_event(cudaEventDefault)};
    DBuf<uint32_t> d_words, d_list, d_keys, d_counts, d_wlen;
    DBuf<uint4> d_entries;
    DBuf<AsmRegion> d_regs;
    DBuf<AsmResult> d_res;
    DBuf<char> d_out;
    DBuf<unsigned long long> d_cursor;
    d_words.ensure(std::max<size_t>(1, words.size()));
    d_entries.ensure(std::max<size_t>(1, entries.size()));
    d_regs.ensure(nR);
    d_list.ensure(nR);
    d_keys.ensure(std::max<uint64_t>(1, global_slots));
    d_counts.ensure(std::max<uint64_t>(1, global_slots));
    d_res.ensure(nR);
    d_wlen.ensure(nR * P.max_paths);
    d_out.ensure(std::max<uint64_t>(1, out_cap));
    d_cursor.ensure(1);
    if (!words.empty()) CK(cudaMemcpyAsync(d_words.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice, st.get()));
    if (!entries.empty()) CK(cudaMemcpyAsync(d_entries.p, entries.data(), entries.size() * sizeof(uint4), cudaMemcpyHostToDevice, st.get()));
    CK(cudaMemcpyAsync(d_regs.p, regs.data(), nR * sizeof(AsmRegion), cudaMemcpyHostToDevice, st.get()));
    CK(cudaMemcpyAsync(d_list.p, list.data(), nR * 4, cudaMemcpyHostToDevice, st.get()));
    CK(cudaMemsetAsync(d_cursor.p, 0, sizeof(unsigned long long), st.get()));
    CK(cudaEventRecord(ev[0].get(), st.get()));
    launch_assemble(d_regs.p, d_list.p, n_smem, d_entries.p, d_words.p, smem_slots, nullptr, nullptr, max_walk, P, d_res.p,
                    d_wlen.p, d_out.p, d_cursor.p, st.get());
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[1].get(), st.get()));
    launch_assemble(d_regs.p, d_list.p + n_smem, n_global, d_entries.p, d_words.p, 0, d_keys.p, d_counts.p, max_walk, P, d_res.p,
                    d_wlen.p, d_out.p, d_cursor.p, st.get());
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[2].get(), st.get()));
    std::vector<AsmResult> res(nR);
    std::vector<uint32_t> wlen(nR * P.max_paths);
    unsigned long long used = 0;
    CK(cudaMemcpyAsync(res.data(), d_res.p, nR * sizeof(AsmResult), cudaMemcpyDeviceToHost, st.get()));
    CK(cudaMemcpyAsync(wlen.data(), d_wlen.p, wlen.size() * 4, cudaMemcpyDeviceToHost, st.get()));
    CK(cudaMemcpyAsync(&used, d_cursor.p, sizeof used, cudaMemcpyDeviceToHost, st.get()));
    CK(cudaStreamSynchronize(st.get()));
    std::string out(used, '\0');
    if (used) CK(cudaMemcpyAsync(&out[0], d_out.p, used, cudaMemcpyDeviceToHost, st.get()));
    CK(cudaStreamSynchronize(st.get()));
    float ms[2] = {0, 0};
    CK(cudaEventElapsedTime(&ms[0], ev[0].get(), ev[1].get()));
    CK(cudaEventElapsedTime(&ms[1], ev[1].get(), ev[2].get()));
    X->asm_stats[2] = ms[0];
    X->asm_stats[3] = ms[1];
    for (size_t r = 0; r < nR; ++r) {
        const AsmResult& R = res[r];
        X->asm_status[r] = (uint8_t)R.status;
        if (R.status != ASM_ASSEMBLED) continue;
        const CandidateRegion& c = D.regions[r];
        const uint32_t a = c.pad_start + R.anchor_i, b = c.pad_end - R.anchor_j;
        const std::string& cons = D.consensus[c.locus];
        std::vector<std::string> alleles;
        uint64_t off = R.byte_off;
        for (uint32_t w = 0; w < R.n_walks; ++w) {
            const uint32_t L = wlen[r * P.max_paths + w];
            if (off + L > used) throw std::runtime_error("assembled walks outside the output buffer");
            std::string s = out.substr(off, L);
            off += L;
            if (s.compare(0, std::string::npos, cons, a, b - a) != 0) alleles.push_back(std::move(s));
        }
        std::sort(alleles.begin(), alleles.end());
        for (const std::string& s : alleles) {
            X->asm_paths.push_back(drprg_denovo_path{(uint32_t)r, a, b, (uint32_t)s.size(), (uint64_t)X->asm_bases.size()});
            X->asm_bases += s;
        }
    }
}

// The map half of a sample from a reads file: strict FASTQ (plain or gzip) in waves of host-framed text, anything else
// through the host parser as one batch
struct FileMapped {
    uint64_t n = 0, dropped = 0, bases = 0, hits = 0, kept = 0;
    size_t waves = 0;
    double ms_ingest = 0, ms_map = 0;
};
FileMapped map_reads_file(drprg_index* X, const char* reads_path, const drprg_map_opts* o, const Inflated* pre) {
    const double t0 = now_ms();
    FileMapped M;
    WaveTotals W;
    if (map_file_in_waves(X, reads_path, o, pre, W)) {
        M.dropped = W.dropped;
        M.bases = W.bases;
        M.hits = W.hits;
        M.kept = W.kept;
        M.n = W.n;
        M.waves = W.waves;
        M.ms_ingest = W.ms_ingest;  // ingest and map alternate wave by wave
        M.ms_map = W.ms_map;
        return M;
    }
    // Not strict 4-line FASTQ, or host ingest forced.  Framing the whole file would decline as well: it runs the same
    // framer over the same records as the waves, and it takes at most 8 GB of text where the waves take any size.
    const FileBatch F = host_parsed_batch(X, reads_path, o ? o->threads : 1);
    drprg_batch* B = F.B.get();
    M.dropped = F.n_dropped;
    M.bases = B->total_bases;
    const double t1 = now_ms();
    sample_begin_any(X, o, F.first_read_len);
    M.n = B->R.n_reads;
    map_batch_any(X, B, 0, &M.hits, &M.kept);
    M.ms_ingest = t1 - t0;
    M.ms_map = now_ms() - t1;
    return M;
}

int run_sample(drprg_index* X, const char* reads_path, const char* vcf_refs, const char* outdir, const drprg_map_opts* o,
               drprg_map_stats* stats, const Inflated* pre = nullptr) {
    need_device(X);
    const double t0 = now_ms();
    // like the reference (File::create of pandora.log comes first, src/lib.rs:592-593): an unusable outdir fails before
    // any GPU work is done
    std::ofstream log(std::string(outdir) + "/pandora.log");
    if (!log) throw std::runtime_error(std::string("cannot write ") + outdir + "/pandora.log");
    const FileMapped M = map_reads_file(X, reads_path, o, pre);
    const double t2 = now_ms();
    genotype(X, vcf_refs, "sample");
    std::ofstream vcf(std::string(outdir) + "/pandora_genotyped.vcf");
    if (!vcf) throw std::runtime_error(std::string("cannot write ") + outdir + "/pandora_genotyped.vcf");
    vcf.write(X->h_vcf.data() + X->vcf_begin, (std::streamsize)X->vcf_len);
    const double t3 = now_ms();
    drprg_map_stats s{};
    s.n_reads = M.n;
    s.n_reads_dropped = M.dropped;
    s.total_bases = M.bases;
    s.n_hits = M.hits;
    s.n_hits_kept = M.kept;
    s.n_loci_present = (uint32_t)X->contigs.size();
    s.n_records = (uint32_t)X->records.size();
    s.exp_depth_covg = X->fit.E;
    s.ms_ingest = M.ms_ingest;
    s.ms_map = M.ms_map;
    s.ms_genotype = t3 - t2;
    s.ms_total = t3 - t0;
    if (stats) *stats = s;
    log << "drprg-cuda map: reads=" << M.n << " dropped=" << M.dropped << " bases=" << M.bases << " hits=" << M.hits
        << " kept=" << M.kept << " loci=" << s.n_loci_present << " records=" << s.n_records << " E=" << s.exp_depth_covg
        << " ingest=" << (M.waves ? "host-framed, " + std::to_string(M.waves) + " wave(s)" : "host") << "\nkernel ms: sketch_lookup=" << X->timings[0] << " sort=" << X->timings[1] << " cluster=" << X->timings[2]
        << " coverage=" << X->timings[3] << "\nwall ms: ingest=" << s.ms_ingest << " map=" << s.ms_map
        << " genotype=" << s.ms_genotype << " total=" << s.ms_total << "\n";
    return 0;
}

DiscoverOpts discover_opts_from(const drprg_discover_opts* o) {
    DiscoverOpts D;
    if (o) {
        if (o->covg_threshold) D.covg_threshold = o->covg_threshold;
        if (o->min_len) D.min_len = o->min_len;
        if (o->max_len) D.max_len = o->max_len;
        if (o->padding != 0xffffffffu) D.padding = o->padding;
        if (o->min_hits) D.min_hits = o->min_hits;
    }
    return D;
}

void refuse_shard_handles(const drprg_index* X) {
    if (X->world > 1 || X->ipc_mapping)
        throw std::runtime_error("one-process-per-GPU handles (drprg_cuda_shard_root / drprg_cuda_shard_attach) keep no read bases: "
                                 "assemble on a single-GPU or drprg_cuda_index_load_multi handle");
}

// `pandora discover` for one sample from the one map pass: map (hit retention on), ML path, candidate regions, local
// assembly, and <outdir>/denovo_paths.txt from the de-novo alleles
void run_discover(drprg_index* X, const char* sample_name, const char* reads_path, const char* outdir, const drprg_map_opts* o,
                  const drprg_discover_opts* d, const drprg_assemble_opts* a, drprg_discover_stats* stats,
                  const Inflated* pre = nullptr) {
    need_device(X);
    refuse_shard_handles(X);
    const char* sample = sample_name ? sample_name : "sample";
    const double t0 = now_ms();
    const std::string path = std::string(outdir) + "/denovo_paths.txt";
    // an unusable outdir fails before any GPU work is done; the file itself is only created once its text is known
    if (access(outdir, W_OK | X_OK) != 0) throw std::runtime_error("cannot write " + path + ": " + strerror(errno));
    struct RetainGuard {  // the caller's retention setting comes back whatever happens
        drprg_index* X;
        bool was;
        ~RetainGuard() {
            for (drprg_index* g : (X->gpus.empty() ? std::vector<drprg_index*>{X} : X->gpus)) g->retain_hits = was;
        }
    } guard{X, X->retain_hits};
    for (drprg_index* g : (X->gpus.empty() ? std::vector<drprg_index*>{X} : X->gpus)) g->retain_hits = true;
    const FileMapped M = map_reads_file(X, reads_path, o, pre);
    const double t1 = now_ms();
    genotype(X, nullptr, sample);  // pandora discover takes no --vcf-refs: the ML path does not depend on them
    const double t2 = now_ms();
    find_candidates(X, discover_opts_from(d));
    assemble_regions(X, a);
    const DiscoverResult& D = X->discover;
    std::vector<std::vector<DenovoVariant>> variants(X->H.loci.size());
    for (const drprg_denovo_path& p : X->asm_paths) {
        const uint32_t l = D.regions[p.region].locus;
        allele_variants(D.consensus[l], p.a, p.b, X->asm_bases.substr(p.offset, p.length), variants[l]);
    }
    drprg_discover_stats s{};
    for (auto& v : variants) {
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
        s.n_loci_with_variants += !v.empty();
        s.n_variants += (uint32_t)v.size();
    }
    const std::string text = denovo_paths_text(X->H, sample, D, variants);
    std::ofstream out(path);
    if (!out) throw std::runtime_error("cannot write " + path);
    out.write(text.data(), (std::streamsize)text.size());
    out.close();
    if (!out) throw std::runtime_error("write error on " + path);
    const double t3 = now_ms();
    s.n_reads = M.n;
    s.n_hits_kept = M.kept;
    s.n_region_reads = D.reads.size();
    s.n_regions = (uint32_t)D.regions.size();
    for (uint8_t st : X->asm_status) {
        s.n_assembled += st == ASM_ASSEMBLED;
        s.n_no_anchor += st == ASM_NO_ANCHOR;
        s.n_too_many_paths += st == ASM_TOO_MANY_PATHS;
        s.n_no_path += st == ASM_NO_PATH;
    }
    s.ms_ingest = M.ms_ingest;
    s.ms_map = M.ms_map;
    s.ms_ml_path = t2 - t1;
    s.ms_discover = t3 - t2;
    s.ms_total = t3 - t0;
    if (stats) *stats = s;
}

// The gzip look-ahead of the batch calls.  A gzip file is inflated on all host cores (gzip_inflate.cpp), and that is still
// most of a sample's time: in a batch of 1 M-read samples on a 16-core host, 91 ms per sample from gzip files against
// 7 ms (map) and 11 ms (discover) from plain ones (profiles/r7_batch_discover_n1.jsonl).  While sample i runs, the gzip
// files of the next few samples are inflated on threads of their own.  They share the cores with each other and with
// sample i's host work, so the look-ahead gains only the time the cores would otherwise be idle, such as sample i's GPU
// work and its waits.
class GzipLookahead {
  public:
    GzipLookahead(size_t n, const char* const* reads_paths, const drprg_map_opts* o)
        : paths_(reads_paths), ahead_(n),
          window_(std::max<size_t>(1, std::min<size_t>({n, (size_t)(o && o->threads ? o->threads : 1), (size_t)8}))) {
        for (size_t i = 0; i < window_; ++i) start(i);
    }
    // the text of sample i (p == nullptr for a plain file); starts the look-ahead of sample i + window; throws the error of
    // the inflate
    Inflated take(size_t i) {
        Inflated pre;
        if (ahead_[i].valid()) pre = ahead_[i].get();
        start(i + window_);
        if (!pre.error.empty()) throw std::runtime_error(pre.error);
        return pre;
    }

  private:
    void start(size_t i) {
        if (i >= ahead_.size() || !file_is_gzip(paths_[i])) return;
        const std::string path = paths_[i];
        ahead_[i] = std::async(std::launch::async, [path]() {
            Inflated r;
            try {
                r.inflate(path);
            } catch (const std::exception& e) {
                r.error = e.what();
            }
            return r;
        });
    }
    const char* const* paths_;
    std::vector<std::future<Inflated>> ahead_;
    const size_t window_;
};
}  // namespace

#define API_BEGIN try {
#define API_END                          \
    }                                    \
    catch (const std::exception& e) {    \
        g_err = e.what();                \
        return 1;                        \
    }                                    \
    catch (...) {                        \
        g_err = "unknown error";         \
        return 1;                        \
    }

extern "C" {
int drprg_cuda_version(void) { return DRPRG_CUDA_VERSION; }
const char* drprg_cuda_last_error(void) { return g_err.c_str(); }
int drprg_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
int drprg_cuda_index_load(const char* prg_path, uint32_t w, uint32_t k, int device, drprg_index** out) {
    API_BEGIN return load_common(read_text_file(prg_path), w, k, device, out);
    API_END
}
int drprg_cuda_index_load_text(const char* prg_text, uint32_t w, uint32_t k, int device, drprg_index** out) {
    API_BEGIN return load_common(prg_text, w, k, device, out);
    API_END
}
int drprg_cuda_index_load_multi(const char* prg_path, uint32_t w, uint32_t k, int n_gpus, const int* devices, drprg_index** out) {
    API_BEGIN return load_multi(read_text_file(prg_path), w, k, n_gpus, devices, out);
    API_END
}
int drprg_cuda_index_n_gpus(drprg_index* X) { return X->gpus.empty() ? (X->device >= 0 ? 1 : 0) : (int)X->gpus.size(); }
void drprg_cuda_index_free(drprg_index* x) { delete x; }

/* one process per GPU: the root rank's accumulator becomes the reduction target of the other ranks */
int drprg_cuda_shard_root(drprg_index* X, int world_size, void* handle64) {
    API_BEGIN need_device(X);
    if (is_multi(X)) throw std::runtime_error("a multi-GPU handle shards inside the library already");
    CK(cudaSetDevice(X->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, X->d_accum.p));
    static_assert(sizeof(h) == 64, "CUDA IPC handles are 64 bytes");
    memcpy(handle64, &h, sizeof h);
    X->world = std::max(1, world_size);
    X->accum_shared = X->world > 1;
    X->hist_on_host = false;
    return 0;
    API_END
}
int drprg_cuda_shard_attach(drprg_index* X, int world_size, const void* handle64) {
    API_BEGIN need_device(X);
    if (is_multi(X)) throw std::runtime_error("a multi-GPU handle shards inside the library already");
    CK(cudaSetDevice(X->device));
    if (X->ipc_mapping) {
        CK(cudaIpcCloseMemHandle(X->ipc_mapping));
        X->ipc_mapping = nullptr;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof h);
    void* p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    X->ipc_mapping = p;
    X->reduce_dst = (int32_t*)p;  // same index on every rank: same accumulator layout
    X->flag_ready = reinterpret_cast<uint32_t*>((int32_t*)p + accum_flag_offset(X->n_accum));
    X->flag_arrivals = X->flag_ready + 1;
    X->world = std::max(1, world_size);
    return 0;
    API_END
}
int drprg_cuda_shard_done(drprg_index* X, void* stream) {
    API_BEGIN need_device(X);
    if (!X->reduce_dst || !X->flag_arrivals) throw std::runtime_error("drprg_cuda_shard_attach was not called");
    CK(cudaSetDevice(X->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t sc[4] = {(int32_t)(X->own_bases & 0xffffff), (int32_t)(X->own_bases >> 24), (int32_t)(X->own_reads & 0xffffff),
                           (int32_t)(X->own_reads >> 24)};
    // a rank without reads still has to wait for the root's zeroing before it touches the scalars
    launch_flag_wait(X->flag_ready, X->epoch, st);
    launch_shard_done(X->reduce_dst + X->n_accum - 4, sc, X->flag_arrivals, st);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
    API_END
}

int drprg_cuda_map_genotype(drprg_index* X, const char* reads_path, const char* vcf_refs, const char* outdir,
                            const drprg_map_opts* o, drprg_map_stats* stats) {
    API_BEGIN return run_sample(X, reads_path, vcf_refs, outdir, o, stats);
    API_END
}
int drprg_cuda_map_genotype_batch(drprg_index* X, size_t n, const char* const* reads_paths, const char* vcf_refs,
                                  const char* const* outdirs, const drprg_map_opts* o, drprg_map_stats* stats) {
    API_BEGIN GzipLookahead ahead(n, reads_paths, o);
    for (size_t i = 0; i < n; ++i) {
        const Inflated pre = ahead.take(i);
        run_sample(X, reads_paths[i], vcf_refs, outdirs[i], o, stats ? stats + i : nullptr, pre.p ? &pre : nullptr);
    }
    return 0;
    API_END
}

int64_t drprg_cuda_pack_reads(const uint8_t* ascii, const uint64_t* off, uint64_t n_reads, uint32_t stride_words,
                              uint32_t* words, uint64_t words_cap, uint64_t* word_off, uint32_t* lens) {
    int64_t r = pack_ascii(ascii, off, n_reads, stride_words, words, words_cap, word_off, lens);
    if (r < 0) g_err = (r == -1) ? "read longer than the fixed stride" : "words buffer too small";
    return r;
}
int drprg_cuda_read_fastx(const char* path, uint32_t threads, uint32_t** words, uint64_t** word_off, uint32_t** lens,
                          uint64_t* n_reads, uint64_t* total_bases, uint32_t* first_read_len) {
    API_BEGIN PackedReads pr;
    load_reads_packed(path, threads, pr);
    *words = (uint32_t*)malloc(std::max<size_t>(1, pr.words.size()) * 4);
    *word_off = (uint64_t*)malloc(pr.word_off.size() * 8);
    *lens = (uint32_t*)malloc(std::max<size_t>(1, pr.lens.size()) * 4);
    memcpy(*words, pr.words.data(), pr.words.size() * 4);
    memcpy(*word_off, pr.word_off.data(), pr.word_off.size() * 8);
    memcpy(*lens, pr.lens.data(), pr.lens.size() * 4);
    *n_reads = pr.lens.size();
    *total_bases = pr.total_bases;
    *first_read_len = pr.first_read_len;
    return 0;
    API_END
}
void drprg_cuda_host_free(void* p) { free(p); }

int drprg_cuda_frame_fastq(const char* path, uint32_t threads, uint8_t** ascii, uint32_t** lens, uint64_t* n_reads,
                           uint64_t* total_bases, int* is_fastq) {
    API_BEGIN* ascii = nullptr;
    *lens = nullptr;
    *n_reads = *total_bases = 0;
    *is_fastq = 0;
    if (file_is_gzip(path)) return 0;  // plain files only
    const ReadsText T(path, nullptr);
    if (!T.may_be_fastq()) return 0;
    std::vector<char> buf(T.src.size / 2 + 64);
    std::vector<FramedSlice> sl;
    if (!fastq_frame_text(T.src, threads, buf.data(), sl)) return 0;
    uint64_t n = 0, bases = 0;
    for (const FramedSlice& z : sl) {
        n += z.st.n_reads;
        bases += z.st.total_bases;
    }
    *ascii = (uint8_t*)malloc(std::max<uint64_t>(1, bases));
    *lens = (uint32_t*)malloc(std::max<uint64_t>(1, n) * 4);
    uint64_t r = 0, at = 0;
    for (const FramedSlice& z : sl)
        for (size_t i = 0; i < z.lens.size(); ++i) {
            memcpy(*ascii + at, buf.data() + z.starts[i], z.lens[i]);
            at += z.lens[i];
            (*lens)[r++] = z.lens[i];
        }
    *n_reads = n;
    *total_bases = bases;
    *is_fastq = 1;
    return 0;
    API_END
}

int drprg_cuda_batch_upload(drprg_index* X, const uint32_t* words, const uint64_t* word_off, uint32_t stride_words,
                            const uint32_t* lens, uint64_t n_reads, uint64_t total_bases, uint32_t read_id_base, void* stream,
                            drprg_batch** out) {
    API_BEGIN if (!stride_words && !word_off) throw std::runtime_error("word_off is required without a fixed stride");
    if (is_multi(X)) *out = multi_upload(X, words, word_off, stride_words, lens, n_reads, total_bases, read_id_base).release();
    else *out = upload_batch(X, words, word_off, stride_words, lens, n_reads, total_bases, read_id_base, (cudaStream_t)stream).release();
    return 0;
    API_END
}
int drprg_cuda_batch_wrap_device(drprg_index* X, const void* d_words, const void* d_word_off, uint32_t stride_words,
                                 const void* d_lens, uint64_t n_reads, uint64_t total_bases, uint32_t read_id_base,
                                 drprg_batch** out) {
    API_BEGIN if (is_multi(X)) throw std::runtime_error("device-resident arrays belong to one GPU: wrap them on a single-GPU handle");
    if (!stride_words && !d_word_off) throw std::runtime_error("word_off is required without a fixed stride");
    drprg_batch* B = new drprg_batch();
    B->R = DevReads{(const uint32_t*)d_words, (const uint64_t*)d_word_off, stride_words, (const uint32_t*)d_lens, n_reads, read_id_base};
    B->total_bases = total_bases;
    B->max_len = stride_words ? stride_words * 16u : UINT32_MAX;
    *out = B;
    return 0;
    API_END
}
int drprg_cuda_batch_from_fastx(drprg_index* X, const char* path, uint32_t threads, drprg_batch** out, uint64_t* n_reads,
                                uint64_t* total_bases, uint64_t* n_dropped, uint32_t* first_read_len, int* parsed_on_device) {
    API_BEGIN FileBatch F = batch_from_file(X, path, threads);
    if (n_reads) *n_reads = F.B->R.n_reads;
    if (total_bases) *total_bases = F.B->total_bases;
    if (n_dropped) *n_dropped = F.n_dropped;
    if (first_read_len) *first_read_len = F.first_read_len;
    if (parsed_on_device) *parsed_on_device = F.on_device ? 1 : 0;
    *out = F.B.release();
    return 0;
    API_END
}
void drprg_cuda_batch_free(drprg_batch* b) { delete b; }

int drprg_cuda_sample_begin(drprg_index* X, const drprg_map_opts* o, uint32_t first_read_len) {
    API_BEGIN sample_begin_any(X, o, first_read_len);
    return 0;
    API_END
}
int drprg_cuda_map_batch(drprg_index* X, drprg_batch* B, void* stream, uint64_t* n_hits, uint64_t* n_kept) {
    API_BEGIN map_batch_any(X, B, (cudaStream_t)stream, n_hits, n_kept);
    return 0;
    API_END
}
int drprg_cuda_accum_device_ptr(drprg_index* X, void** d_ptr, uint64_t* n_int32) {
    API_BEGIN need_device(X);
    CK(cudaSetDevice(X->device));
    flush_scalars(X);
    X->hist_on_host = false;  // the caller may change the accumulators (allreduce)
    *d_ptr = X->d_accum.p;
    *n_int32 = X->n_accum;
    return 0;
    API_END
}
int drprg_cuda_accum_download(drprg_index* X, int32_t* out, uint64_t n) {
    API_BEGIN need_device(X);
    if (n != X->n_accum) throw std::runtime_error("accumulator size mismatch");
    CK(cudaSetDevice(X->device));
    flush_scalars(X);
    CK(cudaMemcpy(out, X->d_accum.p, n * 4, cudaMemcpyDeviceToHost));
    return 0;
    API_END
}
int drprg_cuda_accum_upload(drprg_index* X, const int32_t* in, uint64_t n) {
    API_BEGIN need_device(X);
    if (n != X->n_accum) throw std::runtime_error("accumulator size mismatch");
    CK(cudaSetDevice(X->device));
    CK(cudaMemcpy(X->d_accum.p, in, n * 4, cudaMemcpyHostToDevice));
    X->hist_on_host = false;
    X->scalars_in_buffer = true;
    return 0;
    API_END
}
int drprg_cuda_genotype(drprg_index* X, const char* vcf_refs, const char* sample) {
    API_BEGIN genotype(X, vcf_refs, sample);
    return 0;
    API_END
}
int drprg_cuda_write_vcf(drprg_index* X, const char* path) {
    API_BEGIN if (!X->have_gt) throw std::runtime_error("no genotype results");
    std::ofstream f(path);
    if (!f) throw std::runtime_error(std::string("cannot write ") + path);
    f.write(X->h_vcf.data() + X->vcf_begin, (std::streamsize)X->vcf_len);
    return 0;
    API_END
}
const char* drprg_cuda_vcf_text(drprg_index* X) { return X->have_gt ? X->h_vcf.data() + X->vcf_begin : ""; }
const char* drprg_cuda_vcf_view(drprg_index* X, uint64_t* len) {
    if (len) *len = X->have_gt ? X->vcf_len : 0;
    return X->have_gt ? X->h_vcf.data() + X->vcf_begin : "";
}

uint64_t drprg_cuda_hash64(uint64_t kmer, uint32_t k) { return hash64_host(kmer, k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1)); }
uint64_t drprg_cuda_hash64_inverse(uint64_t hash, uint32_t k) {
    return hash64_inverse_host(hash, k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1));
}

int drprg_cuda_index_info(drprg_index* X, drprg_index_info* o) {
    API_BEGIN o->w = X->H.w;
    o->k = X->H.k;
    o->n_loci = (uint32_t)X->H.loci.size();
    o->total_knodes = X->H.total_knodes();
    o->n_records = X->H.records.size();
    o->n_edges = X->n_edges;
    o->n_path_intervals = X->n_ivs;
    o->table_slots = X->table_slots;
    o->filter_words = X->filter_words;
    return 0;
    API_END
}
const char* drprg_cuda_locus_name(drprg_index* X, uint32_t l) { return l < X->H.loci.size() ? X->H.loci[l].name.c_str() : ""; }
int drprg_cuda_index_knode_base(drprg_index* X, uint32_t* out) {
    memcpy(out, X->H.knode_base.data(), X->H.knode_base.size() * 4);
    return 0;
}
int drprg_cuda_index_knodes(drprg_index* X, uint64_t* hash, uint8_t* strand, uint32_t* n_out, uint32_t* n_iv) {
    size_t g = 0;
    for (auto& L : X->H.loci)
        for (size_t r = 0; r < L.kpath.size(); ++r, ++g) {
            hash[g] = L.khash[r];
            strand[g] = L.kstrand[r];
            n_out[g] = (uint32_t)L.kout[r].size();
            n_iv[g] = (uint32_t)L.kpath[r].size();
        }
    return 0;
}
int drprg_cuda_index_edges(drprg_index* X, uint32_t* edges) {
    size_t e = 0;
    for (size_t l = 0; l < X->H.loci.size(); ++l)
        for (auto& o : X->H.loci[l].kout)
            for (uint32_t t : o) edges[e++] = X->H.knode_base[l] + t;
    return 0;
}
int drprg_cuda_index_paths(drprg_index* X, uint32_t* iv_start, uint32_t* iv_len) {
    size_t e = 0;
    for (auto& L : X->H.loci)
        for (auto& p : L.kpath)
            for (auto& sg : p) {
                iv_start[e] = sg.s;
                iv_len[e] = sg.e - sg.s;
                ++e;
            }
    return 0;
}
int drprg_cuda_index_records(drprg_index* X, uint64_t* hash, uint32_t* prg, uint32_t* knode, uint8_t* strand) {
    size_t i = 0;
    for (auto& r : X->H.records) {
        hash[i] = r.hash;
        prg[i] = r.prg;
        knode[i] = r.knode;
        strand[i] = r.strand;
        ++i;
    }
    return 0;
}
int drprg_cuda_index_min_path_length(drprg_index* X, uint32_t* out) {
    for (size_t l = 0; l < X->H.loci.size(); ++l) out[l] = X->H.loci[l].min_path_len;
    return 0;
}
int drprg_cuda_index_screen_filters(drprg_index* X, uint32_t* kfilter, uint32_t* kfilter_words, uint32_t* kfilter14,
                                    uint32_t* kfilter14_words) {
    API_BEGIN
    const ScreenFilters F = build_screen_filters(X->H);
    if (kfilter) std::copy(F.kfilter.begin(), F.kfilter.end(), kfilter);
    if (kfilter14) std::copy(F.kfilter14.begin(), F.kfilter14.end(), kfilter14);
    *kfilter_words = (uint32_t)F.kfilter.size();
    *kfilter14_words = (uint32_t)F.kfilter14.size();
    return 0;
    API_END
}

int64_t drprg_cuda_sketch_batch(drprg_index* X, drprg_batch* B, void* stream, uint32_t* read, uint32_t* start, uint64_t* hash,
                                uint8_t* strand, uint64_t cap) {
    try {
        need_device(X);
        CK(cudaSetDevice(X->device));
        cudaStream_t st = (cudaStream_t)stream;
        DBuf<unsigned long long> key, val;
        key.ensure(cap);
        val.ensure(cap);
        CK(cudaMemsetAsync(X->d_counters.p, 0, 16, st));
        for (auto& e : B->ev)
            if (e) CK(cudaStreamWaitEvent(st, e.get(), 0));
        launch_sketch_only(B->R, X->H.w, X->H.k, key.p, val.p, X->d_counters.p, cap, X->sm_count, B->max_len, st);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(X->h_counters.p, X->d_counters.p, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        uint64_t n = X->h_counters.p[0];
        if (n > cap) {
            g_err = "sketch output capacity too small";
            return -(int64_t)n;
        }
        std::vector<unsigned long long> hk(n), hv(n);
        CK(cudaMemcpy(hk.data(), key.p, n * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(hv.data(), val.p, n * 8, cudaMemcpyDeviceToHost));
        std::vector<uint64_t> ord(n);
        for (uint64_t i = 0; i < n; ++i) ord[i] = i;
        std::sort(ord.begin(), ord.end(), [&](uint64_t a, uint64_t b) { return hk[a] < hk[b]; });
        for (uint64_t i = 0; i < n; ++i) {
            const uint64_t j = ord[i];
            read[i] = (uint32_t)(hk[j] >> 32);
            start[i] = (uint32_t)hk[j];
            hash[i] = hv[j] >> 1;
            strand[i] = (uint8_t)(hv[j] & 1);
        }
        return (int64_t)n;
    } catch (const std::exception& e) {
        g_err = e.what();
        return INT64_MIN;
    }
}
int64_t drprg_cuda_last_hits(drprg_index* X0, uint32_t* read, uint32_t* start, uint32_t* prg, uint32_t* knode, uint8_t* fwd,
                             uint8_t* kept, uint64_t cap) {
    try {
        need_device(X0);
        // a multi-GPU handle holds one contiguous shard of reads per GPU: the shards are listed in GPU order
        std::vector<drprg_index*> gpus = X0->gpus.empty() ? std::vector<drprg_index*>{X0} : X0->gpus;
        uint64_t total = 0;
        for (drprg_index* X : gpus) total += X->last_n_hits;
        if (total > cap) return -(int64_t)total;
        uint64_t o = 0;
        for (drprg_index* X : gpus) {
            CK(cudaSetDevice(X->device));
            const uint64_t n = X->last_n_hits, na = X->last_n_active;
            // the device keeps the hits grouped by read (slices in no particular order, sorted within a read that can keep
            // hits): pandora's order (read, prg, strand, read_start, k-mer node) is restored here
            std::vector<unsigned long long> key(n);
            std::vector<uint8_t> kp(n);
            std::vector<uint32_t> ar(na), ab(na), ac(na);
            if (n) {
                CK(cudaMemcpy(key.data(), X->gkey.p, n * 8, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(kp.data(), X->gkept.p, n, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(ar.data(), X->act_read.p, na * 4, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(ab.data(), X->act_base.p, na * 4, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(ac.data(), X->act_count.p, na * 4, cudaMemcpyDeviceToHost));
            }
            std::vector<uint32_t> ord(na);
            for (uint32_t i = 0; i < na; ++i) ord[i] = i;
            std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return ar[a] < ar[b]; });
            const uint64_t o0 = o;
            for (uint32_t a : ord) {
                // reads that cannot keep anything are not sorted on the device; their flags are all 0, so sorting the keys alone is exact
                if (!std::is_sorted(key.begin() + ab[a], key.begin() + ab[a] + ac[a])) std::sort(key.begin() + ab[a], key.begin() + ab[a] + ac[a]);
                for (uint32_t j = ab[a]; j < ab[a] + ac[a]; ++j, ++o) {
                    const unsigned long long k = key[j];
                    read[o] = X->last_id_base + ar[a];
                    prg[o] = (uint32_t)(k >> 48);
                    fwd[o] = (uint8_t)(((k >> 47) & 1ull) ^ 1ull);
                    start[o] = (uint32_t)(k >> GKEY_KNODE_BITS) & ((1u << GKEY_START_BITS) - 1u);
                    knode[o] = (uint32_t)k & ((1u << GKEY_KNODE_BITS) - 1u);
                    kept[o] = kp[j];
                }
            }
            if (o - o0 != n) throw std::runtime_error("grouped hits do not add up");
        }
        CK(cudaSetDevice(X0->device));
        return (int64_t)total;
    } catch (const std::exception& e) {
        g_err = e.what();
        return INT64_MIN;
    }
}
int drprg_cuda_gt_params(drprg_index* X, double* out) {
    const FitParams& P = X->fit;
    out[0] = P.E; out[1] = P.bin; out[2] = P.nb_p; out[3] = P.nb_r; out[4] = P.e_rate; out[5] = P.thresh;
    out[6] = P.covg; out[7] = P.min_kmer_covg; out[8] = P.mean; out[9] = P.var; out[10] = (double)P.num_reads;
    return 0;
}
int64_t drprg_cuda_gt_mlpath(drprg_index* X, uint32_t locus, uint32_t* out, uint64_t cap) {
    if (!X->have_gt || locus >= X->present.size() || !X->present[locus]) return -1;
    const auto& p = X->mlpaths[locus];
    for (size_t i = 0; i < p.size() && i < cap; ++i) out[i] = p[i];
    return (int64_t)p.size();
}
int drprg_cuda_gt_counts(drprg_index* X, uint32_t* n_records, uint32_t* n_alleles, uint64_t* n_allele_knodes) {
    *n_records = (uint32_t)X->records.size();
    *n_alleles = X->GA.allele_off.empty() ? 0 : (uint32_t)X->GA.allele_off.size() - 1;
    *n_allele_knodes = X->GA.allele_kn.size();
    return 0;
}
int drprg_cuda_gt_records(drprg_index* X, uint32_t* locus, uint32_t* pos, uint32_t* n_alleles, int32_t* gt, double* gt_conf) {
    ensure_ga(X);
    for (size_t i = 0; i < X->records.size(); ++i) {
        locus[i] = X->records[i]->locus;
        pos[i] = X->records[i]->pos;
        n_alleles[i] = X->GA.rec_off[i + 1] - X->GA.rec_off[i];
        gt[i] = X->GA.gt[i];
        gt_conf[i] = X->GA.gt_conf[i];
    }
    return 0;
}
int drprg_cuda_gt_alleles(drprg_index* X, double* lik, double* gaps, uint32_t* mean_fwd, uint32_t* mean_rev, uint32_t* med_fwd,
                          uint32_t* med_rev, uint32_t* sum_fwd, uint32_t* sum_rev, uint32_t* n_knodes) {
    ensure_ga(X);
    const GenotypeArrays& G = X->GA;
    const size_t na = G.lik.size();
    memcpy(lik, G.lik.data(), na * 8);
    memcpy(gaps, G.gaps.data(), na * 8);
    memcpy(mean_fwd, G.mean_fwd.data(), na * 4);
    memcpy(mean_rev, G.mean_rev.data(), na * 4);
    memcpy(med_fwd, G.med_fwd.data(), na * 4);
    memcpy(med_rev, G.med_rev.data(), na * 4);
    memcpy(sum_fwd, G.sum_fwd.data(), na * 4);
    memcpy(sum_rev, G.sum_rev.data(), na * 4);
    for (size_t a = 0; a < na; ++a) n_knodes[a] = G.allele_off[a + 1] - G.allele_off[a];
    return 0;
}
int drprg_cuda_gt_allele_knodes(drprg_index* X, uint32_t* out) {
    // ranks within the locus, like the oracle
    size_t e = 0;
    for (const SiteRecord* r : X->records)
        for (auto& kn : r->allele_kn)
            for (uint32_t x : kn) out[e++] = x;
    return 0;
}
int drprg_cuda_genotype_rows(int device, uint32_t n_records, const uint32_t* rec_off, const uint32_t* mean_fwd,
                             const uint32_t* mean_rev, const double* gaps, uint32_t exp_depth, double genotyping_error_rate,
                             double min_gt_conf, float minor_af, double* lik, int32_t* gt, double* gt_conf, int32_t* covg_gt,
                             float* frs, float* sb_ratio, int32_t* minor_gt, float* pdp) {
    API_BEGIN
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw std::runtime_error("no CUDA device visible: drprg-cuda has no CPU fallback");
    if (device < 0 || device >= ndev) throw std::runtime_error("bad device ordinal");
    CK(cudaSetDevice(device));
    if (!n_records) return 0;
    const uint32_t na = rec_off[n_records];
    DBuf<uint32_t> d_u32;
    DBuf<double> d_f64;
    DBuf<int32_t> d_i32;
    DBuf<float> d_f32;
    d_u32.ensure((size_t)n_records + 1 + 2 * (size_t)na);
    d_f64.ensure(2 * (size_t)na + n_records);
    d_i32.ensure((size_t)n_records * 3);
    d_f32.ensure((size_t)n_records * 2 + na);
    uint32_t *d_off = d_u32.p, *d_mf = d_off + n_records + 1, *d_mr = d_mf + na;
    double *d_gaps = d_f64.p, *d_lik = d_gaps + na, *d_conf = d_lik + na;
    CK(cudaMemcpy(d_off, rec_off, ((size_t)n_records + 1) * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_mf, mean_fwd, (size_t)na * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_mr, mean_rev, (size_t)na * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_gaps, gaps, (size_t)na * 8, cudaMemcpyHostToDevice));
    DevGenotype G{};
    G.n_records = n_records;
    G.n_alleles = na;
    G.rec_off = d_off;
    G.mean_fwd = d_mf;
    G.mean_rev = d_mr;
    G.gaps = d_gaps;
    G.lik = d_lik;
    G.gt_conf = d_conf;
    G.gt = d_i32.p;
    G.covg_gt = d_i32.p + n_records;
    G.minor_gt = d_i32.p + 2 * (size_t)n_records;
    G.frs = d_f32.p;
    G.sb_ratio = d_f32.p + n_records;
    G.pdp = d_f32.p + 2 * (size_t)n_records;
    ModelParams MP{};
    MP.exp_depth = exp_depth;
    MP.gt_err = genotyping_error_rate > 0 ? genotyping_error_rate : 0.01;
    MP.gt_conf = min_gt_conf;
    MP.minor_af = minor_af;
    launch_genotype_rows(G, MP, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(lik, d_lik, (size_t)na * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(gt_conf, d_conf, (size_t)n_records * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(gt, d_i32.p, (size_t)n_records * 4, cudaMemcpyDeviceToHost));
    if (covg_gt) CK(cudaMemcpy(covg_gt, G.covg_gt, (size_t)n_records * 4, cudaMemcpyDeviceToHost));
    if (minor_gt) CK(cudaMemcpy(minor_gt, G.minor_gt, (size_t)n_records * 4, cudaMemcpyDeviceToHost));
    if (frs) CK(cudaMemcpy(frs, G.frs, (size_t)n_records * 4, cudaMemcpyDeviceToHost));
    if (sb_ratio) CK(cudaMemcpy(sb_ratio, G.sb_ratio, (size_t)n_records * 4, cudaMemcpyDeviceToHost));
    if (pdp) CK(cudaMemcpy(pdp, G.pdp, (size_t)na * 4, cudaMemcpyDeviceToHost));
    return 0;
    API_END
}
/* `pandora index` replacement (SURVEY 8f rank 3): the files drprg's validate_index looks for, next to the PRG */
int drprg_cuda_index_write(drprg_index* X, const char* prg_path) {
    API_BEGIN write_pandora_index(X->H, prg_path);
    return 0;
    API_END
}
/* ---- discover's mapping front half from the map pass (SURVEY 8f rank 1) ---- */
int drprg_cuda_retain_hits(drprg_index* X, int on) {
    for (drprg_index* g : (X->gpus.empty() ? std::vector<drprg_index*>{X} : X->gpus)) g->retain_hits = on != 0;
    return 0;
}
int drprg_cuda_discover_candidates(drprg_index* X, const drprg_discover_opts* o, uint32_t* n_regions, uint64_t* n_region_reads) {
    API_BEGIN need_device(X);
    if (!X->have_gt) throw std::runtime_error("drprg_cuda_genotype has not run for this sample");
    if (!X->retain_hits) throw std::runtime_error("drprg_cuda_retain_hits(idx, 1) must be set before the sample is mapped");
    find_candidates(X, discover_opts_from(o));
    if (n_regions) *n_regions = (uint32_t)X->discover.regions.size();
    if (n_region_reads) *n_region_reads = X->discover.reads.size();
    return 0;
    API_END
}
int drprg_cuda_discover_regions(drprg_index* X, drprg_candidate_region* out) {
    for (size_t i = 0; i < X->discover.regions.size(); ++i) {
        const CandidateRegion& c = X->discover.regions[i];
        out[i] = drprg_candidate_region{c.locus, c.start, c.end, c.pad_start, c.pad_end, c.n_reads, c.read_off};
    }
    return 0;
}
int drprg_cuda_discover_region_reads(drprg_index* X, uint32_t* read, uint32_t* start, uint32_t* end, uint8_t* fwd) {
    for (size_t i = 0; i < X->discover.reads.size(); ++i) {
        const ReadCoordinate& r = X->discover.reads[i];
        read[i] = r.read;
        start[i] = r.start;
        end[i] = r.end;
        fwd[i] = r.fwd;
    }
    return 0;
}
const char* drprg_cuda_discover_consensus(drprg_index* X, uint32_t locus, uint64_t* len) {
    if (locus >= X->discover.consensus.size() || X->discover.consensus[locus].empty()) {
        if (len) *len = 0;
        return nullptr;
    }
    if (len) *len = X->discover.consensus[locus].size();
    return X->discover.consensus[locus].c_str();
}
int drprg_cuda_discover_coverage(drprg_index* X, uint32_t locus, uint32_t* covg) {
    if (locus >= X->discover.coverage.size()) return 1;
    memcpy(covg, X->discover.coverage[locus].data(), X->discover.coverage[locus].size() * 4);
    return 0;
}
int drprg_cuda_discover_assemble(drprg_index* X, const drprg_assemble_opts* o, uint32_t* n_paths, uint64_t* n_path_bases) {
    API_BEGIN need_device(X);
    refuse_shard_handles(X);
    if (!X->have_gt) throw std::runtime_error("drprg_cuda_genotype has not run for this sample");
    if (!X->retain_hits) throw std::runtime_error("drprg_cuda_retain_hits(idx, 1) must be set before the sample is mapped");
    if (!X->discover_ready) throw std::runtime_error("drprg_cuda_discover_candidates has not run for this sample");
    assemble_regions(X, o);
    if (n_paths) *n_paths = (uint32_t)X->asm_paths.size();
    if (n_path_bases) *n_path_bases = X->asm_bases.size();
    return 0;
    API_END
}
int drprg_cuda_discover(drprg_index* X, const char* sample, const char* reads_path, const char* outdir, const drprg_map_opts* o,
                        const drprg_discover_opts* d, const drprg_assemble_opts* a, drprg_discover_stats* stats) {
    API_BEGIN run_discover(X, sample, reads_path, outdir, o, d, a, stats);
    return 0;
    API_END
}
int drprg_cuda_discover_batch(drprg_index* X, size_t n, const char* const* samples, const char* const* reads_paths,
                              const char* const* outdirs, const drprg_map_opts* o, const drprg_discover_opts* d,
                              const drprg_assemble_opts* a, drprg_discover_stats* stats) {
    API_BEGIN need_device(X);
    refuse_shard_handles(X);
    if (n && (!reads_paths || !outdirs)) throw std::runtime_error("reads_paths and outdirs must hold n entries each");
    GzipLookahead ahead(n, reads_paths, o);
    for (size_t i = 0; i < n; ++i) {
        try {
            const Inflated pre = ahead.take(i);
            run_discover(X, samples ? samples[i] : nullptr, reads_paths[i], outdirs[i], o, d, a, stats ? stats + i : nullptr,
                         pre.p ? &pre : nullptr);
        } catch (const std::exception& e) {
            throw std::runtime_error("sample " + std::to_string(i) + " (" + reads_paths[i] + "): " + e.what());
        }
    }
    return 0;
    API_END
}
int drprg_cuda_discover_paths(drprg_index* X, drprg_denovo_path* out, char* bases) {
    if (!X->asm_paths.empty()) memcpy(out, X->asm_paths.data(), X->asm_paths.size() * sizeof(drprg_denovo_path));
    if (!X->asm_bases.empty()) memcpy(bases, X->asm_bases.data(), X->asm_bases.size());
    return 0;
}
int drprg_cuda_discover_region_status(drprg_index* X, uint8_t* status) {
    if (!X->asm_status.empty()) memcpy(status, X->asm_status.data(), X->asm_status.size());
    return 0;
}
int drprg_cuda_last_assemble_stats(drprg_index* X, double* out4) {
    memcpy(out4, X->asm_stats, sizeof X->asm_stats);
    return 0;
}
int drprg_cuda_set_minor_af(drprg_index* X, float minor_af) {
    X->minor_af = minor_af;
    return 0;
}
int drprg_cuda_gt_filter_stats(drprg_index* X, int32_t* covg_gt, float* frs, float* sb_ratio, int32_t* minor_gt, float* pdp) {
    API_BEGIN need_device(X);
    if (!X->have_gt) throw std::runtime_error("no genotype results");
    CK(cudaSetDevice(X->device));
    const size_t nr = X->records.size(), na = X->GA.allele_off.empty() ? 0 : X->GA.allele_off.size() - 1;
    if (!nr) return 0;
    if (covg_gt) CK(cudaMemcpy(covg_gt, X->d_gt_i32.p + nr, nr * 4, cudaMemcpyDeviceToHost));
    if (minor_gt) CK(cudaMemcpy(minor_gt, X->d_gt_i32.p + 2 * nr, nr * 4, cudaMemcpyDeviceToHost));
    if (frs) CK(cudaMemcpy(frs, X->d_gt_f32.p, nr * 4, cudaMemcpyDeviceToHost));
    if (sb_ratio) CK(cudaMemcpy(sb_ratio, X->d_gt_f32.p + nr, nr * 4, cudaMemcpyDeviceToHost));
    if (pdp) CK(cudaMemcpy(pdp, X->d_gt_f32.p + 2 * nr, na * 4, cudaMemcpyDeviceToHost));
    return 0;
    API_END
}
int drprg_cuda_last_timings(drprg_index* X, float* out4) {
    memcpy(out4, X->timings, sizeof X->timings);
    return 0;
}
int drprg_cuda_last_genotype_timings(drprg_index* X, double* out6 /* 7 values */) {
    memcpy(out6, X->gt_ms, 7 * sizeof(double));
    return 0;
}
int drprg_cuda_format_g6(double v, char* out) {
    size_t n = format_g6(v, out);
    out[n] = 0;
    return (int)n;
}
int drprg_cuda_format_g6_device(int device, const double* v, uint32_t n, char* out, uint8_t* len, uint8_t* refused) {
    API_BEGIN CK(cudaSetDevice(device));
    DBuf<double> dv;
    DBuf<char> dout;
    DBuf<uint8_t> dl, dr;
    dv.ensure(n);
    dout.ensure(48ull * n);
    dl.ensure(n);
    dr.ensure(n);
    CK(cudaMemcpy(dv.p, v, (size_t)n * 8, cudaMemcpyHostToDevice));
    launch_format_g6_batch(dv.p, n, dout.p, dl.p, dr.p, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, 48ull * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(len, dl.p, n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(refused, dr.p, n, cudaMemcpyDeviceToHost));
    return 0;
    API_END
}
uint64_t drprg_cuda_launch_count(void) { return launch_count(); }
double drprg_cuda_issue_peak(drprg_index* X) {
    try {
        need_device(X);
        CK(cudaSetDevice(X->device));
        return measure_issue_peak(X->sm_count, 0);
    } catch (const std::exception& e) {
        g_err = e.what();
        return 0.0;
    }
}
}
