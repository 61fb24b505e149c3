// C ABI of include/drprg_cuda.h: the drop-in for Pandora::genotype_with
// (/root/reference/src/lib.rs:580-642) plus the staged interface used for multi-GPU read sharding,
// benches and parity tests.  Owns all device memory of an index (plain cudaMalloc; no torch types).
#include <cuda_runtime.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
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

#include "../../include/drprg_cuda.h"
#include "genotype_host.hpp"
#include "fastq_frame.hpp"
#include "ingest.hpp"
#include "kernels.cuh"
#include "prg_graph.hpp"

using namespace drprg;

namespace {
thread_local std::string g_err;

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #call); \
    } while (0)

template <class T>
struct DBuf {  // grow-only device buffer
    T* p = nullptr;
    size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) cudaFree(p);
        p = nullptr;
        size_t want = n + n / 4 + 1024;
        CK(cudaMalloc(&p, want * sizeof(T)));
        cap = want;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

template <class T>
struct PinnedBuf {  // grow-only pinned host buffer: async D2H into pageable memory would block the host
    T* p = nullptr;
    size_t cap = 0, n = 0;
    void resize(size_t want) {
        if (want > cap) {
            if (p) cudaFreeHost(p);
            p = nullptr;
            cap = want + want / 4 + 256;
            CK(cudaMallocHost(&p, cap * sizeof(T)));
        }
        n = want;
    }
    T* data() { return p; }
    size_t size() const { return n; }
    T* begin() { return p; }
    T* end() { return p + n; }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = n = 0;
    }
};

template <class T>
T* to_device(const std::vector<T>& v) {
    T* d = nullptr;
    CK(cudaMalloc(&d, std::max<size_t>(1, v.size()) * sizeof(T)));
    if (!v.empty()) CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return d;
}

// freed batch buffers are parked here and reused by the next upload: cudaFree synchronises the device and
// cudaMalloc costs ~0.1-1 ms, both of which would sit inside every end-to-end step
struct DevPool {
    struct Slot { void* p; size_t bytes; int device; };
    std::vector<Slot> free_;
    std::mutex m_;
    void* get(size_t bytes, int device) {
        std::lock_guard<std::mutex> g(m_);
        size_t best = free_.size();
        for (size_t i = 0; i < free_.size(); ++i)
            if (free_[i].device == device && free_[i].bytes >= bytes && (best == free_.size() || free_[i].bytes < free_[best].bytes)) best = i;
        if (best != free_.size() && free_[best].bytes <= bytes * 2 + (1 << 20)) {
            void* p = free_[best].p;
            free_.erase(free_.begin() + best);
            return p;
        }
        void* p = nullptr;
        CK(cudaMalloc(&p, bytes));
        return p;
    }
    void put(void* p, size_t bytes, int device) {
        std::lock_guard<std::mutex> g(m_);
        if (free_.size() >= 16) {
            cudaFree(free_.front().p);
            free_.erase(free_.begin());
        }
        free_.push_back({p, bytes, device});
    }
} g_pool;

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
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
    std::vector<drprg_batch*> shards;  // multi-GPU handle: one sub-batch per GPU (this object is then only the container)
    DevReads R{};
    uint32_t *d_words = nullptr, *d_lens = nullptr, *d_seg_read = nullptr, *d_seg_start = nullptr;
    uint64_t* d_off = nullptr;
    bool owned = false;
    size_t b_words = 0, b_lens = 0, b_off = 0, b_seg = 0;
    int device = 0;
    uint64_t total_bases = 0;
    uint32_t max_len = UINT32_MAX;  // longest read (bound); selects the short-read kernel
    // host uploads are split into chunks copied on a separate stream; the sketch kernel of chunk c starts as soon
    // as its bytes have landed, so the H2D copy overlaps the sketch of the previous chunks
    int n_chunks = 1;
    uint64_t chunk_lo[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

struct drprg_index {
    HostIndex H;
    int device = 0, sm_count = 148;
    // device-resident index
    DevTable T{};
    uint2 *d_slots = nullptr, *d_recs = nullptr;
    uint32_t* d_kfilter = nullptr;
    uint32_t *d_filter = nullptr, *d_knode_base = nullptr, *d_edge_off = nullptr, *d_edges = nullptr;
    uint8_t *d_is_terminal = nullptr, *d_needs_mean = nullptr;
    uint32_t *d_locus_unit_off = nullptr, *d_unit_start = nullptr, *d_unit_nodes = nullptr;
    uint32_t *d_locus_level_off = nullptr, *d_level_start = nullptr, *d_level_nodes = nullptr, *d_level_singles = nullptr;
    float mean_run_len = 0.f;
    uint32_t table_slots = 0, filter_words = 0;
    uint64_t n_edges = 0, n_ivs = 0;
    // accumulators: [2*N coverage | P locus reads | 4 scalars]
    int32_t* d_accum = nullptr;
    uint64_t n_accum = 0;
    uint64_t total_bases = 0, n_reads = 0;
    bool scalars_in_buffer = false;
    bool hist_on_host = false;  // h_small holds the coverage histogram + locus read counts of the current accumulators
    // sample state
    SampleOpts opts;
    bool sample_open = false;
    uint32_t first_read_len = 0;
    uint32_t* d_thresh = nullptr;
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
    unsigned long long* d_counters = nullptr;  // CTR_* of kernels.cuh
    unsigned long long* h_counters = nullptr;  // pinned
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
    cudaEvent_t ev[6]{};  // batch timeline: start, lookup done, hits grouped, clustered, coverage merged
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
    uint32_t *d_rec_off = nullptr, *d_allele_off = nullptr, *d_allele_kn = nullptr, *d_knode_locus = nullptr, *d_hist = nullptr;
    DBuf<uint32_t> d_gt_u32;
    DBuf<double> d_gt_f64;
    DBuf<int32_t> d_gt_i32;
    DBuf<float> d_gt_f32;  // frs | strand-bias ratio (per record), depth proportions (per allele)
    float minor_af = -1.0f;  // < 0: drprg's default (1.0, or 0.1 with --illumina)
    // discover's front half from the map pass (SURVEY 8f rank 1): kept hits of the sample, retained on request
    bool retain_hits = false;
    std::vector<RetainedHit> retained;
    DiscoverResult discover;
    uint32_t max_locus_knodes = 0, max_locus_edges = 0;
    cudaEvent_t ev_ml[2] = {nullptr, nullptr};
    cudaStream_t st_ml = nullptr, st_gt = nullptr, st_copy = nullptr, st_acc = nullptr;
    cudaEvent_t ev_acc[3] = {nullptr, nullptr, nullptr};  // [2]: node scores + threshold ready on `st`
    double* d_thresh_f64 = nullptr;
    int* d_thresh_i32 = nullptr;
    PinnedBuf<int> h_thresh;
    uint32_t* d_hist1000 = nullptr;
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
    char* d_vcf_prefix = nullptr;
    uint32_t *d_vcf_prefix_off = nullptr, *d_vcf_slot_off = nullptr, *d_vcf_ctl = nullptr;  // ctl: [0] text bytes, [1] flags
    DBuf<char> d_vcf_slots;
    DBuf<uint32_t> d_vcf_line_len, d_vcf_out_off;
    PinnedBuf<uint32_t> h_vcf_ctl;
    size_t vcf_prefix_bytes = 0, vcf_slot_bytes = 0;
    bool ga_stale = false;  // the per-allele / per-record arrays are in the pinned download buffers, not yet in GA
    bool have_gt = false;
    bool ml_in_flight = false;  // the ML-path kernel of an unfinished drprg_cuda_genotype may still be writing h_path / h_done
    DBuf<double> d_prob, d_M;
    DBuf<uint32_t> d_len, d_up, d_path, d_path_len;

    ~drprg_index() {
        workers.clear();
        replicas.clear();
        if (device < 0) return;
        cudaSetDevice(device);
        if (ipc_mapping) cudaIpcCloseMemHandle(ipc_mapping);
        for (void* p : {(void*)d_slots, (void*)d_recs, (void*)d_filter, (void*)d_knode_base, (void*)d_edge_off, (void*)d_edges,
                        (void*)d_is_terminal, (void*)d_needs_mean, (void*)d_locus_unit_off, (void*)d_unit_start, (void*)d_unit_nodes, (void*)d_accum, (void*)d_thresh, (void*)d_counters, (void*)d_rec_off,
                        (void*)d_allele_off, (void*)d_allele_kn, (void*)d_knode_locus, (void*)d_hist, (void*)d_kfilter, (void*)d_locus_level_off, (void*)d_level_start, (void*)d_level_nodes, (void*)d_level_singles})
            if (p) cudaFree(p);
        if (h_counters) cudaFreeHost(h_counters);
        hi.release(); lo.release(); gkey.release(); gkept.release();
        act_read.release(); act_base.release(); act_count.release(); act_lk.release(); lk_ovf.release(); big_list.release(); cov_keys.release();
        for (auto& b : scratch) b.release();
        read_count.release(); read_base.release();
        partials.release();
        queue.release(); queue_kmer.release();
        d_gt_u32.release(); d_gt_f64.release(); d_gt_i32.release(); d_gt_f32.release();
        d_prob.release(); d_M.release(); d_len.release(); d_up.release(); d_path.release(); d_path_len.release();
        for (auto& e : ev)
            if (e) cudaEventDestroy(e);
        h_path.release(); h_plen.release(); h_u32.release(); h_done.release(); h_f64.release(); h_gt.release(); h_acc.release();
        h_vcf.release(); h_vcf_ctl.release(); d_vcf_slots.release(); d_vcf_line_len.release(); d_vcf_out_off.release();
        for (void* p : {(void*)d_vcf_prefix, (void*)d_vcf_prefix_off, (void*)d_vcf_slot_off, (void*)d_vcf_ctl})
            if (p) cudaFree(p);
        for (auto& e : ev_ml)
            if (e) cudaEventDestroy(e);
        if (st_copy) cudaStreamDestroy(st_copy);
        if (st_acc) cudaStreamDestroy(st_acc);
        for (auto& e : ev_acc)
            if (e) cudaEventDestroy(e);
        if (d_hist1000) cudaFree(d_hist1000);
        if (d_thresh_f64) cudaFree(d_thresh_f64);
        if (d_thresh_i32) cudaFree(d_thresh_i32);
        h_thresh.release();
        h_small.release();
        if (st_ml) cudaStreamDestroy(st_ml);
        if (st_gt) cudaStreamDestroy(st_gt);
    }
};

namespace {
inline size_t accum_flag_offset(uint64_t n_accum) { return (size_t)((n_accum + 31) & ~31ull); }  // 128-byte aligned flag words

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
    X->d_slots = to_device(slots);
    X->d_recs = to_device(recs);
    X->d_filter = to_device(filter);
    X->table_slots = 1u << sb;
    X->filter_words = 1u << fb;
    X->T = DevTable{X->d_slots, sb, X->d_recs, X->d_filter, fb};
    // ---- k-mer screen: the k-mers behind the indexed hashes, both orientations (hash64 is invertible)
    if (H.k >= 8 && H.k <= 15 && distinct > 0) {
        const uint64_t mask = (1ull << (2 * H.k)) - 1;
        std::vector<uint32_t> kmers;
        kmers.reserve(distinct * 2);
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
        // The filter is capped by one SM's shared memory (1.77 Mbit).  Beyond ~300 k k-mers (4x the Mtb-scale panel) more
        // than a third of its bits are set, over 10 % of all read positions are flagged and resolving them costs as much
        // as sketching every read: such an index keeps the sketch kernels.
        const bool screen_pays = kmers.size() <= 300000;
        // ~24 filter bits per k-mer, capped by the shared memory of one SM
        uint32_t nw = (uint32_t)std::min<uint64_t>(SCREEN_MAX_FILTER_WORDS, std::max<uint64_t>(1024, (kmers.size() * 24 + 31) / 32));
        nw = (nw + 3) & ~3u;
        std::vector<uint32_t> kfilter(nw, 0);
        for (uint32_t x : kmers) screen_filter_insert(kfilter.data(), nw, x, H.k);
        if (screen_pays) {
            X->d_kfilter = to_device(kfilter);
            X->T.kfilter = X->d_kfilter;
            X->T.kfilter_words = nw;
        }
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
    X->d_knode_base = to_device(H.knode_base);
    X->d_edge_off = to_device(edge_off);
    X->d_edges = to_device(edges);
    X->d_is_terminal = to_device(term);
    {   // a node's mean log-prob is only ever compared when one of its predecessors has more than one out-edge
        std::vector<uint8_t> needs(N, 0);
        for (size_t l = 0; l < H.loci.size(); ++l) {
            const Locus& L = H.loci[l];
            const uint32_t base = H.knode_base[l];
            for (uint32_t r = 0; r < L.kpath.size(); ++r)
                if (L.kout[r].size() > 1)
                    for (uint32_t o : L.kout[r]) needs[base + o] = 1;
        }
        X->d_needs_mean = to_device(needs);
    }
    {   // processing units of the ML-path kernel: a node with a choice (or none), or a run of <= 32 single-successor nodes
        std::vector<uint32_t> locus_unit_off(1, 0), unit_start(1, 0), unit_nodes;
        for (size_t l = 0; l < H.loci.size(); ++l) {
            const Locus& L = H.loci[l];
            const uint32_t n = (uint32_t)L.kpath.size();
            std::vector<std::vector<uint32_t>> preds(n);
            for (uint32_t r = 0; r < n; ++r)
                for (uint32_t o : L.kout[r]) preds[o].push_back(r);
            std::vector<char> done(n, 0);
            for (uint32_t r = n >= 2 ? n - 1 : 0; r-- > 0;) {  // n-2 .. 0 (the terminus is not a unit)
                if (done[r]) continue;
                done[r] = 1;
                unit_nodes.push_back(r);
                if (L.kout[r].size() == 1) {
                    uint32_t cur = r, len = 1;
                    while (len < 32) {
                        uint32_t best = UINT32_MAX;
                        for (uint32_t p : preds[cur])
                            if (!done[p] && L.kout[p].size() == 1 && (best == UINT32_MAX || p > best)) best = p;
                        if (best == UINT32_MAX) break;
                        done[best] = 1;
                        unit_nodes.push_back(best);
                        cur = best;
                        ++len;
                    }
                }
                unit_start.push_back((uint32_t)unit_nodes.size());
            }
            locus_unit_off.push_back((uint32_t)unit_start.size() - 1);
        }
        {
            uint64_t runs = 0, run_nodes = 0;
            for (size_t l = 0; l < H.loci.size(); ++l)
                for (uint32_t uu = locus_unit_off[l]; uu < locus_unit_off[l + 1]; ++uu)
                    if (H.loci[l].kout[unit_nodes[unit_start[uu]]].size() == 1) {
                        ++runs;
                        run_nodes += unit_start[uu + 1] - unit_start[uu];
                    }
            X->mean_run_len = runs ? (float)run_nodes / (float)runs : 0.f;
        }
        X->d_locus_unit_off = to_device(locus_unit_off);
        X->d_unit_start = to_device(unit_start);
        X->d_unit_nodes = to_device(unit_nodes);
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
        X->d_locus_level_off = to_device(locus_level_off);
        X->d_level_start = to_device(level_start);
        X->d_level_nodes = to_device(level_nodes);
        X->d_level_singles = to_device(level_singles);
    }
    X->n_accum = 2ull * N + H.loci.size() + 4;
    // 16 extra words behind the accumulator hold the cross-GPU flags of a read-sharded run (ready epoch, arrival counter)
    CK(cudaMalloc(&X->d_accum, (accum_flag_offset(X->n_accum) + 16) * sizeof(int32_t)));
    CK(cudaMemset(X->d_accum, 0, (accum_flag_offset(X->n_accum) + 16) * sizeof(int32_t)));
    CK(cudaMalloc(&X->d_thresh, std::max<size_t>(1, H.loci.size()) * sizeof(uint32_t)));
    CK(cudaMalloc(&X->d_counters, CTR_COUNT * sizeof(unsigned long long)));
    CK(cudaMallocHost(&X->h_counters, CTR_COUNT * sizeof(unsigned long long)));

    for (auto& e : X->ev) CK(cudaEventCreate(&e));
    std::vector<uint32_t> knode_locus(N);
    for (size_t l = 0; l < H.loci.size(); ++l) {
        for (uint32_t g = H.knode_base[l]; g < H.knode_base[l + 1]; ++g) knode_locus[g] = (uint32_t)l;
        X->max_locus_knodes = std::max(X->max_locus_knodes, H.knode_base[l + 1] - H.knode_base[l]);
        X->max_locus_edges = std::max(X->max_locus_edges, edge_off[H.knode_base[l + 1]] - edge_off[H.knode_base[l]]);
    }
    X->d_knode_locus = to_device(knode_locus);
    CK(cudaMalloc(&X->d_hist, 200 * sizeof(uint32_t)));
    CK(cudaMalloc(&X->d_hist1000, 1000 * sizeof(uint32_t)));
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
        if (!thr.empty()) CK(cudaMemcpy(X->d_thresh, thr.data(), thr.size() * 4, cudaMemcpyHostToDevice));
        X->thresh_on_device = thr;
    }
    CK(cudaMemset(X->d_accum, 0, X->n_accum * sizeof(int32_t)));
    ++X->epoch;
    if (X->world > 1 && X->accum_shared)  // the other ranks may add to this accumulator from here on
        launch_flag_publish(reinterpret_cast<uint32_t*>(X->d_accum + accum_flag_offset(X->n_accum)), X->epoch, 0);
    X->total_bases = X->n_reads = 0;
    X->own_bases = X->own_reads = 0;
    X->retained.clear();
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

void map_batch(drprg_index* X, drprg_batch* B, cudaStream_t st, uint64_t* n_hits, uint64_t* n_kept) {
    if (!X->sample_open) throw std::runtime_error("drprg_cuda_sample_begin was not called");
    CK(cudaSetDevice(X->device));
    const HostIndex& H = X->H;
    if (B->max_len != UINT32_MAX && B->max_len >= (1u << GKEY_START_BITS)) throw std::runtime_error("reads of 32 Mb or more are not supported");
    // whole-genome reads give ~0.35 hits per 150 bp read; a targeted run overflows once, regrows to the exact count and is redone
    ensure_hit_capacity(X, std::max<uint64_t>(X->hi.cap, std::max<uint64_t>(1u << 20, B->total_bases / 256)));
    ensure_read_capacity(X, B->R.n_reads);
    if (X->T.kfilter) {  // ~2 flagged positions per 150 bp read
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
        CK(cudaMemsetAsync(X->d_counters, 0, CTR_COUNT * sizeof(unsigned long long), st));
        CK(cudaEventRecord(X->ev[0], st));
        for (int c = 0; c < B->n_chunks; ++c) {
            DevReads Rc = B->R;
            Rc.hit_count = X->read_count.p;
            if (B->n_chunks > 1) {
                const uint64_t lo = B->chunk_lo[c], hi = B->chunk_lo[c + 1];
                Rc.hit_count = X->read_count.p + lo;
                if (B->ev[c]) CK(cudaStreamWaitEvent(st, B->ev[c], 0));
                Rc.words = B->R.stride_words ? B->R.words + lo * B->R.stride_words : B->R.words;
                Rc.word_off = B->R.word_off ? B->R.word_off + lo : nullptr;
                Rc.lens = B->R.lens + lo;
                Rc.n_reads = hi - lo;
                Rc.read_id_base = B->R.read_id_base + (uint32_t)lo;
            }
            launch_sketch_lookup(Rc, X->T, H.w, H.k, X->hi.p, X->lo.p, X->d_counters + CTR_HITS, X->hi.cap, X->sm_count, B->max_len, st,
                                 X->queue.p, queue_cap, X->d_counters + CTR_QUEUE, X->queue_kmer.p);
        }
        CK(cudaGetLastError());
        CK(cudaEventRecord(X->ev[1], st));
        PostBuffers PB{};
        PB.hi = X->hi.p; PB.lo = X->lo.p; PB.ctr = X->d_counters;
        PB.read_count = X->read_count.p; PB.read_base = X->read_base.p;
        PB.act_read = X->act_read.p; PB.act_base = X->act_base.p; PB.act_count = X->act_count.p;
        PB.act_lk = X->act_lk.p; PB.lk_ovf = X->lk_ovf.p;
        PB.big_list = X->big_list.p; PB.gkey = X->gkey.p; PB.gkept = X->gkept.p; PB.cov_keys = X->cov_keys.p;
        for (int i = 0; i < 10; ++i) PB.scratch[i] = X->scratch[i].p;
        PB.partials = X->partials.p; PB.n_partials = X->n_partials;
        if (X->reduce_dst && X->flag_ready) launch_flag_wait(X->flag_ready, X->epoch, st);  // root has zeroed its accumulator for this sample
        launch_postprocess(PB, PostCaps{X->hi.cap, queue_cap}, B->R.read_id_base, B->R.n_reads, X->opts.max_diff, X->min_thresh, X->d_thresh,
                           X->d_knode_base, N, P, X->reduce_dst ? X->reduce_dst : X->d_accum,
                           (X->reduce_dst || X->accum_shared) ? 1 : 0,  // several GPUs add into one accumulator: every writer uses red
                           X->sm_count, st,
                           X->ev[2], X->ev[3]);
        CK(cudaEventRecord(X->ev[4], st));
        CK(cudaGetLastError());
        if (!X->reduce_dst && !X->accum_shared) {
            // what the genotype step needs first (coverage histogram, locus read counts: 4 KB) rides on this batch's final
            // synchronisation; it stays valid unless the accumulators change before drprg_cuda_genotype (another batch
            // recomputes it, a reduce from other GPUs invalidates it)
            launch_cov_hist(X->d_accum, N, X->d_is_terminal, X->d_knode_locus, X->d_accum + 2ull * N, X->d_hist1000, st);
            X->h_small.resize(1000 + (size_t)P + 4);
            CK(cudaMemcpyAsync(X->h_small.data(), X->d_hist1000, 1000 * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(X->h_small.data() + 1000, X->d_accum + 2ull * N, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaMemcpyAsync(X->h_counters, X->d_counters, CTR_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nh = X->h_counters[CTR_HITS];
        const uint64_t nq = X->h_counters[CTR_QUEUE_NEED];  // largest screen queue any chunk wanted
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
        fprintf(stderr, "[drprg-cuda] map batch: %llu reads, %d chunks, screen queue %llu (largest chunk), probe survivors %llu, hits %llu\n",
                (unsigned long long)B->R.n_reads, B->n_chunks, X->h_counters[CTR_QUEUE_NEED], X->h_counters[CTR_SURVIVORS], (unsigned long long)nh);
    X->hist_on_host = !X->reduce_dst && !X->accum_shared;
    CK(cudaEventElapsedTime(&X->timings[0], X->ev[0], X->ev[1]));
    CK(cudaEventElapsedTime(&X->timings[1], X->ev[1], X->ev[2]));
    CK(cudaEventElapsedTime(&X->timings[2], X->ev[2], X->ev[3]));
    CK(cudaEventElapsedTime(&X->timings[3], X->ev[3], X->ev[4]));
    X->last_n_hits = nh;
    X->last_n_active = X->h_counters[CTR_ACTIVE];
    X->last_id_base = B->R.read_id_base;
    X->total_bases += B->total_bases;
    X->n_reads += B->R.n_reads;
    X->own_bases += B->total_bases;
    X->own_reads += B->R.n_reads;
    if (X->retain_hits && nh) {  // the kept hits of this batch, grouped by read, pandora order within a read
        const uint64_t na = X->last_n_active;
        std::vector<unsigned long long> key(nh);
        std::vector<uint8_t> kp(nh);
        std::vector<uint32_t> ar(na), ab(na), ac(na);
        CK(cudaMemcpy(key.data(), X->gkey.p, nh * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(kp.data(), X->gkept.p, nh, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(ar.data(), X->act_read.p, na * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(ab.data(), X->act_base.p, na * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(ac.data(), X->act_count.p, na * 4, cudaMemcpyDeviceToHost));
        for (uint64_t a = 0; a < na; ++a)
            for (uint32_t j = ab[a]; j < ab[a] + ac[a]; ++j) {
                if (!kp[j]) continue;  // kept hits sit in slices the cluster kernels sorted
                const unsigned long long k = key[j];
                X->retained.push_back(RetainedHit{B->R.read_id_base + ar[a], (uint32_t)(k >> GKEY_KNODE_BITS) & ((1u << GKEY_START_BITS) - 1u),
                                                  (uint32_t)k & ((1u << GKEY_KNODE_BITS) - 1u), (uint16_t)(k >> 48),
                                                  (uint8_t)(((k >> 47) & 1ull) ^ 1ull)});
            }
    }
    if (n_hits) *n_hits = nh;
    if (n_kept) *n_kept = X->h_counters[CTR_KEPT];
}

void flush_scalars(drprg_index* X) {
    if (X->scalars_in_buffer) return;
    int32_t s[4] = {(int32_t)(X->total_bases & 0xffffff), (int32_t)(X->total_bases >> 24), (int32_t)(X->n_reads & 0xffffff),
                    (int32_t)(X->n_reads >> 24)};
    if (X->accum_shared && X->world > 1) {  // the other ranks have added their scalars (shard_done): this rank's join them
        launch_add_scalars(X->d_accum + X->n_accum - 4, s, 0);
        CK(cudaStreamSynchronize(0));
    } else {
        CK(cudaMemcpy(X->d_accum + X->n_accum - 4, s, sizeof s, cudaMemcpyHostToDevice));
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
        cudaStreamSynchronize(X->st_ml);
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
        launch_flag_wait(reinterpret_cast<uint32_t*>(X->d_accum + accum_flag_offset(X->n_accum)) + 1, X->epoch * (uint32_t)(X->world - 1), 0);
    const bool reuse_hist = X->hist_on_host;  // downloaded at the end of the last map_batch, accumulators untouched since
    if (!reuse_hist) flush_scalars(X);
    if (!X->st_ml) {
        CK(cudaStreamCreateWithFlags(&X->st_ml, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&X->st_gt, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&X->st_acc, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&X->ev_acc[0], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&X->ev_acc[1], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&X->ev_acc[2], cudaEventDisableTiming));
        CK(cudaMalloc(&X->d_thresh_f64, sizeof(double)));
        CK(cudaMalloc(&X->d_thresh_i32, sizeof(int)));
    }
    // On the critical path the host only needs the 1000-bin coverage histogram (built on the device), the locus read
    // counts and the scalars: 4 KB.  The full accumulator (0.3 MB, pinned destination) is needed when the ML paths are
    // verified; it comes down on its own stream, ordered after whatever produced the accumulator on `st` (map_batch, or
    // the caller's allreduce).
    X->h_acc.resize(X->n_accum);
    CK(cudaEventRecord(X->ev_acc[0], st));
    CK(cudaStreamWaitEvent(X->st_acc, X->ev_acc[0], 0));
    CK(cudaMemcpyAsync(X->h_acc.data(), X->d_accum, X->n_accum * 4, cudaMemcpyDeviceToHost, X->st_acc));
    CK(cudaEventRecord(X->ev_acc[1], X->st_acc));
    uint64_t total_bases = X->total_bases;  // this process's batches; after an allreduce the summed scalars are read back
    if (!reuse_hist) {
        launch_cov_hist(X->d_accum, N, X->d_is_terminal, X->d_knode_locus, X->d_accum + 2ull * N, X->d_hist1000, st);
        X->h_small.resize(1000 + (size_t)P + 4);
        CK(cudaMemcpyAsync(X->h_small.data(), X->d_hist1000, 1000 * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(X->h_small.data() + 1000, X->d_accum + 2ull * N, ((size_t)P + 4) * 4, cudaMemcpyDeviceToHost, st));
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
    launch_node_prob(X->d_accum, N, X->d_is_terminal, MP, X->d_prob.p, st);
    launch_prob_hist(X->d_prob.p, N, X->d_is_terminal, X->d_knode_locus, X->d_accum + 2ull * N, X->d_hist, st);
    bool any_present = false;
    for (uint32_t l = 0; l < P; ++l) any_present = any_present || locus_reads[l] > 0;
    // the threshold (valley of the 200-bin histogram) is found on the device too: the ML-path kernel reads it from
    // device memory and starts without a host round trip; the host picks the value up later
    launch_prob_thresh(X->d_hist, any_present, X->fit.thresh, X->d_thresh_f64, X->d_thresh_i32, st);
    X->h_thresh.resize(1);
    CK(cudaMemcpyAsync(X->h_thresh.data(), X->d_thresh_i32, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(X->ev_acc[2], st));
    MP.thresh = (double)X->fit.thresh;  // placeholder for kernels that do not read it (S8); S7 uses d_thresh_f64
    lap(1);
    // ---- S7 on the device: the ML-path kernel is a latency chain per locus (~0.4 ms).  It only decides which loci
    // are reported and whether the path spells alleles the site tables lack (rare), so it runs on its own stream
    // while S8 (per-allele statistics + likelihoods) and the VCF text are produced SPECULATIVELY for the common
    // outcome "every locus with reads is present, no extra records"; the outcome is verified afterwards and
    // anything that deviates is redone on the slow path.
    if (!X->ev_ml[0]) {
        CK(cudaEventCreate(&X->ev_ml[0]));
        CK(cudaEventCreate(&X->ev_ml[1]));
    }
    X->h_path.resize(N);
    X->h_plen.resize(P);
    X->h_done.resize(P);
    std::fill(X->h_done.begin(), X->h_done.end(), 0u);
    CK(cudaStreamWaitEvent(X->st_ml, X->ev_acc[2], 0));  // node scores and threshold are produced on `st`
    CK(cudaMemsetAsync(X->d_path.p, 0, (size_t)N * 4, X->st_ml));  // absent loci leave their slice unwritten
    CK(cudaEventRecord(X->ev_ml[0], X->st_ml));
    // The level-parallel kernel writes every locus's path straight into pinned host memory (UVA: the same pointers
    // are valid on the device) and raises a per-locus flag, so the host can verify the small loci while the big ones
    // are still running; the older kernels leave the paths in device memory and are copied back as a whole.
    const bool ml_streamed = launch_mlpath(
        P, X->d_knode_base, X->d_edge_off, X->d_edges, X->d_prob.p, X->d_accum + 2ull * N, MP, X->d_M.p, X->d_len.p, X->d_up.p, N,
        X->d_path.p, X->d_path_len.p, X->max_locus_knodes, X->max_locus_edges, X->d_needs_mean, X->d_locus_unit_off, X->d_unit_start,
        X->d_unit_nodes, X->mean_run_len, X->st_ml, X->d_locus_level_off, X->d_level_start, X->d_level_nodes, X->d_level_singles,
        X->h_path.data(), X->h_plen.data(), X->h_done.data(), X->d_thresh_f64);
    X->ml_in_flight = true;
    CK(cudaEventRecord(X->ev_ml[1], X->st_ml));
    CK(cudaGetLastError());
    if (!ml_streamed) {
        CK(cudaMemcpyAsync(X->h_path.data(), X->d_path.p, (size_t)N * 4, cudaMemcpyDeviceToHost, X->st_ml));
        CK(cudaMemcpyAsync(X->h_plen.data(), X->d_path_len.p, (size_t)P * 4, cudaMemcpyDeviceToHost, X->st_ml));
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
            for (void* p : {(void*)X->d_rec_off, (void*)X->d_allele_off, (void*)X->d_allele_kn})
                if (p) cudaFree(p);
            X->d_rec_off = to_device(G.rec_off);
            X->d_allele_off = to_device(G.allele_off);
            X->d_allele_kn = to_device(G.allele_kn);
            {   // the static columns of every record line and the slots of the sample columns (VCF text on the device)
                std::vector<char> prefix;
                std::vector<uint32_t> poff(1, 0), soff(1, 0);
                for (size_t i = 0; i < X->records.size(); ++i) {
                    const std::string& t = vcf_record_prefix(H, *X->records[i]);
                    prefix.insert(prefix.end(), t.begin(), t.end());
                    poff.push_back((uint32_t)prefix.size());
                    soff.push_back(soff.back() + (uint32_t)vcf_sample_column_bound(G.rec_off[i + 1] - G.rec_off[i]));
                }
                for (void* p : {(void*)X->d_vcf_prefix, (void*)X->d_vcf_prefix_off, (void*)X->d_vcf_slot_off})
                    if (p) cudaFree(p);
                X->d_vcf_prefix = to_device(prefix);
                X->d_vcf_prefix_off = to_device(poff);
                X->d_vcf_slot_off = to_device(soff);
                X->vcf_prefix_bytes = prefix.size();
                X->vcf_slot_bytes = soff.back();
                if (!X->d_vcf_ctl) CK(cudaMalloc(&X->d_vcf_ctl, 2 * sizeof(uint32_t)));
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
            DevGenotype DG{nr, na, X->d_rec_off, X->d_allele_off, X->d_allele_kn, u, u + na, u + 2 * (size_t)na, u + 3 * (size_t)na,
                           u + 4 * (size_t)na, u + 5 * (size_t)na, f, f + na, f + 2 * (size_t)na, X->d_gt_i32.p};
            // the statistics drprg's filters derive from the record come out of the same kernel (they stay on the device
            // until drprg_cuda_gt_filter_stats asks for them)
            DG.covg_gt = X->d_gt_i32.p + nr;
            DG.minor_gt = X->d_gt_i32.p + 2 * (size_t)nr;
            DG.frs = X->d_gt_f32.p;
            DG.sb_ratio = X->d_gt_f32.p + nr;
            DG.pdp = X->d_gt_f32.p + 2 * (size_t)nr;
            launch_genotype(X->d_accum, DG, MP, s8);
            // the record lines: formatted by the device into the host-mapped text buffer, right behind the header
            X->d_vcf_slots.ensure(X->vcf_slot_bytes + 1);
            X->d_vcf_line_len.ensure(nr);
            X->d_vcf_out_off.ensure((size_t)nr + 1);
            CK(cudaMemsetAsync(X->d_vcf_ctl, 0, 2 * sizeof(uint32_t), s8));
            DevVcfText VT{X->d_vcf_prefix, X->d_vcf_prefix_off, X->d_vcf_slot_off, X->d_vcf_slots.p, X->d_vcf_line_len.p,
                          X->d_vcf_out_off.p, X->h_vcf.data() + hl, (uint32_t)(X->vcf_prefix_bytes + X->vcf_slot_bytes), X->d_vcf_ctl,
                          X->d_vcf_ctl + 1};
            static const bool host_text = getenv("DRPRG_VCF_TEXT") && std::string(getenv("DRPRG_VCF_TEXT")) == "host";
            if (!host_text) launch_vcf_text(DG, VT, s8);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(X->h_vcf_ctl.data(), X->d_vcf_ctl, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s8));
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
    run_s8_and_format(X->st_gt);
    CK(cudaEventSynchronize(X->ev_acc[2]));  // long done: the threshold the device chose
    X->fit.thresh = X->h_thresh.data()[0];
    MP.thresh = (double)X->fit.thresh;
    lap(3);
    // ---- verify the speculation against the ML paths
    const double tw0 = now_ms();
    if (!ml_streamed) CK(cudaStreamSynchronize(X->st_ml));
    CK(cudaEventSynchronize(X->ev_acc[1]));  // the full accumulator is on the host from here on
    const double tw1 = now_ms();
    const uint32_t* path = X->h_path.data();
    const uint32_t* plen = X->h_plen.data();
    const volatile uint32_t* done = X->h_done.data();
    std::atomic<bool> ml_failed{false};
    auto wait_for_locus = [&](uint32_t l) {  // streamed mode: spin until the kernel has published locus l
        if (!ml_streamed) return true;
        for (uint64_t spin = 0; done[l] == 0u; ++spin) {
            if (ml_failed.load(std::memory_order_relaxed)) return false;
            if ((spin & 0xffffu) == 0xffffu && cudaStreamQuery(X->st_ml) != cudaErrorNotReady && done[l] == 0u) {
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
        const cudaError_t mle = cudaStreamSynchronize(X->st_ml);
        X->ml_in_flight = false;
        if (mle != cudaSuccess)
            throw std::runtime_error(std::string("ML-path kernel failed: ") + cudaGetErrorString(mle));
    }
    if (ml_failed.load()) throw std::runtime_error("the ML-path kernel ended without publishing every locus");
    {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, X->ev_ml[0], X->ev_ml[1]));
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
        run_s8_and_format(X->st_gt);
    }
    lap(5);
    X->have_gt = true;
}

void free_batch(drprg_batch* b) {
    if (!b) return;
    for (drprg_batch* sh : b->shards) free_batch(sh);
    b->shards.clear();
    for (auto& e : b->ev)
        if (e) cudaEventDestroy(e);
    if (b->owned) {
        if (b->d_words) g_pool.put(b->d_words, b->b_words, b->device);
        if (b->d_lens) g_pool.put(b->d_lens, b->b_lens, b->device);
        if (b->d_off) g_pool.put(b->d_off, b->b_off, b->device);
        if (b->d_seg_read) g_pool.put(b->d_seg_read, b->b_seg, b->device);
        if (b->d_seg_start) g_pool.put(b->d_seg_start, b->b_seg, b->device);
    }
    delete b;
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
    B->b_seg = sr.size() * 4;
    B->d_seg_read = (uint32_t*)g_pool.get(B->b_seg, X->device);
    B->d_seg_start = (uint32_t*)g_pool.get(B->b_seg, X->device);
    CK(cudaMemcpyAsync(B->d_seg_read, sr.data(), B->b_seg, cudaMemcpyHostToDevice, cs));
    CK(cudaMemcpyAsync(B->d_seg_start, ss.data(), B->b_seg, cudaMemcpyHostToDevice, cs));
    CK(cudaStreamSynchronize(cs));  // the staging vectors die with this scope
    B->R.seg_read = B->d_seg_read;
    B->R.seg_start = B->d_seg_start;
    B->R.n_segs = sr.size();
    B->R.seg_len = seg_len;
}

drprg_batch* upload_batch(drprg_index* X, const uint32_t* words, const uint64_t* word_off, uint32_t stride, const uint32_t* lens,
                          uint64_t n, uint64_t total_bases, uint32_t id_base, cudaStream_t st) {
    need_device(X);
    CK(cudaSetDevice(X->device));
    std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(new drprg_batch(), free_batch);
    B->owned = true;
    const uint64_t nwords = stride ? n * (uint64_t)stride : (n ? word_off[n] : 0);
    B->device = X->device;
    B->b_words = std::max<uint64_t>(1, nwords + 2) * 4;
    B->b_lens = std::max<uint64_t>(1, n) * 4;
    B->d_words = (uint32_t*)g_pool.get(B->b_words, X->device);
    B->d_lens = (uint32_t*)g_pool.get(B->b_lens, X->device);
    if (!stride) {
        B->b_off = (n + 1) * 8;
        B->d_off = (uint64_t*)g_pool.get(B->b_off, X->device);
    }
    const bool chunked = (st == nullptr) && nwords * 4 >= (8u << 20) && stride && stride * 16u <= SHORT_READ_MAX;
    cudaStream_t cs = st;
    if (chunked) {
        if (!X->st_copy) CK(cudaStreamCreateWithFlags(&X->st_copy, cudaStreamNonBlocking));
        cs = X->st_copy;
        B->n_chunks = 4;
    }
    if (!stride) CK(cudaMemcpyAsync(B->d_off, word_off, (n + 1) * 8, cudaMemcpyHostToDevice, cs));
    uint32_t ml = 0;
    for (int c = 0; c < B->n_chunks; ++c) {
        const uint64_t lo = n * (uint64_t)c / B->n_chunks, hi = n * (uint64_t)(c + 1) / B->n_chunks;
        B->chunk_lo[c] = lo;
        B->chunk_lo[c + 1] = hi;
        const uint64_t w0 = stride ? lo * stride : word_off[lo], w1 = stride ? hi * stride : word_off[hi];
        if (w1 > w0) CK(cudaMemcpyAsync(B->d_words + w0, words + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, cs));
        if (hi > lo) CK(cudaMemcpyAsync(B->d_lens + lo, lens + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, cs));
        if (chunked) {
            CK(cudaEventCreateWithFlags(&B->ev[c], cudaEventDisableTiming));
            CK(cudaEventRecord(B->ev[c], cs));
        }
        // the longest read only selects the kernel: a fixed stride that already bounds it needs no scan
        if (!(stride && stride * 16u <= SHORT_READ_MAX))
            for (uint64_t i = lo; i < hi; ++i) ml = std::max(ml, lens[i]);  // overlaps the copy just enqueued
    }
    if (stride && stride * 16u <= SHORT_READ_MAX) ml = stride * 16u;
    B->R = DevReads{B->d_words, B->d_off, stride, B->d_lens, n, id_base};
    B->total_bases = total_bases;
    B->max_len = ml;
    if (ml > SHORT_READ_MAX) build_segments(X, B.get(), lens, n, total_bases, cs);
    return B.release();
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
        R->reduce_dst = root->d_accum;  // UVA: the root's pointer is valid on the peer once access is enabled
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

drprg_batch* multi_upload(drprg_index* root, const uint32_t* words, const uint64_t* word_off, uint32_t stride, const uint32_t* lens,
                          uint64_t n, uint64_t total_bases, uint32_t id_base) {
    const size_t G = root->gpus.size();
    std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(new drprg_batch(), free_batch);
    B->shards.assign(G, nullptr);
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
    for (auto* sh : B->shards) sum += sh->total_bases;
    if (total_bases > sum) B->shards[G - 1]->total_bases += total_bases - sum;
    return B.release();
}

void multi_map_batch(drprg_index* root, drprg_batch* B, uint64_t* n_hits, uint64_t* n_kept) {
    const size_t G = root->gpus.size();
    if (B->shards.size() != G) throw std::runtime_error("the batch was not uploaded through this multi-GPU handle");
    std::vector<uint64_t> nh(G, 0), nk(G, 0);
    for_each_gpu(root, [&](size_t g, drprg_index* X) { map_batch(X, B->shards[g], 0, &nh[g], &nk[g]); });
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

// A reads file as a device-resident batch.  Strict 4-line FASTQ (plain or gzip) is parsed and packed ON THE DEVICE
// (ingest.cu); FASTA and anything unusual goes through the host parser and an upload.  DRPRG_HOST_INGEST=1 forces the
// host parser (tests compare the two).
struct FileBatch {
    drprg_batch* B = nullptr;
    uint64_t n_dropped = 0;
    uint32_t first_read_len = 0;
    bool on_device = false;
};
struct Inflated {  // a gzip reads file inflated ahead of time (batch mode)
    char* p = nullptr;
    size_t n = 0;
    std::string error;
    Inflated() = default;
    Inflated(const Inflated&) = delete;
    Inflated(Inflated&& o) noexcept : p(o.p), n(o.n), error(std::move(o.error)) { o.p = nullptr; }
    Inflated& operator=(Inflated&& o) noexcept {
        if (this != &o) {
            free(p);
            p = o.p;
            n = o.n;
            error = std::move(o.error);
            o.p = nullptr;
        }
        return *this;
    }
    ~Inflated() { free(p); }
};

// the packed reads an ingest left on the device, as a batch of this index
drprg_batch* batch_from_ingest(drprg_index* X, const IngestResult& I, uint32_t read_id_base) {
    std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(new drprg_batch(), free_batch);
    B->owned = true;
    B->device = X->device;
    B->d_words = I.d_words;
    B->d_lens = I.d_lens;
    B->d_off = I.d_word_off;
    B->b_words = I.b_words;
    B->b_lens = I.b_lens;
    B->b_off = I.b_off;
    B->R = DevReads{I.d_words, I.d_word_off, I.stride_words, I.d_lens, I.n_reads, read_id_base};
    B->total_bases = I.total_bases;
    B->max_len = I.stride_words ? I.stride_words * 16u : I.max_len;
    if (I.max_len > SHORT_READ_MAX) {  // the segment table is built from the lengths on the host
        std::vector<uint32_t> lens(I.n_reads);
        CK(cudaMemcpy(lens.data(), I.d_lens, I.n_reads * 4, cudaMemcpyDeviceToHost));
        build_segments(X, B.get(), lens.data(), I.n_reads, I.total_bases, 0);
    }
    return B.release();
}

FileBatch batch_from_file(drprg_index* X, const char* reads_path, uint32_t threads, const Inflated* pre = nullptr) {
    need_device(X);
    CK(cudaSetDevice(X->device));
    FileBatch F;
    if (is_multi(X)) {  // one shard of the reads per GPU
        PackedReads pr;
        load_reads_packed(reads_path, threads, pr);
        const uint64_t n = pr.lens.size();
        if (n > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
        F.B = multi_upload(X, pr.words.data(), pr.word_off.data(), 0, pr.lens.data(), n, pr.total_bases, 0);
        F.n_dropped = pr.n_dropped;
        F.first_read_len = pr.first_read_len;
        return F;
    }
    static const bool host_only = getenv("DRPRG_HOST_INGEST") != nullptr && atoi(getenv("DRPRG_HOST_INGEST")) != 0;
    // gzip: the whole stream is inflated on all host threads first (gzip_inflate.cpp; zlib's one-core gzread only for
    // streams the parallel decoder declines), then the text takes the same device path as a plain file
    Inflated local;
    if (!pre && !host_only && file_is_gzip(reads_path)) {
        inflate_file(reads_path, &local.p, &local.n);
        pre = &local;
    }
    IngestResult I;
    const int dev = X->device;
    if (!host_only && ingest_fastq_device(reads_path, X->device, threads, I, 0, [dev](size_t bytes) { return g_pool.get(bytes, dev); },
                                          pre ? pre->p : nullptr, pre ? pre->n : 0)) {
        std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(batch_from_ingest(X, I, 0), free_batch);
        F.B = B.release();
        F.n_dropped = I.n_dropped;
        F.first_read_len = I.first_read_len;
        F.on_device = true;
        return F;
    }
    PackedReads pr;
    load_reads_packed(reads_path, threads, pr);
    const uint64_t n = pr.lens.size();
    if (n > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
    F.B = upload_batch(X, pr.words.data(), pr.word_off.data(), 0, pr.lens.data(), n, pr.total_bases, 0, 0);
    CK(cudaStreamSynchronize(0));  // pr dies with this scope
    F.n_dropped = pr.n_dropped;
    F.first_read_len = pr.first_read_len;
    return F;
}

// A reads file of any size, mapped wave by wave: plain strict FASTQ (or a gzip file inflated into host memory) is cut at
// record starts into waves of ~1 GiB of text; every wave is framed on the host, uploaded (sequence lines only), packed and
// mapped into the sample's accumulators before the next one is read, so a 30 M-read file (9.4 GB of text, BASELINE
// config 3) needs 0.5 GiB of pinned and 1 GiB of device memory instead of the whole text, and files beyond the 8 GB limit
// of one ingest still take the fast path.  false = the general path (batch_from_file) must handle the file; a sample
// that was begun here is begun again there.
struct WaveTotals {
    uint64_t n = 0, dropped = 0, bases = 0, hits = 0, kept = 0;
    uint32_t first_len = 0;
    size_t waves = 0;
    double ms_ingest = 0, ms_map = 0;
};
bool map_file_in_waves(drprg_index* X, const char* reads_path, const drprg_map_opts* o, const Inflated* pre, WaveTotals& W) {
    static const bool off = [] {
        const char* h = getenv("DRPRG_HOST_INGEST");
        const char* d = getenv("DRPRG_INGEST");
        return (h && atoi(h) != 0) || (d && std::string(d) == "device");
    }();
    if (off) return false;
    // A multi-GPU handle maps the file on its root GPU: a file-fed sample is bound by the host's framing rate (~45 GB/s of
    // text on 16 cores against 1.9 ms of GPU time per 10 M reads), so sharding the waves would leave every GPU idle
    // anyway; read sharding pays for batches that are already packed (drprg_cuda_batch_upload).
    static const size_t wave_bytes = [] {
        const char* e = getenv("DRPRG_WAVE_BYTES");
        return e && atol(e) > 0 ? (size_t)atol(e) : (size_t)(1u << 30);
    }();
    TextSource F;
    struct Closer {
        int fd = -1;
        ~Closer() {
            if (fd >= 0) close(fd);
        }
    } closer;
    Inflated local;
    if (!pre && file_is_gzip(reads_path)) {  // gzip: inflated on all host threads first (gzip_inflate.cpp)
        inflate_file(reads_path, &local.p, &local.n);
        pre = &local;
    }
    if (pre) {
        F.mem = pre->p;
        F.size = pre->n;
    } else {
        closer.fd = open(reads_path, O_RDONLY);
        if (closer.fd < 0) throw std::runtime_error(std::string("cannot open ") + reads_path);
        F.fd = closer.fd;
        F.size = (size_t)lseek(closer.fd, 0, SEEK_END);
    }
    char first = 0;
    if (F.size < 8 || F.read(&first, 0, 1) != 1 || first != '@') return false;
    const uint32_t threads = o ? std::max(1u, o->threads) : 1u;
    const int dev = X->device;
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
        if (!ingest_fastq_text(S, dev, threads, I, 0, [dev](size_t bytes) { return g_pool.get(bytes, dev); })) return false;
        if (W.n + I.n_reads > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
        std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(batch_from_ingest(X, I, (uint32_t)W.n), free_batch);
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

int run_sample(drprg_index* X, const char* reads_path, const char* vcf_refs, const char* outdir, const drprg_map_opts* o,
               drprg_map_stats* stats, const Inflated* pre = nullptr) {
    need_device(X);
    const double t0 = now_ms();
    // like the reference (File::create of pandora.log comes first, src/lib.rs:592-593): an unusable outdir fails before
    // any GPU work is done
    std::ofstream log(std::string(outdir) + "/pandora.log");
    if (!log) throw std::runtime_error(std::string("cannot write ") + outdir + "/pandora.log");
    struct {
        uint64_t n_dropped, total_bases;
    } pr{0, 0};
    uint64_t nh = 0, nk = 0, n = 0;
    bool on_device = true;
    size_t waves = 0;
    double t1 = t0, wave_ingest_ms = -1, wave_map_ms = 0;
    WaveTotals W;
    if (map_file_in_waves(X, reads_path, o, pre, W)) {
        pr.n_dropped = W.dropped;
        pr.total_bases = W.bases;
        nh = W.hits;
        nk = W.kept;
        n = W.n;
        waves = W.waves;
        wave_ingest_ms = W.ms_ingest;  // ingest and map alternate wave by wave
        wave_map_ms = W.ms_map;
    } else {
        FileBatch F = batch_from_file(X, reads_path, o ? o->threads : 1, pre);
        std::unique_ptr<drprg_batch, void (*)(drprg_batch*)> B(F.B, free_batch);
        pr.n_dropped = F.n_dropped;
        pr.total_bases = B->total_bases;
        on_device = F.on_device;
        t1 = now_ms();
        sample_begin_any(X, o, F.first_read_len);
        n = B->R.n_reads;
        map_batch_any(X, B.get(), 0, &nh, &nk);
    }
    const double t2 = now_ms();
    genotype(X, vcf_refs, "sample");
    std::ofstream vcf(std::string(outdir) + "/pandora_genotyped.vcf");
    if (!vcf) throw std::runtime_error(std::string("cannot write ") + outdir + "/pandora_genotyped.vcf");
    vcf.write(X->h_vcf.data() + X->vcf_begin, (std::streamsize)X->vcf_len);
    const double t3 = now_ms();
    drprg_map_stats s{};
    s.n_reads = n;
    s.n_reads_dropped = pr.n_dropped;
    s.total_bases = pr.total_bases;
    s.n_hits = nh;
    s.n_hits_kept = nk;
    s.n_loci_present = (uint32_t)X->contigs.size();
    s.n_records = (uint32_t)X->records.size();
    s.exp_depth_covg = X->fit.E;
    s.ms_ingest = wave_ingest_ms >= 0 ? wave_ingest_ms : t1 - t0;
    s.ms_map = wave_ingest_ms >= 0 ? wave_map_ms : t2 - t1;
    s.ms_genotype = t3 - t2;
    s.ms_total = t3 - t0;
    if (stats) *stats = s;
    log << "drprg-cuda map: reads=" << n << " dropped=" << pr.n_dropped << " bases=" << pr.total_bases << " hits=" << nh
        << " kept=" << nk << " loci=" << s.n_loci_present << " records=" << s.n_records << " E=" << s.exp_depth_covg
        << " ingest=" << (waves ? "host-framed, " + std::to_string(waves) + " wave(s)" : on_device ? "device" : "host") << "\nkernel ms: sketch_lookup=" << X->timings[0] << " sort=" << X->timings[1] << " cluster=" << X->timings[2]
        << " coverage=" << X->timings[3] << "\nwall ms: ingest=" << s.ms_ingest << " map=" << s.ms_map
        << " genotype=" << s.ms_genotype << " total=" << s.ms_total << "\n";
    return 0;
}
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
    CK(cudaIpcGetMemHandle(&h, X->d_accum));
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
    API_BEGIN
    // gzip inputs are inflate-bound (one zlib stream = one core, ~0.6 s per million reads): the next few samples are
    // inflated on spare threads while the GPU works on the current one
    const size_t window = std::max<size_t>(1, std::min<size_t>({n, (size_t)(o && o->threads ? o->threads : 1), (size_t)8}));
    std::vector<std::future<Inflated>> ahead(n);
    auto prefetch = [&](size_t i) {
        if (i >= n || !file_is_gzip(reads_paths[i])) return;
        const std::string path = reads_paths[i];
        ahead[i] = std::async(std::launch::async, [path]() {
            Inflated r;
            try {
                inflate_file(path, &r.p, &r.n);
            } catch (const std::exception& e) {
                r.error = e.what();
            }
            return r;
        });
    };
    for (size_t i = 0; i < window; ++i) prefetch(i);
    for (size_t i = 0; i < n; ++i) {
        Inflated pre;
        if (ahead[i].valid()) pre = ahead[i].get();
        prefetch(i + window);
        if (!pre.error.empty()) throw std::runtime_error(pre.error);
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
    TextSource src;
    src.fd = open(path, O_RDONLY);
    if (src.fd < 0) throw std::runtime_error(std::string("cannot open ") + path);
    struct Closer {
        int fd;
        ~Closer() { close(fd); }
    } closer{src.fd};
    src.size = (size_t)lseek(src.fd, 0, SEEK_END);
    char first = 0;
    if (src.size < 8 || src.read(&first, 0, 1) != 1 || first != '@') return 0;
    std::vector<char> buf(src.size / 2 + 64);
    std::vector<FramedSlice> sl;
    if (!fastq_frame_text(src, threads, buf.data(), sl)) return 0;
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
    if (is_multi(X)) *out = multi_upload(X, words, word_off, stride_words, lens, n_reads, total_bases, read_id_base);
    else *out = upload_batch(X, words, word_off, stride_words, lens, n_reads, total_bases, read_id_base, (cudaStream_t)stream);
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
    *out = F.B;
    if (n_reads) *n_reads = F.B->R.n_reads;
    if (total_bases) *total_bases = F.B->total_bases;
    if (n_dropped) *n_dropped = F.n_dropped;
    if (first_read_len) *first_read_len = F.first_read_len;
    if (parsed_on_device) *parsed_on_device = F.on_device ? 1 : 0;
    return 0;
    API_END
}
void drprg_cuda_batch_free(drprg_batch* b) { free_batch(b); }

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
    *d_ptr = X->d_accum;
    *n_int32 = X->n_accum;
    return 0;
    API_END
}
int drprg_cuda_accum_download(drprg_index* X, int32_t* out, uint64_t n) {
    API_BEGIN need_device(X);
    if (n != X->n_accum) throw std::runtime_error("accumulator size mismatch");
    CK(cudaSetDevice(X->device));
    flush_scalars(X);
    CK(cudaMemcpy(out, X->d_accum, n * 4, cudaMemcpyDeviceToHost));
    return 0;
    API_END
}
int drprg_cuda_accum_upload(drprg_index* X, const int32_t* in, uint64_t n) {
    API_BEGIN need_device(X);
    if (n != X->n_accum) throw std::runtime_error("accumulator size mismatch");
    CK(cudaSetDevice(X->device));
    CK(cudaMemcpy(X->d_accum, in, n * 4, cudaMemcpyHostToDevice));
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

int64_t drprg_cuda_sketch_batch(drprg_index* X, drprg_batch* B, void* stream, uint32_t* read, uint32_t* start, uint64_t* hash,
                                uint8_t* strand, uint64_t cap) {
    try {
        need_device(X);
        CK(cudaSetDevice(X->device));
        cudaStream_t st = (cudaStream_t)stream;
        DBuf<unsigned long long> key, val;
        key.ensure(cap);
        val.ensure(cap);
        CK(cudaMemsetAsync(X->d_counters, 0, 16, st));
        for (auto& e : B->ev)
            if (e) CK(cudaStreamWaitEvent(st, e, 0));
        launch_sketch_only(B->R, X->H.w, X->H.k, key.p, val.p, X->d_counters, cap, X->sm_count, B->max_len, st);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(X->h_counters, X->d_counters, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        uint64_t n = X->h_counters[0];
        if (n > cap) {
            key.release();
            val.release();
            g_err = "sketch output capacity too small";
            return -(int64_t)n;
        }
        std::vector<unsigned long long> hk(n), hv(n);
        CK(cudaMemcpy(hk.data(), key.p, n * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(hv.data(), val.p, n * 8, cudaMemcpyDeviceToHost));
        key.release();
        val.release();
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
    struct Guard {
        DBuf<uint32_t>& a; DBuf<double>& b; DBuf<int32_t>& c; DBuf<float>& d;
        ~Guard() { a.release(); b.release(); c.release(); d.release(); }
    } guard{d_u32, d_f64, d_i32, d_f32};
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
    DiscoverOpts D;
    if (o) {
        if (o->covg_threshold) D.covg_threshold = o->covg_threshold;
        if (o->min_len) D.min_len = o->min_len;
        if (o->max_len) D.max_len = o->max_len;
        if (o->padding != 0xffffffffu) D.padding = o->padding;
        if (o->min_hits) D.min_hits = o->min_hits;
    }
    const std::vector<RetainedHit>* hits = &X->retained;
    std::vector<RetainedHit> all;
    if (X->gpus.size() > 1) {  // shards are contiguous read ranges: concatenation keeps the hits grouped by read
        for (drprg_index* g : X->gpus) all.insert(all.end(), g->retained.begin(), g->retained.end());
        hits = &all;
    }
    discover_candidates(X->H, X->present, X->mlpaths, X->h_acc.data(), *hits, D, X->discover);
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
    dv.release(); dout.release(); dl.release(); dr.release();
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
