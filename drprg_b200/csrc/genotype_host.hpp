// Host-side pieces around the S7/S8 kernels: model parameter estimation (S6, tiny and branchy,
// SURVEY.md §8a row a6), reference-path threading, variant-site enumeration with the
// allele -> k-mer-node CSR the genotype kernel consumes, and the pandora_genotyped.vcf writer
// (/root/reference/src/lib.rs:644-646; schema /root/reference/tests/cases/predict/*.vcf).
#pragma once
#include <functional>
#include <map>
#include <set>
#include <tuple>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "prg_graph.hpp"

namespace drprg {

// Small persistent host thread pool (creating threads per call cost more than the work they did).
// parallel_for(n, fn) runs fn(0..n-1) on the pool plus the calling thread and rethrows the first error.
void parallel_for(size_t n, const std::function<void(size_t)>& fn, size_t max_threads = 8);
// the same on the larger, non-spinning pool used by ingest and gzip inflate (up to 64 threads of the rank's core share)
void parallel_for_io(size_t n, const std::function<void(size_t)>& fn, size_t max_threads = 64);

struct SampleOpts {
    uint32_t min_cluster_size = 10;
    bool illumina = false;
    uint32_t genome_size = 4411532;
    uint32_t max_diff = 250;
    double e_rate = 0.11;
    double gt_error_rate = 0.01;
    double gt_conf = 0.0;
    uint32_t window = 100;  // pandora max_num_kmers_to_average
    uint32_t threads = 1;
};

struct FitParams {
    uint32_t E = 0;
    bool bin = false;
    double nb_p = 0.015, nb_r = 2.0, e_rate = 0.11;
    int thresh = -25;
    uint32_t covg = 0, min_kmer_covg = 0;
    double mean = 0, var = 0;
    uint64_t num_reads = 0;
};

// cov: interleaved (fwd, rev) per global knode, already summed over ranks; saturates at 65535
// everything of estimate_parameters except the probability threshold (set from the device histogram)
FitParams fit_parameters(const HostIndex& H, const int32_t* cov, const int32_t* locus_reads, uint64_t total_bases,
                         const SampleOpts& o);
FitParams fit_parameters_hist(const HostIndex& H, const uint32_t* hist1000, const int32_t* locus_reads, uint64_t total_bases,
                              const SampleOpts& o);
int prob_threshold(const uint32_t* hist200);
double host_node_log_prob(const FitParams& P, uint32_t k, uint32_t f, uint32_t r, bool terminal);

struct SiteRecord {
    uint32_t locus = 0, pos = 0;  // pos 0-based on the reference path
    std::string ref;
    std::vector<std::string> alts;
    std::string vc, graphtype;
    std::vector<std::vector<uint32_t>> allele_kn;  // ranks within the locus, ref allele first
    mutable std::string text_prefix;               // cached VCF columns CHROM..FORMAT
};

// node path threading `seq` from node 0 to the sink (empty if none); top_path = first out-edges
std::vector<uint32_t> thread_sequence(const Locus& L, const std::string& seq);
std::vector<uint32_t> top_path(const Locus& L);
// biallelic records of one locus along `ref` (pandora build_vcf + allele k-mer mapping)
std::vector<SiteRecord> enumerate_sites(const HostIndex& H, uint32_t locus, const std::vector<uint32_t>& ref);
// local node path under an ML k-mer path (ranks)
std::vector<uint32_t> local_path_of(const Locus& L, const std::vector<uint32_t>& kpath);
// records the ML path spells but enumerate_sites did not (pandora add_sample_gt_to_vcf)
using SiteKeySet = std::set<std::tuple<uint32_t, std::string, std::string>>;  // (pos, ref, alt) of the biallelic records
void find_ml_path_records(const HostIndex& H, uint32_t locus, const std::vector<uint32_t>& ref,
                          const std::vector<uint32_t>& lpath, const SiteKeySet& known, std::vector<SiteRecord>& extra);
// sort + merge records sharing (pos, ref); anchor empty alleles
std::vector<SiteRecord> merge_records(const Locus& L, const std::vector<uint32_t>& ref, std::vector<SiteRecord> recs);
// coverage sanity filter of pandora add_consensus_path_to_fastaq: true = drop the locus
bool locus_coverage_outlier(const HostIndex& H, uint32_t locus, const std::vector<uint32_t>& kpath,
                            const std::vector<uint32_t>& lpath, const int32_t* cov, uint32_t global_covg);

// ---- discover's mapping front half from the map pass (discover.cpp, SURVEY 8f rank 1) ------------------------------
struct DiscoverOpts {  // pandora discover defaults (drprg overrides none of them)
    uint32_t covg_threshold = 3, min_len = 1, max_len = 30, padding = 22, min_hits = 2;
};
struct ReadCoordinate {
    uint32_t read, start, end;
    uint8_t fwd;
};
struct CandidateRegion {
    uint32_t locus = 0, start = 0, end = 0, pad_start = 0, pad_end = 0, n_reads = 0;
    uint64_t read_off = 0;
};
struct DiscoverResult {
    std::vector<std::string> consensus;           // per locus: ML sequence (empty when the locus is absent)
    std::vector<std::vector<uint32_t>> coverage;  // per locus: per-base coverage along it
    std::vector<std::vector<uint32_t>> local_path; // per locus: the local nodes the ML sequence spells
    std::vector<CandidateRegion> regions;         // ordered by locus, then position
    std::vector<ReadCoordinate> reads;            // per region, ordered by read id
};
std::vector<uint32_t> ml_path_base_coverage(const HostIndex& H, uint32_t locus, const std::vector<uint32_t>& kpath,
                                            const std::vector<uint32_t>& lpath, const int32_t* cov);
// the per-locus half: consensus, coverage, local path and candidate regions (reads left empty), and the consensus start of
// every global k-mer node on the ML path of a locus with regions (UINT32_MAX elsewhere) for the region-read kernel
void discover_regions(const HostIndex& H, const std::vector<char>& present, const std::vector<std::vector<uint32_t>>& mlpaths,
                      const int32_t* cov, const DiscoverOpts& o, DiscoverResult& R, std::vector<uint32_t>& cons_start);
// discover/denovo_paths.txt [P]: a de-novo allele replacing cons[a, b) as variants against the ML sequence (1-based pos,
// anchored so that neither allele is empty), and the file's text for the loci with variants
struct DenovoVariant {
    uint32_t pos;
    std::string ref, alt;
    bool operator<(const DenovoVariant& o) const { return std::tie(pos, ref, alt) < std::tie(o.pos, o.ref, o.alt); }
    bool operator==(const DenovoVariant& o) const { return pos == o.pos && ref == o.ref && alt == o.alt; }
};
void allele_variants(const std::string& cons, uint32_t a, uint32_t b, const std::string& allele, std::vector<DenovoVariant>& out);
std::string denovo_paths_text(const HostIndex& H, const std::string& sample, const DiscoverResult& D,
                              const std::vector<std::vector<DenovoVariant>>& variants /* per locus, sorted, distinct */);

// pandora-compatible index files next to the PRG (`pandora index` replacement, SURVEY 8f rank 3): <prg>.k{K}.w{W}.idx and
// kmer_prgs/NN/<locus>.k{K}.w{W}.gfa
void write_pandora_index(const HostIndex& H, const std::string& prg_path);

struct GenotypeArrays {  // flattened over records / alleles, device results copied back
    std::vector<uint32_t> rec_off, allele_off, allele_kn;
    std::vector<uint32_t> mean_fwd, mean_rev, med_fwd, med_rev, sum_fwd, sum_rev;
    std::vector<double> gaps, lik, gt_conf;
    std::vector<int32_t> gt;
};
void format_vcf(const HostIndex& H, const std::vector<const SiteRecord*>& recs, const GenotypeArrays& G,
                const std::vector<std::string>& contigs, const std::string& sample, std::string& out);

void format_vcf_header(const std::vector<std::string>& contigs, const std::string& sample, std::string& out);
const std::string& vcf_record_prefix(const HostIndex& H, const SiteRecord& r);  // CHROM .. FORMAT columns, cached
// upper bound of a record's sample column (GT : 6 integer vectors : GAPS : LIKELIHOOD : GT_CONF, newline) with na alleles
inline size_t vcf_sample_column_bound(size_t na) { return 16 + na * (6 * 12 + 2 * 28) + 40; }
size_t format_g6(double v, char* out);  // printf("%g") text of v, out has room for 40 chars
std::map<std::string, std::string> load_fasta(const std::string& path);

// fasta/fastq (plain or gzip) -> 2-bit packed reads
struct PackedReads {
    std::vector<uint32_t> words;
    std::vector<uint64_t> word_off;
    std::vector<uint32_t> lens;
    uint64_t total_bases = 0, n_dropped = 0;
    uint32_t first_read_len = 0;
};
void load_reads_packed(const std::string& path, uint32_t threads, PackedReads& out);
bool inflate_file(const std::string& path, char** out, size_t* n);  // malloc'ed; caller frees
bool file_is_gzip(const std::string& path);
int64_t pack_ascii(const uint8_t* ascii, const uint64_t* off, uint64_t n, uint32_t stride_words, uint32_t* words,
                   uint64_t words_cap, uint64_t* word_off, uint32_t* lens);

}  // namespace drprg
