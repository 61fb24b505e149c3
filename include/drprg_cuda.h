/* drprg_cuda.h — C ABI of the B200-native replacement for the `pandora map --genotype --local`
 * step of `drprg predict`.
 *
 * Reference interface replaced: Pandora::genotype_with(prg, vcf_ref, reads, outdir, args)
 *   /root/reference/src/lib.rs:580-642, called from /root/reference/src/predict.rs:296-302 with
 *   the argv of src/lib.rs:594-609 + src/predict.rs:288-294.  The callee writes
 *   <outdir>/pandora_genotyped.vcf (src/lib.rs:644-646) and <outdir>/pandora.log (src/lib.rs:592).
 *   Success <=> return 0 (the reference maps a non-zero exit status to
 *   DependencyError::ProcessError, src/lib.rs:629-641); drprg_cuda_last_error() carries the text the
 *   reference would have logged from stderr.
 *
 * All pointers are plain host pointers unless a parameter is documented as a device pointer.
 * No torch types cross this boundary.  Every function is thread-compatible (one index per thread).
 */
#ifndef DRPRG_CUDA_H
#define DRPRG_CUDA_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRPRG_CUDA_VERSION 100 /* 0.1.0 */

typedef struct drprg_index drprg_index; /* PRG + k-mer graphs + minimizer table, resident in HBM */
typedef struct drprg_batch drprg_batch; /* 2-bit packed reads, resident in HBM */

/* mirrors the pandora argv drprg builds: -t, -c, -I, -K, -g, --max-covg, --gt-conf (src/lib.rs:594-609,
 * src/predict.rs:288-294) plus pandora defaults drprg never overrides (0 = pandora default):
 * -E genotyping error rate 0.01, -m max_diff 250, -e error rate 0.11 (0.001 and 2k+1 under -I). */
typedef struct {
    uint32_t threads;          /* -t  (host threads for FASTQ parse/pack) */
    uint32_t min_cluster_size; /* -c  (drprg default 10, src/predict.rs:194-196) */
    uint8_t illumina;          /* -I */
    uint8_t debug;             /* -K */
    uint32_t genome_size;      /* -g  (drprg passes 4411532, src/lib.rs:36) */
    uint32_t max_covg;         /* --max-covg (drprg passes u32::MAX = never subsample) */
    double gt_conf;            /* --gt-conf (drprg passes 0) */
    double genotyping_error_rate;
    uint32_t max_diff;
    double error_rate;
} drprg_map_opts;

typedef struct {
    uint64_t n_reads, n_reads_dropped, total_bases;
    uint64_t n_hits, n_hits_kept;
    uint32_t n_loci_present, n_records;
    uint32_t exp_depth_covg;
    double ms_ingest, ms_map, ms_genotype, ms_total;
} drprg_map_stats;

/* ---- lifecycle ------------------------------------------------------------------------------- */
int drprg_cuda_version(void);
const char* drprg_cuda_last_error(void); /* thread-local, valid until the next call */
int drprg_cuda_device_count(void);

/* Parse the PRG text (pandora format, e.g. /root/reference/tests/cases/expected/dr.prg), sketch it with
 * (w,k), build k-mer graphs + minimizer hash table and upload them to `device`.  Replaces what
 * `pandora index` (src/lib.rs:479-510) writes and `pandora map` re-loads (dr.prg.kK.wW.idx, kmer_prgs/).
 * device = -1 builds a host-only handle for index introspection (no GPU needed); every compute entry point
 * refuses such a handle — there is no CPU fallback for the map path. */
int drprg_cuda_index_load(const char* prg_path, uint32_t w, uint32_t k, int device, drprg_index** out);
int drprg_cuda_index_load_text(const char* prg_text, uint32_t w, uint32_t k, int device, drprg_index** out);
void drprg_cuda_index_free(drprg_index*);
/* `pandora index` replacement (SURVEY 8f rank 3; Pandora::index_with, src/lib.rs:479-510, called at src/builder.rs:644-659
 * and per sample at src/predict.rs:281-284): writes <prg_path>.k{K}.w{W}.idx and kmer_prgs/NN/<locus>.k{K}.w{W}.gfa next to
 * the PRG in pandora's text layout — the files drprg's validate_index requires (src/predict.rs:400-418,
 * find_prg_index_in src/lib.rs:1222-1231).  Works on a host-only handle (device = -1). */
int drprg_cuda_index_write(drprg_index*, const char* prg_path);

/* ---- read sharding over the GPUs of one box (BASELINE config 3; SURVEY 8e) ------------------------------------------
 * (a) inside the library: ONE handle drives n_gpus devices (0 = all visible; devices = NULL means 0..n-1).  The index is
 * replicated, every batch is cut into one contiguous shard of reads per GPU, one host thread per GPU issues the
 * launches, and the coverage kernel of every non-root GPU adds straight into the root GPU's accumulator over NVLink
 * (peer-mapped memory, red.global.add: integer sums, bit-exact for any GPU count) — the path's only exchange step needs no
 * separate collective.  Every call that takes a drprg_index* works on such a handle (the drop-in call included), so the
 * reference's single blocking call (Pandora::genotype_with, src/lib.rs:580-590) can use the whole box.  Sharding pays for
 * batches that are already packed (drprg_cuda_batch_upload); a reads FILE is bound by the host's framing rate and is
 * mapped wave by wave on the root GPU. */
int drprg_cuda_index_load_multi(const char* prg_path, uint32_t w, uint32_t k, int n_gpus, const int* devices, drprg_index** out);
int drprg_cuda_index_n_gpus(drprg_index*);
/* (b) one PROCESS per GPU (torchrun / MPI style): the root rank exports its accumulator as a 64-byte CUDA IPC handle,
 * the other ranks attach it and from then on add their coverage into it over NVLink exactly as in (a).  Per sample every
 * rank calls sample_begin and map_batch on its shard; a non-root rank then calls shard_done (its scalars join the root's,
 * the root's arrival counter goes up); the root's drprg_cuda_genotype waits on the device for world_size - 1 arrivals. */
int drprg_cuda_shard_root(drprg_index*, int world_size, void* handle64_out);
int drprg_cuda_shard_attach(drprg_index*, int world_size, const void* handle64);
int drprg_cuda_shard_done(drprg_index*, void* stream);

/* ---- the drop-in call: one sample, files in, pandora_genotyped.vcf out -------------------------- */
int drprg_cuda_map_genotype(drprg_index*, const char* reads_path, const char* vcf_refs_fasta, const char* outdir,
                            const drprg_map_opts*, drprg_map_stats* out_stats /* may be NULL */);
/* config 5: independent samples, one after another on this index's GPU (sample-sharding across GPUs is
 * one process per GPU, each calling this on its share); the gzip files of the next few samples are inflated on host
 * threads of their own while a sample runs.  drprg_cuda_discover_batch is the same for the discover step. */
int drprg_cuda_map_genotype_batch(drprg_index*, size_t n, const char* const* reads_paths, const char* vcf_refs_fasta,
                                  const char* const* outdirs, const drprg_map_opts*, drprg_map_stats* out_stats /* n or NULL */);

/* ---- staged interface (multi-GPU read sharding, benches, parity tests) -------------------------- */
/* host 2-bit packer: ASCII reads (concatenated, off[n+1]) -> words/word_off/lens.  Base i of a read sits in
 * bits [30-2(i%16), 31-2(i%16)] of word i/16 (A0 C1 G2 T3).  A read with a non-ACGT base gets lens=0
 * (pandora drops such reads).  stride_words>0 => fixed stride (word_off may be NULL).  Returns words used. */
int64_t drprg_cuda_pack_reads(const uint8_t* ascii, const uint64_t* off, uint64_t n_reads, uint32_t stride_words,
                              uint32_t* words, uint64_t words_cap, uint64_t* word_off, uint32_t* lens);
/* read a fasta/fastq(.gz) file and pack it (host); caller frees with drprg_cuda_host_free */
int drprg_cuda_read_fastx(const char* path, uint32_t threads, uint32_t** words, uint64_t** word_off, uint32_t** lens,
                          uint64_t* n_reads, uint64_t* total_bases, uint32_t* first_read_len);
void drprg_cuda_host_free(void*);
/* host half of the file ingest (test hook, no GPU): frames a plain strict 4-line FASTQ on the IO threads exactly as
 * drprg_cuda_map_genotype does before the upload; *ascii = the sequence lines back to back in read order, *lens = their
 * lengths.  Returns 0 and *is_fastq = 0 for input the framer declines (FASTA, wrapped records, blank lines: the
 * general parser takes those).  Replaces the reads-file reader behind /root/reference/src/predict.rs:166-170. */
int drprg_cuda_frame_fastq(const char* path, uint32_t threads, uint8_t** ascii, uint32_t** lens, uint64_t* n_reads,
                           uint64_t* total_bases, int* is_fastq);

/* H2D copy of a packed batch (pinned staging inside).  read_id_base = global id of the batch's first read. */
int drprg_cuda_batch_upload(drprg_index*, const uint32_t* words, const uint64_t* word_off /* NULL if stride */,
                            uint32_t stride_words, const uint32_t* lens, uint64_t n_reads, uint64_t total_bases,
                            uint32_t read_id_base, void* stream, drprg_batch** out);
/* adopt device-resident arrays (no copy; caller keeps ownership) */
int drprg_cuda_batch_wrap_device(drprg_index*, const void* d_words, const void* d_word_off, uint32_t stride_words,
                                 const void* d_lens, uint64_t n_reads, uint64_t total_bases, uint32_t read_id_base,
                                 drprg_batch** out);
/* a reads file (fasta/fastq, plain or gzip: src/predict.rs:166-170) as a device-resident batch.  Strict 4-line FASTQ is
 * framed on the host, and only its sequence lines are sent to the device and 2-bit packed there; other inputs use the
 * host parser and an upload.  *parsed_on_device = 1 for the first path, 0 for the host parser. */
int drprg_cuda_batch_from_fastx(drprg_index*, const char* path, uint32_t threads, drprg_batch** out, uint64_t* n_reads,
                                uint64_t* total_bases, uint64_t* n_dropped, uint32_t* first_read_len, int* parsed_on_device);
void drprg_cuda_batch_free(drprg_batch*);

/* start a sample: zero the coverage accumulators, fix the options (thresholds depend on -c/-I and on the
 * length of the sample's first read, pandora's expected_number_kmers_in_short_read_sketch) */
int drprg_cuda_sample_begin(drprg_index*, const drprg_map_opts*, uint32_t first_read_len);
/* S1-S5 for one batch on `stream`: sketch -> lookup -> sort -> cluster/filter -> coverage (+=) */
int drprg_cuda_map_batch(drprg_index*, drprg_batch*, void* stream, uint64_t* n_hits, uint64_t* n_kept);
/* packed int32 accumulator [2*total_knodes coverage (fwd,rev interleaved) | n_loci locus read counts |
 * total_bases lo24,hi | n_reads lo24,hi]: device pointer + element count, for an in-place allreduce(sum)
 * across ranks (NCCL via torch.distributed) before genotyping.  Scalars are flushed by this call. */
int drprg_cuda_accum_device_ptr(drprg_index*, void** d_ptr, uint64_t* n_int32);
int drprg_cuda_accum_download(drprg_index*, int32_t* out, uint64_t n_int32);
int drprg_cuda_accum_upload(drprg_index*, const int32_t* in, uint64_t n_int32);
/* S6-S8 from the accumulators: parameters (host), ML path + genotype kernels; keeps results for the getters */
int drprg_cuda_genotype(drprg_index*, const char* vcf_refs_fasta /* NULL = top path */, const char* sample_name);
int drprg_cuda_write_vcf(drprg_index*, const char* path);
const char* drprg_cuda_vcf_text(drprg_index*);
/* the same text without a copy: pointer + length, valid until the next drprg_cuda_genotype on this handle */
const char* drprg_cuda_vcf_view(drprg_index*, uint64_t* len);

/* ---- one mapping pass for `pandora discover` and `pandora map` (SURVEY 8f rank 1) --------------------------------------
 * drprg runs pandora twice per sample; the first half of `pandora discover` (src/predict.rs:247-256 -> src/lib.rs:513-578) is
 * the same S1-S7 as the map step.  With hit retention switched on BEFORE the sample is mapped, drprg_cuda_discover_candidates
 * (after drprg_cuda_genotype) returns what pandora's local assembler needs, from the pass that ran anyway: per present locus
 * the maximum-likelihood sequence and its per-base coverage, the candidate regions (runs of coverage < covg_threshold with a
 * length in [min_len, max_len], padded) and per region the reads with >= min_hits kept hits inside it (read id, span on the
 * read, strand).  Fields left 0 take pandora discover's defaults (3, 1, 30, 2); padding 0xffffffff = default 22.
 * Retention keeps every kept hit (read id, hit key) in a store on its GPU, appended by a kernel at the end of each batch;
 * the reads over the regions are found there by a kernel, only the result (a few thousand entries) comes to the host. */
typedef struct {
    uint32_t covg_threshold, min_len, max_len, padding, min_hits;
} drprg_discover_opts;
typedef struct {
    uint32_t locus, start, end, pad_start, pad_end, n_reads; /* intervals on the locus's ML sequence, end exclusive */
    uint64_t read_off;                                      /* first entry of the region in the read arrays */
} drprg_candidate_region;
int drprg_cuda_retain_hits(drprg_index*, int on);
int drprg_cuda_discover_candidates(drprg_index*, const drprg_discover_opts* /* NULL = defaults */, uint32_t* n_regions,
                                   uint64_t* n_region_reads);
int drprg_cuda_discover_regions(drprg_index*, drprg_candidate_region* out /* n_regions */);
int drprg_cuda_discover_region_reads(drprg_index*, uint32_t* read, uint32_t* start, uint32_t* end, uint8_t* fwd /* n_region_reads each */);
const char* drprg_cuda_discover_consensus(drprg_index*, uint32_t locus, uint64_t* len); /* NULL: locus absent from the sample */
int drprg_cuda_discover_coverage(drprg_index*, uint32_t locus, uint32_t* covg /* consensus length */);

/* The second half of `pandora discover`: local assembly of every candidate region into de-novo alleles, on the GPU, from the
 * bases of the reads the map pass retained (hit retention keeps the 2-bit words of every read with a kept hit).  Call after
 * drprg_cuda_discover_candidates; refused without retention, before genotyping, and on one-process-per-GPU handles
 * (drprg_cuda_shard_root / _attach).  Per region (padded interval [ps, pe), core [s, e) on the ML sequence C): the
 * region reads' spans, reverse-complemented where fwd = 0, give the oriented 11-mers of a de Bruijn graph whose k-mers seen
 * at least min_dbg_dp times are solid; the anchors are the first solid pair (i, j), i outer, of C[ps+i, +11) inside the
 * left flank and C[pe-11-j, pe-j) inside the right flank, up to 10 each; every walk through solid k-mers from the start to
 * the end anchor (A, C, G, T order, cycles allowed, at most (pe-j) - (ps+i) + max_insertion bases) is enumerated, and more
 * than max_candidate_paths walks abandon the region.  The walks other than C[ps+i, pe-j) are the region's de-novo alleles,
 * sorted.  Fields left 0 take pandora's defaults (2, 25); max_insertion 0xffffffff = default 15; max_candidate_paths <= 64. */
typedef struct {
    uint32_t min_dbg_dp, max_insertion, max_candidate_paths;
} drprg_assemble_opts;
typedef struct {
    uint32_t region;  /* index into drprg_cuda_discover_regions */
    uint32_t a, b;    /* the consensus interval [a, b) the allele replaces */
    uint32_t length;  /* bases at `offset` in the bases buffer of drprg_cuda_discover_paths */
    uint64_t offset;
} drprg_denovo_path;
#define DRPRG_DENOVO_ASSEMBLED 0      /* walks found; none besides the consensus = the reads agree with it */
#define DRPRG_DENOVO_NO_ANCHOR 1      /* no solid anchor pair */
#define DRPRG_DENOVO_TOO_MANY_PATHS 2 /* more than max_candidate_paths walks: abandoned */
#define DRPRG_DENOVO_NO_PATH 3        /* anchors, but no walk between them */
int drprg_cuda_discover_assemble(drprg_index*, const drprg_assemble_opts* /* NULL = defaults */, uint32_t* n_paths,
                                 uint64_t* n_path_bases);
int drprg_cuda_discover_paths(drprg_index*, drprg_denovo_path* out /* n_paths */, char* bases /* n_path_bases */);
int drprg_cuda_discover_region_status(drprg_index*, uint8_t* status /* n_regions, DRPRG_DENOVO_* */);
/* the last assembly's shape: regions counted in a shared-memory k-mer table, regions whose pileup needed a table in global
 * memory, and the device time in ms of the two kernel launches (CUDA events) — 4 doubles */
int drprg_cuda_last_assemble_stats(drprg_index*, double* out4);

/* `pandora discover` for one sample in one blocking call (drprg src/predict.rs:247-256 -> src/lib.rs:513-578): the reads file
 * is mapped through the same ingest as drprg_cuda_map_genotype with hit retention switched on (the caller's setting is
 * restored afterwards), genotyped without --vcf-refs (the ML path does not depend on them), its candidate regions are
 * found and assembled as above, and <outdir>/denovo_paths.txt is written; no VCF.  The file [P: restates pandora 0.10's
 * writer and make_prg update's reader]:
 *     1 samples / Sample <sample> / <L> loci with denovo variants
 *     then per locus with a variant, in PRG order: its name, "<M> nodes", one "(<node id> [<start>, <end>) <seq>)" line per
 *     node of its ML local path (PRG-string coordinates, node ids = this library's local-node ranks), "<V> variants found",
 *     and one "<pos>\t<ref>\t<alt>" line per variant.
 * Variants: every de-novo allele is aligned to the consensus span it replaces (unit-cost edit distance; the traceback from
 * the end extends an open gap while that stays optimal, else prefers substitution, then deletion, then insertion); each
 * maximal run of non-match columns is one variant at its 1-based position on the ML sequence, a run with an empty side
 * anchored by the consensus base before it (after it when it starts at the span's first base).  Per locus the union over its regions, distinct, sorted by (pos, ref, alt).
 * NULL options take the defaults; refused on one-process-per-GPU handles. */
typedef struct {
    uint64_t n_reads, n_hits_kept, n_region_reads;
    uint32_t n_regions, n_assembled, n_no_anchor, n_too_many_paths, n_no_path; /* region statuses: DRPRG_DENOVO_* */
    uint32_t n_loci_with_variants, n_variants;
    double ms_ingest, ms_map, ms_ml_path, ms_discover, ms_total; /* wall clock; discover = regions + assembly + file */
} drprg_discover_stats;
int drprg_cuda_discover(drprg_index*, const char* sample, const char* reads_path, const char* outdir, const drprg_map_opts*,
                        const drprg_discover_opts*, const drprg_assemble_opts*, drprg_discover_stats* /* may be NULL */);
/* `pandora discover` for n independent samples, one after another on this index (the discover half of config 5, next to
 * drprg_cuda_map_genotype_batch): sample i gets exactly what drprg_cuda_discover(X, samples[i], reads_paths[i], outdirs[i],
 * ...) gives it, <outdirs[i]>/denovo_paths.txt byte for byte and out_stats[i].  As in the map batch, the gzip files of the
 * next few samples are inflated on host threads of their own while a sample runs.  The first failing sample stops the call:
 * it returns non-zero, drprg_cuda_last_error() names the sample's index and reads path, and the files of the samples before
 * it stay.  The caller's retention setting is restored.  n = 0 does nothing; n > 0 needs reads_paths and outdirs.  Refused
 * on host-only and one-process-per-GPU handles; a drprg_cuda_index_load_multi handle maps each file on its root GPU. */
int drprg_cuda_discover_batch(drprg_index*, size_t n, const char* const* samples /* NULL = "sample" each */,
                              const char* const* reads_paths, const char* const* outdirs, const drprg_map_opts*,
                              const drprg_discover_opts*, const drprg_assemble_opts*, drprg_discover_stats* out_stats /* n or NULL */);

/* ---- introspection / parity hooks (same .so, used by tests and bench) --------------------------- */
/* pandora's hash64 on a 2k-bit k-mer and its inverse (the k-mer screen is built from the inverse): host functions */
uint64_t drprg_cuda_hash64(uint64_t kmer, uint32_t k);
uint64_t drprg_cuda_hash64_inverse(uint64_t hash, uint32_t k);
typedef struct {
    uint32_t w, k, n_loci, total_knodes;
    uint64_t n_records, n_edges, n_path_intervals;
    uint32_t table_slots, filter_words;
} drprg_index_info;
int drprg_cuda_index_info(drprg_index*, drprg_index_info*);
const char* drprg_cuda_locus_name(drprg_index*, uint32_t locus);
int drprg_cuda_index_knode_base(drprg_index*, uint32_t* out /* n_loci+1 */);
int drprg_cuda_index_knodes(drprg_index*, uint64_t* hash, uint8_t* strand, uint32_t* n_out, uint32_t* n_iv);
int drprg_cuda_index_edges(drprg_index*, uint32_t* edges /* global ids */);
int drprg_cuda_index_paths(drprg_index*, uint32_t* iv_start, uint32_t* iv_len);
int drprg_cuda_index_records(drprg_index*, uint64_t* hash, uint32_t* prg, uint32_t* knode, uint8_t* strand);
int drprg_cuda_index_min_path_length(drprg_index*, uint32_t* out /* n_loci */);
/* the k-mer screen's Bloom filters as the index builds them (k = 15; empty otherwise): over the indexed 15-mers of both
 * orientations and over their 14-mers, in screen_filter_insert's layout.  Pass NULL filters to learn the word counts;
 * both are 0 when the index keeps the sketch kernels. */
int drprg_cuda_index_screen_filters(drprg_index*, uint32_t* kfilter, uint32_t* kfilter_words, uint32_t* kfilter14,
                                    uint32_t* kfilter14_words);
/* S1 only: all (w,k)-minimizers of the batch, ordered (read, start); returns count (or <0) */
int64_t drprg_cuda_sketch_batch(drprg_index*, drprg_batch*, void* stream, uint32_t* read, uint32_t* start,
                                uint64_t* hash, uint8_t* strand, uint64_t cap);
/* hits of the last drprg_cuda_map_batch, sorted (read, prg, fwd first, start, knode) */
int64_t drprg_cuda_last_hits(drprg_index*, uint32_t* read, uint32_t* start, uint32_t* prg, uint32_t* knode,
                             uint8_t* fwd, uint8_t* kept, uint64_t cap);
/* genotype results: out[11] = E, bin, nb_p, nb_r, e_rate, thresh, covg, min_kmer_covg, mean, var, num_reads */
int drprg_cuda_gt_params(drprg_index*, double* out);
int64_t drprg_cuda_gt_mlpath(drprg_index*, uint32_t locus, uint32_t* out, uint64_t cap); /* -1: locus absent */
int drprg_cuda_gt_counts(drprg_index*, uint32_t* n_records, uint32_t* n_alleles, uint64_t* n_allele_knodes);
int drprg_cuda_gt_records(drprg_index*, uint32_t* locus, uint32_t* pos, uint32_t* n_alleles, int32_t* gt, double* gt_conf);
int drprg_cuda_gt_alleles(drprg_index*, double* lik, double* gaps, uint32_t* mean_fwd, uint32_t* mean_rev,
                          uint32_t* med_fwd, uint32_t* med_rev, uint32_t* sum_fwd, uint32_t* sum_rev, uint32_t* n_knodes);
int drprg_cuda_gt_allele_knodes(drprg_index*, uint32_t* out);
/* S8's likelihood / GT / GT_CONF kernel on caller-supplied per-allele rows: rec_off[n_records+1] -> alleles, per allele the
 * MEAN_FWD_COVG, MEAN_REV_COVG and GAPS a pandora VCF record carries (e.g. /root/reference/tests/cases/predict/in.vcf), the
 * sample's integer expected depth E, -E error rate and --gt-conf.  Outputs lik[n_alleles], gt[n_records] (-1 = null call),
 * gt_conf[n_records] and — optional, NULL to skip — the filter statistics described at drprg_cuda_gt_filter_stats.  This
 * is the genotype_kernel of the product path, so the reference's VCF fixtures check it directly. */
int drprg_cuda_genotype_rows(int device, uint32_t n_records, const uint32_t* rec_off, const uint32_t* mean_fwd,
                             const uint32_t* mean_rev, const double* gaps, uint32_t exp_depth, double genotyping_error_rate,
                             double min_gt_conf, float minor_af, double* lik, int32_t* gt, double* gt_conf, int32_t* covg_gt,
                             float* frs, float* sb_ratio, int32_t* minor_gt, float* pdp);
/* SURVEY 8f rank 4: the per-record statistics drprg's Filterer (src/filter.rs:212-301) and MinorAllele (src/minor.rs:70-127)
 * derive from a pandora record come out of the genotype kernel itself, in their f32 arithmetic and after drprg's nulling of
 * calls without depth (src/predict.rs:440-444): covg_gt = Filterer::_covg_for_gt; frs = VcfExt::fraction_read_support
 * (src/lib.rs:980-1011; NaN = None); sb_ratio = the ratio has_strand_bias compares with --min-strand-bias (NaN = None);
 * minor_gt = the allele check_for_minor_alternate would switch the call to (-1 = none) for --maf minor_af; pdp[n_alleles] =
 * VcfExt::depth_proportions, the PDP tag (src/lib.rs:1165-1174; NaN when the position has no depth).  Rust stays the
 * source of truth for the thresholds; these are the inputs of its comparisons, saving the BCF round trip in batch mode. */
int drprg_cuda_gt_filter_stats(drprg_index*, int32_t* covg_gt, float* frs, float* sb_ratio, int32_t* minor_gt, float* pdp);
/* --maf for minor_gt (default: drprg's own, 1.0 or 0.1 with -I, src/minor.rs:11-12,26-33); takes effect at the next genotype */
int drprg_cuda_set_minor_af(drprg_index*, float minor_af);
/* kernel timing of the last map_batch in ms (CUDA events on its stream): [sketch_lookup, sort, cluster, coverage] */
int drprg_cuda_last_timings(drprg_index*, float* out4);
/* host wall time of the last drprg_cuda_genotype in ms: [accumulator download, parameter fit + log-prob histogram,
 * ML-path launch + speculative record list, genotype kernels + VCF text (overlapping the ML-path kernel),
 * wait for the ML paths + verification, slow-path redo (0 when the speculation held),
 * device time of the ML-path kernel (CUDA events on its stream)] — 7 doubles */
int drprg_cuda_last_genotype_timings(drprg_index*, double* out7);
/* the VCF writer's float formatting (printf "%g"); out needs 48 bytes.  Exposed so tests can pin it against printf. */
int drprg_cuda_format_g6(double v, char* out);
/* the same formatting as the DEVICE does it for the VCF record lines (genotype.cu): out = 48 bytes per value, len[i] its
 * length, refused[i] = 1 where the device formatter declines (exponent notation, rounding ties, -0, inf, nan: the host
 * formatter then writes the sample's text).  Test hook. */
int drprg_cuda_format_g6_device(int device, const double* v, uint32_t n, char* out, uint8_t* len, uint8_t* refused);
/* number of kernel launches issued by this library since load (for bench.py's gpu_launches) */
uint64_t drprg_cuda_launch_count(void);
/* measured warp-instructions per second of a pure 32-bit integer multiply-add / shift / logic loop on this index's GPU: the
 * issue-rate ceiling of the k-mer screen (which is bound by instruction issue, not by HBM); 0 on failure */
double drprg_cuda_issue_peak(drprg_index*);

#ifdef __cplusplus
}
#endif
#endif
