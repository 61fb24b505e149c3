//! Safe wrapper over `include/drprg_cuda.h`.
//!
//! Replaces `Pandora::genotype_with` (drprg `src/lib.rs:580-642`) for the map step of
//! `drprg predict` (`src/predict.rs:285-303`): same inputs (PRG, `--vcf-refs`, reads, outdir, the
//! `-t -w -k -c [-I] [-K]` options), same outputs (`<outdir>/pandora_genotyped.vcf`,
//! `<outdir>/pandora.log`), same error convention (an `Err` where the subprocess would have exited
//! non-zero).  NOTE: this crate is source only in this repository — the build container has no
//! Rust toolchain — and is kept deliberately small.
use std::ffi::{CStr, CString};
use std::os::raw::{c_char, c_int};
use std::path::Path;

#[repr(C)]
#[derive(Debug, Clone, Copy)]
pub struct MapOpts {
    pub threads: u32,
    pub min_cluster_size: u32,
    pub illumina: u8,
    pub debug: u8,
    pub genome_size: u32,
    pub max_covg: u32,
    pub gt_conf: f64,
    pub genotyping_error_rate: f64,
    pub max_diff: u32,
    pub error_rate: f64,
}

#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct MapStats {
    pub n_reads: u64,
    pub n_reads_dropped: u64,
    pub total_bases: u64,
    pub n_hits: u64,
    pub n_hits_kept: u64,
    pub n_loci_present: u32,
    pub n_records: u32,
    pub exp_depth_covg: u32,
    pub ms_ingest: f64,
    pub ms_map: f64,
    pub ms_genotype: f64,
    pub ms_total: f64,
}

/// `pandora discover` options drprg leaves at their defaults (src/predict.rs:236-245); 0 = pandora's default
/// (covg threshold 3, region length 1..30, >= 2 hits per read), padding u32::MAX = 22.
#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct DiscoverOpts {
    pub covg_threshold: u32,
    pub min_len: u32,
    pub max_len: u32,
    pub padding: u32,
    pub min_hits: u32,
}

/// A low-coverage interval of a locus's maximum-likelihood sequence (end exclusive) and where its reads start in
/// the arrays of `CandidateReads`.
#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct CandidateRegion {
    pub locus: u32,
    pub start: u32,
    pub end: u32,
    pub pad_start: u32,
    pub pad_end: u32,
    pub n_reads: u32,
    pub read_off: u64,
}

/// What one `discover` call did (`drprg_discover_stats`): region statuses are `DRPRG_DENOVO_*` counts, times are wall ms.
#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct DiscoverStats {
    pub n_reads: u64,
    pub n_hits_kept: u64,
    pub n_region_reads: u64,
    pub n_regions: u32,
    pub n_assembled: u32,
    pub n_no_anchor: u32,
    pub n_too_many_paths: u32,
    pub n_no_path: u32,
    pub n_loci_with_variants: u32,
    pub n_variants: u32,
    pub ms_ingest: f64,
    pub ms_map: f64,
    pub ms_ml_path: f64,
    pub ms_discover: f64,
    pub ms_total: f64,
}

/// Options of the local assembler (`drprg_assemble_opts`); 0 = pandora's default (min DBG depth 2, 25 candidate paths),
/// max_insertion u32::MAX = 15.  max_candidate_paths is at most 64.
#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct AssembleOpts {
    pub min_dbg_dp: u32,
    pub max_insertion: u32,
    pub max_candidate_paths: u32,
}

/// One de-novo allele as the C ABI lists it (`drprg_denovo_path`): it replaces `[a, b)` of its region's locus consensus;
/// its bases are `length` bytes at `offset` of the bases buffer.
#[repr(C)]
#[derive(Debug, Default, Clone, Copy)]
pub struct DenovoPath {
    pub region: u32,
    pub a: u32,
    pub b: u32,
    pub length: u32,
    pub offset: u64,
}

/// Region status of the local assembler (`DRPRG_DENOVO_*`).
pub const DENOVO_ASSEMBLED: u8 = 0;
pub const DENOVO_NO_ANCHOR: u8 = 1;
pub const DENOVO_TOO_MANY_PATHS: u8 = 2;
pub const DENOVO_NO_PATH: u8 = 3;

/// A de-novo allele: region index, the consensus interval `[a, b)` it replaces, its sequence.
#[derive(Debug, Default, Clone)]
pub struct DenovoAllele {
    pub region: u32,
    pub a: u32,
    pub b: u32,
    pub seq: Vec<u8>,
}

/// Reads overlapping the candidate regions: read id, span on the read, strand (parallel arrays).
#[derive(Debug, Default, Clone)]
pub struct CandidateReads {
    pub read: Vec<u32>,
    pub start: Vec<u32>,
    pub end: Vec<u32>,
    pub fwd: Vec<u8>,
}

/// What `Filterer::filter` (drprg src/filter.rs:212-301) and `MinorAllele` (src/minor.rs:70-127) derive from a record's
/// FORMAT tags, computed by the genotype kernel (one entry per VCF record, VCF order).
#[derive(Debug, Default, Clone)]
pub struct FilterStats {
    pub covg_gt: Vec<i32>,
    pub frs: Vec<f32>,
    pub sb_ratio: Vec<f32>,
    pub minor_gt: Vec<i32>,
    pub pdp: Vec<f32>,
}

#[repr(C)]
pub struct RawIndex {
    _private: [u8; 0],
}

extern "C" {
    fn drprg_cuda_version() -> c_int;
    fn drprg_cuda_last_error() -> *const c_char;
    fn drprg_cuda_device_count() -> c_int;
    fn drprg_cuda_index_load(prg_path: *const c_char, w: u32, k: u32, device: c_int, out: *mut *mut RawIndex) -> c_int;
    fn drprg_cuda_index_load_multi(
        prg_path: *const c_char,
        w: u32,
        k: u32,
        n_gpus: c_int,
        devices: *const c_int,
        out: *mut *mut RawIndex,
    ) -> c_int;
    fn drprg_cuda_index_n_gpus(idx: *mut RawIndex) -> c_int;
    fn drprg_cuda_index_write(idx: *mut RawIndex, prg_path: *const c_char) -> c_int;
    fn drprg_cuda_index_free(idx: *mut RawIndex);
    fn drprg_cuda_retain_hits(idx: *mut RawIndex, on: c_int) -> c_int;
    fn drprg_cuda_discover_candidates(
        idx: *mut RawIndex,
        opts: *const DiscoverOpts,
        n_regions: *mut u32,
        n_region_reads: *mut u64,
    ) -> c_int;
    fn drprg_cuda_discover_regions(idx: *mut RawIndex, out: *mut CandidateRegion) -> c_int;
    fn drprg_cuda_discover_region_reads(idx: *mut RawIndex, read: *mut u32, start: *mut u32, end: *mut u32, fwd: *mut u8) -> c_int;
    fn drprg_cuda_discover_consensus(idx: *mut RawIndex, locus: u32, len: *mut u64) -> *const c_char;
    fn drprg_cuda_discover_assemble(
        idx: *mut RawIndex,
        opts: *const AssembleOpts,
        n_paths: *mut u32,
        n_path_bases: *mut u64,
    ) -> c_int;
    fn drprg_cuda_discover(
        idx: *mut RawIndex,
        sample: *const c_char,
        reads_path: *const c_char,
        outdir: *const c_char,
        map_opts: *const MapOpts,
        discover_opts: *const DiscoverOpts,
        assemble_opts: *const AssembleOpts,
        stats: *mut DiscoverStats,
    ) -> c_int;
    fn drprg_cuda_discover_paths(idx: *mut RawIndex, out: *mut DenovoPath, bases: *mut c_char) -> c_int;
    fn drprg_cuda_discover_region_status(idx: *mut RawIndex, status: *mut u8) -> c_int;
    fn drprg_cuda_gt_counts(idx: *mut RawIndex, n_records: *mut u32, n_alleles: *mut u32, n_allele_knodes: *mut u64) -> c_int;
    fn drprg_cuda_gt_filter_stats(
        idx: *mut RawIndex,
        covg_gt: *mut i32,
        frs: *mut f32,
        sb_ratio: *mut f32,
        minor_gt: *mut i32,
        pdp: *mut f32,
    ) -> c_int;
    fn drprg_cuda_map_genotype(
        idx: *mut RawIndex,
        reads_path: *const c_char,
        vcf_refs_fasta: *const c_char,
        outdir: *const c_char,
        opts: *const MapOpts,
        out_stats: *mut MapStats,
    ) -> c_int;
}

#[derive(thiserror::Error, Debug)]
pub enum CudaError {
    /// mirrors DependencyError::ProcessError (drprg src/lib.rs:65-90)
    #[error("drprg-cuda failed: {0}")]
    ProcessError(String),
    #[error("path is not valid UTF-8 / contains NUL: {0}")]
    BadPath(String),
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(drprg_cuda_last_error()).to_string_lossy().into_owned() }
}

fn cpath(p: &Path) -> Result<CString, CudaError> {
    CString::new(p.to_string_lossy().as_bytes()).map_err(|_| CudaError::BadPath(p.to_string_lossy().into_owned()))
}

pub fn version() -> i32 {
    unsafe { drprg_cuda_version() }
}

pub fn device_count() -> i32 {
    unsafe { drprg_cuda_device_count() }
}

/// PRG + k-mer graphs + minimizer table resident in HBM on one GPU (or replicated on several: `load_multi`).
pub struct Index {
    raw: *mut RawIndex,
}

unsafe impl Send for Index {}

impl Index {
    /// Parses and sketches the PRG (milliseconds) and uploads it; replaces the `dr.prg.kK.wW.idx` +
    /// `kmer_prgs/` files `pandora map` would reload.  Works for `outdir/updated.dr.prg` too.
    pub fn load(prg: &Path, w: u32, k: u32, device: i32) -> Result<Self, CudaError> {
        let p = cpath(prg)?;
        let mut raw: *mut RawIndex = std::ptr::null_mut();
        let rc = unsafe { drprg_cuda_index_load(p.as_ptr(), w, k, device, &mut raw) };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(Index { raw })
    }

    /// The same handle driving `n_gpus` GPUs of the box (0 = all visible): batches that are already packed are read-sharded,
    /// the coverage kernel adds into the root GPU's accumulator over NVLink; a reads file is mapped on the root GPU.
    pub fn load_multi(prg: &Path, w: u32, k: u32, n_gpus: i32) -> Result<Self, CudaError> {
        if n_gpus == 1 {
            return Self::load(prg, w, k, 0);
        }
        let p = cpath(prg)?;
        let mut raw: *mut RawIndex = std::ptr::null_mut();
        let rc = unsafe { drprg_cuda_index_load_multi(p.as_ptr(), w, k, n_gpus, std::ptr::null(), &mut raw) };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(Index { raw })
    }

    pub fn n_gpus(&self) -> i32 {
        unsafe { drprg_cuda_index_n_gpus(self.raw) }
    }

    /// Replaces `Pandora::index_with` (drprg src/lib.rs:479-510): writes `<prg>.kK.wW.idx` and `kmer_prgs/` next to the
    /// PRG in pandora's layout (what `validate_index`, src/predict.rs:400-418, looks for).
    pub fn write_pandora_index(&self, prg: &Path) -> Result<(), CudaError> {
        let p = cpath(prg)?;
        if unsafe { drprg_cuda_index_write(self.raw, p.as_ptr()) } != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(())
    }

    /// Keep the sample's kept hits so that `discover_candidates` can be asked after `map_genotype` (the mapping front
    /// half of `Pandora::discover_with`, drprg src/lib.rs:513-578, from the pass that runs anyway).  Call before mapping.
    pub fn retain_hits(&mut self, on: bool) -> Result<(), CudaError> {
        if unsafe { drprg_cuda_retain_hits(self.raw, on as c_int) } != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(())
    }

    /// Candidate regions for pandora's local assembler and the reads over them.
    pub fn discover_candidates(&mut self, opts: Option<&DiscoverOpts>) -> Result<(Vec<CandidateRegion>, CandidateReads), CudaError> {
        let (mut n_regions, mut n_reads) = (0u32, 0u64);
        let o = opts.map_or(std::ptr::null(), |o| o as *const DiscoverOpts);
        if unsafe { drprg_cuda_discover_candidates(self.raw, o, &mut n_regions, &mut n_reads) } != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        let mut regions = vec![CandidateRegion::default(); n_regions as usize];
        let n = n_reads as usize;
        let mut reads = CandidateReads { read: vec![0; n], start: vec![0; n], end: vec![0; n], fwd: vec![0; n] };
        let rc = unsafe {
            drprg_cuda_discover_regions(self.raw, regions.as_mut_ptr())
                | drprg_cuda_discover_region_reads(
                    self.raw,
                    reads.read.as_mut_ptr(),
                    reads.start.as_mut_ptr(),
                    reads.end.as_mut_ptr(),
                    reads.fwd.as_mut_ptr(),
                )
        };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok((regions, reads))
    }

    /// pandora discover's local assembly of every candidate region, on the GPU, from the bases the map pass retained.  Call
    /// after `discover_candidates` (`n_regions` = its region count).  Returns the status of every region and the de-novo
    /// alleles, sorted within a region.
    pub fn discover_assemble(&mut self, opts: Option<&AssembleOpts>, n_regions: usize) -> Result<(Vec<u8>, Vec<DenovoAllele>), CudaError> {
        let (mut n_paths, mut n_bases) = (0u32, 0u64);
        let o = opts.map_or(std::ptr::null(), |o| o as *const AssembleOpts);
        if unsafe { drprg_cuda_discover_assemble(self.raw, o, &mut n_paths, &mut n_bases) } != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        let mut paths = vec![DenovoPath::default(); n_paths as usize];
        let mut bases = vec![0u8; n_bases as usize];
        let mut status = vec![0u8; n_regions];
        let rc = unsafe {
            drprg_cuda_discover_paths(self.raw, paths.as_mut_ptr(), bases.as_mut_ptr() as *mut c_char)
                | drprg_cuda_discover_region_status(self.raw, status.as_mut_ptr())
        };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        let alleles = paths
            .iter()
            .map(|p| DenovoAllele {
                region: p.region,
                a: p.a,
                b: p.b,
                seq: bases[p.offset as usize..(p.offset + p.length as u64) as usize].to_vec(),
            })
            .collect();
        Ok((status, alleles))
    }

    /// Drop-in for `Pandora::discover_with` (drprg src/lib.rs:513-578) for one sample: maps `reads` (hit retention on for
    /// this call only), assembles the candidate regions on the GPU and writes `<outdir>/denovo_paths.txt`.  Blocking.
    pub fn discover(&mut self, sample: &str, reads: &Path, outdir: &Path, opts: &MapOpts) -> Result<DiscoverStats, CudaError> {
        let s = CString::new(sample).map_err(|_| CudaError::ProcessError("sample name contains a NUL byte".into()))?;
        let (r, o) = (cpath(reads)?, cpath(outdir)?);
        let mut stats = DiscoverStats::default();
        let rc = unsafe {
            drprg_cuda_discover(self.raw, s.as_ptr(), r.as_ptr(), o.as_ptr(), opts, std::ptr::null(), std::ptr::null(), &mut stats)
        };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(stats)
    }

    /// The maximum-likelihood sequence of a locus in this sample (`None`: the locus is absent).
    pub fn discover_consensus(&self, locus: u32) -> Option<Vec<u8>> {
        let mut len = 0u64;
        let p = unsafe { drprg_cuda_discover_consensus(self.raw, locus, &mut len) };
        if p.is_null() {
            return None;
        }
        Some(unsafe { std::slice::from_raw_parts(p as *const u8, len as usize) }.to_vec())
    }

    /// Per-record statistics of the last `map_genotype` for drprg's filters (no BCF round trip).
    pub fn filter_stats(&self) -> Result<FilterStats, CudaError> {
        let (mut nr, mut na, mut nk) = (0u32, 0u32, 0u64);
        if unsafe { drprg_cuda_gt_counts(self.raw, &mut nr, &mut na, &mut nk) } != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        let n = nr as usize;
        let mut s = FilterStats { covg_gt: vec![0; n], frs: vec![0.0; n], sb_ratio: vec![0.0; n], minor_gt: vec![0; n], pdp: vec![0.0; na as usize] };
        let rc = unsafe {
            drprg_cuda_gt_filter_stats(self.raw, s.covg_gt.as_mut_ptr(), s.frs.as_mut_ptr(), s.sb_ratio.as_mut_ptr(), s.minor_gt.as_mut_ptr(), s.pdp.as_mut_ptr())
        };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(s)
    }

    /// Drop-in for `Pandora::genotype_with(prg, vcf_ref, reads, outdir, args)`.
    pub fn map_genotype(&mut self, vcf_ref: &Path, reads: &Path, outdir: &Path, opts: &MapOpts) -> Result<MapStats, CudaError> {
        let (r, v, o) = (cpath(reads)?, cpath(vcf_ref)?, cpath(outdir)?);
        let mut stats = MapStats::default();
        let rc = unsafe { drprg_cuda_map_genotype(self.raw, r.as_ptr(), v.as_ptr(), o.as_ptr(), opts, &mut stats) };
        if rc != 0 {
            return Err(CudaError::ProcessError(last_error()));
        }
        Ok(stats)
    }
}

impl Drop for Index {
    fn drop(&mut self) {
        unsafe { drprg_cuda_index_free(self.raw) }
    }
}

impl MapOpts {
    /// The options `Predict::run` passes to pandora (drprg src/predict.rs:288-294, src/lib.rs:594-609).
    pub fn for_predict(threads: u32, min_cluster_size: u32, illumina: bool, debug: bool) -> Self {
        MapOpts {
            threads,
            min_cluster_size,
            illumina: illumina as u8,
            debug: debug as u8,
            genome_size: 4_411_532, // MTB_GENOME_SIZE, src/lib.rs:36
            max_covg: u32::MAX,
            gt_conf: 0.0,
            genotyping_error_rate: 0.01,
            max_diff: 0,
            error_rate: 0.0,
        }
    }
}
