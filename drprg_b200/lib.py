"""ctypes binding of include/drprg_cuda.h (the in-container stand-in for the Rust `drprg-cuda`
crate, crates/drprg-cuda/src/lib.rs).  There is no CPU fallback: loading fails loudly if the CUDA
library has not been built, and every call fails if no GPU is visible."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("DRPRG_CUDA_LIB") or os.path.join(_HERE, "libdrprg_cuda.so")  # env override: A/B builds
_LIB = None


class DrprgCudaError(RuntimeError):
    pass


class MapOpts(C.Structure):
    _fields_ = [
        ("threads", C.c_uint32), ("min_cluster_size", C.c_uint32), ("illumina", C.c_uint8), ("debug", C.c_uint8),
        ("genome_size", C.c_uint32), ("max_covg", C.c_uint32), ("gt_conf", C.c_double),
        ("genotyping_error_rate", C.c_double), ("max_diff", C.c_uint32), ("error_rate", C.c_double),
    ]


class MapStats(C.Structure):
    _fields_ = [
        ("n_reads", C.c_uint64), ("n_reads_dropped", C.c_uint64), ("total_bases", C.c_uint64), ("n_hits", C.c_uint64),
        ("n_hits_kept", C.c_uint64), ("n_loci_present", C.c_uint32), ("n_records", C.c_uint32),
        ("exp_depth_covg", C.c_uint32), ("ms_ingest", C.c_double), ("ms_map", C.c_double), ("ms_genotype", C.c_double),
        ("ms_total", C.c_double),
    ]

    def asdict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class DiscoverOpts(C.Structure):
    _fields_ = [("covg_threshold", C.c_uint32), ("min_len", C.c_uint32), ("max_len", C.c_uint32), ("padding", C.c_uint32), ("min_hits", C.c_uint32)]


class CandidateRegion(C.Structure):
    _fields_ = [("locus", C.c_uint32), ("start", C.c_uint32), ("end", C.c_uint32), ("pad_start", C.c_uint32), ("pad_end", C.c_uint32),
                ("n_reads", C.c_uint32), ("read_off", C.c_uint64)]


class AssembleOpts(C.Structure):
    _fields_ = [("min_dbg_dp", C.c_uint32), ("max_insertion", C.c_uint32), ("max_candidate_paths", C.c_uint32)]


class DenovoPath(C.Structure):
    _fields_ = [("region", C.c_uint32), ("a", C.c_uint32), ("b", C.c_uint32), ("length", C.c_uint32), ("offset", C.c_uint64)]


class DiscoverStats(C.Structure):
    _fields_ = [
        ("n_reads", C.c_uint64), ("n_hits_kept", C.c_uint64), ("n_region_reads", C.c_uint64), ("n_regions", C.c_uint32),
        ("n_assembled", C.c_uint32), ("n_no_anchor", C.c_uint32), ("n_too_many_paths", C.c_uint32), ("n_no_path", C.c_uint32),
        ("n_loci_with_variants", C.c_uint32), ("n_variants", C.c_uint32), ("ms_ingest", C.c_double), ("ms_map", C.c_double),
        ("ms_ml_path", C.c_double), ("ms_discover", C.c_double), ("ms_total", C.c_double),
    ]

    def asdict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


# region status of discover_assemble (DRPRG_DENOVO_* of the header)
ASSEMBLED, NO_ANCHOR, TOO_MANY_PATHS, NO_PATH = 0, 1, 2, 3


class IndexInfo(C.Structure):
    _fields_ = [
        ("w", C.c_uint32), ("k", C.c_uint32), ("n_loci", C.c_uint32), ("total_knodes", C.c_uint32),
        ("n_records", C.c_uint64), ("n_edges", C.c_uint64), ("n_path_intervals", C.c_uint64),
        ("table_slots", C.c_uint32), ("filter_words", C.c_uint32),
    ]


def make_opts(threads=1, min_cluster_size=10, illumina=False, genome_size=4411532, gt_conf=0.0,
              genotyping_error_rate=0.01, max_diff=0, error_rate=0.0, debug=False):
    return MapOpts(threads, min_cluster_size, int(illumina), int(debug), genome_size, 0xFFFFFFFF, gt_conf,
                   genotyping_error_rate, max_diff, error_rate)


# every symbol include/drprg_cuda.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "drprg_cuda_version", "drprg_cuda_last_error", "drprg_cuda_device_count", "drprg_cuda_index_load",
    "drprg_cuda_index_load_text", "drprg_cuda_index_free", "drprg_cuda_index_load_multi", "drprg_cuda_index_n_gpus", "drprg_cuda_index_write",
    "drprg_cuda_shard_root", "drprg_cuda_shard_attach", "drprg_cuda_shard_done", "drprg_cuda_map_genotype", "drprg_cuda_map_genotype_batch",
    "drprg_cuda_pack_reads", "drprg_cuda_read_fastx", "drprg_cuda_frame_fastq", "drprg_cuda_batch_from_fastx", "drprg_cuda_host_free", "drprg_cuda_batch_upload",
    "drprg_cuda_batch_wrap_device", "drprg_cuda_batch_free", "drprg_cuda_sample_begin", "drprg_cuda_map_batch",
    "drprg_cuda_accum_device_ptr", "drprg_cuda_accum_download", "drprg_cuda_accum_upload", "drprg_cuda_genotype",
    "drprg_cuda_write_vcf", "drprg_cuda_vcf_text", "drprg_cuda_vcf_view", "drprg_cuda_index_info", "drprg_cuda_locus_name",
    "drprg_cuda_index_knode_base", "drprg_cuda_index_knodes", "drprg_cuda_index_edges", "drprg_cuda_index_paths",
    "drprg_cuda_index_records", "drprg_cuda_index_min_path_length", "drprg_cuda_index_screen_filters", "drprg_cuda_sketch_batch", "drprg_cuda_last_hits",
    "drprg_cuda_gt_params", "drprg_cuda_gt_mlpath", "drprg_cuda_gt_counts", "drprg_cuda_gt_records",
    "drprg_cuda_gt_alleles", "drprg_cuda_gt_allele_knodes", "drprg_cuda_genotype_rows", "drprg_cuda_gt_filter_stats", "drprg_cuda_set_minor_af", "drprg_cuda_retain_hits", "drprg_cuda_discover_candidates",
    "drprg_cuda_discover_regions", "drprg_cuda_discover_region_reads", "drprg_cuda_discover_consensus", "drprg_cuda_discover_coverage", "drprg_cuda_discover_assemble", "drprg_cuda_discover", "drprg_cuda_discover_batch", "drprg_cuda_discover_paths",
    "drprg_cuda_discover_region_status", "drprg_cuda_last_assemble_stats", "drprg_cuda_last_timings", "drprg_cuda_last_genotype_timings", "drprg_cuda_format_g6", "drprg_cuda_format_g6_device", "drprg_cuda_launch_count", "drprg_cuda_hash64", "drprg_cuda_hash64_inverse", "drprg_cuda_issue_peak",
]


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise DrprgCudaError(f"{SO_PATH} is missing: build it with `python -m drprg_b200.build` "
                                 "(there is no CPU fallback for the map path)")
        L = C.CDLL(SO_PATH)
        L.drprg_cuda_last_error.restype = C.c_char_p
        L.drprg_cuda_locus_name.restype = C.c_char_p
        L.drprg_cuda_vcf_text.restype = C.c_char_p
        L.drprg_cuda_vcf_view.restype = C.c_void_p
        L.drprg_cuda_discover_consensus.restype = C.c_void_p
        for f in ("drprg_cuda_pack_reads", "drprg_cuda_sketch_batch", "drprg_cuda_last_hits", "drprg_cuda_gt_mlpath"):
            getattr(L, f).restype = C.c_int64
        L.drprg_cuda_launch_count.restype = C.c_uint64
        L.drprg_cuda_issue_peak.restype = C.c_double
        for f in ("drprg_cuda_hash64", "drprg_cuda_hash64_inverse"):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_uint64, C.c_uint32]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _check(rc, what):
    if rc != 0:
        raise DrprgCudaError(f"{what}: {lib().drprg_cuda_last_error().decode()}")


def _discover_args(opts, discover_opts, assemble_opts):
    """the three option structs of the discover calls; the keyword dicts override the defaults field by field"""
    d = DiscoverOpts(**dict(dict(covg_threshold=0, min_len=0, max_len=0, padding=0xFFFFFFFF, min_hits=0), **(discover_opts or {})))
    a = AssembleOpts(**dict(dict(min_dbg_dp=0, max_insertion=0xFFFFFFFF, max_candidate_paths=0), **(assemble_opts or {})))
    return opts or make_opts(), d, a


def pack_reads(data, off, stride_words=0):
    """ASCII reads (uint8 data, uint64 off[n+1]) -> (words, word_off, lens) via the library's host packer."""
    L = lib()
    data = np.ascontiguousarray(data, np.uint8)
    off = np.ascontiguousarray(off, np.uint64)
    n = len(off) - 1
    lens = (off[1:] - off[:-1]).astype(np.int64)
    cap = int(n * stride_words) if stride_words else int(((lens + 15) // 16).sum())
    words = np.zeros(max(cap, 1), np.uint32)
    woff = np.zeros(n + 1, np.uint64)
    out_lens = np.zeros(max(n, 1), np.uint32)
    r = L.drprg_cuda_pack_reads(_p(data), _p(off), C.c_uint64(n), C.c_uint32(stride_words), _p(words), C.c_uint64(cap),
                                _p(woff), _p(out_lens))
    if r < 0:
        raise DrprgCudaError(L.drprg_cuda_last_error().decode())
    return words[:cap], woff, out_lens[:n]


def read_fastx(path, threads=8):
    """host parser (fasta/fastq, plain or gzip) -> (words, word_off, lens, n_reads, total_bases, first_read_len)"""
    L = lib()
    words, woff, lens = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint32)()
    n, tb, fl = C.c_uint64(), C.c_uint64(), C.c_uint32()
    _check(L.drprg_cuda_read_fastx(str(path).encode(), C.c_uint32(threads), C.byref(words), C.byref(woff), C.byref(lens),
                                   C.byref(n), C.byref(tb), C.byref(fl)), "drprg_cuda_read_fastx")
    try:
        o = np.ctypeslib.as_array(woff, (n.value + 1,)).copy()
        w = np.ctypeslib.as_array(words, (max(1, int(o[-1])),)).copy()[:int(o[-1])]
        l = np.ctypeslib.as_array(lens, (max(1, n.value),)).copy()[:n.value]
    finally:
        for p in (words, woff, lens):
            L.drprg_cuda_host_free(p)
    return w, o, l, n.value, tb.value, fl.value


def frame_fastq(path, threads=8):
    """host half of the file ingest (no GPU): (ascii uint8[total_bases], lens uint32[n]) or None when the framer declines"""
    L = lib()
    ascii_, lens = C.POINTER(C.c_uint8)(), C.POINTER(C.c_uint32)()
    n, tb, ok = C.c_uint64(), C.c_uint64(), C.c_int()
    _check(L.drprg_cuda_frame_fastq(str(path).encode(), C.c_uint32(threads), C.byref(ascii_), C.byref(lens), C.byref(n),
                                    C.byref(tb), C.byref(ok)), "drprg_cuda_frame_fastq")
    try:
        if not ok.value:
            return None
        a = np.ctypeslib.as_array(ascii_, (max(1, tb.value),)).copy()[:tb.value]
        l = np.ctypeslib.as_array(lens, (max(1, n.value),)).copy()[:n.value]
    finally:
        for p in (ascii_, lens):
            L.drprg_cuda_host_free(p)
    return a, l


class Batch:
    def __init__(self, index, handle, n_reads, keep=()):
        self.index, self.h, self.n_reads, self._keep = index, handle, n_reads, keep

    def free(self):
        if self.h:
            try:
                lib().drprg_cuda_batch_free(self.h)
            except Exception:
                pass
            self.h = None

    def __del__(self):
        self.free()


class Index:
    """PRG + k-mer graphs + minimizer table resident in HBM on one GPU."""

    def __init__(self, prg_path=None, w=11, k=15, device=0, text=None, n_gpus=None, devices=None):
        """n_gpus (0 = all visible) or an explicit device list makes ONE handle shard every batch over several GPUs of the
        box inside the library (drprg_cuda_index_load_multi)."""
        L = lib()
        h = C.c_void_p()
        if n_gpus is not None or devices is not None:
            devs = None if devices is None else (C.c_int * len(devices))(*devices)
            n = len(devices) if devices is not None else int(n_gpus)
            rc = L.drprg_cuda_index_load_multi(str(prg_path).encode(), w, k, C.c_int(n), devs, C.byref(h))
            device = devices[0] if devices else 0
        elif text is not None:
            rc = L.drprg_cuda_index_load_text(text.encode(), w, k, device, C.byref(h))
        else:
            rc = L.drprg_cuda_index_load(str(prg_path).encode(), w, k, device, C.byref(h))
        _check(rc, "drprg_cuda_index_load")
        self.h = h
        self.device = device
        info = IndexInfo()
        _check(L.drprg_cuda_index_info(self.h, C.byref(info)), "index_info")
        self.info = info
        self.w, self.k = info.w, info.k
        self.n_loci, self.total_knodes = info.n_loci, info.total_knodes
        self.names = [L.drprg_cuda_locus_name(self.h, C.c_uint32(i)).decode() for i in range(self.n_loci)]
        self.knode_base = np.zeros(self.n_loci + 1, np.uint32)
        L.drprg_cuda_index_knode_base(self.h, _p(self.knode_base))
        self.n_accum = 2 * self.total_knodes + self.n_loci + 4

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().drprg_cuda_index_free(self.h)
            except Exception:  # interpreter shutdown: module globals may already be gone
                pass
            self.h = None

    def __del__(self):
        self.close()

    def write_pandora_index(self, prg_path):
        """the files `pandora index` would leave next to the PRG: <prg>.k{K}.w{W}.idx and kmer_prgs/NN/<locus>.k{K}.w{W}.gfa"""
        _check(lib().drprg_cuda_index_write(self.h, str(prg_path).encode()), "drprg_cuda_index_write")

    @property
    def n_gpus(self):
        return int(lib().drprg_cuda_index_n_gpus(self.h))

    # ---- one process per GPU: the root rank's accumulator is the reduction target of the others ----
    def shard_root(self, world_size):
        """root rank: returns the 64-byte CUDA IPC handle of the accumulator for the other ranks"""
        buf = C.create_string_buffer(64)
        _check(lib().drprg_cuda_shard_root(self.h, C.c_int(world_size), buf), "drprg_cuda_shard_root")
        return buf.raw

    def shard_attach(self, world_size, handle):
        _check(lib().drprg_cuda_shard_attach(self.h, C.c_int(world_size), C.c_char_p(bytes(handle))), "drprg_cuda_shard_attach")

    def shard_done(self, stream=0):
        _check(lib().drprg_cuda_shard_done(self.h, C.c_void_p(stream)), "drprg_cuda_shard_done")

    # ---- introspection (parity with the oracle) ----
    def knodes(self):
        L, n = lib(), self.total_knodes
        hsh = np.zeros(n, np.uint64); strand = np.zeros(n, np.uint8)
        n_out = np.zeros(n, np.uint32); n_iv = np.zeros(n, np.uint32)
        L.drprg_cuda_index_knodes(self.h, _p(hsh), _p(strand), _p(n_out), _p(n_iv))
        edges = np.zeros(int(n_out.sum()), np.uint32)
        L.drprg_cuda_index_edges(self.h, _p(edges))
        ivs = np.zeros(int(n_iv.sum()), np.uint32); ivl = np.zeros(int(n_iv.sum()), np.uint32)
        L.drprg_cuda_index_paths(self.h, _p(ivs), _p(ivl))
        return dict(hash=hsh, strand=strand, n_out=n_out, n_iv=n_iv, edges=edges, iv_start=ivs, iv_len=ivl)

    def records(self):
        n = int(self.info.n_records)
        hsh = np.zeros(n, np.uint64); prg = np.zeros(n, np.uint32); kn = np.zeros(n, np.uint32); st = np.zeros(n, np.uint8)
        lib().drprg_cuda_index_records(self.h, _p(hsh), _p(prg), _p(kn), _p(st))
        return dict(hash=hsh, prg=prg, knode=kn, strand=st)

    def min_path_lengths(self):
        o = np.zeros(self.n_loci, np.uint32)
        lib().drprg_cuda_index_min_path_length(self.h, _p(o))
        return o

    # ---- staged pipeline ----
    def upload(self, words, word_off, lens, total_bases=None, stride_words=0, read_id_base=0, stream=0):
        words = np.ascontiguousarray(words, np.uint32)
        lens = np.ascontiguousarray(lens, np.uint32)
        woff = None if stride_words else np.ascontiguousarray(word_off, np.uint64)
        if total_bases is None:
            total_bases = int(lens.astype(np.uint64).sum())
        h = C.c_void_p()
        rc = lib().drprg_cuda_batch_upload(self.h, _p(words), _p(woff), C.c_uint32(stride_words), _p(lens),
                                           C.c_uint64(len(lens)), C.c_uint64(int(total_bases)), C.c_uint32(read_id_base),
                                           C.c_void_p(stream), C.byref(h))
        _check(rc, "drprg_cuda_batch_upload")
        return Batch(self, h, len(lens))

    def batch_from_fastx(self, path, threads=8):
        """a reads file as a device-resident batch: strict 4-line FASTQ (plain/gzip) is framed on the host and packed on the
        GPU (info["parsed_on_device"] is True), anything else goes through the host parser.  Returns (Batch, info)."""
        h = C.c_void_p()
        n, tb, nd = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        fl, dev = C.c_uint32(0), C.c_int(0)
        rc = lib().drprg_cuda_batch_from_fastx(self.h, str(path).encode(), C.c_uint32(threads), C.byref(h), C.byref(n), C.byref(tb),
                                               C.byref(nd), C.byref(fl), C.byref(dev))
        _check(rc, "drprg_cuda_batch_from_fastx")
        return Batch(self, h, n.value), dict(n_reads=n.value, total_bases=tb.value, n_dropped=nd.value, first_read_len=fl.value,
                                             parsed_on_device=bool(dev.value))

    def upload_ptrs(self, words_ptr, lens_ptr, n_reads, stride_words, total_bases, read_id_base=0, stream=0, woff_ptr=None):
        """H2D from raw host pointers (e.g. pinned torch tensors) without numpy staging."""
        h = C.c_void_p()
        rc = lib().drprg_cuda_batch_upload(self.h, C.c_void_p(words_ptr), C.c_void_p(woff_ptr) if woff_ptr else None,
                                           C.c_uint32(stride_words), C.c_void_p(lens_ptr), C.c_uint64(n_reads),
                                           C.c_uint64(int(total_bases)), C.c_uint32(read_id_base), C.c_void_p(stream), C.byref(h))
        _check(rc, "drprg_cuda_batch_upload")
        return Batch(self, h, n_reads)

    def wrap_device(self, d_words_ptr, d_lens_ptr, n_reads, stride_words, total_bases, read_id_base=0, d_woff_ptr=None, keep=()):
        h = C.c_void_p()
        rc = lib().drprg_cuda_batch_wrap_device(self.h, C.c_void_p(d_words_ptr), C.c_void_p(d_woff_ptr) if d_woff_ptr else None,
                                                C.c_uint32(stride_words), C.c_void_p(d_lens_ptr), C.c_uint64(n_reads),
                                                C.c_uint64(int(total_bases)), C.c_uint32(read_id_base), C.byref(h))
        _check(rc, "drprg_cuda_batch_wrap_device")
        return Batch(self, h, n_reads, keep)

    def sample_begin(self, opts=None, first_read_len=0):
        self.opts = opts or make_opts()
        _check(lib().drprg_cuda_sample_begin(self.h, C.byref(self.opts), C.c_uint32(first_read_len)), "sample_begin")

    def map_batch(self, batch, stream=0):
        nh, nk = C.c_uint64(), C.c_uint64()
        _check(lib().drprg_cuda_map_batch(self.h, batch.h, C.c_void_p(stream), C.byref(nh), C.byref(nk)), "map_batch")
        return nh.value, nk.value

    def sketch(self, batch, cap=None, stream=0):
        cap = int(cap or max(1024, batch.n_reads * 64))
        rd = np.zeros(cap, np.uint32); st = np.zeros(cap, np.uint32); hs = np.zeros(cap, np.uint64); sd = np.zeros(cap, np.uint8)
        n = lib().drprg_cuda_sketch_batch(self.h, batch.h, C.c_void_p(stream), _p(rd), _p(st), _p(hs), _p(sd), C.c_uint64(cap))
        if n < 0:
            raise DrprgCudaError(f"sketch_batch: {lib().drprg_cuda_last_error().decode()} ({n})")
        return dict(read=rd[:n], start=st[:n], hash=hs[:n], strand=sd[:n])

    def last_hits(self, n):
        a = {k: np.zeros(n, np.uint32) for k in ("read", "start", "prg", "knode")}
        fwd = np.zeros(n, np.uint8); kept = np.zeros(n, np.uint8)
        r = lib().drprg_cuda_last_hits(self.h, _p(a["read"]), _p(a["start"]), _p(a["prg"]), _p(a["knode"]), _p(fwd), _p(kept), C.c_uint64(n))
        if r < 0:
            raise DrprgCudaError("last_hits failed")
        a["fwd"], a["kept"] = fwd, kept
        return a

    def accum_device_ptr(self):
        p, n = C.c_void_p(), C.c_uint64()
        _check(lib().drprg_cuda_accum_device_ptr(self.h, C.byref(p), C.byref(n)), "accum_device_ptr")
        return p.value, n.value

    def accum_download(self):
        o = np.zeros(self.n_accum, np.int32)
        _check(lib().drprg_cuda_accum_download(self.h, _p(o), C.c_uint64(len(o))), "accum_download")
        return o

    def accum_upload(self, a):
        a = np.ascontiguousarray(a, np.int32)
        _check(lib().drprg_cuda_accum_upload(self.h, _p(a), C.c_uint64(len(a))), "accum_upload")

    def coverage(self):
        a = self.accum_download()
        n = self.total_knodes
        cov = a[: 2 * n].reshape(n, 2)
        sc = a[-4:].astype(np.int64)
        return dict(fwd=cov[:, 0].astype(np.uint32), rev=cov[:, 1].astype(np.uint32),
                    locus_reads=a[2 * n: 2 * n + self.n_loci].astype(np.uint32),
                    total_bases=int(sc[0] + (sc[1] << 24)), n_reads=int(sc[2] + (sc[3] << 24)))

    def genotype(self, vcf_refs=None, sample="sample"):
        _check(lib().drprg_cuda_genotype(self.h, str(vcf_refs).encode() if vcf_refs else None, sample.encode()), "genotype")

    def vcf(self):
        return lib().drprg_cuda_vcf_text(self.h).decode()

    def vcf_bytes(self):
        """the VCF text as bytes (no UTF-8 decode: the text is ~1 MB per sample)"""
        return lib().drprg_cuda_vcf_text(self.h)

    def vcf_view(self):
        """zero-copy view of the VCF text in the library's host buffer (valid until the next genotype call)"""
        n = C.c_uint64(0)
        p = lib().drprg_cuda_vcf_view(self.h, C.byref(n))
        return memoryview((C.c_char * n.value).from_address(p)) if n.value else memoryview(b"")

    def write_vcf(self, path):
        _check(lib().drprg_cuda_write_vcf(self.h, str(path).encode()), "write_vcf")

    def params(self):
        o = np.zeros(11, np.float64)
        lib().drprg_cuda_gt_params(self.h, _p(o))
        keys = ["E", "bin", "nb_p", "nb_r", "e_rate", "thresh", "covg", "min_kmer_covg", "mean", "var", "num_reads"]
        return dict(zip(keys, o.tolist()))

    def mlpath(self, locus):
        cap = int(self.knode_base[locus + 1] - self.knode_base[locus]) + 1
        o = np.zeros(cap, np.uint32)
        n = lib().drprg_cuda_gt_mlpath(self.h, C.c_uint32(locus), _p(o), C.c_uint64(cap))
        return None if n < 0 else o[:n].copy()

    def gt_records(self):
        L = lib()
        nr, na, nk = C.c_uint32(), C.c_uint32(), C.c_uint64()
        L.drprg_cuda_gt_counts(self.h, C.byref(nr), C.byref(na), C.byref(nk))
        n, na, nk = nr.value, na.value, nk.value
        locus = np.zeros(n, np.uint32); pos = np.zeros(n, np.uint32); nal = np.zeros(n, np.uint32)
        gt = np.zeros(n, np.int32); conf = np.zeros(n, np.float64)
        L.drprg_cuda_gt_records(self.h, _p(locus), _p(pos), _p(nal), _p(gt), _p(conf))
        lik = np.zeros(na, np.float64); gaps = np.zeros(na, np.float64)
        u = {k: np.zeros(na, np.uint32) for k in ("mean_fwd", "mean_rev", "med_fwd", "med_rev", "sum_fwd", "sum_rev", "n_knodes")}
        L.drprg_cuda_gt_alleles(self.h, _p(lik), _p(gaps), _p(u["mean_fwd"]), _p(u["mean_rev"]), _p(u["med_fwd"]), _p(u["med_rev"]),
                                _p(u["sum_fwd"]), _p(u["sum_rev"]), _p(u["n_knodes"]))
        kn = np.zeros(nk, np.uint32)
        L.drprg_cuda_gt_allele_knodes(self.h, _p(kn))
        d = dict(locus=locus, pos=pos, n_alleles=nal, gt=gt, gt_conf=conf, lik=lik, gaps=gaps, allele_knodes=kn)
        d.update(u)
        return d

    def issue_peak(self):
        """measured warp-instructions/s of a pure INT32 multiply-add / shift / logic loop on this GPU"""
        return float(lib().drprg_cuda_issue_peak(self.h))

    def filter_stats(self):
        """per-record statistics of drprg's Filterer / MinorAllele, computed by the genotype kernel (see the header)"""
        L = lib()
        nr, na, nk = C.c_uint32(), C.c_uint32(), C.c_uint64()
        L.drprg_cuda_gt_counts(self.h, C.byref(nr), C.byref(na), C.byref(nk))
        n, na = nr.value, na.value
        cg = np.zeros(n, np.int32); frs = np.zeros(n, np.float32); sb = np.zeros(n, np.float32)
        mg = np.zeros(n, np.int32); pdp = np.zeros(na, np.float32)
        _check(L.drprg_cuda_gt_filter_stats(self.h, _p(cg), _p(frs), _p(sb), _p(mg), _p(pdp)), "drprg_cuda_gt_filter_stats")
        return dict(covg_gt=cg, frs=frs, sb_ratio=sb, minor_gt=mg, pdp=pdp)

    # ---- discover's mapping front half from the map pass ----
    def retain_hits(self, on=True):
        lib().drprg_cuda_retain_hits(self.h, C.c_int(1 if on else 0))

    def discover_candidates(self, covg_threshold=0, min_len=0, max_len=0, padding=0xFFFFFFFF, min_hits=0):
        """after genotype(): {locus: (consensus, coverage)}, regions [(locus, start, end, pad_start, pad_end, reads)] with
        reads = [(read, start, end, fwd)]"""
        L = lib()
        o = DiscoverOpts(covg_threshold, min_len, max_len, padding, min_hits)
        nr, nrr = C.c_uint32(), C.c_uint64()
        _check(L.drprg_cuda_discover_candidates(self.h, C.byref(o), C.byref(nr), C.byref(nrr)), "drprg_cuda_discover_candidates")
        regs = (CandidateRegion * max(1, nr.value))()
        L.drprg_cuda_discover_regions(self.h, regs)
        n = nrr.value
        rd = np.zeros(n, np.uint32); st = np.zeros(n, np.uint32); en = np.zeros(n, np.uint32); fw = np.zeros(n, np.uint8)
        L.drprg_cuda_discover_region_reads(self.h, _p(rd), _p(st), _p(en), _p(fw))
        loci = {}
        for l in range(self.n_loci):
            ln = C.c_uint64()
            p = L.drprg_cuda_discover_consensus(self.h, C.c_uint32(l), C.byref(ln))
            if not p:
                continue
            cov = np.zeros(ln.value, np.uint32)
            L.drprg_cuda_discover_coverage(self.h, C.c_uint32(l), _p(cov))
            loci[l] = (C.string_at(p, ln.value).decode(), cov)
        regions = []
        for i in range(nr.value):
            r = regs[i]
            a, b = r.read_off, r.read_off + r.n_reads
            regions.append((r.locus, r.start, r.end, r.pad_start, r.pad_end,
                            list(zip(rd[a:b].tolist(), st[a:b].tolist(), en[a:b].tolist(), fw[a:b].tolist()))))
        return loci, regions

    def discover_assemble(self, min_dbg_dp=0, max_insertion=0xFFFFFFFF, max_candidate_paths=0):
        """after discover_candidates(): the local assembler on the GPU -> (status uint8[n_regions], paths) with paths =
        [(region, a, b, sequence)]: the de-novo alleles replacing consensus[a:b] of the region's locus, sorted per region"""
        L = lib()
        o = AssembleOpts(min_dbg_dp, max_insertion, max_candidate_paths)
        n, nb = C.c_uint32(), C.c_uint64()
        _check(L.drprg_cuda_discover_assemble(self.h, C.byref(o), C.byref(n), C.byref(nb)), "drprg_cuda_discover_assemble")
        out = (DenovoPath * max(1, n.value))()
        bases = C.create_string_buffer(max(1, nb.value))
        _check(L.drprg_cuda_discover_paths(self.h, out, bases), "drprg_cuda_discover_paths")
        st = self.last_assemble_stats()
        status = np.zeros(st["regions_shared"] + st["regions_global"], np.uint8)
        _check(L.drprg_cuda_discover_region_status(self.h, _p(status)), "drprg_cuda_discover_region_status")
        raw = bases.raw
        paths = [(p.region, p.a, p.b, raw[p.offset:p.offset + p.length].decode()) for p in out[:n.value]]
        return status, paths

    def last_assemble_stats(self):
        """regions counted in a shared-memory table / in a global one, and the device ms of the two kernel launches"""
        o = np.zeros(4, np.float64)
        lib().drprg_cuda_last_assemble_stats(self.h, _p(o))
        return dict(regions_shared=int(o[0]), regions_global=int(o[1]), ms_shared=float(o[2]), ms_global=float(o[3]))

    def discover(self, reads_path, outdir, opts=None, sample="sample", discover_opts=None, assemble_opts=None):
        """`pandora discover` for one sample: maps the reads file (hit retention on for this call only), finds and assembles
        the candidate regions and writes <outdir>/denovo_paths.txt; returns the stats dict.  discover_opts / assemble_opts:
        keyword dicts of discover_candidates / discover_assemble."""
        st = DiscoverStats()
        o, d, a = _discover_args(opts, discover_opts, assemble_opts)
        rc = lib().drprg_cuda_discover(self.h, sample.encode(), str(reads_path).encode(), str(outdir).encode(), C.byref(o), C.byref(d),
                                       C.byref(a), C.byref(st))
        _check(rc, "drprg_cuda_discover")
        return st.asdict()

    def discover_batch(self, samples, reads_paths, outdirs, opts=None, discover_opts=None, assemble_opts=None):
        """`pandora discover` for several samples on this resident index (drprg_cuda_discover_batch): sample i as
        discover(reads_paths[i], outdirs[i], sample=samples[i]) would run it, while the next gzip files are inflated ahead;
        samples=None names every sample "sample".  Returns one stats dict per sample.  The first failing sample raises,
        naming its index; the files of the samples before it stay."""
        n = len(reads_paths)
        if len(outdirs) != n or (samples is not None and len(samples) != n):
            raise ValueError("samples, reads_paths and outdirs must have one entry per sample")
        strs = lambda xs: (C.c_char_p * max(1, n))(*[str(x).encode() for x in xs])
        st = (DiscoverStats * max(1, n))()
        o, d, a = _discover_args(opts, discover_opts, assemble_opts)
        rc = lib().drprg_cuda_discover_batch(self.h, C.c_size_t(n), None if samples is None else strs(samples), strs(reads_paths),
                                             strs(outdirs), C.byref(o), C.byref(d), C.byref(a), st)
        _check(rc, "drprg_cuda_discover_batch")
        return [st[i].asdict() for i in range(n)]

    def set_minor_af(self, maf):
        lib().drprg_cuda_set_minor_af(self.h, C.c_float(maf))

    def last_timings(self):
        o = np.zeros(4, np.float32)
        lib().drprg_cuda_last_timings(self.h, _p(o))
        return dict(zip(("sketch_lookup", "sort", "cluster", "coverage"), o.tolist()))

    def last_genotype_timings(self):
        o = np.zeros(7, np.float64)
        lib().drprg_cuda_last_genotype_timings(self.h, _p(o))
        return dict(zip(("download", "fit", "launch_ml+records", "s8+vcf_text", "ml_wait+verify", "redo", "mlpath_kernel"), o.tolist()))

    # ---- the drop-in call ----
    def map_genotype(self, reads_path, vcf_refs, outdir, opts=None):
        st = MapStats()
        o = opts or make_opts()
        rc = lib().drprg_cuda_map_genotype(self.h, str(reads_path).encode(), str(vcf_refs).encode() if vcf_refs else None,
                                           str(outdir).encode(), C.byref(o), C.byref(st))
        _check(rc, "drprg_cuda_map_genotype")
        return st.asdict()


def genotype_rows(rec_off, mean_fwd, mean_rev, gaps, exp_depth, err=0.01, min_gt_conf=0.0, device=0, minor_af=1.0, stats=False):
    """the product's genotype_kernel on caller-supplied per-allele rows (parity hook for the reference's VCF fixtures);
    stats=True also returns the fused filter / minor-allele statistics"""
    rec_off = np.ascontiguousarray(rec_off, np.uint32)
    mf = np.ascontiguousarray(mean_fwd, np.uint32)
    mr = np.ascontiguousarray(mean_rev, np.uint32)
    g = np.ascontiguousarray(gaps, np.float64)
    nr, na = len(rec_off) - 1, int(rec_off[-1])
    assert len(mf) == na and len(mr) == na and len(g) == na
    lik = np.zeros(na, np.float64); gt = np.zeros(nr, np.int32); conf = np.zeros(nr, np.float64)
    cg = np.zeros(nr, np.int32); frs = np.zeros(nr, np.float32); sb = np.zeros(nr, np.float32)
    mg = np.zeros(nr, np.int32); pdp = np.zeros(na, np.float32)
    rc = lib().drprg_cuda_genotype_rows(C.c_int(device), C.c_uint32(nr), _p(rec_off), _p(mf), _p(mr), _p(g), C.c_uint32(int(exp_depth)),
                                        C.c_double(err), C.c_double(min_gt_conf), C.c_float(minor_af), _p(lik), _p(gt), _p(conf),
                                        _p(cg), _p(frs), _p(sb), _p(mg), _p(pdp))
    _check(rc, "drprg_cuda_genotype_rows")
    if stats:
        return lik, gt, conf, dict(covg_gt=cg, frs=frs, sb_ratio=sb, minor_gt=mg, pdp=pdp)
    return lik, gt, conf


def launch_count():
    return int(lib().drprg_cuda_launch_count())
