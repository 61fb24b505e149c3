"""GPU parity tests proper: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on
the same seeded inputs.  Integer stages are compared bit-exactly; log-likelihoods at 1e-9 relative."""
import os

import numpy as np
import pytest

import oracle_py as O
from drprg_b200 import lib, sim
from helpers import TOY_PRG, TOY_REFS, assert_genotype_equal, long_reads_sample, panel_sample, reads_from_strings, small_panel

pytestmark = pytest.mark.gpu


def both_indexes(prg, w, k):
    return lib.Index(prg, w, k, device=0), O.Index(prg, w, k)


def gpu_sketch(gx, data, off, stride_words=0):
    words, woff, lens = lib.pack_reads(data, off, stride_words)
    b = gx.upload(words, woff, lens, stride_words=stride_words)
    return gx.sketch(b, cap=max(4096, len(data)))


def oracle_sketch_all(data, off, w, k):
    rd, st, hs, sd = [], [], [], []
    for i in range(len(off) - 1):
        h, s, d = O.sketch(data[int(off[i]):int(off[i + 1])].tobytes(), w, k)
        rd += [i] * len(h); st += s.tolist(); hs += h.tolist(); sd += d.tolist()
    return dict(read=np.array(rd, np.uint32), start=np.array(st, np.uint32), hash=np.array(hs, np.uint64), strand=np.array(sd, np.uint8))


def assert_sketch_equal(a, b):
    for k in ("read", "start", "hash", "strand"):
        assert len(a[k]) == len(b[k]), (k, len(a[k]), len(b[k]))
        assert (a[k] == b[k]).all(), k


@pytest.mark.parametrize("w,k", [(11, 15), (14, 15), (1, 15), (32, 16), (5, 7), (19, 11), (11, 16), (8, 3)])
def test_sketch_parity_edge_cases(w, k):
    gx = lib.Index(TOY_PRG, w, k, device=0)
    rng = np.random.default_rng(w * 100 + k)
    strs = []
    for L in [0, 1, k - 1, k, w + k - 2, w + k - 1, w + k, 100, 150, 151, 191 + k, 192 + k, 193 + k, 400, 1000, 5000]:
        strs.append("".join("ACGT"[i] for i in rng.integers(0, 4, size=L)))
    strs.append("A" * 300)                                  # homopolymer: every k-mer ties
    strs.append("ACGT" * 100)                               # short tandem repeat
    strs.append(strs[9][:70] + "N" + strs[9][71:])          # non-ACGT base drops the read
    strs.append(strs[9].lower())                            # soft-masked bases hash like upper case
    strs.append("AC" * 80 + "GATTACA" * 30)
    data, off = reads_from_strings(strs)
    assert_sketch_equal(gpu_sketch(gx, data, off), oracle_sketch_all(data, off, w, k))


def test_sketch_parity_fixed_stride_and_ragged():
    w, k = 11, 15
    gx = lib.Index(TOY_PRG, w, k, device=0)
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=20, decoys=3, seed=5)
    want = oracle_sketch_all(d, o, w, k)
    assert_sketch_equal(gpu_sketch(gx, d, o, stride_words=10), want)
    assert_sketch_equal(gpu_sketch(gx, d, o, stride_words=0), want)
    rng = np.random.default_rng(3)
    strs = ["".join("ACGT"[i] for i in rng.integers(0, 4, size=int(L))) for L in rng.integers(0, 700, size=300)]
    data, off = reads_from_strings(strs)
    assert_sketch_equal(gpu_sketch(gx, data, off), oracle_sketch_all(data, off, w, k))


@pytest.mark.parametrize("w,k", [(11, 15), (14, 15)])
def test_sketch_parity_short_read_kernel(w, k):
    """the thread-per-read kernel (reads <= 640 bp, compile-time w,k): ragged lengths, ties, drops, padding lanes"""
    gx = lib.Index(TOY_PRG, w, k, device=0)
    rng = np.random.default_rng(w)
    strs = ["".join("ACGT"[i] for i in rng.integers(0, 4, size=int(L))) for L in rng.integers(0, 600, size=700)]
    strs += ["A" * 300, "ACGT" * 100, "AC" * 80 + "GATTACA" * 30, "T" * (w + k - 1), "G" * (w + k - 2), "",
             strs[5][:40] + "N" + strs[5][41:], "C" * 640, "ACG" * 213]
    for L in (w + k - 1, w + k, 2 * w + k - 1, 2 * w + k, 150, 151, 160, 161):
        strs.append("".join("ACGT"[i] for i in rng.integers(0, 4, size=L)))
    data, off = reads_from_strings(strs)
    want = oracle_sketch_all(data, off, w, k)
    assert_sketch_equal(gpu_sketch(gx, data, off), want)                      # ragged offsets
    assert_sketch_equal(gpu_sketch(gx, data, off, stride_words=40), want)     # fixed stride
    # a batch that is not a multiple of the CTA size, and a single read
    assert_sketch_equal(gpu_sketch(gx, *reads_from_strings(strs[:1])), oracle_sketch_all(*reads_from_strings(strs[:1]), w, k))


@pytest.mark.parametrize("w,k", [(11, 15), (14, 15)])
def test_sketch_parity_long_reads_segmented(w, k):
    """long reads are cut into segments for the thread-per-item kernel: every segment boundary must be seamless"""
    gx = lib.Index(TOY_PRG, w, k, device=0)
    rng = np.random.default_rng(k * 7 + w)
    lens = [641, 40 * w + k - 1, 40 * w + k, 40 * w + k + 1, 80 * w + k - 1, 80 * w + k + w, 3000, 12345, 50000, 7, 0, 700]
    strs = ["".join("ACGT"[i] for i in rng.integers(0, 4, size=L)) for L in lens]
    strs += ["A" * 2000, "ACGT" * 800, "AC" * 500 + "GATTACA" * 300, strs[6][:1500] + "N" + strs[6][1501:]]
    data, off = reads_from_strings(strs)
    assert_sketch_equal(gpu_sketch(gx, data, off), oracle_sketch_all(data, off, w, k))


def test_empty_batch():
    gx = lib.Index(TOY_PRG, 11, 15, device=0)
    data, off = reads_from_strings([])
    words, woff, lens = lib.pack_reads(data, off)
    gx.sample_begin(lib.make_opts(illumina=True), 150)
    b = gx.upload(words, woff, lens)
    assert gx.map_batch(b) == (0, 0)
    gx.genotype(TOY_REFS)
    assert [l for l in gx.vcf().splitlines() if not l.startswith("#")] == []


def run_both(prg, refs, data, off, w=11, k=15, illumina=True, genome_size=4411532, stride_words=0, n_batches=1, c=10):
    gx, ox = both_indexes(prg, w, k)
    oo = O.make_opts(illumina=illumina, genome_size=genome_size, min_cluster_size=c)
    go = lib.make_opts(illumina=illumina, genome_size=genome_size, min_cluster_size=c)
    first_len = int(off[1] - off[0]) if len(off) > 1 else 0
    mr = O.MapRun(ox, data, off, oo)
    gx.sample_begin(go, first_len)
    n = len(off) - 1
    hits = []
    bounds = np.linspace(0, n, n_batches + 1).astype(int)
    for bi in range(n_batches):
        lo, hi = int(bounds[bi]), int(bounds[bi + 1])
        sub_off = off[lo:hi + 1] - off[lo]
        sub = data[int(off[lo]):int(off[hi])]
        words, woff, lens = lib.pack_reads(sub, sub_off, stride_words)
        b = gx.upload(words, woff, lens, total_bases=int(sub_off[-1]), stride_words=stride_words, read_id_base=lo)
        nh, nk = gx.map_batch(b)
        h = gx.last_hits(nh)
        assert int(h["kept"].sum()) == nk
        hits.append(h)
    gh = {key: np.concatenate([h[key] for h in hits]) for key in hits[0]}
    return gx, ox, mr, gh, oo


def assert_map_equal(gx, mr, gh):
    oh = mr.hits()
    for key in ("read", "prg", "fwd", "start", "knode", "kept"):
        assert len(gh[key]) == len(oh[key]), (key, len(gh[key]), len(oh[key]))
        assert (gh[key] == oh[key]).all(), key
    cov = gx.coverage()
    f, r = mr.coverage()
    assert (cov["fwd"] == f).all() and (cov["rev"] == r).all()
    assert (cov["locus_reads"] == mr.locus_reads()).all()
    sc = mr.scalars()
    assert cov["total_bases"] == sc["total_bases"] and cov["n_reads"] == sc["n_reads"]


def test_toy_config1_full_pipeline():
    """BASELINE config 1: the reference's toy PRG (gid, pncA), simulated Illumina reads + decoys."""
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=60, decoys=5, seed=1)
    for w in (11, 14):
        gx, ox, mr, gh, oo = run_both(TOY_PRG, TOY_REFS, d, o, w=w, genome_size=2000, stride_words=10)
        assert len(gh["read"]) > 1000
        assert_map_equal(gx, mr, gh)
        og = assert_genotype_equal(gx, ox, mr, oo, TOY_REFS)
        assert len(og.records()["pos"]) == 23


def test_synthetic_panel_illumina_multibatch():
    p, prg, refs = small_panel()
    d, o, g, pl = panel_sample(p, 60000)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, genome_size=len(g), stride_words=10, n_batches=3)
    assert gh["kept"].sum() > 10000
    assert_map_equal(gx, mr, gh)
    og = assert_genotype_equal(gx, ox, mr, oo, refs)
    r = og.records()
    assert (r["gt"] > 0).sum() > 10  # the sample carries alt alleles and they are called


def test_synthetic_panel_nanopore_long_reads():
    """config 4 shape: long noisy reads, no -I (max_diff 250, e_rate 0.11), ragged lengths, multi-chunk sketch."""
    p, prg, refs = small_panel()
    d, o, g, pl = long_reads_sample(p, 600)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, illumina=False, genome_size=len(g))
    assert gh["kept"].sum() > 1000
    assert_map_equal(gx, mr, gh)
    assert_genotype_equal(gx, ox, mr, oo, refs)


def test_low_min_cluster_size_many_clusters():
    """-c 2 lets short spurious clusters through so the overlap filters (filter_clusters/2) do real work."""
    p, prg, refs = small_panel()
    d, o, g, pl = long_reads_sample(p, 300, seed=33, mean_len=6000)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, illumina=False, genome_size=len(g), c=2)
    assert_map_equal(gx, mr, gh)
    assert_genotype_equal(gx, ox, mr, oo, refs)


def test_coverage_is_additive_over_shards():
    """read sharding (BASELINE config 3): per-shard accumulators summed == single run (the allreduce identity)."""
    p, prg, refs = small_panel()
    d, o, g, pl = panel_sample(p, 30000, seed=41)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, genome_size=len(g), stride_words=10)
    whole = gx.accum_download()
    go = lib.make_opts(illumina=True, genome_size=len(g))
    n = len(o) - 1
    parts = []
    for s in range(4):
        lo, hi = n * s // 4, n * (s + 1) // 4
        sub_off = o[lo:hi + 1] - o[lo]
        words, woff, lens = lib.pack_reads(d[int(o[lo]):int(o[hi])], sub_off, 10)
        gx.sample_begin(go, 150)
        gx.map_batch(gx.upload(words, woff, lens, total_bases=int(sub_off[-1]), stride_words=10, read_id_base=lo))
        parts.append(gx.accum_download().astype(np.int64))
    tot = sum(parts)
    # scalars are split lo24/hi: recombine before comparing
    def scal(a):
        return (int(a[-4]) + (int(a[-3]) << 24), int(a[-2]) + (int(a[-1]) << 24))
    assert (tot[:-4] == whole[:-4]).all()
    assert scal(tot) == scal(whole.astype(np.int64))
    gx.sample_begin(go, 150)
    gx.accum_upload(tot.astype(np.int32))
    assert_genotype_equal(gx, ox, mr, oo, refs)


def _drop_in_call_matches_oracle(tmp_path, fq, d, o):
    """maps the reads file fq (the reads d, o) through drprg_cuda_map_genotype into tmp_path and checks the VCF against
    the oracle's; returns the index and pandora.log"""
    gx, ox = both_indexes(TOY_PRG, 11, 15)
    st = gx.map_genotype(fq, TOY_REFS, tmp_path, lib.make_opts(illumina=True, genome_size=2000))
    assert st["n_reads"] == len(o) - 1 and st["n_records"] == 23
    log = (tmp_path / "pandora.log").read_text()
    got = (tmp_path / "pandora_genotyped.vcf").read_text()
    oo = O.make_opts(illumina=True, genome_size=2000)
    og = O.Genotype(ox, O.MapRun(ox, d, o, oo), oo, TOY_REFS)
    strip = lambda t: [l for l in t.splitlines() if not l.startswith("##fileDate")]
    assert strip(got) == strip(og.vcf())
    return gx, log


def test_drop_in_call_writes_pandora_vcf(tmp_path):
    """drprg_cuda_map_genotype == Pandora::genotype_with: files in, outdir/pandora_genotyped.vcf out."""
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=9)
    fq = tmp_path / "reads.fq.gz"
    sim.write_fastq(str(fq), d, o, gz=True)
    gx, log = _drop_in_call_matches_oracle(tmp_path, fq, d, o)
    assert "ingest=host-framed, " in log, log
    with pytest.raises(lib.DrprgCudaError):
        gx.map_genotype(tmp_path / "missing.fq", TOY_REFS, tmp_path)


@pytest.mark.parametrize("fmt", ["wrapped_fastq", "fasta"])
def test_drop_in_call_host_parser_fallback(tmp_path, fmt):
    """a wrapped FASTQ (sequence and quality in lines of 60) or a FASTA of the same reads: the framer declines it, the
    drop-in call maps it through the host parser (pandora.log says so) and writes the oracle's VCF"""
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=9)
    wrap = lambda s: b"".join(s[j:j + 60] + b"\n" for j in range(0, len(s), 60))
    reads = [d[int(o[i]):int(o[i + 1])].tobytes() for i in range(len(o) - 1)]
    fq = tmp_path / ("reads.fq" if fmt == "wrapped_fastq" else "reads.fa")
    fq.write_bytes(b"".join(b"@r%d\n" % i + wrap(r) + b"+\n" + wrap(b"I" * len(r)) if fmt == "wrapped_fastq" else
                            b">r%d\n" % i + wrap(r) for i, r in enumerate(reads)))
    _, log = _drop_in_call_matches_oracle(tmp_path, fq, d, o)
    assert "ingest=host\n" in log, log


def test_batch_of_samples_config5(tmp_path):
    """BASELINE config 5 shape: several samples through drprg_cuda_map_genotype_batch on one resident index;
    every sample's VCF equals the oracle's."""
    import ctypes as C
    p, prg, refs = small_panel()
    gx, ox = both_indexes(prg, 11, 15)
    n_samples = 4
    reads, outs, datas = [], [], []
    for s in range(n_samples):
        d, o, g, pl = panel_sample(p, 20000, seed=100 + 7 * s)
        fq = tmp_path / (f"s{s}.fq.gz" if s % 2 else f"s{s}.fq")  # gzip samples are inflated ahead of time on spare threads
        sim.write_fastq(str(fq), d, o, gz=bool(s % 2))
        od = tmp_path / f"out{s}"
        od.mkdir()
        reads.append(str(fq).encode()); outs.append(str(od).encode()); datas.append((d, o, len(g)))
    L = lib.lib()
    arr_r = (C.c_char_p * n_samples)(*reads)
    arr_o = (C.c_char_p * n_samples)(*outs)
    stats = (lib.MapStats * n_samples)()
    go = lib.make_opts(illumina=True, genome_size=200_000, threads=4)
    rc = L.drprg_cuda_map_genotype_batch(gx.h, C.c_size_t(n_samples), arr_r, refs.encode(), arr_o, C.byref(go), stats)
    assert rc == 0, L.drprg_cuda_last_error()
    strip = lambda t: [l for l in t.splitlines() if not l.startswith("##fileDate")]
    for s in range(n_samples):
        d, o, gl = datas[s]
        oo = O.make_opts(illumina=True, genome_size=200_000)
        og = O.Genotype(ox, O.MapRun(ox, d, o, oo), oo, refs)
        got = open(os.path.join(outs[s].decode(), "pandora_genotyped.vcf")).read()
        assert strip(got) == strip(og.vcf()), s
        assert stats[s].n_reads == len(o) - 1


def test_pandora_mirror_interface(tmp_path):
    """drprg_b200.pandora.Pandora mirrors Pandora::genotype_with / vcf_filename (src/lib.rs:580-646)."""
    from drprg_b200.pandora import DependencyError, Pandora
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=30, decoys=1, seed=4)
    fq = tmp_path / "r.fq"
    sim.write_fastq(str(fq), d, o)
    pan = Pandora.from_path()
    st = pan.genotype_with(TOY_PRG, TOY_REFS, fq, tmp_path, ["-t", "2", "-w", "11", "-k", "15", "-c", "10", "-I"])
    assert (tmp_path / Pandora.vcf_filename()).exists() and st["n_records"] == 23
    with pytest.raises(DependencyError):
        pan.genotype_with(TOY_PRG, TOY_REFS, tmp_path / "nope.fq", tmp_path, ["-w", "11", "-k", "15"])
    with pytest.raises(DependencyError):
        pan.genotype_with(TOY_PRG, TOY_REFS, fq, tmp_path, ["--bogus"])


def test_config2_full_size_properties_and_oracle():
    """BASELINE config 2 at full size (30-locus panel, 1 M x 150 bp reads from a 4.4 Mb genome): size-independent
    properties (hit order, shard additivity, idempotence) plus a direct comparison with the oracle (which finishes in
    seconds on the box's host threads)."""
    from drprg_b200 import workload
    wl = workload.Config2()
    d, o = wl.reads(1_000_000, 0)
    n = len(o) - 1
    words, _, lens = lib.pack_reads(d, o, workload.STRIDE_WORDS)
    gx = lib.Index(wl.prg_path, wl.w, wl.k, device=0)
    go = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE)
    gx.sample_begin(go, workload.READ_LEN)
    nh, nk = gx.map_batch(gx.upload(words, None, lens, total_bases=int(o[-1]), stride_words=workload.STRIDE_WORDS))
    whole = gx.accum_download().astype(np.int64)
    h = gx.last_hits(nh)
    # sortedness: (read, prg, fwd-first, start, knode) strictly increasing
    key = np.stack([h["read"], h["prg"], 1 - h["fwd"], h["start"], h["knode"]]).astype(np.int64)
    order = np.lexsort(key[::-1])
    assert (order == np.arange(nh)).all()
    assert 0.005 < nk / n < 2.0 and nk == int(h["kept"].sum())
    gx.genotype(wl.refs_path)
    vcf_whole = [l for l in gx.vcf().splitlines() if not l.startswith("##fileDate")]
    # shard additivity (the allreduce identity) and idempotence
    tot = np.zeros_like(whole)
    for s in range(8):
        lo, hi = n * s // 8, n * (s + 1) // 8
        gx.sample_begin(go, workload.READ_LEN)
        gx.map_batch(gx.upload(words[lo * 10:hi * 10], None, lens[lo:hi], total_bases=150 * (hi - lo),
                               stride_words=workload.STRIDE_WORDS, read_id_base=lo))
        tot += gx.accum_download().astype(np.int64)
    assert (tot[:-4] == whole[:-4]).all()
    gx.sample_begin(go, workload.READ_LEN)
    gx.accum_upload(np.concatenate([tot[:-4], whole[-4:]]).astype(np.int32))
    gx.genotype(wl.refs_path)
    assert [l for l in gx.vcf().splitlines() if not l.startswith("##fileDate")] == vcf_whole
    # oracle on the same million reads
    ox = O.Index(wl.prg_path, wl.w, wl.k)
    oo = O.make_opts(threads=os.cpu_count() or 1, illumina=True, genome_size=workload.GENOME_SIZE)
    mr = O.MapRun(ox, d, o, oo)
    f, r = mr.coverage()
    N = ox.total_knodes
    assert (whole[:2 * N:2] == f).all() and (whole[1:2 * N:2] == r).all()
    assert (whole[2 * N:2 * N + ox.n_loci] == mr.locus_reads()).all()
    oh = mr.hits()  # every hit and its kept flag, at full size
    for hk in ("read", "prg", "fwd", "start", "knode", "kept"):
        assert len(h[hk]) == len(oh[hk]) and (h[hk] == oh[hk]).all(), hk
    og = O.Genotype(ox, mr, oo, wl.refs_path)
    assert [l for l in og.vcf().splitlines() if not l.startswith("##fileDate")] == vcf_whole


def test_pandora_cuda_cli_drop_in(tmp_path):
    """drprg_b200/pandora_cuda takes the exact argv drprg builds for `pandora map` (src/lib.rs:594-617,
    src/predict.rs:288-294), so `drprg predict -p pandora_cuda` needs no Rust change."""
    import subprocess
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=12)
    fq = tmp_path / "reads.fq"
    sim.write_fastq(str(fq), d, o)
    exe = os.path.join(os.path.dirname(lib.SO_PATH), "pandora_cuda")
    out = tmp_path / "out"
    argv = [exe, "map", "--genotype", "--local", "--gt-conf", "0", "-v", "-o", str(out), "-g", "2000", "--max-covg", "4294967295",
            "--vcf-refs", TOY_REFS, "-t", "2", "-w", "11", "-k", "15", "-c", "10", "-I", TOY_PRG, str(fq)]
    r = subprocess.run(argv, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ox = O.Index(TOY_PRG, 11, 15)
    oo = O.make_opts(illumina=True, genome_size=2000)
    og = O.Genotype(ox, O.MapRun(ox, d, o, oo), oo, TOY_REFS)
    strip = lambda t: [l for l in t.splitlines() if not l.startswith("##fileDate")]
    assert strip((out / "pandora_genotyped.vcf").read_text()) == strip(og.vcf())
    bad = subprocess.run([exe, "map", "-w", "11", "-k", "15", str(tmp_path / "missing.prg"), str(fq)], capture_output=True, text=True)
    assert bad.returncode != 0 and "cannot open" in bad.stderr


@pytest.mark.parametrize("env", [{"DRPRG_MLPATH_GENERIC": "1"}, {"DRPRG_SCREEN": "0"}, {"DRPRG_VCF_TEXT": "host"}])
def test_alternative_kernel_variants_keep_parity(env):
    """three paths that the toy panels only reach when forced, each of which must give the oracle's results: the generic
    ML-path kernel (DRPRG_MLPATH_GENERIC=1), which loci too large for the level-parallel kernel's shared memory take; the
    short-read sketch + lookup kernels without the k-mer screen in front (DRPRG_SCREEN=0), which an index of more than
    300 k k-mers uses; and the host VCF formatter (DRPRG_VCF_TEXT=host), which formats a sample that the device formatter
    cannot print exactly.  The switches are read once per process."""
    import subprocess, sys
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "toy_config1 or nanopore or low_min_cluster or short_read_kernel or screened_lookup"], env=e, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_hit_buffer_regrows_on_targeted_reads():
    """every read on the panel (targeted sequencing): ~20 hits per read overflow the initial hit buffer, which must
    regrow to the exact count and re-run the sketch without changing the result"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 5, 0.1)
    g, placements = sim.make_genome(p, [h[0] for h in hap], size=60_000, seed=6, min_sep=3000)
    regions = [(s, ln) for s, ln, st in placements]
    d, o = sim.simulate_reads(g, 120_000, 150, seed=8, sub_rate=0.002, regions=regions)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, genome_size=len(g), stride_words=10)
    assert len(gh["read"]) > (1 << 20)
    assert_map_equal(gx, mr, gh)


def test_minimizer_in_more_than_255_kmer_nodes():
    """a minimizer k-mer shared by 300 loci has 300 index records: the slot's 8-bit count escapes to a header record
    (pandora has no limit); hits must equal the oracle's"""
    rng = np.random.default_rng(77)
    shared = "".join("ACGT"[i] for i in rng.integers(0, 4, size=90))
    loci = []
    for i in range(300):
        tail = "".join("ACGT"[j] for j in rng.integers(0, 4, size=40))
        loci.append(f">rep{i}\n{shared}{tail}\n")
    text = "".join(loci)
    gx, ox = lib.Index(text=text, w=11, k=15, device=0), O.Index(text=text, w=11, k=15)
    rec = ox.records()
    _, counts = np.unique(rec["hash"], return_counts=True)
    assert counts.max() >= 300
    reads = [shared[:80], shared[5:90], shared + "ACGTACGTAC", loci[7].split("\n")[1], "".join("ACGT"[j] for j in rng.integers(0, 4, size=150))]
    data, off = reads_from_strings(reads)
    oo = O.make_opts(illumina=True, genome_size=100000, min_cluster_size=2)
    go = lib.make_opts(illumina=True, genome_size=100000, min_cluster_size=2)
    mr = O.MapRun(ox, data, off, oo)
    for stride in (0, 10):
        words, woff, lens = lib.pack_reads(data, off, stride)
        gx.sample_begin(go, 80)
        nh, nk = gx.map_batch(gx.upload(words, woff, lens, total_bases=int(off[-1]), stride_words=stride))
        assert nh > 3000
        assert_map_equal(gx, mr, gx.last_hits(nh))


def _fastq_bytes(reads, crlf=False, final_newline=True):
    nl = b"\r\n" if crlf else b"\n"
    t = b"".join(b"@read%d some comment" % i + nl + r + nl + b"+" + nl + b"I" * len(r) + nl for i, r in enumerate(reads))
    return t if final_newline else t[:-len(nl)]


def _map_file_both_ways(gx, path, opts):
    """(hits, info) through batch_from_fastx (framed on the host, packed on the device) and through the host parser +
    upload"""
    out = []
    b, info = gx.batch_from_fastx(path)
    gx.sample_begin(opts, info["first_read_len"])
    nh, nk = gx.map_batch(b)
    out.append((gx.last_hits(nh), info, gx.coverage()))
    words, woff, lens, n, tb, fl = lib.read_fastx(path)
    gx.sample_begin(opts, fl)
    nh, nk = gx.map_batch(gx.upload(words, woff, lens, total_bases=tb))
    out.append((gx.last_hits(nh), dict(n_reads=n, total_bases=tb, first_read_len=fl), gx.coverage()))
    return out


@pytest.mark.parametrize("variant", ["plain", "gzip", "crlf", "no_final_newline"])
def test_device_fastq_ingest_matches_host_parser(tmp_path, variant):
    """SURVEY 8f rank 2: the reads file is framed on the host and its sequence lines are 2-bit packed on the GPU; the
    batch must be the one the host parser builds (same reads, lengths, dropped reads, hits and coverage)."""
    import gzip
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=30, decoys=2, seed=4)
    reads = [d[int(o[i]):int(o[i + 1])].tobytes() for i in range(len(o) - 1)]
    reads[3] = reads[3][:70] + b"N" + reads[3][71:]      # dropped by pandora: non-ACGT
    reads[5] = reads[5].lower()                          # case-insensitive
    reads[7] = reads[7][:20]                             # shorter than w + k - 1
    reads[9] = b""                                       # empty sequence line
    reads[11] = reads[11][:149] + b"x"                   # bad base in the last word
    text = _fastq_bytes(reads, crlf=(variant == "crlf"), final_newline=(variant != "no_final_newline"))
    path = tmp_path / ("r.fq.gz" if variant == "gzip" else "r.fq")
    path.write_bytes(gzip.compress(text) if variant == "gzip" else text)
    gx = lib.Index(TOY_PRG, 11, 15, device=0)
    (hd, idev, cd), (hh, ihost, ch) = _map_file_both_ways(gx, path, lib.make_opts(illumina=True, genome_size=2000))
    assert idev["parsed_on_device"]
    assert idev["n_reads"] == ihost["n_reads"] == len(reads)
    assert idev["total_bases"] == ihost["total_bases"] == sum(len(r) for r in reads)
    assert idev["first_read_len"] == ihost["first_read_len"] == len(reads[0])
    assert idev["n_dropped"] == 2
    assert len(hd["read"]) > 500
    for key in ("read", "prg", "fwd", "start", "knode", "kept"):
        assert len(hd[key]) == len(hh[key]) and (hd[key] == hh[key]).all(), key
    for key in ("fwd", "rev", "locus_reads"):
        assert (cd[key] == ch[key]).all()
    assert cd["total_bases"] == ch["total_bases"] and cd["n_reads"] == ch["n_reads"]


def test_device_fastq_ingest_long_reads_and_fallbacks(tmp_path):
    """ragged layout + segment table for long reads; FASTA, wrapped or blank-line input falls back to the host parser,
    which rejects a record whose quality line is not as long as its sequence"""
    p, prg, refs = small_panel()
    d, o, g, pl = long_reads_sample(p, 200)
    reads = [d[int(o[i]):int(o[i + 1])].tobytes() for i in range(len(o) - 1)]
    fq = tmp_path / "long.fq"
    fq.write_bytes(_fastq_bytes(reads))
    gx = lib.Index(prg, 11, 15, device=0)
    opts = lib.make_opts(illumina=False, genome_size=len(g))
    (hd, idev, cd), (hh, ihost, ch) = _map_file_both_ways(gx, fq, opts)
    assert idev["parsed_on_device"] and idev["n_reads"] == len(reads)
    assert len(hd["read"]) > 1000
    for key in ("read", "prg", "fwd", "start", "knode", "kept"):
        assert len(hd[key]) == len(hh[key]) and (hd[key] == hh[key]).all(), key
    assert (cd["fwd"] == ch["fwd"]).all() and (cd["rev"] == ch["rev"]).all()
    # fallbacks
    fa = tmp_path / "r.fa"
    fa.write_bytes(b"".join(b">r%d\n" % i + r[:80] + b"\n" + r[80:160] + b"\n" for i, r in enumerate(reads[:20])))
    b, info = gx.batch_from_fastx(fa)
    assert not info["parsed_on_device"] and info["n_reads"] == 20
    blank = tmp_path / "blank.fq"
    blank.write_bytes(_fastq_bytes(reads[:10]) + b"\n")
    b, info = gx.batch_from_fastx(blank)
    assert not info["parsed_on_device"] and info["n_reads"] == 10
    bad = tmp_path / "bad.fq"  # record 3 of 10: quality one shorter than the sequence
    bad.write_bytes(b"".join(b"@r%d\n" % i + r + b"\n+\n" + b"I" * (len(r) - (i == 3)) + b"\n" for i, r in enumerate(reads[:10])))
    with pytest.raises(lib.DrprgCudaError, match="malformed FASTQ record"):
        gx.batch_from_fastx(bad)
    with pytest.raises(lib.DrprgCudaError, match="malformed FASTQ record"):
        gx.map_genotype(bad, refs, tmp_path, opts)


@pytest.mark.parametrize("env", [{"DRPRG_FRAME_SLICE": "2048"}, {"DRPRG_WAVE_BYTES": "30000", "DRPRG_FRAME_SLICE": "4096"}])
def test_file_ingest_variants_keep_parity(env):
    """a strict FASTQ file is framed on the host in slices of 1 MiB of text, which only the sequence lines leave; with
    2 KB slices every test file is cut at many record boundaries, and the batch must still be the host parser's.  The
    drop-in call maps a file wave by wave (DRPRG_WAVE_BYTES, default 1 GiB of text per wave): with 30 KB waves every test
    file takes several and the VCF must not change."""
    import subprocess, sys
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "device_fastq_ingest or drop_in_call or cli_drop_in or batch_of_samples"], env=e, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def _panel_path_reads(seed, n, lens_choices):
    """reads cut from the toy panel's reference sequences (so their minimizers are indexed), random strand, a few
    substitutions, assorted lengths; plus homopolymer / repeat / non-ACGT / random decoys"""
    rng = np.random.default_rng(seed)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    comp = str.maketrans("ACGT", "TGCA")
    strs = []
    for i in range(n):
        g = refs[int(rng.integers(0, len(refs)))]
        L = int(lens_choices[i % len(lens_choices)])
        st = int(rng.integers(0, max(1, len(g) - L)))
        r = list(g[st:st + L])
        for _ in range(int(rng.integers(0, 3))):
            if r:
                r[int(rng.integers(0, len(r)))] = "ACGT"[int(rng.integers(0, 4))]
        r = "".join(r)
        if rng.integers(0, 2):
            r = r.translate(comp)[::-1]
        strs.append(r)
    strs += ["A" * 300, "ACGT" * 100, "AC" * 80 + "GATTACA" * 30, "", "ACGTN" * 30, strs[0].lower(),
             strs[1][:30] + "N" + strs[1][31:], refs[0][:25], refs[0][:24], refs[0][:640], refs[1][:641]]
    strs += ["".join("ACGT"[j] for j in rng.integers(0, 4, size=int(L))) for L in rng.integers(0, 700, size=60)]
    return strs


@pytest.mark.parametrize("w", [11, 14, 1, 5, 19, 32])
def test_screened_lookup_edge_cases(w):
    """k = 15 batches go through the k-mer screen + resolve kernels: hits must equal the oracle's for every window size
    (compiled W = 11, 14 and the generic resolve), read lengths around the word / chunk / segment boundaries, ragged and
    fixed-stride layouts, both strands, ties, dropped reads"""
    k = 15
    lens = [25, 26, 31, 32, 33, 47, 48, 49, 100, 127, 128, 129, 142, 143, 144, 145, 150, 151, 159, 160, 161, 174, 175, 176,
            200, 255, 256, 257, 300, 454, 455, 456, 500, 639, 640]
    strs = _panel_path_reads(100 + w, 350, lens)
    data, off = reads_from_strings(strs)
    gx, ox, mr, gh, oo = run_both(TOY_PRG, TOY_REFS, data, off, w=w, k=k, genome_size=2000, c=2)
    assert len(gh["read"]) > 2000
    assert_map_equal(gx, mr, gh)
    gx2, ox2, mr2, gh2, _ = run_both(TOY_PRG, TOY_REFS, data, off, w=w, k=k, genome_size=2000, c=2, stride_words=44)
    for key in gh:
        assert (gh[key] == gh2[key]).all(), key
    # short-read-only batch (the one-chunk screen instantiation) and a long-read batch (segments)
    short = [s for s in strs if len(s) <= 160]
    d2, o2 = reads_from_strings(short)
    gx3, ox3, mr3, gh3, _ = run_both(TOY_PRG, TOY_REFS, d2, o2, w=w, k=k, genome_size=2000, c=2, stride_words=10)
    assert_map_equal(gx3, mr3, gh3)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    longs = [refs[0] + refs[1][:300], refs[1], refs[0][:700] + "ACGT" * 200 + refs[1][100:], "A" * 1500, refs[0][:641]] + short[:20]
    d3, o3 = reads_from_strings(longs)
    gx4, ox4, mr4, gh4, _ = run_both(TOY_PRG, TOY_REFS, d3, o3, w=w, k=k, genome_size=2000, c=2, illumina=False)
    assert_map_equal(gx4, mr4, gh4)


def test_chunked_upload_and_its_overflow_path():
    """a host upload of >= 8 MB is split into four chunks whose screen/resolve kernels start as each chunk lands.  Targeted
    reads overflow the initial hit buffer in a middle chunk: the batch is redone with larger buffers and must equal the
    oracle (and a second sample on the same handle, which needs no redo, must give the same hits)."""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 5, 0.1)
    g, placements = sim.make_genome(p, [h[0] for h in hap], size=60_000, seed=6, min_sep=3000)
    regions = [(s, ln) for s, ln, st in placements]
    d, o = sim.simulate_reads(g, 230_000, 150, seed=9, sub_rate=0.002, regions=regions)
    gx, ox, mr, gh, oo = run_both(prg, refs, d, o, genome_size=len(g), stride_words=10)   # 9.2 MB of words: chunked
    assert len(gh["read"]) > (2 << 20)
    assert_map_equal(gx, mr, gh)
    # second sample on the same handle: buffers are large enough now, no redo, same answer
    words, woff, lens = lib.pack_reads(d, o, 10)
    gx.sample_begin(lib.make_opts(illumina=True, genome_size=len(g), min_cluster_size=10), 150)
    nh, nk = gx.map_batch(gx.upload(words, woff, lens, total_bases=int(o[-1]), stride_words=10))
    h2 = gx.last_hits(nh)
    for key in gh:
        assert (gh[key] == h2[key]).all(), key
    assert_map_equal(gx, mr, h2)
