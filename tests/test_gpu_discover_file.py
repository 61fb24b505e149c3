"""`pandora discover` in one call (drprg_cuda_discover): denovo_paths.txt equals the restatement of tests/denovo_paths_oracle.py
byte for byte, whichever way the reads reach the map pass and whichever front end asks (lib.Index.discover,
Pandora.discover_with, `pandora_cuda discover` with drprg's argv); planted novel variants come back as records; retention
is restored afterwards; and the refusals give a clear error."""
import gzip
import os
import shutil
import subprocess
import sys
import tempfile

import pytest

import denovo_paths_oracle as P
import discover_py as D
import oracle_py as O
from drprg_b200 import lib, sim
from drprg_b200.pandora import DependencyError, Pandora
from helpers import TOY_PRG, TOY_REFS, panel_sample, reads_from_strings, small_panel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "drprg_b200", "pandora_cuda")
MTB = 4411532  # drprg's fixed -g


def toy_hole():
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=5)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    reads = [d[int(o[i]):int(o[i + 1])].tobytes().decode() for i in range(len(o) - 1)]
    comp = str.maketrans("ACGT", "TGCA")
    hole = refs[0][400:425]
    keep = [r for r in reads if hole not in r and hole not in r.translate(comp)[::-1]]
    return reads_from_strings(keep)


def discover_file(tmp, name, prg, reads, genome_size, **kw):
    out = tmp / name
    out.mkdir()
    ix = lib.Index(prg, 11, 15, **(kw or dict(device=0)))
    st = ix.discover(reads, out, lib.make_opts(illumina=True, genome_size=genome_size))
    return (out / "denovo_paths.txt").read_text(), st


@pytest.fixture(scope="module")
def panel(tmp_path_factory):
    p, prg, refs = small_panel()
    d, o, g, pl = panel_sample(p, 12_000, seed=61)
    tmp = tmp_path_factory.mktemp("panel")
    fq = tmp / "reads.fq"
    sim.write_fastq(str(fq), d, o)
    want, _, _ = P.oracle_file(prg, d, o, MTB)
    return dict(prg=prg, refs=refs, d=d, o=o, fq=fq, want=want, tmp=tmp)


def test_toy_sample_with_an_uncovered_stretch(tmp_path):
    d, o = toy_hole()
    fq = tmp_path / "reads.fq"
    sim.write_fastq(str(fq), d, o)
    got, st = discover_file(tmp_path, "out", TOY_PRG, fq, 2000)
    want, _, regions = P.oracle_file(TOY_PRG, d, o, 2000)
    assert got == want
    assert st["n_regions"] == len(regions) >= 1 and st["n_reads"] == len(o) - 1


def test_panel_file_equals_the_restatement_on_every_ingest(panel, tmp_path):
    got, st = discover_file(tmp_path, "plain", panel["prg"], panel["fq"], MTB)
    assert got == panel["want"]
    n, genes = P.drprg_loci(got)
    assert n == st["n_loci_with_variants"] == len(genes) >= 1
    assert sum(len(v) for _, v in P.read_denovo_paths(got)[1].values()) == st["n_variants"]
    assert st["n_assembled"] + st["n_no_anchor"] + st["n_too_many_paths"] + st["n_no_path"] == st["n_regions"]
    gz = tmp_path / "reads.fq.gz"
    with open(panel["fq"], "rb") as f, gzip.open(gz, "wb") as g:
        shutil.copyfileobj(f, g)
    assert discover_file(tmp_path, "gz", panel["prg"], gz, MTB)[0] == panel["want"]
    fa = tmp_path / "reads.fa"  # FASTA goes through the host parser: a multi-GPU handle shards it over its GPUs
    d, o = panel["d"], panel["o"]
    fa.write_text("".join(f">r{i}\n{d[int(o[i]):int(o[i + 1])].tobytes().decode()}\n" for i in range(len(o) - 1)))
    assert discover_file(tmp_path, "multi", panel["prg"], fa, MTB, devices=[0, 0, 0])[0] == panel["want"]
    assert discover_file(tmp_path, "multi_fq", panel["prg"], panel["fq"], MTB, devices=[0, 0, 0])[0] == panel["want"]
    code = (f"import sys; sys.path[:0] = [{ROOT!r}]\n"
            "from drprg_b200 import lib\n"
            f"ix = lib.Index({panel['prg']!r}, 11, 15, device=0)\n"
            f"ix.discover({str(panel['fq'])!r}, {str(tmp_path)!r}, lib.make_opts(illumina=True, genome_size={MTB}))\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, DRPRG_WAVE_BYTES="30000"), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert (tmp_path / "denovo_paths.txt").read_text() == panel["want"]


def test_pandora_mirror_and_cli_with_drprgs_argv(panel, tmp_path):
    (tmp_path / "reads").mkdir()
    shutil.copy(panel["fq"], tmp_path / "reads" / "s1.fq")
    query = tmp_path / "query.tsv"
    query.write_text("sample\treads/s1.fq\n")  # relative: resolved against the query file's directory
    args = ["-t", "2", "-w", "11", "-k", "15", "-c", "10", "-I"]
    path = Pandora.from_path().discover_with(panel["prg"], query, tmp_path / "py", args)
    assert open(path).read() == panel["want"]
    env = {k: v for k, v in os.environ.items() if k != "DRPRG_REAL_PANDORA"}
    out = tmp_path / "cli"
    argv = [EXE, "discover", "-g", str(MTB), "--max-covg", str(2**32 - 1), "-v", "-o", str(out)] + args + ["-K", panel["prg"], str(query)]
    r = subprocess.run(argv, env=env, capture_output=True, text=True, cwd=str(tmp_path / "reads"))
    assert r.returncode == 0, r.stderr
    assert (out / "denovo_paths.txt").read_text() == panel["want"]
    assert sorted(os.listdir(out)) == ["denovo_paths.txt"]


def test_planted_variants_are_records():
    """a SNP, a 3 bp deletion and a 6 bp insertion the PRG does not know: each is a record of its locus that makes the
    same sequence out of the ML sequence, and the SNP is at its own position"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 31, 0.1)
    seqs, variants = sim.insert_novel_variants(p, hap, ["snp", "del3", "ins6"], seed=2)
    g, pl = sim.make_genome(p, seqs, size=200_000, seed=32, min_sep=3000)
    d, o = sim.simulate_reads(g, 200_000 * 40 // 150, 150, 33, 0.002)
    tmp = tempfile.mkdtemp(prefix="drprg_planted_")
    try:
        fq = os.path.join(tmp, "reads.fq")
        sim.write_fastq(fq, d, o)
        ix = lib.Index(prg, 11, 15, device=0)
        ix.discover(fq, tmp, lib.make_opts(illumina=True, genome_size=len(g)))
        _, got = P.read_denovo_paths(open(os.path.join(tmp, "denovo_paths.txt")).read())
    finally:
        shutil.rmtree(tmp)
    for li, v, ref_len, alt, old in variants:
        nodes, recs = got[ix.names[li]]
        cons = "".join(q for _, _, _, q in nodes)  # the locus's ML sequence
        at = cons.find(old[v - 30:v]) + 30  # the variant's offset on the ML sequence
        assert at >= 30 and cons[at:at + 30] == old[v:v + 30], (li, v)
        planted = cons[:at] + alt + cons[at + ref_len:]
        hits = [(pos, r, a) for pos, r, a in recs if cons[pos - 1:pos - 1 + len(r)] == r
                and cons[:pos - 1] + a + cons[pos - 1 + len(r):] == planted]
        assert hits, (li, v, ref_len, alt, recs)
        if ref_len == 1 and len(alt) == 1:
            assert (at + 1, cons[at], alt) in recs
        else:
            assert all(r and a and (r[0] == a[0] or r[-1] == a[-1]) for _, r, a in hits)  # anchored


def test_sample_without_novel_variants(tmp_path):
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=5)
    fq = tmp_path / "reads.fq"
    sim.write_fastq(str(fq), d, o)
    got, st = discover_file(tmp_path, "out", TOY_PRG, fq, 2000)
    assert got == "1 samples\nSample sample\n0 loci with denovo variants\n" == P.oracle_file(TOY_PRG, d, o, 2000)[0]
    assert st["n_variants"] == 0


def test_targeted_reads_grow_the_retained_hit_store_across_batches():
    """~800x over one locus, about 20 kept hits per read, in 4 staged batches: the retained-hit store is too small in the
    first batch and again in later ones, and regrows keeping what earlier batches appended; regions and reads equal the
    oracle's"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 41, 0.1)
    seqs, _ = sim.insert_novel_variants(p, hap, ["snp"], seed=1)
    g, pl = sim.make_genome(p, seqs, size=200_000, seed=42, min_sep=3000)
    s, n, _ = pl[0]
    d, o = sim.simulate_reads(g, n * 800 // 150, 150, 43, 0.002, regions=[(s - 100, n + 200)])
    ox = O.Index(prg, 11, 15)
    oo = O.make_opts(illumina=True, genome_size=len(g))
    mr = O.MapRun(ox, d, o, oo)
    og = O.Genotype(ox, mr, oo, refs)
    want_loci, want = D.discover(ox, mr, og, open(prg).read().splitlines())
    hits = mr.hits()
    n_reads = len(o) - 1
    assert (hits["kept"] == 1).sum() > 10 * n_reads
    gx = lib.Index(prg, 11, 15, device=0)
    words, woff, lens = lib.pack_reads(d, o, 10)
    gx.retain_hits(True)
    gx.sample_begin(lib.make_opts(illumina=True, genome_size=len(g)), 150)
    for q in range(4):
        lo, hi = n_reads * q // 4, n_reads * (q + 1) // 4
        gx.map_batch(gx.upload(words[lo * 10:hi * 10], None, lens[lo:hi], total_bases=int(o[hi] - o[lo]), stride_words=10,
                               read_id_base=lo))
    gx.genotype(refs)
    _, got = gx.discover_candidates()
    assert got == want and any(r[5] for r in want)


def test_retention_is_restored_after_discover(panel, tmp_path):
    opts = lib.make_opts(illumina=True, genome_size=MTB)
    fresh = lib.Index(panel["prg"], 11, 15, device=0)
    (tmp_path / "a").mkdir()
    fresh.map_genotype(panel["fq"], panel["refs"], tmp_path / "a", opts)
    ix = lib.Index(panel["prg"], 11, 15, device=0)
    (tmp_path / "b").mkdir()
    ix.discover(panel["fq"], tmp_path / "b", opts)
    ix.map_genotype(panel["fq"], panel["refs"], tmp_path / "b", opts)
    assert (tmp_path / "b" / "pandora_genotyped.vcf").read_bytes() == (tmp_path / "a" / "pandora_genotyped.vcf").read_bytes()
    with pytest.raises(lib.DrprgCudaError, match="retain_hits"):  # retention was off before discover, and is off again
        ix.discover_candidates()


def test_refusals(panel, tmp_path):
    ix = lib.Index(TOY_PRG, 11, 15, device=0)
    with pytest.raises(lib.DrprgCudaError, match="cannot open"):
        ix.discover(tmp_path / "missing.fq", tmp_path)
    with pytest.raises(lib.DrprgCudaError, match="cannot write"):
        ix.discover(panel["fq"], tmp_path / "no" / "such" / "dir")
    root = lib.Index(TOY_PRG, 11, 15, device=0)
    root.shard_root(2)
    with pytest.raises(lib.DrprgCudaError, match="one-process-per-GPU"):
        root.discover(panel["fq"], tmp_path)
    query = tmp_path / "two.tsv"
    query.write_text(f"a\t{panel['fq']}\nb\t{panel['fq']}\n")
    with pytest.raises(DependencyError, match="exactly one"):
        Pandora.from_path().discover_with(TOY_PRG, query, tmp_path / "py", ["-w", "11", "-k", "15"])
    env = {k: v for k, v in os.environ.items() if k != "DRPRG_REAL_PANDORA"}
    r = subprocess.run([EXE, "discover", "-o", str(tmp_path / "cli"), "-w", "11", "-k", "15", TOY_PRG, str(query)], env=env,
                       capture_output=True, text=True)
    assert r.returncode != 0 and "exactly one" in r.stderr
    query.write_text(f"a\t{panel['fq']}\n")
    r = subprocess.run([EXE, "discover", "--covg-threshold", "5", TOY_PRG, str(query)], env=env, capture_output=True, text=True)
    assert r.returncode != 0 and "unsupported option --covg-threshold" in r.stderr
    r = subprocess.run([EXE, "discover", "-o", str(tmp_path / "cli"), "-w", "11", "-k", "15", TOY_PRG,
                        str(tmp_path / "missing.tsv")], env=env, capture_output=True, text=True)
    assert r.returncode != 0 and "cannot read" in r.stderr
    assert not (tmp_path / "denovo_paths.txt").exists()
