"""The local assembler of `pandora discover` on the GPU (drprg_cuda_discover_assemble): region statuses and de-novo allele
sets equal the oracle's restatement (tests/denovo_oracle.py) on the same reads, on every way the reads reach the map pass;
and, independently of the oracle, novel variants planted in a sample come back as their true haplotypes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import denovo_oracle as A
import discover_py as D
import oracle_py as O
from drprg_b200 import lib, sim
from helpers import TOY_PRG, TOY_REFS, panel_sample, small_panel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle(prg, refs, d, o, genome_size, **asm):
    ox = O.Index(prg, 11, 15)
    oo = O.make_opts(illumina=True, genome_size=genome_size)
    mr = O.MapRun(ox, d, o, oo)
    og = O.Genotype(ox, mr, oo, refs)
    loci, regions = D.discover(ox, mr, og, open(prg).read().splitlines())
    reads = [d[int(o[i]):int(o[i + 1])].tobytes().decode() for i in range(len(o) - 1)]
    return regions, A.assemble(loci, regions, reads, **asm)


def as_sets(regions, results):
    status = [r[0] for r in results]
    paths = sorted((i, a, b, s) for i, (st, a, b, ps) in enumerate(results) for s in ps)
    return status, paths


def gpu_run(prg, refs, d, o, genome_size, devices=None, n_batches=1, **asm):
    gx = lib.Index(prg, 11, 15, devices=devices) if devices else lib.Index(prg, 11, 15, device=0)
    words, woff, lens = lib.pack_reads(d, o, 10)
    n = len(lens)
    gx.retain_hits(True)
    gx.sample_begin(lib.make_opts(illumina=True, genome_size=genome_size), 150)
    for q in range(n_batches):
        lo, hi = n * q // n_batches, n * (q + 1) // n_batches
        gx.map_batch(gx.upload(words[lo * 10:hi * 10], None, lens[lo:hi], total_bases=int(o[hi] - o[lo]), stride_words=10,
                               read_id_base=lo))
    gx.genotype(refs)
    _, regions = gx.discover_candidates()
    status, paths = gx.discover_assemble(**asm)
    return gx, regions, status.tolist(), sorted(paths)


def check(prg, refs, d, o, genome_size, asm=None, **kw):
    asm = asm or {}
    want_regions, want = oracle(prg, refs, d, o, genome_size, **asm)
    gx, regions, status, paths = gpu_run(prg, refs, d, o, genome_size, **kw, **asm)
    assert [r[:5] for r in regions] == [r[:5] for r in want_regions]
    want_status, want_paths = as_sets(want_regions, want)
    assert status == want_status
    assert paths == want_paths
    return gx, status, paths


def toy_hole():
    d, o = sim.toy_dataset(TOY_PRG, TOY_REFS, depth=40, decoys=2, seed=5)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    reads = [d[int(o[i]):int(o[i + 1])].tobytes().decode() for i in range(len(o) - 1)]
    comp = str.maketrans("ACGT", "TGCA")
    hole = refs[0][400:425]
    keep = [r for r in reads if hole not in r and hole not in r.translate(comp)[::-1]]
    dd = np.frombuffer("".join(keep).encode(), np.uint8).copy()
    return dd, np.arange(len(keep) + 1, dtype=np.uint64) * np.uint64(150)


def test_toy_sample_with_an_uncovered_stretch():
    d, o = toy_hole()
    gx, status, paths = check(TOY_PRG, TOY_REFS, d, o, 2000)
    assert len(status) >= 1


def test_panel_sample_staged_batches_and_shards():
    p, prg, refs = small_panel()
    d, o, g, pl = panel_sample(p, 12_000, seed=61)
    gx, status, paths = check(prg, refs, d, o, len(g))
    assert status.count(lib.ASSEMBLED) > 0
    st = gx.last_assemble_stats()
    assert st["regions_shared"] == len(status) and st["regions_global"] == 0
    check(prg, refs, d, o, len(g), n_batches=3)                 # the same reads in 3 staged batches
    check(prg, refs, d, o, len(g), devices=[0, 0, 0])           # a multi-GPU handle: three shards on one GPU
    check(prg, refs, d, o, len(g), asm=dict(min_dbg_dp=3, max_insertion=5, max_candidate_paths=4))


def test_pileup_beyond_the_shared_memory_table():
    """about 800x over one locus with a novel SNP in it: the region's pileup has more k-mer positions than a CTA's
    shared-memory table holds, so its k-mers are counted in global scratch"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 41, 0.1)
    seqs, variants = sim.insert_novel_variants(p, hap, ["snp"], seed=1)
    g, pl = sim.make_genome(p, seqs, size=200_000, seed=42, min_sep=3000)
    s, n, _ = pl[0]
    d, o = sim.simulate_reads(g, n * 800 // 150, 150, 43, 0.002, regions=[(s - 100, n + 200)])
    gx, status, paths = check(prg, refs, d, o, len(g))
    assert gx.last_assemble_stats()["regions_global"] >= 1


def test_reads_file_in_small_waves_through_the_pandora_mirror(tmp_path):
    """Pandora.genotype_with(..., retain_hits=True) on a reads FILE mapped in 30 KB waves (the bases of every wave are gone
    when the next one is mapped), then discover_paths()"""
    p, prg, refs = small_panel()
    d, o, g, pl = panel_sample(p, 12_000, seed=61)
    fq = tmp_path / "reads.fq"
    sim.write_fastq(str(fq), d, o)
    code = (
        "import json, sys\n"
        f"sys.path[:0] = [{ROOT!r}]\n"
        "from drprg_b200.pandora import Pandora\n"
        "pan = Pandora.from_path()\n"
        f"pan.genotype_with({prg!r}, {refs!r}, {str(fq)!r}, {str(tmp_path)!r}, ['-t', '4', '-w', '11', '-k', '15', '-c', '10', '-I'],"
        " retain_hits=True)\n"
        "by_name = pan.discover_paths()\n"
        "ix = pan._index\n"
        "_, regions = ix.discover_candidates()\n"
        "status, paths = ix.discover_assemble()\n"
        "print(json.dumps(dict(by_name=by_name, status=status.tolist(), paths=paths, regions=[r[:5] for r in regions])))\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, DRPRG_WAVE_BYTES="30000"), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert "wave(s)" in open(tmp_path / "pandora.log").read() and " 1 wave(s)" not in open(tmp_path / "pandora.log").read()
    want_regions, want = oracle(prg, refs, d, o, 4411532)  # drprg's -g is fixed at the Mtb genome size in genotype_with
    want_status, want_paths = as_sets(want_regions, want)
    assert [tuple(r) for r in got["regions"]] == [r[:5] for r in want_regions]
    assert got["status"] == want_status
    assert sorted(tuple(x) for x in got["paths"]) == want_paths
    names = lib.Index(prg, 11, 15, device=-1).names
    by_name = {}
    for i, a, b, s in want_paths:
        by_name.setdefault(names[want_regions[i][0]], []).append([a, b, s])
    assert got["by_name"] == by_name


def test_novel_variants_come_back_as_their_haplotypes():
    """a SNP, a 3 bp deletion and a 6 bp insertion that the PRG does not know, 40x of 150 bp reads: the region over each
    is assembled, and one of its alleles is the sample's true sequence between the anchors"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, 31, 0.1)
    seqs, variants = sim.insert_novel_variants(p, hap, ["snp", "del3", "ins6"], seed=2)
    g, pl = sim.make_genome(p, seqs, size=200_000, seed=32, min_sep=3000)
    d, o = sim.simulate_reads(g, 200_000 * 40 // 150, 150, 33, 0.002)
    gx, regions, status, paths = gpu_run(prg, refs, d, o, len(g))
    loci, _ = gx.discover_candidates()
    for li, v, ref_len, alt, _ in variants:
        cons, new = loci[li][0], seqs[li].decode()
        over = [i for i, r in enumerate(regions) if r[0] == li and r[1] <= v + ref_len and r[2] >= v - 1]
        assert over, ("no candidate region over the variant", li, v)
        for i in over:
            assert status[i] == lib.ASSEMBLED, (li, v, status[i])
            a, b = next((a, b) for r, a, b, s in paths if r == i)
            k = A.DISCOVER_K
            lo, hi = new.find(cons[a:a + k]), new.find(cons[b - k:b], max(0, v - k))
            assert (i, a, b, new[lo:hi + k]) in paths, (li, v, alt)


def test_refusals():
    """no retention, no genotype, no candidates, and one-process-per-GPU handles: a clear error, no result"""
    d, o = toy_hole()
    words, woff, lens = lib.pack_reads(d, o, 10)
    gx = lib.Index(TOY_PRG, 11, 15, device=0)
    opts = lib.make_opts(illumina=True, genome_size=2000)
    gx.retain_hits(True)
    gx.sample_begin(opts, 150)
    gx.map_batch(gx.upload(words, woff, lens, total_bases=int(o[-1]), stride_words=10))
    with pytest.raises(lib.DrprgCudaError, match="genotype"):
        gx.discover_assemble()
    gx.genotype(TOY_REFS)
    with pytest.raises(lib.DrprgCudaError, match="discover_candidates"):
        gx.discover_assemble()
    gx.discover_candidates()
    gx.discover_assemble()
    gx.retain_hits(False)
    gx.sample_begin(opts, 150)
    gx.map_batch(gx.upload(words, woff, lens, total_bases=int(o[-1]), stride_words=10))
    gx.genotype(TOY_REFS)
    with pytest.raises(lib.DrprgCudaError, match="retain_hits"):
        gx.discover_assemble()
    root = lib.Index(TOY_PRG, 11, 15, device=0)
    root.shard_root(2)
    with pytest.raises(lib.DrprgCudaError, match="one-process-per-GPU"):
        root.discover_assemble()
