"""`pandora discover` for nanopore samples, drprg's default read type (no -I): ~4 kb reads at 5 % error, so nearly every read
is cut into segments by the map pass.  Staged runs (ragged and fixed-stride uploads, one batch and several) give the
candidate regions, region reads, statuses and alleles of the oracle (oracle/discover_py.py, tests/denovo_oracle.py); every
front end that reads a file (lib.Index.discover on plain, gzip and FASTA input and in small waves, `pandora_cuda discover`
with drprg's argv, lib.Index.discover_batch, a two-shard handle) writes the restated denovo_paths.txt of
tests/denovo_paths_oracle.py byte for byte; a deep pileup of long reads takes the global k-mer table and equals the
oracle; and the planted variants of the oracle's file are records of the GPU's."""
import gzip
import os
import shutil
import subprocess
import sys

import pytest

import denovo_oracle as A
import denovo_paths_oracle as P
import discover_py as D
import oracle_py as O
from drprg_b200 import lib, sim
from helpers import small_panel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "drprg_b200", "pandora_cuda")
MTB = 4411532  # drprg's fixed -g
GENOME = 200_000
KINDS = ["snp", "del3", "ins6", "snp", "ins6"]


def opts(**kw):
    return lib.make_opts(illumina=False, genome_size=MTB, **kw)


def nanopore_sample(seed, depth=34, mean_len=4000, regions=None, n_reads=None):
    """a small-panel sample with the 5 novel variants of KINDS planted and ~depth x of nanopore-like reads (5 % error)"""
    p, prg, refs = small_panel()
    hap = sim.sample_haplotype(p, seed, 0.1)
    seqs, variants = sim.insert_novel_variants(p, hap, KINDS, seed=seed + 1)
    g, pl = sim.make_genome(p, seqs, size=GENOME, seed=seed + 2, min_sep=3000)
    if regions == "locus0":
        regions = [pl[0][:2]]
    n = n_reads or GENOME * depth // mean_len
    d, o = sim.simulate_long_reads(g, n, mean_len=mean_len, seed=seed + 3, regions=regions)
    return dict(prg=prg, refs=refs, d=d, o=o, variants=variants)


def write_reads(path, d, o, fmt):
    if fmt == "fa":
        path.write_text("".join(f">r{i}\n{d[int(o[i]):int(o[i + 1])].tobytes().decode()}\n" for i in range(len(o) - 1)))
    else:
        sim.write_fastq(str(path), d, o, gz=fmt == "fq.gz")
    return path


def staged_oracle(s):
    """discover's regions (with their reads) and the assembler's results, from the oracle's own map pass"""
    ox = O.Index(s["prg"], 11, 15)
    oo = O.make_opts(illumina=False, genome_size=MTB)
    mr = O.MapRun(ox, s["d"], s["o"], oo)
    og = O.Genotype(ox, mr, oo, s["refs"])
    loci, regions = D.discover(ox, mr, og, open(s["prg"]).read().splitlines())
    d, o = s["d"], s["o"]
    reads = [d[int(o[i]):int(o[i + 1])].tobytes().decode() for i in range(len(o) - 1)]
    return regions, A.assemble(loci, regions, reads)


def staged_gpu(s, n_batches=1, stride=False):
    """the staged calls on batches uploaded ragged (word_off) or, with stride, at one fixed stride of the longest read"""
    d, o = s["d"], s["o"]
    n = len(o) - 1
    sw = int(((o[1:] - o[:-1]).max() + 15) // 16) if stride else 0
    words, woff, lens = lib.pack_reads(d, o, sw)
    gx = lib.Index(s["prg"], 11, 15, device=0)
    gx.retain_hits(True)
    gx.sample_begin(opts(), int(lens[0]))
    for q in range(n_batches):
        lo, hi = n * q // n_batches, n * (q + 1) // n_batches
        if stride:
            b = gx.upload(words[lo * sw:hi * sw], None, lens[lo:hi], total_bases=int(o[hi] - o[lo]), stride_words=sw, read_id_base=lo)
        else:
            b = gx.upload(words[int(woff[lo]):int(woff[hi])], woff[lo:hi + 1] - woff[lo], lens[lo:hi], total_bases=int(o[hi] - o[lo]),
                          read_id_base=lo)
        gx.map_batch(b)
    gx.genotype(s["refs"])
    _, regions = gx.discover_candidates()
    status, paths = gx.discover_assemble()
    return gx, regions, status.tolist(), sorted(paths)


def check_staged(s, want, **kw):
    want_regions, results = want
    gx, regions, status, paths = staged_gpu(s, **kw)
    assert [r[:5] for r in regions] == [r[:5] for r in want_regions]   # candidate regions
    assert [r[5] for r in regions] == [r[5] for r in want_regions]     # their reads: {read, start, end, fwd}
    assert status == [r[0] for r in results]
    assert paths == sorted((i, a, b, x) for i, (_, a, b, ps) in enumerate(results) for x in ps)
    return gx, status


@pytest.fixture(scope="module")
def sample(tmp_path_factory):
    s = nanopore_sample(81)
    d, o = s["d"], s["o"]
    assert ((o[1:] - o[:-1]) > 640).mean() > 0.95  # nearly every read takes the map pass's segment table
    s["tmp"] = tmp = tmp_path_factory.mktemp("nanopore")
    s["fq"] = write_reads(tmp / "reads.fq", d, o, "fq")
    s["want"], s["loci"], s["regions"] = P.oracle_file(s["prg"], d, o, MTB, illumina=False)
    assert int(s["want"].splitlines()[2].split()[0]) >= 3
    return s


@pytest.fixture(scope="module")
def staged_want(sample):
    return staged_oracle(sample)


def discover_file(tmp, name, prg, reads, **kw):
    out = tmp / name
    out.mkdir()
    ix = lib.Index(prg, 11, 15, **(kw or dict(device=0)))
    st = ix.discover(reads, out, opts())
    return (out / "denovo_paths.txt").read_text(), st


def test_staged_one_ragged_batch(sample, staged_want):
    gx, status = check_staged(sample, staged_want)
    assert status.count(lib.ASSEMBLED) > 0 and len(status) == len(sample["regions"])
    assert sum(len(r[5]) for r in staged_want[0]) > len(status)   # regions with several long reads over them


def test_staged_three_ragged_batches(sample, staged_want):
    check_staged(sample, staged_want, n_batches=3)


def test_staged_fixed_stride_batches(sample, staged_want):
    """one stride for every read: the longest read's words, so each batch still takes the segment table"""
    check_staged(sample, staged_want, stride=True)
    check_staged(sample, staged_want, n_batches=3, stride=True)


def test_file_equals_the_restatement_on_every_ingest(sample, tmp_path):
    got, st = discover_file(tmp_path, "plain", sample["prg"], sample["fq"])
    assert got == sample["want"]
    assert st["n_reads"] == len(sample["o"]) - 1 and st["n_regions"] == len(sample["regions"])
    assert st["n_assembled"] + st["n_no_anchor"] + st["n_too_many_paths"] + st["n_no_path"] == st["n_regions"]
    gz = tmp_path / "reads.fq.gz"
    with open(sample["fq"], "rb") as f, gzip.open(gz, "wb") as g:
        shutil.copyfileobj(f, g)
    assert discover_file(tmp_path, "gz", sample["prg"], gz)[0] == sample["want"]
    fa = write_reads(tmp_path / "reads.fa", sample["d"], sample["o"], "fa")  # the general host parser
    assert discover_file(tmp_path, "fa", sample["prg"], fa)[0] == sample["want"]


def test_file_in_small_waves(sample, tmp_path):
    """the FASTQ mapped in ~25-read waves: every wave's words are retained before the next wave replaces them"""
    code = ("import sys\n"
            f"sys.path[:0] = [{ROOT!r}]\n"
            "from drprg_b200 import lib\n"
            f"ix = lib.Index({sample['prg']!r}, 11, 15, device=0)\n"
            f"ix.discover({str(sample['fq'])!r}, {str(tmp_path)!r}, lib.make_opts(illumina=False, genome_size={MTB}))\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, DRPRG_WAVE_BYTES="200000"), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert (tmp_path / "denovo_paths.txt").read_text() == sample["want"]


def test_cli_with_drprgs_argv_without_illumina(sample, tmp_path):
    (tmp_path / "reads").mkdir()
    shutil.copy(sample["fq"], tmp_path / "reads" / "s1.fq")
    query = tmp_path / "query.tsv"
    query.write_text("sample\treads/s1.fq\n")
    env = {k: v for k, v in os.environ.items() if k != "DRPRG_REAL_PANDORA"}
    out = tmp_path / "cli"
    argv = [EXE, "discover", "-g", str(MTB), "--max-covg", str(2**32 - 1), "-v", "-o", str(out), "-t", "2", "-w", "11", "-k", "15",
            "-c", "10", "-K", sample["prg"], str(query)]
    r = subprocess.run(argv, env=env, capture_output=True, text=True, cwd=str(tmp_path / "reads"))
    assert r.returncode == 0, r.stderr
    assert (out / "denovo_paths.txt").read_text() == sample["want"]


def test_batch_of_three_samples(sample, tmp_path):
    others = [nanopore_sample(91, depth=25), nanopore_sample(95, depth=25)]
    reads = [sample["fq"]] + [write_reads(tmp_path / f"s{i}.{fmt}", s["d"], s["o"], fmt) for i, (s, fmt) in
                              enumerate(zip(others, ("fq.gz", "fq")), 1)]
    want = [sample["want"]] + [P.oracle_file(s["prg"], s["d"], s["o"], MTB, illumina=False)[0] for s in others]
    out = [tmp_path / f"out{i}" for i in range(3)]
    for d in out:
        d.mkdir()
    stats = lib.Index(sample["prg"], 11, 15, device=0).discover_batch(None, reads, out, opts(threads=4))
    no_times = lambda st: {k: v for k, v in st.items() if not k.startswith("ms_")}
    for i in range(3):
        got, st = discover_file(tmp_path, f"single{i}", sample["prg"], reads[i])
        assert (out[i] / "denovo_paths.txt").read_text() == got == want[i], i
        assert no_times(stats[i]) == no_times(st), i


@pytest.mark.parametrize("devices", [[0, 0], [0, 1]], ids=["one_gpu", "two_gpus"])
def test_two_shard_handle(sample, tmp_path, devices):
    if len(set(devices)) > int(lib.lib().drprg_cuda_device_count()):
        pytest.skip("needs two GPUs")
    assert discover_file(tmp_path, "multi", sample["prg"], sample["fq"], devices=devices)[0] == sample["want"]


def test_deep_pileup_of_long_reads_takes_the_global_table():
    """~1000 long reads centred on one locus: several regions have more than 8 192 k-mer positions in their pileup"""
    s = nanopore_sample(81, n_reads=1000, regions="locus0")
    want = staged_oracle(s)
    npos = [sum(max(0, e - st - A.DISCOVER_K + 1) for _, st, e, _ in r[5]) for r in want[0]]
    assert max(npos) > 8192
    gx, status = check_staged(s, want)
    assert gx.last_assemble_stats()["regions_global"] == sum(n > 8192 for n in npos) >= 1


def planted_records(text, names, variants):
    """the planted variants that are records of a denovo_paths.txt: the same edit of the locus's ML sequence"""
    _, got = P.read_denovo_paths(text)
    found = []
    for li, v, ref_len, alt, old in variants:
        if names[li] not in got:
            continue
        nodes, recs = got[names[li]]
        cons = "".join(q for _, _, _, q in nodes)
        at = cons.find(old[v - 30:v]) + 30
        if at < 30:
            continue
        planted = cons[:at] + alt + cons[at + ref_len:]
        if any(cons[p - 1:p - 1 + len(r)] == r and cons[:p - 1] + a + cons[p - 1 + len(r):] == planted for p, r, a in recs):
            found.append((li, v))
    return found


def test_planted_variants_of_the_oracle_are_records(sample, tmp_path):
    names = lib.Index(sample["prg"], 11, 15, device=-1).names
    want = planted_records(sample["want"], names, sample["variants"])
    assert want
    got, _ = discover_file(tmp_path, "out", sample["prg"], sample["fq"])
    assert set(want) <= set(planted_records(got, names, sample["variants"]))
