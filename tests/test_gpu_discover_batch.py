"""`pandora discover` for a batch of samples on one resident index (drprg_cuda_discover_batch, lib.Index.discover_batch):
every denovo_paths.txt equals the file a single drprg_cuda_discover call on a fresh handle writes and the restatement of
tests/denovo_paths_oracle.py, whatever the sample's format (plain FASTQ, gzip FASTQ inflated ahead, FASTA through the host
parser); the stats equal the single call's; the caller's retention setting comes back; the first failing sample stops the
batch and is named; a drprg_cuda_index_load_multi handle writes the same files; and the refusals."""
import ctypes as C

import pytest

import denovo_paths_oracle as P
from drprg_b200 import lib, sim
from helpers import TOY_PRG, small_panel

pytestmark = pytest.mark.gpu
MTB = 4411532  # drprg's fixed -g
OPTS = dict(illumina=True, genome_size=MTB, threads=4)  # 4 host threads: the gzip look-ahead runs 4 samples deep


def opts():
    return lib.make_opts(**OPTS)


def panel_reads(p, seed, kinds, n_reads, sub_rate):
    """reads of a sample of the small panel with novel variants of `kinds` planted (none for [])"""
    hap = sim.sample_haplotype(p, seed, 0.1)
    seqs, _ = sim.insert_novel_variants(p, hap, kinds, seed=seed + 1)
    g, _ = sim.make_genome(p, seqs, size=200_000, seed=seed + 2, min_sep=3000)
    return sim.simulate_reads(g, n_reads, 150, seed + 3, sub_rate)


# (seed, planted variants, reads, substitution rate, file format); sample 3 has no novel variants at all
SPECS = [(71, ["snp", "del3", "ins6"], 12_000, 0.002, "fq"),
         (72, ["ins6", "snp", "del3"], 12_000, 0.002, "fq.gz"),
         (73, ["del3", "ins6", "snp"], 12_000, 0.002, "fa"),
         (91, [], 20_000, 0.0, "fq"),
         (74, ["snp", "snp", "ins6"], 12_000, 0.002, "fq.gz")]


@pytest.fixture(scope="module")
def batch(tmp_path_factory):
    p, prg, refs = small_panel()
    tmp = tmp_path_factory.mktemp("batch")
    reads, want = [], []
    for i, (seed, kinds, n, sub, fmt) in enumerate(SPECS):
        d, o = panel_reads(p, seed, kinds, n, sub)
        path = tmp / f"s{i}.{fmt}"
        if fmt == "fa":
            path.write_text("".join(f">r{j}\n{d[int(o[j]):int(o[j + 1])].tobytes().decode()}\n" for j in range(len(o) - 1)))
        else:
            sim.write_fastq(str(path), d, o, gz=fmt.endswith(".gz"))
        reads.append(path)
        want.append(P.oracle_file(prg, d, o, MTB)[0])
    assert want[3] == "1 samples\nSample sample\n0 loci with denovo variants\n"
    assert all(int(w.splitlines()[2].split()[0]) >= 1 for k, w in enumerate(want) if k != 3)
    return dict(prg=prg, refs=refs, reads=reads, want=want)


def outdirs(tmp_path, n, tag="out"):
    out = [tmp_path / f"{tag}{i}" for i in range(n)]
    for d in out:
        d.mkdir()
    return out


def text(d):
    return (d / "denovo_paths.txt").read_text()


def without_times(st):
    return {k: v for k, v in st.items() if not k.startswith("ms_")}


def test_every_file_equals_the_single_call_and_the_restatement(batch, tmp_path):
    ix = lib.Index(batch["prg"], 11, 15, device=0)
    out = outdirs(tmp_path, len(SPECS))
    stats = ix.discover_batch(None, batch["reads"], out, opts())
    assert len(stats) == len(SPECS)
    for i in range(len(SPECS)):
        single = tmp_path / f"single{i}"
        single.mkdir()
        st = lib.Index(batch["prg"], 11, 15, device=0).discover(batch["reads"][i], single, opts())
        assert (out[i] / "denovo_paths.txt").read_bytes() == (single / "denovo_paths.txt").read_bytes(), i
        assert text(out[i]) == batch["want"][i], i
        assert without_times(stats[i]) == without_times(st), i
    assert stats[3]["n_variants"] == 0 and all(stats[i]["n_variants"] > 0 for i in (0, 1, 2, 4))


@pytest.mark.parametrize("retain", [False, True])
def test_retention_is_restored_and_map_is_unchanged(batch, tmp_path, retain):
    fresh = lib.Index(batch["prg"], 11, 15, device=0)
    (tmp_path / "fresh").mkdir()
    fresh.map_genotype(batch["reads"][0], batch["refs"], tmp_path / "fresh", opts())
    ix = lib.Index(batch["prg"], 11, 15, device=0)
    ix.retain_hits(retain)
    out = outdirs(tmp_path, 2)
    ix.discover_batch(["a", "b"], batch["reads"][:2], out, opts())
    for i, name in enumerate(("a", "b")):  # the sample's name is the file's second line, the rest is unchanged
        assert text(out[i]).splitlines()[1] == f"Sample {name}"
        assert text(out[i]).splitlines()[2:] == batch["want"][i].splitlines()[2:]
    (tmp_path / "after").mkdir()
    ix.map_genotype(batch["reads"][0], batch["refs"], tmp_path / "after", opts())
    got = (tmp_path / "after" / "pandora_genotyped.vcf").read_bytes()
    assert got == (tmp_path / "fresh" / "pandora_genotyped.vcf").read_bytes()
    if retain:  # retention stayed on: the map call above kept its hits
        ix.discover_candidates()
    else:
        with pytest.raises(lib.DrprgCudaError, match="retain_hits"):
            ix.discover_candidates()


def test_the_first_failing_sample_stops_the_batch(batch, tmp_path):
    ix = lib.Index(batch["prg"], 11, 15, device=0)
    reads = list(batch["reads"])
    reads[2] = tmp_path / "missing.fq"
    out = outdirs(tmp_path, len(reads))
    with pytest.raises(lib.DrprgCudaError, match=r"sample 2 \(.*missing\.fq\): cannot open") as e:
        ix.discover_batch(None, reads, out, opts())
    assert [(d / "denovo_paths.txt").exists() for d in out] == [True, True, False, False, False]
    assert text(out[0]) == batch["want"][0] and text(out[1]) == batch["want"][1]
    (tmp_path / "again").mkdir()
    ix.discover(batch["reads"][2], tmp_path / "again", opts())
    assert text(tmp_path / "again") == batch["want"][2]
    with pytest.raises(lib.DrprgCudaError, match="sample 0 .*cannot write"):  # an unusable outdir is named too
        ix.discover_batch(None, batch["reads"][:1], [tmp_path / "no" / "such" / "dir"], opts())


def test_multi_gpu_handle_writes_the_same_files(batch, tmp_path):
    ix = lib.Index(batch["prg"], 11, 15, devices=[0, 0])  # two shards on one GPU: the whole sharded path
    out = outdirs(tmp_path, len(SPECS))
    ix.discover_batch(None, batch["reads"], out, opts())
    for i in range(len(SPECS)):
        assert text(out[i]) == batch["want"][i], i


def test_refusals_and_an_empty_batch(batch, tmp_path):
    host = lib.Index(TOY_PRG, 11, 15, device=-1)
    with pytest.raises(lib.DrprgCudaError, match="host-only"):
        host.discover_batch(None, batch["reads"][:1], [tmp_path], opts())
    root = lib.Index(TOY_PRG, 11, 15, device=0)
    root.shard_root(2)
    with pytest.raises(lib.DrprgCudaError, match="one-process-per-GPU"):
        root.discover_batch(None, batch["reads"][:1], [tmp_path], opts())
    ix = lib.Index(batch["prg"], 11, 15, device=0)
    assert ix.discover_batch(None, [], [], opts()) == []
    L = lib.lib()
    assert L.drprg_cuda_discover_batch(ix.h, C.c_size_t(0), None, None, None, None, None, None, None) == 0
    arr = (C.c_char_p * 1)(str(tmp_path).encode())
    assert L.drprg_cuda_discover_batch(ix.h, C.c_size_t(1), None, None, arr, None, None, None, None) != 0
    assert b"reads_paths and outdirs" in L.drprg_cuda_last_error()
    arr_r = (C.c_char_p * 1)(str(batch["reads"][0]).encode())
    assert L.drprg_cuda_discover_batch(ix.h, C.c_size_t(1), None, arr_r, None, None, None, None, None) != 0
    assert list(tmp_path.iterdir()) == []
    with pytest.raises(ValueError):
        ix.discover_batch(["a"], batch["reads"][:2], outdirs(tmp_path, 2))
