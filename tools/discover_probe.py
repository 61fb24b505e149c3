"""`pandora discover` at config-2 scale: the benchmark panel (workload.Config2) with a sample genome carrying 20 variants
the PRG does not know (a SNP, a 3 bp deletion or a 6 bp insertion in each of the first 20 loci), 1 M simulated 150 bp
reads.  Reports, in one run on one GPU:
  the card and its power limit; map_batch wall time with hit retention off and on, alternated, with spreads; the same at
  config-3 size (--big-batches batches of 2 x --reads reads per sample, the 1 M reads twice over); the bytes the retention
  keeps; the candidate regions and their assembly statuses; which k-mer table path the regions take and the assembly
  kernels' device time (CUDA events inside the library); the oracle assembler's wall time on the same regions and whether
  its results equal the GPU's; how many planted variants come back as their true haplotype; drprg_cuda_discover on the
  reads as a plain and a gzip FASTQ with its stage split, alternated with drprg_cuda_map_genotype on the same file; whether
  the file equals the test-side restatement (tests/denovo_paths_oracle.py) of the same ML paths, regions and oracle
  alleles; and how many planted variants are records of the file.
With --nanopore the sample is config 4's shape instead: --reads reads (default 15 000, 34x) of ~10 kb (lognormal sigma 0.3)
at 5 % error split 40/30/30 into substitutions, insertions and deletions, uploaded ragged and mapped without -I; the
config-3 section is left out.

    python tools/discover_probe.py [--reads 1000000] [--reps 5] [--big-batches 15] [--nanopore] [--out LOG]
"""
import argparse
import gzip
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]

import denovo_oracle as A  # noqa: E402
import denovo_paths_oracle as P  # noqa: E402
import oracle_py as O  # noqa: E402
from drprg_b200 import lib, sim, workload  # noqa: E402

KINDS = ("snp", "del3", "ins6")


def spread(v):
    v = sorted(v)
    return f"median {v[len(v) // 2]:.3f} min {v[0]:.3f} max {v[-1]:.3f}"


def write_fastq_ragged(path, data, off, gz):
    """reads of any length, gzip at level 1 (a 300x nanopore sample is ~2.6 GB of FASTQ)"""
    with (gzip.open(path, "wb", compresslevel=1) if gz else open(path, "wb")) as f:
        for i in range(0, len(off) - 1, 4096):
            f.write(b"".join(b"@r%d\n%s\n+\n%s\n" % (j, s, b"I" * len(s))
                             for j in range(i, min(i + 4096, len(off) - 1))
                             for s in [data[int(off[j]):int(off[j + 1])].tobytes()]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, help="default 1 000 000 (150 bp) or, with --nanopore, 15 000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--big-batches", type=int, default=15)
    ap.add_argument("--nanopore", action="store_true", help="config-4 reads: ~10 kb at 5 % error, no -I")
    ap.add_argument("--out", help="also write the report to this file")
    a = ap.parse_args()
    a.reads = a.reads or (15_000 if a.nanopore else 1_000_000)
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    log(f"card: {q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'}")
    w = workload.Config2()
    hap = sim.sample_haplotype(w.panel, workload.PANEL_SEED + 1, 0.10)
    seqs, variants = sim.insert_novel_variants(w.panel, hap, [KINDS[i % 3] for i in range(20)], seed=5)
    genome, _ = sim.make_genome(w.panel, seqs, size=workload.GENOME_SIZE, seed=workload.PANEL_SEED + 5)
    if a.nanopore:
        d, o = sim.simulate_long_reads(genome, a.reads, mean_len=10_000, sigma=0.3, seed=workload.PANEL_SEED + 2, err=0.05,
                                       mix=(0.4, 0.3, 0.3))
        log(f"sample: {a.reads} nanopore reads, {int(o[-1])} bases ({o[-1] / workload.GENOME_SIZE:.1f}x), mean "
            f"{o[-1] / a.reads:.0f} bp, 5 % error, {len(variants)} planted variants, config-2 panel ({len(w.panel.loci)} loci)")
    else:
        d, o = sim.simulate_reads(genome, a.reads, workload.READ_LEN, seed=workload.PANEL_SEED + 2, sub_rate=0.002)
        log(f"sample: {a.reads} reads of {workload.READ_LEN} bp, {len(variants)} planted variants, config-2 panel ({len(w.panel.loci)} loci)")
    first_len = int(o[1] - o[0])
    stride = 0 if a.nanopore else workload.STRIDE_WORDS  # long reads go up ragged (word_off)
    gx = lib.Index(w.prg_path, w.w, w.k, device=0)
    words, woff, lens = lib.pack_reads(d, o, stride)
    batch = gx.upload(words, woff, lens, total_bases=int(o[-1]), stride_words=stride)
    opts = lib.make_opts(illumina=not a.nanopore, genome_size=workload.GENOME_SIZE)
    ms = {False: [], True: []}
    for rep in range(a.reps + 1):  # the first round warms both arms up
        for on in ((False, True) if rep % 2 == 0 else (True, False)):
            gx.retain_hits(on)
            gx.sample_begin(opts, first_len)
            t = time.perf_counter()
            nh, nk = gx.map_batch(batch)  # returns after its stream has been synchronised
            if rep:
                ms[on].append((time.perf_counter() - t) * 1e3)
    log(f"map_batch ms, retention off: {spread(ms[False])}  (n={len(ms[False])})")
    log(f"map_batch ms, retention on:  {spread(ms[True])}  (n={len(ms[True])})")
    if not a.nanopore:
        big = gx.upload(np.concatenate([words, words]), None, np.concatenate([lens, lens]), total_bases=2 * int(o[-1]),
                        stride_words=workload.STRIDE_WORDS)
        ms = {False: [], True: []}
        for rep in range(a.reps + 1):
            for on in ((False, True) if rep % 2 == 0 else (True, False)):
                gx.retain_hits(on)
                gx.sample_begin(opts, first_len)
                t = time.perf_counter()
                for _ in range(a.big_batches):
                    gx.map_batch(big)
                if rep:
                    ms[on].append((time.perf_counter() - t) * 1e3)
        n_big = 2 * a.reads * a.big_batches
        log(f"{n_big} reads in {a.big_batches} batches of {2 * a.reads}, all map_batch calls ms, retention off: {spread(ms[False])}  (n={len(ms[False])})")
        log(f"{n_big} reads in {a.big_batches} batches of {2 * a.reads}, all map_batch calls ms, retention on:  {spread(ms[True])}  (n={len(ms[True])})")
        del big
    # the last call above left retention on or off depending on the parity of reps: map once more with it on
    gx.retain_hits(True)
    gx.sample_begin(opts, first_len)
    nh, nk = gx.map_batch(batch)
    h = gx.last_hits(nh)
    kept_reads = np.unique(h["read"][h["kept"] == 1])
    words_kept = int(((lens[kept_reads].astype(np.int64) + 15) // 16).sum())
    log(f"retained: {nk} kept hits of {len(kept_reads)} of {a.reads} reads ({100 * len(kept_reads) / a.reads:.2f} %): {12 * nk} bytes "
        f"of hits + {8 * len(kept_reads)} bytes of rows in the GPU's store, {4 * words_kept} bytes of 2-bit words on the host")
    gx.genotype(w.refs_path)
    loci, regions = gx.discover_candidates()
    n_region_reads = sum(len(r[5]) for r in regions)
    log(f"candidate regions: {len(regions)}, region reads: {n_region_reads}, k-mer positions in the largest pileup: "
        f"{max([sum(max(0, e - s - A.DISCOVER_K + 1) for _, s, e, _ in r[5]) for r in regions], default=0)}")
    kt = []
    for rep in range(a.reps + 1):
        status, paths = gx.discover_assemble()
        st = gx.last_assemble_stats()
        if rep:
            kt.append(st["ms_shared"] + st["ms_global"])
    names = ("assembled", "no anchor", "too many paths", "no path")
    counts = np.bincount(status, minlength=4)
    log("status: " + ", ".join(f"{n} {c}" for n, c in zip(names, counts.tolist())) + f"; de-novo alleles: {len(paths)}")
    log(f"k-mer tables: {st['regions_shared']} regions in shared memory, {st['regions_global']} in global scratch")
    log(f"assembly kernels ms (CUDA events, both launches): {spread(kt)}  (n={len(kt)})")
    reads = {}
    for r in regions:
        for rd, _, _, _ in r[5]:
            if rd not in reads:
                reads[rd] = d[int(o[rd]):int(o[rd + 1])].tobytes().decode()
    t = time.perf_counter()
    want = A.assemble(loci, regions, reads)
    log(f"oracle assembler (Python, one host thread) on the same regions: {(time.perf_counter() - t) * 1e3:.1f} ms")
    want_paths = sorted((i, a_, b, s) for i, (_, a_, b, ps) in enumerate(want) for s in ps)
    same = [x[0] for x in want] == status.tolist() and want_paths == sorted(paths)
    log(f"GPU statuses and alleles equal the oracle's: {same}")
    found = 0
    for li, v, ref_len, alt, _ in variants:
        cons, new = loci[li][0], seqs[li].decode()
        for i, r in enumerate(regions):
            if r[0] != li or r[1] > v + ref_len or r[2] < v - 1 or status[i] != lib.ASSEMBLED:
                continue
            ab = [(a_, b) for rr, a_, b, _ in paths if rr == i]
            if not ab:
                continue
            a_, b = ab[0]
            k = A.DISCOVER_K
            lo, hi = new.find(cons[a_:a_ + k]), new.find(cons[b - k:b], max(0, v - k))
            if lo >= 0 and hi >= 0 and (i, a_, b, new[lo:hi + k]) in paths:
                found += 1
                break
    log(f"planted variants recovered as their true haplotype: {found} of {len(variants)}")

    # the whole discover call on files, next to the map call on the same file
    gx.retain_hits(False)  # map_genotype runs with the caller's setting; discover switches retention on for itself
    tmp = tempfile.mkdtemp(prefix="drprg_discover_probe_")
    try:
        text = None
        for gz in (False, True):
            fq = os.path.join(tmp, "reads.fq" + (".gz" if gz else ""))
            if a.nanopore:
                write_fastq_ragged(fq, d, o, gz)
            else:
                sim.write_fastq_fast(fq, d, o, gz=gz)
            runs = {"discover": [], "map": []}
            for rep in range(a.reps + 1):
                for what in (("discover", "map") if rep % 2 == 0 else ("map", "discover")):
                    if what == "discover":
                        st = gx.discover(fq, tmp, opts)
                    else:
                        st = gx.map_genotype(fq, w.refs_path, tmp, opts)
                    if rep:
                        runs[what].append(st)
            kind = "gzip" if gz else "plain"
            for key in ("ms_ingest", "ms_map", "ms_ml_path", "ms_discover", "ms_total"):
                log(f"drprg_cuda_discover, {kind} FASTQ, {key}: {spread([r[key] for r in runs['discover']])}")
            for key in ("ms_ingest", "ms_map", "ms_genotype", "ms_total"):
                log(f"drprg_cuda_map_genotype, {kind} FASTQ, {key}: {spread([r[key] for r in runs['map']])}")
            st = runs["discover"][-1]
            log(f"drprg_cuda_discover, {kind} FASTQ: reads {st['n_reads']}, kept hits {st['n_hits_kept']}, regions {st['n_regions']}, "
                f"region reads {st['n_region_reads']}, assembled {st['n_assembled']}, no anchor {st['n_no_anchor']}, too many paths "
                f"{st['n_too_many_paths']}, no path {st['n_no_path']}, loci with variants {st['n_loci_with_variants']}, variants {st['n_variants']}")
            t = open(os.path.join(tmp, "denovo_paths.txt")).read()
            text = t if text is None else text
            log(f"denovo_paths.txt of the {kind} FASTQ equals the plain one: {t == text}")
    finally:
        shutil.rmtree(tmp)
    # the restatement from the ML paths and regions of the discover call's own genotyping (in-memory map above, same reads)
    # and the oracle assembler's alleles: checks the variant form and the layout, not the map pass (the tests do that)
    gx.retain_hits(True)
    gx.sample_begin(opts, first_len)
    gx.map_batch(batch)
    gx.genotype(None)
    loci, regions = gx.discover_candidates()
    reads = {rd: d[int(o[rd]):int(o[rd + 1])].tobytes().decode() for r in regions for rd, _, _, _ in r[5]}
    want = A.assemble(loci, regions, reads)
    ox = O.Index(w.prg_path, w.w, w.k)
    want_text = P.file_from(ox, open(w.prg_path).read().splitlines(), {l: gx.mlpath(l).tolist() for l in loci}, loci, regions, want)
    same_file = want_text == text
    log(f"denovo_paths.txt equals the restatement: {same_file}")
    _, got = P.read_denovo_paths(text)
    records = 0
    for li, v, ref_len, alt, old in variants:
        if gx.names[li] not in got:
            continue
        nodes, recs = got[gx.names[li]]
        cons = "".join(q for _, _, _, q in nodes)
        at = cons.find(old[v - 30:v]) + 30
        if at < 30:
            continue
        planted = cons[:at] + alt + cons[at + ref_len:]
        records += any(cons[p - 1:p - 1 + len(r)] == r and cons[:p - 1] + al + cons[p - 1 + len(r):] == planted for p, r, al in recs)
    log(f"planted variants that are records of denovo_paths.txt (same edit of the ML sequence): {records} of {len(variants)}")
    same = same and same_file
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
