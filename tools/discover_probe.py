"""discover's local assembler at config-2 scale: the benchmark panel (workload.Config2) with a sample genome carrying
20 variants the PRG does not know (a SNP, a 3 bp deletion or a 6 bp insertion in each of the first 20 loci), 1 M
simulated 150 bp reads.  Reports, in one run on one GPU:
  the card and its power limit; map_batch wall time with hit retention off and on, alternated, with spreads; the bytes the
  retention keeps; the candidate regions and their assembly statuses; which k-mer table path the regions take and the
  assembly kernels' device time (CUDA events inside the library); the oracle assembler's wall time on the same regions and
  whether its results equal the GPU's; and how many planted variants come back as their true haplotype.

    python tools/discover_probe.py [--reads 1000000] [--reps 5] [--out LOG]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import denovo_oracle as A  # noqa: E402
from drprg_b200 import lib, sim, workload  # noqa: E402

KINDS = ("snp", "del3", "ins6")


def spread(v):
    v = sorted(v)
    return f"median {v[len(v) // 2]:.3f} min {v[0]:.3f} max {v[-1]:.3f}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="also write the report to this file")
    a = ap.parse_args()
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
    d, o = sim.simulate_reads(genome, a.reads, workload.READ_LEN, seed=workload.PANEL_SEED + 2, sub_rate=0.002)
    log(f"sample: {a.reads} reads of {workload.READ_LEN} bp, {len(variants)} planted variants, config-2 panel ({len(w.panel.loci)} loci)")
    gx = lib.Index(w.prg_path, w.w, w.k, device=0)
    words, woff, lens = lib.pack_reads(d, o, workload.STRIDE_WORDS)
    batch = gx.upload(words, woff, lens, total_bases=int(o[-1]), stride_words=workload.STRIDE_WORDS)
    opts = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE)
    ms = {False: [], True: []}
    for rep in range(a.reps + 1):  # the first round warms both arms up
        for on in ((False, True) if rep % 2 == 0 else (True, False)):
            gx.retain_hits(on)
            gx.sample_begin(opts, workload.READ_LEN)
            t = time.perf_counter()
            nh, nk = gx.map_batch(batch)  # returns after its stream has been synchronised
            if rep:
                ms[on].append((time.perf_counter() - t) * 1e3)
    log(f"map_batch ms, retention off: {spread(ms[False])}  (n={len(ms[False])})")
    log(f"map_batch ms, retention on:  {spread(ms[True])}  (n={len(ms[True])})")
    # the last call above left retention on or off depending on the parity of reps: map once more with it on
    gx.retain_hits(True)
    gx.sample_begin(opts, workload.READ_LEN)
    nh, nk = gx.map_batch(batch)
    h = gx.last_hits(nh)
    kept_reads = np.unique(h["read"][h["kept"] == 1])
    words_kept = int(((lens[kept_reads].astype(np.int64) + 15) // 16).sum())
    log(f"retained: {len(kept_reads)} of {a.reads} reads ({100 * len(kept_reads) / a.reads:.2f} %), {4 * words_kept} bytes of "
        f"2-bit words + {16 * len(kept_reads)} bytes of per-read entries")
    gx.genotype(w.refs_path)
    loci, regions = gx.discover_candidates()
    n_region_reads = sum(len(r[5]) for r in regions)
    log(f"candidate regions: {len(regions)}, region reads: {n_region_reads}")
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
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
