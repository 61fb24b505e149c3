"""Shared dataset builders for the parity tests (seeded, small enough for the oracle to finish in seconds)."""
import os
import tempfile

import numpy as np

import oracle_py as O
from drprg_b200 import sim

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOY_PRG = os.path.join(GOLDEN, "toy.dr.prg")
TOY_REFS = os.path.join(GOLDEN, "toy.genes.fa")

_cache = {}


def reads_from_strings(strs):
    data = np.frombuffer("".join(strs).encode(), np.uint8).copy()
    off = np.zeros(len(strs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in strs])
    return data, off


def small_panel(seed=7, n_loci=5, n_sites=500):
    key = ("panel", seed, n_loci, n_sites)
    if key not in _cache:
        p = sim.make_panel(seed=seed, n_loci=n_loci, n_sites=n_sites, len_lo=900, len_hi=2200,
                           frac=(0.7, 0.12, 0.12, 0.06))
        d = tempfile.mkdtemp(prefix="drprg_panel_")
        prg, fa = p.write(d)
        _cache[key] = (p, prg, fa)
    return _cache[key]


def panel_sample(panel, n_reads, seed=11, genome_size=200_000, alt_frac=0.1, read_len=150, sub_rate=0.002):
    hap = sim.sample_haplotype(panel, seed, alt_frac)
    g, placements = sim.make_genome(panel, [h[0] for h in hap], size=genome_size, seed=seed + 1, min_sep=3000)
    d, o = sim.simulate_reads(g, n_reads, read_len, seed + 2, sub_rate)
    return d, o, g, placements


def long_reads_sample(panel, n_reads, seed=21, genome_size=200_000, mean_len=4000):
    hap = sim.sample_haplotype(panel, seed, 0.1)
    g, placements = sim.make_genome(panel, [h[0] for h in hap], size=genome_size, seed=seed + 1, min_sep=3000)
    d, o = sim.simulate_long_reads(g, n_reads, mean_len=mean_len, seed=seed + 2)
    return d, o, g, placements


def assert_genotype_equal(gx, ox, mr, oo, refs):
    og = O.Genotype(ox, mr, oo, refs)
    gx.genotype(refs)
    gp, op = gx.params(), og.params()
    for key in op:
        assert gp[key] == op[key], (key, gp[key], op[key])
    for l in range(ox.n_loci):
        a, b = gx.mlpath(l), og.mlpath(l)
        assert (a is None) == (b is None), l
        if a is not None:
            assert len(a) == len(b) and (a == b).all(), ("ml path", l)
    gr, orr = gx.gt_records(), og.records()
    for key in ("locus", "pos", "n_alleles", "gt", "mean_fwd", "mean_rev", "med_fwd", "med_rev", "sum_fwd", "sum_rev",
                "n_knodes", "allele_knodes", "gaps"):
        assert len(gr[key]) == len(orr[key]), key
        assert (gr[key] == orr[key]).all(), key
    # log-likelihoods: fp64 on both sides, 1e-9 relative (BASELINE.json north_star)
    np.testing.assert_allclose(gr["lik"], orr["lik"], rtol=1e-9, atol=0)
    np.testing.assert_allclose(gr["gt_conf"], orr["gt_conf"], rtol=1e-9, atol=1e-9)
    strip = lambda t: [l for l in t.splitlines() if not l.startswith("##fileDate")]
    assert strip(gx.vcf()) == strip(og.vcf())
    assert bytes(gx.vcf_view()) == gx.vcf_bytes()  # the zero-copy view is the same text
    # the filter / minor-allele statistics fused into the genotype kernel (SURVEY 8f rank 4) against the Rust restatement
    import rust_filters
    rust_filters.check_against(gx.filter_stats(), np.concatenate([[0], np.cumsum(gr["n_alleles"])]), gr["mean_fwd"], gr["mean_rev"],
                               gr["gaps"], gr["gt"], gr["gt_conf"], 0.1 if oo.illumina else 1.0)
    return og
