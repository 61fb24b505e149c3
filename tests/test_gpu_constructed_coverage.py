"""S6-S8 (parameter fit, ML path, genotyping and the VCF text) held to the oracle on hand-built coverage.

The parity tests get their coverage from simulated reads, which is always smooth and moderate.  Here the accumulator is
written directly (Index.accum_upload) and the oracle genotypes the same numbers (MapRun.from_coverage), so every
construction can aim at one edge of the genotyping code: exact ties, saturated strands, each branch of the fit, the
loci the speculative pass gets wrong, and the generic ML-path kernel with loci in shared and in global memory.  Every
construction first asserts, from the oracle's side, that it reaches the regime it is meant for, so that it cannot
silently stop testing its edge; test_constructions_reach_their_regimes does that without a GPU."""
import math
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle_py as O
from drprg_b200 import sim
from helpers import TOY_PRG, TOY_REFS, assert_genotype_equal, panel_sample, small_panel

W, K = 11, 15
SAT = 65535            # each strand counter saturates here (uint16 in pandora)
WINDOW = 100           # pandora's max_kmers_to_average: the ML path's moving window
NB_CLAMP = 0.999999    # nb_p when mean / var >= 0.985
SMEM_BUDGET = 220 * 1024


# ---------------------------------------------------------------------------------------------------------- plumbing
def _is_text(prg):
    return prg.startswith(">")


_oracle_idx, _gpu_idx = {}, {}


def oracle_index(prg):
    if prg not in _oracle_idx:
        _oracle_idx[prg] = O.Index(text=prg, w=W, k=K) if _is_text(prg) else O.Index(prg, W, K)
    return _oracle_idx[prg]


def gpu_index(prg):
    from drprg_b200 import lib
    if prg not in _gpu_idx:
        _gpu_idx[prg] = lib.Index(text=prg, w=W, k=K, device=0) if _is_text(prg) else lib.Index(prg, W, K, device=0)
    return _gpu_idx[prg]


def encode_accum(fwd, rev, locus_reads, total_bases, n_reads):
    """the accumulator layout: [fwd, rev interleaved | locus_reads | total_bases lo24, hi | n_reads lo24, hi]"""
    n = len(fwd)
    a = np.zeros(2 * n + len(locus_reads) + 4, np.int64)
    a[0:2 * n:2], a[1:2 * n:2] = fwd, rev
    a[2 * n:2 * n + len(locus_reads)] = locus_reads
    a[-4:] = [total_bases & 0xFFFFFF, total_bases >> 24, n_reads & 0xFFFFFF, n_reads >> 24]
    assert a.max() < 2 ** 31 and a.min() >= 0
    return a.astype(np.int32)


class Case:
    """per-node coverage of one construction (uncapped: the GPU gets these numbers, the oracle each strand capped at
    65535, which is what its counting would have left) and the sample's scalars and options"""

    def __init__(self, prg, refs, fwd, rev, locus_reads, total_bases, genome_size, n_reads=100_000, illumina=True):
        self.prg, self.refs, self.genome_size, self.illumina = prg, refs, genome_size, illumina
        self.fwd, self.rev = np.asarray(fwd, np.int64), np.asarray(rev, np.int64)
        self.locus_reads = np.asarray(locus_reads, np.int64)
        self.total_bases, self.n_reads = int(total_bases), int(n_reads)

    def oracle_opts(self):
        return O.make_opts(illumina=self.illumina, genome_size=self.genome_size)

    def oracle_maprun(self):
        ox = oracle_index(self.prg)
        return O.MapRun.from_coverage(ox, np.minimum(self.fwd, SAT), np.minimum(self.rev, SAT), self.locus_reads,
                                      self.total_bases, self.n_reads)

    def oracle(self):
        return O.Genotype(oracle_index(self.prg), self.oracle_maprun(), self.oracle_opts(), self.refs)


def genotype_both(case, gx=None):
    """the construction through the GPU (sample_begin, accum_upload, genotype) and the oracle; every result compared"""
    from drprg_b200 import lib
    gx = gx or gpu_index(case.prg)
    gx.sample_begin(lib.make_opts(illumina=case.illumina, genome_size=case.genome_size), 150)
    gx.accum_upload(encode_accum(case.fwd, case.rev, case.locus_reads, case.total_bases, case.n_reads))
    return assert_genotype_equal(gx, oracle_index(case.prg), case.oracle_maprun(), case.oracle_opts(), case.refs)


def split(c, rng=None):
    """a total per node -> (fwd, rev); with rng the split is uneven"""
    c = np.asarray(c, np.int64)
    if rng is None:
        f = (c + 1) // 2
    else:
        f = np.floor(c * rng.uniform(0.3, 0.7, size=c.shape)).astype(np.int64)
    return f, c - f


def inner_mask(ox, present=None):
    """True for the k-mer nodes that are neither start nor end of their locus (of the present loci, if given)"""
    m = np.ones(ox.total_knodes, bool)
    m[ox.knode_base[:-1]] = False
    m[ox.knode_base[1:] - 1] = False
    if present is not None:
        for l in range(ox.n_loci):
            if not present[l]:
                m[ox.knode_base[l]:ox.knode_base[l + 1]] = False
    return m


def locus_of(ox):
    return np.repeat(np.arange(ox.n_loci), np.diff(ox.knode_base))


def vcf_contigs(og):
    return [l[len("##contig=<ID="):].rstrip(">").split(",")[0] for l in og.vcf().splitlines() if l.startswith("##contig=")]


def vcf_body(og):
    return [l for l in og.vcf().splitlines() if not l.startswith("#")]


def nb_log_prob(c, P):
    """pandora's negative-binomial node score (the oracle's knode_log_prob), for the regime checks"""
    v = (math.lgamma(c + P["nb_r"]) - math.lgamma(P["nb_r"]) - math.lgamma(c + 1.0) + P["nb_r"] * math.log(P["nb_p"])
         + c * math.log(1.0 - P["nb_p"]))
    return max(v, -3.4028234663852886e38 / 1000.0)


def prob_hist(cov, mask, P):
    h = np.zeros(200, np.int64)
    for c in cov[mask].tolist():
        p = nb_log_prob(c, P)
        if -200.0 <= p < 0.0:
            h[int(math.floor(p + 200.0))] += 1
    return h


def prob_thresh(d):
    """pandora's find_prob_thresh on the 200-bin histogram"""
    p1 = int(np.argmax(d))
    p2 = -1
    for i in range(200):
        if abs(i - p1) <= 10 or d[i] == 0:
            continue
        if p2 < 0 or d[i] > d[p2]:
            p2 = i
    if p2 < 0:
        return max(-200, p1 - 210)
    a, b = min(p1, p2), max(p1, p2)
    return int(a + np.argmin(d[a:b + 1])) - 200


def exponent_values(og):
    r = og.records()
    v = np.concatenate([r["lik"], r["gt_conf"]])
    return v[["e" in "%g" % x for x in v.tolist()]]


# ------------------------------------------------------------------------------------------------------ the inputs
_cache = {}


def toy_plus_short():
    """the toy PRG plus two short loci whose ML paths are shorter than the 100-node window: (PRG text, sample genome)"""
    if "toy_plus" not in _cache:
        rng = np.random.default_rng(91)
        R = lambda n: sim.random_dna(rng, n).tobytes()
        short = [sim.Locus("s1", [R(30), sim.Site([[b"A"], [b"C"]]), R(8), sim.Site([[b"GT"], [b"G"], [b"TT"]]), R(30)]),
                 sim.Locus("s2", [R(25), sim.Site([[R(3)], [R(5)]]), R(25)])]
        text = open(TOY_PRG).read().rstrip("\n") + "\n" + "".join(f">{l.name}\n{l.prg_text()}\n" for l in short)
        genes = [l.strip().encode() for l in open(TOY_REFS) if not l.startswith(">")]
        genes += [short[0].spell(lambda s: len(s.alleles) - 1), short[1].spell(lambda s: 0)]
        genome = b"".join(R(400) + g for g in genes) + R(400)
        _cache["toy_plus"] = (text, np.frombuffer(genome, np.uint8).copy())
    return _cache["toy_plus"]


def realistic(which):
    """coverage of simulated reads (one oracle map pass each, cached): 'panel' = small_panel at ~45x, 'toy' = the toy
    PRG plus two short loci at ~40x.  Returns (prg, refs, fwd, rev, locus_reads, total_bases, genome_size)."""
    if which not in _cache:
        if which == "panel":
            p, prg, refs = small_panel()
            d, o, g, pl = panel_sample(p, 60000)
        else:
            prg, g = toy_plus_short()
            refs = TOY_REFS
            d, o = sim.simulate_reads(g, len(g) * 40 // 150, 150, 5, 0.002)
        ox = oracle_index(prg)
        mr = O.MapRun(ox, d, o, O.make_opts(illumina=True, genome_size=len(g)))
        f, r = mr.coverage()
        f, r, lr = f.astype(np.int64), r.astype(np.int64), mr.locus_reads().astype(np.int64)
        rng = np.random.default_rng(23)
        for l in np.flatnonzero(lr == 0):  # loci too short for a cluster of hits: coverage like the reads would give
            lo, hi = ox.knode_base[l], ox.knode_base[l + 1]
            f[lo:hi], r[lo:hi], lr[l] = rng.integers(15, 30, hi - lo), rng.integers(15, 30, hi - lo), 40
        _cache[which] = (prg, refs, f, r, lr, int(mr.scalars()["total_bases"]), len(g))
    return _cache[which]


def real_case(which, **kw):
    prg, refs, f, r, lr, tb, gs = realistic(which)
    args = dict(prg=prg, refs=refs, fwd=f.copy(), rev=r.copy(), locus_reads=lr.copy(), total_bases=tb, genome_size=gs)
    args.update(kw)
    return Case(**args)


# ------------------------------------------------------------------------------------------------ the constructions
# Each entry: name -> (build() -> Case, regime(case, oracle genotype)).  The regime check asserts, from the oracle's
# results and the index, that the construction reaches the edge it is named for.
def _uniform(which):
    def build():
        c = real_case(which)
        c.fwd[:], c.rev[:] = 15, 15
        c.total_bases = 40 * c.genome_size
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        P = og.params()
        assert P["var"] == 0 and P["nb_p"] == 0.015  # every node ties: mean >= var, the fallback model
        paths = [og.mlpath(l) for l in range(ox.n_loci)]
        assert all(p is not None and len(p) for p in paths)
        if which == "toy":  # ML paths shorter and longer than the window
            assert min(len(p) for p in paths) < WINDOW < max(len(p) for p in paths)
        else:  # small_panel has nodes with more than four successors (the level kernel's serial loop)
            assert (ox.knodes()["n_out"] > 4).sum() > 0
    return build, regime


def _zero_loci(which):
    def build():
        c = real_case(which)
        kb = oracle_index(c.prg).knode_base
        for l in (0, 2):
            c.fwd[kb[l]:kb[l + 1]], c.rev[kb[l]:kb[l + 1]] = 0, 0
        c.total_bases = 20 * c.genome_size  # covg 20: the coverage filter is off, the zero loci stay in the VCF
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        assert og.params()["covg"] <= 20 and c.locus_reads[[0, 2]].min() > 0
        assert {ox.names[0], ox.names[2]} <= set(vcf_contigs(og))
        assert len(og.mlpath(0)) and len(og.mlpath(2))
    return build, regime


def _rounded(which):
    def build():
        c = real_case(which)
        c.fwd, c.rev = np.round(c.fwd / 10).astype(np.int64) * 10, np.round(c.rev / 10).astype(np.int64) * 10
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        r = og.records()
        depth = r["mean_fwd"].astype(np.int64) + r["mean_rev"]
        off = np.concatenate([[0], np.cumsum(r["n_alleles"].astype(np.int64))])
        ties = sum(len(set(depth[off[i]:off[i + 1]].tolist())) < r["n_alleles"][i] for i in range(len(r["pos"])))
        assert ties > 0  # records whose alleles have exactly the same depth
        paths = [og.mlpath(l) for l in range(ox.n_loci)]
        assert all(p is not None and len(p) for p in paths)
        if which == "toy":
            assert min(len(p) for p in paths) < WINDOW < max(len(p) for p in paths)
    return build, regime


def _saturated():
    def build():
        c = real_case("panel")
        # 500 times the reads' coverage, on top of 7500 per strand: every node is deep, so no node without coverage
        # pulls the ML path off the covered alleles
        c.fwd, c.rev = c.fwd * 500 + 7500, c.rev * 500 + 7500
        ox = oracle_index(c.prg)
        og = real_case("panel").oracle()
        r = og.records()
        off = np.concatenate([[0], np.cumsum(r["n_knodes"].astype(np.int64))])
        aoff = np.concatenate([[0], np.cumsum(r["n_alleles"].astype(np.int64))])
        for i in range(0, len(r["pos"]), 7):  # the k-mers of every 7th record: one strand over the cap, the other under
            for a in range(aoff[i], aoff[i + 1]):
                g = ox.knode_base[r["locus"][i]] + r["allele_knodes"][off[a]:off[a + 1]]
                c.fwd[g] += 66_000 + 13 * i
                if i % 3 == 0:  # and both strands over
                    c.rev[g] += 70_000
        c.total_bases = 4000 * c.genome_size  # covg 4000: the ML paths' coverage mode (~20 000) passes the filter
        return c

    def regime(c, og):
        m = inner_mask(oracle_index(c.prg))
        over_one = ((c.fwd > SAT) & (c.rev < SAT))[m]
        assert over_one.sum() > 50 and ((c.fwd > SAT) & (c.rev > SAT))[m].sum() > 20
        assert ((np.minimum(c.fwd, SAT) + np.minimum(c.rev, SAT))[m] > 1000).mean() > 0.5
        assert len(exponent_values(og)) > 0  # values the device formatter leaves to the host
        assert len(vcf_contigs(og)) == oracle_index(c.prg).n_loci
    return build, regime


def _nb_clamped():
    def build():
        c = real_case("panel")
        ox = oracle_index(c.prg)
        # the inner nodes in pairs at 40 +- 7 and 40 +- 6 (one node at 40 if their number is odd): mean 40 and a
        # variance just above 40, so that mean / var >= 0.985 and nb_p = 0.015 + mean / var is clamped
        m = inner_mask(ox)
        n = int(m.sum())
        x = int(round(4.3 * n / 26))
        y = (n - 2 * x) // 2
        vals = np.array([47, 33] * x + [46, 34] * y + [40] * (n - 2 * x - 2 * y), np.int64)
        assert 40 < (vals - 40).var() and 40 / (vals - 40).var() >= 0.986
        vals = vals[np.random.default_rng(5).permutation(n)]
        tot = np.full(ox.total_knodes, 40, np.int64)
        tot[m] = vals
        c.fwd, c.rev = split(tot, np.random.default_rng(6))
        c.total_bases = 40 * c.genome_size
        return c

    def regime(c, og):
        P = og.params()
        assert P["mean"] < P["var"] and P["mean"] / P["var"] >= 0.985 and P["nb_p"] == NB_CLAMP
    return build, regime


def _empty_prob_hist():
    def build():
        c = real_case("panel")
        rng = np.random.default_rng(8)
        c.fwd, c.rev = split(rng.integers(14_000, 30_000, len(c.fwd)), rng)
        c.total_bases = 4000 * c.genome_size  # covg 4000: the histogram [400, 1000) is empty, E = 1
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        P = og.params()
        assert og.params()["thresh"] == -200 and P["E"] == 1
        m = inner_mask(ox, c.locus_reads > 0)
        assert prob_hist(np.minimum(c.fwd, SAT) + np.minimum(c.rev, SAT), m, P).sum() == 0  # no inner node in [-200, 0)
        assert len(vcf_contigs(og)) == ox.n_loci
    return build, regime


def _mean_ge_var():
    def build():
        c = real_case("panel")
        rng = np.random.default_rng(9)
        c.fwd, c.rev = rng.poisson(20, len(c.fwd)), rng.poisson(20, len(c.fwd))
        c.total_bases = 40 * c.genome_size
        return c

    def regime(c, og):
        P = og.params()
        assert P["mean"] >= P["var"] > 0 and P["nb_p"] == 0.015 and P["num_reads"] > 30 and P["covg"] > 2
    return build, regime


def _overdispersed(seed, **kw):
    c = real_case("panel", **kw)
    rng = np.random.default_rng(seed)
    c.fwd, c.rev = split(rng.poisson(rng.gamma(4.0, 10.0, len(c.fwd))), rng)
    return c


def _few_reads():
    def build():
        c = _overdispersed(10, total_bases=40 * realistic("panel")[6])
        c.locus_reads[:] = [30, 31, 29, 30, 30]  # num_reads = 150 // 5 = 30
        return c

    def regime(c, og):
        P = og.params()
        assert P["num_reads"] == 30 and P["mean"] < P["var"] and P["covg"] > 2 and P["nb_p"] == 0.015
    return build, regime


def _low_covg():
    def build():
        return _overdispersed(11, total_bases=2 * realistic("panel")[6] + 7)

    def regime(c, og):
        P = og.params()
        assert P["covg"] == 2 and P["mean"] < P["var"] and P["num_reads"] > 30 and P["nb_p"] == 0.015
    return build, regime


ABSENT = 1


def _absent_locus():
    def build():
        c = real_case("panel")
        ox = oracle_index(c.prg)
        lo, hi = ox.knode_base[ABSENT], ox.knode_base[ABSENT + 1]
        c.locus_reads[ABSENT] = 0
        c.fwd[lo:hi], c.rev[lo:hi] = 0, 0
        # coverage without reads, which every histogram of the fit must leave out: one value for the whole locus, the
        # one whose score is closest to -100 (a peak of its own in the score histogram, were it counted)
        P = c.oracle().params()
        t = min(range(1, 1000), key=lambda t: abs(nb_log_prob(t, P) + 100.0))
        c.fwd[lo:hi], c.rev[lo:hi] = split(np.full(hi - lo, t))
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        assert ox.names[ABSENT] not in vcf_contigs(og) and og.mlpath(ABSENT) is None
        lo, hi = ox.knode_base[ABSENT], ox.knode_base[ABSENT + 1]
        z = Case(c.prg, c.refs, c.fwd.copy(), c.rev.copy(), c.locus_reads, c.total_bases, c.genome_size)
        z.fwd[lo:hi], z.rev[lo:hi] = 0, 0
        assert z.oracle().params() == og.params()
        # were the locus counted, both histograms would change: the moments of the fit and the threshold
        P = og.params()
        cov = c.fwd + c.rev
        with_it = inner_mask(ox, np.ones(ox.n_loci, bool))
        without = inner_mask(ox, c.locus_reads > 0)
        assert cov[with_it].var() != cov[without].var()
        assert prob_thresh(prob_hist(cov, with_it, P)) != P["thresh"] == prob_thresh(prob_hist(cov, without, P))
    return build, regime


def _no_locus():
    def build():
        c = real_case("panel")
        c.locus_reads[:] = 0
        return c

    def regime(c, og):
        P = og.params()
        assert vcf_contigs(og) == [] and vcf_body(og) == [] and P["thresh"] == -25 and P["E"] == P["covg"] == 45
    return build, regime


OUTLIER = 3


def _outlier():
    def build():
        c = real_case("panel")
        ox = oracle_index(c.prg)
        lo, hi = ox.knode_base[OUTLIER], ox.knode_base[OUTLIER + 1]
        c.fwd[lo:hi] *= 50  # the locus's coverage mode is far above 10 * covg
        c.rev[lo:hi] *= 50
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        assert og.params()["covg"] > 20 and c.locus_reads[OUTLIER] > 0
        assert ox.names[OUTLIER] not in vcf_contigs(og) and len(vcf_contigs(og)) == ox.n_loci - 1
    return build, regime


def _all_zero():
    def build():
        c = real_case("panel")
        c.fwd[:], c.rev[:] = 0, 0
        return c

    def regime(c, og):
        assert og.params()["covg"] > 20
        assert (c.locus_reads > 0).all() and vcf_contigs(og) == [] and vcf_body(og) == []
    return build, regime


def _hist_edge():
    def build():
        c = real_case("panel")
        ox = oracle_index(c.prg)
        idx = np.flatnonzero(inner_mask(ox))[::7]
        tot = np.array([999, 1000, 1000, 1001] * (len(idx) // 4 + 1))[:len(idx)]
        c.fwd[idx], c.rev[idx] = split(tot)
        c.total_bases = 20 * c.genome_size  # covg 20: no coverage filter
        return c

    def regime(c, og):
        ox = oracle_index(c.prg)
        cov = (c.fwd + c.rev)[inner_mask(ox)]
        assert (cov == 999).sum() > 50 and (cov == 1000).sum() > 100 and (cov == 1001).sum() > 50
        assert len(vcf_contigs(og)) == ox.n_loci
    return build, regime


# Not here: an ML path that spells a TOO_MANY_ALTS record.  Random, tied and zero coverage on the toy PRG and
# small_panel, with and without --vcf-refs, and hand-built PRGs with adjacent sites, empty alleles and nested sites never
# produced one in the oracle: every stretch where such an ML path leaves the reference path is an allele of the site
# table.  A clamped nb_p cannot empty the score histogram either (its nodes near the mean score about -3), so the -200
# threshold is reached under the fallback model (fit_empty_prob_hist); fit_nb_clamped reaches -200 on its own.
CASES = {
    "ties_uniform_toy": _uniform("toy"), "ties_uniform_panel": _uniform("panel"),
    "ties_zero_loci_panel": _zero_loci("panel"),
    "ties_rounded_toy": _rounded("toy"), "ties_rounded_panel": _rounded("panel"),
    "saturated": _saturated(),
    "fit_nb_clamped": _nb_clamped(), "fit_empty_prob_hist": _empty_prob_hist(), "fit_mean_ge_var": _mean_ge_var(),
    "fit_few_reads": _few_reads(), "fit_low_covg": _low_covg(), "fit_absent_locus": _absent_locus(),
    "fit_no_locus": _no_locus(), "fit_cov_hist_edge": _hist_edge(),
    "slow_outlier_locus": _outlier(), "slow_all_zero": _all_zero(),
}


def built(name):
    key = ("case", name)
    if key not in _cache:
        _cache[key] = CASES[name][0]()
    return _cache[key]


# ------------------------------------------------------------------------ panels for the generic ML-path kernel
def mlpath_sizing(ox):
    """launch_mlpath's choice for this index at pandora's window (100): whether the level-parallel kernel's shared
    memory fits, and the generic kernel's shared-memory sizing and which loci fit it"""
    n_out = ox.knodes()["n_out"].astype(np.int64)
    kb = ox.knode_base.astype(np.int64)
    nodes = np.diff(kb)
    edges = np.array([n_out[kb[l]:kb[l + 1]].sum() for l in range(ox.n_loci)])
    mn, me = int(nodes.max()), int(edges.max())
    level_smem = (mn + 1) * 64 + (me + 1) * 4 + mn * 12 + 32
    per_node = 24 + 4 + 4 * 7 + 4  # 7 lifting levels for a window of 100
    smem_nodes, smem_edges = (mn + 3) & ~1, me + 2
    halved = smem_nodes * per_node + 16 + 4 * smem_edges > SMEM_BUDGET
    if halved:
        smem_nodes, smem_edges = ((SMEM_BUDGET // 2) // per_node) & ~1, (SMEM_BUDGET // 2) // 4
    in_smem = (nodes <= smem_nodes) & (edges <= smem_edges)
    return dict(level_fits=level_smem <= SMEM_BUDGET, halved=halved, in_smem=in_smem, nodes=nodes, edges=edges)


def _dense_panel(big):
    """dense loci (a site every 4 bp) of the given (length, seed), then three loci of the small_panel kind (PRG text, refs)"""
    key = ("dense", big)
    if key not in _cache:
        loci = []
        for i, (L, seed) in enumerate(big):
            l = sim.make_panel(seed=seed, n_loci=1, n_sites=L // 4, len_lo=L, len_hi=L).loci[0]
            loci.append(sim.Locus(f"big{i}", l.parts, l.ref))
        loci += sim.make_panel(seed=7, n_loci=3, n_sites=200, len_lo=500, len_hi=900).loci
        p = sim.Panel(loci)
        d = tempfile.mkdtemp(prefix="drprg_dense_")
        _cache[key] = p.write(d)
    return _cache[key]


DENSE = {"smem_3k": ((1150, 3),), "global_9k": ((9000, 4), (6000, 5))}


def dense_regime(name, ox):
    s = mlpath_sizing(ox)
    assert not s["level_fits"]  # the level-parallel kernel is refused: every locus takes mlpath_kernel
    if name == "smem_3k":  # ~3 000 nodes: every locus in shared memory
        assert not s["halved"] and s["in_smem"].all() and s["nodes"].max() > 3000
    else:  # shared memory sized for half the budget: the two big loci run from global memory, side by side
        assert s["halved"] and (~s["in_smem"]).sum() == 2 and s["in_smem"][2:].all() and s["nodes"].max() > 24_000


def dense_cases(name):
    prg, refs = _dense_panel(DENSE[name])
    ox = oracle_index(prg)
    n, gs = ox.total_knodes, 100_000
    rng = np.random.default_rng(len(name))
    lr = np.full(ox.n_loci, 200)
    random = Case(prg, refs, rng.integers(0, 40, n), rng.integers(0, 40, n), lr, 40 * gs, gs)
    tied = Case(prg, refs, np.full(n, 20), np.full(n, 20), lr, 40 * gs, gs)
    f, r = rng.integers(30_000, 90_000, n), rng.integers(20_000, 70_000, n)
    saturated = Case(prg, refs, f, r, lr, 10_000 * gs, gs)
    return dict(random=random, tied=tied, saturated=saturated)


# --------------------------------------------------------------------------------------------------------- the tests
def test_constructions_reach_their_regimes():
    """no GPU: every construction, genotyped by the oracle alone, reaches the regime it is named for, and the dense
    panels have the sizes that send their loci to the generic ML-path kernel's shared- and global-memory branches"""
    for name in CASES:
        c = built(name)
        CASES[name][1](c, c.oracle())
    for name in DENSE:
        dense_regime(name, oracle_index(_dense_panel(DENSE[name])[0]))
    sat = dense_cases("global_9k")["saturated"]
    assert (sat.fwd > SAT).any() and (sat.rev < SAT).any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_constructed_coverage_matches_oracle(name):
    c = built(name)
    og = genotype_both(c)
    CASES[name][1](c, og)


@pytest.mark.gpu
def test_saturated_values_leave_the_device_formatter():
    """likelihoods of saturated alleles print in exponent notation, which the device's "%g" refuses: the text comes from
    the host formatter, with no environment switch, and equals the oracle's (test_constructed_coverage_matches_oracle)"""
    import ctypes as C
    from drprg_b200 import lib
    v = np.ascontiguousarray(exponent_values(built("saturated").oracle()), np.float64)
    n = len(v)
    assert n > 0
    out, ln, refused = np.zeros(48 * n, np.uint8), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    rc = lib.lib().drprg_cuda_format_g6_device(C.c_int(0), v.ctypes.data_as(C.c_void_p), C.c_uint32(n),
                                               out.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p),
                                               refused.ctypes.data_as(C.c_void_p))
    assert rc == 0 and refused.all()
    gx = gpu_index(built("saturated").prg)
    genotype_both(built("saturated"), gx)
    text = gx.vcf()
    assert any(("%g" % x) in text for x in v.tolist())


@pytest.mark.gpu
def test_consecutive_samples_on_one_handle():
    """batch mode keeps the record lists and site tables of one genotype() call for the next: a sequence of samples
    whose outcome changes (a locus dropped, saturated strands) with --vcf-refs switched on and off, on one handle, each
    equal to a fresh oracle run"""
    from drprg_b200 import lib
    prg = realistic("panel")[0]
    gx = lib.Index(prg, W, K, device=0)
    clean = real_case("panel")
    refs = clean.refs
    seq = [(clean, refs), (built("slow_outlier_locus"), None), (clean, refs), (built("saturated"), None),
           (clean, None), (built("slow_outlier_locus"), refs), (clean, refs)]
    for c, r in seq:
        c = Case(c.prg, r, c.fwd, c.rev, c.locus_reads, c.total_bases, c.genome_size)
        genotype_both(c, gx)


@pytest.mark.gpu
@pytest.mark.parametrize("panel", list(DENSE))
def test_generic_mlpath_kernel_without_the_switch(panel):
    """a locus too large for the level-parallel kernel sends every locus to the generic kernel: with ~3 000 nodes all
    of them in shared memory; with 27 k and 19 k nodes shared memory is sized for half the budget, the two big loci run
    from global memory side by side and the small ones stay in shared memory"""
    prg = _dense_panel(DENSE[panel])[0]
    dense_regime(panel, oracle_index(prg))
    for kind, c in dense_cases(panel).items():
        og = genotype_both(c)
        assert len(vcf_contigs(og)) > 0, kind


@pytest.mark.gpu
def test_constructed_coverage_under_the_generic_kernel():
    """the same constructions through the generic ML-path kernel (DRPRG_MLPATH_GENERIC=1, read once per process)"""
    e = dict(os.environ, DRPRG_MLPATH_GENERIC="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "constructed_coverage_matches_oracle or consecutive_samples"], env=e, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
