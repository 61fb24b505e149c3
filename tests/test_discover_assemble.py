"""The local assembler of `pandora discover` as the oracle restates it (tests/denovo_oracle.py): one hand-built pileup per
outcome.  The GPU kernel is held to this restatement in tests/test_gpu_discover_assemble.py."""
import numpy as np

import denovo_oracle as D

K = D.DISCOVER_K
COMP = str.maketrans("ACGT", "TGCA")


def consensus(n, seed=3):
    rng = np.random.default_rng(seed)
    while True:
        s = "".join("ACGT"[x] for x in rng.integers(0, 4, n))
        kmers = [s[p:p + K - 1] for p in range(n - K + 2)]
        if len(set(kmers)) == len(kmers):  # no repeated (K-1)-mer: the consensus alone spells exactly one walk
            return s


def run(cons, ps, pe, s, e, seqs, reverse_every=0):
    """the region through assemble(): every reverse_every-th read arrives reverse-complemented with fwd = 0"""
    read_seqs, reads = {}, []
    for i, q in enumerate(seqs):
        rev = reverse_every and i % reverse_every == 0
        read_seqs[i] = "GG" + (q.translate(COMP)[::-1] if rev else q) + "TT"
        reads.append((i, 2, 2 + len(q), 0 if rev else 1))
    loci = {0: (cons, None)}
    return D.assemble(loci, [(0, s, e, ps, pe, reads)], read_seqs)[0]


def sub(seq, pos, base):
    return seq[:pos] + base + seq[pos + 1:]


def test_snp_bubble_gives_one_allele():
    cons = consensus(80)
    alt_base = "ACGT"[("ACGT".index(cons[40]) + 1) % 4]
    alt = sub(cons, 40, alt_base)
    st, a, b, paths = run(cons, 0, 80, 30, 50, [cons] * 3 + [alt] * 3, reverse_every=2)
    assert (st, a, b) == (D.ASSEMBLED, 0, 80)
    assert paths == [alt]


def test_insertion_of_six_bases_gives_one_allele():
    cons = consensus(80)
    alt = cons[:40] + "ACGTTG" + cons[40:]
    st, a, b, paths = run(cons, 0, 80, 30, 50, [alt] * 4)
    assert (st, a, b) == (D.ASSEMBLED, 0, 80)
    assert paths == [alt]


def test_deletion_of_three_bases_gives_one_allele():
    cons = consensus(80)
    alt = cons[:40] + cons[43:]
    st, a, b, paths = run(cons, 0, 80, 30, 50, [alt] * 4, reverse_every=3)
    assert (st, a, b, paths) == (D.ASSEMBLED, 0, 80, [alt])


def test_agreeing_reads_assemble_to_no_allele():
    cons = consensus(80)
    assert run(cons, 0, 80, 30, 50, [cons] * 5) == (D.ASSEMBLED, 0, 80, [])


def test_unsolid_first_anchor_falls_through_to_the_next_pair():
    """no read covers the first base: the pair (i = 1, j = 0) decides the region"""
    cons = consensus(80)
    st, a, b, paths = run(cons, 0, 80, 30, 50, [cons[1:]] * 3)
    assert (st, a, b, paths) == (D.ASSEMBLED, 1, 80, [])
    # the last base is not covered either: (1, 1)
    st, a, b, paths = run(cons, 0, 80, 30, 50, [cons[1:-1]] * 3)
    assert (st, a, b, paths) == (D.ASSEMBLED, 1, 79, [])


def test_more_than_the_maximum_of_walks_abandons_the_region():
    """five independent SNP bubbles, both alleles solid at each: 2^5 = 32 walks > 25"""
    cons = consensus(120, seed=5)
    seqs = [cons] * 3
    for pos in (30, 45, 60, 75, 90):
        alt = sub(cons, pos, "ACGT"[("ACGT".index(cons[pos]) + 2) % 4])
        seqs += [alt[pos - 15:pos + 16]] * 3
    st, a, b, paths = run(cons, 0, 120, 20, 100, seqs)
    assert (st, paths) == (D.TOO_MANY_PATHS, [])
    # four bubbles (16 walks) still assemble: 15 alleles besides the consensus
    st, a, b, paths = run(cons, 0, 120, 20, 100, seqs[:-3])
    assert st == D.ASSEMBLED and len(paths) == 15 and paths == sorted(paths)


def test_flank_shorter_than_k_has_no_anchor():
    cons = consensus(80)
    assert run(cons, 0, 80, K - 1, 50, [cons] * 5)[0] == D.NO_ANCHOR
    assert run(cons, 0, 80, 30, 80 - K + 1, [cons] * 5)[0] == D.NO_ANCHOR


def test_anchors_without_a_path_between_them():
    """both flanks are solid but no read spans the region"""
    cons = consensus(80)
    st, a, b, paths = run(cons, 0, 80, 30, 50, [cons[:35]] * 3 + [cons[45:]] * 3)
    assert (st, a, b, paths) == (D.NO_PATH, 0, 80, [])
