"""discover/denovo_paths.txt as restated in tests/denovo_paths_oracle.py, on hand-built alleles (no GPU): the variant form
(alignment, traceback placement, anchoring, union over regions) and the file read back by the restated drprg and make_prg
readers."""
import denovo_paths_oracle as P


def test_snp():
    cons = "ACGTACGTAC"
    assert P.allele_variants(cons, 2, 8, "GTTCGT") == [(5, "A", "T")]


def test_two_snps_separated_by_a_match_are_two_records():
    cons = "ACGTACGTAC"
    assert P.allele_variants(cons, 2, 8, "GCAAGT") == [(4, "T", "C"), (6, "C", "A")]


def test_deletion_in_a_homopolymer_is_placed_by_the_traceback():
    """the traceback from the end takes the diagonal first, so the deleted bases are the leftmost of the run, and the
    deletion is anchored by the consensus base before it"""
    cons = "TTCGAAAAAAGCTT"
    assert P.allele_variants(cons, 2, 12, "CGAAAGC") == [(4, "GAAA", "G")]


def test_insertion_is_anchored_by_the_base_before_it():
    cons = "TTCGATGCTT"
    assert P.allele_variants(cons, 2, 8, "CGACCCTGC") == [(5, "A", "ACCC")]


def test_an_open_gap_is_extended_so_one_indel_is_one_record():
    """CTGC inserted after GGAT: a traceback that always takes the diagonal first aligns A--T--CACAGTCT against
    ATCTGCCACAGTCT, two insertions (TC, GC) of equal cost; extending the open gap keeps the insertion one record"""
    cons = "GGATCACAGTCTAC"
    assert P.allele_variants(cons, 2, 12, "ATCTGCCACAGTCT") == [(4, "T", "TCTGC")]


def test_indel_at_the_first_base_is_anchored_by_the_base_after_it():
    cons = "TTAAACGT"
    assert P.allele_variants(cons, 2, 8, "AACGT") == [(3, "AA", "A")]
    assert P.allele_variants(cons, 2, 8, "GAAACGT") == [(3, "A", "GA")]


def test_a_variant_from_two_overlapping_regions_is_listed_once():
    cons = "TTCGATGCTTGACCA"
    allele = "CGTTGC"  # cons[2:8] = CGATGC with A -> T
    wider = cons[1] + allele + cons[8]
    assert P.allele_variants(cons, 2, 8, allele) == P.allele_variants(cons, 1, 9, wider) == [(5, "A", "T")]
    assert P.locus_variants(cons, [(2, 8, allele), (1, 9, wider), (9, 14, "TGTCC")]) == [(5, "A", "T"), (12, "A", "T")]


def test_file_read_back_by_drprg_and_make_prg_readers():
    loci = [
        ("geneA", [(0, 0, 5, "ACGTA"), (2, 9, 12, "CCG"), (7, 45, 45, "")], [(3, "G", "T"), (7, "C", "CAT")]),
        ("geneB", [(0, 0, 4, "TTGA")], []),
        ("geneC", [(0, 0, 6, "GGGCCC")], [(1, "GG", "G")]),
    ]
    text = P.denovo_paths_text("mysample", loci)
    assert text.splitlines()[:6] == ["1 samples", "Sample mysample", "2 loci with denovo variants", "geneA", "3 nodes", "(0 [0, 5) ACGTA)"]
    assert "(7 [45, 45) )" in text.splitlines()
    assert P.drprg_loci(text) == (2, ["geneA", "geneC"])
    sample, got = P.read_denovo_paths(text)
    assert sample == "mysample"
    assert got == {name: (nodes, variants) for name, nodes, variants in loci if variants}


def test_a_sample_without_variants():
    text = P.denovo_paths_text("s", [("geneB", [(0, 0, 4, "TTGA")], [])])
    assert text == "1 samples\nSample s\n0 loci with denovo variants\n"
    assert P.drprg_loci(text) == (0, [])
    assert P.read_denovo_paths(text) == ("s", {})
