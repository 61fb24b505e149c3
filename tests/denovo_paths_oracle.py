"""ORACLE — TEST INFRASTRUCTURE ONLY.  Restatement of the file `pandora discover` leaves for drprg, discover/denovo_paths.txt,
built from the discover front half (oracle/discover_py.py) and the local assembler (tests/denovo_oracle.py).  Every choice
here is [P]: pandora 0.10's writer and make_prg update's reader are restated, not checked against a pandora binary.

  variants   a de-novo allele A replaces R = cons[a:b]; R and A are aligned globally with unit-cost edit distance, the
             traceback from the end extends an open gap while that stays optimal, and otherwise prefers the diagonal (match
             or substitution), then a deletion (a base of R), then an insertion.  Each maximal run of non-match columns is
             one variant (1-based pos on the ML sequence, ref, alt).  A run with an empty side is anchored by the consensus
             base before it, or by the base after it when it starts at R[0].
             The variants of a locus are the union over its regions' alleles, distinct, sorted by (pos, ref, alt).
  file       "1 samples", "Sample <name>", "<L> loci with denovo variants", then per locus with a variant (PRG order) its
             name, "<M> nodes", one "(<id> [<start>, <end>) <seq>)" line per node of its ML local path, "<V> variants found"
             and one "<pos>\\t<ref>\\t<alt>" line per variant.
"""
import re

import denovo_oracle as A
import discover_py as D
import oracle_py as O


def allele_variants(cons, a, b, allele):
    """-> [(pos, ref, alt)] of one de-novo allele replacing cons[a:b]"""
    R, Al = cons[a:b], allele
    n, m = len(R), len(Al)
    d = [[0] * (m + 1) for _ in range(n + 1)]
    for i in range(n + 1):
        d[i][0] = i
    for j in range(m + 1):
        d[0][j] = j
    for i in range(1, n + 1):
        for j in range(1, m + 1):
            d[i][j] = min(d[i - 1][j - 1] + (R[i - 1] != Al[j - 1]), d[i - 1][j] + 1, d[i][j - 1] + 1)
    cols, i, j, op = [], n, m, None  # (R index or None, allele index or None); op: the last column's kind
    while i or j:
        diag = i and j and d[i][j] == d[i - 1][j - 1] + (R[i - 1] != Al[j - 1])
        dele = i and d[i][j] == d[i - 1][j] + 1
        ins = j and d[i][j] == d[i][j - 1] + 1
        if op == "D" and dele or op == "I" and ins:
            pass  # an open gap is extended
        else:
            op = "M" if diag else "D" if dele else "I"
        if op != "I":
            i -= 1
        if op != "D":
            j -= 1
        cols.append((i if op != "I" else None, j if op != "D" else None))
    cols.reverse()
    match = lambda c: c[0] is not None and c[1] is not None and R[c[0]] == Al[c[1]]
    out, ri, c = [], 0, 0
    while c < len(cols):
        if match(cols[c]):
            ri, c = ri + 1, c + 1
            continue
        i0, ref, alt = ri, "", ""
        while c < len(cols) and not match(cols[c]):
            if cols[c][0] is not None:
                ref += R[cols[c][0]]
                ri += 1
            if cols[c][1] is not None:
                alt += Al[cols[c][1]]
            c += 1
        pos = a + i0 + 1
        if not ref or not alt:
            if i0 == 0 and a + ri < len(cons):
                ref, alt = ref + cons[a + ri], alt + cons[a + ri]
            elif a + i0 > 0:
                x = cons[a + i0 - 1]
                ref, alt, pos = x + ref, x + alt, pos - 1
        out.append((pos, ref, alt))
    return out


def locus_variants(cons, alleles):
    """alleles = [(a, b, sequence)] of one locus -> its distinct variants, sorted by (pos, ref, alt)"""
    return sorted({v for a, b, s in alleles for v in allele_variants(cons, a, b, s)})


def denovo_paths_text(sample, loci):
    """loci = [(name, [(node id, start, end, seq)], [(pos, ref, alt)])] in PRG order; loci without variants are left out"""
    loci = [l for l in loci if l[2]]
    out = ["1 samples", f"Sample {sample}", f"{len(loci)} loci with denovo variants"]
    for name, nodes, variants in loci:
        out.append(name)
        out.append(f"{len(nodes)} nodes")
        out += [f"({n} [{s}, {e}) {q})" for n, s, e, q in nodes]
        out.append(f"{len(variants)} variants found")
        out += [f"{p}\t{r}\t{a}" for p, r, a in variants]
    return "\n".join(out) + "\n"


_DRPRG_COUNT = re.compile(r"^(?P<n>\d+) loci with denovo variants$")  # drprg src/lib.rs:648-697
_NODE = re.compile(r"^\((\d+) \[(\d+), (\d+)\) ([ACGTN]*)\)$")


def drprg_loci(text):
    """drprg's reader: the `N loci with denovo variants` count and the gene names, each the line before `… nodes`"""
    lines = text.splitlines()
    n = next(int(m["n"]) for m in map(_DRPRG_COUNT.match, lines) if m)
    genes = [lines[i - 1] for i, l in enumerate(lines) if l.endswith(" nodes") and i > 0]
    return n, genes


def read_denovo_paths(text):
    """make_prg update's reader: -> (sample, {locus: ([(node id, start, end, seq)], [(pos, ref, alt)])}); lines are
    stripped and tab-split, so no field may be empty"""
    lines = [l.strip() for l in text.splitlines()]
    assert lines[0] == "1 samples" and lines[1].startswith("Sample ")
    sample, n_loci = lines[1][len("Sample "):], int(lines[2].split()[0])
    out, i = {}, 3
    for _ in range(n_loci):
        name, n_nodes = lines[i], int(lines[i + 1].split()[0])
        nodes = []
        for l in lines[i + 2:i + 2 + n_nodes]:
            m = _NODE.match(l)
            assert m, l
            nodes.append((int(m[1]), int(m[2]), int(m[3]), m[4]))
        i += 2 + n_nodes
        n_var = int(lines[i].split()[0])
        variants = []
        for l in lines[i + 1:i + 1 + n_var]:
            f = l.split("\t")
            assert len(f) == 3 and all(f), l
            variants.append((int(f[0]), f[1], f[2]))
        out[name] = (nodes, variants)
        i += 1 + n_var
    assert i == len(lines)
    return sample, out


def file_from(ox, text_lines, mlpaths, loci, regions, results, sample="sample"):
    """the restated file from discover's front half (loci, regions as discover_py.discover returns them), the assembler's
    results per region (denovo_oracle.assemble) and the ML k-mer path of every present locus (mlpaths[locus])"""
    alleles = {}
    for r, (status, a, b, seqs) in zip(regions, results):
        alleles.setdefault(r[0], []).extend((a, b, s) for s in seqs)
    out = []
    for locus in range(ox.n_loci):
        if locus not in loci:
            continue
        starts, lens, adj, kpaths = D._locus_tables(ox, locus)
        lp = D.local_path(starts, lens, adj, kpaths, list(mlpaths[locus]))
        body = text_lines[2 * locus + 1]
        nodes = [(n, int(starts[n]), int(starts[n] + lens[n]), body[starts[n]:starts[n] + lens[n]]) for n in lp]
        out.append((text_lines[2 * locus][1:].split()[0], nodes, locus_variants(loci[locus][0], alleles.get(locus, []))))
    return denovo_paths_text(sample, out)


def oracle_file(prg, d, o, genome_size, sample="sample", illumina=True, **asm):
    """the restated denovo_paths.txt of reads (d, o) against prg, genotyped without --vcf-refs -> (text, loci, regions)"""
    ox = O.Index(prg, 11, 15)
    oo = O.make_opts(illumina=illumina, genome_size=genome_size)
    mr = O.MapRun(ox, d, o, oo)
    og = O.Genotype(ox, mr, oo, None)
    text_lines = open(prg).read().splitlines()
    loci, regions = D.discover(ox, mr, og, text_lines)
    reads = [d[int(o[i]):int(o[i + 1])].tobytes().decode() for i in range(len(o) - 1)]
    results = A.assemble(loci, regions, reads, **asm)
    mlpaths = {l: og.mlpath(l).tolist() for l in loci}
    return file_from(ox, text_lines, mlpaths, loci, regions, results, sample), loci, regions

