"""ORACLE — TEST INFRASTRUCTURE ONLY.  CPU restatement (plain Python, small inputs) of the local assembler of `pandora
discover` that drprg launches at src/predict.rs:247-256 -> src/lib.rs:513-578: the second half of discover, after the
candidate regions and their reads (oracle/discover_py.py).  Upstream pandora runs a GATB de Bruijn graph
(denovo_discovery/local_assembly.cpp); its source is not in the reference tree, so parity is unpinned and this restatement is the
arbiter the GPU kernel (drprg_b200/csrc/assemble.cu) is held to.  Every choice marked [P] is this restatement's, not a
pinned upstream behaviour; README lists them under known risks."""

DISCOVER_K = 11            # discover -k: de Bruijn graph k-mer size
MIN_DBG_DP = 2             # --min-dbg-dp: a k-mer seen this often is solid [P: absolute count, no GATB abundance model]
KMER_ATTEMPTS = 10         # anchor k-mers tried per flank
MAX_INSERTION = 15         # --max-ins: a walk may spell this many bases more than the consensus it replaces
MAX_CANDIDATE_PATHS = 25   # --max-num-candidate-paths: more complete walks abandon the region

ASSEMBLED, NO_ANCHOR, TOO_MANY_PATHS, NO_PATH = 0, 1, 2, 3  # region status
_COMP = str.maketrans("ACGT", "TGCA")


def pileup(read_seqs, reads):
    """the region reads in consensus orientation: [start, end) of each read, reverse-complemented when fwd == 0"""
    out = []
    for rd, st, en, fw in reads:
        s = read_seqs[rd][st:en]
        out.append(s if fw else s.translate(_COMP)[::-1])
    return out


def kmer_counts(seqs, k=DISCOVER_K):
    """oriented k-mer counts [P: not canonical, unlike GATB's bidirected graph]"""
    c = {}
    for s in seqs:
        for p in range(len(s) - k + 1):
            x = s[p:p + k]
            c[x] = c.get(x, 0) + 1
    return c


def assemble_region(cons, ps, pe, s, e, seqs, k=DISCOVER_K, min_dbg_dp=MIN_DBG_DP, max_insertion=MAX_INSERTION,
                    max_candidate_paths=MAX_CANDIDATE_PATHS):
    """-> (status, a, b, sorted de-novo alleles replacing cons[a:b]); a = b = 0 unless an anchor pair was found"""
    counts = kmer_counts(seqs, k)
    solid = lambda x: counts.get(x, 0) >= min_dbg_dp
    starts = [i for i in range(KMER_ATTEMPTS) if ps + i + k <= s]
    ends = [j for j in range(KMER_ATTEMPTS) if pe - k - j >= e]
    pair = next(((i, j) for i in starts for j in ends if solid(cons[ps + i:ps + i + k]) and solid(cons[pe - k - j:pe - j])), None)
    if pair is None:
        return NO_ANCHOR, 0, 0, []
    i, j = pair
    a, b = ps + i, pe - j
    start, end, max_len = cons[a:a + k], cons[b - k:b], (b - a) + max_insertion
    walks = []
    stack = [start]  # depth first, A C G T in that order; a walk ends where it first reaches the end anchor [P]
    while stack:
        w = stack.pop()
        if w[-k:] == end:
            walks.append(w)
            if len(walks) > max_candidate_paths:
                return TOO_MANY_PATHS, a, b, []
            continue
        if len(w) + 1 > max_len:
            continue
        for x in "TGCA":  # pushed in reverse: A is explored first
            if solid(w[1 - k:] + x):
                stack.append(w + x)
    if not walks:
        return NO_PATH, a, b, []
    return ASSEMBLED, a, b, sorted(w for w in walks if w != cons[a:b])


def assemble(loci, regions, read_seqs, **opts):
    """loci / regions as discover() returns them, read_seqs[read id] = read bases -> [(status, a, b, [alleles])] per region"""
    return [assemble_region(loci[r[0]][0], r[3], r[4], r[1], r[2], pileup(read_seqs, r[5]), **opts) for r in regions]
