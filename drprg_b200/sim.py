"""Synthetic panels, genomes and reads for the map hot path (SURVEY.md §8d configs).

Nothing here is on the measured path: it only makes inputs (PRG text in pandora's format, a
--vcf-refs FASTA, a genome with the loci embedded and simulated reads) with fixed seeds so that
tests, bench.py and the CPU baseline all see the same bytes.

PRG grammar (reference fixture /root/reference/tests/cases/expected/dr.prg, SURVEY.md A.1): tokens
separated by single spaces; odd marker n opens and closes site n, n+1 separates its alleles; sites
are numbered 5,7,9,... in depth-first order per locus; alleles may be empty and may nest.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

BASES = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = np.zeros(256, np.uint8)
for a, b in zip(b"ACGTNacgtn", b"TGCANtgcan"):
    _COMP[a] = b
_CODE = np.full(256, 4, np.uint8)
for i, c in enumerate(b"ACGT"):
    _CODE[c] = i
    _CODE[c + 32] = i


def random_dna(rng, n, gc=0.65):
    p = np.array([(1 - gc) / 2, gc / 2, gc / 2, (1 - gc) / 2])
    return BASES[rng.choice(4, size=n, p=p)]


def revcomp(a):
    return _COMP[a[::-1]]


# --------------------------------------------------------------------------------------------
@dataclass
class Site:
    """One variation site: alleles[0] is the reference allele.  An allele is a list of parts,
    each part either bytes (sequence) or a nested Site."""
    alleles: list
    ref_start: int = 0  # offset of the site on the locus reference sequence


@dataclass
class Locus:
    name: str
    parts: list  # bytes | Site, alternating sequence / site
    ref: bytes = b""

    def prg_text(self):
        counter = [5]

        def emit(parts):
            toks = []
            for p in parts:
                if isinstance(p, (bytes, bytearray)):
                    toks.append(p.decode())
                else:
                    n = counter[0]
                    counter[0] += 2
                    toks.append(str(n))
                    for i, al in enumerate(p.alleles):
                        if i:
                            toks.append(str(n + 1))
                        toks.extend(emit_allele(al))
                    toks.append(str(n))
            return toks

        def emit_allele(al):
            # an allele must start and end with a sequence token (possibly empty)
            parts = list(al)
            if not parts or not isinstance(parts[0], (bytes, bytearray)):
                parts.insert(0, b"")
            if not isinstance(parts[-1], (bytes, bytearray)):
                parts.append(b"")
            return emit(parts)

        parts = list(self.parts)
        if not isinstance(parts[0], (bytes, bytearray)):
            parts.insert(0, b"")
        if not isinstance(parts[-1], (bytes, bytearray)):
            parts.append(b"")
        return " ".join(emit(parts))

    def spell(self, chooser):
        """Sequence of the path where chooser(site) -> allele index (called depth-first)."""
        out = bytearray()

        def go(parts):
            for p in parts:
                if isinstance(p, (bytes, bytearray)):
                    out.extend(p)
                else:
                    go(p.alleles[chooser(p)])

        go(self.parts)
        return bytes(out)


@dataclass
class Panel:
    loci: list
    seed: int = 0

    def prg_text(self):
        return "".join(f">{l.name}\n{l.prg_text()}\n" for l in self.loci)

    def refs_fasta(self):
        return "".join(f">{l.name}\n{l.ref.decode()}\n" for l in self.loci)

    def write(self, outdir, stem="dr"):
        os.makedirs(outdir, exist_ok=True)
        prg = os.path.join(outdir, f"{stem}.prg")
        fa = os.path.join(outdir, "genes.fa")
        with open(prg, "w") as f:
            f.write(self.prg_text())
        with open(fa, "w") as f:
            f.write(self.refs_fasta())
        return prg, fa


def make_panel(seed=20231017, n_loci=30, n_sites=5000, len_lo=800, len_hi=3800, gc=0.65, min_gap=1,
               frac=(0.85, 0.08, 0.06, 0.01)):
    """Synthetic M. tuberculosis-scale panel (SURVEY §8d config 2).  Site mix: biallelic SNP,
    multi-allelic SNP/MNP (2-4 alts), indel 1-20 bp (anchored), nested (a SNP inside an allele)."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(len_lo, len_hi + 1, size=n_loci)
    per = np.maximum(0, np.floor(n_sites * lens / lens.sum()).astype(int))
    loci = []
    for li in range(n_loci):
        L = int(lens[li])
        ref = random_dna(rng, L, gc)
        want = int(per[li])
        # choose site starts with spacing; keep 30 bp clear at both ends
        cand = np.sort(rng.choice(np.arange(30, L - 60), size=min(want, max(0, (L - 90) // 2)), replace=False))
        parts, cur = [], 0
        for s in cand:
            s = int(s)
            if s < cur + min_gap:
                continue
            kind = rng.choice(4, p=frac)
            if kind == 0:  # SNP
                rlen = 1
                r = ref[s:s + 1].tobytes()
                alt = BASES[(int(_CODE[ref[s]]) + int(rng.integers(1, 4))) % 4:][:1].tobytes()
                site = Site([[r], [alt]])
            elif kind == 1:  # multi-allelic SNP / MNP
                rlen = int(rng.integers(1, 5))
                r = ref[s:s + rlen].tobytes()
                alts = set()
                for _ in range(int(rng.integers(2, 5))):
                    a = bytearray(r)
                    j = int(rng.integers(0, rlen))
                    a[j] = int(BASES[(int(_CODE[a[j]]) + int(rng.integers(1, 4))) % 4])
                    if bytes(a) != r:
                        alts.add(bytes(a))
                site = Site([[r]] + [[a] for a in sorted(alts)])
            elif kind == 2:  # indel with anchor base
                n = int(rng.integers(1, 21))
                if rng.random() < 0.5:  # deletion
                    rlen = 1 + n
                    r = ref[s:s + rlen].tobytes()
                    site = Site([[r], [r[:1]]])
                else:
                    rlen = 1
                    r = ref[s:s + 1].tobytes()
                    site = Site([[r], [r + random_dna(rng, n, gc).tobytes()]])
            else:  # nested: ref allele = x (SNP) y ; alt allele = different block
                rlen = int(rng.integers(6, 13))
                r = ref[s:s + rlen].tobytes()
                j = int(rng.integers(1, rlen - 1))
                alt_b = BASES[(int(_CODE[r[j]]) + int(rng.integers(1, 4))) % 4:][:1].tobytes()
                inner = Site([[r[j:j + 1]], [alt_b]])
                other = random_dna(rng, int(rng.integers(4, 16)), gc).tobytes()
                if other == r:
                    other = other + b"A"
                site = Site([[r[:j], inner, r[j + 1:]], [other]])
            if s + rlen > L - 30:
                continue
            site.ref_start = s
            parts.append(ref[cur:s].tobytes())
            parts.append(site)
            cur = s + rlen
        parts.append(ref[cur:].tobytes())
        loci.append(Locus(f"g{li:02d}", parts, ref.tobytes()))
    return Panel(loci, seed)


def sample_haplotype(panel, seed, alt_frac=0.10):
    """Per locus: the sample's sequence (alt allele at ~alt_frac of sites) and the choices."""
    rng = np.random.default_rng(seed)
    out = []
    for l in panel.loci:
        choices = []

        def chooser(site):
            c = 0
            if rng.random() < alt_frac:
                c = int(rng.integers(1, len(site.alleles)))
            choices.append(c)
            return c

        out.append((l.spell(chooser), choices))
    return out


def insert_novel_variants(panel, hap, kinds, seed=0):
    """Variants the PRG does not know, in the sample's locus sequences: kinds[i] in ("snp", "del3", "ins6") goes into locus i,
    in the middle of its longest stretch between sites.  hap = sample_haplotype(panel, ...).  Returns (sequences,
    [(locus, offset, ref_len, alt, sequence without the variant)])."""
    rng = np.random.default_rng(seed)

    def spell(parts, it):  # replays the site choices of sample_haplotype, depth first like Locus.spell
        out = bytearray()
        for q in parts:
            out += q if isinstance(q, (bytes, bytearray)) else spell(q.alleles[next(it)], it)
        return bytes(out)

    seqs, variants = [h[0] for h in hap], []
    for li, kind in enumerate(kinds):
        L = panel.loci[li]
        i = max((j for j, q in enumerate(L.parts) if isinstance(q, (bytes, bytearray))), key=lambda j: len(L.parts[j]))
        v = len(spell(L.parts[:i], iter(hap[li][1]))) + len(L.parts[i]) // 2
        old = seqs[li]
        if kind == "snp":
            ref_len, alt = 1, BASES[(int(_CODE[old[v]]) + int(rng.integers(1, 4))) % 4:][:1].tobytes()
        elif kind == "del3":
            ref_len, alt = 3, b""
        else:
            ref_len, alt = 0, random_dna(rng, 6).tobytes()
        seqs[li] = old[:v] + alt + old[v + ref_len:]
        variants.append((li, v, ref_len, alt.decode(), old.decode()))
    return seqs, variants


def make_genome(panel, hap_seqs, size=4_411_532, seed=1, gc=0.65, min_sep=5000):
    """Random genome with the sample's locus sequences embedded (random strand, >= min_sep apart)."""
    rng = np.random.default_rng(seed)
    g = random_dna(rng, size, gc)
    n = len(hap_seqs)
    slots = np.sort(rng.choice(np.arange(1, size // (min_sep * 2) - 1), size=n, replace=False)) * (min_sep * 2)
    placements = []
    for s, seq in zip(slots, hap_seqs):
        a = np.frombuffer(seq, np.uint8)
        strand = int(rng.integers(0, 2))
        if strand:
            a = revcomp(a)
        g[s:s + len(a)] = a
        placements.append((int(s), len(a), strand))
    return g, placements


def simulate_reads(genome, n_reads, read_len=150, seed=2, sub_rate=0.002, regions=None):
    """Illumina-like reads: uniform start, random strand, substitutions only.  Returns (data, off):
    uint8 ASCII bases concatenated and uint64 offsets (n+1).  regions = list of (start, len) limits
    sampling to those intervals (toy configs)."""
    rng = np.random.default_rng(seed)
    G = len(genome)
    if regions is None:
        starts = rng.integers(0, G - read_len + 1, size=n_reads)
    else:
        reg = np.array(regions)
        w = np.maximum(reg[:, 1] - read_len + 1, 1).astype(float)
        which = rng.choice(len(reg), size=n_reads, p=w / w.sum())
        starts = reg[which, 0] + (rng.random(n_reads) * w[which]).astype(np.int64)
    idx = starts[:, None] + np.arange(read_len)[None, :]
    reads = genome[idx]
    strand = rng.integers(0, 2, size=n_reads).astype(bool)
    reads[strand] = _COMP[reads[strand][:, ::-1]]
    nerr = rng.binomial(n_reads * read_len, sub_rate)
    if nerr:
        ei = rng.integers(0, n_reads, size=nerr)
        ej = rng.integers(0, read_len, size=nerr)
        reads[ei, ej] = BASES[(_CODE[reads[ei, ej]] + rng.integers(1, 4, size=nerr)) % 4]
    data = np.ascontiguousarray(reads).reshape(-1)
    off = (np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(read_len))
    return data, off


def simulate_long_reads(genome, n_reads, mean_len=10000, sigma=0.3, seed=3, err=0.05, mix=(0.4, 0.3, 0.3),
                        regions=None):
    """Nanopore-like reads: lognormal length, err split sub/ins/del.  Returns (data, off)."""
    rng = np.random.default_rng(seed)
    G = len(genome)
    lens = np.clip(rng.lognormal(np.log(mean_len) - sigma * sigma / 2, sigma, size=n_reads), 200, G // 4).astype(np.int64)
    chunks, off = [], [0]
    for i in range(n_reads):
        L = int(lens[i])
        if regions is None:
            s = int(rng.integers(0, G - L))
        else:
            r = regions[int(rng.integers(0, len(regions)))]
            s = int(np.clip(r[0] + rng.integers(-L // 2, max(1, r[1] - L // 2)), 0, G - L))
        a = genome[s:s + L].copy()
        if rng.random() < 0.5:
            a = revcomp(a)
        u = rng.random(L)
        sub = u < err * mix[0]
        ins = (u >= err * mix[0]) & (u < err * (mix[0] + mix[1]))
        dele = (u >= err * (mix[0] + mix[1])) & (u < err)
        a[sub] = BASES[(_CODE[a[sub]] + rng.integers(1, 4, size=int(sub.sum()))) % 4]
        keep = ~dele
        reps = np.ones(L, np.int64)
        reps[ins] = 2
        a2 = np.repeat(a[keep], reps[keep])
        # inserted copies become random bases
        dup = np.zeros(len(a2), bool)
        pos = np.cumsum(reps[keep]) - 1
        dup[pos[reps[keep] == 2]] = True
        a2[dup] = BASES[rng.integers(0, 4, size=int(dup.sum()))]
        chunks.append(a2)
        off.append(off[-1] + len(a2))
    return np.concatenate(chunks), np.array(off, np.uint64)


def write_fastq(path, data, off, gz=False):
    import gzip
    op = gzip.open if gz else open
    with op(path, "wb") as f:
        for i in range(len(off) - 1):
            s = data[int(off[i]):int(off[i + 1])].tobytes()
            f.write(b"@r%d\n" % i + s + b"\n+\n" + b"I" * len(s) + b"\n")


def write_fastq_fast(path, data, off, gz=False, seed=7):
    """vectorised FASTQ writer for equal-length reads (benchmarks: a million records in a fraction of a second): fixed-width
    headers, qualities drawn from the four binned Illumina symbols so that gzip sees realistic entropy"""
    import zlib
    n = len(off) - 1
    L = int(off[1] - off[0]) if n else 0
    if n == 0 or not (np.diff(off) == L).all():
        return write_fastq(path, data, off, gz)
    rng = np.random.default_rng(seed)
    head = 11  # "@r" + 8 digits + newline
    rec = head + L + 3 + L + 1
    out = np.empty((n, rec), np.uint8)
    out[:, 0], out[:, 1] = ord("@"), ord("r")
    ids = np.arange(n, dtype=np.int64)
    for d in range(8):
        out[:, 2 + d] = ord("0") + (ids // 10 ** (7 - d)) % 10
    out[:, 10] = 10
    out[:, head:head + L] = np.asarray(data, np.uint8).reshape(n, L)
    out[:, head + L], out[:, head + L + 1], out[:, head + L + 2] = 10, ord("+"), 10
    out[:, head + L + 3:head + 2 * L + 3] = np.frombuffer(b"F:,#", np.uint8)[rng.choice(4, size=(n, L), p=(0.85, 0.08, 0.05, 0.02))]
    out[:, rec - 1] = 10
    raw = out.tobytes()
    with open(path, "wb") as f:
        if gz:
            co = zlib.compressobj(1, zlib.DEFLATED, 31)  # one gzip member, like `gzip -1`
            f.write(co.compress(raw))
            f.write(co.flush())
        else:
            f.write(raw)


# --------------------------------------------------------------------------------------------
def pack_reads(data, off, stride_words=0):
    """2-bit pack ASCII reads (A0 C1 G2 T3, base i of a read in bits [30-2*(i%16), 31-2*(i%16)] of
    word i//16, i.e. earlier bases more significant).  Returns (words uint32, word_off uint64[n+1],
    lens uint32[n]).  A read with any non-ACGT base gets len 0 (pandora drops the whole read).
    stride_words > 0 forces a fixed stride per read (all reads must fit)."""
    n = len(off) - 1
    lens = (off[1:] - off[:-1]).astype(np.int64)
    code = _CODE[data]
    bad = code > 3
    nwords = (lens + 15) // 16
    if stride_words:
        assert nwords.max(initial=0) <= stride_words
        woff = np.arange(n + 1, dtype=np.uint64) * np.uint64(stride_words)
    else:
        woff = np.zeros(n + 1, np.uint64)
        np.cumsum(nwords, out=woff[1:])
    total_words = int(woff[-1])
    words = np.zeros(total_words, np.uint32)
    if len(data):
        read_of = np.repeat(np.arange(n), lens)
        pos = np.arange(len(data)) - np.repeat(off[:-1].astype(np.int64), lens)
        widx = woff[read_of].astype(np.int64) + pos // 16
        shift = (30 - 2 * (pos % 16)).astype(np.uint32)
        np.bitwise_or.at(words, widx, (code & 3).astype(np.uint32) << shift)
        out_lens = lens.astype(np.uint32)
        if bad.any():
            out_lens[np.unique(read_of[bad])] = 0
    else:
        out_lens = lens.astype(np.uint32)
    return words, woff, out_lens


def toy_dataset(prg_path, refs_path, depth=50, decoys=10, seed=1, read_len=150, sub_rate=0.002):
    """Config 1 (SURVEY §8d): reads tiled from a random-allele path of each toy locus plus random
    decoy reads.  Returns (data, off)."""
    rng = np.random.default_rng(seed)
    name, seqs = None, {}
    for line in open(refs_path):
        line = line.strip()
        if line.startswith(">"):
            name = line[1:].split()[0]
            seqs[name] = ""
        elif name:
            seqs[name] += line
    flank = 300
    pieces, regions, cur = [], [], 0
    for nm, s in seqs.items():
        f = random_dna(rng, flank)
        body = np.frombuffer(s.encode(), np.uint8)
        pieces += [f, body]
        regions.append((cur, flank + len(body) + flank))
        cur += flank + len(body)
    pieces.append(random_dna(rng, flank))
    genome = np.concatenate(pieces)
    total = sum(len(s) for s in seqs.values())
    n = int(depth * total / read_len)
    d1, o1 = simulate_reads(genome, n, read_len, seed + 1, sub_rate, regions=[(0, len(genome))])
    dec = random_dna(rng, read_len * n * decoys // 1)
    d = np.concatenate([d1, dec])
    o = np.arange(n + n * decoys + 1, dtype=np.uint64) * np.uint64(read_len)
    return d, o
