"""The k-mer screen tests the 14-mers at even read positions only: a flagged position q stands for the candidate k-mers at
p = q - 1 and p = q, which are then tested against the filter of the indexed 15-mers before they are queued.  Reads cut
from the panel's sequences at every offset put indexed minimizers at every read position, odd and even, at the first
position p = 0 and the last p = nk - 1, on both strands, with an even and an odd number nk of k-mer positions.  Long
reads are screened in segments of 40 w positions (an even length, so every segment starts at an even position); reads
of 1000 and 1333 bases put indexed minimizers on either side of their segment boundaries.  The device hits must equal
the oracle's and those of the sketch kernels without the screen (DRPRG_SCREEN=0, run in a subprocess because the switch
is read once per process)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("read", "prg", "fwd", "start", "knode", "kept")
W, K = 11, 15


def _revcomp(s):
    return s.translate(str.maketrans("ACGT", "TGCA"))[::-1]


def _map(prg, data, off):
    from drprg_b200 import lib
    gx = lib.Index(prg, W, K, device=0)
    go = lib.make_opts(illumina=True, genome_size=200_000, min_cluster_size=2)
    words, woff, lens = lib.pack_reads(data, off)
    gx.sample_begin(go, int(off[1] - off[0]))
    nh, _ = gx.map_batch(gx.upload(words, woff, lens, total_bases=int(off[-1])))
    return gx.last_hits(nh)


@pytest.fixture(scope="module")
def panel():
    from helpers import small_panel
    _, prg, refs = small_panel()
    seqs = [l.strip() for l in open(refs) if not l.startswith(">")]
    return prg, sorted(seqs, key=len, reverse=True)


def _short_reads(seqs):
    reads = []
    for L in (150, 151):  # nk = 136 (the last position's candidate comes from q = nk) and nk = 137
        g = seqs[0]
        for s in range(0, len(g) - L + 1):
            r = g[s:s + L]
            reads.append(_revcomp(r) if s % 2 else r)
            reads.append(r if s % 2 else _revcomp(r))
    return reads


def _long_reads(seqs):
    reads = []
    for L in (1000, 1333):  # segment boundaries at 440 and 880
        for g in seqs[:2]:
            for s in range(0, len(g) - L + 1, 3):
                r = g[s:s + L]
                reads.append(r)
                reads.append(_revcomp(r))
    return reads + [seqs[0][:30], seqs[1][5:200]]  # short reads in a segmented batch


def _check(prg, reads, tmp_path, want_starts):
    import oracle_py as O
    from helpers import reads_from_strings
    data, off = reads_from_strings(reads)
    ox = O.Index(prg, W, K)
    oh = O.MapRun(ox, data, off, O.make_opts(illumina=True, genome_size=200_000, min_cluster_size=2)).hits()
    starts = set(oh["start"].tolist())
    assert want_starts <= starts, sorted(want_starts - starts)
    gh = _map(prg, data, off)
    for key in KEYS:
        assert len(gh[key]) == len(oh[key]) and (gh[key] == oh[key]).all(), key
    # the same batch through the sketch kernels, without the screen
    np.savez(tmp_path / "reads.npz", data=data, off=off)
    env = dict(os.environ, DRPRG_SCREEN="0", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), prg, str(tmp_path / "reads.npz"), str(tmp_path / "hits.npz")],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    sh = np.load(tmp_path / "hits.npz")
    for key in KEYS:
        assert len(sh[key]) == len(gh[key]) and (sh[key] == gh[key]).all(), key
    return oh


@pytest.mark.gpu
def test_screen_every_other_position_short_reads(panel, tmp_path):
    prg, seqs = panel
    oh = _check(prg, _short_reads(seqs), tmp_path, {0, 1, 2, 3, 134, 135, 136})
    assert oh["fwd"].any() and not oh["fwd"].all()


@pytest.mark.gpu
def test_screen_every_other_position_across_segments(panel, tmp_path):
    prg, seqs = panel
    seg = 40 * W
    _check(prg, _long_reads(seqs), tmp_path, {0, 1, seg - 2, seg - 1, seg, seg + 1, 2 * seg - 1, 2 * seg, 2 * seg + 1, 985, 1318})


if __name__ == "__main__":  # DRPRG_SCREEN=0 run of _check: PRG, reads .npz, hits .npz out
    f = np.load(sys.argv[2])
    h = _map(sys.argv[1], f["data"], f["off"])
    np.savez(sys.argv[3], **{key: h[key] for key in KEYS})
