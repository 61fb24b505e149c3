"""The resolve kernel of the k-mer screen takes the queue in warp tiles of 128 entries, collects the probe survivors of a
tile in a ring in the warp's shared memory, tests them 32 at a time and tests what is left after the warp's last tile.
Every prefix of a list of short reads cut from the panel (then mixed with random 150 bp decoys, whose queue entries are
all Bloom false positives) is mapped as one batch: queues from a few entries to several tiles, tiles with fewer than 32
survivors (a partial test only) and with more (full tests, then a partial one).  A batch this small has more warps than
tiles, so every warp takes at most one tile; survivors carried over into a warp's next tile need a queue longer than
128 entries per warp of the grid and are covered by the 1 M-read oracle comparisons."""
import numpy as np
import pytest

import oracle_py as O
from drprg_b200 import lib
from helpers import TOY_PRG, TOY_REFS, reads_from_strings

pytestmark = pytest.mark.gpu
W, K = 11, 15


def test_resolve_every_small_batch_size():
    rng = np.random.default_rng(5)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    reads = []
    for i in range(160):
        if i >= 40 and i % 4 == 3:
            reads.append("".join("ACGT"[j] for j in rng.integers(0, 4, size=150)))
            continue
        g = refs[int(rng.integers(0, len(refs)))]
        L = int(rng.integers(W + K - 1, W + K + 16))  # 1..17 windows: the queue grows by a few entries per read
        st = int(rng.integers(0, len(g) - L))
        r = g[st:st + L]
        reads.append(r.translate(str.maketrans("ACGT", "TGCA"))[::-1] if rng.integers(0, 2) else r)
    gx, ox = lib.Index(TOY_PRG, W, K, device=0), O.Index(TOY_PRG, W, K)
    oo = O.make_opts(illumina=True, genome_size=2000, min_cluster_size=2)
    go = lib.make_opts(illumina=True, genome_size=2000, min_cluster_size=2)
    for n in range(1, len(reads) + 1):
        data, off = reads_from_strings(reads[:n])
        oh = O.MapRun(ox, data, off, oo).hits()
        for stride in (0, 10):
            words, woff, lens = lib.pack_reads(data, off, stride)
            gx.sample_begin(go, len(reads[0]))
            nh, _ = gx.map_batch(gx.upload(words, woff, lens, total_bases=int(off[-1]), stride_words=stride))
            gh = gx.last_hits(nh)
            for key in ("read", "prg", "fwd", "start", "knode", "kept"):
                assert len(gh[key]) == len(oh[key]) and (gh[key] == oh[key]).all(), (n, stride, key)
