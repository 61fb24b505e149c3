"""The post-process kernels of the map step (cluster.cu): grouping by read, clustering and the k-mer coverage count, at
the sizes where their own choices matter.  The coverage count keeps one copy of 32-bit counters per CTA for a range of
56 k keys and cuts the batch's key slots into stretches of at least 32 k slots; the per-stretch partials are summed by
the merge.
- a hot key: one k-mer node counted more than 65 535 times inside one (range, stretch) job;
- range edges: the benchmark panel's 76 532 keys are two ranges, checked against the oracle at every key;
- batch sizes around one stretch, and a batch of one active read, each followed by another batch of the same sample
  (the per-read hit counters must be back at zero for it)."""
import math
import os

import numpy as np
import pytest

import oracle_py as O
from drprg_b200 import lib, workload
from helpers import TOY_PRG, TOY_REFS, reads_from_strings
from test_gpu_parity import assert_map_equal

pytestmark = pytest.mark.gpu
W, K = 11, 15
CV_RANGE = 56 * 1024   # keys per coverage range (cluster.cu)
CV_STRETCH_MIN = 32768  # key slots of the shortest stretch (cluster.cu)


@pytest.fixture(scope="module")
def toy():
    gx = lib.Index(TOY_PRG, W, K, device=0)
    go = lib.make_opts(illumina=True, genome_size=2000, min_cluster_size=2)
    refs = [l.strip() for l in open(TOY_REFS) if not l.startswith(">")]
    return gx, go, refs


def map_reads(gx, go, reads, new_sample=True, read_id_base=0):
    """maps the reads as one batch; returns (hits, kept hits, accumulator as int64)"""
    data, off = reads_from_strings(reads)
    words, woff, lens = lib.pack_reads(data, off)
    if new_sample:
        gx.sample_begin(go, len(reads[0]))
    nh, nk = gx.map_batch(gx.upload(words, woff, lens, total_bases=int(off[-1]), read_id_base=read_id_base))
    return nh, nk, gx.accum_download().astype(np.int64)


def panel_read(refs, L, pick):
    g = refs[pick % len(refs)]
    st = (pick * 7919) % (len(g) - L)
    return g[st:st + L]


def read_with(gx, go, refs, L, want):
    """a read of length L cut from the panel whose single-read map satisfies want(hits, kept, accum): (read, its map)"""
    for pick in range(400):
        r = panel_read(refs, L, pick)
        m = map_reads(gx, go, [r])
        if want(*m):
            return r, m
    raise AssertionError("no such read in the toy panel")


def slots_of(gx, m):
    """key slots one read with map m fills: its hits, two locus slots, one more per kept cluster beyond two"""
    nh, _, acc = m
    n_lk = int(acc[2 * gx.total_knodes:2 * gx.total_knodes + gx.n_loci].sum())
    return nh + 2 + max(0, n_lk - 2) if nh else 0


def scalars(acc):
    return int(acc[-4]) + (int(acc[-3]) << 24), int(acc[-2]) + (int(acc[-1]) << 24)


def test_hot_key_past_16_bits_in_one_job(toy):
    """more than 65 535 copies of one read in every stretch: its k-mer nodes' counters pass 16 bits inside one job"""
    import torch

    gx, go, refs = toy
    L = 60
    read, (nh1, nk1, acc1) = read_with(gx, go, refs, L, lambda nh, nk, acc: nk > 0)
    ox = O.Index(TOY_PRG, W, K)
    d1, o1 = reads_from_strings([read])
    mr = O.MapRun(ox, d1, o1, O.make_opts(illumina=True, genome_size=2000, min_cluster_size=2))
    f, r = mr.coverage()
    N = gx.total_knodes
    assert (acc1[0:2 * N:2] == f).all() and (acc1[1:2 * N:2] == r).all() and (acc1[2 * N:2 * N + gx.n_loci] == mr.locus_reads()).all()
    # one stretch per CTA of the count grid (one range, one CTA per SM): 70 000 copies per stretch
    n = 70_000 * torch.cuda.get_device_properties(0).multi_processor_count
    stride = 4  # 60 bp in 2-bit codes
    words, _, _ = lib.pack_reads(d1, o1, stride)
    d_words = torch.from_numpy(np.ascontiguousarray(words, np.uint32).view(np.int32)).cuda().repeat(n)
    d_lens = torch.full((n,), L, dtype=torch.int32, device="cuda")
    gx.sample_begin(go, L)
    nh, nk = gx.map_batch(gx.wrap_device(d_words.data_ptr(), d_lens.data_ptr(), n, stride, n * L, keep=(d_words, d_lens)))
    acc = gx.accum_download().astype(np.int64)
    assert nh == n * nh1 and nk == n * nk1
    assert (acc[:-4] == n * acc1[:-4]).all()
    assert scalars(acc) == (n * L, n)
    assert acc[:2 * N].max() > 65535 * torch.cuda.get_device_properties(0).multi_processor_count


def test_benchmark_panel_two_key_ranges_against_oracle():
    """the benchmark panel's keys span two ranges; every counter, the first of the second range and the very last one
    (the last locus) included, equals the oracle's"""
    wl = workload.Config2()
    gx, ox = lib.Index(wl.prg_path, wl.w, wl.k, device=0), O.Index(wl.prg_path, wl.w, wl.k)
    n_keys = 2 * ox.total_knodes + ox.n_loci
    assert CV_RANGE < n_keys <= 2 * CV_RANGE
    d, o = wl.reads(300_000, 0)
    oo = O.make_opts(threads=os.cpu_count() or 1, illumina=True, genome_size=workload.GENOME_SIZE)
    go = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE)
    mr = O.MapRun(ox, d, o, oo)
    words, _, lens = lib.pack_reads(d, o, workload.STRIDE_WORDS)
    gx.sample_begin(go, workload.READ_LEN)
    nh, nk = gx.map_batch(gx.upload(words, None, lens, total_bases=int(o[-1]), stride_words=workload.STRIDE_WORDS))
    gh = gx.last_hits(nh)
    assert int(gh["kept"].sum()) == nk
    assert_map_equal(gx, mr, gh)
    acc = gx.accum_download()
    assert acc[CV_RANGE] > 0 and acc[n_keys - 1] > 0  # both ends of the second range are counted


def test_batches_around_one_stretch_then_the_next_batch(toy):
    """batches whose key slots are just below, at and above one stretch, a few stretches, and one active read: each
    gives the sum of its reads' single-read maps, and so does another batch of the same sample mapped after it.
    The slots end with the two locus slots of every active read; in the batches of kept reads only, each of those pairs
    starts with a counted locus key, so a trailing stretch of two slots or more holds a counted key."""
    gx, go, refs = toy
    L = 60
    a, ma = read_with(gx, go, refs, L, lambda nh, nk, acc: nk > 0)
    sa = slots_of(gx, ma)
    b, mb = read_with(gx, go, refs, 30, lambda nh, nk, acc: nh > 0 and math.gcd(sa, slots_of(gx, (nh, nk, acc))) == 1)
    sb = slots_of(gx, mb)
    follow = [a, b, b, a, a]
    exp_follow = 3 * ma[2][:-4] + 2 * mb[2][:-4]

    def mixed(target):  # reads a and b, exactly `target` slots
        nb = next(j for j in range(sa) if (target - j * sb) % sa == 0)
        na = (target - nb * sb) // sa
        assert na * sa + nb * sb == target
        return na, nb

    def kept_only(after):  # reads a only, 2 .. sa + 1 slots past `after`
        na = (after + 2 + sa - 1) // sa
        assert 2 <= na * sa - after <= sa + 1
        return na, 0

    cases = [mixed(CV_STRETCH_MIN - 1), mixed(CV_STRETCH_MIN), mixed(CV_STRETCH_MIN + 1), kept_only(CV_STRETCH_MIN),
             kept_only(3 * CV_STRETCH_MIN), (1, 0)]
    for na, nb in cases:
        reads = [a] * na + [b] * nb
        np.random.default_rng(na + nb).shuffle(reads)
        nh, nk, acc = map_reads(gx, go, reads)
        assert nh == na * ma[0] + nb * mb[0] and nk == na * ma[1] + nb * mb[1], (na, nb)
        assert (acc[:-4] == na * ma[2][:-4] + nb * mb[2][:-4]).all(), (na, nb)
        nh2, _, acc2 = map_reads(gx, go, follow, new_sample=False, read_id_base=len(reads))
        assert nh2 == 3 * ma[0] + 2 * mb[0], (na, nb)
        assert (acc2[:-4] == acc[:-4] + exp_follow).all(), (na, nb)
