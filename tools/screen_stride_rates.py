"""Rates of the k-mer screen on the CPU, from the library's own screen filters (drprg_cuda_index_screen_filters) and
config-3 reads: the 15-mer screen at every position against the 14-mer screen at every other position whose two
candidate 15-mers are then tested against the 15-mer filter.  Per read it prints, for each scheme, the flagged positions,
the candidate 15-mers, the candidates that pass the 15-mer filter (the queue entries) and the indexed 15-mers (the true
positives, which both schemes must keep).  Exact quantities of the filters; no GPU is used.
   python tools/screen_stride_rates.py [--subshards N]
The sub-shards are drawn with torch's CPU generator from the workload's seeds, so they are reads of the config-3
simulator but not bit-for-bit the sub-shards the GPU generates."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCREEN_MUL = 0x9E3779B1
M32 = (1 << 32) - 1


def library_filters(ix):
    from drprg_b200 import lib
    L = lib.lib()
    n15, n14 = C.c_uint32(), C.c_uint32()
    L.drprg_cuda_index_screen_filters(ix.h, None, C.byref(n15), None, C.byref(n14))
    f15 = np.zeros(n15.value, np.uint32)
    f14 = np.zeros(n14.value, np.uint32)
    rc = L.drprg_cuda_index_screen_filters(ix.h, f15.ctypes.data_as(C.c_void_p), C.byref(n15),
                                           f14.ctypes.data_as(C.c_void_p), C.byref(n14))
    assert rc == 0
    return f15, f14


def in_filter(F, x, k):
    """screen_filter_insert's test, vectorized: x are right-aligned k-mers (uint64 array)"""
    x = x.astype(np.uint64)
    p = (x * np.uint64((SCREEN_MUL << (32 - 2 * k)) & M32)) & np.uint64(M32)
    idx = (p * np.uint64(len(F))) >> np.uint64(32)
    w = F[idx.astype(np.int64)].astype(np.uint64)
    return ((w >> (x & np.uint64(31))) & (w >> ((p >> np.uint64(11)) & np.uint64(31))) & np.uint64(1)).astype(bool)


def kmers_at(codes, k):
    """[n, L] 2-bit codes -> [n, L - k + 1] right-aligned k-mers"""
    n, L = codes.shape
    out = np.zeros((n, L - k + 1), np.uint64)
    for j in range(k):
        out = (out << np.uint64(2)) | codes[:, j:L - k + 1 + j].astype(np.uint64)
    return out


def indexed_kmers(ix, k):
    from drprg_b200 import lib
    L = lib.lib()
    hs = np.unique(ix.records()["hash"])
    fw = np.array([L.drprg_cuda_hash64_inverse(int(h), k) for h in hs], np.uint64)
    rc = np.zeros_like(fw)
    t = fw.copy()
    for _ in range(k):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - (t & np.uint64(3)))
        t >>= np.uint64(2)
    return np.unique(np.concatenate([fw, rc]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subshards", type=int, default=4)
    args = ap.parse_args()
    from drprg_b200 import lib, workload
    wl = workload.Config3(total_reads=workload.Config3.SUBSHARD * args.subshards)
    ix = lib.Index(wl.prg_path, wl.w, wl.k, device=-1)
    k = wl.k
    f15, f14 = library_filters(ix)
    kset = indexed_kmers(ix, k)
    n14 = len(np.unique(np.concatenate([kset >> np.uint64(2), kset & np.uint64((1 << 2 * (k - 1)) - 1)])))
    print(json.dumps({"indexed_15mers_both_strands": int(len(kset)), "indexed_14mers": n14,
                      "filter15_words": int(len(f15)), "filter14_words": int(len(f14)),
                      "filter15_bits_per_entry": round(32 * len(f15) / len(kset), 2),
                      "filter14_bits_per_entry": round(32 * len(f14) / n14, 2)}))
    tot = {}
    n_reads = 0
    for i in range(args.subshards):
        codes = wl.subshard_codes(i, device="cpu").numpy()
        n, L = codes.shape
        k15 = kmers_at(codes, k)          # p in [0, nk)
        k14 = kmers_at(codes, k - 1)      # q in [0, nk]
        nk = L - k + 1
        true = np.isin(k15, kset)
        pass15 = in_filter(f15, k15, k)
        # stride 1: every position against the 15-mer filter
        s1 = dict(flags=pass15.sum(), candidates=pass15.sum(), queue=pass15.sum(), true=true.sum())
        # stride 2: even q in [0, nk] against the 14-mer filter; candidates p = q - 1 (q > 0) and p = q (q < nk)
        q = np.arange(0, nk + 1, 2)
        flag = in_filter(f14, k14[:, q], k - 1)
        cand = np.zeros((n, nk), bool)
        qa = q[q > 0]
        cand[:, qa - 1] |= flag[:, q > 0]
        qb = q[q < nk]
        cand[:, qb] |= flag[:, q < nk]
        s2 = dict(flags=flag.sum(), candidates=cand.sum(), queue=(cand & pass15).sum(), true=(cand & true).sum())
        assert s2["true"] == s1["true"], "a true indexed k-mer escaped the stride-2 screen"
        for name, d in (("stride1", s1), ("stride2", s2)):
            for key, v in d.items():
                tot[(name, key)] = tot.get((name, key), 0) + int(v)
        n_reads += n
    for name, tested in (("stride1", nk), ("stride2", len(q))):
        print(json.dumps({"scheme": name, "reads": n_reads, "tested_positions_per_read": tested,
                          "flags_per_read": round(tot[(name, "flags")] / n_reads, 4),
                          "flag_rate_per_tested_position": round(tot[(name, "flags")] / n_reads / tested, 5),
                          "candidates_per_read": round(tot[(name, "candidates")] / n_reads, 4),
                          "candidates_passing_15mer_filter_per_read": round(tot[(name, "queue")] / n_reads, 4),
                          "true_indexed_15mers_per_read": round(tot[(name, "true")] / n_reads, 4)}))


if __name__ == "__main__":
    main()
