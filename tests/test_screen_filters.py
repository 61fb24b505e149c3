"""The k-mer screen's filters as the library builds them at index load: the 15-mer filter must contain every indexed k-mer
in both orientations, and the 14-mer filter the screen tests at even read positions both 14-mers of each of them —
otherwise a read's indexed k-mer could go unflagged and its hit be lost.  Host only: no GPU is needed."""
import ctypes as C

import numpy as np

from drprg_b200 import lib
from helpers import TOY_PRG, small_panel

SCREEN_MUL = 0x9E3779B1


def _filters(ix):
    L = lib.lib()
    n15, n14 = C.c_uint32(), C.c_uint32()
    assert L.drprg_cuda_index_screen_filters(ix.h, None, C.byref(n15), None, C.byref(n14)) == 0
    f15, f14 = np.zeros(n15.value, np.uint32), np.zeros(n14.value, np.uint32)
    assert L.drprg_cuda_index_screen_filters(ix.h, f15.ctypes.data_as(C.c_void_p), C.byref(n15),
                                             f14.ctypes.data_as(C.c_void_p), C.byref(n14)) == 0
    return f15, f14


def _contains(F, x, k):
    p = (x * ((SCREEN_MUL << (32 - 2 * k)) & 0xffffffff)) & 0xffffffff
    w = int(F[(p * len(F)) >> 32])
    return (w >> (x & 31)) & (w >> ((p >> 11) & 31)) & 1 == 1


def _revcomp(x, k):
    y = 0
    for _ in range(k):
        y = (y << 2) | (3 - (x & 3))
        x >>= 2
    return y


def test_screen_filters_hold_every_indexed_kmer_and_its_14mers():
    L = lib.lib()
    for prg in (TOY_PRG, small_panel()[1]):
        ix = lib.Index(prg, 11, 15, device=-1)
        f15, f14 = _filters(ix)
        assert len(f15) % 4 == 0 and len(f14) % 4 == 0 and len(f14) >= len(f15)
        hashes = np.unique(ix.records()["hash"])
        assert len(hashes)
        for h in hashes.tolist():
            y = int(L.drprg_cuda_hash64_inverse(h, 15))
            for x in (y, _revcomp(y, 15)):
                assert _contains(f15, x, 15), (prg, x)
                assert _contains(f14, x >> 2, 14) and _contains(f14, x & ((1 << 28) - 1), 14), (prg, x)


def test_no_screen_filters_for_other_k():
    ix = lib.Index(TOY_PRG, 11, 13, device=-1)
    assert [len(f) for f in _filters(ix)] == [0, 0]
