"""CPU: the host side of vdjgraph_query.  The Python binding's offsets and window counts, the test model
of the answers on hand-made examples, and the stats struct's layout in the header and in ctypes."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from tests.query_model import NodeIndex, answers, decode_kmers, window_starts
from tests.util import pack_codes
from vdjer_b200 import graph
from vdjer_b200.graph import NIL, query_batch, window_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _index(kmers):
    codes = np.array([["ACGT".index(ch) for ch in s] for s in kmers], np.uint8)
    return NodeIndex(*pack_codes(codes))


def test_offsets_and_window_counts():
    text, offsets = query_batch([b"ACGTA", "", "AC", b"NNNNNNN", "ACG"])
    assert text.tobytes() == b"ACGTAACNNNNNNNACG"
    assert offsets.dtype == np.uint64 and offsets.tolist() == [0, 5, 5, 7, 14, 17]
    assert window_counts(offsets, 3).tolist() == [3, 0, 0, 5, 1]
    assert window_counts(offsets, 1).tolist() == [5, 0, 2, 7, 3]
    assert window_counts(offsets, 8).tolist() == [0, 0, 0, 0, 0]
    assert window_starts(offsets, 3).tolist() == [0, 1, 2, 7, 8, 9, 10, 11, 14]
    empty_text, empty_offsets = query_batch([])
    assert empty_text.size == 0 and empty_offsets.tolist() == [0]
    assert window_counts(empty_offsets, 3).size == 0


def test_model_on_hand_made_queries():
    idx = _index(["ACG", "CGT", "TTT", "GGA"])
    got = answers([b"ACGTT", b"TTTT", b"AC", b"ACNGT", b"GGACG", b""], 3, idx)
    want = [[0, 1, NIL], [2, 2], [], [NIL, NIL, NIL], [3, NIL, 0], []]
    assert [a.tolist() for a in got] == want
    assert all(a.dtype == np.uint32 for a in got)


def test_model_keys_above_64_bits():
    """k > 32: the bases past the 32nd are in the high word."""
    rng = np.random.default_rng(5)
    seqs = ["".join("ACGT"[c] for c in rng.integers(0, 4, 60)) for _ in range(4)]
    nodes = [s[3:3 + 40] for s in seqs] + [seqs[0][10:50]]
    idx = _index(nodes)
    got = answers(seqs, 40, idx)
    for q, a in enumerate(got):
        assert len(a) == 21
        assert a[3] == q
        others = [w for w in range(21) if w != 3 and not (q == 0 and w == 10)]
        assert np.all(a[others] == NIL)
    assert got[0][10] == 4


def test_decode_kmers_round_trip():
    kmers = ["ACGTTGCA" * 6 + "TT", "T" * 50, "A" * 33]
    for s in kmers:
        codes = np.array([["ACGT".index(ch) for ch in s]], np.uint8)
        lo, hi = pack_codes(codes)
        assert decode_kmers(lo, hi, len(s)) == [s.encode()]


def test_query_stats_layout_matches_header():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "vdjgraph.h"
int main(void){
 printf("%zu %zu %zu %zu %zu\n", sizeof(vdjgraph_query_stats), offsetof(vdjgraph_query_stats, n_found),
   offsetof(vdjgraph_query_stats, d2h_bytes), offsetof(vdjgraph_query_stats, ms_kernels), offsetof(vdjgraph_query_stats, ms_total));
 return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    S = graph._QueryStats
    assert got == [C.sizeof(S), S.n_found.offset, S.d2h_bytes.offset, S.ms_kernels.offset, S.ms_total.offset]
