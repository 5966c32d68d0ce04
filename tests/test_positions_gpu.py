"""GPU: node positions past 2^32, against the oracle, along every build route.

A position (stamp) is r*w + o for window o of record r, w = L - k + 1, kept in 40 bits: in the run records, the
narrow queue tuples, the occurrence log, the stamp -> record division, the coarse out_first bound, the sorts and
the distributed finish's node rows.  To reach 2^32 cheaply the input is A ++ F ++ B: A and B are seeded
synthetic records, F is enough all-N records to push B's stamps past 2^32.  An all-N record has no gated and no
N-free window, so it changes nothing in the graph but the numbering of every record after it: the expected graph
is the oracle's graph of A ++ B with first_pos moved by |F|*w wherever it is at or past |A|*w.

B holds more reads of A's clone library, reads of clones A does not have (nodes first seen past 2^32) and copies
of some of A's records (first occurrence, the distinct-read decision and edge order compare stamps on both
sides of 2^32).  Every build sees the same input; the fixtures assert that it really crosses the boundary."""
import numpy as np
import pytest

from oracle import loader
from tests import hashmap_model
from tests.query_model import NodeIndex, answers
from tests.util import assert_graph_equal, assert_pre_table_equal, kmer_codes_at, pack_codes
from vdjer_b200 import GraphBuilder, MultiBuilder, PinnedRecords, shard, synth

pytestmark = pytest.mark.gpu

L, K, MF, MQ = 255, 35, 2, 90
W = L - K + 1
RB = 2 * L + 1
TWO32 = 1 << 32
N_BEFORE = 2 * (TWO32 // (2 * W))     # |A| + |F|, even: window 2^32 falls inside one of B's first two records
NIL = 0xFFFFFFFF


def _records(buf):
    """NUL-terminated record buffer -> [n, RB] view of its records."""
    return buf[: buf.size // RB * RB].reshape(-1, RB)


def _buffer(head, n_fill, tail):
    """head ++ n_fill all-N records ++ tail as one NUL-terminated buffer, written in place."""
    out = np.empty((len(head) + n_fill + len(tail)) * RB + 1, np.uint8)
    recs = out[:-1].reshape(-1, RB)
    recs[: len(head)] = head
    fill = recs[len(head): len(head) + n_fill]
    fill[:, 0] = ord("0")
    fill[:, 1: 1 + L] = ord("N")
    fill[:, 1 + L:] = ord("#")
    recs[len(head) + n_fill:] = tail
    out[-1] = 0
    return out


def _nul(recs):
    return np.concatenate([recs.reshape(-1), np.zeros(1, np.uint8)])


class Case:
    """A, B and the expected graph.  A's records fill the primary buffer first; B's primary records follow F
    there and B's secondary records make up the secondary buffer."""

    def __init__(self):
        ap, as_ = synth.generate(n_pairs=1500, read_length=L, seed=601, n_clones=40, threads=4)
        bp, bs = synth.generate(n_pairs=1500, read_length=L, seed=601, n_clones=40, threads=4, pair_offset=1500)
        np_, ns = synth.generate(n_pairs=200, read_length=L, seed=602, n_clones=8, threads=4)   # clones A lacks
        self.A = np.concatenate([_records(ap), _records(as_)])
        pairs = self.A.reshape(-1, 2, RB)
        copies = pairs[np.random.default_rng(603).choice(len(pairs), 400, replace=False)].reshape(-1, RB)
        self.B_p = np.concatenate([copies[:200], _records(bp), _records(np_), copies[200:]])
        self.B_s = np.concatenate([_records(bs), _records(ns)])
        self.n_fill = N_BEFORE - len(self.A)
        assert len(self.A) % 2 == 0 and self.n_fill > 0 and self.n_fill % 2 == 0
        # what the oracle sees: A ++ B
        self.primary = _nul(np.concatenate([self.A, self.B_p]))
        self.secondary = _nul(self.B_s)
        self.want = loader.build(self.primary, self.secondary, L, K, MF, MQ, kind="port")
        fp = self.want["first_pos"].copy()
        fp[fp >= np.uint64(len(self.A) * W)] += np.uint64(self.n_fill * W)
        self.shifted = dict(self.want, first_pos=fp)
        self.n_records = N_BEFORE + len(self.B_p) + len(self.B_s)
        self.n_windows = self.n_records * W
        self.codes = kmer_codes_at(self.primary, self.secondary, L, K, self.want["first_pos"])
        self.kmer_lo, self.kmer_hi = pack_codes(self.codes)

    def assert_crosses(self):
        """The input reaches what it is meant to test: nodes on both sides of 2^32, an edge across it and
        stamps that need more than 32 bits."""
        fp = self.shifted["first_pos"]
        assert fp.min() < TWO32 <= fp.max()
        succ = self.want["out_succ"]
        has = succ != NIL
        dst = np.where(has, fp[np.where(has, succ, 0)], 0)
        assert ((fp[:, None] < TWO32) & has & (dst >= TWO32)).any(), "no edge from below 2^32 to at or past it"
        assert int(self.n_windows).bit_length() >= 33

    def forward(self):
        """The forward reads of A ++ F ++ B (what vdjgraph_build_forward takes): about 5 GB."""
        return _buffer(self.A[0::2], self.n_fill // 2, self.B_p[0::2]), _nul(self.B_s[0::2])

    def text(self):
        """A ++ F ++ B in the reference's record format: about 10 GB."""
        return _buffer(self.A, self.n_fill, self.B_p), self.secondary


@pytest.fixture(scope="module")
def case(built):
    c = Case()
    c.assert_crosses()
    return c


@pytest.fixture(scope="module")
def fwd(case):
    return case.forward()


@pytest.fixture(scope="module")
def layout(case):
    slots, nb = hashmap_model.layout(case.codes)
    return np.where(slots < 0, NIL, slots).astype(np.uint32), nb


def _check(got, case, what, keys=False, stats=True):
    assert_graph_equal(got, case.shifted, what)
    if stats:
        st = got.stats
        assert st["n_records"] == case.n_records and st["n_windows"] == case.n_windows, what
        for name in ["n_gated", "n_pre_total", "n_hits"]:
            assert st[name] == case.want[name], f"{what}: {name}"
    if keys:
        assert np.array_equal(got.kmer_lo, case.kmer_lo) and np.array_equal(got.kmer_hi, case.kmer_hi), f"{what}: k-mers"


def _check_layout(got, layout, what):
    slots, nb = layout
    assert got.stats["hm_buckets"] == nb and got.hm_slots is not None, what
    assert np.array_equal(got.hm_slots, slots), f"{what}: hash-map layout"


def test_text_records_past_2_32(case):
    """vdjgraph_build from the reference's doubled record buffers (10 GB staged)."""
    primary, secondary = case.text()
    with GraphBuilder(L, K, MF, MQ, export_keys=True) as gb:
        got = gb.build(primary, secondary)
    del primary
    _check(got, case, "text", keys=True)


def test_forward_reads_past_2_32(case, fwd, layout):
    """vdjgraph_build_forward from pageable and from page-locked buffers: graph, k-mers, pre-table, hash-map
    layout and the narrow 16-byte tuple (33 stamp bits leave 19 fingerprint bits at k = 35)."""
    fp, fs = fwd
    with GraphBuilder(L, K, MF, MQ, export_keys=True, hashmap_layout=True) as gb:
        got = gb.build_forward(fp, fs)
        _check(got, case, "forward", keys=True)
        assert got.stats["tuple_bytes"] == 16
        _check_layout(got, layout, "forward")
        assert_pre_table_equal(gb.pre_table(), case.want, case.primary, case.secondary, L, K, "forward")
        with PinnedRecords(fp, fs):
            pinned = gb.build_forward(fp, fs)
        _check(pinned, case, "forward, page-locked", keys=True)
        _check_layout(pinned, layout, "forward, page-locked")


def test_query_past_2_32(case, fwd):
    """vdjgraph_query after the build: reads of A and of B, and both joined end to end, window by window."""
    index = NodeIndex(case.kmer_lo, case.kmer_hi)
    a = [r[1: 1 + L].tobytes() for r in case.A[::15]]
    b = [r[1: 1 + L].tobytes() for r in case.B_p[::15]] + [r[1: 1 + L].tobytes() for r in case.B_s[::15]]
    seqs = a + b + [x + y for x, y in zip(a, b)]
    with GraphBuilder(L, K, MF, MQ) as gb:
        gb.build_forward(*fwd)
        got, stats = gb.query(seqs)
    want = answers(seqs, K, index)
    assert stats["n_found"] > 0
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), f"query {i}"


def test_wide_tuples_past_2_32(case, fwd):
    with GraphBuilder(L, K, MF, MQ, wide_tuples=True) as gb:
        got = gb.build_forward(*fwd)
        assert got.stats["tuple_bytes"] == 24
        _check(got, case, "wide")
        assert_pre_table_equal(gb.pre_table(), case.want, case.primary, case.secondary, L, K, "wide")


def test_exact_read_comparison_past_2_32(case, fwd, monkeypatch):
    """No read fingerprint bits: every distinct-read decision compares the packed reads of records derived from
    stamps, many of them at or past 2^32."""
    monkeypatch.setenv("VDJGRAPH_FP_BITS", "0")
    with GraphBuilder(L, K, MF, MQ) as gb:
        got = gb.build_forward(*fwd)
        _check(got, case, "fp0")
        assert_pre_table_equal(gb.pre_table(), case.want, case.primary, case.secondary, L, K, "fp0")


def test_rounds_past_2_32(case, fwd):
    """Four super-partition rounds: survivor records and the merged flat table carry the stamps."""
    with GraphBuilder(L, K, MF, MQ, rounds=4, export_keys=True) as gb:
        got = gb.build_forward(*fwd)
    assert got.stats["rounds"] == 4
    _check(got, case, "rounds=4", keys=True)


@pytest.mark.parametrize("G", [2, 4])
def test_sharded_past_2_32(case, fwd, layout, G):
    """Sharded over G contexts of one device, rank boundaries inside F: the distributed finish's node rows
    (first_pos in 40 bits), its k-mer array and the hash-map layout."""
    fp, fs = fwd
    parts = [shard.split_records(fp, fs, L, lo // 2, hi // 2) for lo, hi in shard.shard_ranges(case.n_records, G)]
    assert all(len(case.A) < lo < N_BEFORE for lo, _ in shard.shard_ranges(case.n_records, G)[1:])
    builders = [GraphBuilder(L, K, MF, MQ, device=0, export_keys=True, hashmap_layout=True) for _ in range(G)]
    try:
        got = shard.build_local(builders, parts, forward=True)
        stats = [b.fetch_stats() for b in builders]
    finally:
        for b in builders:
            b.close()
    _check(got, case, f"sharded G={G}", keys=True, stats=False)
    _check_layout(got, layout, f"sharded G={G}")
    for name in ["n_pre_total", "n_hits", "n_gated"]:
        assert sum(s[name] for s in stats) == case.want[name], name


def test_multi_past_2_32(case, fwd, layout):
    with MultiBuilder(L, K, MF, MQ, devices=[0, 0], export_keys=True, hashmap_layout=True) as mb:
        got = mb.build_forward(*fwd)
        stats = [mb.rank_stats(r) for r in range(2)]
    _check(got, case, "multi", keys=True, stats=False)
    _check_layout(got, layout, "multi")
    for name in ["n_pre_total", "n_hits", "n_gated"]:
        assert sum(s[name] for s in stats) == case.want[name], name
