"""GPU: vdjgraph_query looks sequences up in the built graph on the device.

Expected answers come from the oracle's graph (or the golden fixtures): node k-mers are the bases at the
nodes' first positions, and tests/query_model.py answers every window from them."""
import os

import numpy as np
import pytest

from oracle import loader
from tests.cases import CASES, make_inputs
from tests.query_model import NodeIndex, answers, decode_kmers
from tests.util import GOLDEN_DIR, digest_of, kmer_codes_at, pack_codes
from vdjer_b200 import GraphBuilder, VdjGraphError, forward_reads, shard, synth
from vdjer_b200.graph import NIL, query_batch, window_counts

pytestmark = pytest.mark.gpu

ERR_PARAM, ERR_BASE, ERR_STATE = -1, -3, -7
_COMP = bytes.maketrans(b"ACGTN", b"TGCAN")


def _inputs(L, k, seed, pairs=3000, clones=100):
    return synth.generate(n_pairs=pairs, read_length=L, seed=seed, n_clones=clones, threads=4, p_n=0.01)


def _reads(primary, secondary, L):
    """The forward reads' bases (with their Ns)."""
    out = []
    for buf in (primary, secondary):
        fwd = forward_reads(buf, L)[:-1].reshape(-1, 2 * L + 1)
        out += [r[1:1 + L].tobytes() for r in fwd]
    return out


def _query_all(gb, seqs):
    text, offsets = query_batch(seqs)
    return gb.query_flat(text, offsets)


@pytest.mark.parametrize("partitions", [1, 256])
@pytest.mark.parametrize("rounds", [1, 4])
@pytest.mark.parametrize("L,k", [(50, 35), (50, 25), (100, 50), (20, 3), (30, 1), (64, 10), (64, 11)])
def test_every_node_finds_itself(built, L, k, rounds, partitions):
    """Sliced (one round) and flat merged (several rounds) tables; k below, at and above the minimizer length."""
    primary, secondary = _inputs(L, k, seed=600 + k, pairs=1500 if L > 50 else 3000)
    want = loader.build(primary, secondary, L, k, 2, 60, kind="port")
    with GraphBuilder(L, k, 2, 60, export_keys=True, rounds=rounds, partitions=partitions) as gb:
        g = gb.build(primary, secondary)
        assert g.n_nodes == want["n_nodes"] > 0
        lo, hi = pack_codes(kmer_codes_at(primary, secondary, L, k, want["first_pos"]))
        assert np.array_equal(g.kmer_lo, lo) and np.array_equal(g.kmer_hi, hi)
        got, stats = _query_all(gb, decode_kmers(g.kmer_lo, g.kmer_hi, k))
    assert np.array_equal(got, np.arange(g.n_nodes, dtype=np.uint32))
    assert stats["n_queries"] == stats["n_windows"] == stats["n_found"] == g.n_nodes


@pytest.mark.parametrize("rounds", [1, 4])
@pytest.mark.parametrize("L,k", [(50, 35), (50, 25), (100, 50)])
def test_reads_and_mixed_queries_match_the_model(built, L, k, rounds):
    primary, secondary = _inputs(L, k, seed=700 + k)
    want = loader.build(primary, secondary, L, k, 2, 60, kind="port")
    index = NodeIndex.from_graph(want, primary, secondary, L, k)
    reads = _reads(primary, secondary, L)
    assert any(b"N" in r for r in reads)
    rng = np.random.default_rng(k)
    seqs = list(reads)
    seqs += [r.translate(_COMP)[::-1] for r in reads[::3]]                      # reverse complements
    seqs += [b"".join(reads[i:i + 200 // L]) for i in range(0, len(reads), 7)]  # windows across read borders
    seqs += [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes() for n in rng.integers(0, 300, 500)]  # random
    with GraphBuilder(L, k, 2, 60, rounds=rounds) as gb:
        gb.build(primary, secondary)
        got, stats = gb.query(seqs)
    model = answers(seqs, k, index)
    assert len(got) == len(seqs)
    for q, (a, b) in enumerate(zip(got, model)):
        assert np.array_equal(a, b), f"query {q}: {a} != {b}"
    flat = np.concatenate(model)
    assert stats["n_windows"] == flat.size and stats["n_found"] == int((flat != NIL).sum())
    assert stats["n_queries"] == len(seqs) and stats["h2d_bytes"] >= sum(map(len, seqs))
    assert stats["d2h_bytes"] >= 4 * flat.size and stats["ms_total"] >= stats["ms_kernels"] > 0
    assert 0 < stats["n_found"] < flat.size


@pytest.mark.parametrize("name", sorted(CASES))
def test_golden_graph_nodes_are_found_at_their_index(built, name):
    case = CASES[name]
    gold = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    primary, secondary = make_inputs(case)
    L, k = case["L"], case["k"]
    codes = kmer_codes_at(primary, secondary, L, k, gold["first_pos"])
    seqs = [row.tobytes() for row in np.frombuffer(b"ACGT", np.uint8)[codes]]
    with GraphBuilder(L, k, case["mf"], case["mq"]) as gb:
        gb.build(primary, secondary)
        got, stats = _query_all(gb, seqs)
    assert np.array_equal(got, np.arange(len(seqs), dtype=np.uint32))
    assert stats["n_found"] == len(seqs)


def test_chunk_boundaries_do_not_change_the_answers(built, monkeypatch):
    """1 KB chunks: thousands of chunks, queries never split, one query longer than a chunk in a chunk of its own."""
    L, k = 50, 35
    primary, secondary = _inputs(L, k, seed=801)
    reads = _reads(primary, secondary, L)
    rng = np.random.default_rng(3)
    seqs = reads[:3000] + [b"".join(reads[3000:3100])] + [b""] * 50 + [b"ACGT"] * 50 + reads[3100:4000]
    order = rng.permutation(len(seqs))
    seqs = [seqs[i] for i in order]
    want = loader.build(primary, secondary, L, k, 3, 90, kind="port")
    model = answers(seqs, k, NodeIndex.from_graph(want, primary, secondary, L, k))
    with GraphBuilder(L, k, 3, 90) as gb:
        gb.build(primary, secondary)
        big, _ = gb.query(seqs)
        monkeypatch.setenv("VDJGRAPH_QUERY_CHUNK_KB", "1")
        small, stats = gb.query(seqs)
    assert stats["h2d_bytes"] > sum(map(len, seqs))
    for a, b, m in zip(big, small, model):
        assert np.array_equal(a, m) and np.array_equal(b, m)


def test_query_state(built):
    L = 50
    primary, secondary = _inputs(L, 35, seed=802)
    with GraphBuilder(L, 35, 3, 90) as gb:
        with pytest.raises(VdjGraphError) as e:
            gb.query([b"A" * 40])
        assert e.value.code == ERR_STATE                       # before any run
        gb.stage(primary, secondary)
        with pytest.raises(VdjGraphError) as e:
            gb.query([b"A" * 40])
        assert e.value.code == ERR_STATE                       # staged, not run
        gb.run()
        before = gb.fetch()
        reads = _reads(primary, secondary, L)[:2000]
        first, _ = gb.query(reads)
        after = gb.fetch()
        assert digest_of(lambda n: getattr(before, n)) == digest_of(lambda n: getattr(after, n))
        gb.build(primary, secondary)
        again, _ = gb.query(reads)
        assert all(np.array_equal(a, b) for a, b in zip(first, again))
        gb.set_params(k=25, mf=2, mq=60)
        with pytest.raises(VdjGraphError) as e:
            gb.query(reads)
        assert e.value.code == ERR_STATE                       # parameters changed since the run
        gb.build(primary, secondary)
        got, _ = gb.query(reads)
    want = loader.build(primary, secondary, L, 25, 2, 60, kind="port")
    model = answers(reads, 25, NodeIndex.from_graph(want, primary, secondary, L, 25))
    assert all(len(a) == L - 25 + 1 and np.array_equal(a, m) for a, m in zip(got, model))


def test_query_input_errors_leave_the_output_untouched(built):
    L, k = 50, 35
    primary, secondary = _inputs(L, k, seed=803)
    reads = _reads(primary, secondary, L)[:100]
    with GraphBuilder(L, k, 3, 90) as gb:
        gb.build(primary, secondary)
        for bad in (b"R", b"a", b"c", b"\0"):
            seqs = reads[:50] + [reads[50][:20] + bad + reads[50][21:]] + reads[51:]
            text, offsets = query_batch(seqs)
            out = np.full(int(window_counts(offsets, k).sum()), 0xA5A5A5A5, np.uint32)
            with pytest.raises(VdjGraphError) as e:
                gb.query_flat(text, offsets, out=out)
            assert e.value.code == ERR_BASE and "query 50" in str(e.value)
            assert np.all(out == 0xA5A5A5A5)
        text, offsets = query_batch(reads)
        n = int(window_counts(offsets, k).sum())
        out = np.full(n + 1, 0xA5A5A5A5, np.uint32)
        for wrong in (n - 1, n + 1):
            with pytest.raises(VdjGraphError) as e:
                gb.query_flat(text, offsets, out=out, n_windows=wrong)
            assert e.value.code == ERR_PARAM
        dec = offsets.copy()
        dec[10], dec[11] = dec[11], dec[10]
        with pytest.raises(VdjGraphError) as e:
            gb.query_flat(text, dec, out=out, n_windows=n)
        assert e.value.code == ERR_PARAM
        assert np.all(out == 0xA5A5A5A5)
        got, stats = gb.query([])
        assert got == [] and stats["n_queries"] == stats["n_windows"] == 0
        got, stats = gb.query([b"", b"ACGT", b"N" * 40])           # no windows, or only windows with an N
        assert [a.tolist() for a in got] == [[], [], [NIL] * 6] and stats["n_found"] == 0


def test_graph_without_nodes_answers_nil(built):
    L, k = 50, 35
    primary, secondary = _inputs(L, k, seed=804, pairs=300)
    reads = _reads(primary, secondary, L)[:200]
    with GraphBuilder(L, k, 32766, 90) as gb:                      # no k-mer is frequent enough
        assert gb.build(primary, secondary).n_nodes == 0
        got, stats = gb.query(reads)
        assert all(np.all(a == NIL) for a in got) and stats["n_found"] == 0
        assert gb.build(b"", b"").n_nodes == 0                      # no records at all
        got, stats = gb.query(reads)
        assert all(len(a) == L - k + 1 and np.all(a == NIL) for a in got) and stats["n_found"] == 0
        with pytest.raises(VdjGraphError) as e:
            gb.query([b"ACGTR" * 10])
        assert e.value.code == ERR_BASE


def test_sharded_build_over_two_ranks_is_not_queryable(built):
    """Every rank's table holds only the k-mers it owns: a query there would miss the others' nodes."""
    L, k = 50, 35
    primary, secondary = _inputs(L, k, seed=805)
    rb = 2 * L + 1
    total = primary.size // rb + secondary.size // rb
    parts = [shard.split_records(primary, secondary, L, lo, hi) for lo, hi in shard.shard_ranges(total, 2)]
    builders = [GraphBuilder(L, k, 3, 90, device=0) for _ in range(2)]
    try:
        g = shard.build_local(builders, parts)
        assert g.n_nodes > 0
        for b in builders:
            with pytest.raises(VdjGraphError) as e:
                b.query([b"A" * 40])
            assert e.value.code == ERR_STATE
    finally:
        for b in builders:
            b.close()
