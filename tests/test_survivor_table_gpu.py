"""GPU: the survivor table (table 2) built hot k-mers first, with displaced-home marks.

Every lookup in table 2 (pass 2, the exports, vdjgraph_query) ends at a home slot that holds another
k-mer unless that home carries CNT2_DISP, the mark t2_insert leaves when it moves a k-mer past its
home.  At VDJGRAPH_LOAD2=0.9 most homes are taken and probe chains are long, so a lost or stale mark
would drop nodes or edges.  VDJGRAPH_HOT2 only orders the inserts; no result may depend on it."""
import numpy as np
import pytest

from oracle import loader
from tests.query_model import NodeIndex, answers, decode_kmers
from tests.util import assert_graph_equal
from vdjer_b200 import GraphBuilder, forward_reads, shard, synth

pytestmark = pytest.mark.gpu

DENSE = "0.9"
NONE_HOT = "1000000"    # above every count (counts stop at 32765)
CASES = [
    # L, k, mf, mq, pairs, clones, seed
    (50, 35, 3, 90, 40000, 800, 901),
    (50, 25, 1, 20, 20000, 150, 902),      # heavy branching: many successor and predecessor lookups
    (100, 50, 2, 120, 10000, 300, 903),    # wide tuples
]
IDS = ["L50k35", "L50k25", "L100k50"]


def _inputs(case):
    L, k, mf, mq, pairs, clones, seed = case
    return synth.generate(n_pairs=pairs, read_length=L, seed=seed, n_clones=clones, threads=4)


def _sharded(primary, secondary, L, k, mf, mq, G):
    rb = 2 * L + 1
    total = (primary.size // rb) + (secondary.size // rb)
    parts = [shard.split_records(primary, secondary, L, lo, hi) for lo, hi in shard.shard_ranges(total, G)]
    builders = [GraphBuilder(L, k, mf, mq, device=0) for _ in range(G)]
    try:
        return shard.build_local(builders, parts)
    finally:
        for b in builders:
            b.close()


@pytest.mark.parametrize("route", ["one_round", "rounds4", "shard2", "shard4"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_dense_table_matches_oracle(built, case, route, monkeypatch):
    """One round (pass 2 and the export on the dense table), four rounds (the merged finish copies every
    survivor record, stale marks included, into a new table) and 2 and 4 contexts sharded on one GPU."""
    monkeypatch.setenv("VDJGRAPH_LOAD2", DENSE)
    L, k, mf, mq = case[:4]
    primary, secondary = _inputs(case)
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    if route.startswith("shard"):
        got = _sharded(primary, secondary, L, k, mf, mq, int(route[5:]))
    else:
        with GraphBuilder(L, k, mf, mq, rounds=4 if route == "rounds4" else 1) as gb:
            got = gb.build(primary, secondary)
        assert got.stats["n_hits"] == want["n_hits"]
    assert_graph_equal(got, want, f"{route} load {DENSE}")


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_hot_threshold_does_not_change_the_graph(built, case, monkeypatch):
    """All survivors hot, none hot and the default order: the same graph, counters and node k-mers."""
    L, k, mf, mq = case[:4]
    primary, secondary = _inputs(case)
    graphs = []
    for hot in ["1", NONE_HOT, None]:
        if hot is None:
            monkeypatch.delenv("VDJGRAPH_HOT2", raising=False)
        else:
            monkeypatch.setenv("VDJGRAPH_HOT2", hot)
        with GraphBuilder(L, k, mf, mq, export_keys=True) as gb:
            graphs.append(gb.build(primary, secondary))
    ref = graphs[0]
    for g in graphs[1:]:
        for name in ["first_pos", "frequency", "out_deg", "in_deg", "out_succ", "in_pred", "kmer_lo", "kmer_hi"]:
            assert np.array_equal(getattr(g, name), getattr(ref, name)), name
        for name in ["n_hits", "n_hits_ungated", "n_pre", "n_pre_total"]:
            assert g.stats[name] == ref.stats[name], name


@pytest.mark.parametrize("rounds", [1, 4])
def test_queries_on_a_dense_table_answer_like_the_graph(built, rounds, monkeypatch):
    """Node k-mers, reads, their reverse complements and random sequences, looked up in a table at load
    0.9 (one round) or in the merged table rebuilt from its records (four rounds)."""
    monkeypatch.setenv("VDJGRAPH_LOAD2", DENSE)
    L, k, mf, mq = 50, 25, 2, 60
    primary, secondary = synth.generate(n_pairs=5000, read_length=L, seed=911, n_clones=120, threads=4, p_n=0.01)
    reads = []
    for buf in (primary, secondary):
        fwd = forward_reads(buf, L)[:-1].reshape(-1, 2 * L + 1)
        reads += [r[1:1 + L].tobytes() for r in fwd]
    rng = np.random.default_rng(911)
    comp = bytes.maketrans(b"ACGTN", b"TGCAN")
    with GraphBuilder(L, k, mf, mq, export_keys=True, rounds=rounds) as gb:
        g = gb.build(primary, secondary)
        assert g.n_nodes > 0
        nodes = decode_kmers(g.kmer_lo, g.kmer_hi, k)
        seqs = nodes + reads + [r.translate(comp)[::-1] for r in reads[::3]]
        seqs += [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes() for n in rng.integers(0, 300, 500)]
        got, stats = gb.query(seqs)
    model = answers(seqs, k, NodeIndex(g.kmer_lo, g.kmer_hi))
    assert np.array_equal(np.concatenate(got[:len(nodes)]), np.arange(g.n_nodes, dtype=np.uint32))
    for q, (a, b) in enumerate(zip(got, model)):
        assert np.array_equal(a, b), f"query {q}: {a} != {b}"


def test_hot_kmers_first_take_most_windows_off_the_slow_path(built, monkeypatch):
    """A skewed sample (300 k pairs from 400 clones): inserting the hot survivors first at least halves
    the pass-2 windows that leave their home slot, against an insert order blind to counts."""
    L, k, mf, mq = 50, 35, 3, 90
    primary, secondary = synth.generate(n_pairs=300_000, read_length=L, seed=913, n_clones=400, threads=8)
    slow = {}
    with GraphBuilder(L, k, mf, mq) as gb:
        gb.stage(primary, secondary)
        for label, hot in [("none_hot", NONE_HOT), ("default", None)]:
            if hot is None:
                monkeypatch.delenv("VDJGRAPH_HOT2", raising=False)
            else:
                monkeypatch.setenv("VDJGRAPH_HOT2", hot)
            gb.run()
            slow[label] = gb.fetch_stats()["n_slow2"]
    assert slow["none_hot"] > 0
    assert slow["default"] * 2 < slow["none_hot"], slow
