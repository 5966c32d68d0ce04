"""GPU: the call order of a context (include/vdjgraph.h, "Call order"), through the Python binding on one GPU.

A call made in a state that does not accept it fails with VDJGRAPH_ERR_STATE and changes nothing.  A call that
fails otherwise leaves the records staged (a failed stage: nothing staged), so the next build starts from them.
The sharded phases are driven by hand here; a one-rank build is shard_stage(p, s, 1, 0, 0, total)."""
import numpy as np
import pytest

from vdjer_b200 import GraphBuilder, VdjGraphError, shard, synth
from vdjer_b200.graph import SHARD_HIST, SHARD_HLL

pytestmark = pytest.mark.gpu

ERR_PARAM, ERR_STRAND, ERR_STATE = -1, -2, -7
L, K, MF, MQ = 50, 35, 3, 90
FIELDS = ["first_pos", "frequency", "out_deg", "in_deg", "out_succ", "in_pred"]


def _inputs(seed):
    return synth.generate(n_pairs=3000, read_length=L, seed=seed, n_clones=100, threads=4)


def _refused(fn, *args) -> str:
    with pytest.raises(VdjGraphError) as e:
        fn(*args)
    assert e.value.code == ERR_STATE, str(e.value)
    return str(e.value)


def _query(gb):
    return gb.query([b"ACGT" * 12])


def _assert_same(got, want):
    assert got.n_nodes == want.n_nodes > 0
    for name in FIELDS:
        assert np.array_equal(getattr(got, name), getattr(want, name)), name


def _stage(builders, parts):
    """shard_stage of every rank; returns the record counts"""
    counts = [b._n_records(p, s) for b, (p, s) in zip(builders, parts)]
    base = np.concatenate([[0], np.cumsum(counts)])
    for r, (b, (p, s)) in enumerate(zip(builders, parts)):
        b.shard_stage(p, s, len(builders), r, int(base[r]), sum(counts))
    return counts


def _plan(builders, counts):
    pieces = [b.shard_count() for b in builders]
    hist_all, hll, cnt = shard.plan_inputs([x[0] for x in pieces], [x[1] for x in pieces], counts)
    for b in builders:
        b.shard_plan(hist_all, hll, cnt)


def _set_peers(builders):
    table = [b.shard_buffers()[0] for b in builders]
    for b in builders:
        b.shard_set_peers(table)


def _build(builders):
    """from PLANNED: the peers, every round's scatter and passes, the finish; rank 0's graph"""
    _set_peers(builders)
    for _ in range(builders[0].shard_rounds()):
        for b in builders:
            b.shard_scatter()
        surv = [b.shard_passes() for b in builders]
    for b in builders:
        b.shard_gather_plan(surv)
    _set_peers(builders)
    for step in range(3):
        for b in builders:
            b.shard_finish_step(step, False)
    for b in builders:
        b.shard_finish()
    return builders[0].fetch()


def test_a_fresh_context_refuses_every_build_call(built):
    hist, hll = np.zeros((1, SHARD_HIST), np.uint64), np.zeros(SHARD_HLL, np.uint8)
    with GraphBuilder(L, K, MF, MQ) as gb:
        for call in (gb.run, gb.fetch, gb.fetch_stats, gb.pre_table, lambda: _query(gb), gb.shard_count,
                     lambda: gb.shard_plan(hist, hll, np.zeros(1, np.uint64)), gb.shard_rounds, gb.shard_scatter,
                     gb.shard_passes, lambda: gb.shard_gather_plan([0]), lambda: gb.shard_finish_step(0, False),
                     gb.shard_finish):
            assert "in state EMPTY" in _refused(call)


def test_staged_records_are_run_before_the_graph_is_read(built):
    primary, secondary = _inputs(901)
    with GraphBuilder(L, K, MF, MQ) as gb:
        gb.stage(primary, secondary)
        for call in (gb.fetch, gb.fetch_stats, lambda: _query(gb), gb.pre_table):
            assert "in state STAGED" in _refused(call)
        gb.run()
        assert gb.fetch().n_nodes > 0
        assert gb.fetch_stats()["n_nodes"] > 0
        _query(gb)
        assert gb.pre_table().frequency.size > 0


def test_shard_phases_out_of_order_are_refused(built):
    primary, secondary = _inputs(902)
    with GraphBuilder(L, K, MF, MQ, rounds=2) as gb:
        counts = _stage([gb], [(primary, secondary)])
        _plan([gb], counts)
        assert "in state PLANNED" in _refused(gb.shard_scatter)          # before set_peers
        _set_peers([gb])
        assert "in state PEERS_SET" in _refused(gb.shard_passes)         # before scatter
        assert gb.shard_rounds() == 2
        gb.shard_scatter()
        surv = gb.shard_passes()
        _refused(gb.shard_gather_plan, [surv])                           # before the last round
        gb.shard_scatter()                                               # ... which goes on
        surv = gb.shard_passes()
        assert "in state PASSES_DONE" in _refused(gb.shard_scatter)     # no round left
        gb.shard_gather_plan([surv])
        _set_peers([gb])
        assert "in state FINISH_PLANNED" in _refused(gb.shard_finish_step, 1, False)   # step 1 before step 0
        gb.shard_finish_step(0, False)
        gb.shard_finish_step(1, False)
        assert "in state FINISH_STEP1" in _refused(gb.shard_finish)    # before step 2
        gb.shard_finish_step(2, False)
        gb.shard_finish()
        got = gb.fetch()
        _assert_same(got, gb.build(primary, secondary))


def test_set_params_drops_the_build(built):
    primary, secondary = _inputs(903)
    with GraphBuilder(L, K, MF, MQ) as gb:
        gb.build(primary, secondary)
        gb.set_params(mf=2, mq=60)                                       # same geometry: the records stay staged
        for call in (gb.fetch, gb.fetch_stats, lambda: _query(gb)):
            assert "in state STAGED" in _refused(call)
        gb.run()
        got = gb.fetch()
        _assert_same(got, gb.build(primary, secondary))
        gb.set_params(k=25)                                              # new k: the records are gone
        assert "in state EMPTY" in _refused(gb.run)
        gb.stage(primary, secondary)
        gb.run()
        assert gb.fetch().n_nodes > 0


def test_set_params_in_the_middle_of_a_sharded_build(built):
    primary, secondary = _inputs(904)
    with GraphBuilder(L, K, MF, MQ) as gb:
        counts = _stage([gb], [(primary, secondary)])
        _plan([gb], counts)
        gb.set_params(mf=2, mq=60)
        assert "in state STAGED" in _refused(gb.shard_set_peers, [gb.shard_buffers()[0]])
        assert "in state STAGED" in _refused(gb.shard_scatter)
        _plan([gb], counts)                                              # shard_count starts the build again
        got = _build([gb])
        _assert_same(got, gb.build(primary, secondary))


def test_a_failed_plan_keeps_the_records_staged(built):
    primary, secondary = _inputs(905)
    with GraphBuilder(L, K, MF, MQ) as gb:
        counts = _stage([gb], [(primary, secondary)])
        _plan([gb], counts)
        _build([gb])
        assert gb.fetch_stats()["n_nodes"] > 0
        hist, hll = gb.shard_count()
        with pytest.raises(VdjGraphError) as e:
            gb.shard_plan(hist[None], hll, np.array([counts[0] + 2], np.uint64))   # counts that do not add up
        assert e.value.code == ERR_PARAM
        assert "in state STAGED" in _refused(gb.fetch_stats)             # not the previous build's counters
        _plan([gb], counts)
        got = _build([gb])
        _assert_same(got, gb.build(primary, secondary))


def test_a_failed_stage_leaves_nothing_staged(built):
    primary, secondary = _inputs(906)
    with GraphBuilder(L, K, MF, MQ) as gb:
        gb.build(primary, secondary)
        bad = primary.copy()
        bad[(2 * L + 1) * 3] = ord("2")                                  # strand byte of record 3
        with pytest.raises(VdjGraphError) as e:
            gb.stage(bad, secondary)
        assert e.value.code == ERR_STRAND
        for call in (gb.fetch_stats, gb.fetch, gb.run):
            assert "in state EMPTY" in _refused(call)


def test_two_ranks_on_one_gpu(built):
    primary, secondary = _inputs(907)
    rb = 2 * L + 1
    total = primary.size // rb + secondary.size // rb
    parts = [shard.split_records(primary, secondary, L, lo, hi) for lo, hi in shard.shard_ranges(total, 2)]
    builders = [GraphBuilder(L, K, MF, MQ, device=0) for _ in range(2)]
    counts = [builders[0]._n_records(p, s) for p, s in parts]
    try:
        g = shard.build_local(builders, parts)
        assert builders[1].fetch_stats()["n_records"] == counts[1]       # every rank has its counters ...
        assert "other than 0" in _refused(builders[1].fetch)             # ... rank 0 the graph
        for b in builders:
            assert "ranks" in _refused(_query, b)
        _plan(builders, counts)                                          # the same staged records again
        again = _build(builders)
    finally:
        for b in builders:
            b.close()
    _assert_same(again, g)
