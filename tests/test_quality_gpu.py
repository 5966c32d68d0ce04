"""GPU: the prune's quality-flag bound against the oracle on qualities that split the gate from HIQ.

On synth.generate's qualities "phred >= 20" and "phred >= 30" are the same bit, so a build that set the
flags k_prune bounds quality sums with (window all >= HIQ, record start all >= HIQ) from the gate would
pass every other comparison with the oracle.  Here the qualities are redrawn (tests/quality_profiles.py)
and the pruned pass-1 table, the graph and the counters are compared on every build route;
tests/test_quality_host.py shows each case here would fail under that mistake."""
import functools

import numpy as np
import pytest

from oracle import loader
from tests import quality_profiles as qp
from tests.util import assert_graph_equal, assert_pre_table_equal
from vdjer_b200 import GraphBuilder, MultiBuilder, PinnedRecords, forward_reads, shard

pytestmark = pytest.mark.gpu

COUNTERS = ["n_pre_total", "n_gated", "n_hits"]


@functools.lru_cache(maxsize=None)
def _inputs(profile, L, k):
    return qp.shape_inputs(profile, L, k)


def _sharded(primary, secondary, L, k, mf, mq, G, **kw):
    rb = 2 * L + 1
    total = (primary.size // rb) + (secondary.size // rb)
    parts = [shard.split_records(primary, secondary, L, lo, hi) for lo, hi in shard.shard_ranges(total, G)]
    builders = [GraphBuilder(L, k, mf, mq, device=0, **kw) for _ in range(G)]
    try:
        g = shard.build_local(builders, parts)
        stats = [b.fetch_stats() for b in builders]
    finally:
        for b in builders:
            b.close()
    return g, stats


def _check(got, pre, counters, want, primary, secondary, L, k, what):
    if pre is not None:
        assert_pre_table_equal(pre, want, primary, secondary, L, k, what)
    assert_graph_equal(got, want, what)
    for name in COUNTERS:
        assert counters[name] == want[name], f"{what}: {name} {counters[name]} != {want[name]}"


@pytest.mark.parametrize("shape", range(len(qp.SHAPES)), ids=[f"L{L}k{k}" for L, k in qp.SHAPES])
@pytest.mark.parametrize("profile", sorted(qp.PROFILES))
def test_mq_sweep_matches_oracle(built, profile, shape):
    """One staging per input, then every (mf, mq) of the sweep on it."""
    L, k = qp.SHAPES[shape]
    primary, secondary = _inputs(profile, L, k)
    with GraphBuilder(L, k) as gb:
        gb.stage(primary, secondary)
        for mf, mq in qp.sweep(shape):
            gb.set_params(mf=mf, mq=mq)
            gb.run()
            got, pre = gb.fetch(), gb.pre_table()
            want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
            _check(got, pre, got.stats, want, primary, secondary, L, k, f"{profile} L{L} k{k} mf{mf} mq{mq}")


def _summed(stats):
    return {name: sum(s[name] for s in stats) for name in COUNTERS}


def _route_build(route, primary, secondary, L, k, mf, mq):
    """(graph, pruned pass-1 table or None, counters) of one build through `route`"""
    if route.startswith("shard"):
        got, stats = _sharded(primary, secondary, L, k, mf, mq, int(route[5:]))
        return got, None, _summed(stats)
    if route == "multi2":
        with MultiBuilder(L, k, mf, mq, devices=[0, 0]) as mb:
            got = mb.build(primary, secondary)
            return got, None, _summed([mb.rank_stats(r) for r in range(2)])
    kw = dict(partitions=1) if route == "partitions1" else dict(partitions=256) if route == "partitions256" else \
        dict(wide_tuples=True) if route == "wide_tuples" else dict(rounds=int(route[6:])) if route.startswith("rounds") \
        else {}
    with GraphBuilder(L, k, mf, mq, **kw) as gb:
        if route == "forward":
            got = gb.build_forward(forward_reads(primary, L), forward_reads(secondary, L))
        elif route == "pinned":
            with PinnedRecords(primary, secondary):
                got = gb.build(primary, secondary)
        else:
            got = gb.build(primary, secondary)
        pre = None if route.startswith("rounds") else gb.pre_table()   # kept by one-round builds only
    return got, pre, got.stats


@pytest.mark.parametrize("profile", qp.ROUTE_PROFILES)
@pytest.mark.parametrize("route", qp.ROUTES)
def test_routes_match_oracle(built, route, profile, monkeypatch):
    """Doubled text (pageable, page-locked), forward reads, partition counts, 24-byte tuples, rounds, no read
    fingerprints (every distinct-read decision compares the packed reads), sharded over 2 and 4 contexts
    (quality rows read from a peer's records) and vdjgraph_multi_* on one GPU named twice."""
    if route == "fp_bits0":
        monkeypatch.setenv("VDJGRAPH_FP_BITS", "0")
    L, k = qp.ROUTE_SHAPE
    primary, secondary = _inputs(profile, L, k)
    for mf, mq in qp.ROUTE_FLAGS:
        want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
        got, pre, counters = _route_build(route, primary, secondary, L, k, mf, mq)
        if route == "wide_tuples":
            assert got.stats["tuple_bytes"] == 24
        _check(got, pre, counters, want, primary, secondary, L, k, f"{route} {profile} mf{mf} mq{mq}")


def test_mid_size_matches_oracle(built):
    """300 k pairs: k_prune's warp-wide row path sees many border k-mers per warp across many hash units."""
    m = qp.MID
    L, k, mf, mq = m["L"], m["k"], m["mf"], m["mq"]
    primary, secondary = qp.mid_inputs()
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    with GraphBuilder(L, k, mf, mq) as gb:
        got = gb.build(primary, secondary)
        pre = gb.pre_table()
    _check(got, pre, got.stats, want, primary, secondary, L, k, "mid-size")
    assert np.count_nonzero(want["pre_freq"] <= 3) > 10_000     # survivors that needed their quality rows
