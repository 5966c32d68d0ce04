"""CPU: the quality profiles of tests/quality_profiles.py and what they buy.

Every case of tests/test_quality_gpu.py is shown able to fail: on its input, a build that logged the
window-all->=HIQ flag from the quality gate instead (hiq = gate) would keep at least FLOOR k-mers the
reference prunes.  The model that counts them is checked against the oracle on the same inputs."""
import numpy as np
import pytest

from oracle import loader
from tests import quality_profiles as qp
from tests.spec_model import order_free_build
from vdjer_b200 import forward_reads, synth

FLOOR = 20


def _agrees_with_oracle(model, primary, secondary, L, k, mf, mq):
    got = model.prune(mf, mq)
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    assert (got["n_pre_total"], got["n_pre"]) == (want["n_pre_total"], want["n_pre"]), (mf, mq)
    return got


@pytest.mark.parametrize("shape", range(len(qp.SHAPES)), ids=[f"L{L}k{k}" for L, k in qp.SHAPES])
@pytest.mark.parametrize("profile", sorted(qp.PROFILES))
def test_mq_sweep_inputs_can_fail(built, profile, shape):
    """One GPU test per (profile, shape) runs the whole mq sweep on one input: the window mutant flips at
    least FLOOR prune decisions over the sweep.  It cannot flip any at mq 20 or 40, nor at 21 unless a
    phred is 0 (a border k-mer then has count <= 2: at 20 none passes the distinct-read test, at 40 the
    mutant's bound reaches T only where the real one does, at 21 every sum is >= 20 + a seed phred), and
    rarely just above a multiple of 20; those cases are there for the edges of T and of
    20 * (count - 1) < T.  flat30 has gate == HIQ on every base: nothing can flip, it tests sums and
    bounds equal to T instead."""
    L, k = qp.SHAPES[shape]
    primary, secondary = qp.shape_inputs(profile, L, k)
    model = qp.PruneModel(primary, secondary, L, k)
    res = [model.prune(mf, mq) for mf, mq in qp.sweep(shape)]
    assert all(r["unsound"] == 0 for r in res), "k_prune's bound keeps a k-mer whose sums are below T"
    for mf, mq in [qp.sweep(shape)[4], qp.sweep(shape)[-3]]:
        _agrees_with_oracle(model, primary, secondary, L, k, mf, mq)
    flips = [r["window"] for r in res]
    for (mf, mq), n in zip(qp.sweep(shape), flips):
        if mq in (20, 40) or (mq == 21 and profile != "wide"):
            assert n == 0, (mf, mq)
    if profile == "flat30":
        assert sum(r["both"] for r in res) == 0
    else:
        assert sum(flips) >= FLOOR, dict(zip(qp.MQ_SWEEP, flips))


@pytest.mark.parametrize("profile", qp.ROUTE_PROFILES)
def test_route_inputs_can_fail(built, profile):
    """Every (mf, mq) the route tests build, on their input: at least FLOOR flips each."""
    L, k = qp.ROUTE_SHAPE
    primary, secondary = qp.shape_inputs(profile, L, k)
    model = qp.PruneModel(primary, secondary, L, k)
    for mf, mq in qp.ROUTE_FLAGS:
        r = _agrees_with_oracle(model, primary, secondary, L, k, mf, mq)
        assert r["unsound"] == 0 and r["window"] >= FLOOR, (mf, mq, r)


def test_mid_size_input_can_fail(built):
    m = qp.MID
    primary, secondary = qp.mid_inputs()
    r = qp.PruneModel(primary, secondary, m["L"], m["k"]).prune(m["mf"], m["mq"])
    assert r["unsound"] == 0 and r["window"] >= FLOOR and r["n_border"] > 50_000, r


@pytest.mark.parametrize("profile", sorted(qp.PROFILES))
def test_order_free_spec_matches_oracle_on_profile(built, profile):
    """SURVEY Appendix A's order-free form (tests/spec_model.py) equals the sequential oracle on inputs
    whose qualities separate the gate from HIQ, including one read length with two mask words."""
    for L, k, mf, mq, seed in [(40, 21, 2, 60, 31), (70, 31, 3, 90, 32), (40, 15, 1, 214, 33)]:
        primary, secondary = qp.quality_inputs(profile, L, n_pairs=500, seed=seed, n_clones=10)
        want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
        got = order_free_build(primary, secondary, L, k, mf, mq)
        for a in ["first_pos", "frequency", "out_deg", "out_succ", "in_deg", "in_pred"]:
            assert np.array_equal(got[a], want[a]), (profile, L, k, a)
        assert got["n_pre_total"] == want["n_pre_total"] and got["n_gated"] == want["n_gated"]
        assert qp.flag_sensitivity(primary, secondary, L, k, mf, mq)["n_pre"] == want["n_pre"]


@pytest.mark.parametrize("profile", sorted(qp.PROFILES))
def test_requantize_keeps_bases_and_mirrors_mate_qualities(built, profile):
    L = 60
    primary, _ = synth.generate(n_pairs=400, read_length=L, seed=5, n_clones=10, p_n=0.02, threads=1)
    out = qp.requantize(primary, L, profile, seed=9)
    rb = 2 * L + 1
    assert out.size == primary.size and out[-1] == 0
    a, b = primary[:-1].reshape(-1, 2, rb), out[:-1].reshape(-1, 2, rb)
    assert np.array_equal(a[:, :, :1 + L], b[:, :, :1 + L]), "bases or strand bytes changed"
    q = b[:, :, 1 + L:].astype(np.int64) - 33
    assert np.array_equal(q[:, 1], q[:, 0, ::-1]), "reverse-complement qualities are not the reverse"
    values, _ = qp.PROFILES[profile]
    n = b[:, 0, 1:1 + L] == ord("N")
    assert n.any()
    assert np.isin(q[:, 0][~n], values).all()
    if profile == "n_keeps_quality":
        assert np.isin(q[:, 0][n], values).all() and (q[:, 0][n] != 2).any()
    else:
        assert (q[:, 0][n] == 2).all()
    if profile in ("hug", "novaseq", "wide"):   # qualities between the gate and HIQ occur
        assert ((q >= 20) & (q < 30)).any()
    # still valid input of the forward-reads route: its even records are the reads
    fwd = forward_reads(out, L)
    assert np.array_equal(fwd[:-1].reshape(-1, rb), b[:, 0])
