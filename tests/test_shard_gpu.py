"""GPU: the sharded build (SURVEY 8e) gives exactly the single-device result.

G ranks run as G contexts inside this process on ONE GPU (peer buffers are plain device pointers;
across processes the same phases run over CUDA IPC mappings, see vdjer_b200/shard.py and
tests/test_shard_dist.py): every tuple is written by the scatter kernel into the buffer of the
rank that owns its hash partition, reads are compared and quality rows fetched across ranks, and
rank 0 finishes over the gathered survivor records."""
import os

import numpy as np
import pytest

from oracle import loader
from tests.cases import CASES, make_inputs
from tests.util import GOLDEN_DIR, assert_graph_equal
from vdjer_b200 import GraphBuilder, MultiBuilder, shard, synth

pytestmark = pytest.mark.gpu


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


@pytest.mark.parametrize("G", [2, 4, 8])
@pytest.mark.parametrize("L,k,mf,mq,pairs,clones,seed", [
    (50, 35, 3, 90, 40000, 800, 201),
    (50, 25, 1, 20, 20000, 150, 202),      # heavy branching: edge order across owners
    (100, 50, 2, 120, 10000, 300, 203),    # wide tuples
])
def test_sharded_equals_single_device_and_oracle(built, G, L, k, mf, mq, pairs, clones, seed):
    primary, secondary = synth.generate(n_pairs=pairs, read_length=L, seed=seed, n_clones=clones, threads=4)
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    got, stats = _sharded(primary, secondary, L, k, mf, mq, G)
    assert_graph_equal(got, want, f"G={G}")
    assert sum(s["n_pre_total"] for s in stats) == want["n_pre_total"]      # k-mers are owned by exactly one rank
    assert sum(s["n_gated"] for s in stats) == want["n_gated"]
    assert sum(s["n_hits"] for s in stats) == want["n_hits"]
    with GraphBuilder(L, k, mf, mq) as gb:
        single = gb.build(primary, secondary)
    for name in ["first_pos", "frequency", "out_deg", "in_deg", "out_succ", "in_pred"]:
        assert np.array_equal(getattr(got, name), getattr(single, name)), name


@pytest.mark.parametrize("G", [2, 8])
def test_sharded_duplicates_and_strand_across_ranks(built, G):
    """Identical reads that land on different ranks must still count as ONE read for
    hasMultipleUniqueReads (:349-352): the exact comparison reads the peer's packed reads."""
    L, k = 50, 35
    primary, secondary = synth.generate(n_pairs=6000, read_length=L, seed=205, n_clones=60, threads=4)
    rb = 2 * L + 1
    body = primary[:-1].reshape(-1, rb)
    primary = np.concatenate([body, body, body[::-1]]).reshape(-1)      # every record three times, far apart
    primary = np.concatenate([primary, np.zeros(1, np.uint8)])
    want = loader.build(primary, secondary, L, k, 2, 60, kind="port")
    got, _ = _sharded(primary, secondary, L, k, 2, 60, G)
    assert_graph_equal(got, want, f"dups G={G}")


def test_sharded_empty_rank(built):
    """A rank without records (fewer records than ranks) takes part in every phase."""
    L, k = 50, 35
    primary, secondary = synth.generate(n_pairs=3000, read_length=L, seed=206, n_clones=30, threads=2)
    want = loader.build(primary, secondary, L, k, 2, 60, kind="port")
    rb = 2 * L + 1
    total = primary.size // rb + secondary.size // rb
    parts = [shard.split_records(primary, secondary, L, 0, total)] + [(np.zeros(0, np.uint8), np.zeros(0, np.uint8))] * 3
    builders = [GraphBuilder(L, k, 2, 60, device=0) for _ in range(4)]
    try:
        got = shard.build_local(builders, parts)
    finally:
        for b in builders:
            b.close()
    assert_graph_equal(got, want, "empty ranks")


def test_multi_process_parity_over_nvlink(built):
    """One process per GPU (torchrun), peer buffers mapped with CUDA IPC, tuples written over NVLink
    by the scatter kernel: bit-exact against the oracle (tests/mgpu_parity.py).  Needs >= 2 GPUs."""
    import os
    import subprocess
    import sys

    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs on the box")
    world = 8 if n >= 8 else 4 if n >= 4 else 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "tests", "mgpu_parity.py")],
                       capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("PARITY OK") == 3, r.stdout[-2000:]


@pytest.mark.parametrize("G", [2, 4])
def test_sharded_from_forward_reads_only(built, G):
    """vdjgraph_shard_stage_forward: every rank stages forward reads only, the reverse-complement
    records are derived on its device; record numbers stay those of the doubled buffers."""
    from vdjer_b200 import forward_reads
    L, k, mf, mq = 50, 35, 3, 90
    primary, secondary = synth.generate(n_pairs=40000, read_length=L, seed=207, n_clones=600, threads=4)
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    rb = 2 * L + 1
    total = primary.size // rb + secondary.size // rb
    parts = []
    for lo, hi in shard.shard_ranges(total, G):          # even boundaries: a read stays with its reverse complement
        p, s = shard.split_records(primary, secondary, L, lo, hi)
        parts.append((forward_reads(p, L), forward_reads(s, L)))
    builders = [GraphBuilder(L, k, mf, mq, device=0) for _ in range(G)]
    try:
        got = shard.build_local(builders, parts, forward=True)
    finally:
        for b in builders:
            b.close()
    assert_graph_equal(got, want, f"forward G={G}")


def _exports_equal(got, single, what):
    """The k-mer array and the hash-map layout of a sharded finish equal the one-device build's."""
    for name in ["kmer_lo", "kmer_hi", "hm_slots"]:
        a, b = getattr(got, name), getattr(single, name)
        assert a is not None and np.array_equal(a, b), f"{what}: {name}"
    assert got.stats["hm_buckets"] == single.stats["hm_buckets"], what


@pytest.mark.parametrize("how", ["shard2", "shard8", "multi4"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_sharded_exports_of_golden_cases(built, name, how):
    """Every golden case through the distributed finish with k-mers and hash-map layout exported: the graph
    equals the compiled reference's (frequency saturation at 32765 included), the exports the one-device build's."""
    case = CASES[name]
    L, k, mf, mq = case["L"], case["k"], case["mf"], case["mq"]
    gold = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    gold["n_nodes"] = len(gold["first_pos"])
    primary, secondary = make_inputs(case)
    kw = dict(export_keys=True, hashmap_layout=True)
    with GraphBuilder(L, k, mf, mq, **kw) as gb:
        single = gb.build(primary, secondary)
    assert_graph_equal(single, gold, f"{name} one device")
    if how == "multi4":
        with MultiBuilder(L, k, mf, mq, devices=[0] * 4, **kw) as mb:
            got = mb.build(primary, secondary)
    else:
        got, _ = _sharded(primary, secondary, L, k, mf, mq, int(how[5:]), **kw)
    assert_graph_equal(got, gold, f"{name} {how}")
    _exports_equal(got, single, f"{name} {how}")


def _four_way_input(k):
    """Reads f1 + p + C + s + f2 for a random core k-mer C, every pair of flanking bases p, s and three pairs of
    far flanks: C (and its reverse complement) has four successors and four predecessors, each seen in
    several distinct reads."""
    rng = np.random.default_rng(11)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))

    core = rnd(k)
    flanks = [(rnd(8), rnd(8)) for _ in range(3)]
    reads = [f1 + p + core + s + f2 for f1, f2 in flanks for p in "ACGT" for s in "ACGT"]
    return synth.records_from_reads(reads), np.zeros(1, np.uint8)


@pytest.mark.parametrize("G", [2, 8])
def test_sharded_fourth_successor_and_predecessor(built, G):
    """A node's fourth edge does not fit its 32-byte row in the distributed finish and goes through the
    overflow list."""
    L, k, mf, mq = 30, 12, 2, 40
    primary, secondary = _four_way_input(k)
    want = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    assert np.count_nonzero((want["out_deg"] == 4) & (want["in_deg"] == 4)) >= 2
    kw = dict(export_keys=True, hashmap_layout=True)
    got, stats = _sharded(primary, secondary, L, k, mf, mq, G, **kw)
    assert_graph_equal(got, want, f"four-way G={G}")
    assert sum(s["n_pre_total"] for s in stats) == want["n_pre_total"]
    with GraphBuilder(L, k, mf, mq, **kw) as gb:
        single = gb.build(primary, secondary)
    assert_graph_equal(single, want, "four-way one device")
    _exports_equal(got, single, f"four-way G={G}")
