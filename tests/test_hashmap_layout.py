"""The layout of the reference's `nodes` map (dense_hash_map bucket of every node), three ways:
the real container (compiled reference, oracle/_ref/libvdjglue.so), the sequential model
(tests/hashmap_model.py) and the library's device-side export (VDJGRAPH_FLAG_HASHMAP_LAYOUT)."""
import numpy as np
import pytest

from oracle import loader
from tests import hashmap_model
from tests.util import kmer_codes_at
from vdjer_b200 import synth

CASES = [
    (50, 35, 3, 90, 6000, 120, 101),
    (50, 25, 1, 20, 5000, 60, 103),      # many nodes per read: long probe chains in the small tables
    (100, 50, 2, 120, 3000, 80, 109),    # k = 50: six full Murmur words and a two-character tail
    (36, 35, 2, 40, 3000, 10, 120),
    (20, 8, 2, 40, 300, 5, 7),           # a handful of nodes: the 32-bucket table
]


def _case(L, k, mf, mq, pairs, clones, seed):
    primary, secondary = synth.generate(n_pairs=pairs, read_length=L, seed=seed, n_clones=clones, threads=2)
    g = loader.build(primary, secondary, L, k, mf, mq, kind="port")
    return primary, secondary, g


@pytest.mark.skipif(not loader.have_glue(), reason="oracle/_ref/libvdjglue.so not built (no /root/reference)")
@pytest.mark.parametrize("L,k,mf,mq,pairs,clones,seed", CASES)
def test_model_reproduces_the_reference_container(built, L, k, mf, mq, pairs, clones, seed):
    primary, secondary, g = _case(L, k, mf, mq, pairs, clones, seed)
    ids, buckets = loader.reference_iteration_order(primary, secondary, L, k, mf, mq, g["n_nodes"])
    slots, nb = hashmap_model.layout(kmer_codes_at(primary, secondary, L, k, g["first_pos"]))
    assert nb == buckets
    assert np.array_equal(slots[slots >= 0].astype(np.uint32), ids)


@pytest.mark.gpu
@pytest.mark.parametrize("L,k,mf,mq,pairs,clones,seed", CASES + [(50, 35, 3, 90, 60000, 1500, 4242)])
def test_device_layout_matches_model_and_reference(built, L, k, mf, mq, pairs, clones, seed):
    from vdjer_b200 import GraphBuilder
    primary, secondary, g = _case(L, k, mf, mq, pairs, clones, seed)
    with GraphBuilder(L, k, mf, mq, hashmap_layout=True) as gb:
        got = gb.build(primary, secondary)
    assert got.n_nodes == g["n_nodes"]
    slots, nb = hashmap_model.layout(kmer_codes_at(primary, secondary, L, k, g["first_pos"]))
    assert got.stats["hm_buckets"] == nb and got.hm_slots is not None
    want = np.where(slots < 0, 0xFFFFFFFF, slots).astype(np.uint32)
    assert np.array_equal(got.hm_slots, want)
    if loader.have_glue():
        ids, buckets = loader.reference_iteration_order(primary, secondary, L, k, mf, mq, g["n_nodes"])
        assert buckets == nb and np.array_equal(got.hm_slots[got.hm_slots != 0xFFFFFFFF], ids)


@pytest.mark.gpu
def test_layout_of_sharded_and_multi_round_builds(built):
    """The layout is computed from the finished graph, whichever way it was built."""
    from vdjer_b200 import GraphBuilder
    L, k, mf, mq = 50, 35, 3, 90
    primary, secondary, g = _case(L, k, mf, mq, 20000, 400, 55)
    slots, nb = hashmap_model.layout(kmer_codes_at(primary, secondary, L, k, g["first_pos"]))
    want = np.where(slots < 0, 0xFFFFFFFF, slots).astype(np.uint32)
    with GraphBuilder(L, k, mf, mq, hashmap_layout=True, rounds=4) as gb:
        got = gb.build(primary, secondary)
    assert np.array_equal(got.hm_slots, want)
    from vdjer_b200 import MultiBuilder, shard
    for G in (2, 4):
        total = (primary.size // (2 * L + 1)) + (secondary.size // (2 * L + 1))
        parts = [shard.split_records(primary, secondary, L, lo, hi) for lo, hi in shard.shard_ranges(total, G)]
        builders = [GraphBuilder(L, k, mf, mq, device=0, hashmap_layout=True, rounds=2 if G == 2 else 0) for _ in range(G)]
        try:
            got = shard.build_local(builders, parts)
        finally:
            for b in builders:
                b.close()
        assert got.stats["hm_buckets"] == nb and np.array_equal(got.hm_slots, want), f"sharded G={G}"
    with MultiBuilder(L, k, mf, mq, devices=[0, 0], hashmap_layout=True) as mb:
        got = mb.build(primary, secondary)
    assert got.stats["hm_buckets"] == nb and np.array_equal(got.hm_slots, want), "multi"
