"""The drop-in seam: glue/vdjgraph_glue.inc rebuilds the reference's `nodes` map, node pool and
toNodes/fromNodes lists from vdjgraph_result arrays; the reference's OWN downstream code
(identify_root_nodes :653, condense_graph :598, dump_graph :1133) must then write a vdjer.dot that
is byte-identical to the one it writes after its own build_pre_graph/prune_pre_graph/build_graph2.

CPU test: arrays from the oracle (same layout).  GPU test: arrays from libvdjgraph.
Needs oracle/_ref/libvdjglue.so (compiled from /root/reference by oracle/Makefile; travels to the
GPU box prebuilt)."""
import os

import pytest

from oracle import loader
from tests.cases import CASES, make_inputs

needs_glue = pytest.mark.skipif(not loader.have_glue(), reason="oracle/_ref/libvdjglue.so not built (no /root/reference)")

# k = 50 is left out: dump_graph copies k characters + NUL into char buf[50] (:1179-1181)
DOT_CASES = ["igh_default_k35", "igh_sensitive_k25", "permissive_k25", "igk_2x75_k35", "pooled_2x100_k35",
             "k16", "k33", "noisy", "mq0", "secondary_only", "hand_edges"]


def _dots(tmp_path, name, graph):
    case = CASES[name]
    primary, secondary = make_inputs(case)
    a, b = str(tmp_path / "ref.dot"), str(tmp_path / "glue.dot")
    want = loader.glue_dot(primary, secondary, case["L"], case["k"], case["mf"], case["mq"], a)
    g = graph(primary, secondary, case)
    got = loader.glue_dot(primary, secondary, case["L"], case["k"], case["mf"], case["mq"], b, graph=g)
    return want, got, open(a, "rb").read(), open(b, "rb").read()


@needs_glue
@pytest.mark.parametrize("name", DOT_CASES)
def test_vdjer_dot_identical_from_oracle_arrays(tmp_path, built, name):
    want, got, ref_dot, glue_dot = _dots(
        tmp_path, name, lambda p, s, c: loader.build(p, s, c["L"], c["k"], c["mf"], c["mq"], kind="port"))
    assert got == want, f"{name}: (nodes, roots) {got} != {want}"
    assert glue_dot == ref_dot, f"{name}: vdjer.dot differs"
    assert len(ref_dot) > 40 or want[0] == 0


@needs_glue
@pytest.mark.parametrize("name", ["igh_default_k35", "permissive_k25", "pooled_2x100_k35", "k16", "hand_edges"])
def test_vdjer_dot_identical_with_bulk_loaded_map(tmp_path, built, name):
    """The glue's fast path: `nodes` loaded in one pass (sparsehash unserialize) from the bucket layout --
    here the sequential model's (tests/hashmap_model.py), on the GPU the library's -- instead of replaying
    the inserts.  Same vdjer.dot, i.e. same iteration order, ids, edges and condensed sequences."""
    from tests import hashmap_model
    from tests.util import kmer_codes_at
    import numpy as np

    def with_layout(p, s, c):
        g = loader.build(p, s, c["L"], c["k"], c["mf"], c["mq"], kind="port")
        slots, _ = hashmap_model.layout(kmer_codes_at(p, s, c["L"], c["k"], g["first_pos"]))
        g["hm_slots"] = np.where(slots < 0, 0xFFFFFFFF, slots).astype(np.uint32)
        return g

    want, got, ref_dot, glue_dot = _dots(tmp_path, name, with_layout)
    assert got == want, f"{name}: (nodes, roots) {got} != {want}"
    assert glue_dot == ref_dot, f"{name}: vdjer.dot differs"


@needs_glue
@pytest.mark.parametrize("damage", ["missing", "out_of_range"])
def test_bulk_load_rejects_a_layout_that_does_not_name_every_node(tmp_path, built, damage):
    """The glue fills the map's buckets in parallel from the exported layout; a layout that leaves a node out
    (or names one that does not exist) must fail the rebuild, not leave a map with a wrong element count."""
    from tests import hashmap_model
    from tests.util import kmer_codes_at
    import numpy as np
    c = CASES["igh_default_k35"]
    p, s = make_inputs(c)
    g = loader.build(p, s, c["L"], c["k"], c["mf"], c["mq"], kind="port")
    slots, _ = hashmap_model.layout(kmer_codes_at(p, s, c["L"], c["k"], g["first_pos"]))
    hm = np.where(slots < 0, 0xFFFFFFFF, slots).astype(np.uint32)
    at = int(np.flatnonzero(hm != 0xFFFFFFFF)[3])
    hm[at] = 0xFFFFFFFF if damage == "missing" else g["n_nodes"] + 5
    g["hm_slots"] = hm
    with pytest.raises(RuntimeError):
        loader.glue_dot(p, s, c["L"], c["k"], c["mf"], c["mq"], str(tmp_path / "x.dot"), graph=g)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [False, True])
@pytest.mark.parametrize("name", DOT_CASES)
def test_vdjer_dot_identical_from_cuda_graph(tmp_path, built, name, layout):
    """Everything the glue reads from the library is the reference's own: the graph arrays equal the ones
    the compiled reference stored for this case (tests/golden), and the map layout equals the sequential
    model's (pinned to the reference's container by test_hashmap_layout.py).  vdjer.dot is a function of
    the records and these arrays only; where the reference's downstream code is built, it is compared
    byte for byte as well."""
    import numpy as np

    from tests import hashmap_model
    from tests.util import GOLDEN_DIR, assert_graph_equal, kmer_codes_at
    from vdjer_b200 import GraphBuilder

    def cuda(p, s, c):
        with GraphBuilder(c["L"], c["k"], c["mf"], c["mq"], hashmap_layout=layout) as gb:
            return gb.build(p, s)

    case = CASES[name]
    primary, secondary = make_inputs(case)
    g = cuda(primary, secondary, case)
    gold = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    gold["n_nodes"] = len(gold["first_pos"])
    assert_graph_equal(g, gold, name)
    if layout:
        slots, nb = hashmap_model.layout(kmer_codes_at(primary, secondary, case["L"], case["k"], gold["first_pos"]))
        assert g.stats["hm_buckets"] == nb
        assert np.array_equal(g.hm_slots, np.where(slots < 0, 0xFFFFFFFF, slots).astype(np.uint32))
    if not loader.have_glue():
        return
    want, got, ref_dot, glue_dot = _dots(tmp_path, name, cuda)
    assert got == want, f"{name}: (nodes, roots) {got} != {want}"
    assert glue_dot == ref_dot, f"{name}: vdjer.dot differs"


@needs_glue
def test_glue_rebuild_timer(built):
    """The measurement hook behind profiles/glue_rebuild_time.py (cost of the reference-side rebuild
    after the library call) runs and returns a plausible wall time."""
    case = CASES["igh_default_k35"]
    primary, secondary = make_inputs(case)
    g = loader.build(primary, secondary, case["L"], case["k"], case["mf"], case["mq"], kind="port")
    ms = loader.glue_rebuild_ms(primary, secondary, case["L"], case["k"], g)
    assert 0 <= ms < 60_000
