"""CPU: bench.py's reference arm (the reference's own CPU functions, or the oracle port when the
compiled reference is absent) prints the contract's JSON line; non-zero ranks of a torchrun launch
stay silent.  The CUDA arm needs a B200 and is exercised by the driver."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, args=()):
    env = dict(os.environ)
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample-pairs", "3000", *args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_json_line(built):
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "graph_build_prune_windows_per_sec" and d["unit"] == "windows/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] == 1
    assert d["cpu_baseline"]["value"] == d["value"] and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "igh_2x50_5M"


def test_reference_arm_other_ranks_are_silent(built):
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == []


def test_reference_arm_dumps_the_graph_of_its_last_step(built, tmp_path):
    """--dump-outputs: the same float64 arrays in every run, and they are the graph of the timed sample."""
    import numpy as np

    from oracle import loader
    from vdjer_b200 import synth
    for d in ("a", "b"):
        d = json.loads(_run(args=["--dump-outputs", str(tmp_path / d)])[0])["outputs_dumped"]
        assert d["nodes"] == d["rows"] > 0
    wl = dict(synth.CONFIGS["igh_2x50_5M"])
    primary, secondary = synth.generate(**dict(wl, n_pairs=3000))
    want = loader.build(primary, secondary, wl["read_length"], wl["k"], wl["mf"], wl["mq"], kind="port")
    want.update(n_nodes=[want["n_nodes"]], node_index=np.arange(want["n_nodes"]))
    for name in ["n_nodes", "node_index", "first_pos", "frequency", "out_deg", "in_deg", "out_succ", "in_pred"]:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b), name
        assert np.array_equal(a, np.asarray(want[name], dtype=np.float64)), name


def test_dump_of_a_large_graph_is_a_fixed_sample_below_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np

    import bench
    n = 1_000_000
    rng = np.random.default_rng(1)
    g = dict(first_pos=np.arange(n, dtype=np.uint64) * 7, frequency=rng.integers(1, 32766, n).astype(np.uint16),
             out_deg=rng.integers(0, 5, n).astype(np.uint8), in_deg=rng.integers(0, 5, n).astype(np.uint8),
             out_succ=rng.integers(0, 2**32, (n, 4)).astype(np.uint32), in_pred=rng.integers(0, 2**32, (n, 4)).astype(np.uint32))
    for d in ("a", "b"):
        info = bench.dump_outputs(str(tmp_path / d), g)
        assert info["nodes"] == n and 0 < info["rows"] < n
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) < 64_000_000
    idx = np.load(tmp_path / "a" / "node_index.npy")
    assert idx.size == info["rows"] and np.all(np.diff(idx) > 0)
    assert np.array_equal(idx, np.load(tmp_path / "b" / "node_index.npy"))
    rows = idx.astype(np.int64)
    for name, a in g.items():
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), a[rows].astype(np.float64)), name
