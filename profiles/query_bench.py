"""vdjgraph_query on BASELINE configs[1] (synth igh_2x50_5M, seed 12345 as in bench.py; 5 M pairs, L = 50,
k = 35): windows per second of the query kernels and end to end, on two batches.

  (a) every forward read of the input, one query each: 10 M queries, 1.6e8 windows
  (b) 100 k queries of 400 bp, each 8 consecutive forward reads: windows across read borders, many of them
      not in the graph

Each batch runs with its text and answer arrays page-locked (registered, as a caller that takes them from
vdjgraph_host_alloc has them: DMA straight from / to them) and pageable (bounced through the library's
page-locked chunks).  One warm-up call, then REPS timed calls; medians are reported.  A seeded sample of 1e5
windows per batch is checked against an index built from the fetched graph's k-mers (export_keys=True); the
script exits non-zero on a mismatch.  Prints one JSON line (and writes it to --out).

    python profiles/query_bench.py [--out FILE] [--reps 5] [--pairs N]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.query_model import NodeIndex, answers_at  # noqa: E402
from vdjer_b200 import GraphBuilder, PinnedRecords, forward_reads, synth  # noqa: E402
from vdjer_b200.graph import NIL  # noqa: E402


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def read_bases(buf, L) -> np.ndarray:
    """[n_reads, L] bases of the forward reads of a record buffer."""
    return forward_reads(buf, L)[:-1].reshape(-1, 2 * L + 1)[:, 1:1 + L]


def measure(gb, text, offsets, n_windows, reps, pinned):
    out = np.empty(n_windows, np.uint32)
    lock = PinnedRecords(text, out) if pinned else None
    try:
        gb.query_flat(text, offsets, out=out)   # warm-up
        runs = []
        for _ in range(reps):
            t0 = time.perf_counter()
            _, st = gb.query_flat(text, offsets, out=out)
            st["wall_ms_python"] = (time.perf_counter() - t0) * 1e3
            runs.append(st)
    finally:
        if lock:
            lock.close()
    med = {key: statistics.median(r[key] for r in runs) for key in ("ms_kernels", "ms_total", "wall_ms_python")}
    st = runs[-1]
    return out, {
        "buffers": "page-locked" if pinned else "pageable",
        "reps": reps,
        "ms_kernels_median": round(med["ms_kernels"], 3),
        "ms_total_median": round(med["ms_total"], 3),
        "ms_kernels_all": [round(r["ms_kernels"], 3) for r in runs],
        "ms_total_all": [round(r["ms_total"], 3) for r in runs],
        "windows_per_s_kernels": n_windows / (med["ms_kernels"] * 1e-3),
        "windows_per_s_total": n_windows / (med["ms_total"] * 1e-3),
        "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"],
        "h2d_plus_d2h_GB_per_s_total": (st["h2d_bytes"] + st["d2h_bytes"]) / (med["ms_total"] * 1e-3) / 1e9,
        "n_found": st["n_found"],
    }


def check_sample(name, got, text, per_query_bytes, windows_per_query, k, index, rng, n=100_000):
    w = np.sort(rng.choice(got.size, size=min(n, got.size), replace=False))
    starts = (w // windows_per_query) * per_query_bytes + (w % windows_per_query)
    want = answers_at(text, starts, k, index)
    bad = np.nonzero(got[w] != want)[0]
    return {"batch": name, "windows": int(w.size), "mismatches": int(bad.size),
            "found_in_sample": int((want != NIL).sum()),
            "first_mismatch": None if not bad.size else {"window": int(w[bad[0]]), "got": int(got[w[bad[0]]]), "want": int(want[bad[0]])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--pairs", type=int, default=0, help="override configs[1]'s 5 M pairs (rehearsals)")
    args = ap.parse_args()
    wl = dict(synth.CONFIGS["igh_2x50_5M"])
    if args.pairs:
        wl["n_pairs"] = args.pairs
    L, k, mf, mq = wl["read_length"], wl["k"], wl["mf"], wl["mq"]
    gen = {kk: v for kk, v in wl.items() if kk not in ("k", "mf", "mq")}
    primary, secondary = synth.generate(seed=12345, **gen)
    bases = np.concatenate([read_bases(primary, L), read_bases(secondary, L)])   # [10 M, 50]
    n_reads = bases.shape[0]
    text_a = np.ascontiguousarray(bases).reshape(-1)
    off_a = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(L)
    per_b, n_b = 8 * L, min(100_000, n_reads // 8)
    text_b = np.ascontiguousarray(bases[: n_b * 8]).reshape(-1)
    off_b = np.arange(n_b + 1, dtype=np.uint64) * np.uint64(per_b)
    wa, wb = L - k + 1, per_b - k + 1

    info = gpu_info()
    with GraphBuilder(L, k, mf, mq, export_keys=True) as gb:
        g = gb.build(primary, secondary)
        index = NodeIndex(g.kmer_lo, g.kmer_hi)
        rng = np.random.default_rng(2024)
        result = {"metric": "vdjgraph_query windows/s", "workload": "igh_2x50_5M", "seed": 12345,
                  "n_pairs": wl["n_pairs"], "L": L, "k": k, "n_nodes": g.n_nodes, **info, "batches": {}, "sample_check": []}
        for name, text, off, per_q, w_per_q in (("a_reads", text_a, off_a, L, wa), ("b_400bp", text_b, off_b, per_b, wb)):
            n_w = (off.size - 1) * w_per_q
            entry = {"n_queries": int(off.size - 1), "n_windows": int(n_w), "text_bytes": int(text.size)}
            for pinned in (True, False):
                got, m = measure(gb, text, off, n_w, args.reps, pinned)
                entry["page_locked" if pinned else "pageable"] = m
                result["sample_check"].append(dict(check_sample(name, got, text, per_q, w_per_q, k, index, rng),
                                                   buffers=m["buffers"]))
            entry["found_fraction"] = entry["page_locked"]["n_found"] / n_w
            result["batches"][name] = entry
    result["sample_check_ok"] = all(c["mismatches"] == 0 for c in result["sample_check"])
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if result["sample_check_ok"] else 1)


if __name__ == "__main__":
    main()
