"""Alternates bench.py runs over library builds and knob settings, and reports what the survivor
table (table 2) and pass 2 cost in each.

    python profiles/survivor_table_ab.py --out /tmp/ab.json --repeat 5 \\
        --variant old:VDJGRAPH_LIB=build/old/libvdjgraph.so --variant new:

Each --variant is LABEL:ENV=VALUE,ENV=VALUE (nothing after the colon: the in-tree library with its
defaults); a relative VDJGRAPH_LIB is taken from the repository root, e.g. build/old/libvdjgraph.so =
the parent commit's library built by its own Makefile and copied there (build/ is not tracked).
The variants run in turn, --repeat times over, so that a slow minute of a shared host lands on all
of them.  Every run is a fresh process: bench.py's device-resident step (--steps after
--warmup), with the CPU baseline and the forward-reads measurement left out.  The JSON written to
--out keeps every run's step time, the kernel times of the table-2 build and of pass 2, the pass-2
slow-path fraction and the digest check, plus the card's name and power limit read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return {}
    return dict(zip(q.split(","), (v.strip() for v in out.split(","))))


def parse_variant(spec: str) -> tuple[str, dict]:
    label, _, envs = spec.partition(":")
    env = {}
    for kv in filter(None, envs.split(",")):
        k, _, v = kv.partition("=")
        env[k] = v
    return label, env


def run_once(workload: str, env: dict, steps: int, warmup: int) -> dict:
    cmd = [sys.executable, "bench.py", "--workload", workload, "--steps", str(steps), "--warmup", str(warmup),
           "--no-cpu-baseline", "--no-forward"]
    e = dict(os.environ)
    for k, v in env.items():
        e[k] = os.path.join(ROOT, v) if k == "VDJGRAPH_LIB" and not os.path.isabs(v) else v
    r = subprocess.run(cmd, cwd=ROOT, env=e, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit(f"{' '.join(cmd)} with {env} failed ({r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    d = json.loads(lines[-1])
    km, c = d["kernel_ms"], d["config"]
    return {"ms_per_step": d["ms_per_step"], "ms_table2": km["ms_table2"], "ms_pass2": km["ms_pass2"],
            "ms_prune": km["ms_prune"], "ms_pass1": km["ms_pass1"], "kernel_ms": km,
            "slow_path_fraction_pass2": c["slow_path_fraction_pass2"], "table2_slots": c["table2_slots"],
            "nodes": c["nodes"], "digest_ok": (d.get("digest_check") or {}).get("ok"), "clocks": d.get("clocks")}


def summary(runs: list[dict]) -> dict:
    out = {}
    for key in ("ms_per_step", "ms_table2", "ms_pass2", "ms_prune", "slow_path_fraction_pass2"):
        v = [r[key] for r in runs]
        out[key] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    v = [r["ms_table2"] + r["ms_pass2"] for r in runs]
    out["ms_table2_plus_pass2"] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", action="append", required=True, help="LABEL:ENV=VALUE,...")
    ap.add_argument("--workload", default="igh_2x50_5M")
    ap.add_argument("--repeat", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    variants = [parse_variant(s) for s in args.variant]
    result = {"card": card(), "workload": args.workload, "steps": args.steps, "warmup": args.warmup,
              "variants": {label: {"env": env, "runs": []} for label, env in variants}}
    t0 = time.time()
    for i in range(args.repeat):
        for label, env in variants:
            r = run_once(args.workload, env, args.steps, args.warmup)
            result["variants"][label]["runs"].append(r)
            print(f"[{time.time() - t0:6.0f} s] {label} #{i}: {r['ms_per_step']:.3f} ms/step  table2 {r['ms_table2']:.3f}  "
                  f"pass2 {r['ms_pass2']:.3f}  slow2 {r['slow_path_fraction_pass2']:.4f}  digest {r['digest_ok']}", flush=True)
    for label, v in result["variants"].items():
        v["summary"] = summary(v["runs"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], **{k: v["summary"] for k, v in result["variants"].items()}}, indent=1))


if __name__ == "__main__":
    main()
