#!/usr/bin/env python
"""bench.py -- V'DJer de Bruijn graph build+prune throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

A step = one graph build (estimate -> pass 1 -> prune -> pass 2 -> export) over the whole
synthetic read set.  Unit: windows (k-mer positions) per second, W = records * (L-k+1).

  value     device-resident: reads already packed in HBM, K x vdjgraph_run, CUDA events on the
            library's stream (inside the library), max over ranks
  e2e       K x vdjgraph_build on HOST text buffers (the reference's record format): host
            packing + H2D + kernels + D2H of the graph, wall clock, max over ranks
  roofline  dominant kernel's algorithmic bytes (SURVEY 8d) / its CUDA-event time vs the measured
            HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the reference's own functions (oracle/_ref, compiled from /root/reference) or the
            oracle port, on a bounded subsample, one core (the stage is single-threaded in the
            reference: assembler2_vdj.c:1381-1415; --t only sizes the traversal pool :1287-1299)

--impl reference times that CPU path alone with the same metric/config.
N > 1 (torchrun): ONE graph over the reads of all ranks (weak scaling: every rank contributes the
N=1 workload, its own pairs of the same repertoire).  k-mers are hash-sharded by minimizer, the scatter
kernel writes each run into the owning GPU's buffer through peer-mapped memory, survivors are gathered
on rank 0 which ranks the nodes and builds the edge lists (DESIGN.md "Multi-GPU").  All ranks draw
disjoint reads from the SAME clone library (one pooled repertoire sequenced N times deeper).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "graph_build_prune_windows_per_sec"
UNIT = "windows/s"
DEFAULT_WORKLOAD = "igh_2x50_5M"  # BASELINE.json configs[1]
NCU_SUMMARY = "profiles/ncu_r2_summary.json"
GRAPH_ARRAYS = ["first_pos", "frequency", "out_deg", "in_deg", "out_succ", "in_pred"]
DUMP_BYTES = 64_000_000   # --dump-outputs writes less than this in all


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled every few ms from a
    thread (nvidia-smi -lms is too coarse for a sub-second region); nvidia-smi as a fallback."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thread = None
        self.how = None

    def _poll_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        self.how = "nvml"
        while True:
            self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
            try:
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for name, bit in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
            if self._stop.wait(0.004):
                break

    def _poll_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.how = "nvidia-smi"
        while True:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                self.sm.append(float(out[0])); self.max_mhz = float(out[1])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], out[2:6]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            if self._stop.wait(0.02):
                break

    def _run(self):
        try:
            self._poll_nvml()
        except Exception:
            self._poll_smi()

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        time.sleep(0.02)   # first sample lands before the timed region starts

    def stop(self) -> dict:
        self._stop.set()
        self.thread.join(timeout=15)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.how}


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel` from the committed
    ncu --set full capture (profiles/ncu_r1_summary.json, made by profiles/prof_r1.sh on the default
    workload); None when there is no capture."""
    path = os.path.join(ROOT, NCU_SUMMARY)
    try:
        ks = json.load(open(path))["kernels"]
        for name, d in ks.items():
            if name.startswith(kernel):
                return d["dram_traffic_bytes_per_launch"]
    except Exception:
        pass
    return None


def atomic_rates():
    """L2-resident random load+RED / load / RED rates (G ops/s) measured on this pool by
    vdjer_b200/microbench (profiles/microbench_r1.json, 32 MB table row); None if absent."""
    try:
        row = json.load(open(os.path.join(ROOT, "profiles", "microbench_r1.json")))["rows"][0]
        return {"load_red": row["load_red_ilp4"], "load": row["load_ilp4"], "red": row["red_ilp4"], "table_mb": row["table_mb"]}
    except Exception:
        return None


def algorithmic_bytes(L, k, h, gated=1.0, h_rmw=None):
    """Bytes per window of each pass and of the whole path (DESIGN.md section 4).
    SURVEY.md 8d charges every window a slot read-modify-write in pass 1 (gated = 1.0) and every
    pass-2 hit a read-modify-write (h_rmw = h).  In the reference only the windows that pass the
    quality gate reach the pass-1 table (include_kmer :240-259), and here the gated occurrences
    are not counted again in pass 2 (its count is seeded from pass 1), so the figures reported as
    `roofline` charge the pass-1 64 B to the gated fraction and the pass-2 64 B to the UNGATED
    hits only; the SURVEY formula is kept beside them as `survey_formula`."""
    w = L - k + 1
    b_in = 1.25 * L / (2 * w)
    p1 = b_in + 64.0 * gated                            # packed read bytes + one slot sector RMW per gated window
    p2 = b_in + 32.0 + 64.0 * (h if h_rmw is None else h_rmw)   # packed read bytes + membership probe + count RMW
    return p1, p2, p1 + p2


def cpu_baseline(wl: dict, sample_pairs: int, extras: bool = False):
    """The reference's graph build on one host core, on the first `sample_pairs` pairs' worth of
    the same generator.  Only place bench.py touches oracle/."""
    from oracle import loader
    from vdjer_b200 import synth
    gen = {k: v for k, v in wl.items() if k not in ("k", "mf", "mq", "n_pairs")}
    primary, secondary = synth.generate(n_pairs=sample_pairs, **gen)
    kind = "reference" if loader.have_reference() else "port"
    import contextlib
    with open(os.devnull, "w") as dn, contextlib.redirect_stderr(dn):
        fd = os.dup(2); os.dup2(dn.fileno(), 2)   # the reference logs progress to stderr
        try:
            t0 = time.perf_counter()
            r = loader.build(primary, secondary, wl["read_length"], wl["k"], wl["mf"], wl["mq"], kind=kind)
            dt = time.perf_counter() - t0
        finally:
            os.dup2(fd, 2); os.close(fd)
    t_graph = r["t_pass1"] + r["t_prune"] + r["t_pass2"]
    out = {"value": r["n_windows"] / t_graph, "unit": UNIT, "cores": 1, "kind": kind,
           "sample": f"first {sample_pairs} pairs of the same generator ({r['n_windows']} windows, "
                     f"{t_graph:.1f} s: pass1 {r['t_pass1']:.1f} prune {r['t_prune']:.1f} pass2 {r['t_pass2']:.1f}; "
                     f"{'compiled reference -O2' if kind == 'reference' else 'oracle port'}; the stage is single-threaded in the reference)",
           "_windows": r["n_windows"], "_seconds": t_graph, "_wall": dt}
    if extras and kind == "reference":
        # the reference's own flags (-g, no -O: Makefile:8), on a quarter of the sample
        try:
            gp, gs = synth.generate(n_pairs=max(1, sample_pairs // 4), **gen)
            fd = os.dup(2)
            with open(os.devnull, "w") as dn:
                os.dup2(dn.fileno(), 2)
                try:
                    rg = loader.build(gp, gs, wl["read_length"], wl["k"], wl["mf"], wl["mq"], kind="reference", variant="g")
                finally:
                    os.dup2(fd, 2); os.close(fd)
            tg = rg["t_pass1"] + rg["t_prune"] + rg["t_pass2"]
            out["reference_flags_g"] = {"value": rg["n_windows"] / tg, "unit": UNIT,
                                        "sample": f"first {max(1, sample_pairs // 4)} pairs, compiled -g without -O like the reference's Makefile:8 ({tg:.1f} s)"}
        except Exception as e:   # the -g library is optional
            out["reference_flags_g"] = {"unavailable": str(e)[:100]}
    out["_primary"], out["_secondary"] = primary, secondary
    out["_graph"] = r
    return out


def dump_outputs(out_dir: str, graph) -> dict:
    """--dump-outputs: the graph the caller of the timed path received in the last step (node rows in
    creation order, as vdjgraph_fetch returns them) as DIR/<array>.npy in float64, so that two builds
    can be compared output for output.  Every value is an integer below 2^53, so float64 holds it
    exactly.  A graph too large for DUMP_BYTES is sampled: node_index.npy holds the rows kept, a
    seeded choice that depends only on the node count; n_nodes.npy holds the count."""
    arrays = {n: (graph[n] if isinstance(graph, dict) else getattr(graph, n)) for n in GRAPH_ARRAYS}
    n = len(arrays["first_pos"])
    row_bytes = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))   # + node_index
    rows = min(n, (DUMP_BYTES - 4096) // row_bytes)                                   # 4096: .npy headers
    index = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    out = {"n_nodes": np.array([n]), "node_index": index, **{name: a[index] for name, a in arrays.items()}}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    return {"dir": out_dir, "nodes": n, "rows": rows, "dtype": "float64"}


def run_reference(args, wl, rank):
    if rank != 0:
        return
    per_step = []
    cb = None
    for i in range(args.warmup + args.steps):
        cb = cpu_baseline(wl, args.cpu_sample_pairs)
        if i >= args.warmup:
            per_step.append(cb["_seconds"])
    t = float(np.mean(per_step))
    value = cb["_windows"] / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
            "config": {"workload": args.workload, "read_length": wl["read_length"], "k": wl["k"], "mf": wl["mf"],
                       "mq": wl["mq"], "pairs_per_step": args.cpu_sample_pairs,
                       "note": "bounded subsample of the workload; CPU stage is single-threaded in the reference"},
            "cpu_baseline": {k: v for k, v in cb.items() if not k.startswith("_")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    line["cpu_baseline"]["value"] = value
    if args.dump_outputs:
        line["outputs_dumped"] = dump_outputs(args.dump_outputs, cb["_graph"])
    print(json.dumps(line), flush=True)


def _sha_graph(g) -> str:
    import hashlib
    h = hashlib.sha256()
    for name, dt in [("first_pos", np.uint64), ("frequency", np.uint16), ("out_deg", np.uint8), ("in_deg", np.uint8),
                     ("out_succ", np.uint32), ("in_pred", np.uint32)]:
        h.update(np.ascontiguousarray(getattr(g, name), dtype=dt).tobytes())
    return h.hexdigest()


def digest_check(workload: str, graph):
    """The graph of the timed workload against the digest the COMPILED REFERENCE left for it
    (tests/golden/full_digests.json, written by tests/golden/make_full_digest.py): counters and a
    SHA-256 per result array.  None when the workload has no digest."""
    import hashlib
    path = os.path.join(ROOT, "tests", "golden", "full_digests.json")
    try:
        want = json.load(open(path))[workload]
    except Exception:
        return None
    dt = dict(first_pos=np.uint64, frequency=np.uint16, out_deg=np.uint8, in_deg=np.uint8, out_succ=np.uint32, in_pred=np.uint32)
    got = {n: hashlib.sha256(np.ascontiguousarray(getattr(graph, n), dtype=t).tobytes()).hexdigest() for n, t in dt.items()}
    ok = got == want["sha256"] and graph.n_nodes == want["n_nodes"] and graph.stats["n_pre_total"] == want["n_pre_total"]
    if not ok:
        raise SystemExit(f"bench: the graph of {workload} differs from the reference digest in {path}")
    return {"ok": True, "nodes": graph.n_nodes, "sha256_first_pos": got["first_pos"][:16],
            "source": "tests/golden/full_digests.json (compiled reference on this exact workload)"}


def shard_parity_check(torch, dist, db, local_rank: int, rank: int, world: int):
    """N > 1: a small seeded read set is built once on rank 0 alone and once sharded over all ranks
    (the same DistributedBuilder, peer mappings and kernels the timed steps use); the two graphs must
    hash the same.  Every rank exits non-zero on a mismatch."""
    from vdjer_b200 import GraphBuilder, shard, synth
    L, k, mf, mq = 50, 35, 3, 90
    primary, secondary = synth.generate(n_pairs=60000, read_length=L, seed=4242, n_clones=1500, threads=2)
    n_rec = (primary.size + secondary.size) // (2 * L + 1)
    lo, hi = shard.shard_ranges(n_rec, world)[rank]
    mine = shard.split_records(primary, secondary, L, lo, hi)
    old = (db.b._p.read_length, db.b._p.kmer_size, db.b._p.min_node_freq, db.b._p.min_base_quality)
    db.b.set_params(read_length=L, k=k, mf=mf, mq=mq)
    g = db.build(np.ascontiguousarray(mine[0]), np.ascontiguousarray(mine[1]), copy=True)
    db.b.set_params(read_length=old[0], k=old[1], mf=old[2], mq=old[3])
    ok = torch.ones(1, device=f"cuda:{local_rank}")
    out = None
    if rank == 0:
        with GraphBuilder(L, k, mf, mq, device=local_rank) as one:
            ref = one.build(primary, secondary)
        a, b = _sha_graph(g), _sha_graph(ref)
        out = {"ok": a == b, "sha": a[:16], "nodes": g.n_nodes, "ranks": world,
               "case": "60000 pairs 2x50, seed 4242: sharded over all ranks vs rank 0 alone, SHA-256 of every result array"}
        if a != b:
            ok.zero_()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if float(ok[0]) == 0:
        raise SystemExit("bench: the sharded graph differs from the single-GPU graph")
    return out


def glue_cost(args, wl, cb, device, primary, secondary, fwd_in, n_nodes):
    """What the reference-side glue (glue/vdjgraph_glue.inc) costs after the library call, per node, on
    the CPU-baseline sample: (a) `nodes` bulk-loaded from the map layout the library exports
    (VDJGRAPH_FLAG_HASHMAP_LAYOUT, computed on the device), (b) the inserts replayed on one thread as in
    round 1; and what the layout costs the library call on the full workload.  Part of the cpu_baseline
    leg (it drives the reference's own containers through oracle/_ref/libvdjglue.so)."""
    from oracle import loader
    if not loader.have_glue():
        return None
    from vdjer_b200 import GraphBuilder, PinnedRecords, forward_reads
    L, k, mf, mq = wl["read_length"], wl["k"], wl["mf"], wl["mq"]
    out = {}
    try:
        with GraphBuilder(L, k, mf, mq, device=device, hashmap_layout=True) as gl:
            if fwd_in:
                fp, fs = primary, secondary
            else:
                fp, fs = forward_reads(primary, L), forward_reads(secondary, L)
            pin = None if args.pageable else PinnedRecords(fp, fs)
            gl.build_forward(fp, fs, copy=False)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                g = gl.build_forward(fp, fs, copy=False)
            out["e2e_ms_with_layout"] = (time.perf_counter() - t0) / args.steps * 1e3
            out["ms_hashmap_layout"] = g.stats["ms_hashmap"]
            out["hm_buckets"] = g.stats["hm_buckets"]
            if pin is not None:
                pin.close()
            gs = gl.build(cb["_primary"], cb["_secondary"])
        # the glue spreads its work over --t threads (VDJGRAPH_GLUE_THREADS overrides); BASELINE runs the
        # reference with --t = host cores, the glue uses at most 16
        nt = min(16, os.cpu_count() or 1)

        def timed(threads: int, replay: bool) -> float:
            os.environ["VDJGRAPH_GLUE_THREADS"] = str(threads)
            if replay:
                os.environ["VDJGRAPH_GLUE_REPLAY"] = "1"
            try:
                return min(loader.glue_rebuild_ms(cb["_primary"], cb["_secondary"], L, k, gs) for _ in range(2))
            finally:
                os.environ.pop("VDJGRAPH_GLUE_THREADS", None)
                os.environ.pop("VDJGRAPH_GLUE_REPLAY", None)

        bulk, replay, bulk1, replay1 = timed(nt, False), timed(nt, True), timed(1, False), timed(1, True)
        per = 1e3 / max(1, gs.n_nodes)
        out.update({"nodes_sample": gs.n_nodes, "threads": nt, "ms_sample": bulk, "us_per_node": bulk * per,
                    "us_per_node_replayed_inserts": replay * per,
                    "us_per_node_one_thread": bulk1 * per, "us_per_node_replayed_inserts_one_thread": replay1 * per,
                    "ms_at_this_graph": bulk * per * n_nodes * 1e-3,
                    "ms_at_this_graph_replayed_inserts": replay * per * n_nodes * 1e-3,
                    "note": "vdjgraph_rebuild_nodes on the sample's graph (scales with the node count): node pool, `nodes` map "
                            "bulk-loaded through sparsehash's unserialize from the exported layout, edge lists, on `threads` "
                            "threads (--t); `replayed_inserts` = the round-1 way (one sparsehash insert per node on one thread "
                            "while the others build flags and lists)"})
    except Exception as e:   # noqa: BLE001
        out["unavailable"] = str(e)[:200]
    return out


def bind_to_gpu_numa_node(index: int):
    """N ranks on one host: run this rank (generator threads, first touch of its record buffers, staging)
    on the cores of the NUMA node its GPU hangs off, so that the page-locked records are DMAed from local
    memory.  Returns a note for the line's config, or None when the topology is not exposed."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:      # nvml pads the domain to 8 hex digits, sysfs uses 4
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return f"rank bound to NUMA node {node} of its GPU ({len(cpus)} cores)"
    except Exception:   # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--pairs", type=int, default=0, help="override the workload's pair count (debug)")
    ap.add_argument("--pageable", action="store_true",
                    help="leave the record buffers pageable (the reference's calloc): staging bounces them through page-locked chunks")
    ap.add_argument("--forward-sharded", action="store_true", help="(accepted for old command lines; the forward-reads path is always measured)")
    ap.add_argument("--forward-inputs", action="store_true",
                    help="generate forward reads only (half the host memory: configs[4] at full size) and run everything, "
                         "`e2e` included, through vdjgraph_*_forward; the doubled text is never materialised")
    ap.add_argument("--no-forward", action="store_true", help="skip the forward-reads-only end-to-end measurement")
    ap.add_argument("--rounds", type=int, default=0, help="rounds over groups of hash units (0 = auto: 1 unless the working set exceeds HBM)")
    ap.add_argument("--cpu-sample-pairs", type=int, default=1_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the graph of the last step as DIR/<array>.npy (float64; "
                         "a fixed, seeded sample of the nodes when it exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    from vdjer_b200 import synth
    wl = dict(synth.CONFIGS[args.workload])
    if args.pairs:
        wl["n_pairs"] = args.pairs
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, wl, rank)
        return

    import torch
    import torch.distributed as dist
    from vdjer_b200 import GraphBuilder
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU path")
    torch.cuda.set_device(local_rank)
    numa_note = None
    if world > 1:
        numa_note = bind_to_gpu_numa_node(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    L, k, mf, mq = wl["read_length"], wl["k"], wl["mf"], wl["mq"]
    gen = {kk: v for kk, v in wl.items() if kk not in ("k", "mf", "mq")}
    t0 = time.perf_counter()
    # N > 1: ONE repertoire (same seed = same clone library), every rank draws its own disjoint
    # n_pairs reads from it: the pooled repertoire of BASELINE configs[4], sequenced N times deeper
    fwd_in = bool(args.forward_inputs)
    primary, secondary = synth.generate(seed=12345, pair_offset=rank * wl["n_pairs"], forward_only=fwd_in, **gen)
    t_gen = time.perf_counter() - t0
    # The record buffers are page-locked once, outside every timed region: a caller that allocates
    # them with vdjgraph_host_alloc (INTEGRATION.md section 3) has them page-locked from the start.
    from vdjer_b200 import PinnedRecords
    pinned = None if args.pageable else PinnedRecords(primary, secondary)

    # staging threads: all cores for one rank; N ranks on one host share them
    host_threads = 0 if world == 1 else max(2, len(os.sched_getaffinity(0)) // (1 if numa_note else world))
    if os.environ.get("VDJGRAPH_HOST_THREADS"):
        host_threads = int(os.environ["VDJGRAPH_HOST_THREADS"])
    gb = GraphBuilder(L, k, mf, mq, device=local_rank, host_threads=host_threads, rounds=args.rounds)
    sharded = world > 1
    if sharded:
        # one graph over the reads of all ranks: k-mers hash-sharded by minimizer, runs exchanged by the scatter
        # kernel through peer-mapped memory, every rank finishes its own survivors and stores the node rows into
        # rank 0's result buffer (vdjer_b200/shard.py)
        from vdjer_b200 import shard
        db = shard.DistributedBuilder(gb, dist, device=f"cuda:{local_rank}")   # small exchanges ride NCCL
        stage, run = (lambda: db.stage(primary, secondary, forward=fwd_in)), db.run
        build = lambda: db.build(primary, secondary, copy=False, forward=fwd_in)  # noqa: E731
    elif fwd_in:
        stage, run = (lambda: gb.stage_forward(primary, secondary)), gb.run
        build = lambda: gb.build_forward(primary, secondary, copy=False)  # noqa: E731
    else:
        stage, run = (lambda: gb.stage(primary, secondary)), gb.run
        build = lambda: gb.build(primary, secondary, copy=False)  # noqa: E731
    # ---- device-resident metric ------------------------------------------------------------
    stage()
    for _ in range(args.warmup):
        run()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    dev_ms, per_kernel = [], []
    for _ in range(args.steps):
        run()
        g = gb.fetch_stats()
        dev_ms.append(g["ms_device"])
        per_kernel.append(g)
    barrier()
    wall_dev = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    # the graph of the last timed step (rank 0), copied out before the checks below restage the builder
    last_graph = (db.fetch() if sharded else gb.fetch()) if args.dump_outputs else None
    stats = per_kernel[-1]
    phase_ms = dict(db.phase_ms) if sharded else None
    W = stats["n_windows"]
    # one device: CUDA events on the library's stream.  Sharded: a step spans several devices and
    # the host exchanges between its phases, so it is timed between barriers (device-synchronised)
    ms_dev = wall_dev * 1e3 if sharded else float(np.mean(dev_ms))

    # ---- multi-GPU: is the sharded graph the single-GPU graph?  (small seeded case, every run) ----
    parity = None
    if sharded:
        parity = shard_parity_check(torch, dist, db, local_rank, rank, world)

    # ---- end to end through the C ABI on host buffers ------------------------------------------
    # `e2e` is the path INTEGRATION.md 3c makes the default: add_to_buffer hands every read over once
    # (forward reads only, vdjgraph_build_forward), the reverse-complement records are derived on the
    # device.  The doubled text of the unmodified bam_read.c is measured beside it (`e2e_text_records`).
    def timed(build_fn):
        for _ in range(min(args.warmup, 2)):
            build_fn()
        barrier()
        t0 = time.perf_counter()
        g = None
        for _ in range(args.steps):
            g = build_fn()   # the C caller's view: result arrays in pinned host memory
            if g is not None:
                chk = int(g.frequency[:: max(1, g.n_nodes // 1024)].sum())   # the result is read on the host
        barrier()
        ms = (time.perf_counter() - t0) / args.steps * 1e3
        st = gb.fetch_stats()
        if g is not None:
            st.update(g.stats)
        return ms, st, g, (chk if g is not None else None)

    digest = None
    ms_txt, txt_stats = None, None
    if fwd_in:
        ms_e2e, e2e_stats, graph, checksum = timed(build)
    else:
        ms_txt, txt_stats, graph, checksum = timed(build)
        if world == 1 and not args.pairs:
            digest = digest_check(args.workload, graph)      # the timed workload is the one pinned against the reference
        if args.no_forward:
            ms_e2e, e2e_stats, ms_txt, txt_stats = ms_txt, txt_stats, None, None
        else:
            from vdjer_b200 import forward_reads
            fp, fs = forward_reads(primary, L), forward_reads(secondary, L)      # what a producer appending each read once holds
            pinned_f = None if args.pageable else PinnedRecords(fp, fs)
            build_f = (lambda: db.build(fp, fs, copy=False, forward=True)) if sharded else (lambda: gb.build_forward(fp, fs, copy=False))  # noqa: E731
            ms_e2e, e2e_stats, g2, checksum_f = timed(build_f)
            if g2 is not None and (g2.n_nodes != graph.n_nodes or checksum_f != checksum):
                raise SystemExit("forward-reads build differs from the build on the doubled buffers")
            if pinned_f is not None:
                pinned_f.close()
            del fp, fs
    fwd_used = fwd_in or not args.no_forward

    # max over ranks of the times, sums of the counters
    sums = {}
    if sharded:
        t = torch.tensor([ms_dev, ms_e2e, ms_txt or 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
        ms_txt = float(t[2]) if ms_txt is not None else None
        names = ["n_windows", "n_hits", "n_gated", "n_pre_total", "n_slow1", "n_slow2", "n_hits_ungated", "kernel_launches", "n_runs", "h2d_bytes"]
        t = torch.tensor([float(stats[n]) for n in names[:-1]] + [float(e2e_stats["h2d_bytes"])], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        sums = {n: float(v) for n, v in zip(names, t)}
        W_total = sums["n_windows"]
    else:
        W_total = float(W)

    if rank == 0:
        peak, peak_src = peaks()
        h = (sums["n_hits"] / W_total) if sharded else stats["n_hits"] / W
        gated = (sums["n_gated"] / W_total) if sharded else stats["n_gated"] / W
        h_u = (sums["n_hits_ungated"] / W_total) if sharded else stats["n_hits_ungated"] / W
        a1, a2, a_all = algorithmic_bytes(L, k, h, gated, h_u)
        s1, s2, s_all = algorithmic_bytes(L, k, h)
        kern = {n: float(np.mean([s[n] for s in per_kernel])) for n in
                ["ms_estimate", "ms_scatter", "ms_init1", "ms_pass1", "ms_prune", "ms_table2", "ms_pass2", "ms_export"]}
        dom = "k_pass1" if kern["ms_pass1"] >= kern["ms_pass2"] else "k_pass2"
        dom_ms = max(kern["ms_pass1"], kern["ms_pass2"])
        dom_bytes = W * (a1 if dom == "k_pass1" else a2)
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
        survey_achieved = W * (s1 if dom == "k_pass1" else s2) / (dom_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": W_total / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
            "config": {"workload": args.workload, "read_length": L, "k": k, "mf": mf, "mq": mq,
                       "pairs_per_gpu": wl["n_pairs"], "records_per_gpu": stats["n_records"], "windows_per_gpu": W,
                       "l2_policy": "inputs_larger_than_L2 (packed reads + tables >> 126 MB, tables re-initialised every step)",
                       "parallelism": (f"one graph over {world} GPUs: k-mers hash-sharded by minimizer (hash units dealt to GPUs by measured load), "
                                       "scatter kernel writes runs into the owner's peer-mapped buffer, every GPU ranks and links its own survivors "
                                       "(peer loads for neighbours owned elsewhere, device-side barriers) and stores the node rows into rank 0's result buffer; "
                                       "step timed between barriers") if sharded else "1 GPU",
                       "distinct_gated_kmers": int(sums["n_pre_total"]) if sharded else stats["n_pre_total"],
                       "nodes": stats["n_nodes"],
                       "gated_fraction": (sums["n_gated"] / W_total) if sharded else stats["n_gated"] / W, "pass2_hit_fraction_h": h,
                       "pass2_ungated_hit_fraction": h_u,
                       "table1_slots": stats["table1_slots"], "table2_slots": stats["table2_slots"],
                       "hash_partitions": stats["partitions"], "rounds": stats["rounds"],
                       "exchange_unit": "run = consecutive N-free windows of a read that share a minimizer bucket (m=10), one 32-byte record",
                       "runs": int(sums["n_runs"]) if sharded else stats["n_runs"],
                       "windows_per_run": W_total / max(1.0, sums["n_runs"] if sharded else stats["n_runs"]),
                       "run_bytes_per_window": stats["run_bytes"] * (sums["n_runs"] if sharded else stats["n_runs"]) / W_total,
                       "window_histogram": "k_count (runs / windows per minimizer bucket + HyperLogLog registers: what the plan needs) runs "
                                           "chunk by chunk behind k_pack while the reads are staged, once per read set; it is part "
                                           "of `e2e` (inside ms_stage), not of a device-resident step",
                       "slow_path_fraction_pass1": stats["n_slow1"] / max(1, stats["n_gated"]),
                       "slow_path_fraction_pass2": stats["n_slow2"] / max(1, W),
                       "generator_s": round(t_gen, 2),
                       **({"host_binding": numa_note} if numa_note else {}),
                       **({"weak_scaling_note": "every rank draws its own reads from the SAME clone library (one pooled repertoire sequenced "
                                                "N times deeper): distinct k-mers grow more slowly than windows"} if sharded else {})},
            "e2e": {"value": W_total / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(sums["h2d_bytes"]) if sharded else e2e_stats["h2d_bytes"],
                    "d2h_bytes_per_step": e2e_stats["d2h_bytes"],
                    "ms_stage": e2e_stats["ms_stage"], "ms_device": e2e_stats["ms_device"], "ms_fetch": e2e_stats["ms_fetch"],
                    "inputs": ("forward reads only, every read handed over once (vdjgraph_build_forward, the default of the "
                               "INTEGRATION.md 3c glue): the reverse-complement records are derived on the device; same graph, "
                               "checked against the doubled-text build in this run"
                               if fwd_used else "the reference's record buffers (every read and its reverse complement)"),
                    "host_buffers": "pageable, bounced through page-locked chunks by host threads" if args.pageable else
                                    "page-locked (vdjgraph_host_register once, untimed): staging DMAs straight from the caller's records"},
            "gpu_launches": int(sums["kernel_launches"] if sharded else stats["kernel_launches"]) * args.steps,
            "kernel_ms": kern, "wall_ms_per_step_device_loop": wall_dev * 1e3,
            "roofline": {"bound": "hbm", "limiter": "scattered 32-byte sector requests into the L2-resident table slice (latency / L1 request "
                                                     "rate), not DRAM bandwidth: see profiles/ncu_r2_summary.json",
                         "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": ncu_traffic(dom) if (args.workload == DEFAULT_WORKLOAD and not args.pairs and not sharded) else None,
                         "traffic_source": NCU_SUMMARY + " (ncu --set full, same workload, one launch; regenerated each round by profiles/prof_r2.sh)",
                         "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
                         "survey_formula": {"achieved": survey_achieved, "frac": survey_achieved / peak,
                                            "algorithmic_bytes_per_window": s1 if dom == "k_pass1" else s2},
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_window": a1 if dom == "k_pass1" else a2,
                         "windows_per_launch": W},
            "roofline_path": {"algorithmic_bytes_per_window": a_all, "achieved": W_total * a_all / (ms_dev * 1e-3) / 1e9 / world,
                              "frac": W_total * a_all / (ms_dev * 1e-3) / 1e9 / world / peak,
                              "survey_formula": {"algorithmic_bytes_per_window": s_all,
                                                 "frac": W_total * s_all / (ms_dev * 1e-3) / 1e9 / world / peak},
                              "note": "whole step (all kernels) per GPU against the HBM copy peak"},
            "clocks": clocks,
        }
        ar = atomic_rates()
        if ar:
            # SURVEY 8d "atomic roof": pass 1 = one L2 load + RED per gated window; pass 2 = one L2 load per
            # N-free window + one RED per ungated hit.  Rates: random sectors in an L2-resident table.
            n_g = gated * W
            t1 = n_g / (ar["load_red"] * 1e9) * 1e3
            n_valid = W   # N-free windows ~ all windows (N rate 0.05 %)
            t2 = (n_valid / (ar["load"] * 1e9) + h_u * W / (ar["red"] * 1e9)) * 1e3
            line["roofline_atomic"] = {
                "source": "profiles/microbench_r1.json (random 32-B sectors, 32 MB table: L2-resident)",
                "rates_G_ops_per_s": ar,
                "k_pass1": {"roof_ms": t1, "measured_ms": kern["ms_pass1"], "frac": t1 / kern["ms_pass1"]},
                "k_pass2": {"roof_ms": t2, "measured_ms": kern["ms_pass2"], "frac": t2 / kern["ms_pass2"]},
            }
        if ms_txt is not None:
            line["e2e_text_records"] = {
                "value": W_total / (ms_txt * 1e-3), "unit": UNIT, "ms_per_step": ms_txt,
                "h2d_bytes_per_step": (int(sums["h2d_bytes"]) * 2) if sharded else txt_stats["h2d_bytes"],
                "d2h_bytes_per_step": txt_stats["d2h_bytes"],
                "ms_stage": txt_stats["ms_stage"], "ms_device": txt_stats["ms_device"], "ms_fetch": txt_stats["ms_fetch"],
                "note": "vdjgraph_build on the unmodified bam_read.c buffers (every read followed by its reverse complement: "
                        "twice the host-to-device bytes for the same graph)"}
        if digest is not None:
            line["digest_check"] = digest
        if parity is not None:
            line["parity_check"] = parity
        if sharded:
            line["shard_phase_ms_rank0"] = {k2: round(v, 3) for k2, v in phase_ms.items()}
        if not args.no_cpu_baseline:
            cb = cpu_baseline(wl, args.cpu_sample_pairs, extras=True)
            line["cpu_baseline"] = {k2: v for k2, v in cb.items() if not k2.startswith("_")}
            if not sharded:
                gr = glue_cost(args, wl, cb, local_rank, primary, secondary, fwd_in, stats["n_nodes"])
                if gr:
                    # the drop-in cost as V'DJer sees it: the library call (with the layout of the reference's
                    # `nodes` map computed on the device) plus the reference-side rebuild of ITS structures
                    line["cpu_baseline"]["glue_rebuild"] = gr
                    if "ms_at_this_graph" in gr:
                        line["e2e"]["ms_with_glue_rebuild"] = gr["e2e_ms_with_layout"] + gr["ms_at_this_graph"]
        if last_graph is not None:
            line["outputs_dumped"] = dump_outputs(args.dump_outputs, last_graph)
        print(json.dumps(line), flush=True)
    if world > 1:
        db.close()
    gb.close()
    if pinned is not None:
        pinned.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
