"""ctypes binding of include/vdjgraph.h.

Names follow the reference's stage (assembler2_vdj.c): `primary` is assemble()'s `input`,
`secondary` its `unaligned_input`; k / mf / mq are --k / --mf / --mq (params.c:53-73 defaults:
35 / 3 / 90).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path() -> str:
    # VDJGRAPH_LIB: another build of the same library (tuning experiments, profiles/variants.sh)
    return os.environ.get("VDJGRAPH_LIB") or os.path.join(_HERE, "libvdjgraph.so")


class VdjGraphError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"vdjgraph error {code}: {msg}")
        self.code = code


class _Params(C.Structure):
    _fields_ = [
        ("read_length", C.c_int32), ("kmer_size", C.c_int32), ("min_node_freq", C.c_int32),
        ("min_base_quality", C.c_int32), ("device", C.c_int32), ("host_threads", C.c_int32),
        ("table_capacity", C.c_uint64), ("flags", C.c_uint32), ("partitions", C.c_uint32),
        ("rounds", C.c_uint32), ("reserved", C.c_uint32),
    ]


class _Result(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_uint64),
        ("first_pos", C.POINTER(C.c_uint64)), ("frequency", C.POINTER(C.c_uint16)),
        ("out_deg", C.POINTER(C.c_uint8)), ("in_deg", C.POINTER(C.c_uint8)),
        ("out_succ", C.POINTER(C.c_uint32)), ("in_pred", C.POINTER(C.c_uint32)),
        ("kmer_lo", C.POINTER(C.c_uint64)), ("kmer_hi", C.POINTER(C.c_uint64)),
        ("n_records", C.c_uint64), ("n_windows", C.c_uint64), ("n_gated", C.c_uint64),
        ("n_pre_total", C.c_uint64), ("n_pre", C.c_uint64), ("n_hits", C.c_uint64),
        ("n_slow1", C.c_uint64), ("n_slow2", C.c_uint64), ("n_hits_ungated", C.c_uint64),
        ("ms_stage", C.c_float), ("ms_device", C.c_float), ("ms_estimate", C.c_float),
        ("ms_scatter", C.c_float), ("ms_init1", C.c_float), ("ms_pass1", C.c_float), ("ms_prune", C.c_float), ("ms_table2", C.c_float),
        ("ms_pass2", C.c_float), ("ms_export", C.c_float), ("ms_fetch", C.c_float),
        ("table1_slots", C.c_uint64), ("table2_slots", C.c_uint64),
        ("partitions", C.c_uint32), ("tuple_bytes", C.c_uint32), ("rounds", C.c_uint32), ("reserved", C.c_uint32),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("n_runs", C.c_uint64), ("run_bytes", C.c_uint32), ("reserved2", C.c_uint32),
        ("hm_buckets", C.c_uint64), ("hm_slots", C.POINTER(C.c_uint32)), ("ms_hashmap", C.c_float), ("reserved3", C.c_float),
    ]


class _QueryStats(C.Structure):
    _fields_ = [("n_queries", C.c_uint64), ("n_windows", C.c_uint64), ("n_found", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("ms_kernels", C.c_float), ("ms_total", C.c_float)]


class _PreTable(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer_lo", C.POINTER(C.c_uint64)),
                ("kmer_hi", C.POINTER(C.c_uint64)), ("frequency", C.POINTER(C.c_uint16))]


FLAG_EXPORT_KEYS = 1
FLAG_WIDE_TUPLES = 2
FLAG_HASHMAP_LAYOUT = 4

EXPORTS = [
    "vdjgraph_version", "vdjgraph_last_error", "vdjgraph_create", "vdjgraph_destroy",
    "vdjgraph_set_params", "vdjgraph_build", "vdjgraph_stage", "vdjgraph_run", "vdjgraph_fetch",
    "vdjgraph_stage_forward", "vdjgraph_build_forward",
    "vdjgraph_fetch_pre_table", "vdjgraph_stats", "vdjgraph_query",
    "vdjgraph_host_alloc", "vdjgraph_host_free", "vdjgraph_host_register", "vdjgraph_host_unregister",
    "vdjgraph_shard_stage", "vdjgraph_shard_stage_forward", "vdjgraph_shard_count", "vdjgraph_shard_plan", "vdjgraph_shard_rounds", "vdjgraph_shard_buffers",
    "vdjgraph_shard_set_peers", "vdjgraph_shard_scatter", "vdjgraph_shard_passes", "vdjgraph_shard_gather_plan",
    "vdjgraph_shard_finish_bytes", "vdjgraph_shard_finish_step", "vdjgraph_shard_finish", "vdjgraph_shard_release_retired", "vdjgraph_ipc_export", "vdjgraph_ipc_open",
    "vdjgraph_ipc_close", "vdjgraph_enable_peer_access",
    "vdjgraph_multi_create", "vdjgraph_multi_destroy", "vdjgraph_multi_build", "vdjgraph_multi_build_forward", "vdjgraph_multi_stats",
]

SHARD_NBUF, SHARD_HIST, SHARD_HLL = 6, 768, 32768   # buffers; uint64 counts; uint8 registers
BUF_GATHER = 5


class _ShardInfo(C.Structure):
    _fields_ = [("n_ranks", C.c_uint32), ("rank", C.c_uint32), ("record_base", C.c_uint64), ("total_records", C.c_uint64)]

_lib = None


def load_library():
    """Load libvdjgraph.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise VdjGraphError(-5, f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(make -C vdjer_b200/csrc); there is no CPU fallback")
    lib = C.CDLL(path)
    lib.vdjgraph_version.restype = C.c_int
    lib.vdjgraph_last_error.restype = C.c_char_p
    lib.vdjgraph_create.argtypes = [C.POINTER(_Params), C.POINTER(C.c_void_p)]
    lib.vdjgraph_destroy.argtypes = [C.c_void_p]
    lib.vdjgraph_destroy.restype = None
    lib.vdjgraph_set_params.argtypes = [C.c_void_p, C.POINTER(_Params)]
    lib.vdjgraph_build.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(_Result)]
    lib.vdjgraph_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    lib.vdjgraph_build_forward.argtypes = lib.vdjgraph_build.argtypes
    lib.vdjgraph_stage_forward.argtypes = lib.vdjgraph_stage.argtypes
    lib.vdjgraph_run.argtypes = [C.c_void_p]
    lib.vdjgraph_fetch.argtypes = [C.c_void_p, C.POINTER(_Result)]
    lib.vdjgraph_stats.argtypes = [C.c_void_p, C.POINTER(_Result)]
    lib.vdjgraph_fetch_pre_table.argtypes = [C.c_void_p, C.POINTER(_PreTable)]
    lib.vdjgraph_query.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(_QueryStats)]
    lib.vdjgraph_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    lib.vdjgraph_host_free.argtypes = [C.c_void_p]
    lib.vdjgraph_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.vdjgraph_host_unregister.argtypes = [C.c_void_p]
    lib.vdjgraph_shard_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(_ShardInfo)]
    lib.vdjgraph_shard_stage_forward.argtypes = lib.vdjgraph_shard_stage.argtypes
    lib.vdjgraph_shard_count.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.vdjgraph_shard_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.vdjgraph_shard_rounds.argtypes = [C.c_void_p]
    lib.vdjgraph_shard_buffers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    lib.vdjgraph_shard_set_peers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.vdjgraph_shard_scatter.argtypes = [C.c_void_p]
    lib.vdjgraph_shard_passes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.vdjgraph_shard_gather_plan.argtypes = [C.c_void_p, C.c_void_p]
    lib.vdjgraph_shard_finish_bytes.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.vdjgraph_shard_finish_step.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.vdjgraph_shard_finish.argtypes = [C.c_void_p]
    lib.vdjgraph_shard_release_retired.argtypes = [C.c_void_p]
    lib.vdjgraph_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.vdjgraph_ipc_open.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.vdjgraph_ipc_close.argtypes = [C.c_void_p]
    lib.vdjgraph_enable_peer_access.argtypes = [C.c_int, C.c_int]
    lib.vdjgraph_multi_create.argtypes = [C.POINTER(_Params), C.POINTER(C.c_int), C.c_uint32, C.POINTER(C.c_void_p)]
    lib.vdjgraph_multi_destroy.argtypes = [C.c_void_p]
    lib.vdjgraph_multi_destroy.restype = None
    lib.vdjgraph_multi_build.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(_Result)]
    lib.vdjgraph_multi_build_forward.argtypes = lib.vdjgraph_multi_build.argtypes
    lib.vdjgraph_multi_stats.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_Result)]
    _lib = lib
    return lib


def _as_u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        a = buf
        if a.dtype != np.uint8:
            a = a.view(np.uint8)
        return np.ascontiguousarray(a)
    return np.frombuffer(buf, dtype=np.uint8)


class PinnedRecords:
    """Page-locks record buffers for as long as it lives (vdjgraph_host_register): staging then DMAs
    straight out of them, as it does from buffers a C caller takes from vdjgraph_host_alloc."""

    def __init__(self, *arrays):
        self._lib = load_library()
        self._held = []
        for a in arrays:
            a = _as_u8(a)
            if a.size == 0:
                continue
            rc = self._lib.vdjgraph_host_register(a.ctypes.data, a.size)
            if rc != 0:
                self.close()
                raise VdjGraphError(rc, (self._lib.vdjgraph_last_error() or b"").decode())
            self._held.append(a)

    def close(self):
        for a in self._held:
            self._lib.vdjgraph_host_unregister(a.ctypes.data)
        self._held = []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def forward_reads(records, read_length: int) -> np.ndarray:
    """The even records (the reads themselves) of a reference-format buffer in which every read is
    followed by its reverse complement (bam_read.c:206-244): what a producer that appends each read
    once would hand to vdjgraph_stage_forward.  NUL-terminated like the input."""
    rb = 2 * read_length + 1
    a = _as_u8(records)
    n = a.size // rb
    if n % 2:
        raise ValueError("odd number of records: not a read / reverse-complement buffer")
    fwd = a[: n * rb].reshape(n // 2, 2 * rb)[:, :rb]
    return np.concatenate([fwd.reshape(-1), np.zeros(1, np.uint8)])


def host_alloc(n_bytes: int) -> np.ndarray:
    """uint8 array in page-locked memory from vdjgraph_host_alloc (freed with host_free)."""
    lib = load_library()
    p = C.c_void_p()
    rc = lib.vdjgraph_host_alloc(n_bytes, C.byref(p))
    if rc != 0:
        raise VdjGraphError(rc, (lib.vdjgraph_last_error() or b"").decode())
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n_bytes, 1),))[:n_bytes]


def host_free(a: np.ndarray):
    load_library().vdjgraph_host_free(C.c_void_p(a.ctypes.data))


NIL = 0xFFFFFFFF   # vdjgraph_query's answer for a window with an N or whose k-mer is not a node


def query_batch(seqs) -> tuple[np.ndarray, np.ndarray]:
    """Sequences (bytes or str) -> (text, offsets): one uint8 array of all their bytes and uint64 offsets [n+1];
    query i is text[offsets[i]:offsets[i+1]], the form vdjgraph_query takes."""
    bs = [s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs]
    offsets = np.zeros(len(bs) + 1, np.uint64)
    np.cumsum(np.fromiter((len(b) for b in bs), np.uint64, count=len(bs)), out=offsets[1:])
    return np.frombuffer(b"".join(bs), np.uint8), offsets


def window_counts(offsets, k: int) -> np.ndarray:
    """Windows of every query: max(0, len - k + 1)."""
    lens = np.diff(np.asarray(offsets, np.uint64).astype(np.int64))
    return np.maximum(lens - (k - 1), 0)


@dataclass
class Graph:
    """The graph after build_graph2 (:1408): node i is the node with reference id i+1."""
    n_nodes: int
    first_pos: np.ndarray   # u64 [n]  r*w + o of node->kmer
    frequency: np.ndarray   # u16 [n]
    out_deg: np.ndarray     # u8  [n]
    in_deg: np.ndarray      # u8  [n]
    out_succ: np.ndarray    # u32 [n,4] toNodes, list order
    in_pred: np.ndarray     # u32 [n,4] fromNodes, list order
    kmer_lo: np.ndarray | None
    kmer_hi: np.ndarray | None
    stats: dict = field(default_factory=dict)
    hm_slots: np.ndarray | None = None   # u32 [hm_buckets]: node per bucket of the reference's `nodes` map (hashmap_layout=True)


@dataclass
class PreTable:
    """pre_nodes after prune_pre_graph (:1393), unordered."""
    kmer_lo: np.ndarray
    kmer_hi: np.ndarray
    frequency: np.ndarray


def _np_from(ptr, n, dtype, cols=1, copy=True):
    if n == 0 or not ptr:
        shape = (0, cols) if cols > 1 else (0,)
        return np.zeros(shape, dtype=dtype)
    a = np.ctypeslib.as_array(ptr, shape=(n * cols,))
    if copy:
        a = a.copy()
    return a.reshape(n, cols) if cols > 1 else a


class GraphBuilder:
    """One libvdjgraph context (CUDA context, streams, staging buffers) reused across builds."""

    def __init__(self, read_length: int, k: int = 35, mf: int = 3, mq: int = 90, device: int = -1,
                 host_threads: int = 0, table_capacity: int = 0, export_keys: bool = False,
                 partitions: int = 0, wide_tuples: bool = False, rounds: int = 0, hashmap_layout: bool = False):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        self._p = _Params(read_length, k, mf, mq, device, host_threads, table_capacity,
                          (FLAG_EXPORT_KEYS if export_keys else 0) | (FLAG_WIDE_TUPLES if wide_tuples else 0) |
                          (FLAG_HASHMAP_LAYOUT if hashmap_layout else 0),
                          partitions, rounds, 0)
        self._check(self._lib.vdjgraph_create(C.byref(self._p), C.byref(self._ctx)))
        self._keep = None

    def _check(self, rc: int):
        if rc != 0:
            raise VdjGraphError(rc, (self._lib.vdjgraph_last_error() or b"").decode())

    def close(self):
        if self._ctx:
            self._lib.vdjgraph_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_params(self, read_length=None, k=None, mf=None, mq=None):
        if read_length is not None:
            self._p.read_length = read_length
        if k is not None:
            self._p.kmer_size = k
        if mf is not None:
            self._p.min_node_freq = mf
        if mq is not None:
            self._p.min_base_quality = mq
        self._check(self._lib.vdjgraph_set_params(self._ctx, C.byref(self._p)))

    def _counts(self, primary, secondary):
        rec = 2 * self._p.read_length + 1
        p, s = _as_u8(primary), _as_u8(secondary)
        # a trailing NUL (the reference's buffers are C strings) is not a record
        return p, s, p.size // rec, s.size // rec

    def _n_records(self, primary, secondary) -> int:
        _, _, n_p, n_s = self._counts(primary, secondary)
        return n_p + n_s

    def stage(self, primary, secondary=b""):
        p, s, n_p, n_s = self._counts(primary, secondary)
        self._keep = (p, s)
        self._check(self._lib.vdjgraph_stage(self._ctx, p.ctypes.data, n_p, s.ctypes.data, n_s))

    def run(self):
        self._check(self._lib.vdjgraph_run(self._ctx))

    def fetch(self, copy: bool = True) -> Graph:
        r = _Result()
        self._check(self._lib.vdjgraph_fetch(self._ctx, C.byref(r)))
        return self._graph(r, copy)

    def fetch_stats(self) -> dict:
        """Counters and timings of the last run() without the device-to-host copy of the graph."""
        r = _Result()
        self._check(self._lib.vdjgraph_stats(self._ctx, C.byref(r)))
        return self._stats(r)

    def build(self, primary, secondary=b"", copy: bool = True) -> Graph:
        """vdjgraph_build: HOST buffers in, graph out (stage + run + fetch).

        copy=False returns views of the library's page-locked result arrays, exactly what a C
        caller gets: valid until the next stage/build/close on this builder."""
        p, s, n_p, n_s = self._counts(primary, secondary)
        r = _Result()
        self._check(self._lib.vdjgraph_build(self._ctx, p.ctypes.data, n_p, s.ctypes.data, n_s, C.byref(r)))
        return self._graph(r, copy)

    def stage_forward(self, primary_reads, secondary_reads=b""):
        """vdjgraph_stage_forward: buffers of FORWARD reads only (see forward_reads())."""
        p, s, n_p, n_s = self._counts(primary_reads, secondary_reads)
        self._keep = (p, s)
        self._check(self._lib.vdjgraph_stage_forward(self._ctx, p.ctypes.data, n_p, s.ctypes.data, n_s))

    def build_forward(self, primary_reads, secondary_reads=b"", copy: bool = True) -> Graph:
        """vdjgraph_build_forward: the graph of the doubled buffers from their forward reads alone;
        the reverse-complement records are derived on the device (half the H2D bytes)."""
        p, s, n_p, n_s = self._counts(primary_reads, secondary_reads)
        r = _Result()
        self._check(self._lib.vdjgraph_build_forward(self._ctx, p.ctypes.data, n_p, s.ctypes.data, n_s, C.byref(r)))
        return self._graph(r, copy)

    # ---- sharded build phases (see include/vdjgraph.h and vdjer_b200/shard.py) -------------------
    def shard_stage(self, primary, secondary, n_ranks: int, rank: int, record_base: int, total_records: int,
                    forward: bool = False):
        """forward: the buffers hold forward reads only (forward_reads()); record_base and total_records
        stay in the doubled numbering (two records per read)."""
        p, s, n_p, n_s = self._counts(primary, secondary)
        self._keep = (p, s)
        info = _ShardInfo(n_ranks, rank, record_base, total_records)
        fn = self._lib.vdjgraph_shard_stage_forward if forward else self._lib.vdjgraph_shard_stage
        self._check(fn(self._ctx, p.ctypes.data, n_p, s.ctypes.data, n_s, C.byref(info)))

    def shard_count(self):
        hist = np.zeros(SHARD_HIST, np.uint64)
        hll = np.zeros(SHARD_HLL, np.uint8)
        self._check(self._lib.vdjgraph_shard_count(self._ctx, hist.ctypes.data, hll.ctypes.data))
        return hist, hll

    def shard_plan(self, hist_all: np.ndarray, hll_merged: np.ndarray, record_counts: np.ndarray):
        h = np.ascontiguousarray(hist_all, np.uint64)
        m = np.ascontiguousarray(hll_merged, np.uint8)
        r = np.ascontiguousarray(record_counts, np.uint64)
        self._check(self._lib.vdjgraph_shard_plan(self._ctx, h.ctypes.data, m.ctypes.data, r.ctypes.data))

    def shard_rounds(self) -> int:
        """Super-partition rounds the plan settled on (scatter + passes run once per round)."""
        n = self._lib.vdjgraph_shard_rounds(self._ctx)
        if n < 0:
            self._check(n)
        return n

    def shard_buffers(self):
        ptrs = (C.c_void_p * SHARD_NBUF)()
        sizes = (C.c_size_t * SHARD_NBUF)()
        self._check(self._lib.vdjgraph_shard_buffers(self._ctx, ptrs, sizes))
        return [int(x or 0) for x in ptrs], [int(x) for x in sizes]

    def shard_set_peers(self, table):
        """table[rank][buffer] = device pointer (ints; 0 = none)."""
        flat = (C.c_void_p * (len(table) * SHARD_NBUF))(*[C.c_void_p(p or None) for row in table for p in row])
        self._check(self._lib.vdjgraph_shard_set_peers(self._ctx, flat))

    def shard_scatter(self):
        self._check(self._lib.vdjgraph_shard_scatter(self._ctx))

    def shard_passes(self) -> int:
        n = C.c_uint64(0)
        self._check(self._lib.vdjgraph_shard_passes(self._ctx, C.byref(n)))
        return int(n.value)

    def shard_gather_plan(self, survivors_all):
        a = np.ascontiguousarray(survivors_all, np.uint64)
        self._check(self._lib.vdjgraph_shard_gather_plan(self._ctx, a.ctypes.data))

    def shard_finish_bytes(self, survivors_all, rank: int) -> int:
        """Bytes rank `rank`'s exchange buffer (BUF_GATHER) must hold for the finish of these survivor counts."""
        a = np.ascontiguousarray(survivors_all, np.uint64)
        n = C.c_size_t(0)
        self._check(self._lib.vdjgraph_shard_finish_bytes(self._ctx, a.ctypes.data, rank, C.byref(n)))
        return int(n.value)

    def shard_finish_step(self, step: int, device_barrier: bool):
        """Step 0, 1, 2 of the distributed finish.  device_barrier: the devices meet in peer memory and the call
        returns at once; otherwise it returns with the stream synchronised and the caller holds the barrier."""
        self._check(self._lib.vdjgraph_shard_finish_step(self._ctx, step, 1 if device_barrier else 0))

    def shard_finish(self):
        """Every rank, after the three steps; the graph is then on rank 0's device."""
        self._check(self._lib.vdjgraph_shard_finish(self._ctx))

    def shard_release_retired(self):
        self._check(self._lib.vdjgraph_shard_release_retired(self._ctx))

    def query(self, seqs) -> tuple[list[np.ndarray], dict]:
        """vdjgraph_query: the node (creation rank) of every k-mer window of every sequence in `seqs` (bytes or
        str over ACGTN), NIL where the window holds an N or its k-mer is not a node of the last built graph.
        Returns one uint32 view per sequence into a single flat array, and the call's counters."""
        text, offsets = query_batch(seqs)
        flat, stats = self.query_flat(text, offsets)
        ends = np.cumsum(window_counts(offsets, self._p.kmer_size))
        return (np.split(flat, ends[:-1]) if len(seqs) else []), stats

    def query_flat(self, text, offsets, out: np.ndarray | None = None, n_windows: int | None = None) -> tuple[np.ndarray, dict]:
        """vdjgraph_query on a batch already in the library's form (query_batch()): the answers of all windows in
        query order in one uint32 array (`out` when given: one page-locked by vdjgraph_host_alloc or
        PinnedRecords is written by DMA).  n_windows defaults to the exact count."""
        t = _as_u8(text)
        off = np.ascontiguousarray(offsets, np.uint64)
        if n_windows is None:
            n_windows = int(window_counts(off, self._p.kmer_size).sum())
        if out is None:
            out = np.empty(max(n_windows, 0), np.uint32)
        if out.dtype != np.uint32 or not out.flags.c_contiguous or out.size < n_windows:
            raise ValueError("out must be a contiguous uint32 array of at least n_windows elements")
        st = _QueryStats()
        self._check(self._lib.vdjgraph_query(self._ctx, t.ctypes.data, off.ctypes.data, max(off.size - 1, 0),
                                             out.ctypes.data, n_windows, C.byref(st)))
        return out, {k: (float(getattr(st, k)) if k.startswith("ms_") else int(getattr(st, k))) for k, _ in _QueryStats._fields_}

    def pre_table(self) -> PreTable:
        t = _PreTable()
        self._check(self._lib.vdjgraph_fetch_pre_table(self._ctx, C.byref(t)))
        n = int(t.n)
        return PreTable(_np_from(t.kmer_lo, n, np.uint64), _np_from(t.kmer_hi, n, np.uint64),
                        _np_from(t.frequency, n, np.uint16))

    @staticmethod
    def _stats(r: _Result) -> dict:
        return {k: (float(getattr(r, k)) if k.startswith("ms_") else int(getattr(r, k)))
                for k, _ in _Result._fields_
                if k.startswith(("n_", "ms_", "table", "h2d", "d2h", "kernel", "partitions", "tuple", "rounds", "run_bytes", "hm_buckets"))}

    def _graph(self, r: _Result, copy: bool = True) -> Graph:
        n = int(r.n_nodes)
        stats = self._stats(r)
        return Graph(
            n, _np_from(r.first_pos, n, np.uint64, 1, copy), _np_from(r.frequency, n, np.uint16, 1, copy),
            _np_from(r.out_deg, n, np.uint8, 1, copy), _np_from(r.in_deg, n, np.uint8, 1, copy),
            _np_from(r.out_succ, n, np.uint32, 4, copy), _np_from(r.in_pred, n, np.uint32, 4, copy),
            _np_from(r.kmer_lo, n, np.uint64, 1, copy) if r.kmer_lo else None,
            _np_from(r.kmer_hi, n, np.uint64, 1, copy) if r.kmer_hi else None, stats,
            _np_from(r.hm_slots, int(r.hm_buckets), np.uint32, 1, copy) if r.hm_slots else None)


class MultiBuilder:
    """One graph over several GPUs of THIS process (vdjgraph_multi_*): one context per entry of `devices`
    (1, 2, 4 or 8 ordinals; the same one may repeat, for tests on one GPU), one host thread per device inside
    every build.  The result is the one-device result; it is fetched from devices[0]."""

    def __init__(self, read_length: int, k: int = 35, mf: int = 3, mq: int = 90, devices=(0,), host_threads: int = 0,
                 export_keys: bool = False, partitions: int = 0, wide_tuples: bool = False, rounds: int = 0,
                 hashmap_layout: bool = False):
        self._lib = load_library()
        self._m = C.c_void_p()
        self.devices = [int(d) for d in devices]
        self._p = _Params(read_length, k, mf, mq, -1, host_threads, 0,
                          (FLAG_EXPORT_KEYS if export_keys else 0) | (FLAG_WIDE_TUPLES if wide_tuples else 0) |
                          (FLAG_HASHMAP_LAYOUT if hashmap_layout else 0),
                          partitions, rounds, 0)
        dev = (C.c_int * len(self.devices))(*self.devices)
        self._check(self._lib.vdjgraph_multi_create(C.byref(self._p), dev, len(self.devices), C.byref(self._m)))

    _check = GraphBuilder._check
    _counts = GraphBuilder._counts
    _graph = GraphBuilder._graph
    _stats = staticmethod(GraphBuilder._stats)

    def close(self):
        if self._m:
            self._lib.vdjgraph_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def build(self, primary, secondary=b"", copy: bool = True) -> Graph:
        p, s, n_p, n_s = self._counts(primary, secondary)
        r = _Result()
        self._check(self._lib.vdjgraph_multi_build(self._m, p.ctypes.data, n_p, s.ctypes.data, n_s, C.byref(r)))
        return self._graph(r, copy)

    def build_forward(self, primary_reads, secondary_reads=b"", copy: bool = True) -> Graph:
        p, s, n_p, n_s = self._counts(primary_reads, secondary_reads)
        r = _Result()
        self._check(self._lib.vdjgraph_multi_build_forward(self._m, p.ctypes.data, n_p, s.ctypes.data, n_s, C.byref(r)))
        return self._graph(r, copy)

    def rank_stats(self, rank: int) -> dict:
        """Counters and timings of one rank's share of the last build."""
        r = _Result()
        self._check(self._lib.vdjgraph_multi_stats(self._m, rank, C.byref(r)))
        return self._stats(r)
