"""vdjer_b200 -- B200-native de Bruijn graph build for V'DJer.

Host-side Python mirror of the C ABI in include/vdjgraph.h (ctypes over the in-tree
libvdjgraph.so).  The library replaces the block assembler2_vdj.c:1381-1415 of the reference
(build_pre_graph x2 -> prune_pre_graph -> build_graph2 x2); there is no CPU fallback here:
importing works anywhere, but creating a GraphBuilder without the CUDA library or a B200 raises.
"""
from .graph import GraphBuilder, MultiBuilder, Graph, PinnedRecords, PreTable, VdjGraphError, forward_reads, host_alloc, host_free, lib_path, NIL, query_batch, window_counts  # noqa: F401
from . import synth  # noqa: F401

__all__ = ["GraphBuilder", "MultiBuilder", "Graph", "PinnedRecords", "PreTable", "VdjGraphError", "forward_reads", "host_alloc", "host_free", "lib_path", "NIL", "query_batch", "window_counts", "synth"]
