"""Sequential model of vdjgraph_query for the tests: an index from packed k-mer to node, built from a
graph's node k-mers, and the answer of every window of a batch of queries."""
from __future__ import annotations

import numpy as np

from tests.util import kmer_codes_at, pack_codes
from vdjer_b200.graph import NIL, query_batch, window_counts

_KEY = np.dtype([("hi", "<u8"), ("lo", "<u8")])
_CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i


class NodeIndex:
    """Node i is the node whose packed k-mer is (lo[i], hi[i]) (the library's key layout)."""

    def __init__(self, lo, hi):
        keys = np.empty(len(lo), _KEY)
        keys["lo"], keys["hi"] = lo, hi
        self.order = np.argsort(keys, kind="stable")
        self.keys = keys[self.order]

    @classmethod
    def from_graph(cls, graph: dict, primary, secondary, L: int, k: int) -> "NodeIndex":
        """From an oracle or golden graph: the node k-mers are the bases at their first positions."""
        return cls(*pack_codes(kmer_codes_at(primary, secondary, L, k, graph["first_pos"])))

    def lookup(self, lo, hi) -> np.ndarray:
        q = np.empty(len(lo), _KEY)
        q["lo"], q["hi"] = lo, hi
        if len(self.keys) == 0:
            return np.full(len(q), NIL, np.uint32)
        pos = np.minimum(np.searchsorted(self.keys, q), len(self.keys) - 1)
        return np.where(self.keys[pos] == q, self.order[pos], NIL).astype(np.uint32)


def decode_kmers(lo, hi, k: int) -> list[bytes]:
    """Packed k-mers back to their bases."""
    lo = np.asarray(lo, np.uint64)
    hi = np.asarray(hi, np.uint64)
    codes = np.empty((len(lo), k), np.uint8)
    for j in range(k):
        word, bit = (lo, 2 * j) if j < 32 else (hi, 2 * (j - 32))
        codes[:, j] = (word >> np.uint64(bit)) & np.uint64(3)
    text = np.frombuffer(b"ACGT", np.uint8)[codes]
    return [row.tobytes() for row in text]


def window_starts(offsets, k: int) -> np.ndarray:
    """Byte position in the batch of every window, in query order."""
    offsets = np.asarray(offsets, np.uint64).astype(np.int64)
    counts = window_counts(offsets, k)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    return np.repeat(offsets[:-1], counts) + (np.arange(int(counts.sum())) - np.repeat(first, counts))


def answers_at(text, starts, k: int, index: NodeIndex) -> np.ndarray:
    """The answer of the windows that start at the given bytes of the batch: the node of the window's k-mer,
    or NIL when the window holds a byte other than ACGT or its k-mer is not a node."""
    text = np.asarray(text, np.uint8)
    starts = np.asarray(starts, np.int64)
    if len(starts) == 0:
        return np.zeros(0, np.uint32)
    codes = _CODE[text[starts[:, None] + np.arange(k)[None, :]]]
    has_n = (codes == 255).any(axis=1)
    lo, hi = pack_codes(np.where(codes == 255, 0, codes))
    out = index.lookup(lo, hi)
    out[has_n] = NIL
    return out


def answers_flat(text, offsets, k: int, index: NodeIndex) -> np.ndarray:
    """The answer of every window of the batch, in query order."""
    return answers_at(text, window_starts(offsets, k), k, index)


def answers(seqs, k: int, index: NodeIndex) -> list[np.ndarray]:
    text, offsets = query_batch(seqs)
    ends = np.cumsum(window_counts(offsets, k))
    return np.split(answers_flat(text, offsets, k, index), ends[:-1]) if len(seqs) else []
