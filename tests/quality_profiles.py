"""Quality profiles for the tests of the prune's quality-flag bound, and a CPU model of that bound.

synth.generate draws phred 2-19 or 30-40 only (N: 2), so on its output "phred >= 20" (the pass-1
gate, the `good` mask) and "phred >= HIQ = 30" (the `hiq` mask) are the same bit on every base, and
the flags k_prune bounds the quality sums with (LOG_A: window all >= HIQ, LOG_B: the record's first
k phreds all >= HIQ) cannot be told apart from the gate.  requantize() redraws the qualities of such
input from profiles that do separate them; flag_sensitivity() counts the k-mers whose prune decision
would change if a build derived those flags from the gate instead, i.e. how many wrong answers a
comparison with the oracle on that input would see."""
from __future__ import annotations

import numpy as np

from vdjer_b200 import synth

GATE_Q, HIQ, QSUM_SAT, N_PHRED = 20, 30, 214, 2
MAX_LOG_RANKS = 11   # ceil(214 / 20)

# the flag mutants: window        LOG_A = the window passes the gate (every logged window does)
#                   record_start  LOG_B = the record's first k bases pass the gate
#                   both          both of them (what hiq = gate in k_pack gives)
MUTANTS = ("window", "record_start", "both")

# name -> (phred values, weights); None weights = uniform
PROFILES = {
    # NovaSeq's binned qualities 2 / 12 / 23 / 37
    "novaseq": ((2, 12, 23, 37), (3, 5, 17, 75)),
    # both sides of the gate (20) and of HIQ (30); 19 is rare enough that many windows pass the gate
    "hug": ((19, 20, 21, 29, 30, 31), (2, 20, 20, 20, 19, 19)),
    # every base exactly Q20 or Q30, a few Q2 bases to cut windows: sums and bounds land on T exactly
    "flat20": ((20, 2), (97, 3)),
    "flat30": ((30, 2), (97, 3)),
    # every phred '!'..'~' (those below the gate at 3 % in all, so that windows pass it): seeds above 214,
    # the 214 -> 255 saturation within one or two additions
    "wide": (tuple(range(94)), (0.15,) * 20 + (97 / 74,) * 74),
    # NovaSeq bins, and N bases keep the phred drawn for them instead of 2: the seed of a k-mer sums the
    # record's first k quality bytes, N positions included (:337-339)
    "n_keeps_quality": ((2, 12, 23, 37), (3, 5, 17, 75)),
}

_CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i


def requantize(records, L: int, profile: str, seed: int) -> np.ndarray:
    """A copy of a record buffer (every read followed by its reverse complement, NUL-terminated) in which
    the qualities of every forward record are drawn from `profile` and those of its reverse-complement
    record are the same draws reversed.  Bases and strand bytes are kept; N bases get phred 2 unless the
    profile is n_keeps_quality."""
    values, weights = PROFILES[profile]
    rb = 2 * L + 1
    out = np.array(records, dtype=np.uint8, copy=True)
    n = out.size // rb
    if n % 2:
        raise ValueError("odd number of records: not a read / reverse-complement buffer")
    pairs = out[: n * rb].reshape(n // 2, 2, rb)
    p = None if weights is None else np.asarray(weights, np.float64) / sum(weights)
    q = np.random.default_rng(seed).choice(np.asarray(values, np.uint8), size=(n // 2, L), p=p)
    if profile != "n_keeps_quality":
        q[pairs[:, 0, 1:1 + L] == ord("N")] = N_PHRED
    pairs[:, 0, 1 + L:] = q + 33
    pairs[:, 1, 1 + L:] = (q + 33)[:, ::-1]
    return out


def quality_inputs(profile: str, L: int, n_pairs: int, seed: int, n_clones: int):
    """(primary, secondary) from synth.generate with the qualities redrawn from `profile`; n_keeps_quality
    inputs carry 1 % N bases so that many records have an N among their first k bases."""
    p_n = 0.01 if profile == "n_keeps_quality" else 0.0005
    primary, secondary = synth.generate(n_pairs=n_pairs, read_length=L, seed=seed, n_clones=n_clones, p_n=p_n,
                                        threads=2)
    return requantize(primary, L, profile, 2 * seed), requantize(secondary, L, profile, 2 * seed + 1)


def _records(buf, L):
    rb = 2 * L + 1
    a = np.asarray(buf, np.uint8)
    return a[: (a.size // rb) * rb].reshape(-1, rb)


def _window_all(mask, k):
    """[R, L] bool -> [R, L-k+1] bool: all of mask[r, i:i+k]."""
    bad = np.concatenate([np.zeros((mask.shape[0], 1), np.int16), np.cumsum(~mask, axis=1, dtype=np.int16)], axis=1)
    return (bad[:, k:] - bad[:, :-k]) == 0


class PruneModel:
    """Pass 1 of one input, reduced once (counts, distinct reads, the exact quality sums and the logged
    flags of every k-mer that can need its sums); prune() then decides any (mf, mq) from it."""

    def __init__(self, primary, secondary, L: int, k: int):
        recs = np.concatenate([_records(primary, L), _records(secondary, L)])
        w = L - k + 1
        codes = _CODE[recs[:, 1:1 + L]]
        qual = recs[:, 1 + L:] - np.uint8(33)          # (unsigned char)(ch - '!')
        acgt = codes < 4
        good, hiq = acgt & (qual >= GATE_Q), acgt & (qual >= HIQ)
        win_good, win_hiq = (_window_all(good, k), _window_all(hiq, k)) if w > 0 else (good[:, :0], hiq[:, :0])
        rec_gate, rec_hiq = good[:, :k].all(axis=1), hiq[:, :k].all(axis=1)

        r, i = np.nonzero(win_good)                    # gated windows in stamp order (r * w + i)
        c = np.where(acgt, codes, 0).astype(np.uint8)
        lo = np.zeros(r.size, np.uint64)
        hi = np.zeros(r.size, np.uint64)
        for j in range(k):
            if j < 32:
                lo |= c[r, i + j].astype(np.uint64) << np.uint64(2 * j)
            else:
                hi |= c[r, i + j].astype(np.uint64) << np.uint64(2 * (j - 32))
        order = np.lexsort((hi, lo))                   # stable: each k-mer's occurrences stay in stamp order
        r, i, lo, hi = r[order], i[order], lo[order], hi[order]
        new = np.ones(r.size, bool)
        new[1:] = (lo[1:] != lo[:-1]) | (hi[1:] != hi[:-1])
        starts = np.flatnonzero(new)
        sizes = np.diff(np.append(starts, r.size))
        self.n_pre_total = starts.size
        self.cnt = np.minimum(sizes, 32765)
        # hasMultipleUniqueReads: the occurrences come from reads that differ in sequence or strand byte
        if r.size:
            _, read_class = np.unique(recs[:, :1 + L].copy().view(f"V{1 + L}").ravel(), return_inverse=True)
            cls = read_class.ravel()[r]
            self.multi = np.minimum.reduceat(cls, starts) != np.maximum.reduceat(cls, starts)
        else:
            self.multi = np.zeros(0, bool)

        # k-mers that can be border k-mers (count <= NB <= 11): exact sums, the first occurrence contributing
        # its RECORD's first k qualities (:337-339), and the flags k_prune bounds them with
        small = self.multi & (self.cnt <= MAX_LOG_RANKS)
        self.small = np.flatnonzero(small)
        sel = np.repeat(small, sizes)
        br, bi = r[sel], i[sel]
        is_first = new[sel]
        bstarts = np.flatnonzero(is_first)
        off = np.where(is_first, 0, bi)
        if br.size:
            rows = qual[br[:, None], off[:, None] + np.arange(k)[None, :]].astype(np.int32)
            self.sums = np.add.reduceat(rows, bstarts, axis=0)
        else:
            self.sums = np.zeros((0, k), np.int32)

        def bound(a, b):
            """k_prune: a later occurrence adds HIQ or GATE_Q by LOG_A, the first one HIQ or 0 by LOG_B"""
            if not br.size:
                return np.zeros(0, np.int64)
            add = np.where(a[br, bi], HIQ, GATE_Q)
            return np.add.reduceat(add, bstarts) - add[bstarts] + np.where(b[br[bstarts]], HIQ, 0)

        self.bounds = dict(real=bound(win_hiq, rec_hiq), window=bound(win_good, rec_hiq),
                           record_start=bound(win_hiq, rec_gate), both=bound(win_good, rec_gate))

    def prune(self, mf: int, mq: int) -> dict:
        """n_pre_total, n_pre (survivors), n_border (k-mers whose sums must be looked at), unsound (border
        k-mers the real flags' bound keeps although a sum is < T: must be 0) and, per mutant, the number of
        k-mers whose prune decision it flips: its bound reaches T although a quality sum is below T."""
        T = min(mq, 254, QSUM_SAT)
        cand = (self.cnt >= mf) & self.multi
        border = cand & (GATE_Q * (self.cnt - 1) < T)
        b = border[self.small]                         # every border k-mer is one of the small ones
        sums_ok = (self.sums >= T).all(axis=1)
        out = dict(n_pre_total=int(self.n_pre_total), n_pre=int((cand & ~border).sum() + (sums_ok & b).sum()),
                   n_border=int(border.sum()), unsound=int((b & (self.bounds["real"] >= T) & ~sums_ok).sum()))
        for name in MUTANTS:
            out[name] = int((b & (self.bounds[name] >= T) & ~sums_ok).sum())
        return out


def flag_sensitivity(primary, secondary, L: int, k: int, mf: int, mq: int) -> dict:
    """The prune of pass-1 k-mers (prune_pre_graph :467-484) with k_prune's lower bound taken literally,
    with the flags the device must log and with each of MUTANTS: see PruneModel.prune."""
    return PruneModel(primary, secondary, L, k).prune(mf, mq)


# ---------------------------------------------------------------------------------------------------
# the cases of tests/test_quality_gpu.py (tests/test_quality_host.py shows each of them can fail)
# ---------------------------------------------------------------------------------------------------
# read length / k: one and two mask words (L > 64: windows straddle bit 64), the longest read
SHAPES = [(50, 35), (50, 25), (75, 35), (100, 35), (100, 50), (150, 41), (255, 50)]
# T = min(mq, 214) across every NB = ceil(T / 20) from 1 to 11 and both sides of 20 * (count - 1) < T
MQ_SWEEP = [20, 21, 40, 59, 60, 61, 89, 90, 91, 120, 121, 150, 200, 213, 214, 215, 254]
_PAIRS = {50: 8000, 75: 6000, 100: 4000, 150: 2500, 255: 1200}


def sweep(shape_index: int):
    """(mf, mq) of the mq sweep of one shape; mf in {1, 2, 3} rotates with the shape, so that over the
    shapes every mq meets every mf"""
    return [(1 + (n + shape_index) % 3, mq) for n, mq in enumerate(MQ_SWEEP)]


def shape_inputs(profile: str, L: int, k: int):
    return quality_inputs(profile, L, _PAIRS[L], seed=1000 + L + k, n_clones=300)


# every other build route on both qualities that split the gate from HIQ, at L = 100 (two mask words)
ROUTES = ["text", "pinned", "forward", "partitions1", "partitions256", "wide_tuples", "rounds2", "rounds8",
          "fp_bits0", "shard2", "shard4", "multi2"]
ROUTE_PROFILES = ["novaseq", "hug"]
ROUTE_SHAPE = (100, 35)
ROUTE_FLAGS = [(2, 60), (3, 90)]

# one mid-size input: many border k-mers per warp of k_prune, across many hash units
MID = dict(profile="novaseq", L=100, k=35, mf=2, mq=60, n_pairs=300_000, seed=4242, n_clones=30_000)


def mid_inputs():
    return quality_inputs(MID["profile"], MID["L"], MID["n_pairs"], MID["seed"], MID["n_clones"])
