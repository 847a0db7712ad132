"""Which shape the session-order sort takes — TEST INFRASTRUCTURE, no tests.

``abr_env_reset_sorted`` (abr_capi.cu) orders the sessions by trace with the counting sort of ``abr_sort.cu`` when
``sort_shape`` gives it a shape, and with CUB's radix sort (``abr_sort_by_trace``) otherwise.  The counting sort cuts
the sessions into runs of ``S``, and one block per run places its sessions ``kSortChunk`` at a time, in rounds of 32
lanes that find their peers with one ballot per key bit.  None of that changes the order, so comparing orders alone
cannot show which of those shapes a test went through.  This module restates, from the source:

* ``sort_shape``: the path (``count``, ``radix-traces``, ``radix-cells``), ``S``, the number of runs, chunks per run,
  key bits, the fill of the last chunk and of the last 32-lane round, and the dynamic shared memory of the place kernel;
* ``reference_order``: the order both paths must install, numpy's stable argsort of the trace ids with an invalid id
  (< 0 or >= n_traces) sorting as trace 0, the trace the reset puts such a session on;
* ``make_ids``: the trace-id patterns of the cases;
* ``SORT_CASES`` / ``case_cells`` / ``reachable_cells``: the cases of ``test_gpu_sort_forms.py`` and the cells they
  must reach; ``SEQUENCE`` / ``sequence_cells``: the calls one environment takes in a row, and the changes of shape
  between them that the zero-left-behind rule of the histogram has to survive.

``test_sort_forms_ledger.py`` checks, on the CPU, that the sources still contain what this restatement relies on and
that the cases reach every reachable cell.
"""
from __future__ import annotations

from dataclasses import dataclass
from functools import lru_cache

import numpy as np

# constants of abr_sort.cu (the ledger checks them against the source)
K_SORT_CHUNK = 512
K_SORT_THREADS = 256
K_MAX_TRACES = 11264               # cursors + two chunk buffers within 48 KB of shared memory
K_MAX_CELLS = 1 << 18              # (trace, run) cells of the one-launch scan
K_MAX_S = 1 << 20
SMEM_48K = 48 * 1024


@dataclass(frozen=True)
class Shape:
    path: str             # "count", "radix-traces", "radix-cells" or "empty"
    S: int                # sessions per run (count and radix-cells: the S the loop ended on)
    n_blocks: int         # runs (count only)
    chunks: int           # kSortChunk chunks of a full run (count only)
    key_bits: int         # ballots per round (count only)
    end_bit: int          # bits the radix sort looks at (radix only)
    last_chunk: int       # sessions in the last chunk of the last run (1..512)
    last_round: int       # lanes in the last 32-lane round (1..32)
    smem: int             # dynamic shared memory of abr_sort_place, bytes (count only)


def key_bits_of(n_traces):
    """launch_sort_gather: the least k with 2^k >= n_traces."""
    k = 0
    while (1 << k) < n_traces:
        k += 1
    return k


def end_bit_of(n_traces):
    """launch_sort_by_trace: as key_bits_of, but at least 1 and at most 31."""
    e = 1
    while e < 31 and (1 << e) < n_traces:
        e += 1
    return e


def sort_shape(n, n_traces):
    """sort_shape of abr_sort.cu plus the choice abr_env_reset_sorted makes from it."""
    if n <= 0:
        return Shape("empty", K_SORT_CHUNK, 0, 0, 0, 0, 0, 0, 0)
    S = K_SORT_CHUNK
    last_round = (n - 1) % 32 + 1
    radix = lambda path, S: Shape(path, S, 0, 0, 0, end_bit_of(n_traces), 0, last_round, 0)
    if n_traces > K_MAX_TRACES:
        return radix("radix-traces", S)
    blocks = -(-n // S)
    while blocks * n_traces > K_MAX_CELLS and S < K_MAX_S:
        S *= 2
        blocks = -(-n // S)
    if blocks * n_traces > K_MAX_CELLS:
        return radix("radix-cells", S)
    last_run = n - (blocks - 1) * S
    return Shape("count", S, blocks, S // K_SORT_CHUNK, key_bits_of(n_traces), 0, (last_run - 1) % K_SORT_CHUNK + 1,
                 last_round, 4 * (n_traces + 2 * K_SORT_CHUNK))


def bucket(tid, n_traces):
    """The trace a session sorts as: its id, or 0 for an invalid one."""
    tid = np.asarray(tid, np.int64)
    return np.where((tid < 0) | (tid >= n_traces), 0, tid)


def reference_order(tid, n_traces):
    """perm[p] = caller's index of the session at environment position p: the stable sort by bucket."""
    return np.argsort(bucket(tid, n_traces), kind="stable").astype(np.int32)


def invalid_ids(n_traces):
    """-1, n_traces, and 2^end_bit + 1 (whose low end_bit bits name trace 1)."""
    return np.array([-1, n_traces, (1 << end_bit_of(n_traces)) + 1], np.int64)


def make_ids(pattern, n, n_traces, seed=0):
    """Trace ids [n] int32 of a named pattern."""
    rng = np.random.default_rng(seed)
    s = np.arange(n, dtype=np.int64)
    if pattern == "interleaved":
        t = s % n_traces
    elif pattern == "reversed":                       # descending runs: every session moves
        t = (n_traces - 1) - (s * n_traces) // max(n, 1)
    elif pattern == "random":
        t = rng.integers(0, n_traces, n)
    elif pattern == "few":                            # three traces, one of them the last
        t = rng.choice(np.array(sorted({0, n_traces // 2, n_traces - 1})), n)
    elif pattern == "one":                            # every session on the last trace
        t = np.full(n, n_traces - 1)
    elif pattern == "chunks":                         # runs of one trace that end exactly at chunk boundaries
        t = (s // K_SORT_CHUNK * 7919) % n_traces
    elif pattern == "invalid":                        # random, then every tenth session gets an invalid id
        t = rng.integers(0, n_traces, n)
        bad = invalid_ids(n_traces)
        t[::10] = bad[(s[::10] // 10) % bad.size]
    else:
        raise ValueError(pattern)
    return t.astype(np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# cells
# ---------------------------------------------------------------------------------------------------------------------
def shape_cells(sh: Shape):
    cells = {("path", sh.path)}
    if sh.path != "count":
        return cells
    cells.add(("S", "512" if sh.S == K_SORT_CHUNK else "max" if sh.S == K_MAX_S else "between"))
    cells.add(("chunks per run", "one" if sh.chunks == 1 else "several"))
    cells.add(("key bits", "0" if sh.key_bits == 0 else "1-10" if sh.key_bits <= 10 else "11-14"))
    cells.add(("shared memory", "48 KB" if sh.smem == SMEM_48K else "below"))
    cells.add(("last round", "full" if sh.last_round == 32 else "partial"))
    cells.add(("last chunk", "full" if sh.last_chunk == K_SORT_CHUNK else "partial"))
    return cells


def id_cells(path, tid, n_traces):
    cells = set()
    b = bucket(tid, n_traces)
    if b.size and (b == b[0]).all():
        cells.add(("ids", path, "one trace"))
    if ((tid < 0) | (tid >= n_traces)).any():
        cells.add(("ids", path, "invalid"))
    return cells


def reachable_cells():
    cells = {("path", p) for p in ("count", "radix-traces", "radix-cells")}
    cells |= {("S", s) for s in ("512", "between", "max")}
    cells |= {("chunks per run", c) for c in ("one", "several")}
    cells |= {("key bits", k) for k in ("0", "1-10", "11-14")}
    cells |= {("shared memory", m) for m in ("below", "48 KB")}
    cells |= {("last round", r) for r in ("full", "partial")}
    cells |= {("last chunk", r) for r in ("full", "partial")}
    cells |= {("ids", p, "one trace") for p in ("count", "radix-traces")}
    # all sessions on one trace at the cells fallback would be a second run of 23 * 2^20 sessions; the large case
    # carries the invalid ids instead
    cells |= {("ids", p, "invalid") for p in ("count", "radix-traces", "radix-cells")}
    return cells


@dataclass(frozen=True)
class SortCase:
    name: str
    N: int
    n_traces: int
    pattern: str
    offsets: bool = True

    @property
    def big(self):
        return sort_shape(self.N, self.n_traces).S == K_MAX_S

    def shape(self):
        return sort_shape(self.N, self.n_traces)

    def ids(self):
        return make_ids(self.pattern, self.N, self.n_traces, seed=self.N ^ self.n_traces)


@lru_cache(maxsize=None)
def case_cells(c: SortCase):
    sh = c.shape()
    return shape_cells(sh) | id_cells(sh.path, c.ids(), c.n_traces)


BIG = 23 << 20      # the most sessions the counting sort takes over 11 264 traces (S = 2^20, 24 runs at 23 * 2^20 + 1)

SORT_CASES = (
    SortCase("1x1", 1, 1, "one", offsets=False),
    SortCase("33x1", 33, 1, "one"),
    SortCase("513x2-reversed", 513, 2, "reversed"),
    SortCase("513x2-invalid", 513, 2, "invalid"),
    SortCase("1Mix2-chunks", 1 << 20, 2, "chunks"),
    SortCase("70001x1024-random", 70001, 1024, "random"),
    SortCase("100000x8192-interleaved", 100000, 8192, "interleaved"),
    SortCase("100000x8192-invalid", 100000, 8192, "invalid"),
    SortCase("100000x11264-interleaved", 100000, 11264, "interleaved"),
    SortCase("100000x11264-few", 100000, 11264, "few"),
    SortCase("100000x11265-reversed", 100000, 11265, "reversed"),
    SortCase("100000x11265-invalid", 100000, 11265, "invalid"),
    SortCase("5000x13000-one", 5000, 13000, "one", offsets=False),
    SortCase("4Mix1024-interleaved", 4 << 20, 1024, "interleaved"),
    SortCase("4Mix1024-chunks", 4 << 20, 1024, "chunks"),
    SortCase("23Mix11264-interleaved", BIG, 11264, "interleaved"),
    SortCase("23Mi+1x11264-invalid", BIG + 1, 11264, "invalid"),
)


# One environment over 8 192 traces (a capacity of 100 000 sessions), one reset_sorted after another: S from 4 096
# down to 512 and back, an empty batch, and a histogram that has to grow.
SEQUENCE_TRACES = 8192
SEQUENCE = (2000, 100000, 513, 0, 33, 100000, 70001, 1)


def sequence_cells(ns, n_traces):
    cells = set()
    hist = 0                                            # the capacity abr_env_reset_sorted keeps, in cells
    prev, paths = None, []
    for n in ns:
        sh = sort_shape(n, n_traces)
        if sh.path == "empty":
            cells.add(("sequence", "empty batch"))
            continue
        if sh.path == "count":
            want = (n_traces * sh.n_blocks + 63) & ~63
            if want > hist:
                cells.add(("sequence", "hist allocated" if hist == 0 else "hist grown"))
                hist = want + want // 2
            else:
                cells.add(("sequence", "hist reused"))
        if prev is not None and sh.path == "count":      # against the last counting call
            if sh.S < prev.S:
                cells.add(("sequence", "S down"))
            if sh.S > prev.S:
                cells.add(("sequence", "S up"))
            if sh.n_blocks != prev.n_blocks:
                cells.add(("sequence", "runs change"))
        paths.append(sh.path)
        if sh.path == "count":
            prev = sh
    if any(paths[i:i + 3] == ["count", "radix-cells", "count"] for i in range(len(paths))):
        cells.add(("sequence", "count, radix, count"))
    return cells


SEQUENCE_MUST = {("sequence", c) for c in ("empty batch", "hist allocated", "hist grown", "hist reused", "S down",
                                          "S up", "runs change")}

# The large cases share one environment of 23 * 2^20 + 1 sessions: the counting sort at S = 2^20, the cells fallback,
# then the counting sort again on the histogram the first call left behind.
BIG_SEQUENCE = (BIG, BIG + 1, 100000)
BIG_SEQUENCE_MUST = {("sequence", "count, radix, count"), ("sequence", "S down"), ("sequence", "hist reused")}
