"""CPU only: the restatement in sort_forms.py against abr_sort.cu / abr_capi.cu, and the case table of
test_gpu_sort_forms.py against every path, run size, chunk count, key width, shared-memory size, round fill and id
pattern of the session-order sort that a legal call can reach."""
import os
import re

import numpy as np
import pytest

import sort_forms as sf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abrsimulator_b200", "csrc")


def source(name):
    """The file with comments dropped and every run of whitespace made one space."""
    with open(os.path.join(CSRC, name)) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    return " ".join(text.split())


# ---- drift guard: what the restatement relies on is still in the sources ----
SORT_EXPRESSIONS = (
    "constexpr int kSortChunk = %d;" % sf.K_SORT_CHUNK,
    "constexpr int kSortThreads = %d;" % sf.K_SORT_THREADS,
    # sort_shape
    "*S = kSortChunk; *n_blocks = 0;",
    "if (n <= 0 || n_traces > %d) return;" % sf.K_MAX_TRACES,
    "long long blocks = ((long long)n + *S - 1) / *S;",
    "const long long max_cells = 1 << %d;" % (sf.K_MAX_CELLS.bit_length() - 1),
    "while (blocks * n_traces > max_cells && *S < (1 << %d)) { *S *= 2; blocks = ((long long)n + *S - 1) / *S; }"
    % (sf.K_MAX_S.bit_length() - 1),
    "if (blocks * n_traces > max_cells) return;",
    "*n_blocks = (int)blocks;",
    # key widths of the two paths
    "int key_bits = 0; while ((1 << key_bits) < n_traces) ++key_bits;",
    "int end_bit = 1; while (end_bit < 31 && (1ll << end_bit) < (long long)n_traces) ++end_bit;",
    # the counting sort: runs, chunks, rounds, shared memory
    "const int hi = min(n, (b + 1) * S);",
    "for (int c0 = b * S; c0 < hi; c0 += kSortChunk) {",
    "for (int k = 0; k < kSortChunk / 32; ++k) {",
    "const bool valid = c0 + 32 * k + lane < hi;",
    "for (int bit = 0; bit < key_bits; ++bit) {",
    "hist[(size_t)(t0 + kSortThreads * k) * n_blocks + b] = 0;",
    "abr_sort_place<<<n_blocks, kSortThreads, sizeof(int) * ((size_t)n_traces + 2 * kSortChunk), st>>>",
    # the radix path sorts the clamped keys
    "keys[i] = (t < 0 || t >= n_traces) ? 0 : t; iota[i] = i;",
    "SortPairs(cub_tmp, cub_bytes, keys_in, keys_out, iota, d_perm, n, 0, end_bit, st);",
)


@pytest.mark.parametrize("expr", SORT_EXPRESSIONS)
def test_sort_expressions(expr):
    assert expr in source("abr_sort.cu")


def test_invalid_ids_sort_as_trace_zero_in_both_kernels_of_the_counting_sort():
    assert source("abr_sort.cu").count("const int bucket = (t < 0 || t >= n_traces) ? 0 : t;") == 2


@pytest.mark.parametrize("expr", [
    "sort_shape(n_sessions, env->v.n_traces, &S, &n_blocks); if (n_blocks > 0) {",
    "const size_t cells = (((size_t)env->v.n_traces * n_blocks) + 63) & ~(size_t)63;",
    "if (fresh) CUDA_TRY(cudaMemset(env->sort_hist.p, 0, env->sort_hist.bytes));",
    "const size_t n = want + want / 2 > 256 ? want + want / 2 : 256;",
    "if (n_sessions > 0) { int S = 0, n_blocks = 0;",
])
def test_capi_expressions(expr):
    assert expr in source("abr_capi.cu")


def test_reset_puts_an_invalid_id_on_trace_zero():
    """What the sort's bucket rule mirrors: the reset counts one error and resets the session onto trace 0."""
    assert "if (tr < 0 || tr >= v.n_traces) { ++n_bad; tr = 0; }" in source("abr_step.cu")


# ---- the restatement against itself ----
@pytest.mark.parametrize("n,n_traces,want", [
    (1, 1, ("count", 512, 1, 0)), (512, 1, ("count", 512, 1, 0)), (513, 2, ("count", 512, 2, 1)),
    (70001, 1024, ("count", 512, 137, 10)), (100000, 8192, ("count", 4096, 25, 13)),
    (100000, 11264, ("count", 8192, 13, 14)), (100000, 11265, ("radix-traces", 512, 0, 0)),
    (4 << 20, 1024, ("count", 16384, 256, 10)), (sf.BIG, 11264, ("count", 1 << 20, 23, 14)),
    (sf.BIG + 1, 11264, ("radix-cells", 1 << 20, 0, 0)), (0, 7, ("empty", 512, 0, 0)),
])
def test_sort_shape(n, n_traces, want):
    sh = sf.sort_shape(n, n_traces)
    assert (sh.path, sh.S, sh.n_blocks, sh.key_bits) == want
    if sh.path == "count":
        assert sh.n_blocks * n_traces <= sf.K_MAX_CELLS and sh.smem <= sf.SMEM_48K
        assert (sh.n_blocks - 1) * sh.S < n <= sh.n_blocks * sh.S


def test_48k_boundary():
    assert sf.sort_shape(100000, 11264).smem == 49152
    assert sf.sort_shape(100000, 11265).path == "radix-traces"
    assert sf.sort_shape(sf.BIG, 11264).path == "count" and sf.sort_shape(sf.BIG + 1, 11264).path == "radix-cells"


def test_key_widths():
    assert [sf.key_bits_of(t) for t in (1, 2, 3, 1024, 1025, 8192, 11264)] == [0, 1, 2, 10, 11, 13, 14]
    assert [sf.end_bit_of(t) for t in (1, 2, 3, 1024, 11265, 13000)] == [1, 1, 2, 10, 14, 14]


@pytest.mark.parametrize("pattern", ["interleaved", "reversed", "random", "few", "one", "chunks", "invalid"])
@pytest.mark.parametrize("n,n_traces", [(1, 1), (513, 2), (5000, 13000), (70001, 1024)])
def test_reference_order_is_a_stable_permutation(pattern, n, n_traces):
    tid = sf.make_ids(pattern, n, n_traces)
    perm = sf.reference_order(tid, n_traces)
    assert perm.dtype == np.int32 and np.array_equal(np.sort(perm), np.arange(n))
    b = sf.bucket(tid, n_traces)[perm]
    assert np.all(np.diff(b) >= 0)
    assert np.all(np.diff(perm)[np.diff(b) == 0] > 0)            # stable: caller's order within a trace


def test_invalid_ids_sort_as_trace_zero():
    n_traces = 11265
    tid = np.array([5, -1, 0, n_traces, 3, (1 << 14) + 1, 0], np.int32)
    assert sf.reference_order(tid, n_traces).tolist() == [1, 2, 3, 5, 6, 4, 0]
    bad = sf.make_ids("invalid", 1000, n_traces)
    assert set(sf.invalid_ids(n_traces).tolist()) <= set(bad.tolist())
    # the raw key's low end_bit bits, what a radix sort of the unclamped ids would use, order them otherwise
    low = bad.astype(np.int64) & ((1 << sf.end_bit_of(n_traces)) - 1)
    assert not np.array_equal(np.argsort(low, kind="stable"), sf.reference_order(bad, n_traces))


# ---- coverage: the case table reaches every reachable cell ----
def missing_cells(cases):
    got = set().union(*(sf.case_cells(c) for c in cases))
    return sf.reachable_cells() - got


def test_case_table_reaches_every_reachable_cell():
    got = set().union(*(sf.case_cells(c) for c in sf.SORT_CASES))
    assert got <= sf.reachable_cells(), sorted(got - sf.reachable_cells())
    missing = sorted(missing_cells(sf.SORT_CASES))
    assert not missing, missing


@pytest.mark.parametrize("case", sf.SORT_CASES, ids=[c.name for c in sf.SORT_CASES])
def test_a_case_alone_in_a_cell_cannot_go(case):
    """Without a case that is the only one to reach a cell the table no longer covers every cell."""
    others = [c for c in sf.SORT_CASES if c is not case]
    alone = sf.case_cells(case) - set().union(*(sf.case_cells(c) for c in others))
    assert missing_cells(others) == alone


@pytest.mark.parametrize("shape", [
    (1, 1), (33, 1), (513, 2), (1 << 20, 2), (100000, 8192), (100000, 11264), (100000, 11265), (4 << 20, 1024),
    (sf.BIG, 11264), (sf.BIG + 1, 11264)])
def test_case_table_has_the_shapes(shape):
    assert shape in {(c.N, c.n_traces) for c in sf.SORT_CASES}


def test_case_table_is_consistent():
    names = [c.name for c in sf.SORT_CASES]
    assert len(set(names)) == len(names)
    patterns = {c.pattern for c in sf.SORT_CASES}
    assert patterns == {"interleaved", "reversed", "random", "few", "one", "chunks", "invalid"}
    assert [c.name for c in sf.SORT_CASES if c.big] == ["23Mix11264-interleaved", "23Mi+1x11264-invalid"]


def test_chunk_pattern_ends_runs_at_chunk_boundaries():
    for c in sf.SORT_CASES:
        if c.pattern == "chunks" and c.N <= (1 << 20):
            tid = c.ids()
            change = np.flatnonzero(np.diff(tid)) + 1
            assert change.size and np.all(change % sf.K_SORT_CHUNK == 0), c.name


def test_sequences_change_shape():
    assert sf.sequence_cells(sf.SEQUENCE, sf.SEQUENCE_TRACES) >= sf.SEQUENCE_MUST
    assert sf.sequence_cells(sf.BIG_SEQUENCE, 11264) >= sf.BIG_SEQUENCE_MUST
    assert max(sf.SEQUENCE) == 100000 and max(sf.BIG_SEQUENCE) == sf.BIG + 1
