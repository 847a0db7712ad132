"""CPU only: the restatement in step_forms.py against the kernel sources and the C oracle, and the case table of
test_gpu_step_forms.py against every access path, head outcome, speculation outcome and compiled form of the
chunk-step kernels that a legal call can reach."""
import os
import re

import numpy as np
import pytest

import step_forms as sf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abrsimulator_b200", "csrc")


def source(name):
    """The file with comments dropped and every run of whitespace made one space."""
    with open(os.path.join(CSRC, name)) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    return " ".join(text.split())


# ---- drift guard: what the restatement relies on is still in the kernels ----
@pytest.mark.parametrize("decl", [
    "constexpr long long kPrefetchMinBytes = 192ll << 20;",
    "constexpr int kTile = %d;" % sf.K_TILE,
    "constexpr int kTileBlocksPerSM = %d;" % sf.K_TILE_BLOCKS_PER_SM,
    "constexpr int kStepTiles = %d;" % sf.K_STEP_TILES,
    "constexpr int kRolloutBlock = %d;" % sf.K_ROLLOUT_BLOCK,
    "constexpr int kStatsBlock = %d;" % sf.K_STATS_BLOCK,
    "constexpr int kStatsSessionsPerBlock = %d;" % sf.K_STATS_SESSIONS_PER_BLOCK,
    "constexpr int kWrapGuard = 1 << %d;" % (sf.K_WRAP_GUARD.bit_length() - 1),
    "constexpr int kStatsGroup = %d;" % sf.K_STATS_GROUP,
    "constexpr size_t kSmemOptInLimit = %d * 1024;" % (sf.K_SMEM_OPT_IN_LIMIT // 1024),
    "#define ABR_STEP_PF_DIST %d" % sf.K_PF_DIST,
])
def test_step_constants(decl):
    assert decl in source("abr_step.cu")


def test_prefetch_threshold():
    assert sf.K_PREFETCH_MIN_BYTES == 192 << 20


@pytest.mark.parametrize("expr", [
    "constexpr int kIdxMaxT = %d;" % sf.K_IDX_MAX_T,
    "int idx_cells(int T) { return T <= kIdxMaxT ? 2 * T : 0; }",
    "int idx_stride(int T_max) { return T_max <= kIdxMaxT ? (2 * T_max + 2 + 7) & ~7 : 0; }",
    "int cum_stride(int T_max) { return (T_max + 8 + 3) & ~3; }",
    "int cum_smem_doubles(int T_max) { return cum_stride(T_max) + 2; }",
    "if (lo != 0 || (hi & 0x800fffff) != 0 || e < 523 || e > 1523) return 0.0;",
])
def test_common_expressions(expr):
    assert expr in source("abr_common.cuh")


STEP_EXPRESSIONS = (
    # trace tables: the fixed M line, scale, the index rows, cell_of
    "int M = idx_stride(v.T_max) > 0 ? idx_cells(T) : 0;",
    "scale = ddiv((double)M, c); if (!(scale > 0.0) || !(scale < kInf)) M = 0;",
    "while (j <= T - 1 && (int)cell_of(c_row[j], scale, M) < b) ++j; i_row[b] = (uint16_t)(j - 1);",
    "const double y = dadd(dmul(x, scale), 6755399441055744.0); return min((uint32_t)__double2loint(y), (uint32_t)(M - 1));",
    # head_fast: staged and global success tests; head_any
    "j = j0 + (c1 <= t ? 1 : 0) + (c2 <= t ? 1 : 0) + (c3 <= t ? 1 : 0);",
    "ok = t < h.c_j1;",
    "const int q0 = j0 & ~3;",
    "ok = n_le >= 1 && n_le <= 7;",
    "return ok && t < s.P;",
    "do { target = dsub(target, s.P); ++n; } while (target >= s.P && n < kWrapGuard);",
    "j = 0; j_hi = s.T - 1;",
    "if (j_hi - j > 8) {",
    "if (s.M == 0 || !head_fast<SMEM>(s, raw, h)) head_any<SMEM>(s, raw, h, walk_error);",
    # run-ahead speculation
    "const bool can_speculate = SMEM || s.M > 0;",
    "if (calm && can_speculate) ok1 = head_fast<SMEM>(s, dadd(h.target, lk1.size), h1);",
    "calm = !__any_sync(lanes, moved);",
    "if (!can_speculate || !head_fast<SMEM>(s, raw, h1)) head_any<SMEM>(s, raw, h1, werr);",
    # launch_step: form, grid, buffer, staging, prefetch
    "const bool fast = !policy && !live && o.has_core() && v.p.track_history == 0 && v.p.track_acc == 0 && "
    "v.p.auto_reset != 0;",
    "int tiles_per_block = (total_tiles + sm_count * kTileBlocksPerSM - 1) / (sm_count * kTileBlocksPerSM);",
    "if (tiles_per_block < kStepTiles) tiles_per_block = kStepTiles;",
    "if (smem_bytes > kSmemOptInLimit || idx_stride(v.T_max) == 0) { smem_doubles = 0; smem_bytes = 0; }",
    "if (tr_first == tr_last && tr_first != staged) {",
    "parity ^= 1u;",
    "if (tr == staged) {",
    "const bool stream_from_hbm = (long long)v.n * 121 >= kPrefetchMinBytes;",
    "if (stream_from_hbm && k + ABR_STEP_PF_DIST < tiles_per_block && j + 32 <= v.n && (threadIdx.x & 31) == 0) {",
    # launch_rollout: form, use_smem
    "const bool plain = !live && v.p.track_history == 0 && v.p.auto_reset != 0;",
    "const bool fast = plain && out.has_core() && !out.actions;",
    "const bool none = plain && out.none();",
    "const bool uni = v.uniform_util != 0;",
    "if (fast && uni) return go(abr_rollout_kernel<P, true, false, false, kAhead, OT>, o);",
    "if (none && uni) return go(abr_rollout_kernel<P, true, true, false, kAhead, double>, o_none);",
    "if (fast || none) return cudaErrorInvalidValue;",
    "const bool use_smem = staged && same && __ldg(&v.trace_meta[tr0].M) > 0;",
    "size_t smem_bytes = ((size_t)smem_doubles + 2 * (size_t)v.V * v.A) * sizeof(double) + "
    "(size_t)idx_stride(v.T_max) * sizeof(uint16_t);",
    # position edges
    "int seg = (n >= 0.0 && n < 2147483648.0) ? (int)((uint32_t)n % (uint32_t)T) : (int)fmod(n, (double)T);",
    "if (n < 2147480000.0) {",
    # statistics trees
    "for (int d = 16; d > 0; d >>= 1) x = dadd(x, __shfl_down_sync(0xffffffffu, x, d));",
    "for (int w = 1; w < kRolloutBlock / 32; ++w) x = dadd(x, s_part[w][threadIdx.x]);",
    "for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) x[j] = dadd(x[j], v.acc[(size_t)j * v.cap + i]);",
    "x = (l < (int)(blockDim.x >> 5)) ? sm[l] : 0.0;",
    "double s = x[0]; #pragma unroll for (int k = 1; k < 8; ++k) s = dadd(s, x[k]);",
    "for (int g0 = q; g0 < n_groups; g0 += 32) {",
    "x[k] = g0 + 4 * k < n_groups ? __ldcg(group_partials + (size_t)(g0 + 4 * k) * ABR_NUM_ACC + j) : 0.0;",
    "out[t] = dadd(dadd(dadd(sm[0][t], sm[1][t]), sm[2][t]), sm[3][t]);",
)


@pytest.mark.parametrize("expr", STEP_EXPRESSIONS)
def test_step_expressions(expr):
    assert expr in source("abr_step.cu")


def test_statistics_tree_choice():
    """abr_stats_partial reuses the episode's block partials while they are fresh and runs stage 1 otherwise."""
    text = source("abr_capi.cu")
    assert "env->fresh_partials = steps > 0 ? rollout_num_blocks(env->v.n) : 0;" in text
    assert "const int np = fresh ? env->fresh_partials : stats_num_partials(env->v.n);" in text
    assert text.count("env->fresh_partials = 0;") == 3


# ---- the restatement against the oracle and against itself ----
def test_trace_tables_reproduce_the_oracles_positions():
    """C restated bit for bit: the oracle's reset position C[seg] + (C[seg+1] - C[seg]) * phi at every segment."""
    from oracle import oracle as orc
    for world in ("mixed", "edges", "long70000"):
        bitrates, sizes, bw, tl, ti = sf.make_world(world)
        tab = sf.trace_tables(bw, tl, ti, orc.DEFAULTS["payload"])
        tid = np.repeat(np.arange(len(tl)), 64).astype(np.int32)
        rng = np.random.default_rng(0)
        off = rng.uniform(0, 1, tid.size) * (tl * ti)[tid]
        ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, tid.size)
        ref.reset(tid, off)
        seg, phi = ref.field("seg"), ref.field("phase")
        C = tab.C[tid]
        c0, c1 = C[np.arange(tid.size), seg], C[np.arange(tid.size), seg + 1]
        assert np.array_equal((c0 + (c1 - c0) * phi).view(np.uint64), ref.field("pos").view(np.uint64)), world


def test_index_bounds_every_position():
    """idx[b] <= j <= idx[b + 1] for the segment j of every position x of cell b (what head_any relies on)."""
    bitrates, sizes, bw, tl, ti = sf.make_world("mixed")
    tab = sf.trace_tables(bw, tl, ti, 0.95)
    rng = np.random.default_rng(1)
    for k in range(len(tl)):
        x = rng.uniform(0, tab.P[k], 20000)
        j = np.searchsorted(tab.C[k, :tab.T[k] + 1], x, side="right") - 1
        b = sf.cell_of(x, tab.scale[k], int(tab.M[k]))
        assert np.all(tab.idx[k][b] <= j) and np.all(j <= tab.idx[k][b + 1]), k


def test_tables_without_index_rows():
    """T_max > kIdxMaxT: the table has no rows, so no trace gets an index, however short; T_max = kIdxMaxT: all do."""
    for T_max, want in ((65535, True), (65536, False), (70000, False)):
        bitrates, sizes, bw, tl, ti = sf.make_world(f"long{T_max}")
        tab = sf.trace_tables(bw, tl, ti, 0.95)
        assert (sf.idx_stride(T_max) > 0) == want
        assert np.all((tab.M > 0) == want) and np.all(tab.ok)


def test_cell_of_rounds_to_nearest():
    assert list(sf.cell_of(np.array([0.0, 0.49, 0.5, 1.5, 2.5, 7.0, 1e9]), 1.0, 8)) == [0, 0, 0, 2, 2, 7, 7]


def test_statistics_trees_are_sums():
    """Both restated trees add every session once (up to rounding) and differ from each other in their order."""
    rng = np.random.default_rng(2)
    for n in (1, 63, 64, 65, 2049, 70001):
        acc = rng.uniform(-1, 1, (sf.NUM_ACC, n))
        for tree in (sf.stats_fused, sf.stats_stage1):
            np.testing.assert_allclose(tree(acc), acc.sum(axis=1), rtol=1e-12, atol=1e-12)
    assert sf.stats_fused(np.ones((sf.NUM_ACC, 5))).tolist() == [5.0] * sf.NUM_ACC


# ---- coverage: the case table reaches every reachable cell ----
def test_case_table_reaches_every_reachable_cell():
    cells = sf.reachable_cells()
    got = set().union(*(c.reaches for c in sf.STEP_CASES))
    assert got <= cells, sorted(got - cells, key=str)
    missing = sorted(cells - got, key=str)
    assert not missing, missing


def test_case_table_is_consistent():
    names = [c.name for c in sf.STEP_CASES]
    assert len(set(names)) == len(names)
    for c in sf.STEP_CASES:
        assert c.reaches and c.form() is not None, c.name
        assert c.kernel in ("step", "policy", "fused", "run", "run_host", "lookahead") and c.steps >= 1
        bitrates, sizes, bw, tl, ti = sf.make_world(c.world)
        tid, off = sf.make_layout(c, tl, ti)
        assert tid.size == c.N and tid.min() >= 0 and tid.max() < len(tl)
        if c.kernel == "fused":
            assert all(cell[1] == c.form() for cell in c.reaches if cell[0] == "fused")


MUST_REACH = [
    ("short traces without index, per-step", lambda c: c.world in ("long65536", "long70000") and c.kernel == "step"),
    ("short traces without index, fused", lambda c: c.world in ("long65536", "long70000") and c.kernel == "fused"),
    ("short traces without index, lookahead", lambda c: c.world in ("long65536", "long70000")
     and c.kernel == "lookahead"),
    ("T_max = kIdxMaxT, all kernels", lambda c: c.world == "long65535"),
    ("2^21 + 77 sessions, per-step", lambda c: c.N == (1 << 21) + 77 and c.kernel == "step"),
    ("FAST + UNI", lambda c: c.kernel == "fused" and c.form()[1:5] == (True, False, False, True)),
    ("NOOUT + UNI", lambda c: c.kernel == "fused" and c.form()[1:5] == (True, True, False, True)),
    ("no index, no speculation", lambda c: sf.spec("global", "no_index") in c.reaches),
    ("safety net, staged", lambda c: sf.head("step", "smem", "guard") in c.reaches),
    ("sleep past 2^31 segments", lambda c: ("edge", "sleep_fmod") in c.reaches),
    ("live idle past 2^31 segments", lambda c: ("edge", "live_fmod") in c.reaches),
]


@pytest.mark.parametrize("what,pred", MUST_REACH, ids=[w for w, _ in MUST_REACH])
def test_case_table_reaches(what, pred):
    assert any(pred(c) for c in sf.STEP_CASES), what


def test_big_case_layout():
    """The 2^21 + 77 case: the prefetch on, more than kStepTiles tiles per block, partial last tile and block, two or
    more restages in a block (both parities), straddling lanes, a mixed tile in every full block."""
    c = next(c for c in sf.STEP_CASES if c.layout == "bign")
    bitrates, sizes, bw, tl, ti = sf.make_world(c.world)
    tid, _ = sf.make_layout(c, tl, ti)
    p = sf.step_paths(tid, int(bw.shape[1]))
    tpb, grid = sf.step_grid(c.N)
    assert sf.step_prefetch(c.N) and tpb > sf.K_STEP_TILES
    assert p.partial_last_tile and p.partial_last_block
    assert (p.restages[:-1] >= 2).all() and p.straddle > 0 and (p.mixed_per_block[:-1] >= 1).all()
    assert p.smem.any() and (~p.smem).any()


def test_budget():
    """Oracle session-steps of the GPU file."""
    total = sum(c.cost() for c in sf.STEP_CASES)
    assert total <= 1.2e7, total
