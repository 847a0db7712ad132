"""CPU only: the restatement in search_forms.py against the kernel sources, and the case table of
test_gpu_search_forms.py against every form and path of the two search kernels that a legal call can reach."""
import os
import re

import pytest

import search_forms as sf

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
@pytest.mark.parametrize("name,value", [("kMaxH", sf.K_MAX_H), ("kMaxA", sf.K_MAX_A),
                                        ("kMpcWarpsPerBlock", sf.K_MPC_WARPS_PER_BLOCK),
                                        ("kPrefixCache", sf.K_PREFIX_CACHE), ("kMaxLivePrefix", sf.K_MAX_LIVE_PREFIX),
                                        ("kMaxLiveRow", sf.K_MAX_LIVE_ROW)])
def test_mpc_constants(name, value):
    assert re.findall(rf"constexpr int {name} = (\d+);", source("abr_mpc.cu")) == [str(value)]


MPC_EXPRESSIONS = (
    # launch_mpc: warps per session, the block cap, branch and bound
    "const long long warps_needed_full = (long long)sms * 16;",
    "const int wps = (a.N >= warps_needed_full || combos < 32 * 36 * 4) ? 1 : kMpcWarpsPerBlock;",
    "const int spb = kMpcWarpsPerBlock / wps;",
    "const long long max_blocks = (long long)sms * 64;",
    "const bool clamp = a.mode == ABR_MPC_ROBUST;",
    "const bool prune = clamp && !(a.flags & ABR_MPC_EXHAUSTIVE) && a.p.smooth_penalty >= 0.0 && a.p.rebuf_penalty >= 0.0;",
    # abr_mpc_kernel: the grid-stride loop over sessions and the per-session path
    "for (long long s = (long long)blockIdx.x * SPB + slot; s < a.N; s += (long long)gridDim.x * SPB)",
    "if (h == 1) {",
    "for (int i = 0; i < h - 2; ++i) n_pre *= A;",
    "const bool compact = PRUNE && h >= 4 && n_pre / A <= kPrefixCache && n_pre <= kMaxLivePrefix && "
    "n_pre * A <= kMaxLiveRow;",
    "if (p.smooth_penalty == 1.0) {",
    "if (PRUNE && compact) o = search_compact<AT, CLAMP, true, WPS>(",
    # search: the parent-state cache
    "const int P = h - 2;",
    "const int n_par = P >= 2 ? n_prefix / A : 0;",
    "const bool use_cache = P >= 2 && n_par <= kPrefixCache;",
)


@pytest.mark.parametrize("expr", MPC_EXPRESSIONS)
def test_mpc_dispatch_expressions(expr):
    assert expr in source("abr_mpc.cu")


def test_mpc_compiled_ladder_sizes():
    text = source("abr_mpc.cu")
    switch = text[text.index("switch (a.A) {"):]
    switch = switch[:switch.index("}")]
    cases = re.findall(r"case (\d+): ABR_MPC_LAUNCH\((\d+)\); break;", switch)
    assert all(a == b for a, b in cases)
    assert tuple(int(a) for a, _ in cases) == sf.COMPILED_A
    assert "default: ABR_MPC_LAUNCH(0); break;" in switch


@pytest.mark.parametrize("expr", [
    "constexpr int kLookaheadBlock = %d;" % sf.K_LOOKAHEAD_BLOCK,
    "const int per_warp = 32 / A;",
    "const int g = lane / A, a0 = lane - g * A;",
    "const bool active = g < per_warp && i < v.n;",
    "const int per_block = (kLookaheadBlock / 32) * (32 / v.A);",
    "if (v.p.auto_reset) abr_lookahead_kernel<true><<<",
])
def test_lookahead_layout_expressions(expr):
    assert expr in source("abr_step.cu")


def test_lookahead_limit():
    with open(os.path.join(CSRC, "abr_capi.cu")) as f:
        text = f.read()
    assert "if (combos > %d.0)" % sf.LOOKAHEAD_MAX_COMBOS in text


# ---- coverage: the case table reaches every reachable cell ----
def reached(sms=sf.B200_SMS):
    """[(case, h, cell, stride)] of every searched horizon of every case."""
    return [(c, h, cell, stride) for c in sf.MPC_CASES for h, (cell, stride) in c.forms(sms).items()]


def test_case_table_reaches_every_reachable_cell():
    cells = sf.reachable_mpc_cells()
    got = {cell for _, _, cell, _ in reached()}
    print(f"\nreachable cells: {len(cells)}, reached by the {len(sf.MPC_CASES)} cases: {len(got & cells)}")
    assert got <= cells
    missing = sorted(cells - got, key=str)
    assert not missing, missing


def test_case_table_is_consistent():
    ids = [c.id for c in sf.MPC_CASES]
    assert len(set(ids)) == len(ids)
    for c in sf.MPC_CASES:
        assert (c.A, c.H) in sf.legal_mpc_shapes() and 1 <= c.K <= 64 and c.n >= 2 * len(c.hs)
        assert len(set(c.hs)) == len(c.hs) and all(1 <= h <= c.H for h in c.hs)
        assert c.mode != "ref" or c.hs == (c.H,)          # mode 0 without ABR_MPC_TRUNCATE: no truncated horizon


def test_stride_cases_visit_other_sessions():
    """A slot that serves several sessions must meet a distinct session next, not a copy of the one it served: a stale
    shared table would go unseen on a copy."""
    cases = [c for c in sf.MPC_CASES if any(st for _, st in c.forms().values())]
    assert cases
    for c in cases:
        assert c.N > c.slot_step() and c.slot_step() % c.n != 0, c.id


@pytest.mark.parametrize("case", [c for c in sf.MPC_CASES if c.ties], ids=lambda c: c.id)
def test_ties_cases_tie_across_live_prefixes(case):
    """At least half the distinct sessions of a ties case have an optimum tied exactly with a sequence in another
    live prefix, so the kernel's first minimum depends on the (value, index) compare, not on list order."""
    import numpy as np
    assert all(cell[0] == 4 and cell[2] == "compact" for cell, _ in case.forms().values())
    b, kw = sf.mpc_inputs(case, seed=sf.MPC_CASES.index(case))
    exp, _, _ = sf.mpc_expected(case, b, kw)
    assert exp["n_errors"] == 0 and len(np.unique(exp["action"])) >= 2
    assert 2 * sf.prefix_ties(case, b, kw, exp) >= case.n


def _must_reach():
    """What the suite did not execute before these cases existed; each entry: (what, predicate on (case, h, cell,
    stride))."""
    key = lambda cell: dict(zip(("wps", "AT", "path", "mode", "vw1"), cell))
    items = [
        ("runtime A, compacted search", lambda c, h, k, s: key(k)["AT"] == 0 and key(k)["path"] == "compact"),
        ("runtime A, parent-state cache", lambda c, h, k, s: key(k)["AT"] == 0 and key(k)["path"] == "cache"
         and key(k)["mode"] != "prune"),
        ("runtime A, branch and bound with the cache", lambda c, h, k, s: key(k)["AT"] == 0 and key(k)["path"] == "cache"
         and key(k)["mode"] == "prune"),
        ("branch and bound with the cache, A = 8, h = 5", lambda c, h, k, s: c.A == 8 and h == 5
         and key(k)["path"] == "cache" and key(k)["mode"] == "prune"),
        ("branch and bound with the cache, A = 12, h = 4", lambda c, h, k, s: c.A == 12 and h == 4
         and key(k)["path"] == "cache" and key(k)["mode"] == "prune"),
        ("compacted at its limits, A = 4, h = 6", lambda c, h, k, s: c.A == 4 and h == 6 and key(k)["path"] == "compact"),
        ("compacted, largest row count, A = 11, h = 4", lambda c, h, k, s: c.A == 11 and h == 4
         and key(k)["path"] == "compact"),
        ("block per session, compacted, exact ties", lambda c, h, k, s: c.ties and key(k)["wps"] == 4
         and key(k)["path"] == "compact"),
        ("H = 8 in the MPC kernel", lambda c, h, k, s: h == 8),
        ("A = 1 in the MPC kernel", lambda c, h, k, s: c.A == 1),
        ("history of more than 32 samples, mode 0", lambda c, h, k, s: c.K > 32 and key(k)["mode"] == "ref"),
        ("history of more than 32 samples, robust", lambda c, h, k, s: c.K > 32 and key(k)["mode"] == "prune"),
    ]
    for path in sf.PATHS:
        items.append((f"a block slot serving several sessions, {path}",
                      lambda c, h, k, s, path=path: s and key(k)["path"] == path))
    for A in (1, 7, 16):
        paths = {(cell[2], cell[3]) for a, H in sf.legal_mpc_shapes() if a == A
                 for cell in sf.reachable_mpc_cells_of(A, H)}
        for path, mode in sorted(paths):
            items.append((f"A = {A}, {path}, {mode}", lambda c, h, k, s, A=A, path=path, mode=mode:
                          c.A == A and key(k)["path"] == path and key(k)["mode"] == mode))
    return items


@pytest.mark.parametrize("what,pred", _must_reach(), ids=[w for w, _ in _must_reach()])
def test_case_table_reaches(what, pred):
    assert any(pred(*r) for r in reached()), what


def test_budget():
    """What the oracle enumerates for the GPU file: Σ over cases of distinct sessions × A^h × h."""
    total = sum(c.cost() for c in sf.MPC_CASES)
    assert total <= 6e7, total
    assert sum(c.cost() for c in sf.LOOKAHEAD_CASES) <= 1.2e8


# ---- lookahead ----
def test_lookahead_cases_reach_every_lane_layout():
    forms = {sf.lookahead_form(c.A, c.auto_reset) for c in sf.LOOKAHEAD_CASES}
    for A in (1, 2, 5, 7, 11, 16):
        for auto_reset in (0, 1):
            assert sf.lookahead_form(A, auto_reset) in forms
    assert (32, False, True) in forms and (32, False, False) in forms                 # A = 1: 32 one-lane sessions
    assert {f for f in forms if f[1]} >= {(6, True, r) for r in (True, False)}         # idle lanes (A = 5)
    assert {(2, True, r) for r in (True, False)} <= forms                               # two sessions per warp
    for c in sf.LOOKAHEAD_CASES:
        per_block = (sf.K_LOOKAHEAD_BLOCK // 32) * (32 // c.A)
        assert c.n % per_block != 0, c.id                                              # a partly filled last block
        assert c.A ** c.H <= sf.LOOKAHEAD_MAX_COMBOS
    shapes = {(c.A, c.H, c.auto_reset) for c in sf.LOOKAHEAD_CASES}
    for r in (0, 1):
        assert {(A, H, r) for A in (1, 2, 5, 7, 11, 16) for H in (1, 3)} <= shapes
        assert {(A, 8, r) for A in (1, 2, 5)} | {(16, 5, r)} <= shapes
