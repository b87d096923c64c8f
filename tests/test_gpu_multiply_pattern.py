"""-m gpu tests of multiply with fixed operand patterns (spb_mm_pattern_*, sp.MultiplyPattern): every run must equal
spb_multiply_mm on arrays with the plan's indices and the run's values, bit for bit -- indices, entry order, values compared
as bits (NaNs matched), shape and the unsorted flag -- and the oracle where the size allows.  Covered: every operand state
under both transpose flags, one array for both operands, scale vectors and C, the empty products, one plan running many value
sets (fast path and fallback alternating: runs emptied and refilled, zero_nan with a leading run that depends on B's order,
infinities opposite an emptied run, exact cancellation in the merge and the hash bin, long runs, everything dropped) under
every policy, the bins (merge builds, hash windows and split items, rows expand-sort-compress would take), the fixed launch
count of the fast path, a poisoned pool, where the values live, a 2^23 + 4097 entry pattern, the errors, and the C++ class."""
import contextlib
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _thresholds
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    import spsparse_b200 as sp
    with sp.Context(0) as c:
        yield c


@contextlib.contextmanager
def _env(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@contextlib.contextmanager
def _context(**env):
    """A context created with the given environment (SPB_POOL_POISON is read at context creation)."""
    import spsparse_b200 as sp
    with _env(**env):
        c = sp.Context(0)
    try:
        yield c
    finally:
        c.close()


def _launches(ctx):
    n = C.c_uint64()
    assert ctx.lib.spb_ctx_launch_count(ctx.h, C.byref(n)) == 0
    return n.value


class Op:
    """Host pattern of one operand: shape, index arrays and the sort flag it is uploaded with."""

    def __init__(self, shape, idx, so=None):
        self.shape, self.idx, self.so = tuple(int(s) for s in shape), [np.asarray(a, np.int32) for a in idx], so

    @property
    def n(self):
        return len(self.idx[0])

    def up(self, ctx, val):
        import spsparse_b200 as sp
        return sp.CooArray.from_host(ctx, self.shape, self.idx, np.asarray(val, np.float64), self.so)

    def coo(self, val):
        return O.Coo(self.shape, self.idx, np.asarray(val, np.float64), self.so)


def _vec(ctx, v):
    import spsparse_b200 as sp
    return None if v is None else sp.CooArray.from_host(ctx, v.shape, v.idx, v.val)


def _down(R):
    idx, val = R.to_host()
    out = (tuple(R.shape), R.sort_order, [np.asarray(a) for a in idx], np.asarray(val))
    R.free()
    return out


def same(got, want, what=""):
    assert got[0] == want[0] and got[1] == want[1], f"{what}: shape / sort flag {got[:2]} != {want[:2]}"
    assert len(got[3]) == len(want[3]), f"{what}: nnz {len(got[3])} != {len(want[3])}"
    for k in range(2):
        assert np.array_equal(got[2][k], want[2][k]), f"{what}: index {k} differs"
    g, w = got[3], want[3]
    ok = (g.view(np.uint64) == w.view(np.uint64)) | (np.isnan(g) & np.isnan(w))
    assert ok.all(), f"{what}: {int((~ok).sum())} values differ in their bits"


class Case:
    def __init__(self, A, tA, B, tB, Cst=1.0, si=None, sj=None, sk=None, pol=O.ADD, zn=False):
        self.A, self.tA, self.B, self.tB, self.Cst, self.si, self.sj, self.sk, self.pol, self.zn = \
            A, tA, B, tB, Cst, si, sj, sk, pol, zn

    def plan(self, ctx):
        import spsparse_b200 as sp
        dA, dB = self.A.up(ctx, np.ones(self.A.n)), self.B.up(ctx, np.ones(self.B.n))
        si, sj, sk = _vec(ctx, self.si), _vec(ctx, self.sj), _vec(ctx, self.sk)
        p = sp.MultiplyPattern(ctx, self.Cst, si, dA, self.tA, sj, dB, self.tB, sk, self.pol, self.zn)
        for x in (dA, dB, si, sj, sk):   # the plan keeps what it needs
            if x is not None:
                x.free()
        return p

    def fresh(self, ctx, av, bv):
        import spsparse_b200 as sp
        dA, dB = self.A.up(ctx, av), self.B.up(ctx, bv)
        si, sj, sk = _vec(ctx, self.si), _vec(ctx, self.sj), _vec(ctx, self.sk)
        R, st = sp.multiply(ctx, self.Cst, si, dA, self.tA, sj, dB, self.tB, sk, self.pol, self.zn, stats=True)
        for x in (dA, dB, si, sj, sk):
            if x is not None:
                x.free()
        return _down(R), st

    def oracle(self, orc, av, bv):
        r = orc.multiply_mm(self.Cst, self.si, self.A.coo(av), self.tA, self.sj, self.B.coo(bv), self.tB, self.sk,
                            self.pol, self.zn)
        return r.idx, r.val


def check_runs(ctx, case, value_sets, orc=None, plan=None):
    """Runs every (a, b) value set through one plan; each result must equal spb_multiply_mm (and the oracle).  Returns the
    plan's and the fresh path's statistics per set."""
    own = plan is None
    plan = plan or case.plan(ctx)
    out = []
    try:
        for t, (av, bv) in enumerate(value_sets):
            R, st = plan.run(av, bv, stats=True)
            got = _down(R)
            want, fst = case.fresh(ctx, av, bv)
            same(got, want, f"value set {t}")
            assert len(got[3]) <= plan.nnz_bound
            if orc is not None:
                idx, val = case.oracle(orc, av, bv)
                assert all(np.array_equal(got[2][k], idx[k]) for k in range(2)), f"value set {t}: oracle indices"
                ok = (got[3].view(np.uint64) == val.view(np.uint64)) | (np.isnan(got[3]) & np.isnan(val))
                assert ok.all(), f"value set {t}: oracle values"
            out.append((st, fst))
    finally:
        if own:
            plan.free()
    return out


def _rand_pattern(rng, shape, n, dup=0.3):
    """Random (row, col) entries with about `dup` of them repeating an earlier tuple, unsorted."""
    r = rng.integers(0, shape[0], n)
    c = rng.integers(0, shape[1], n)
    k = int(n * dup)
    src = rng.integers(0, n - k, k)
    r[n - k:], c[n - k:] = r[src], c[src]
    p = rng.permutation(n)
    return [r[p], c[p]]


def _sorted_unique(idx, so):
    """The distinct tuples of idx in the order so (an operand that may be flagged sorted)."""
    key = np.unique(np.stack([idx[so[0]], idx[so[1]]], 1), axis=0)
    out = [None, None]
    out[so[0]], out[so[1]] = key[:, 0], key[:, 1]
    return out


def _vals(rng, n):
    return _thresholds.values(rng, n)


# ---- plan shapes ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tA", [".", "T"])
@pytest.mark.parametrize("tB", [".", "T"])
@pytest.mark.parametrize("sa", ["unsorted", "needed", "other"])
@pytest.mark.parametrize("sb", ["unsorted", "needed", "other"])
def test_operand_states(ctx, orc, tA, tB, sa, sb):
    rng = np.random.default_rng([tA == "T", tB == "T", len(sa), len(sb)])
    m, k, q = 40, 30, 35
    a_shape = (m, k) if tA == "." else (k, m)
    b_shape = (k, q) if tB == "." else (q, k)
    a_need = (0, 1) if tA == "." else (1, 0)
    b_need = (1, 0) if tB == "." else (0, 1)   # the reference's order for B: (col, inner)
    ops = []
    for shape, st, need in ((a_shape, sa, a_need), (b_shape, sb, b_need)):
        idx = _rand_pattern(rng, shape, 300)
        so = None if st == "unsorted" else (need if st == "needed" else need[::-1])
        if so is not None:
            idx = _sorted_unique(idx, so)
        ops.append(Op(shape, idx, so))
    A, B = ops
    for zn in (False, True):
        case = Case(A, tA, B, tB, zn=zn)
        sets = []
        for t in range(4):
            av, bv = _vals(rng, A.n), _vals(rng, B.n)
            if t % 2:   # zeros: a fallback whenever an operand is folded
                av[rng.integers(0, A.n, 40)] = 0.0
                bv[rng.integers(0, B.n, 40)] = 0.0
            if zn and t == 3:
                bv[rng.integers(0, B.n, 20)] = np.nan
            sets.append((av, bv))
        res = check_runs(ctx, case, sets, orc)
        assert not res[0][0].fallback and not res[2][0].fallback


def test_same_array_for_both_operands(ctx, orc):
    """A * diag(s) * A^T from one array and one value pointer (config 3)."""
    import spsparse_b200 as sp
    import torch
    rng = np.random.default_rng(3)
    A = Op((50, 60), _rand_pattern(rng, (50, 60), 400))
    s = O.Coo((60,), [np.arange(0, 60, 2)], _vals(rng, 30))
    dA = A.up(ctx, np.ones(A.n))
    ds = _vec(ctx, s)
    plan = sp.MultiplyPattern(ctx, 1.0, None, dA, ".", ds, dA, "T", None)
    dA.free(); ds.free()
    case = Case(A, ".", A, "T", sj=s)
    try:
        for t in range(3):
            v = _vals(rng, A.n)
            if t == 1:
                v[:50] = 0.0
            tv = torch.from_numpy(v).cuda()
            R, st = plan.run(tv, tv, stats=True)
            got = _down(R)
            want, _ = case.fresh(ctx, v, v)
            same(got, want, f"set {t}")
            idx, val = case.oracle(orc, v, v)
            assert np.array_equal(got[3].view(np.uint64), val.view(np.uint64))
    finally:
        plan.free()


def test_scales_and_C(ctx, orc):
    rng = np.random.default_rng(5)
    m, k, q = 64, 48, 57
    A = Op((m, k), _rand_pattern(rng, (m, k), 500))
    B = Op((k, q), _rand_pattern(rng, (k, q), 500))
    # zero values, absent indices and an entry at the last index of every scale vector
    si = O.Coo((m,), [np.r_[np.arange(0, m - 1, 3), m - 1]], np.r_[_vals(rng, len(range(0, m - 1, 3))), 0.5])
    si.val[::4] = 0.0
    sj = O.Coo((k,), [np.r_[np.arange(1, k - 1, 2), k - 1]], np.r_[_vals(rng, len(range(1, k - 1, 2))), -2.0])
    sj.val[::5] = 0.0
    sk = O.Coo((q,), [np.r_[np.arange(0, q - 1, 2), q - 1]], np.r_[_vals(rng, len(range(0, q - 1, 2))), 3.0])
    sk.val[1::6] = 0.0
    for Cst in (2.5, -0.75):
        case = Case(A, ".", B, ".", Cst, si, sj, sk)
        sets = [(_vals(rng, A.n), _vals(rng, B.n)) for _ in range(2)]
        check_runs(ctx, case, sets, orc)


@pytest.mark.parametrize("which", ["C0", "empty_scale", "empty_A"])
def test_empty_products(ctx, which):
    import spsparse_b200 as sp
    rng = np.random.default_rng(7)
    A = Op((20, 30), _rand_pattern(rng, (20, 30), 100) if which != "empty_A" else [[], []])
    B = Op((30, 25), _rand_pattern(rng, (30, 25), 100))
    sj = O.Coo((30,), [np.array([], np.int32)], np.array([])) if which == "empty_scale" else None
    case = Case(A, ".", B, ".", 0.0 if which == "C0" else 1.0, sj=sj)
    plan = case.plan(ctx)
    try:
        assert plan.nnz_bound == 0
        for _ in range(2):
            R = plan.run(np.ones(A.n), np.ones(B.n))
            assert tuple(R.shape) == (20, 25) and R.size() == 0
            want, _ = case.fresh(ctx, np.ones(A.n), np.ones(B.n))
            same(_down(R), want)
    finally:
        plan.free()
    assert isinstance(sp.MultiplyPattern, type)


# ---- value sets -------------------------------------------------------------------------------------------------------------
def _mix_case(rng, pol, zn):
    """A and B unsorted with duplicates, a run of 300 copies of one tuple in A (folded by the warp kernel), an inner index
    whose B row holds NaN / +-inf, and entries arranged so that B's leading NaN run differs between (inner, col) and (col,
    inner) order."""
    m, k, q = 30, 20, 24
    ai = _rand_pattern(rng, (m, k), 400)
    bi = _rand_pattern(rng, (k, q), 300)
    # the long run: (3, 4) 300 times
    ai = [np.r_[ai[0], np.full(300, 3)], np.r_[ai[1], np.full(300, 4)]]
    # B: (inner 0, col 5) = NaN first in (inner, col) order, (inner 1, col 0) the first kept entry in (col, inner) order
    bi = [np.r_[[0, 1, 0], bi[0]], np.r_[[5, 0, 6], bi[1]]]
    # A row 2 uses inner 7 only through the tuple (2, 7); B row 7 holds an infinity
    ai = [np.r_[ai[0], 2, 2], np.r_[ai[1], 7, 7]]
    bi = [np.r_[bi[0], 7], np.r_[bi[1], 9]]
    return Op((m, k), ai), Op((k, q), bi)


def _mix_sets(rng, A, B):
    """(a, b, expect_fallback) value sets, fast and fallback runs alternating."""
    ia = [np.flatnonzero((A.idx[0] == A.idx[0][t]) & (A.idx[1] == A.idx[1][t])) for t in range(A.n)]
    ib = [np.flatnonzero((B.idx[0] == B.idx[0][t]) & (B.idx[1] == B.idx[1][t])) for t in range(B.n)]
    run_27 = np.flatnonzero((A.idx[0] == 2) & (A.idx[1] == 7))
    run_long = np.flatnonzero((A.idx[0] == 3) & (A.idx[1] == 4))
    b_inf = np.flatnonzero((B.idx[0] == 7) & (B.idx[1] == 9))
    base_a, base_b = _vals(rng, A.n), _vals(rng, B.n)
    sets = [(base_a, base_b, False)]
    a = base_a.copy()   # duplicates cancelling to an explicit 0.0 (still present: fast path)
    r = ia[0]
    if len(r) >= 2:
        a[r] = 0.0
        a[r[0]], a[r[1]] = 1.25, -1.25
    sets.append((a, base_b, False))
    a = base_a.copy()   # a whole run of A emptied by zeros
    a[ia[5]] = 0.0
    sets.append((a, base_b, True))
    sets.append((base_a, base_b, False))   # refilled
    b = base_b.copy()   # a whole run of B emptied
    b[ib[9]] = 0.0
    sets.append((base_a, b, True))
    sets.append((base_a, base_b, False))   # refilled
    b = base_b.copy()   # leading NaNs of B in (inner, col) order that are not leading in (col, inner) order
    b[0] = np.nan
    sets.append((base_a, b, False))
    b = base_b.copy()   # +-inf in B opposite the emptied A run (2, 7)
    b[b_inf] = np.inf
    a = base_a.copy()
    a[run_27] = 0.0
    sets.append((a, b, True))
    b[b_inf] = -np.inf
    sets.append((base_a, b, False))
    a = base_a.copy()   # the long run, order-sensitive values
    a[run_long] = _vals(rng, len(run_long)) * 1e3
    sets.append((a, base_b, False))
    a = base_a.copy()   # the long run emptied
    a[run_long] = 0.0
    sets.append((a, base_b, True))
    sets.append((np.zeros(A.n), np.zeros(B.n), True))   # everything dropped
    sets.append((base_a, base_b, False))
    return sets


@pytest.mark.parametrize("pol", [O.ADD, O.LEAVE_ALONE, O.REPLACE])
@pytest.mark.parametrize("zn", [False, True])
def test_one_plan_many_value_sets(ctx, orc, pol, zn):
    rng = np.random.default_rng(11 + pol * 2 + zn)
    A, B = _mix_case(rng, pol, zn)
    case = Case(A, ".", B, ".", pol=pol, zn=zn)
    sets = _mix_sets(rng, A, B)
    res = check_runs(ctx, case, [(a, b) for a, b, _ in sets], orc)
    for t, ((a, b, fb), (st, _)) in enumerate(zip(sets, res)):
        if not zn or t != 6:   # with zero_nan the leading NaN of set 6 may be the only entry of its run
            assert bool(st.fallback) == fb, f"set {t}: fallback {st.fallback}"
        if st.fallback:
            assert st.empty_runs_a + st.empty_runs_b > 0
        else:
            assert st.empty_runs_a == 0 and st.empty_runs_b == 0 and st.mm.ms_symbolic == 0


def test_zero_nan_bound_in_the_reference_order(ctx, orc):
    """B: (inner 0, col 5) = NaN sorts before the first kept (inner 0, col 6) in (inner, col) order, but after the first kept
    (inner 1, col 0) in the reference's (col, inner) order: it is kept, and its output is NaN."""
    A = Op((2, 2), [[0, 0], [0, 1]])
    B = Op((2, 8), [[0, 1, 0], [5, 0, 6]])
    case = Case(A, ".", B, ".", zn=True)
    res = check_runs(ctx, case, [(np.array([1.0, 2.0]), np.array([np.nan, 3.0, 4.0]))], orc)
    assert not res[0][0].fallback


def test_empty_run_is_not_zero(ctx, orc):
    """An A run emptied by zeros opposite an infinity in B: no term (0 * inf would be NaN)."""
    A = Op((2, 3), [[0, 0, 0, 1], [0, 1, 1, 2]])
    B = Op((3, 2), [[0, 1, 2], [0, 0, 1]])
    case = Case(A, ".", B, ".")
    res = check_runs(ctx, case, [(np.array([1.0, 0.0, 0.0, 2.0]), np.array([3.0, np.inf, 5.0])),
                                 (np.array([1.0, 2.0, -2.0, 2.0]), np.array([3.0, np.inf, 5.0]))], orc)
    assert res[0][0].fallback and res[0][0].empty_runs_a == 1 and not res[1][0].fallback


def test_long_run_folds_left_to_right(ctx, orc):
    """Runs of 257, 1000 and 4099 copies, signed values of very different magnitudes: a tree sum gives other bits."""
    rng = np.random.default_rng(17)
    lens = [257, 1000, 4099]
    r = np.concatenate([np.full(L, i) for i, L in enumerate(lens)])
    A = Op((3, 4), [r, np.zeros(len(r), np.int32)])
    B = Op((4, 2), [[0, 0], [0, 1]])
    case = Case(A, ".", B, ".")
    sets = []
    for _ in range(3):
        a = rng.standard_normal(len(r)) * np.exp2(rng.uniform(-30, 30, len(r)))
        sets.append((a, np.array([1.0, -1.0])))
    check_runs(ctx, case, sets, orc)


# ---- bins -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [2, 4, 6, 8])
def test_merge_builds(ctx, orc, L):
    rng = np.random.default_rng(L)
    m, k, q = 200, 150, 120
    rows = np.repeat(np.arange(m), L)
    cols = np.concatenate([rng.choice(k, L, replace=False) for _ in range(m)])
    A = Op((m, k), [rows, cols])
    B = Op((k, q), _rand_pattern(rng, (k, q), 600, dup=0.1))
    case = Case(A, ".", B, ".")
    av, bv = _vals(rng, A.n), _vals(rng, B.n)
    a2 = av.copy()
    a2[[0, 1]] = 0.0
    res = check_runs(ctx, case, [(av, bv), (a2, bv), _cancel_at(A, B, av, bv), (av, bv)], orc)
    assert res[0][0].mm.rows_merge > 0 and res[0][0].mm.rows_hash == 0 and res[1][0].fallback


def _cancel_at(A, B, av, bv):
    """Values for which one output of the row of A's first entry sums to exactly 0: the last column is given to the B rows of
    two entries of that row only (its inner indices are distinct), and their terms are 1*2 and -1*2."""
    c = B.shape[1] - 1
    B.idx[1][B.idx[1] == c] = c - 1
    t = [x for x in np.flatnonzero(A.idx[0] == A.idx[0][0]) if (B.idx[0] == A.idx[1][x]).any()][:2]
    e0 = np.flatnonzero(B.idx[0] == A.idx[1][t[0]])[0]
    e1 = np.flatnonzero(B.idx[0] == A.idx[1][t[1]])[0]
    B.idx[1][e0] = B.idx[1][e1] = c
    a, b = av.copy(), bv.copy()
    a[t[0]], a[t[1]] = 1.0, -1.0
    b[e0] = b[e1] = 2.0
    return a, b


def _hash_case(rng, m=40, k=300, q=2000, per_row=60, per_b=40):
    rows = np.repeat(np.arange(m), per_row)
    cols = np.concatenate([rng.choice(k, per_row, replace=False) for _ in range(m)])
    A = Op((m, k), [rows, cols])
    B = Op((k, q), [np.repeat(np.arange(k), per_b), np.concatenate([rng.choice(q, per_b, replace=False) for _ in range(k)])])
    return A, B


@pytest.mark.parametrize("env", [{}, {"SPB_HASH_WIN_COLS": "256"}, {"SPB_HASH_WIN_COLS": "256", "SPB_HASH_ITEM_CAP": "100"},
                                 {"SPB_HASH_ITEM_CAP": "37"}])
def test_hash_rows(ctx, orc, env):
    rng = np.random.default_rng(23)
    A, B = _hash_case(rng)
    case = Case(A, ".", B, ".")
    av, bv = _vals(rng, A.n), _vals(rng, B.n)
    with _env(**env):
        res = check_runs(ctx, case, [(av, bv), _cancel_at(A, B, av, bv), (av, bv)], orc)
    assert res[0][0].mm.rows_hash > 0 and res[0][0].mm.rows_esc == 0


def test_rows_esc_would_take_go_to_the_hash_bin(ctx, orc):
    """Rows of 9..12 inner indices with fewer than 512 products: spb_multiply_mm runs them through expand-sort-compress, the
    plan through the hash bin."""
    rng = np.random.default_rng(29)
    m, k, q = 50, 100, 400
    L = 9 + np.arange(m) % 4
    rows = np.repeat(np.arange(m), L)
    cols = np.concatenate([rng.choice(k, n, replace=False) for n in L])
    A = Op((m, k), [rows, cols])
    B = Op((k, q), [np.repeat(np.arange(k), 3), rng.integers(0, q, 3 * k)])
    case = Case(A, ".", B, ".")
    res = check_runs(ctx, case, [(_vals(rng, A.n), _vals(rng, B.n)) for _ in range(2)], orc)
    st, fst = res[0]
    assert fst.rows_esc > 0 and st.mm.rows_esc == 0 and st.mm.rows_hash >= fst.rows_esc


# ---- path pins --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("zn", [False, True])
def test_fast_path_launch_count(ctx, zn):
    rng = np.random.default_rng(31)
    A, B = _hash_case(rng, m=30)
    case = Case(A, ".", B, ".", zn=zn)
    plan = case.plan(ctx)
    try:
        counts = []
        for _ in range(3):
            av, bv = _vals(rng, A.n), _vals(rng, B.n)
            l0 = _launches(ctx)
            R, st = plan.run(av, bv, stats=True)
            counts.append(_launches(ctx) - l0)
            R.free()
            assert not st.fallback and st.mm.ms_symbolic == 0 and st.mm.ms_prepare == 0
        # two folds of two kernels (+ the leading-run bound each with zero_nan), the hash numeric kernel, the merge numeric
        # kernel where merge rows exist; no sort, count or bitmap kernel
        want = 4 + (2 if zn else 0) + (1 if st.mm.rows_hash else 0) + (1 if st.mm.rows_merge else 0)
        assert counts == [want] * 3, counts
    finally:
        plan.free()


def _poison_sequence(c):
    import spsparse_b200 as sp
    rng = np.random.default_rng(37)
    A, B = _mix_case(rng, O.ADD, True)
    case = Case(A, ".", B, ".", zn=True)
    sets = _mix_sets(rng, A, B)
    plan = case.plan(c)
    out = []
    l0 = _launches(c)
    for a, b, _ in sets[:6]:
        R, st = plan.run(a, b, stats=True)
        out.append((_down(R), st.fallback, st.empty_runs_a, st.empty_runs_b, st.mm.nnz_c, st.mm.rows_merge, st.mm.rows_hash))
    plan.free()
    assert isinstance(sp.MultiplyPattern, type)
    return out, _launches(c) - l0


@pytest.mark.parametrize("pattern", ["00", "ff", "7f"])
def test_poisoned_pool(pattern):
    with _context() as c:
        want, want_l = _poison_sequence(c)
    with _context(SPB_POOL_POISON=pattern) as c:
        got, got_l = _poison_sequence(c)
    assert got_l == want_l
    for g, w in zip(got, want):
        same(g[0], w[0])
        assert g[1:] == w[1:]


# ---- placement, size and errors ---------------------------------------------------------------------------------------------
def test_values_in_device_and_host_memory(ctx, orc):
    import torch
    rng = np.random.default_rng(41)
    A, B = _mix_case(rng, O.ADD, False)
    case = Case(A, ".", B, ".")
    plan = case.plan(ctx)
    try:
        av, bv = _vals(rng, A.n), _vals(rng, B.n)
        want, _ = case.fresh(ctx, av, bv)
        ta = torch.from_numpy(np.r_[0.0, av]).cuda()[1:]   # element offset 1: 8-byte, not 16-byte aligned
        tb = torch.from_numpy(np.r_[0.0, bv]).cuda()[1:]
        same(_down(plan.run(ta, tb)), want, "device, offset 1")
        same(_down(plan.run(av, bv)), want, "host")
        same(_down(plan.run(ta.data_ptr(), tb.data_ptr())), want, "raw pointers")
        same(_down(plan.run(av, tb)), want, "host A, device B")
    finally:
        plan.free()


def test_scale_2_23_plus_4097(ctx):
    """A config-5-family pattern of 2^23 + 4097 entries, hub rows and a run of 300: creation sorts with 9-bit row passes and
    the in-row sort."""
    rng = np.random.default_rng(43)
    m = 1 << 25
    n = (1 << 23) + 4097
    rows = rng.integers(0, m, n)
    rows[:6000] = 12345   # hub rows
    rows[6000:9000] = m - 1
    rows[9000:9300] = 777  # a run of 300 copies
    cols = (rows + rng.integers(-2, 3, n)) % m
    cols[9000:9300] = 778
    p = rng.permutation(n)
    A = Op((m, m), [rows[p], cols[p]])
    nb = 1 << 20
    br = rng.integers(0, m, nb)
    B = Op((m, m), [br, (br + rng.integers(-2, 3, nb)) % m])
    w = O.Coo((m,), [np.arange(0, m, 1, dtype=np.int32)[::7]], _vals(rng, len(range(0, m, 7))))
    case = Case(A, ".", B, ".", sj=w)
    av, bv = _vals(rng, A.n), _vals(rng, B.n)
    a2 = av.copy()
    a2[np.flatnonzero(A.idx[0] == 777)] = 0.0
    res = check_runs(ctx, case, [(av, bv), (a2, bv)])
    assert not res[0][0].fallback and res[1][0].fallback


def test_errors(ctx):
    import spsparse_b200 as sp
    from spsparse_b200._lib import MMPatternStats, SpbError
    rng = np.random.default_rng(47)
    A, B = _mix_case(rng, O.ADD, False)
    plan = Case(A, ".", B, ".").plan(ctx)
    try:
        with pytest.raises(ValueError):
            plan.run(np.ones(A.n - 1), np.ones(B.n))
        with pytest.raises(ValueError):
            plan.run(np.ones(A.n), np.ones(B.n + 1))
        with pytest.raises(TypeError):
            plan.run([1.0] * A.n, np.ones(B.n))
        import torch
        t = torch.zeros(A.n + 1, dtype=torch.float64, device="cuda")
        with pytest.raises(SpbError):
            plan.run(t.data_ptr() + 4, t.data_ptr())   # misaligned
        with pytest.raises(SpbError):
            plan.run(0, t.data_ptr())                  # null
        h, st = C.c_void_p(), MMPatternStats()
        assert ctx.lib.spb_mm_pattern_run(None, None, None, C.byref(h), C.byref(st)) != 0
        assert ctx.lib.spb_mm_pattern_run(plan.h, None, None, None, None) != 0
        assert ctx.lib.spb_mm_pattern_create(None, 1.0, None, None, b".", None, None, b".", None, 1, 0, C.byref(h), None) != 0
        dA, dB = A.up(ctx, np.ones(A.n)), B.up(ctx, np.ones(B.n))
        with pytest.raises(SpbError):
            sp.MultiplyPattern(ctx, 1.0, None, dA, ".", None, dB, "T", None)   # inner dimensions differ
        with pytest.raises(SpbError):
            sp.MultiplyPattern(ctx, 1.0, None, dA, ".", None, dB, ".", None, 7)  # unknown policy
        dA.free(); dB.free()
    finally:
        plan.free()


def test_cpp_multiply_pattern():
    exe = os.path.join(ROOT, "tests", "cpp", "_bin", "multiply_pattern_test")
    assert os.path.exists(exe), "tests/cpp/_bin/multiply_pattern_test is built by __graft_entry__.build()"
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    out = r.stdout[-4000:] + r.stderr[-2000:]
    assert r.returncode == 0 and "0 failure(s)" in out, out
