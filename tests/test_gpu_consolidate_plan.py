"""-m gpu tests of consolidate with a fixed index pattern (spb_consolidate_plan_*, sp.ConsolidatePlan): the pattern is sorted
once and every run with new values must equal spb_consolidate on an array with the plan's indices and those values, bit for
bit -- indices, values compared as bits (NaNs matched), the sort-order flag, and for rank 2 dim_beginnings -- and the oracle
where the size allows.  Covered: the reference fixtures, one plan with many value sets (zeros that empty whole runs, NaNs in
and after the leading run, infinities, exact cancellation, everything dropped), where the values live (device at element
offset 1 through a tensor and a raw pointer, host memory), a poisoned pool, tile boundaries of the kept count, a 2^23 + 4097
entry pattern, plan outputs fed to multiply, the fixed launch count of a run, the errors, and the C++ class."""
import contextlib
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _cases
import _golden
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M8 = 100_000_000
TILE = 4096


@pytest.fixture(scope="module")
def ctx():
    import spsparse_b200 as sp
    with sp.Context(0) as c:
        yield c


@contextlib.contextmanager
def _context(**env):
    """A context created with the given environment (SPB_POOL_POISON is read at context creation)."""
    import spsparse_b200 as sp
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        c = sp.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    try:
        yield c
    finally:
        c.close()


def _launches(ctx):
    n = C.c_uint64()
    assert ctx.lib.spb_ctx_launch_count(ctx.h, C.byref(n)) == 0
    return n.value


def _result(R):
    """(Coo, dim_beginnings or None) of a device result; frees it."""
    from _gpu import down
    out = down(R)
    db = R.dim_beginnings() if R.rank == 2 else None
    R.free()
    return out, db


def fresh(ctx, shape, idx, val, so, pol, zn):
    import spsparse_b200 as sp
    A = sp.CooArray.from_host(ctx, shape, idx, val)
    R = sp.consolidate(ctx, A, so, pol, zn)
    A.free()
    return _result(R)


def planned(plan, val, pol, zn):
    R, st = plan.run(val, pol, zn, stats=True)
    assert st.passes == 0 and st.n_in == plan.n
    out, db = _result(R)
    assert st.n_out == out.n
    return out, db


def same(got, want, what=""):
    g, gdb = got
    w, wdb = want
    assert _cases.same_coo(g, w), what
    assert g.sort_order == w.sort_order, what
    if wdb is not None:
        assert np.array_equal(gdb, wdb), what


def make_plan(ctx, shape, idx, so):
    """A plan over the pattern, built from an uploaded array that is freed before any run."""
    import spsparse_b200 as sp
    A = sp.CooArray.from_host(ctx, shape, idx, np.ones(len(idx[0])))
    plan = sp.ConsolidatePlan(ctx, A, so)
    A.free()
    return plan


# ---- 1. the reference's fixtures ------------------------------------------------------------------------------------
def test_fixtures_from_the_reference(ctx):
    p = _golden.pack("consolidate_cases")
    for s in range(int(p["count"])):
        a, want = _golden.get_coo(p, f"c{s}_in"), _golden.get_coo(p, f"c{s}_out")
        pol, zn, *so = (int(x) for x in p[f"c{s}_args"])
        plan = make_plan(ctx, a.shape, a.idx, tuple(so))
        g, db = planned(plan, a.val, pol, zn)
        plan.free()
        assert _cases.same_coo(g, want), f"consolidate case {s}"
        assert g.sort_order == tuple(so[:a.rank]), s
        if a.rank == 2:
            assert np.array_equal(db, p[f"c{s}_db"]), f"dim_beginnings case {s}"


# ---- 2. one plan, many value sets (and 7. the launch count of a run) --------------------------------------------------
def _run_mix(rank):
    """Runs of 1 .. 6000 duplicates, scrambled (the mix of test_duplicate_runs_of_every_length)."""
    rng = np.random.default_rng(41)
    lens = np.concatenate([rng.integers(1, 12, 3000), rng.integers(200, 330, 300), rng.integers(1000, 6000, 40),
                           [257, 256, 255, 264, 2048, 2304]])
    keys = rng.permutation(len(lens))
    run = np.repeat(np.arange(len(lens)), lens)         # run number of every entry, before scrambling
    o = rng.permutation(len(run))
    run = run[o]
    if rank == 2:
        return (200, 1 << 20), [keys[run] // 700, keys[run] % 700 * 1000], run
    return (1 << 22,), [keys[run] * 1000 + 7], run


def _value_sets(run):
    """name -> values for the entries of a pattern whose run number (distinct index tuple) is run[i]."""
    rng = np.random.default_rng(7)
    n, nruns = len(run), int(run.max()) + 1
    pos = 0.5 + rng.random(n)
    dead = rng.random(nruns) < 0.3                       # runs emptied by +-0
    zeros = pos.copy()
    zeros[dead[run]] = np.where(rng.random(int(dead[run].sum())) < 0.5, 0.0, -0.0)
    refill = 0.5 + rng.random(n)
    nan = rng.standard_normal(n)
    nan[rng.random(n) < 0.1] = np.nan
    nan[rng.random(n) < 0.1] = 0.0
    inf = rng.standard_normal(n)
    inf[rng.random(n) < 0.05] = np.inf
    inf[rng.random(n) < 0.05] = -np.inf
    cancel = rng.integers(-3, 4, n).astype(np.float64)    # small integers: many runs sum to exactly 0 (kept, C5)
    return {"nonzero": pos, "zeroed_runs": zeros, "refilled": refill, "nan": nan, "inf": inf, "cancel": cancel,
            "mixed": _cases._values(rng, n, "mixed"), "all_dropped": np.where(rng.random(n) < 0.5, 0.0, -0.0)}


def _with_leading_nans(shape, idx, vals, so):
    """The value set with every entry of the first few sorted runs NaN or 0: the leading run spans several tuples and
    tiles' worth of positions."""
    key = idx[so[0]].astype(np.int64) * (shape[so[1]] if len(shape) == 2 else 1) + (idx[so[1]] if len(shape) == 2 else 0)
    order = np.argsort(key, kind="stable")
    v = vals.copy()
    head = order[:9000]
    v[head] = np.where(np.arange(len(head)) % 3 == 0, 0.0, np.nan)
    return v


@pytest.mark.parametrize("rank,so", [(1, (0,)), (2, (0, 1)), (2, (1, 0))])
def test_one_plan_many_value_sets(ctx, orc, rank, so):
    shape, idx, run = _run_mix(rank)
    plan = make_plan(ctx, shape, idx, so)
    assert plan.n_runs == len(np.unique(run))
    sets = _value_sets(run)
    sets["leading_nan"] = _with_leading_nans(shape, idx, sets["nan"], so)
    for name, vals in sets.items():
        for pol in _cases.POLICIES:
            for zn in (0, 1):
                what = (name, pol, zn)
                l0 = _launches(ctx)
                got = planned(plan, vals, pol, zn)
                # no sort at run time: the bound (zero_nan only), the gather, the reduce, the long runs (ADD / REPLACE)
                assert _launches(ctx) - l0 == (1 if zn else 0) + 2 + (1 if pol in (O.ADD, O.REPLACE) else 0), what
                same(got, fresh(ctx, shape, idx, vals, so, pol, zn), what)
                want = orc.consolidate(O.Coo(shape, idx, vals), so, pol, zn)
                assert _cases.same_coo(got[0], want), what
                if name == "all_dropped":
                    assert got[0].n == 0
    plan.free()


def test_empty_pattern(ctx):
    import spsparse_b200 as sp
    for shape, so in (((4, 4), (0, 1)), ((4, 4), (1, 0)), ((9,), (0,))):
        A = sp.CooArray.from_host(ctx, shape, [np.zeros(0, np.int32)] * len(shape), np.zeros(0))
        plan = sp.ConsolidatePlan(ctx, A, so)
        A.free()
        assert plan.n_runs == 0
        R, st = plan.run(np.zeros(0), stats=True)
        assert R.size() == 0 and R.sort_order == so and st.n_out == 0    # algorithm.hpp:263,318 (C1)
        if len(shape) == 2:
            assert len(R.dim_beginnings()) == 0
        R.free()
        plan.free()


# ---- 3. where the values live ---------------------------------------------------------------------------------------
def test_values_in_device_and_host_memory(ctx):
    import torch
    shape, idx, run = _run_mix(2)
    vals = _value_sets(run)["mixed"]
    n = len(vals)
    plan = make_plan(ctx, shape, idx, (0, 1))
    buf = torch.empty(n + 1, dtype=torch.float64, device="cuda")
    buf[1:] = torch.from_numpy(vals)
    torch.cuda.synchronize()
    host = np.empty(n + 1)
    host[1:] = vals
    for pol in _cases.POLICIES:
        for zn in (0, 1):
            want = fresh(ctx, shape, idx, vals, (0, 1), pol, zn)
            same(planned(plan, buf[1:], pol, zn), want, ("tensor at offset 1", pol, zn))
            same(planned(plan, buf.data_ptr() + 8, pol, zn), want, ("device pointer at offset 1", pol, zn))
            same(planned(plan, host[1:], pol, zn), want, ("host at offset 1", pol, zn))
    plan.free()


# ---- 4. a poisoned pool ---------------------------------------------------------------------------------------------
def _poison_sequence(c):
    import spsparse_b200 as sp
    out = []
    for rank, so in ((2, (0, 1)), (2, (1, 0)), (1, (0,))):
        shape, idx, run = _run_mix(rank)
        sets = _value_sets(run)
        plan = make_plan(c, shape, idx, so)
        for vals in (sets["zeroed_runs"], sets["refilled"]):
            for pol in _cases.POLICIES:
                for zn in (0, 1):
                    R, st = plan.run(vals, pol, zn, stats=True)
                    out.append((_result(R), (st.n_in, st.n_kept, st.n_out, st.key_bits, st.passes)))
        plan.free()
    # and a larger pattern whose tiles are full: 3 * 4096 + 1 entries, a third of them zero
    rng = np.random.default_rng(5)
    n = 3 * TILE + 1
    idx = [rng.integers(0, 50, n), rng.integers(0, 60, n)]
    vals = np.where(rng.random(n) < 0.33, 0.0, rng.standard_normal(n))
    plan = make_plan(c, (50, 60), idx, (0, 1))
    R, st = plan.run(vals, sp.ADD, 1, stats=True)
    out.append((_result(R), (st.n_in, st.n_kept, st.n_out, st.key_bits, st.passes)))
    plan.free()
    return out, _launches(c)


@pytest.mark.parametrize("pattern", ["00", "ff", "7f"])
def test_poisoned_pool(pattern):
    with _context() as c:
        want, want_launches = _poison_sequence(c)
    with _context(SPB_POOL_POISON=pattern) as c:
        got, got_launches = _poison_sequence(c)
    assert got_launches == want_launches
    assert len(got) == len(want)
    for k, ((g, gst), (w, wst)) in enumerate(zip(got, want)):
        same(g, w, k)
        assert gst == wst, k


# ---- 5. tile boundaries and scale -------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [TILE - 1, TILE, TILE + 1, 3 * TILE + 1])
def test_kept_count_on_and_beside_tile_boundaries(ctx, orc, n):
    rng = np.random.default_rng(n)
    shape = (300, 400)
    idx = [rng.integers(0, 300, n), rng.integers(0, 400, n)]
    plan = make_plan(ctx, shape, idx, (0, 1))
    base = 0.5 + rng.random(n)
    for kept in sorted({k for k in (TILE - 1, TILE, TILE + 1, 2 * TILE - 1, 2 * TILE, 2 * TILE + 1, 3 * TILE - 1,
                                     3 * TILE, 3 * TILE + 1, n - 1, n) if 0 < k <= n}):
        vals = base.copy()
        vals[rng.permutation(n)[:n - kept]] = 0.0
        for pol, zn in ((O.ADD, 0), (O.REPLACE, 1), (O.LEAVE_ALONE, 0)):
            R, st = plan.run(vals, pol, zn, stats=True)
            assert st.n_kept == kept
            got = _result(R)
            same(got, fresh(ctx, shape, idx, vals, (0, 1), pol, zn), (kept, pol, zn))
            assert _cases.same_coo(got[0], orc.consolidate(O.Coo(shape, idx, vals), (0, 1), pol, zn)), (kept, pol, zn)
    plan.free()


def test_scale_2_23_plus_4097(ctx, orc):
    """2^23 + 4097 entries in a 10^8 x 10^8 shape: large enough that plan creation takes the 9-bit row passes plus the
    in-row sort (the organisation a fresh consolidate of the same pattern reports).  Hub rows, one run longer than 2^16, and
    dropped zeros."""
    import spsparse_b200 as sp
    rng = np.random.default_rng(23)
    n = (1 << 23) + 4097
    rows = rng.integers(0, M8, n)
    cols = rng.integers(0, M8, n)
    dup = rng.random(n) < 0.3                                   # duplicates of other entries
    src = rng.integers(0, n, int(dup.sum()))
    rows[dup], cols[dup] = rows[src], cols[src]
    hub = rng.random(n) < 0.02                                  # two hub rows of ~84k entries each
    rows[hub] = np.where(rng.random(int(hub.sum())) < 0.5, 12345, M8 - 1)
    cols[hub] = rng.integers(0, 5000, int(hub.sum()))
    rows[:70000], cols[:70000] = 777, 4242                      # one run of 70000 duplicates (> 2^16)
    o = rng.permutation(n)
    idx = [rows[o].astype(np.int32), cols[o].astype(np.int32)]
    shape = (M8, M8)
    plan = make_plan(ctx, shape, idx, (0, 1))
    v = rng.standard_normal(n)
    v[rng.random(n) < 0.1] = 0.0
    v[rng.random(n) < 0.01] = np.nan
    for pol in _cases.POLICIES:
        for zn in (0, 1):
            got = planned(plan, v, pol, zn)
            A = sp.CooArray.from_host(ctx, shape, idx, v)
            R, st = sp.consolidate(ctx, A, (0, 1), pol, zn, stats=True)
            A.free()
            assert st.digit_bits == 9 and st.passes == 3, (st.digit_bits, st.passes)   # the row passes + in-row sort
            same(got, _result(R), (pol, zn))
    want = orc.consolidate(O.Coo(shape, idx, v), (0, 1), O.ADD, True)
    assert _cases.same_coo(planned(plan, v, O.ADD, 1)[0], want)
    plan.free()


# ---- 6. plan outputs feed multiply ------------------------------------------------------------------------------------
def test_plan_outputs_feed_multiply(ctx, orc):
    import spsparse_b200 as sp
    from _gpu import down
    rng = np.random.default_rng(66)
    m, k, p = 300, 400, 350
    na, nb = 6000, 7000
    ia = [rng.integers(0, m, na), rng.integers(0, k, na)]
    ib = [rng.integers(0, k, nb), rng.integers(0, p, nb)]
    ibt = [ib[1], ib[0]]                                        # B stored transposed, for transpose_B = 'T'
    plan_a = make_plan(ctx, (m, k), ia, (0, 1))
    plan_b = make_plan(ctx, (k, p), ib, (1, 0))                 # the order multiply wants B in for '.'
    plan_bt = make_plan(ctx, (p, k), ibt, (0, 1))               # ... and for 'T'
    plan_bi = make_plan(ctx, (k, p), ib, (0, 1))                # by inner index: multiply_prepared
    va = 0.5 + rng.random(na)
    vb = rng.standard_normal(nb)
    va_gone = va.copy()
    va_gone[np.isin(ia[0], np.arange(0, m, 3))] = 0.0           # every third row of A vanishes
    for a_vals in (va, va_gone):
        Araw = sp.CooArray.from_host(ctx, (m, k), ia, a_vals)
        Braw = sp.CooArray.from_host(ctx, (k, p), ib, vb)
        want = down(sp.multiply(ctx, 1.0, None, Araw, ".", None, Braw, ".", None))
        Araw.free(); Braw.free()
        ref = orc.multiply_mm(1.0, None, O.Coo((m, k), ia, a_vals), ".", None, O.Coo((k, p), ib, vb), ".", None)
        assert _cases.same_coo(want, ref)
        Ap = plan_a.run(a_vals)
        for B, tB in ((plan_b.run(vb), "."), (plan_bt.run(vb), "T")):
            got = down(sp.multiply(ctx, 1.0, None, Ap, ".", None, B, tB, None))
            assert _cases.same_coo(got, want), tB
            B.free()
        Bi = plan_bi.run(vb)
        C_, _ = sp.multiply_prepared(ctx, 1.0, None, Ap, 0, None, Bi, 0, None)
        assert _cases.same_coo(down(C_), want)
        C_.free(); Bi.free(); Ap.free()
    for pl in (plan_a, plan_b, plan_bt, plan_bi):
        pl.free()


# ---- 8. errors --------------------------------------------------------------------------------------------------------
def test_errors(ctx):
    import spsparse_b200 as sp
    A = sp.CooArray.from_host(ctx, (4, 4), [[1, 2, 1], [1, 3, 1]], [1., 2., 3.])
    for bad in ((0, 0), (0, 2), (-1, 1)):
        with pytest.raises(sp.SpbError) as e:
            sp.ConsolidatePlan(ctx, A, bad)
        assert e.value.code == 2, bad
    plan = sp.ConsolidatePlan(ctx, A, (0, 1))
    h = C.c_void_p()
    assert ctx.lib.spb_consolidate_plan_run(plan.h, None, 1, 0, C.byref(h), None) == 2      # null values, n > 0
    for pol in (-1, 3, 7):
        with pytest.raises(sp.SpbError) as e:
            plan.run(np.ones(3), pol)
        assert e.value.code == 2, pol
    plan.free()
    A.free()
    # out-of-bounds indices: refused at creation, as spb_consolidate refuses them
    B = sp.CooArray.from_host(ctx, (4, 4), [[1, 4], [1, 1]], [1., 1.])
    with pytest.raises(sp.SpbError) as e:
        sp.ConsolidatePlan(ctx, B, (0, 1))
    assert e.value.code == 2
    with pytest.raises(sp.SpbError):
        sp.consolidate(ctx, B, (0, 1))
    B.free()


# ---- 9. the C++ class -------------------------------------------------------------------------------------------------
def test_cpp_consolidate_plan():
    exe = os.path.join(ROOT, "tests", "cpp", "_bin", "consolidate_plan_test")
    assert os.path.exists(exe), "tests/cpp/_bin/consolidate_plan_test is built by __graft_entry__.build()"
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    out = r.stdout[-4000:] + r.stderr[-2000:]
    assert r.returncode == 0 and "0 failure(s)" in out, out
