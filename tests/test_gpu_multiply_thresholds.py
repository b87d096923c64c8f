"""-m gpu: multiply at the thresholds where it changes bin, kernel build or branch (cases: tests/_thresholds.py).  Every
result equals the oracle's bit for bit, and every case pins the path it took: the bin totals of spb_mm_stats, launch
count differences between runs with and without a branch, and (hash numeric kernel) the SPB_TRACE counts of work items,
steps, warp-pipelined steps and entry barriers, read from a child process because the library reads SPB_TRACE once."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _cases
import _thresholds as T

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _launches(ctx):
    n = C.c_uint64()
    assert ctx.lib.spb_ctx_launch_count(ctx.h, C.byref(n)) == 0
    return n.value


def _run(ctx, case, A=None):
    """One multiply of the case: (result, stats, kernels launched).  A: an uploaded A handle to use instead."""
    import spsparse_b200 as sp
    from _gpu import up, down
    hs = [up(ctx, case[x]) for x in ("si", "sj", "B", "sk")]
    a = A if A is not None else up(ctx, case["A"])
    n0 = _launches(ctx)
    R, st = sp.multiply(ctx, case["C"], hs[0], a, ".", hs[1], hs[2], ".", hs[3], stats=True)
    n = _launches(ctx) - n0
    got = down(R)
    for h in hs + [R] + ([a] if A is None else []):
        if h is not None:
            h.free()
    return got, st, n


def _want(orc, case):
    return orc.multiply_mm(case["C"], case["si"], case["A"], ".", case["sj"], case["B"], ".", case["sk"])


def _check(case, want, got, st, onepass=False):
    assert _cases.same_coo(got, want), case["name"]
    e = case["expect"]
    assert st.rows_merge == e["merge"] and st.nnz_c == want.n, (case["name"], st.asdict(), e)
    if not onepass:   # (the one-pass merge reports its own counters only)
        assert (st.rows_esc, st.rows_hash, st.products_hash, st.products_esc) == \
               (e["esc"], e["hash"], e["products_hash"], e["products_esc"]), (case["name"], st.asdict(), e)


@pytest.fixture
def context(monkeypatch):
    """Context factory: the knobs read at context creation set first."""
    import spsparse_b200 as sp
    made = []

    def make(**env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        c = sp.Context(0)
        made.append(c)
        return c
    yield make
    for c in made:
        c.close()


PLAIN = [T.merge_bin, T.hash_vs_esc] + [lambda n=n: T.bitmap_width(n) for n in (T.HASH_MAX_COLS, T.HASH_MAX_COLS + 1, 2 * T.HASH_MAX_COLS + 1)]


@pytest.mark.parametrize("build", PLAIN, ids=["merge_bin", "hash_vs_esc", "bitmap_W", "bitmap_W+1", "bitmap_2W+1"])
def test_bins_at_their_thresholds(orc, context, monkeypatch, build):
    """Merge (8 / 9 entries, 1024 / 1025 products, an empty or scalej-masked ninth entry, rows zeroed by scalei), hash
    versus ESC (511 / 512 / 513 products) and the bitmap's width (W, W+1, 2W+1 columns, outputs at W-1, W, n_cols-1).
    Wide matrices run with k_hash_win_bounds and with the bitmap kernel's own window search: one launch apart."""
    case = build()
    want = _want(orc, case)
    ctx = context()
    got, st, n = _run(ctx, case)
    _check(case, want, got, st)
    monkeypatch.setenv("SPB_HASH_NO_WIN_BOUNDS", "1")
    got, st, n_own = _run(ctx, case)
    _check(case, want, got, st)
    n_win = -(-case["B"].shape[1] // T.HASH_MAX_COLS)
    assert n - n_own == (1 if n_win > 1 and case["expect"]["hash"] else 0), (n, n_own)


@pytest.mark.parametrize("stage", [16, 8, 4])
def test_merge_staging_flushes(orc, context, monkeypatch, stage):
    """Rows of 15, 16, 17, 32, 33 outputs and exact cancellations on the first / last output of a flushed run; the same
    matrix without cancellation launches no compaction."""
    case = T.merge_staging()
    want = _want(orc, case)
    ctx = context()
    monkeypatch.setenv("SPB_MERGE_STAGE", str(stage))
    got, st, n = _run(ctx, case)
    _check(case, want, got, st)
    assert want.n < sum(T.analyse(case)["outputs"])   # tombstones were written ...
    plain = T.merge_staging(cancel=False)
    got, st, n_plain = _run(ctx, plain)
    _check(plain, _want(orc, plain), got, st)
    assert st.nnz_c == sum(T.analyse(plain)["outputs"]) and n - n_plain >= 3   # ... and compacted: flags, scan, compaction


@pytest.mark.parametrize("longest", range(1, 9))
def test_merge_kernel_builds(orc, context, longest):
    """Longest A row 1..8 (kernels for 2/4/6/8 lists).  Mean B row > 16: the longest row is found up front (k_row_maxlen,
    one launch); <= 16: the count kernel reports it.  Once known, it is cached with A's row structure."""
    import spsparse_b200 as sp
    from _gpu import up
    ctx = context()
    cases = {lb: T.nl_build(longest, lb) for lb in (False, True)}
    cases[True]["A"] = cases[False]["A"]   # one A for both: rows of the same 16 inner indices
    wants = {lb: _want(orc, c) for lb, c in cases.items()}

    def fresh():
        a = up(ctx, cases[False]["A"])
        ac = sp.consolidate(ctx, a, (0, 1))
        a.free()
        return ac

    first_minus_second = {}
    for lb in (False, True):
        A = fresh()
        runs = []
        for _ in range(2):
            got, st, n = _run(ctx, cases[lb], A)
            _check(cases[lb], wants[lb], got, st)
            runs.append(n)
        A.free()
        first_minus_second[lb] = runs[0] - runs[1]
    assert first_minus_second[True] - first_minus_second[False] == 1, first_minus_second
    # short B rows first (the count kernel records the longest row), then long ones: no k_row_maxlen
    A = fresh()
    _run(ctx, cases[False], A)
    got, st, n_after_short = _run(ctx, cases[True], A)
    _check(cases[True], wants[True], got, st)
    got, st, n_again = _run(ctx, cases[True], A)
    A.free()
    assert n_after_short == n_again


@pytest.mark.parametrize("kind", ["pass", "outputs", "products"])
def test_one_pass_merge_and_its_fallback(orc, context, monkeypatch, kind):
    """SPB_MERGE_ONEPASS=1 takes short rows of <= 16 outputs in one kernel; a row of 17 outputs or of 1025 products makes it
    fail fast, and the two-pass answer follows (two launches more: the longest-row pass and the failed kernel)."""
    case = T.onepass(kind)
    want = _want(orc, case)
    ctx = context()
    got, st, n_two = _run(ctx, case)
    _check(case, want, got, st)
    monkeypatch.setenv("SPB_MERGE_ONEPASS", "1")
    got, st, n_one = _run(ctx, case)
    _check(case, want, got, st, onepass=kind == "pass")
    if kind == "pass":
        assert st.ms_symbolic == 0.0 and n_one < n_two
    else:
        assert n_one == n_two + 2


@pytest.mark.parametrize("f", [8191, 8192, 8193])
@pytest.mark.parametrize("collapse", [False, True])
def test_small_row_sort_capacity(orc, context, monkeypatch, f, collapse):
    """A row of 8191 / 8192 / 8193 products in a matrix wider than the bitmap, next to a row of 12000: rows of at most 8192
    products are listed by k_hash_symbolic_small (one launch more than with SPB_HASH_SMALL=0)."""
    case = T.small_sort(f, collapse)
    want = _want(orc, case)
    ctx = context()
    got, st, n = _run(ctx, case)
    _check(case, want, got, st)
    monkeypatch.setenv("SPB_HASH_SMALL", "0")
    got, st, n_bitmap = _run(ctx, case)
    _check(case, want, got, st)
    assert n - n_bitmap == (1 if case["expect"]["small"] else 0)


@pytest.mark.parametrize("words", [4607, 4608, 4609])
@pytest.mark.parametrize("walk", [None, "0"])
def test_sparse_bitmap_walk_capacity(orc, context, monkeypatch, words, walk):
    """Outputs in 4607 / 4608 / 4609 bitmap words, with the sparse walk allowed and with SPB_HASH_SPARSE_WALK=0.  Only the
    result and the bin are observable: which walk a unit took is not (both give the same result), so an off-by-one in the
    walk's capacity test would pass; an overflow of its 4608-entry list would not."""
    case = T.sparse_walk(words)
    want = _want(orc, case)
    if walk is not None:
        monkeypatch.setenv("SPB_HASH_SPARSE_WALK", walk)
    got, st, n = _run(context(), case)
    _check(case, want, got, st)


@pytest.mark.parametrize("offset", [0, 1])
def test_esc_chunk_boundary(orc, context, offset):
    """ESC rows whose products reach 2^27 (one chunk) exactly at a row end, or one product past it: two chunks.  With
    SPB_ESC_CHUNK=2^28 the same input is one chunk and launches fewer kernels.  Where the cut falls is not observable
    from outside; tests/test_thresholds_cpu.py checks that the ESC prefix is 2^27 (+ 1) at the end of ESC_BOUNDARY_ROW."""
    case = T.esc_chunk(offset)
    want = _want(orc, case)
    got, st, n = _run(context(), case)
    _check(case, want, got, st)
    assert st.products_esc == T.ESC_CHUNK + offset + 1000 * 511
    got, st, n_one = _run(context(SPB_ESC_CHUNK=str(1 << 28)), case)
    _check(case, want, got, st)
    assert n > n_one


@pytest.mark.parametrize("delta", [-2, 0, 1])
def test_row_panels_cut_at_a_row_start(orc, context, delta):
    """Two panels whose chunk is one product before, exactly on, or one product after the first product of row
    PANEL_CUT_ROW: the second panel starts at that row, that row, and the next.  Other max_products values too: the
    panel count and every panel's first row follow k_panel_bounds' rule (_thresholds.panel_rows), and the panels
    concatenated are the oracle's product."""
    import spsparse_b200 as sp
    from _gpu import up
    from test_gpu_multiply import gpu_mm_panels
    case = T.panels(delta)
    want = _want(orc, case)
    prod = T.analyse(case, columns=False)["products"]
    F = int(prod.sum())
    ctx = context()
    for mp in (-(-F // 2), F - 1, F // 7, F // 59, 1):
        rows = T.panel_rows(prod, mp)
        if mp in (-(-F // 2), F - 1):
            assert rows == [0, T.PANEL_CUT_ROW + (delta > 0)]
        hs = [up(ctx, case[x]) for x in ("A", "B")]
        plan = sp.MultiplyPlan(ctx, case["C"], None, hs[0], ".", None, hs[1], ".", None, max_products_per_panel=mp)
        got_rows = [plan.info(p)[0] for p in range(plan.n_panels)]
        plan.free()
        for h in hs:
            h.free()
        assert got_rows == rows, (mp, got_rows, rows)
        got, n_panels = gpu_mm_panels(ctx, case["C"], None, case["A"], ".", None, case["B"], ".", None, max_products=mp)
        assert n_panels == len(rows) and _cases.same_coo(got, want), mp


# ---- hash numeric kernel, traced: run in a child process started with SPB_TRACE=1 ------------------------------------
def _traced_cases():
    out = [T.hash_items(v, s) for v in (2, 1, 0) for s in (False, True)]
    return out + [T.hash_steps(v, s) for v in (2, 1, 0) for s in (31, 32, 33, 0)]


def _child():
    """Runs every traced case in its own context; prints one JSON line per case to stdout, a marker to stderr before it."""
    from oracle import oracle as O
    import spsparse_b200 as sp
    orc = O.port()
    for case in _traced_cases():
        os.environ.update(case["ctx_env"])
        want = _want(orc, case)
        with sp.Context(0) as ctx:
            print(f"@@case {case['name']}", file=sys.stderr, flush=True)
            got, st, n = _run(ctx, case)
            sys.stderr.flush()
        print(json.dumps(dict(name=case["name"], same=_cases.same_coo(got, want), nnz=want.n, stats=st.asdict())), flush=True)


def _parse_trace(err):
    import re
    out, cur = {}, None
    for line in err.splitlines():
        if line.startswith("@@case "):
            cur = line.split()[1]
        m = re.search(r"mm hash numeric: (\d+) items \((\d+)\), (\d+) staged chunks, (\d+) steps \((\d+) warp-pipelined\), (\d+) entry barriers", line)
        if m and cur:
            v = [int(x) for x in m.groups()]
            out[cur] = dict(items=v[0], chunks=v[2], steps=v[3], piped=v[4], barriers=v[5])
    return out


def test_hash_items_and_step_order_traced():
    """Hash rows of CAP-1 .. 2 CAP+1 outputs for every variant (with and without a scalek that excludes columns, with
    exact cancellation on items' first and last outputs), and rows whose steps span 31 / 32 / 33 entries or put 32 lanes
    on one output: results bit-identical, and the kernel's own counts of items, steps, warp-pipelined steps and entry
    barriers equal a replay of its schedule (_thresholds.hash_trace)."""
    env = dict(os.environ, SPB_TRACE="1")
    code = f"import sys; sys.path[:0] = [{HERE!r}, {os.path.dirname(HERE)!r}]; import test_gpu_multiply_thresholds as t; t._child()"
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]
    trace = _parse_trace(p.stderr)
    results = {r["name"]: r for r in map(json.loads, p.stdout.splitlines())}
    for case in _traced_cases():
        r = results[case["name"]]
        e = case["expect"]
        st = r["stats"]
        assert r["same"], case["name"]
        assert (st["rows_merge"], st["rows_esc"], st["rows_hash"], st["products_hash"], st["nnz_c"]) == \
               (e["merge"], e["esc"], e["hash"], e["products_hash"], r["nnz"]), (case["name"], st)
        variant = int(case["ctx_env"]["SPB_HASH_VARIANT"])
        assert trace[case["name"]] == T.hash_trace(case, variant), case["name"]
