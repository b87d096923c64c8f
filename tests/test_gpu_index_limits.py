"""-m gpu tests at the int32 index limit: every extent exactly 2^31, so index 2^31 - 1 is legal in every dimension (the
reference's IndexT is int32).  Indices crowd both ends of the range.  Every multiply bin (register merge in all its builds,
LOCAL and one-pass variants, expand-sort-compress, the bitmap + hash-accumulator bin in its ~1366 column windows), row panels,
prepared / compressed operands and the one-rank row partition are compared bit for bit with the oracle run on the relabelled
problem (tests/_limits.py; checked against the oracle's loop nest in tests/test_index_limits_cpu.py).  Consolidate and the row
structure are tested with a 31-bit column part.

Memory: a dense pointer over 2^31 inner indices is 8 GB, every densified scale vector 16 GB (scalej adds a 2 GB mask), so no
call here uses all three scale vectors at once (at most ~42 GB per call); the context's cached blocks are handed back at the end."""
import numpy as np
import pytest

import _cases
import _limits as L
from oracle import oracle as O

pytestmark = pytest.mark.gpu

N, TOP = L.N, L.TOP
TS = [(".", "."), ("T", "."), (".", "T"), ("T", "T")]
# scale vectors of one call: si and sk together, or sj alone; entry 2^31-1 present and non-zero, present and 0, or absent
SCALES = [None, ("ik", "nonzero"), ("ik", "zero"), ("ik", "absent"), ("j", "nonzero"), ("j", "zero"), ("j", "absent")]


@pytest.fixture(scope="module")
def ctx():
    import spsparse_b200 as sp
    with sp.Context(0) as c:
        yield c
        c.trim()


def _scales(A, B, which, seed):
    """(si, sj, sk) over the indices op(A) / op(B) use, for SCALES entry `which`."""
    if which is None:
        return None, None, None
    rng = np.random.default_rng(seed)
    dims, mode = which
    si = L.scale_vector(rng, A.idx[0], mode) if "i" in dims else None
    sj = L.scale_vector(rng, np.concatenate([A.idx[1], B.idx[0]]), mode) if "j" in dims else None
    sk = L.scale_vector(rng, B.idx[1], mode) if "k" in dims else None
    return si, sj, sk


def _case(seed, roles, tA, tB, which=None, **kw):
    """Arguments of multiply (stored operands under the transpose flags, scale vectors) for op(A) x op(B) from
    _limits.mm_inputs."""
    A, B = L.mm_inputs(seed, roles, **kw)
    si, sj, sk = _scales(A, B, which, seed)
    return (1.5, si, L.transposed(A, tA), tA, sj, L.transposed(B, tB), tB, sk)


def _mm(ctx, orc, args):
    """GPU multiply of args, compared with the relabelled oracle; returns (stats, reference product)."""
    import spsparse_b200 as sp
    from _gpu import up, down
    Cst, si, A, tA, sj, B, tB, sk = args
    hs = [up(ctx, x) for x in (si, A, sj, B, sk)]
    R, st = sp.multiply(ctx, Cst, hs[0], hs[1], tA, hs[2], hs[3], tB, hs[4], stats=True)
    got = down(R)
    for h in hs + [R]:
        if h is not None:
            h.free()
    want, wst = L.relabeled_mm(orc, *args, want_stats=True)
    assert st.products == wst["F"]
    assert _cases.same_coo(got, want)
    return st, want


def _top_outputs_checked(want):
    """The product really has outputs in column 2^31-1 (one of them NaN) -- what the merge used to lose."""
    top = want.idx[1] == TOP
    return top.any() and np.isnan(want.val[top]).any()


@pytest.mark.parametrize("which", SCALES)
def test_default_bins(ctx, orc, which):
    """The default bins (short rows: the register merge) with 2^31-1 as row, inner index, column, and all three; both
    transpose flags of both operands."""
    for roles in ("i", "j", "k", "ijk"):
        for t, (tA, tB) in enumerate(TS):
            args = _case(31 + t, roles, tA, tB, which)
            st, want = _mm(ctx, orc, args)
            assert st.rows_merge > 0 and st.rows_esc == 0 and st.rows_hash == 0, (roles, tA, tB)
            if which is None and "k" in roles:
                assert _top_outputs_checked(want), (roles, tA, tB)


@pytest.mark.parametrize("nl", [2, 4, 6, 8])
def test_every_merge_build(orc, monkeypatch, nl):
    """Each register-merge build (NL = 2, 4, 6, 8 lists for the count and the numeric kernel) on rows of NL - 1 and NL
    inner indices; the 8-list numeric kernel also with its 8- and 4-output staging."""
    import spsparse_b200 as sp
    monkeypatch.setenv("SPB_MERGE_NL_COUNT", str(nl))
    monkeypatch.setenv("SPB_MERGE_NL_NUMERIC", str(nl))
    with sp.Context(0) as c2:
        for stage in ([None, "8", "4"] if nl == 8 else [None]):
            if stage:
                monkeypatch.setenv("SPB_MERGE_STAGE", stage)
            for ln in (nl - 1, nl):
                for roles, (tA, tB), which in (("k", (".", "."), None), ("ijk", ("T", "T"), None), ("ijk", (".", "T"), ("ik", "nonzero")),
                                               ("jk", ("T", "."), ("j", "nonzero"))):
                    args = _case(100 * nl + ln, roles, tA, tB, which, row_len=ln)
                    st, want = _mm(c2, orc, args)
                    assert st.rows_merge > 0 and st.rows_esc == 0 and st.rows_hash == 0
                    if which is None:
                        assert _top_outputs_checked(want)
        c2.trim()


@pytest.mark.parametrize("inner_lo", [0, N - 600])
def test_local_merge(orc, monkeypatch, inner_lo):
    """SPB_MERGE_LOCAL=1: all inner indices within 600 of each other (at the bottom of the range, or ending at 2^31-1), so
    the block stages its stretch of B in shared memory; columns up to 2^31-1."""
    import spsparse_b200 as sp
    monkeypatch.setenv("SPB_MERGE_LOCAL", "1")
    with sp.Context(0) as c2:
        for ln in (2, 4, 6, 8):
            for (tA, tB), which in (((".", "."), None), (("T", "T"), ("ik", "nonzero")), (("T", "."), ("j", "zero"))):
                args = _case(7 + ln, "ik", tA, tB, which, row_len=ln, inner_lo=inner_lo)
                st, want = _mm(c2, orc, args)
                assert st.rows_merge > 0 and st.rows_esc == 0 and st.rows_hash == 0
                if which is None:
                    assert _top_outputs_checked(want)
        c2.trim()


def test_one_pass_merge(orc, monkeypatch):
    """SPB_MERGE_ONEPASS=1: rows of at most 16 outputs (A rows of 1..4 entries, B rows of at most 3), so the one-pass kernel
    keeps its result (no symbolic phase was timed)."""
    import spsparse_b200 as sp
    monkeypatch.setenv("SPB_MERGE_ONEPASS", "1")
    with sp.Context(0) as c2:
        for ln in (1, 2, 3, 4):
            for roles in ("k", "ijk"):
                for (tA, tB), which in (((".", "."), None), (("T", "T"), ("ik", "nonzero")), ((".", "T"), ("j", "nonzero"))):
                    args = _case(50 + ln, roles, tA, tB, which, row_len=ln, b_len=3)
                    st, want = _mm(c2, orc, args)
                    assert st.rows_merge > 0 and st.rows_esc == 0 and st.rows_hash == 0 and st.ms_symbolic == 0.0
                    if which is None:
                        assert _top_outputs_checked(want)
        c2.trim()


def _esc_env(monkeypatch, merge_max, chunk, hash_min="off"):
    monkeypatch.setenv("SPB_MERGE_MAX_PRODUCTS", str(merge_max))
    monkeypatch.setenv("SPB_ESC_CHUNK", str(chunk))
    monkeypatch.setenv("SPB_HASH_MIN_PRODUCTS", str(hash_min))


def test_expand_sort_compress(orc, monkeypatch):
    """Every row through expand-sort-compress, in chunks of 37 products: keys (row number, column) with a 31-bit column part."""
    import spsparse_b200 as sp
    _esc_env(monkeypatch, 0, 37)
    with sp.Context(0) as c2:
        for roles in ("k", "ijk", "i"):
            for t, (tA, tB) in enumerate(TS):
                for which in (None, ("ik", "nonzero"), ("j", "zero")):
                    st, want = _mm(c2, orc, _case(70 + t, roles, tA, tB, which))
                    assert st.rows_esc > 0 and st.rows_merge == 0 and st.rows_hash == 0
        c2.trim()


@pytest.mark.parametrize("variant,small", [(0, "0"), (1, "0"), (2, "0"), (2, "1"), (0, "1")])
def test_hash_bin(orc, monkeypatch, variant, small):
    """Every row through the bitmap + hash-accumulator bin: SPB_HASH_SMALL=0 runs the bitmap in ~1366 column windows of
    2^31 columns, "1" lists the columns by a shared-memory sort; rows cut into work items of at most 3 outputs."""
    import spsparse_b200 as sp
    _esc_env(monkeypatch, 0, 1 << 27, hash_min=0)
    monkeypatch.setenv("SPB_HASH_VARIANT", str(variant))
    monkeypatch.setenv("SPB_HASH_SMALL", small)
    monkeypatch.setenv("SPB_HASH_ITEM_CAP", "3")
    with sp.Context(0) as c2:
        for roles in ("k", "ijk"):
            for t, (tA, tB) in enumerate(TS):
                for which in (None, ("ik", "zero"), ("j", "nonzero")):
                    st, want = _mm(c2, orc, _case(90 + t + variant, roles, tA, tB, which))
                    assert st.rows_hash > 0 and st.rows_merge == 0 and st.rows_esc == 0
                    if which is None:
                        assert _top_outputs_checked(want)
        c2.trim()


@pytest.mark.parametrize("max_products", [1, 1 << 30])
def test_row_panels(ctx, orc, max_products):
    """MultiplyPlan: the panels concatenated are the product (one row of op(A) per panel with max_products = 1, one panel
    with 2^30)."""
    import spsparse_b200 as sp
    from _gpu import up, down
    for roles, (tA, tB), which in (("ijk", (".", "."), None), ("ik", ("T", "T"), ("ik", "nonzero")), ("jk", (".", "T"), ("j", "zero"))):
        Cst, si, A, tA, sj, B, tB, sk = _case(11, roles, tA, tB, which)
        want = L.relabeled_mm(orc, Cst, si, A, tA, sj, B, tB, sk)
        hs = [up(ctx, x) for x in (si, A, sj, B, sk)]
        plan = sp.MultiplyPlan(ctx, Cst, hs[0], hs[1], tA, hs[2], hs[3], tB, hs[4], O.ADD, False, max_products)
        hs[1].free(); hs[3].free()
        parts = []
        for p in range(plan.n_panels):
            R = plan.panel(p)
            parts.append(down(R))
            R.free()
        shape, n_panels = plan.shape, plan.n_panels
        plan.free()
        for h in (hs[0], hs[2], hs[4]):
            if h is not None:
                h.free()
        got = O.Coo(shape, [np.concatenate([c.idx[d] for c in parts]) for d in (0, 1)], np.concatenate([c.val for c in parts]))
        assert _cases.same_coo(got, want), (roles, tA, tB, n_panels)
        assert (n_panels > 1) == (max_products == 1), n_panels


def test_prepared_compressed_b_and_one_rank_partition(ctx, orc):
    """multiply_prepared with B in compressed form (wrap_csr over its 2^31 + 1 pointer) and the row partition with one rank
    (row_lo = [0, 2^31]): the same product."""
    import spsparse_b200 as sp
    from spsparse_b200.dist import RowPartition
    from _gpu import up, down
    for roles, which in (("ijk", None), ("ijk", ("ik", "nonzero")), ("jk", ("j", "zero"))):
        Cst, si, A, _, sj, B, _, sk = _case(21, roles, ".", ".", which)
        want = L.relabeled_mm(orc, Cst, si, A, ".", sj, B, ".", sk)
        hs = [up(ctx, x) for x in (si, A, sj, B, sk)]
        Ac, Bc = sp.consolidate(ctx, hs[1], (0, 1)), sp.consolidate(ctx, hs[3], (0, 1))
        (_, p1), pv = Bc.device_ptrs()
        ptr, ext = Bc.dense_ptr()
        assert ext == N
        Bcsr = sp.CooArray.wrap_csr(ctx, (N, N), 0, ptr, p1, pv, Bc.size())
        C1, st1 = sp.multiply_prepared(ctx, Cst, hs[0], Ac, 0, hs[2], Bcsr, 0, hs[4])
        assert _cases.same_coo(down(C1), want), (roles, which)
        for h in (C1, Bcsr, Ac, Bc):
            h.free()
        rp = RowPartition(ctx, 0, 1, N, B.n + 1)
        C2, _ = rp.multiply(Cst, hs[0], hs[1], hs[2], hs[3], hs[4])
        assert _cases.same_coo(down(C2), want), (roles, which)
        C2.free()
        rp.close()
        for h in hs:
            if h is not None:
                h.free()


def test_matrix_vector(ctx, orc):
    """Matrix x vector: row 2^31-1, inner index 2^31-1, V index 2^31-1, both transpose flags, si and sj with entries at the end."""
    import spsparse_b200 as sp
    from _gpu import up, down
    for seed in range(6):
        rng = np.random.default_rng(600 + seed)
        flavour = ["pos", "int", "mixed"][seed % 3]
        n = 400
        ai, aj = L.crowded(rng, n, pool=50), L.crowded(rng, n, pool=50)
        Aop = O.Coo((N, N), [ai, aj], _cases._values(rng, n, flavour))
        vi = np.append(L.crowded(rng, 150, pool=50), [TOP, TOP])   # a duplicate at 2^31-1: consolidated first
        V = O.Coo((N,), [vi], _cases._values(rng, len(vi), flavour))
        si = L.scale_vector(rng, ai, ["nonzero", "zero", "absent"][seed % 3]) if seed % 2 == 0 else None
        sj = L.scale_vector(rng, np.concatenate([aj, vi]), ["absent", "nonzero", "zero"][seed % 3]) if seed % 3 != 2 else None
        for tA in (".", "T"):
            A = L.transposed(Aop, tA)
            want = orc.multiply_mv(1.5, si, A, tA, sj, V)
            hs = [up(ctx, x) for x in (si, A, sj, V)]
            R = sp.multiply(ctx, 1.5, hs[0], hs[1], tA, hs[2], hs[3])
            got = down(R)
            for h in hs + [R]:
                if h is not None:
                    h.free()
            assert got.shape == (N,) and _cases.same_coo(got, want), (seed, tA)


# ---- consolidate and row structure with a 31-bit column part ---------------------------------------------------------
def _crowded_coo(rng, shape, n, edge_frac, flavour, pool=None):
    idx = []
    for _ in shape:
        x = rng.integers(0, N, n) if pool is None else rng.integers(0, N, pool)[rng.integers(0, pool, n)]
        e = rng.random(n) < edge_frac
        x[e] = L.EDGE[rng.integers(0, len(L.EDGE), int(e.sum()))]
        idx.append(x)
    return O.Coo(shape, idx, _cases._values(rng, n, flavour))


def test_consolidate_large_default_path(ctx, orc):
    """2^23 + 4097 entries in a 2^31 x 2^31 shape, 5 % of every index at the ends of the range (hub rows of ~70 000 entries at
    0, 1, 2, 2^31-3 .. 2^31-1): the default organisation (row-digit passes + in-row column sort; 31-bit row part in four 8-bit
    passes), compared in full with the oracle, both orders."""
    import spsparse_b200 as sp
    from _gpu import up, down
    rng = np.random.default_rng(31)
    n = (1 << 23) + 4097
    a = _crowded_coo(rng, (N, N), n, 0.05, "mixed")
    dup = rng.random(n) < 0.2
    src = rng.integers(0, n, n)
    for d in range(2):
        a.idx[d][dup] = a.idx[d][src[dup]]
    for so, pol, zn in (((0, 1), O.ADD, 1), ((1, 0), O.REPLACE, 0)):
        A = up(ctx, a)
        R, st = sp.consolidate(ctx, A, so, pol, zn, stats=True)
        got, db = down(R), R.dim_beginnings()
        A.free(); R.free()
        assert st.key_bits == 62 and st.digit_bits == 8 and st.passes == 4, (st.key_bits, st.digit_bits, st.passes)
        want = orc.consolidate(a, so, pol, zn)
        assert _cases.same_coo(got, want), (so, pol, zn)
        assert np.array_equal(db, orc.dim_beginnings(want))


@pytest.mark.parametrize("mode,walk,fused,rwarp,r9", [("1", "1", "0", None, None), ("1", "0", "0", None, None), ("1", "2", "0", None, None),
                                                      ("1", "1", "1", None, None), ("1", "1", "0", "0", None), ("1", "0", "0", "2", None),
                                                      ("0", "0", "0", "2", None), ("0", "0", "0", None, "1")])
def test_consolidate_forced_organisations(ctx, orc, monkeypatch, mode, walk, fused, rwarp, r9):
    """The sort's organisations forced on a 2^31 x 2^31 shape with indices at both ends: row passes + in-row column sort (each
    in-row kernel, fused into the reduce or not), full-key passes, each reduce kernel, 9-bit digits over the 62-bit key; all policies, zero_nan,
    both orders, sorted_permutation."""
    import spsparse_b200 as sp
    from _gpu import up, down
    monkeypatch.setenv("SPB_SEGMENT_SORT", mode)
    monkeypatch.setenv("SPB_SEGMENT_WALK", walk)
    monkeypatch.setenv("SPB_FUSED_REDUCE", fused)
    if rwarp is not None:
        monkeypatch.setenv("SPB_REDUCE_WARP", rwarp)
    if r9 is not None:
        monkeypatch.setenv("SPB_RADIX9", r9)
    rng = np.random.default_rng(41)
    cases = [_crowded_coo(rng, (N, N), 60000, 0.3, "mixed", pool=20000),     # duplicates; rows at the ends of thousands of entries
             _crowded_coo(rng, (N, N), 50000, 0.02, "int", pool=30000),      # short rows, a few dozen at the ends
             _crowded_coo(rng, (N, N), 4097, 0.5, "pos", pool=500)]
    for s, a in enumerate(cases):
        for so in ((0, 1), (1, 0)):
            for pol in _cases.POLICIES:
                zn = (s + pol) % 2
                A = up(ctx, a)
                R = sp.consolidate(ctx, A, so, pol, zn)
                got, db = down(R), R.dim_beginnings()
                A.free(); R.free()
                want = orc.consolidate(a, so, pol, zn)
                assert _cases.same_coo(got, want), (s, so, pol)
                assert np.array_equal(db, orc.dim_beginnings(want)), (s, so, pol)
            A = up(ctx, a)
            perm = A.sorted_permutation(so)
            A.free()
            assert np.array_equal(perm, orc.sorted_permutation(a, so)), (s, so)


def test_consolidate_rank1_full_extent(ctx, orc):
    """Rank 1, extent 2^31, 300 000 entries (many tiles) crowding both ends: every policy, zero_nan on and off."""
    import spsparse_b200 as sp
    from _gpu import up, down
    rng = np.random.default_rng(51)
    for flavour in ("mixed", "int"):
        a = _crowded_coo(rng, (N,), 300_000, 0.2, flavour, pool=100_000)
        for pol in _cases.POLICIES:
            for zn in (0, 1):
                A = up(ctx, a)
                R = sp.consolidate(ctx, A, (0,), pol, zn)
                got = down(R)
                A.free(); R.free()
                assert _cases.same_coo(got, orc.consolidate(a, (0,), pol, zn)), (flavour, pol, zn)


def test_row_structure_at_full_extent(ctx, orc):
    """dim_beginnings, the dense pointer over 2^31 row values (long stretches of empty rows between the ends) and
    dense_ptr_range at (2^31-5, 2^31), (0, 2^31), (2^31, 2^31), checked on the device."""
    import spsparse_b200 as sp
    import torch
    from _gpu import DevView, up
    rng = np.random.default_rng(61)
    a = _crowded_coo(rng, (N, N), 20000, 0.4, "pos", pool=300)
    A = up(ctx, a)
    R = sp.consolidate(ctx, A, (0, 1))
    A.free()
    want = orc.consolidate(a, (0, 1))
    assert np.array_equal(R.dim_beginnings(), orc.dim_beginnings(want))
    rows = want.idx[0].astype(np.int64)
    n = len(rows)
    ptr, ext = R.dense_ptr()
    assert ext == N
    full = torch.as_tensor(DevView(ptr, N + 1, "<i4"), device="cuda")
    assert bool((full[1:] >= full[:-1]).all().item()) and int(full[0].item()) == 0 and int(full[N].item()) == n
    # ptr[v] = entries in rows below v: at every row, its neighbours, both ends and a random sample
    probe = np.unique(np.concatenate([rows, np.clip(rows - 1, 0, N), rows + 1, [0, 1, N - 2, N - 1, N], rng.integers(0, N + 1, 100_000)]))
    got = full[torch.as_tensor(probe, device="cuda")].cpu().numpy()
    assert np.array_equal(got, np.searchsorted(rows, probe, side="left"))
    for lo, hi in ((N - 5, N), (0, N), (N, N)):
        part = torch.as_tensor(DevView(R.dense_ptr_range(lo, hi), hi - lo + 1, "<i4"), device="cuda")
        assert torch.equal(part, full[lo:hi + 1]), (lo, hi)
        del part
    del full
    R.free()
