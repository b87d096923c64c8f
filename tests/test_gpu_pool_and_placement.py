"""-m gpu tests of three inputs the rest of the suite never varies: what the device memory pool held before a call, where the
caller's arrays sit in memory, and the sizes at which the sort's tiles begin and end.

* Poisoned pool: SPB_POOL_POISON fills every block the context's pool hands out with one byte (00, ff, 7f), so a kernel that
  reads a slot nobody wrote sees that byte instead of the zeros of fresh driver memory or the previous call's data.  One
  context per pattern runs a mixed sequence (consolidate in every organisation, the row structure, every multiply bin, row
  panels, prepared operands, matrix x vector, the one-rank row partition, the dense conversions), so cached blocks come back
  with slack and with old data in them.  Every result equals the oracle, and the statistics and launch count equal those of
  the same sequence in an unpoisoned context.
* Placement: the caller's arrays handed over with spb_coo_wrap_device at element offset 1 (4-byte index, 8-byte value
  pointers), so pass 0 and the histogram take their plain kernels on full tiles (one launch fewer than the aligned run, whose
  full tiles take the bulk-copy kernel), and multiply / mv read a sorted wrapped operand in place.
* Tile boundaries: 4095 .. 3*4096 + 1 entries and 2^23 + {0, 1, 4095}, with 1, 2 or 4097 dropped zeros so that the
  kept count lands on and beside a tile boundary; aligned and unaligned, bulk and per-thread loads, 8- and 9-bit digits,
  full-key passes and the in-row sort.  st.passes and st.digit_bits confirm the organisation that ran."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

import _cases
from oracle import oracle as O

pytestmark = pytest.mark.gpu

PATTERNS = ["00", "ff", "7f"]
M8 = 100_000_000
RS_TILE = 4096
_WANT = {}   # oracle answers by case key: the same inputs recur under every pattern and placement


# ---- helpers ---------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _env(**kv):
    """Sets (value) or removes (None) environment variables for the block; restores them afterwards."""
    old = {k: os.environ.get(k) for k in kv}
    for k, v in kv.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
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
    """A context created under `env` (for the knobs read at context creation)."""
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


def _cons_fields(st):
    return (st.n_in, st.n_kept, st.n_out, st.key_bits, st.passes, st.digit_bits)


def _mm_fields(st):
    return (st.products, st.nnz_a, st.nnz_b, st.rows_a, st.rows_merge, st.rows_esc, st.products_esc, st.nnz_c, st.rows_hash,
            st.products_hash)


def _same(got, want):
    if isinstance(want, O.Coo):
        return _cases.same_coo(got, want)
    if want.dtype == np.float64:   # dense arrays: bit for bit, any NaN equals any NaN
        na, nb = np.isnan(got), np.isnan(want)
        return got.shape == want.shape and np.array_equal(na, nb) and np.array_equal(got[~na].view(np.uint64), want[~nb].view(np.uint64))
    return np.array_equal(got, want)


def _want(key, fn):
    if key not in _WANT:
        _WANT[key] = fn()
    return _WANT[key]


class _Wrapped:
    """A COO array copied into torch device buffers at the given element offsets (one per index array, then the values) and
    wrapped with spb_coo_wrap_device; the buffers live as long as this object."""

    def __init__(self, ctx, a, offs, sort_order=None):
        import spsparse_b200 as sp
        import torch
        self.keep, ptrs = [], []
        for arr, off, dt in zip(list(a.idx) + [a.val], offs, [torch.int32] * a.rank + [torch.float64]):
            t = torch.empty(a.n + 1, dtype=dt, device="cuda")
            t[off:off + a.n].copy_(torch.from_numpy(np.ascontiguousarray(arr, np.int32 if dt == torch.int32 else np.float64)))
            self.keep.append(t)
            ptrs.append(t.data_ptr() + off * t.element_size())
        torch.cuda.synchronize()
        self.h = sp.CooArray.wrap_device(ctx, a.shape, ptrs[:-1], ptrs[-1], a.n, sort_order)

    def free(self):
        import torch
        self.h.free()
        torch.cuda.synchronize()
        self.keep = []


def _cons(ctx, H, so, pol, zn):
    """consolidate of handle H: (result, dim_beginnings or None, stats)"""
    import spsparse_b200 as sp
    from _gpu import down
    R, st = sp.consolidate(ctx, H, so, pol, zn, stats=True)
    got, db = down(R), (R.dim_beginnings() if R.rank == 2 else None)
    R.free()
    return got, db, st


def _check_cons(ctx, orc, key, a, H, so, pol, zn):
    got, db, st = _cons(ctx, H, so, pol, zn)
    want = _want(("cons",) + key, lambda: orc.consolidate(a, so, pol, zn))
    assert _cases.same_coo(got, want), key
    if db is not None:
        assert np.array_equal(db, _want(("db",) + key, lambda: orc.dim_beginnings(want))), key
    assert st.n_out == want.n
    return st


def _mm(ctx, args, pol=O.ADD, zn=0):
    import spsparse_b200 as sp
    from _gpu import up, down
    Cst, si, A, tA, sj, B, tB, sk = args
    hs = [up(ctx, x) for x in (si, A, sj, B, sk)]
    R, st = sp.multiply(ctx, Cst, hs[0], hs[1], tA, hs[2], hs[3], tB, hs[4], pol, zn, stats=True)
    got = down(R)
    for h in hs + [R]:
        if h is not None:
            h.free()
    return got, st


def _case_args(c):
    return (c["C"], c["si"], c["A"], c["tA"], c["sj"], c["B"], c["tB"], c["sk"])


def _cancel_case(seed, m=1200):
    """Short rows whose terms cancel to exactly 0 (whole rows of C vanish, some outputs vanish, +inf - inf = NaN kept) next to
    ordinary rows: tombstones and compaction in every bin."""
    rng = np.random.default_rng(seed)
    nj, nk = 400, 3000
    bj, bk, bv = [], [], []
    for j in range(100):
        cols = np.sort(rng.choice(nk, 6, replace=False))
        vals = rng.integers(1, 5, 6).astype(np.float64)
        for jj in (2 * j, 2 * j + 1):
            bj += [jj] * 6; bk += cols.tolist(); bv += vals.tolist()
    nb = 2500
    bj += rng.integers(200, nj, nb).tolist(); bk += rng.integers(0, nk, nb).tolist(); bv += rng.integers(1, 5, nb).astype(float).tolist()
    B = O.Coo((nj, nk), [np.array(bj), np.array(bk)], np.array(bv))
    ai, aj, av = [], [], []
    for i in range(m):
        p, q = int(rng.integers(0, 100)), int(rng.integers(200, nj))
        kind = i % 4
        if kind == 0:
            ai += [i, i]; aj += [2 * p, 2 * p + 1]; av += [3.0, -3.0]
        elif kind == 1:
            ai += [i, i, i]; aj += [2 * p, 2 * p + 1, q]; av += [2.0, -2.0, 1.5]
        elif kind == 2:
            for qq in rng.choice(np.arange(200, nj), 4, replace=False):
                ai.append(i); aj.append(int(qq)); av.append(float(rng.integers(1, 4)))
        else:
            ai += [i, i]; aj += [2 * p, 2 * p + 1]; av += [np.inf, -np.inf]
    A = O.Coo((m, nj), [np.array(ai), np.array(aj)], np.array(av))
    return (1.0, None, A, ".", None, B, ".", None)


def _hub_case(rng, shape, n, hubs, kmax=None):
    """Random entries, 30 % duplicates of earlier tuples, `hubs` rows of 1000 .. 9000 entries (longer than the in-row sort
    handles)."""
    i = rng.integers(0, shape[0], n)
    k = rng.integers(0, kmax or shape[1], n)
    dup = rng.random(n) < 0.3
    src = rng.integers(0, n, n)
    i[dup], k[dup] = i[src[dup]], k[src[dup]]
    for h in range(hubs):
        ln = int(rng.integers(1000, 9000))
        at = int(rng.integers(0, max(n - ln, 1)))
        i[at:at + ln] = 17 + 5 * h
        k[at:at + ln] = rng.integers(0, 5000, len(i[at:at + ln]))
    return i, k


def _dropping(rng, n, drops):
    """Non-zero values but for exactly `drops` zeros (either sign), which consolidate drops.  (A NaN is dropped only ahead of
    the first kept entry, so NaNs would not fix the kept count.)"""
    v = (0.5 + rng.random(n)) * np.where(rng.random(n) < 0.5, -1.0, 1.0)
    v[rng.choice(n, drops, replace=False)] = np.where(rng.random(drops) < 0.5, 0.0, -0.0)
    return v


def _large(x):
    """2^23 + x entries in a 10^8 x 10^8 shape (the default organisation: 9-bit row passes + in-row sort), 30 % duplicates,
    three hub rows longer than the in-row sort handles, 2 / 1 / 4097 dropped entries for x = 0 / 1 / 4095 (kept counts
    2^23 - 2, 2^23, 2^23 - 2).  Returns (array, sort order, policy, zero_nan)."""
    n = (1 << 23) + x
    drops, pol, zn = {0: (2, O.ADD, 1), 1: (1, O.REPLACE, 0), 4095: (4097, O.LEAVE_ALONE, 1)}[x]
    rng = np.random.default_rng(7000 + x)
    i, k = _hub_case(rng, (M8, M8), n, 3)
    return O.Coo((M8, M8), [i, k], _dropping(rng, n, drops)), (0, 1), pol, zn, drops


_LARGE = {}


def _large_case(x):
    if x not in _LARGE:
        _LARGE[x] = _large(x)
    return _LARGE[x]


# ---- 1. the switch is live -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern", PATTERNS)
def test_poison_fills_every_block(pattern):
    """spb_coo_alloc returns blocks holding the pattern: fresh ones, and cached ones that held uploaded data before (with
    slack: a smaller request gets the larger block back).  A malformed value is refused."""
    import spsparse_b200 as sp
    from spsparse_b200._lib import vp
    byte = int(pattern, 16)
    with _context(SPB_POOL_POISON=pattern) as c:
        rng = np.random.default_rng(1)
        for n in (1000, 950, 300_000, 290_000, 1, 3 << 20):
            U = sp.CooArray.from_host(c, (5000, 5000), [rng.integers(0, 5000, n), rng.integers(0, 5000, n)], rng.random(n))
            U.free()   # its blocks go back to the pool holding data; the next request of a similar size gets them
            h = vp()
            assert c.lib.spb_coo_alloc(c.h, 2, (C.c_uint64 * 2)(5000, 5000), n - n // 40, C.byref(h)) == 0
            a = sp.CooArray(c, h)
            idx, val = a.to_host()
            a.free()
            for x in idx + [val]:
                assert (x.view(np.uint8) == byte).all(), (pattern, n)
    for bad in ("", "1ff", "zz"):
        with pytest.raises(sp.SpbError):
            with _context(SPB_POOL_POISON=bad):
                pass


# ---- 2. the poisoned matrix ------------------------------------------------------------------------------------------
class _Run:
    """One run of a sequence: results are checked against the oracle as they come, statistics are kept by case key."""

    def __init__(self, ctx, orc):
        self.ctx, self.orc, self.stats = ctx, orc, {}

    def cons(self, key, a, so, pol, zn, **env):
        from _gpu import up
        with _env(**env):
            A = up(self.ctx, a)
            st = _check_cons(self.ctx, self.orc, key, a, A, so, pol, zn)
            A.free()
        self.stats[("cons",) + key] = _cons_fields(st)

    def mm(self, key, args, pol=O.ADD, zn=0, **env):
        with _env(**env):
            got, st = _mm(self.ctx, args, pol, zn)
        want = _want(("mm",) + key, lambda: self.orc.multiply_mm(*args, pol, zn))
        assert _cases.same_coo(got, want), key
        self.stats[("mm",) + key] = _mm_fields(st)
        return st

    def check(self, key, got, fn, st=None):
        assert _same(got, _want(key, fn)), key
        if st is not None:
            self.stats[key] = st


def _seq_default(r):
    """The sequence of the default context."""
    import spsparse_b200 as sp
    from spsparse_b200.dist import RowPartition
    from _gpu import up, down, dev_to_numpy
    ctx, orc = r.ctx, r.orc
    # consolidate: fresh seeds (0 .. 4099 entries, both orders, every policy, zero_nan), mixed sizes
    for s in range(1000, 1040):
        c = _cases.consolidate_case(s)
        r.cons(("seed", s), O.Coo(tuple(c["shape"]), c["idx"], c["val"]), tuple(c["sort_order"]), c["policy"], c["zero_nan"])
    # duplicate runs longer than 256 (k_long_runs), crossing tiles
    rng = np.random.default_rng(41)
    lens = np.concatenate([rng.integers(1, 12, 600), rng.integers(200, 330, 60), rng.integers(1000, 3000, 8), [257, 256, 255, 264]])
    keys = rng.permutation(len(lens))
    o = rng.permutation(int(lens.sum()))
    a = O.Coo((200, 1 << 20), [np.repeat(keys // 700, lens)[o], np.repeat(keys % 700 * 1000, lens)[o]],
              _cases._values(rng, int(lens.sum()), "mixed"))
    for pol in _cases.POLICIES:
        r.cons(("runs", pol), a, (0, 1), pol, pol % 2)
    # row passes + in-row sort with hub rows (long-row re-sort), each reduce kernel, the fused kernel; full-key passes
    rng = np.random.default_rng(43)
    i, k = _hub_case(rng, (2000, 1 << 18), 60000, 3)
    hub = O.Coo((2000, 1 << 18), [i, k], _cases._values(rng, len(i), "mixed"))
    for name, env in (("seg", {}), ("seg_rw0", {"SPB_REDUCE_WARP": "0"}), ("seg_rw2", {"SPB_REDUCE_WARP": "2"}),
                      ("seg_fused", {"SPB_FUSED_REDUCE": "1"}), ("seg_table", {"SPB_SEGMENT_WALK": "0"})):
        for so, pol in (((0, 1), O.ADD), ((1, 0), O.REPLACE)):
            r.cons(("hub", name, so), hub, so, pol, 1, SPB_SEGMENT_SORT="1", **env)
    r.cons(("hub", "full", (0, 1)), hub, (0, 1), O.ADD, 0, SPB_SEGMENT_SORT="0", SPB_REDUCE_WARP="2")
    # the default large path: 9-bit row passes, in-row sort, hub rows re-sorted by full key
    a, so, pol, zn, _ = _large_case(4095)
    r.cons(("large", 4095), a, so, pol, zn)
    assert r.stats[("cons", "large", 4095)][4:] == (3, 9)
    # sorted_permutation
    for s in (1004, 1008, 1009):   # 1004 is a rank-1 case
        c = _cases.consolidate_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        for so in ((0,),) if a.rank == 1 else ((0, 1), (1, 0)):
            A = up(ctx, a)
            r.check(("perm", s, so), A.sorted_permutation(so), lambda: orc.sorted_permutation(a, so))
            A.free()
    # dense pointer over rows with gaps of thousands of empty rows (listed and filled by the gap kernel), ranges of it
    rng = np.random.default_rng(47)
    rows = np.array([0, 3, 5000, 5001, 20000, 61234, 99999])
    a = O.Coo((100_000, 64), [rows[rng.integers(0, len(rows), 3000)], rng.integers(0, 64, 3000)], _cases._values(rng, 3000, "int"))
    A = up(ctx, a)
    R = sp.consolidate(ctx, A, (0, 1))
    A.free()
    want = _want(("cons", "gaps"), lambda: orc.consolidate(a, (0, 1)))
    ptr, ext = R.dense_ptr()
    ctx.sync()
    full = dev_to_numpy(ptr, ext + 1, "<i4")
    r.check(("dense_ptr", "gaps"), full, lambda: np.searchsorted(want.idx[0], np.arange(ext + 1), side="left").astype(np.int32))
    for lo, hi in ((0, 100_000), (4000, 21000), (99_990, 100_000), (7, 7), (5001, 5002)):
        p = R.dense_ptr_range(lo, hi)
        ctx.sync()
        assert np.array_equal(dev_to_numpy(p, hi - lo + 1, "<i4"), full[lo:hi + 1]), (lo, hi)
    r.check(("db", "gaps"), R.dim_beginnings(), lambda: orc.dim_beginnings(want))
    R.free()
    # multiply: the register merge (default builds, 2- and 4-list builds, LOCAL, one pass) with exact cancellation
    canc = _cancel_case(404)
    for name, env in (("default", {}), ("nl2", {"SPB_MERGE_NL_COUNT": "2", "SPB_MERGE_NL_NUMERIC": "2"}),
                      ("nl4", {"SPB_MERGE_NL_COUNT": "4", "SPB_MERGE_NL_NUMERIC": "4"}), ("local", {"SPB_MERGE_LOCAL": "1"}),
                      ("onepass", {"SPB_MERGE_ONEPASS": "1"})):
        st = r.mm(("cancel", name), canc, **env)
        assert st.rows_merge > 0 and st.rows_esc == 0 and st.rows_hash == 0
    for s in range(2000, 2024):
        c = _cases.mm_case(s, big=(s % 4 == 0))
        r.mm(("seed", s), _case_args(c), c["policy"], c["zero_nan"])
    # row panels
    Cst, si, A_, tA, sj, B_, tB, sk = canc
    hs = [up(ctx, x) for x in (A_, B_)]
    plan = sp.MultiplyPlan(ctx, Cst, None, hs[0], tA, None, hs[1], tB, None, O.ADD, False, 2000)
    hs[0].free(); hs[1].free()
    parts = []
    for p in range(plan.n_panels):
        R = plan.panel(p)
        parts.append(down(R))
        R.free()
    assert plan.n_panels > 3
    shape = plan.shape
    plan.free()
    got = O.Coo(shape, [np.concatenate([q.idx[d] for q in parts]) for d in (0, 1)], np.concatenate([q.val for q in parts]))
    r.check(("mm", "cancel", "default"), got, None)
    # multiply_prepared with B in compressed form, and the one-rank row partition
    c = _cases.mm_case(2008, big=True)
    A_ = orc.transpose(c["A"], (1, 0)) if c["tA"] == "T" else c["A"]
    B_ = orc.transpose(c["B"], (1, 0)) if c["tB"] == "T" else c["B"]
    Ah, Bh, Sh = up(ctx, A_), up(ctx, B_), up(ctx, c["sj"])
    Ac, Bc = sp.consolidate(ctx, Ah, (0, 1)), sp.consolidate(ctx, Bh, (0, 1))
    (_, p1), pv = Bc.device_ptrs()
    ptr, ext = Bc.dense_ptr()
    Bcsr = sp.CooArray.wrap_csr(ctx, B_.shape, 0, ptr, p1, pv, Bc.size())
    C1, st1 = sp.multiply_prepared(ctx, 1.0, None, Ac, 0, Sh, Bcsr, 0, None)
    r.check(("prepared", 2008), down(C1), lambda: orc.multiply_mm(1.0, None, A_, ".", c["sj"], B_, ".", None), _mm_fields(st1))
    for h in (C1, Bcsr, Ac, Bc):
        h.free()
    rp = RowPartition(ctx, 0, 1, B_.shape[0], B_.n + 1)
    C2, _ = rp.multiply(c["C"], None, Ah, Sh, Bh, None, c["policy"], c["zero_nan"])
    r.check(("rowpart", 2008), down(C2), lambda: orc.multiply_mm(c["C"], None, A_, ".", c["sj"], B_, ".", None, c["policy"], c["zero_nan"]))
    C2.free()
    rp.close()
    for h in (Ah, Bh, Sh):
        if h is not None:   # sj is absent in some cases
            h.free()
    # matrix x vector
    for s in range(9000, 9020):
        c = _cases.mv_case(s)
        args = (c["C"], c["si"], c["A"], c["tA"], c["sj"], c["V"])
        hs = [up(ctx, x) for x in args[1:3] + args[4:]]
        R = sp.multiply(ctx, c["C"], hs[0], hs[1], c["tA"], hs[2], hs[3], duplicate_policy=c["policy"], zero_nan=c["zero_nan"])
        r.check(("mv", s), down(R), lambda: orc.multiply_mv(*args, c["policy"], c["zero_nan"]))
        for h in hs + [R]:
            if h is not None:
                h.free()
    # the dense conversions and transpose
    for s in range(300, 318):
        c = _cases.dense_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        dA = up(ctx, a)
        r.check(("to_dense", s), sp.to_dense(ctx, dA, c["policy"]), lambda: orc.to_dense(a, c["policy"]))
        dense = _WANT[("to_dense", s)]
        S = sp.to_sparse(ctx, dense)
        r.check(("to_sparse", s), down(S), lambda: orc.to_sparse(dense))
        T = sp.transpose(ctx, dA, tuple(c["perm"]))
        r.check(("transpose", s), down(T), lambda: orc.transpose(a, tuple(c["perm"])))
        for h in (dA, S, T):
            h.free()


def _seq_esc(r):
    """Every row through expand-sort-compress, in chunks of 37 products."""
    st = r.mm(("cancel", "esc"), _cancel_case(404))
    assert st.rows_esc > 0 and st.rows_merge == 0 and st.rows_hash == 0
    for s in range(2100, 2112):
        c = _cases.mm_case(s, big=(s % 4 == 0))
        r.mm(("seed", s), _case_args(c), c["policy"], c["zero_nan"])


def _seq_hash(r):
    """Every row through the bitmap + hash-accumulator bin: whole rows, work items of 3 outputs, 32-column windows."""
    for name, env in (("plain", {"SPB_HASH_SMALL": "1"}), ("items", {"SPB_HASH_ITEM_CAP": "3", "SPB_HASH_SMALL": "0"}),
                      ("windows", {"SPB_HASH_WIN_COLS": "32", "SPB_HASH_ITEM_CAP": "7", "SPB_HASH_SMALL": "0"})):
        st = r.mm(("cancel", name), _cancel_case(404), **env)
        assert st.rows_hash > 0 and st.rows_merge == 0 and st.rows_esc == 0
        for s in (2000, 2004, 2008, 2013):
            r.mm(("seed", s, name), _case_args(_cases.mm_case(s, big=(s % 4 == 0))), **env)


def _seq_bulk_off(r):
    """Per-thread tile loads in every radix pass after the first."""
    rng = np.random.default_rng(53)
    i, k = _hub_case(rng, (2000, 1 << 18), 60000, 2)
    a = O.Coo((2000, 1 << 18), [i, k], _cases._values(rng, len(i), "mixed"))
    for seg in ("0", "1"):
        for r9 in ("0", "1"):
            r.cons(("bulk0", seg, r9), a, (0, 1), O.ADD, 1, SPB_SEGMENT_SORT=seg, SPB_RADIX9=r9)


_SEQUENCES = {
    "default": ({}, _seq_default),
    "esc": ({"SPB_MERGE_MAX_PRODUCTS": "0", "SPB_ESC_CHUNK": "37", "SPB_HASH_MIN_PRODUCTS": "off"}, _seq_esc),
    "hash0": ({"SPB_MERGE_MAX_PRODUCTS": "0", "SPB_HASH_MIN_PRODUCTS": "0", "SPB_HASH_VARIANT": "0"}, _seq_hash),
    "hash1": ({"SPB_MERGE_MAX_PRODUCTS": "0", "SPB_HASH_MIN_PRODUCTS": "0", "SPB_HASH_VARIANT": "1"}, _seq_hash),
    "hash2": ({"SPB_MERGE_MAX_PRODUCTS": "0", "SPB_HASH_MIN_PRODUCTS": "0", "SPB_HASH_VARIANT": "2"}, _seq_hash),
    "bulk_off": ({"SPB_BULK_LOAD": "0"}, _seq_bulk_off),
}
_CLEAN = {}   # sequence name -> (statistics, launch count) of the unpoisoned run


@pytest.mark.parametrize("pattern", PATTERNS)
def test_poisoned_pool_matrix(orc, pattern):
    """Each sequence in a context whose pool blocks arrive filled with `pattern`: every result equals the oracle, and the bin
    and organisation statistics and the launch count equal those of the same sequence in an unpoisoned context."""
    for name, (knobs, seq) in _SEQUENCES.items():
        if name not in _CLEAN:
            with _context(SPB_POOL_POISON=None, **knobs) as c:
                r = _Run(c, orc)
                seq(r)
                _CLEAN[name] = (r.stats, _launches(c))
        with _context(SPB_POOL_POISON=pattern, **knobs) as c:
            r = _Run(c, orc)
            seq(r)
            stats, launches = r.stats, _launches(c)
        clean_stats, clean_launches = _CLEAN[name]
        assert stats.keys() == clean_stats.keys()
        for key in stats:
            assert stats[key] == clean_stats[key], (name, key)
        assert launches == clean_launches, name


# ---- 3. placement of the caller's arrays -----------------------------------------------------------------------------
OFFSETS = {"row": (1, 0, 0), "col": (0, 1, 0), "val": (0, 0, 1), "all": (1, 1, 1)}


def _bulk_saved(n):
    """Launches the unaligned sort of n entries saves: the aligned one runs the bulk pass-0 kernel on its full tiles and the
    plain one on the partial last tile; the unaligned one runs the plain kernel alone."""
    return 1 if n >= RS_TILE and n % RS_TILE else 0


def _placement_case(n, seed, shape=(3000, 5000)):
    rng = np.random.default_rng(seed)
    idx = [rng.integers(0, s, n) for s in shape]
    dup = rng.random(n) < 0.2
    src = rng.integers(0, n, n)
    for x in idx:
        x[dup] = x[src[dup]]
    return O.Coo(shape, idx, _cases._values(rng, n, "mixed"))


@pytest.mark.parametrize("where", list(OFFSETS))
def test_unaligned_caller_arrays(ctx_default, orc, where):
    """consolidate, sorted_permutation and multiply (tA, tB in {., T}) on wrapped arrays of which `where` sits at element offset
    1: the same answers and statistics as the aligned wrap, and one launch fewer wherever the aligned sort has full tiles and
    a partial one."""
    ctx = ctx_default
    offs = OFFSETS[where]
    aligned = (0, 0, 0)

    def run(off, fn):
        n0 = _launches(ctx)
        out = fn(off)
        return out, _launches(ctx) - n0

    for n in (3000, 4096, 5000, 8192, 9001):
        a = _placement_case(n, 100 + n)
        for so, pol, zn in (((0, 1), O.ADD, 1), ((1, 0), O.REPLACE, 0), ((0, 1), O.LEAVE_ALONE, 1)):
            def cons(off):
                W = _Wrapped(ctx, a, off)
                st = _check_cons(ctx, orc, ("place", n, so, pol, zn), a, W.h, so, pol, zn)
                W.free()
                return _cons_fields(st)
            (st_a, l_a), (st_u, l_u) = run(aligned, cons), run(offs, cons)
            assert st_a == st_u and l_a - l_u == _bulk_saved(n), (n, so, l_a, l_u)

            def perm(off):
                W = _Wrapped(ctx, a, off)
                p = W.h.sorted_permutation(so)
                W.free()
                assert np.array_equal(p, _want(("perm", n, so), lambda: orc.sorted_permutation(a, so))), (n, so)
            (_, l_a), (_, l_u) = run(aligned, perm), run(offs, perm)
            # sorted_permutation sorts the index arrays with the entry numbers as payload: the values' place does not matter
            assert l_a - l_u == (_bulk_saved(n) if offs[0] or offs[1] else 0), (n, so)
    # multiply: both operands prepared (sorted) from the wrapped arrays
    import spsparse_b200 as sp
    from _gpu import down
    for tA in (".", "T"):
        for tB in (".", "T"):
            opA, opB = _placement_case(5000, 7, (800, 600)), _placement_case(4500, 8, (600, 900))
            A = orc.transpose(opA, (1, 0)) if tA == "T" else opA
            B = orc.transpose(opB, (1, 0)) if tB == "T" else opB

            def mm(off):
                WA, WB = _Wrapped(ctx, A, off), _Wrapped(ctx, B, off)
                R, st = sp.multiply(ctx, 1.5, None, WA.h, tA, None, WB.h, tB, None, O.ADD, True, stats=True)
                got = down(R)
                R.free(); WA.free(); WB.free()
                want = _want(("place_mm", tA, tB), lambda: orc.multiply_mm(1.5, None, A, tA, None, B, tB, None, O.ADD, True))
                assert _cases.same_coo(got, want), (tA, tB)
                return _mm_fields(st)
            (st_a, l_a), (st_u, l_u) = run(aligned, mm), run(offs, mm)
            assert st_a == st_u and l_a - l_u == _bulk_saved(A.n) + _bulk_saved(B.n), (tA, tB, l_a, l_u)


@pytest.mark.parametrize("where", list(OFFSETS))
def test_unaligned_sorted_operands_used_in_place(ctx_default, orc, where):
    """A wrapped operand flagged sorted in the order multiply / mv need is read where it lies (A of the matrix product, A and
    V of the matrix x vector product); B flagged sorted is re-bucketed from the wrapped arrays with every entry kept."""
    import spsparse_b200 as sp
    from _gpu import down
    ctx = ctx_default
    offs = OFFSETS[where]
    A = orc.consolidate(_placement_case(6000, 11, (700, 500)), (0, 1))
    B = orc.consolidate(_placement_case(5000, 12, (500, 800)), (0, 1))
    WA, WB = _Wrapped(ctx, A, offs, (0, 1)), _Wrapped(ctx, B, offs, (0, 1))
    R, st = sp.multiply(ctx, 2.5, None, WA.h, ".", None, WB.h, ".", None, stats=True)
    got = down(R)
    R.free(); WB.free()
    assert _cases.same_coo(got, orc.multiply_mm(2.5, None, A, ".", None, B, ".", None)) and st.products > 0
    rng = np.random.default_rng(13)
    V = orc.consolidate(O.Coo((500,), [rng.integers(0, 500, 300)], _cases._values(rng, 300, "mixed")), (0,))
    WV = _Wrapped(ctx, V, offs[1:], (0,))   # rank 1: its index (offset of the column index) and its values
    R = sp.multiply(ctx, -1.5, None, WA.h, ".", None, WV.h)
    got = down(R)
    R.free(); WA.free(); WV.free()
    assert _cases.same_coo(got, orc.multiply_mv(-1.5, None, A, ".", None, V))


@pytest.mark.parametrize("offs", [(1, 0), (0, 1), (1, 1)])
def test_unaligned_rank1(ctx_default, orc, offs):
    """Rank 1: consolidate with every policy, sorted_permutation, and mv with an unsorted wrapped vector."""
    import spsparse_b200 as sp
    from _gpu import down
    ctx = ctx_default
    for n in (3000, 5000, 8192, 12289):
        rng = np.random.default_rng(n)
        a = O.Coo((1 << 20,), [rng.integers(0, 1 << 20, n) // 16], _cases._values(rng, n, "mixed"))
        for pol in _cases.POLICIES:
            def cons(off):
                n0 = _launches(ctx)
                W = _Wrapped(ctx, a, off)
                st = _cons_fields(_check_cons(ctx, orc, ("r1", n, pol), a, W.h, (0,), pol, pol % 2))
                W.free()
                return st, _launches(ctx) - n0
            (st_a, l_a), (st_u, l_u) = cons((0, 0)), cons(offs)
            assert st_a == st_u and l_a - l_u == _bulk_saved(n), (n, pol, l_a, l_u)
        W = _Wrapped(ctx, a, offs)
        p = W.h.sorted_permutation((0,))
        W.free()
        assert np.array_equal(p, _want(("r1perm", n), lambda: orc.sorted_permutation(a, (0,))))
    rng = np.random.default_rng(5)
    A = _placement_case(3000, 14, (400, 1 << 20))
    V = O.Coo((1 << 20,), [rng.integers(0, 1 << 20, 5000)], _cases._values(rng, 5000, "mixed"))
    W = _Wrapped(ctx, V, offs)
    from _gpu import up
    Ah = up(ctx, A)
    R = sp.multiply(ctx, 1.0, None, Ah, ".", None, W.h, duplicate_policy=O.REPLACE, zero_nan=True)
    got = down(R)
    R.free(); Ah.free(); W.free()
    assert _cases.same_coo(got, orc.multiply_mv(1.0, None, A, ".", None, V, O.REPLACE, True))


@pytest.fixture(scope="module")
def ctx_default():
    import spsparse_b200 as sp
    with sp.Context(0) as c:
        yield c
        c.trim()


# ---- 4. tile boundaries and load paths -------------------------------------------------------------------------------
def _organisation(seg, r9):
    """(passes, digit bits) of a 54-bit key (10^8 x 10^8): full-key passes or row passes + in-row sort, 8- or 9-bit digits."""
    return {("0", "0"): (7, 8), ("0", "1"): (6, 9), ("1", "0"): (4, 8), ("1", "1"): (3, 9)}[(seg, r9)]


def _tile_case(n, drops, t):
    rng = np.random.default_rng(n * 10 + drops)
    rows = rng.integers(0, M8, max(n // 3, 1))[rng.integers(0, max(n // 3, 1), n)]   # ~3 entries a row
    k = rng.integers(0, M8, n)
    dup = rng.random(n) < 0.3
    src = rng.integers(0, n, n)
    k[dup] = k[src[dup]]
    zn = t % 2
    return O.Coo((M8, M8), [rows, k], _dropping(rng, n, drops)), [(0, 1), (1, 0)][t % 2], _cases.POLICIES[t % 3], zn


def test_tile_boundaries(orc):
    """n in {4095, 4096, 4097, 8191, 8192, 8193, 3*4096+1} with 1, 2 or 4097 dropped entries (kept counts on and beside a tile
    boundary), aligned and unaligned, bulk and per-thread loads, 8- and 9-bit digits, full-key passes and the in-row sort."""
    t = 0
    with _context(SPB_BULK_LOAD="1") as c1, _context(SPB_BULK_LOAD="0") as c0:
        for n in (4095, 4096, 4097, 8191, 8192, 8193, 3 * 4096 + 1):
            for drops in (1, 2, 4097):
                if drops >= n:
                    continue
                t += 1
                a, so, pol, zn = _tile_case(n, drops, t)
                for bulk, ctx in (("1", c1), ("0", c0)):
                    for seg in ("0", "1"):
                        for r9 in ("0", "1"):
                            launches = []
                            for off in ((0, 0, 0), (1, 1, 1)):
                                with _env(SPB_SEGMENT_SORT=seg, SPB_RADIX9=r9):
                                    n0 = _launches(ctx)
                                    W = _Wrapped(ctx, a, off)
                                    st = _check_cons(ctx, orc, ("tile", n, drops), a, W.h, so, pol, zn)
                                    W.free()
                                    launches.append(_launches(ctx) - n0)
                                key = (n, drops, bulk, seg, r9, off)
                                assert (st.passes, st.digit_bits) == _organisation(seg, r9), key
                                assert st.n_in == n and st.n_kept == n - drops, key
                            assert launches[0] - launches[1] == (_bulk_saved(n) if bulk == "1" else 0), (n, drops, bulk, seg, r9, launches)


@pytest.mark.parametrize("x", [0, 1, 4095])
def test_tile_boundaries_large(orc, x):
    """2^23 + x entries on the default organisation (three 9-bit row passes + in-row sort, hub rows re-sorted by their full
    key), kept counts 2^23 - 2, 2^23, 2^23 - 2: aligned and unaligned, bulk and per-thread loads; the scalar histogram
    (SPB_VEC_LOAD=0) and MATCH.ANY ranks (SPB_RANK_MODE=1) once each."""
    a, so, pol, zn, drops = _large_case(x)
    n = a.n
    extra = {1: {"SPB_VEC_LOAD": "0"}, 4095: {"SPB_RANK_MODE": "1"}}.get(x)
    with _context(SPB_BULK_LOAD="1") as c1, _context(SPB_BULK_LOAD="0") as c0:
        for bulk, ctx in (("1", c1), ("0", c0)):
            launches = []
            for off in ((0, 0, 0), (1, 1, 1)):
                n0 = _launches(ctx)
                W = _Wrapped(ctx, a, off)
                st = _check_cons(ctx, orc, ("large", x), a, W.h, so, pol, zn)
                W.free()
                launches.append(_launches(ctx) - n0)
                assert (st.key_bits, st.passes, st.digit_bits) == (54, 3, 9) and st.n_kept == n - drops, (bulk, off)
            assert launches[0] - launches[1] == (_bulk_saved(n) if bulk == "1" else 0), (bulk, launches)
        if extra:
            with _env(**extra):
                W = _Wrapped(c1, a, (0, 0, 0))
                st = _check_cons(c1, orc, ("large", x), a, W.h, so, pol, zn)
                W.free()
            assert (st.passes, st.digit_bits) == (3, 9)
        c1.trim(); c0.trim()
