"""Cross-check: restatement (oracle/spsparse_oracle.c) against the genuine reference on seeded inputs of its own,
beyond those of test_oracle_golden.py.  The reference's answers are stored in tests/golden/live_cases*.npz (their origin:
tests/golden/make_golden.py, live_cases); when oracle/_ref is built (SPSPARSE_REFERENCE) the reference also runs live
and must give exactly the stored answers."""
import numpy as np
import pytest

import _cases
import _golden
from oracle import oracle as O


def _same(a, b):
    if isinstance(a, O.Coo):
        return _cases.same_coo(a, b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.fixture(scope="module")
def want():
    p = _golden.pack("live_cases")
    ref = O.reference()

    def get(key, live):
        """The reference's answer stored under key; with oracle/_ref built, live(reference) must be the same."""
        stored = _golden.get_coo(p, key) if key + "_shape" in p else p[key]
        if ref is not None:
            assert _same(live(ref), stored), f"the reference disagrees with the stored answer {key}"
        return stored
    return get


def test_consolidate_live(orc, want):
    for s in range(120, 260):
        c = _cases.consolidate_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        args = (a, tuple(c["sort_order"]), c["policy"], c["zero_nan"])
        g, w = orc.consolidate(*args), want(f"c{s}_out", lambda r: r.consolidate(*args))
        assert _cases.same_coo(g, w), s
        assert np.array_equal(orc.sorted_permutation(a, args[1]), want(f"c{s}_perm", lambda r: r.sorted_permutation(a, args[1])))
        if a.rank == 2:
            assert np.array_equal(orc.dim_beginnings(g), want(f"c{s}_db", lambda r: r.dim_beginnings(w)))


def test_multiply_mm_live(orc, want):
    for s in range(300, 700):
        c = _cases.mm_case(s, big=(s % 40 == 0))
        A, B = c["A"], c["B"]
        acon = orc.consolidate(A, (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        bcon = orc.consolidate(B, (0, 1) if c["tB"] == "T" else (1, 0), c["policy"], c["zero_nan"])
        if (A.n and not acon.n) or (B.n and not bcon.n):
            continue  # the reference segfaults here (see tests/golden/make_golden.py)
        args = (c["C"], c["si"], A, c["tA"], c["sj"], B, c["tB"], c["sk"], c["policy"], c["zero_nan"])
        assert _cases.same_coo(orc.multiply_mm(*args), want(f"m{s}_out", lambda r: r.multiply_mm(*args))), s


def test_multiply_mv_live(orc, want):
    for s in range(150, 400):
        c = _cases.mv_case(s)
        acon = orc.consolidate(c["A"], (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        if c["A"].n and not acon.n:
            continue  # reference UB: empty consolidated A (multiply_sparse.hpp:302-303 comment)
        args = (c["C"], c["si"], c["A"], c["tA"], c["sj"], c["V"], c["policy"], c["zero_nan"])
        assert _cases.same_coo(orc.multiply_mv(*args), want(f"v{s}_out", lambda r: r.multiply_mv(*args))), s


def test_join_live(orc, want):
    rng = np.random.default_rng(7)
    for i in range(300):
        lists = [np.unique(rng.integers(0, 30, int(rng.integers(0, 20)))).astype(np.int32) for _ in range(3)]
        assert np.array_equal(orc.join(lists[0], lists[1]), want(f"j{i}_2", lambda r: r.join(lists[0], lists[1])))
        assert np.array_equal(orc.join(*lists), want(f"j{i}_3", lambda r: r.join(*lists)))


def test_dense_ops_live(orc, want):
    for s in range(100, 220):
        c = _cases.dense_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        perm = tuple(c["perm"])
        assert _cases.same_coo(orc.transpose(a, perm), want(f"d{s}_T", lambda r: r.transpose(a, perm))), s
        for policy in _cases.POLICIES:
            g, w = orc.to_dense(a, policy), want(f"d{s}_dense{policy}", lambda r: r.to_dense(a, policy))
            assert np.array_equal(g.view(np.uint64), w.view(np.uint64)), (s, policy)
        assert _cases.same_coo(orc.to_sparse(g), want(f"d{s}_sparse", lambda r: r.to_sparse(w))), s
