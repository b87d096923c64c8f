"""Regenerates tests/golden/*.npz from the GENUINE reference (oracle/_ref/libspsparse_ref.so).

Needs a checkout of the original spsparse to build oracle/_ref:
    SPSPARSE_REFERENCE=<checkout> make -C oracle ref && python tests/golden/make_golden.py
The fixtures pin the oracle (tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_*.py)
to the reference's own outputs, so the tests need no copy of the reference.  Packs over 1 MB are stored in parts
(tests/golden/_pack.py).

    python tests/golden/make_golden.py live               # live_cases: the reference's answers for tests/test_oracle_vs_reference.py
    python tests/golden/make_golden.py live restatement   # ... written from the restatement instead (see live_cases)
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import oracle as O  # noqa: E402
import _cases  # noqa: E402
from _pack import Packer  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ref = O.reference()


def put(d, prefix, coo):
    if coo is None:
        d[prefix + "_none"] = np.array(1)
        return
    d[prefix + "_shape"] = np.array(coo.shape, np.int64)
    for k, a in enumerate(coo.idx):
        d[f"{prefix}_idx{k}"] = a
    d[prefix + "_val"] = coo.val
    d[prefix + "_so"] = np.array(coo.sort_order if coo.sort_order is not None else (-1,), np.int32)


def reference_test_inputs(seed, mv):
    """tests/test_multiply_sparse.cpp:84-98 / :138-152 via ref_testcase_inputs (libstdc++ RNG)."""
    f = ref.lib.ref_testcase_inputs
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    f.argtypes = [C.c_uint, C.c_int, C.c_int, C.POINTER(C.c_int64), i32p, i32p, f64p,
                  C.POINTER(C.c_int64), i32p, i32p, f64p]
    f.restype = None
    a0, a1, b0, b1 = (np.zeros(25, np.int32) for _ in range(4))
    av, bv = np.zeros(25), np.zeros(25)
    na, nb = C.c_int64(), C.c_int64()
    p32 = lambda a: a.ctypes.data_as(i32p)
    p64 = lambda a: a.ctypes.data_as(f64p)
    f(5, seed, int(mv), C.byref(na), p32(a0), p32(a1), p64(av), C.byref(nb), p32(b0), p32(b1), p64(bv))
    A = O.Coo((5, 5), [a0[:na.value], a1[:na.value]], av[:na.value])
    B = O.Coo((5,), [b0[:nb.value]], bv[:nb.value]) if mv else O.Coo((5, 5), [b0[:nb.value], b1[:nb.value]], bv[:nb.value])
    return A, B


def dense_ops():
    """4b. transpose / to_dense (DenseAccum, all policies) / to_sparse  (SURVEY 8f rank 3)"""
    d = Packer()
    nd = 60
    for s in range(nd):
        c = _cases.dense_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        put(d, f"d{s}_in", a)
        d[f"d{s}_args"] = np.array(list(c["perm"]) + [c["policy"]], np.int32)
        put(d, f"d{s}_T", ref.transpose(a, tuple(c["perm"])))
        dense = ref.to_dense(a, c["policy"])
        d[f"d{s}_dense"] = dense
        put(d, f"d{s}_sparse", ref.to_sparse(dense))
    d["count"] = np.array(nd)
    d.save(os.path.join(HERE, "dense_ops_cases.npz"))


def live_cases(impl):
    """The answers tests/test_oracle_vs_reference.py compares the restatement with, on its own seeded inputs (the same
    loops as there).  The committed live_cases pack was written by `live restatement`: the restatement's answers,
    which that test, run live against the genuine reference, found identical on every one of these inputs (commit
    5e24c53, whose CPU suite passed in full with oracle/_ref built; spsparse_oracle.c, _cases.py and the test are
    unchanged since).  `live` rewrites the pack from the reference itself."""
    orc = O.port()
    d = Packer()
    for s in range(120, 260):
        c = _cases.consolidate_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        r = impl.consolidate(a, tuple(c["sort_order"]), c["policy"], c["zero_nan"])
        put(d, f"c{s}_out", r)
        d[f"c{s}_perm"] = impl.sorted_permutation(a, tuple(c["sort_order"]))
        if a.rank == 2:
            d[f"c{s}_db"] = impl.dim_beginnings(r)
    for s in range(300, 700):
        c = _cases.mm_case(s, big=(s % 40 == 0))
        A, B = c["A"], c["B"]
        acon = orc.consolidate(A, (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        bcon = orc.consolidate(B, (0, 1) if c["tB"] == "T" else (1, 0), c["policy"], c["zero_nan"])
        if (A.n and not acon.n) or (B.n and not bcon.n):
            continue  # the reference segfaults here (see main)
        put(d, f"m{s}_out", impl.multiply_mm(c["C"], c["si"], A, c["tA"], c["sj"], B, c["tB"], c["sk"], c["policy"], c["zero_nan"]))
    for s in range(150, 400):
        c = _cases.mv_case(s)
        acon = orc.consolidate(c["A"], (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        if c["A"].n and not acon.n:
            continue  # reference UB: empty consolidated A
        put(d, f"v{s}_out", impl.multiply_mv(c["C"], c["si"], c["A"], c["tA"], c["sj"], c["V"], c["policy"], c["zero_nan"]))
    rng = np.random.default_rng(7)
    for i in range(300):
        lists = [np.unique(rng.integers(0, 30, int(rng.integers(0, 20)))).astype(np.int32) for _ in range(3)]
        d[f"j{i}_2"] = impl.join(lists[0], lists[1])
        d[f"j{i}_3"] = impl.join(*lists)
    for s in range(100, 220):
        c = _cases.dense_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        put(d, f"d{s}_T", impl.transpose(a, tuple(c["perm"])))
        for policy in _cases.POLICIES:
            dense = impl.to_dense(a, policy)
            d[f"d{s}_dense{policy}"] = dense
        put(d, f"d{s}_sparse", impl.to_sparse(dense))
    return d.save(os.path.join(HERE, "live_cases.npz"))


def main():
    # 1. the reference's own randomized tests, seeds 1..999 (BASELINE config 1)
    d = Packer()
    eye = O.Coo((5,), [np.arange(5)], np.ones(5), (0,))
    for seed in range(1, 1000):
        A, B = reference_test_inputs(seed, mv=False)
        put(d, f"mm{seed}_A", A); put(d, f"mm{seed}_B", B)
        put(d, f"mm{seed}_C", ref.multiply_mm(1.0, None, A, ".", eye, B, ".", None))  # :104-110
        A, V = reference_test_inputs(seed, mv=True)
        put(d, f"mv{seed}_A", A); put(d, f"mv{seed}_V", V)
        put(d, f"mv{seed}_C", ref.multiply_mv(1.0, None, A, ".", None, V))  # :158-163
    d.save(os.path.join(HERE, "reference_random_tests.npz"))

    # 2. consolidate fuzz: all policies / zero_nan / NaN / +-0 / cancellation / rank 1 and 2
    d = Packer()
    ncons = 120
    for s in range(ncons):
        c = _cases.consolidate_case(s)
        a = O.Coo(tuple(c["shape"]), c["idx"], c["val"])
        r = ref.consolidate(a, tuple(c["sort_order"]), c["policy"], c["zero_nan"])
        put(d, f"c{s}_in", a); put(d, f"c{s}_out", r)
        d[f"c{s}_args"] = np.array([c["policy"], c["zero_nan"]] + list(c["sort_order"]), np.int32)
        if a.rank == 2:
            d[f"c{s}_db"] = ref.dim_beginnings(r)
    d["count"] = np.array(ncons)
    d.save(os.path.join(HERE, "consolidate_cases.npz"))

    # 3. multiply MM fuzz with scale vectors, transposes, policies, pre-sorted operands
    d = Packer()
    nmm = 300
    for s in range(nmm):
        c = _cases.mm_case(s, big=(s % 25 == 24))
        A, B = c["A"], c["B"]
        if s % 4 == 1:  # exercise Consolidate<>'s "already sorted" shortcut (algorithm.hpp:360-362)
            A = ref.consolidate(A, (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        if s % 4 == 2:
            B = ref.consolidate(B, (0, 1) if c["tB"] == "T" else (1, 0), c["policy"], c["zero_nan"])
        if A.n == 0 or B.n == 0:
            A, B = c["A"], c["B"]
        # The reference dereferences an empty dim_beginnings list (algorithm.hpp:197,
        # multiply_sparse.hpp:176-177) when an operand consolidates to nothing (all values 0/NaN):
        # it segfaults.  Such cases are stored with the only sensible answer, an empty product.
        acon = ref.consolidate(A, (1, 0) if c["tA"] == "T" else (0, 1), c["policy"], c["zero_nan"])
        bcon = ref.consolidate(B, (0, 1) if c["tB"] == "T" else (1, 0), c["policy"], c["zero_nan"])
        if (A.n and not acon.n) or (B.n and not bcon.n):
            shp = (A.shape[1 if c["tA"] == "T" else 0], B.shape[0 if c["tB"] == "T" else 1])
            r = O.Coo(shp, [np.empty(0, np.int32)] * 2, np.empty(0))
            d[f"m{s}_refub"] = np.array(1)
        else:
            r = ref.multiply_mm(c["C"], c["si"], A, c["tA"], c["sj"], B, c["tB"], c["sk"], c["policy"], c["zero_nan"])
        for nm, x in (("si", c["si"]), ("A", A), ("sj", c["sj"]), ("B", B), ("sk", c["sk"]), ("out", r)):
            put(d, f"m{s}_{nm}", x)
        d[f"m{s}_args"] = np.array([c["C"], ord(c["tA"]), ord(c["tB"]), c["policy"], c["zero_nan"]], np.float64)
    d["count"] = np.array(nmm)
    d.save(os.path.join(HERE, "multiply_mm_cases.npz"))

    # 4. multiply MV fuzz
    d = Packer()
    nmv = 150
    for s in range(nmv):
        c = _cases.mv_case(s)
        r = ref.multiply_mv(c["C"], c["si"], c["A"], c["tA"], c["sj"], c["V"], c["policy"], c["zero_nan"])
        for nm, x in (("si", c["si"]), ("A", c["A"]), ("sj", c["sj"]), ("V", c["V"]), ("out", r)):
            put(d, f"v{s}_{nm}", x)
        d[f"v{s}_args"] = np.array([c["C"], ord(c["tA"]), c["policy"], c["zero_nan"]], np.float64)
    d["count"] = np.array(nmv)
    d.save(os.path.join(HERE, "multiply_mv_cases.npz"))

    dense_ops()

    # 5. known answer of BASELINE config 2's generator at reduced size (SURVEY App. C #2 family)
    orc = O.port()
    a = orc.gen_dup_coo(0x5EED0002, 0, 300000, 210000, 12, 1024)
    r = ref.consolidate(a, (0, 1))
    w = np.arange(1, r.n + 1, dtype=np.uint64)
    chk = [int((w * a.astype(np.uint64)).sum()) for a in r.idx]  # position-weighted, mod 2^64
    np.savez_compressed(os.path.join(HERE, "config2_small.npz"), nnz=np.array(r.n), sum=np.array(r.val.sum()),
                        chk=np.array(chk, np.uint64), idx0=r.idx[0][::64], idx1=r.idx[1][::64], val=r.val[::64])
    print("golden fixtures written")


if __name__ == "__main__":
    if sys.argv[1:] == ["live", "restatement"]:
        print(live_cases(O.port()))
        sys.exit()
    assert ref is not None, "build oracle/_ref first"
    if sys.argv[1:] == ["live"]:
        print(live_cases(ref))
    elif sys.argv[1:] == ["dense"]:  # only the newest pack
        dense_ops()
    else:
        main()
