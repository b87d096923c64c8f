"""ctypes front-end for the parity oracle -- TEST INFRASTRUCTURE ONLY.

Loads ``oracle/liboracle.so`` (the plain-C restatement, ``spsparse_oracle.c``) and, when it has
been built, ``oracle/_ref/libspsparse_ref.so`` (the GENUINE reference headers behind the same C
interface, ``ref_shim.cpp``).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
CPU-baseline / ``--impl reference`` legs may import this module; nothing under ``spsparse_b200/``
does.  Reference citations live in the C sources.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LEAVE_ALONE, ADD, REPLACE = 0, 1, 2  # spsparse.hpp:25-26
ROW_MAJOR, COL_MAJOR = (0, 1), (1, 0)  # spsparse.cpp:30-31

_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f64p = C.POINTER(C.c_double)


class _Mat(C.Structure):
    _fields_ = [("shape", C.c_uint64 * 2), ("n", C.c_int64), ("idx0", _i32p), ("idx1", _i32p),
                ("val", _f64p), ("sort_order", C.c_int * 2)]


class _Vec(C.Structure):
    _fields_ = [("shape", C.c_uint64), ("n", C.c_int64), ("idx", _i32p), ("val", _f64p),
                ("sort_order", C.c_int)]


@dataclass
class Coo:
    """Host COO matrix/vector as the caller of the reference would hold it."""
    shape: tuple
    idx: list  # list of int32 arrays, one per dimension
    val: np.ndarray
    sort_order: tuple = None  # None => unsorted / edit mode (sort_order[0] == -1)

    def __post_init__(self):
        self.idx = [np.ascontiguousarray(a, dtype=np.int32) for a in self.idx]
        self.val = np.ascontiguousarray(self.val, dtype=np.float64)
        self.shape = tuple(int(s) for s in self.shape)

    @property
    def n(self):
        return int(self.val.shape[0])

    @property
    def rank(self):
        return len(self.shape)


def _p32(a):
    return a.ctypes.data_as(_i32p)


def _p64f(a):
    return a.ctypes.data_as(_f64p)


def _mat(m: Coo):
    s = _Mat()
    s.shape[0], s.shape[1] = m.shape
    s.n = m.n
    s.idx0, s.idx1, s.val = _p32(m.idx[0]), _p32(m.idx[1]), _p64f(m.val)
    so = m.sort_order if m.sort_order is not None else (-1, 0)
    s.sort_order[0], s.sort_order[1] = so
    return s


def _vec(v: Coo):
    if v is None:
        return None
    s = _Vec()
    s.shape = v.shape[0]
    s.n = v.n
    s.idx, s.val = _p32(v.idx[0]), _p64f(v.val)
    s.sort_order = -1 if v.sort_order is None else v.sort_order[0]
    return s


def _ref(x):
    return None if x is None else C.byref(x)


class InnerDimError(Exception):
    pass


class Impl:
    """One implementation of the oracle interface (prefix 'orc' = restatement, 'ref' = genuine)."""

    def __init__(self, lib: C.CDLL, prefix: str):
        self.lib, self.prefix = lib, prefix
        self.kind = "port" if prefix == "orc" else "reference"
        f = self._f
        f("free").argtypes = [C.c_void_p]
        f("free").restype = None
        f("sorted_permutation").argtypes = [C.c_int, C.c_int64, _i32p, _i32p, C.POINTER(C.c_int), _i64p]
        f("sorted_permutation").restype = None
        f("consolidate").argtypes = [C.c_int, C.c_int64, _i32p, _i32p, _f64p, C.POINTER(C.c_int),
                                     C.c_int, C.c_int, _i32p, _i32p, _f64p]
        f("consolidate").restype = C.c_int64
        f("join").argtypes = [_i32p, C.c_int64, _i32p, C.c_int64, _i32p, C.c_int64, _i32p]
        f("join").restype = C.c_int64
        mm = [C.c_double, C.POINTER(_Vec), C.POINTER(_Mat), C.c_char, C.POINTER(_Vec), C.POINTER(_Mat),
              C.c_char, C.POINTER(_Vec), C.c_int, C.c_int, C.POINTER(C.c_uint64), _i64p,
              C.POINTER(_i32p), C.POINTER(_i32p), C.POINTER(_f64p)]
        if prefix == "orc":
            f("dim_beginnings").argtypes = [C.c_int64, _i32p, _i64p]
            f("multiply_mm").argtypes = mm + [_i64p]
            f("multiply_mm_pairs").argtypes = mm
            f("multiply_mm_pairs").restype = C.c_int
            f("gen_dup_coo").argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int64,
                                         _i32p, _i32p, _f64p]
            f("gen_dup_coo").restype = None
        else:
            f("dim_beginnings").argtypes = [C.c_int64, _i32p, _i32p, C.POINTER(C.c_int), _i64p]
            f("multiply_mm").argtypes = mm + [_f64p]
            f("consolidate_timed").argtypes = [C.c_int64, _i32p, _i32p, _f64p, C.POINTER(C.c_int),
                                               C.c_int, C.c_int, _i64p, _f64p]
            f("consolidate_timed").restype = C.c_double
        f("dim_beginnings").restype = C.c_int64
        u64p = C.POINTER(C.c_uint64)
        f("transpose").argtypes = [C.c_int, C.c_int64, _i32p, _i32p, C.POINTER(C.c_int), _i32p, _i32p]
        f("transpose").restype = None
        f("to_dense").argtypes = [C.c_int, u64p, C.c_int64, _i32p, _i32p, _f64p, C.c_int, _f64p]
        f("to_dense").restype = C.c_int
        f("to_sparse").argtypes = [C.c_int, u64p, _f64p, _i32p, _i32p, _f64p]
        f("to_sparse").restype = C.c_int64
        f("multiply_mm").restype = C.c_int
        f("multiply_mv").argtypes = [C.c_double, C.POINTER(_Vec), C.POINTER(_Mat), C.c_char,
                                     C.POINTER(_Vec), C.POINTER(_Vec), C.c_int, C.c_int,
                                     C.POINTER(C.c_uint64), _i64p, C.POINTER(_i32p), C.POINTER(_f64p)]
        f("multiply_mv").restype = C.c_int

    def _f(self, name):
        return getattr(self.lib, f"{self.prefix}_{name}")

    # ---- algorithm.hpp:411-427
    def sorted_permutation(self, a: Coo, sort_order):
        perm = np.empty(a.n, dtype=np.int64)
        so = (C.c_int * 2)(*(list(sort_order) + [0])[:2])
        i1 = _p32(a.idx[1]) if a.rank > 1 else None
        self._f("sorted_permutation")(a.rank, a.n, _p32(a.idx[0]), i1, so, perm.ctypes.data_as(_i64p))
        return perm

    # ---- algorithm.hpp:251-319
    def consolidate(self, a: Coo, sort_order, policy=ADD, zero_nan=False) -> Coo:
        n = a.n
        o0 = np.empty(max(n, 1), dtype=np.int32)
        o1 = np.empty(max(n, 1), dtype=np.int32)
        ov = np.empty(max(n, 1), dtype=np.float64)
        so = (C.c_int * 2)(*(list(sort_order) + [0])[:2])
        i1 = _p32(a.idx[1]) if a.rank > 1 else None
        m = self._f("consolidate")(a.rank, n, _p32(a.idx[0]), i1, _p64f(a.val), so, int(policy),
                                   int(bool(zero_nan)), _p32(o0), _p32(o1), _p64f(ov))
        idx = [o0[:m].copy()] + ([o1[:m].copy()] if a.rank > 1 else [])
        return Coo(a.shape, idx, ov[:m].copy(), tuple(sort_order))

    # ---- algorithm.hpp:74-118
    def dim_beginnings(self, a: Coo):
        assert a.sort_order is not None
        out = np.empty(a.n + 1, dtype=np.int64)
        if self.prefix == "orc":
            m = self._f("dim_beginnings")(a.n, _p32(a.idx[a.sort_order[0]]), out.ctypes.data_as(_i64p))
        else:
            so = (C.c_int * 2)(*a.sort_order)
            m = self._f("dim_beginnings")(a.n, _p32(a.idx[0]), _p32(a.idx[1]), so, out.ctypes.data_as(_i64p))
        return out[:m].copy()

    # ---- algorithm.hpp:46-57 (copy :30-37 is the identity permutation)
    def transpose(self, a: Coo, perm) -> Coo:
        n = a.n
        o0 = np.empty(max(n, 1), dtype=np.int32)
        o1 = np.empty(max(n, 1), dtype=np.int32)
        pm = (C.c_int * 2)(*(list(perm) + [0])[:2])
        i1 = _p32(a.idx[1]) if a.rank > 1 else None
        self._f("transpose")(a.rank, n, _p32(a.idx[0]), i1, pm, _p32(o0), _p32(o1))
        idx = [o0[:n].copy()] + ([o1[:n].copy()] if a.rank > 1 else [])
        return Coo(tuple(a.shape[p] for p in perm), idx, np.array(a.val, dtype=np.float64, copy=True), None)

    # ---- VectorCooArray.hpp:313-321 + accum.hpp:110-140
    def to_dense(self, a: Coo, policy=ADD) -> np.ndarray:
        dense = np.empty(tuple(int(x) for x in a.shape), dtype=np.float64)
        shp = (C.c_uint64 * 2)(*(list(a.shape) + [1])[:2])
        i1 = _p32(a.idx[1]) if a.rank > 1 else None
        rc = self._f("to_dense")(a.rank, shp, a.n, _p32(a.idx[0]), i1, _p64f(a.val), int(policy), _p64f(dense))
        if rc != 0:
            raise ValueError("to_dense: index out of bounds")
        return dense

    # ---- algorithm.hpp:433-440
    def to_sparse(self, dense: np.ndarray) -> Coo:
        dense = np.ascontiguousarray(dense, dtype=np.float64)
        cells = max(dense.size, 1)
        o0 = np.empty(cells, dtype=np.int32)
        o1 = np.empty(cells, dtype=np.int32)
        ov = np.empty(cells, dtype=np.float64)
        shp = (C.c_uint64 * 2)(*(list(dense.shape) + [1])[:2])
        m = self._f("to_sparse")(dense.ndim, shp, _p64f(dense), _p32(o0), _p32(o1), _p64f(ov))
        idx = [o0[:m].copy()] + ([o1[:m].copy()] if dense.ndim > 1 else [])
        return Coo(tuple(dense.shape), idx, ov[:m].copy(), None)

    # ---- xiter.hpp Join2Xiter / Join3Xiter
    def join(self, a, b, c=None):
        a = np.ascontiguousarray(a, dtype=np.int32)
        b = np.ascontiguousarray(b, dtype=np.int32)
        cc = None if c is None else np.ascontiguousarray(c, dtype=np.int32)
        out = np.empty(max(len(a), 1), dtype=np.int32)
        m = self._f("join")(_p32(a), len(a), _p32(b), len(b), None if cc is None else _p32(cc),
                            -1 if cc is None else len(cc), _p32(out))
        return out[:m].copy()

    def _take(self, n, pi, pk, pv):
        def arr(p, dt):
            if n == 0 or not p:
                return np.empty(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(n,)).astype(dt, copy=True)
        i = arr(pi, np.int32)
        k = arr(pk, np.int32) if pk is not None else None
        v = arr(pv, np.float64)
        for p in (pi, pk, pv):
            if p is not None and p:
                self._f("free")(C.cast(p, C.c_void_p))
        return i, k, v

    # ---- multiply_sparse.hpp:152-248
    def multiply_mm(self, Cst, si, A: Coo, tA, sj, B: Coo, tB, sk, policy=ADD, zero_nan=False,
                    pairs=False, want_stats=False):
        mA, mB = _mat(A), _mat(B)
        vi, vj, vk = _vec(si), _vec(sj), _vec(sk)
        shp = (C.c_uint64 * 2)()
        n = C.c_int64()
        pi, pk, pv = _i32p(), _i32p(), _f64p()
        args = [float(Cst), _ref(vi), C.byref(mA), tA.encode(), _ref(vj), C.byref(mB), tB.encode(), _ref(vk),
                int(policy), int(bool(zero_nan)), shp, C.byref(n), C.byref(pi), C.byref(pk), C.byref(pv)]
        stats = None
        if pairs:
            rc = self._f("multiply_mm_pairs")(*args)
        elif self.prefix == "orc":
            st = (C.c_int64 * 4)()
            rc = self._f("multiply_mm")(*args, st)
            stats = dict(F=st[0], nnzA=st[1], nnzB=st[2], rowsA=st[3])
        else:
            sec = C.c_double()
            rc = self._f("multiply_mm")(*args, C.byref(sec))
            stats = dict(seconds=sec.value)
        i, k, v = self._take(n.value, pi, pk, pv)
        if rc != 0:
            raise InnerDimError()
        out = Coo((shp[0], shp[1]), [i, k], v, None)  # left in edit mode (SURVEY App. A M10)
        return (out, stats) if want_stats else out

    # ---- multiply_sparse.hpp:281-365
    def multiply_mv(self, Cst, si, A: Coo, tA, sj, V: Coo, policy=ADD, zero_nan=False) -> Coo:
        mA = _mat(A)
        vi, vj, vv = _vec(si), _vec(sj), _vec(V)
        shp = C.c_uint64()
        n = C.c_int64()
        pi, pv = _i32p(), _f64p()
        rc = self._f("multiply_mv")(float(Cst), _ref(vi), C.byref(mA), tA.encode(), _ref(vj), C.byref(vv),
                                    int(policy), int(bool(zero_nan)), C.byref(shp), C.byref(n),
                                    C.byref(pi), C.byref(pv))
        i, _, v = self._take(n.value, pi, None, pv)
        if rc != 0:
            raise InnerDimError()
        return Coo((shp.value,), [i], v, None)

    # ---- SURVEY Appendix C, config 2 family (restatement library only)
    def gen_dup_coo(self, seed, i0, n, ubase, bits, zero_every=0):
        row = np.empty(n, dtype=np.int32)
        col = np.empty(n, dtype=np.int32)
        val = np.empty(n, dtype=np.float64)
        self.lib.orc_gen_dup_coo(seed, i0, n, ubase, bits, zero_every, _p32(row), _p32(col), _p64f(val))
        return Coo((1 << bits, 1 << bits), [row, col], val, None)

    def consolidate_timed(self, a: Coo, sort_order=ROW_MAJOR, policy=ADD, zero_nan=False):
        """Genuine reference only: seconds spent inside spsparse::consolidate, nnz out, sum of values."""
        assert self.prefix == "ref"
        so = (C.c_int * 2)(*sort_order)
        n_out, s = C.c_int64(), C.c_double()
        sec = self._f("consolidate_timed")(a.n, _p32(a.idx[0]), _p32(a.idx[1]), _p64f(a.val), so, int(policy),
                                           int(bool(zero_nan)), C.byref(n_out), C.byref(s))
        return sec, n_out.value, s.value


def reference_dir():
    """The checkout of the original spsparse (github.com/citibeth/spsparse) that SPSPARSE_REFERENCE names, or None when
    the variable is unset.  A value that names no such checkout is an error, not a reason to skip the reference."""
    d = os.environ.get("SPSPARSE_REFERENCE")
    if not d:
        return None
    if not (os.path.isfile(os.path.join(d, "slib", "spsparse", "spsparse.cpp")) and os.path.isdir(os.path.join(d, "tests"))):
        raise FileNotFoundError(f"SPSPARSE_REFERENCE={d!r} is not a checkout of spsparse (slib/spsparse/spsparse.cpp and tests/)")
    return d


def build(ref: bool = True) -> None:
    """Compile the oracle (and, when SPSPARSE_REFERENCE names a checkout of the original spsparse, the genuine
    reference; oracle/Makefile reads the same variable)."""
    subprocess.run(["make", "-s", "-C", HERE, "oracle"], check=True)
    if ref and reference_dir():
        subprocess.run(["make", "-s", "-C", HERE, "ref"], check=True)


_cache = {}


def port() -> Impl:
    """The plain-C restatement (always available; built on demand)."""
    if "orc" not in _cache:
        so = os.path.join(HERE, "liboracle.so")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(HERE, "spsparse_oracle.c")):
            build(ref=False)
        _cache["orc"] = Impl(C.CDLL(so), "orc")
    return _cache["orc"]


def reference() -> Impl | None:
    """The genuine reference behind the same interface, or None when oracle/_ref was not built."""
    if "ref" not in _cache:
        so = os.path.join(HERE, "_ref", "libspsparse_ref.so")
        _cache["ref"] = Impl(C.CDLL(so), "ref") if os.path.exists(so) else None
    return _cache["ref"]
