"""Host-side Python mirror of the reference's interface for the hot path, over the C ABI.

Names follow the reference (slib/spsparse): ``CooArray`` plays ``VectorCooArray``
(VectorCooArray.hpp:8-158) with device-resident storage; ``consolidate`` / ``multiply`` take the
same arguments in the same order as algorithm.hpp:251-256 and multiply_sparse.hpp:152-164 /
281-291.  The C++ template layer in include/spsparse/ is the drop-in for C++ callers; this module
is what tests/ and bench.py drive.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import ConsolidateStats, MMPatternStats, MMStats, check, vp

LEAVE_ALONE, ADD, REPLACE = 0, 1, 2  # DuplicatePolicy, spsparse.hpp:25-26
ROW_MAJOR, COL_MAJOR = (0, 1), (1, 0)  # spsparse.cpp:30-31

ERR_INNER_DIM, ERR_NOT_SORTED = 3, 4


class Context:
    """One GPU + one CUDA stream (pass torch's ``stream.cuda_stream`` to share it)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = _lib.load()
        h = vp()
        check(self.lib.spb_ctx_create(device, vp(stream) if stream else None, C.byref(h)))
        self.h, self.device = h, device

    def sync(self):
        check(self.lib.spb_ctx_sync(self.h))

    def trim(self) -> int:
        """Hands the context's cached device blocks back to the driver (spb_ctx_trim); returns the bytes released."""
        freed = C.c_uint64(0)
        check(self.lib.spb_ctx_trim(self.h, C.byref(freed)))
        return freed.value

    def close(self):
        if self.h:
            self.lib.spb_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _order(so):
    if so is None:
        return None
    so = list(so) + [0]
    return (C.c_int * 2)(so[0], so[1])


class CooArray:
    """Device-resident COO array (int32 indices, fp64 values, rank 1 or 2)."""

    def __init__(self, ctx: Context, handle):
        self.ctx, self.h = ctx, handle

    # -- construction -------------------------------------------------------------------------
    @classmethod
    def from_host(cls, ctx, shape, idx, val, sort_order=None):
        shape = [int(s) for s in shape]
        rank = len(shape)
        idx = [np.ascontiguousarray(a, dtype=np.int32) for a in idx]
        val = np.ascontiguousarray(val, dtype=np.float64)
        n = int(val.shape[0])
        ptrs = (_lib.i32p * rank)(*[a.ctypes.data_as(_lib.i32p) for a in idx])
        h = vp()
        check(ctx.lib.spb_coo_upload(ctx.h, rank, (C.c_uint64 * rank)(*shape), ptrs, val.ctypes.data_as(_lib.f64p),
                                     n, _order(sort_order), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_netcdf(cls, ctx, path, vname):
        """The array stored under `vname` by ncio_spsparse (reference slib/spsparse/netcdf.hpp:86-138; classic-format files,
        spsparse_b200/ncio.py), uploaded as unsorted COO."""
        from . import ncio
        shape, idx, val = ncio.read_spsparse(path, vname)
        if any(s > 2 ** 31 for s in shape):
            raise ValueError(f"{vname}: shape {shape} does not fit 32-bit indices")
        return cls.from_host(ctx, shape, idx, val)

    def to_netcdf(self, path, vname):
        """Writes the array the way ncio_spsparse does (one array per file here; ncio.write_spsparse takes several)."""
        from . import ncio
        _, shape, _, _ = self._info()
        idx, val = self.to_host()
        ncio.write_spsparse(path, {vname: (tuple(shape), idx, val)})

    @classmethod
    def wrap_device(cls, ctx, shape, idx_ptrs, val_ptr, n, sort_order=None):
        shape = [int(s) for s in shape]
        rank = len(shape)
        ptrs = (vp * rank)(*[vp(int(p)) for p in idx_ptrs])
        h = vp()
        check(ctx.lib.spb_coo_wrap_device(ctx.h, rank, (C.c_uint64 * rank)(*shape), ptrs, vp(int(val_ptr)), int(n),
                                          _order(sort_order), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def wrap_csr(cls, ctx, shape, lead_dim, ptr, other_idx, val, n):
        """Consolidated matrix in compressed form (device pointers; see spb_coo_wrap_csr)."""
        h = vp()
        check(ctx.lib.spb_coo_wrap_csr(ctx.h, (C.c_uint64 * 2)(*[int(x) for x in shape]), int(lead_dim), vp(int(ptr)),
                                       vp(int(other_idx)), vp(int(val)), int(n), C.byref(h)))
        return cls(ctx, h)

    def dense_ptr(self):
        """(device pointer, extent) of the dense pointer over the leading sorted index (cached in the array)."""
        p = vp()
        ext = C.c_uint64()
        check(self.ctx.lib.spb_coo_dense_ptr(self.ctx.h, self.h, C.byref(p), C.byref(ext)))
        return p.value, int(ext.value)

    def dense_ptr_range(self, lo, hi):
        """Device pointer to the hi - lo + 1 values of the dense pointer for leading-index values lo..hi."""
        p = vp()
        check(self.ctx.lib.spb_coo_dense_ptr_range(self.ctx.h, self.h, int(lo), int(hi), C.byref(p)))
        return p.value

    # -- accessors ----------------------------------------------------------------------------
    def _info(self):
        rank = C.c_int()
        shape = (C.c_uint64 * 2)()
        n = C.c_uint64()
        so = (C.c_int * 2)()
        check(self.ctx.lib.spb_coo_info(self.h, C.byref(rank), shape, C.byref(n), so))
        r = rank.value
        return r, tuple(int(shape[k]) for k in range(r)), int(n.value), tuple(int(so[k]) for k in range(r))

    @property
    def rank(self):
        return self._info()[0]

    @property
    def shape(self):
        return self._info()[1]

    def size(self):
        return self._info()[2]

    @property
    def sort_order(self):
        so = self._info()[3]
        return None if so[0] < 0 else so

    def device_ptrs(self):
        idx = (vp * 2)()
        val = vp()
        check(self.ctx.lib.spb_coo_device_ptrs(self.h, idx, C.byref(val)))
        return [idx[k] for k in range(self.rank)], val.value

    def to_host(self, out=None):
        """Copies the entries to the host.  ``out=(idx_arrays, val_array)`` reuses caller buffers
        (e.g. pinned memory); they must be contiguous, int32 / float64, of exactly size() entries."""
        rank, shape, n, _ = self._info()
        if out is not None:
            idx, val = out
            assert all(a.dtype == np.int32 and a.flags.c_contiguous and a.shape[0] == n for a in idx)
            assert val.dtype == np.float64 and val.flags.c_contiguous and val.shape[0] == n
        else:
            idx = [np.empty(n, dtype=np.int32) for _ in range(rank)]
            val = np.empty(n, dtype=np.float64)
        ptrs = (_lib.i32p * rank)(*[a.ctypes.data_as(_lib.i32p) for a in idx])
        check(self.ctx.lib.spb_coo_download(self.ctx.h, self.h, ptrs, val.ctypes.data_as(_lib.f64p)))
        return idx, val

    def sorted_permutation(self, sort_order):
        """spsparse::sorted_permutation (algorithm.hpp:411-427)."""
        perm = np.empty(self.size(), dtype=np.uint64)
        check(self.ctx.lib.spb_sorted_permutation(self.ctx.h, self.h, _order(sort_order), perm.ctypes.data_as(_lib.u64p)))
        return perm.astype(np.int64)

    def dim_beginnings(self):
        """spsparse::dim_beginnings (algorithm.hpp:74-118)."""
        cnt = C.c_uint64()
        cap = self.size() + 1
        out = np.empty(cap, dtype=np.uint64)
        check(self.ctx.lib.spb_dim_beginnings(self.ctx.h, self.h, out.ctypes.data_as(_lib.u64p), cap, C.byref(cnt)))
        return out[:cnt.value].astype(np.int64)

    def free(self):
        if self.h:
            self.ctx.lib.spb_coo_free(self.ctx.h, self.h)
            self.h = None


def consolidate(ctx: Context, A: CooArray, sort_order, duplicate_policy=ADD, zero_nan=False, stats=False):
    """spsparse::consolidate (algorithm.hpp:251-319): returns the new, sorted array."""
    h = vp()
    st = ConsolidateStats()
    check(ctx.lib.spb_consolidate(ctx.h, A.h, _order(sort_order), int(duplicate_policy), int(bool(zero_nan)),
                                  C.byref(h), C.byref(st)))
    out = CooArray(ctx, h)
    return (out, st) if stats else out


def _plan_values(values, n):
    """(pointer, keep-alive) for n values given to a plan run: a CUDA float64 tensor, a numpy array (host memory) or a raw
    device pointer."""
    if isinstance(values, int):
        return values, None
    if isinstance(values, np.ndarray):
        v = np.ascontiguousarray(values, dtype=np.float64)
        if v.ndim != 1 or v.shape[0] != n:
            raise ValueError(f"values: {v.shape} for a plan of {n} entries")
        return v.ctypes.data, v
    if hasattr(values, "data_ptr") and getattr(values, "is_cuda", False):
        import torch
        if values.dtype != torch.float64 or values.dim() != 1 or values.numel() != n or values.stride(0) != 1:
            raise ValueError(f"values: need a contiguous float64 tensor of {n} entries")
        return values.data_ptr(), values
    raise TypeError("values: a CUDA float64 tensor, a numpy array or a device pointer")


class ConsolidatePlan:
    """``consolidate`` for a fixed index pattern (spb_consolidate_plan_*): the pattern of ``A`` is sorted once, and every
    ``run(values)`` returns what ``consolidate`` returns for ``A``'s indices with those values -- bit for bit -- with one
    gather pass and the duplicate-reduce instead of a sort.  ``A`` may be freed once the plan exists.  Device values are read on
    the context's stream: values written on another stream must be complete (synchronise, or share the stream)."""

    def __init__(self, ctx: Context, A: CooArray, sort_order):
        self.ctx = ctx
        self.n = A.size()
        h, runs = vp(), C.c_uint64()
        check(ctx.lib.spb_consolidate_plan_create(ctx.h, A.h, _order(sort_order), C.byref(h), C.byref(runs)))
        self.h, self.n_runs = h, int(runs.value)

    def _values(self, values):
        return _plan_values(values, self.n)

    def run(self, values, duplicate_policy=ADD, zero_nan=False, stats=False):
        ptr, _keep = self._values(values)   # _keep: a converted numpy copy must outlive the call
        h, st = vp(), ConsolidateStats()
        check(self.ctx.lib.spb_consolidate_plan_run(self.h, vp(ptr) if ptr else None, int(duplicate_policy),
                                                    int(bool(zero_nan)), C.byref(h), C.byref(st)))
        out = CooArray(self.ctx, h)
        return (out, st) if stats else out

    def free(self):
        if self.h:
            self.ctx.lib.spb_consolidate_plan_destroy(self.h)
            self.h = None


class MultiplyPattern:
    """``multiply`` for fixed operand patterns (spb_mm_pattern_*): the indices of ``A`` and ``B``, both transpose flags, ``Cst``,
    the scale vectors, the policy and ``zero_nan`` are fixed once, and every ``run(a_values, b_values)`` returns what
    ``multiply`` returns for ``A``'s and ``B``'s indices with those values -- bit for bit -- without sorting anything or
    repeating the symbolic phase.  ``A``, ``B`` and the scale vectors may be freed once the pattern exists.  Values are
    ``A.size()`` / ``B.size()`` doubles in entry order: CUDA float64 tensors, numpy arrays or device pointers (the same object
    may be passed twice); device values are read on the context's stream."""

    def __init__(self, ctx: Context, Cst, scalei, A, transpose_A, scalej, B, transpose_B, scalek,
                 duplicate_policy=ADD, zero_nan=False):
        self.ctx = ctx
        self.n_a, self.n_b = A.size(), B.size()
        h, bound = vp(), C.c_uint64()
        check(ctx.lib.spb_mm_pattern_create(ctx.h, float(Cst), _h(scalei), A.h, transpose_A.encode(), _h(scalej), B.h,
                                            transpose_B.encode(), _h(scalek), int(duplicate_policy), int(bool(zero_nan)),
                                            C.byref(h), C.byref(bound)))
        self.h, self.nnz_bound = h, int(bound.value)

    def run(self, a_values, b_values, stats=False):
        pa, _ka = _plan_values(a_values, self.n_a)   # _ka / _kb: converted numpy copies must outlive the call
        pb, _kb = _plan_values(b_values, self.n_b)
        if b_values is a_values:
            pb = pa   # one array for both operands: one staging of host values
        h, st = vp(), MMPatternStats()
        check(self.ctx.lib.spb_mm_pattern_run(self.h, vp(pa) if pa else None, vp(pb) if pb else None, C.byref(h), C.byref(st)))
        out = CooArray(self.ctx, h)
        return (out, st) if stats else out

    def free(self):
        if self.h:
            self.ctx.lib.spb_mm_pattern_destroy(self.h)
            self.h = None


def copy(ctx: Context, A: CooArray):
    """spsparse::copy (algorithm.hpp:30-37) into a fresh array."""
    h = vp()
    check(ctx.lib.spb_coo_copy(ctx.h, A.h, C.byref(h)))
    return CooArray(ctx, h)


def transpose(ctx: Context, A: CooArray, perm):
    """spsparse::transpose (algorithm.hpp:46-57): new dimension k takes old dimension perm[k]."""
    h = vp()
    check(ctx.lib.spb_coo_transpose(ctx.h, A.h, (C.c_int * 2)(*(list(perm) + [0])[:2]), C.byref(h)))
    return CooArray(ctx, h)


def to_dense(ctx: Context, A: CooArray, duplicate_policy=ADD):
    """VectorCooArray::to_dense (VectorCooArray.hpp:313-321; DenseAccum policies accum.hpp:110-140) -> numpy array."""
    dense = np.empty(tuple(A.shape), dtype=np.float64)
    if dense.size:
        check(ctx.lib.spb_coo_to_dense(ctx.h, A.h, int(duplicate_policy), dense.ctypes.data_as(_lib.f64p)))
    return dense


def to_sparse(ctx: Context, dense):
    """spsparse::to_sparse (algorithm.hpp:433-440): the elements != 0 of a dense array, in storage order."""
    dense = np.ascontiguousarray(dense, dtype=np.float64)
    h = vp()
    check(ctx.lib.spb_dense_to_coo(ctx.h, dense.ndim, (C.c_uint64 * dense.ndim)(*dense.shape),
                                   dense.ctypes.data_as(_lib.f64p), C.byref(h)))
    return CooArray(ctx, h)


def _h(x):
    return x.h if x is not None else None


def multiply(ctx: Context, Cst, scalei, A, transpose_A, scalej, B, transpose_B=None, scalek=None,
             duplicate_policy=ADD, zero_nan=False, stats=False):
    """spsparse::multiply.  With a rank-2 ``B`` this is the matrix*matrix form
    (multiply_sparse.hpp:152-248); with a rank-1 ``B`` (then ``transpose_B``/``scalek`` must be
    omitted) it is the matrix*vector form (multiply_sparse.hpp:281-365)."""
    h = vp()
    if B.rank == 1:
        check(ctx.lib.spb_multiply_mv(ctx.h, float(Cst), _h(scalei), A.h, transpose_A.encode(), _h(scalej), B.h,
                                      int(duplicate_policy), int(bool(zero_nan)), C.byref(h)))
        return CooArray(ctx, h)
    st = MMStats()
    check(ctx.lib.spb_multiply_mm(ctx.h, float(Cst), _h(scalei), A.h, transpose_A.encode(), _h(scalej), B.h,
                                  transpose_B.encode(), _h(scalek), int(duplicate_policy), int(bool(zero_nan)),
                                  C.byref(h), C.byref(st)))
    out = CooArray(ctx, h)
    return (out, st) if stats else out


def multiply_prepared(ctx: Context, Cst, scalei, A, a_row_dim, scalej, B, b_inner_dim, scalek):
    """SpGEMM on operands consolidated beforehand (A by (row, inner), B by (inner, col))."""
    h = vp()
    st = MMStats()
    check(ctx.lib.spb_multiply_mm_prepared(ctx.h, float(Cst), _h(scalei), A.h, int(a_row_dim), _h(scalej), B.h,
                                           int(b_inner_dim), _h(scalek), C.byref(h), C.byref(st)))
    return CooArray(ctx, h), st


class MultiplyPlan:
    """spsparse::multiply formed in row panels (spb_mm_plan_*): the A-row loop of the reference carries no state between
    rows (multiply_sparse.hpp:192-246), so ``panel(0), panel(1), ...`` concatenated are the result of ``multiply`` -- for
    products too large for one array (R-MAT 2^24 A*A)."""

    def __init__(self, ctx: Context, Cst, scalei, A, transpose_A, scalej, B, transpose_B, scalek,
                 duplicate_policy=ADD, zero_nan=False, max_products_per_panel=1 << 30):
        self.ctx = ctx
        self._keep = (scalei, scalej, scalek)  # used by the plan, not copied
        h, n, f = vp(), C.c_uint64(), C.c_uint64()
        check(ctx.lib.spb_mm_plan_create(ctx.h, float(Cst), _h(scalei), A.h, transpose_A.encode(), _h(scalej), B.h,
                                         transpose_B.encode(), _h(scalek), int(duplicate_policy), int(bool(zero_nan)),
                                         int(max_products_per_panel), C.byref(h), C.byref(n), C.byref(f)))
        self.h, self.n_panels, self.products = h, int(n.value), int(f.value)
        shp = (C.c_uint64 * 2)()
        check(ctx.lib.spb_mm_plan_info(self.h, self.n_panels, None, None, None, shp))
        self.shape = (int(shp[0]), int(shp[1]))

    def info(self, p):
        """(first row index, last row index, intermediate products) of panel p"""
        a, b, f = C.c_int32(), C.c_int32(), C.c_uint64()
        check(self.ctx.lib.spb_mm_plan_info(self.h, int(p), C.byref(a), C.byref(b), C.byref(f), None))
        return int(a.value), int(b.value), int(f.value)

    def symbolic(self, p) -> MMStats:
        st = MMStats()
        check(self.ctx.lib.spb_mm_plan_symbolic(self.h, int(p), C.byref(st)))
        return st

    def panel(self, p, stats=False):
        h, st = vp(), MMStats()
        check(self.ctx.lib.spb_mm_plan_panel(self.h, int(p), C.byref(h), C.byref(st)))
        out = CooArray(self.ctx, h)
        return (out, st) if stats else out

    def free(self):
        if self.h:
            self.ctx.lib.spb_mm_plan_destroy(self.h)
            self.h = None


# ---- synthetic inputs on the device (SURVEY.md Appendix C) ------------------------------------
def gen_dup_coo(ctx, seed, i0, n, ubase, bits, zero_every=0):
    h = vp()
    check(ctx.lib.spb_gen_dup_coo(ctx.h, seed, i0, n, ubase, bits, zero_every, C.byref(h)))
    return CooArray(ctx, h)


def gen_banded(ctx, seed, m, r0, r1):
    h = vp()
    check(ctx.lib.spb_gen_banded(ctx.h, seed, m, r0, r1, C.byref(h)))
    return CooArray(ctx, h)


def gen_regrid(ctx, seed, ny, nx, gy, gx):
    h = vp()
    check(ctx.lib.spb_gen_regrid(ctx.h, seed, ny, nx, gy, gx, C.byref(h)))
    return CooArray(ctx, h)


def gen_rmat(ctx, seed, scale, nedges):
    h = vp()
    check(ctx.lib.spb_gen_rmat(ctx.h, seed, scale, nedges, C.byref(h)))
    return CooArray(ctx, h)


def gen_vector(ctx, seed, dim):
    h = vp()
    check(ctx.lib.spb_gen_vector(ctx.h, seed, dim, C.byref(h)))
    return CooArray(ctx, h)
