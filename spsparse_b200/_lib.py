"""ctypes binding of the C ABI in include/spsparse_b200.h.  Fails loudly when the CUDA library is
missing or cannot be loaded -- there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPB_LIB") or os.path.join(HERE, "lib", "libspsparse_b200.so")  # SPB_LIB: A/B experiments

i32p = C.POINTER(C.c_int32)
f64p = C.POINTER(C.c_double)
u64p = C.POINTER(C.c_uint64)
intp = C.POINTER(C.c_int)
vp = C.c_void_p


class ConsolidateStats(C.Structure):
    _fields_ = [("n_in", C.c_uint64), ("n_kept", C.c_uint64), ("n_out", C.c_uint64),
                ("key_bits", C.c_int), ("passes", C.c_int),
                ("ms_total", C.c_float), ("ms_sort", C.c_float), ("ms_reduce", C.c_float),
                ("ms_pass", C.c_float), ("digit_bits", C.c_int)]


class MMStats(C.Structure):
    _fields_ = [("products", C.c_uint64), ("nnz_a", C.c_uint64), ("nnz_b", C.c_uint64),
                ("rows_a", C.c_uint64), ("rows_merge", C.c_uint64), ("rows_esc", C.c_uint64),
                ("products_esc", C.c_uint64), ("nnz_c", C.c_uint64),
                ("rows_hash", C.c_uint64), ("products_hash", C.c_uint64),
                ("ms_prepare", C.c_float), ("ms_symbolic", C.c_float), ("ms_numeric", C.c_float),
                ("ms_total", C.c_float),
                ("ms_merge_count", C.c_float), ("ms_hash_count", C.c_float), ("ms_esc", C.c_float),
                ("ms_merge_numeric", C.c_float), ("ms_hash_emit", C.c_float), ("ms_hash_splits", C.c_float),
                ("ms_hash_numeric", C.c_float)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RowpartStats(C.Structure):
    _fields_ = [("a", ConsolidateStats), ("b", ConsolidateStats), ("mm", MMStats),
                ("rows_fetched", C.c_uint64), ("entries_fetched", C.c_uint64),
                ("ms_consolidate_a", C.c_float), ("ms_consolidate_b", C.c_float), ("ms_fetch", C.c_float),
                ("ms_side_stream", C.c_float), ("ms_fetch_wait", C.c_float), ("ms_total", C.c_float)]


# every symbol include/spsparse_b200.h declares: (name, restype, argtypes)
SIGNATURES = {
    "spb_last_error": (C.c_char_p, []),
    "spb_version": (C.c_int, []),
    "spb_ctx_create": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
    "spb_ctx_destroy": (C.c_int, [vp]),
    "spb_ctx_sync": (C.c_int, [vp]),
    "spb_ctx_device": (C.c_int, [vp, intp, C.POINTER(vp)]),
    "spb_ctx_trim": (C.c_int, [vp, u64p]),
    "spb_host_prefault": (C.c_int, [vp, C.c_uint64]),
    "spb_ctx_launch_count": (C.c_int, [vp, u64p]),
    "spb_coo_upload": (C.c_int, [vp, C.c_int, u64p, C.POINTER(i32p), f64p, C.c_uint64, intp, C.POINTER(vp)]),
    "spb_coo_wrap_device": (C.c_int, [vp, C.c_int, u64p, C.POINTER(vp), vp, C.c_uint64, intp, C.POINTER(vp)]),
    "spb_coo_alloc": (C.c_int, [vp, C.c_int, u64p, C.c_uint64, C.POINTER(vp)]),
    "spb_coo_info": (C.c_int, [vp, intp, u64p, u64p, intp]),
    "spb_coo_device_ptrs": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "spb_coo_dense_ptr": (C.c_int, [vp, vp, C.POINTER(vp), u64p]),
    "spb_coo_dense_ptr_range": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
    "spb_coo_copy": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "spb_coo_transpose": (C.c_int, [vp, vp, C.POINTER(C.c_int), C.POINTER(vp)]),
    "spb_coo_to_dense": (C.c_int, [vp, vp, C.c_int, C.POINTER(C.c_double)]),
    "spb_dense_to_coo": (C.c_int, [vp, C.c_int, u64p, C.POINTER(C.c_double), C.POINTER(vp)]),
    "spb_coo_wrap_csr": (C.c_int, [vp, u64p, C.c_int, vp, vp, vp, C.c_uint64, C.POINTER(vp)]),
    "spb_coo_set_sorted": (C.c_int, [vp, intp]),
    "spb_coo_download": (C.c_int, [vp, vp, C.POINTER(i32p), f64p]),
    "spb_coo_free": (C.c_int, [vp, vp]),
    "spb_consolidate": (C.c_int, [vp, vp, intp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(ConsolidateStats)]),
    "spb_sorted_permutation": (C.c_int, [vp, vp, intp, u64p]),
    "spb_consolidate_plan_create": (C.c_int, [vp, vp, intp, C.POINTER(vp), u64p]),
    "spb_consolidate_plan_run": (C.c_int, [vp, vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(ConsolidateStats)]),
    "spb_consolidate_plan_destroy": (C.c_int, [vp]),
    "spb_dim_beginnings": (C.c_int, [vp, vp, u64p, C.c_uint64, u64p]),
    "spb_multiply_mm": (C.c_int, [vp, C.c_double, vp, vp, C.c_char, vp, vp, C.c_char, vp, C.c_int, C.c_int,
                                  C.POINTER(vp), C.POINTER(MMStats)]),
    "spb_multiply_mm_prepared": (C.c_int, [vp, C.c_double, vp, vp, C.c_int, vp, vp, C.c_int, vp,
                                           C.POINTER(vp), C.POINTER(MMStats)]),
    "spb_mm_plan_create": (C.c_int, [vp, C.c_double, vp, vp, C.c_char, vp, vp, C.c_char, vp, C.c_int, C.c_int, C.c_uint64,
                                     C.POINTER(vp), u64p, u64p]),
    "spb_mm_plan_info": (C.c_int, [vp, C.c_uint64, i32p, i32p, u64p, u64p]),
    "spb_mm_plan_symbolic": (C.c_int, [vp, C.c_uint64, C.POINTER(MMStats)]),
    "spb_mm_plan_panel": (C.c_int, [vp, C.c_uint64, C.POINTER(vp), C.POINTER(MMStats)]),
    "spb_mm_plan_destroy": (C.c_int, [vp]),
    "spb_rowpart_create": (C.c_int, [vp, C.c_int, C.c_int, u64p, C.c_uint64, C.POINTER(vp)]),
    "spb_rowpart_handle": (C.c_int, [vp, vp, C.c_uint64]),
    "spb_rowpart_attach": (C.c_int, [vp, vp, C.c_uint64]),
    "spb_rowpart_multiply": (C.c_int, [vp, C.c_double, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.POINTER(vp),
                                       C.POINTER(RowpartStats)]),
    "spb_rowpart_destroy": (C.c_int, [vp]),
    "spb_multiply_mv": (C.c_int, [vp, C.c_double, vp, vp, C.c_char, vp, vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "spb_gen_dup_coo": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_uint64, C.POINTER(vp)]),
    "spb_gen_banded": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
    "spb_gen_regrid": (C.c_int, [vp, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(vp)]),
    "spb_gen_rmat": (C.c_int, [vp, C.c_uint64, C.c_int, C.c_uint64, C.POINTER(vp)]),
    "spb_gen_vector": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libspsparse_b200.so and binds every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m spsparse_b200.build` "
                          "(or __graft_entry__.build()); spsparse_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


class SpbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"spsparse_b200 error {code}: {msg}")
        self.code = code


def check(rc: int):
    if rc != 0:
        raise SpbError(rc, load().spb_last_error().decode(errors="replace"))
