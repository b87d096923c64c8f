/*
 * spsparse_b200.h -- C ABI of the B200-native spsparse hot path (libspsparse_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  The reference
 * (citibeth/spsparse) is a header-only C++ template library with no FFI of its own, so each entry
 * point below names the reference routine it replaces (paths relative to the reference tree);
 * the C++ template layer in include/spsparse/ (same names and argument order as the reference)
 * is a thin host wrapper over these calls -- see INTEGRATION.md.
 *
 * Types: IndexT = int32 (non-negative), ValT = double, rank 1 or 2 -- the instantiation used by
 * every reference test (tests/test_multiply_sparse.cpp:90-97, tests/test_array.cpp:68).
 *
 * Conventions
 *  - every function returns 0 (SPB_OK) or an SPB_ERR_* code; spb_last_error() gives the text
 *    (thread-local).  Nothing throws across the ABI.  There is NO CPU fallback: a missing or
 *    failing GPU is an error.
 *  - calls are synchronous for the caller unless noted; one CUDA stream per context.
 *  - `spb_coo` handles own device memory unless created by spb_coo_wrap_device; free them with
 *    spb_coo_free.  No function keeps a host pointer after it returns.
 */
#ifndef SPSPARSE_B200_H
#define SPSPARSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct spb_ctx spb_ctx; /* device + stream + workspace pool */
typedef struct spb_coo spb_coo; /* device-resident COO array (struct-of-arrays, like
                                   VectorCooArray::index_vecs/val_vec, VectorCooArray.hpp:22-23) */

enum {
    SPB_OK = 0,
    SPB_ERR_CUDA = 1,       /* CUDA runtime failure (message has the CUDA error string) */
    SPB_ERR_ARG = 2,        /* bad argument (null pointer, rank, index out of bounds, ...) */
    SPB_ERR_INNER_DIM = 3,  /* multiply: inner dimensions differ (multiply_sparse.hpp:172-174) */
    SPB_ERR_NOT_SORTED = 4, /* dim_beginnings on an unsorted array (algorithm.hpp:82-84) */
    SPB_ERR_TOO_LARGE = 5   /* 2^31 or more entries in one array (the reference's own cap, algorithm.hpp:419) */
};

/* DuplicatePolicy, same order as spsparse.hpp:25-26 */
enum { SPB_LEAVE_ALONE = 0, SPB_ADD = 1, SPB_REPLACE = 2 };

const char *spb_last_error(void);
int spb_version(void);

/* ---- context --------------------------------------------------------------------------- */
/* cuda_stream: a cudaStream_t to run on (e.g. torch's current stream), or NULL to create one. */
int spb_ctx_create(int device, void *cuda_stream, spb_ctx **out);
int spb_ctx_destroy(spb_ctx *ctx);
int spb_ctx_sync(spb_ctx *ctx);
int spb_ctx_device(const spb_ctx *ctx, int *device, void **cuda_stream);
/* The context keeps freed device blocks for reuse (the hot path asks for the same multi-GB scratch sizes every call).
 * spb_ctx_trim waits for the stream and hands every cached block back to the driver -- for processes that share the GPU
 * with another allocator; released_bytes (may be NULL) reports how much. */
int spb_ctx_trim(spb_ctx *ctx, uint64_t *released_bytes);
/* Host-side helper for callers that download multi-GB results into freshly reserved (never touched) memory, e.g. the tail of
 * a std::vector after reserve(): writes a zero into every page of [p, p + bytes) from several threads, so that the page
 * faults of the first touch -- 1 GB/s from one thread, the dominant cost of spsparse::multiply into an empty VectorCooArray --
 * are taken in parallel.  Needs no GPU and no context. */
int spb_host_prefault(void *p, uint64_t bytes);
/* kernels launched through this context so far (measurement aid) */
int spb_ctx_launch_count(const spb_ctx *ctx, uint64_t *launches);

/* ---- COO arrays  (VectorCooArray, VectorCooArray.hpp:8-158) ---------------------------- */
/* sort_order: NULL or {-1,..} = unsorted/edit mode; else the order the data is ALREADY sorted
 * and consolidated in (what VectorCooArray::sort_order records, VectorCooArray.hpp:33-34,131-135). */
int spb_coo_upload(spb_ctx *ctx, int rank, const uint64_t *shape, const int32_t *const *idx,
                   const double *val, uint64_t n, const int *sort_order, spb_coo **out);
/* Wraps caller-owned device arrays without copying (used for NCCL-gathered operands). */
int spb_coo_wrap_device(spb_ctx *ctx, int rank, const uint64_t *shape, int32_t *const *d_idx,
                        double *d_val, uint64_t n, const int *sort_order, spb_coo **out);
/* Uninitialised device storage for n entries (filled by the generators below or by the caller). */
int spb_coo_alloc(spb_ctx *ctx, int rank, const uint64_t *shape, uint64_t n, spb_coo **out);
int spb_coo_info(const spb_coo *a, int *rank, uint64_t *shape /*[rank]*/, uint64_t *n,
                 int *sort_order /*[rank]*/);
int spb_coo_device_ptrs(const spb_coo *a, int32_t **d_idx /*[rank]*/, double **d_val);
/* Dense pointer over the leading sorted index of a consolidated rank-2 array: ptr[v] = offset of the first
 * entry whose index[sort_order[0]] >= v, for v in [0, extent]; device memory owned by (and cached in) `a`. */
int spb_coo_dense_ptr(spb_ctx *ctx, const spb_coo *a, uint32_t **d_ptr, uint64_t *extent);
/* The same pointer for the leading-index values lo..hi only: d_ptr[v - lo] for v in [lo, hi], hi - lo + 1 values,
 * offsets absolute within `a`.  Costs O(rows of a + hi - lo) instead of O(extent): what a rank of the
 * row-partitioned multiply uses for its own shard of B. */
int spb_coo_dense_ptr_range(spb_ctx *ctx, const spb_coo *a, uint64_t lo, uint64_t hi, uint32_t **d_ptr);
/* Wraps a consolidated matrix given in compressed form (caller-owned device memory, not copied): a dense
 * pointer d_ptr[shape[lead_dim]+1] over dimension lead_dim, plus the other dimension's index and the value of
 * every entry.  Only usable as the B operand of spb_multiply_mm_prepared (b_inner_dim = lead_dim) -- this is how
 * the multi-GPU path hands over the replicated B without shipping its redundant row-index array. */
int spb_coo_wrap_csr(spb_ctx *ctx, const uint64_t *shape, int lead_dim, uint32_t *d_ptr, int32_t *d_other_idx,
                     double *d_val, uint64_t n, spb_coo **out);
int spb_coo_set_sorted(spb_coo *a, const int *sort_order); /* VectorCooArray::set_sorted :131-135 */
int spb_coo_download(spb_ctx *ctx, const spb_coo *a, int32_t *const *idx, double *val);
int spb_coo_free(spb_ctx *ctx, spb_coo *a);

/* ---- consolidate  (spsparse::consolidate, algorithm.hpp:251-319; sorted_permutation :411-427;
 *      the in-place form VectorCooArray::consolidate, VectorCooArray.hpp:299-311) -------------
 * Stable sort by (idx[sort_order[0]], idx[sort_order[1]]), zero inputs dropped, NaN inputs dropped
 * only in the leading run when zero_nan, duplicates merged by `policy`; index columns keep the
 * array's own dimension order.  `out` is a new array flagged sorted by sort_order. */
typedef struct {
    uint64_t n_in, n_kept, n_out; /* entries in, after the input-zero drop, after merging */
    int key_bits, passes;         /* significant key bits, radix passes run */
    float ms_total, ms_sort, ms_reduce;
    float ms_pass; /* mean duration of one radix scatter pass (passes after the first), 0 if only one */
    int digit_bits; /* width of a radix digit: 8, or 9 where that saves a pass */
} spb_consolidate_stats;
int spb_consolidate(spb_ctx *ctx, const spb_coo *in, const int *sort_order, int policy, int zero_nan,
                    spb_coo **out, spb_consolidate_stats *stats /* may be NULL */);

/* ---- consolidate with a fixed index pattern  (spsparse::consolidate, algorithm.hpp:251-319) ----------------------
 * For callers that assemble the same (row, column) pattern again and again with new values (a time step, a regridding
 * step): the pattern is sorted once, and every later consolidate of new values over it is one gather pass plus the
 * duplicate-reduce -- no sort.  The result of a run depends on the values as consolidate's does (zeros dropped, NaNs of the
 * leading run dropped with zero_nan, the policy's fold) and is bit-identical to spb_consolidate on the same data.
 *
 * spb_consolidate_plan_create  sorts the index pattern of `in` once (stable, every entry kept, nothing merged); the values
 *                              of `in` are not read.  Index bounds are checked here, with spb_consolidate's errors.  `in`
 *                              may be freed afterwards.  The plan holds 12 bytes of device memory per entry (the sorted
 *                              packed keys and the 32-bit permutation).  n_runs (may be NULL): distinct index tuples.
 * spb_consolidate_plan_run     what spb_consolidate(ctx, X, sort_order, policy, zero_nan) returns, where X has the plan's
 *                              indices and the values `val`: n doubles in the entry order of the array the plan was made
 *                              from.  `val` may be device memory of the plan's device (any 8-byte alignment) or host memory
 *                              (staged as spb_coo_upload stages it).  `out` is a new array flagged sorted by sort_order.
 *                              stats: passes = 0 (no radix pass runs), ms_sort = the gather pass (with zero_nan also the
 *                              search for the leading run's end), n_kept / n_out of this run.
 * spb_consolidate_plan_destroy releases the plan; call it before destroying the plan's context. */
typedef struct spb_cons_plan spb_cons_plan;
int spb_consolidate_plan_create(spb_ctx *ctx, const spb_coo *in, const int *sort_order, spb_cons_plan **out,
                                uint64_t *n_runs /* may be NULL */);
int spb_consolidate_plan_run(spb_cons_plan *plan, const double *val, int policy, int zero_nan, spb_coo **out,
                             spb_consolidate_stats *stats /* may be NULL */);
int spb_consolidate_plan_destroy(spb_cons_plan *plan);

/* ---- sorted_permutation  (spsparse::sorted_permutation, algorithm.hpp:411-427) -----------
 * perm[t] = position in `in` of the entry that a stable sort by sort_order puts at position t.
 * Writes in->n values to host memory.  Nothing is dropped or merged. */
int spb_sorted_permutation(spb_ctx *ctx, const spb_coo *in, const int *sort_order, uint64_t *perm);

/* ---- dim_beginnings  (spsparse::dim_beginnings, algorithm.hpp:74-118) -------------------
 * Offsets of the first entry of every non-empty value of dimension sort_order[0], plus the
 * sentinel n.  Writes min(count, cap) offsets to host memory, returns the full count. */
int spb_dim_beginnings(spb_ctx *ctx, const spb_coo *sorted, uint64_t *out, uint64_t cap, uint64_t *count);

/* ---- copy / transpose / to_dense / to_sparse: the steps either side of the path -----------
 * spb_coo_copy       spsparse::copy into a fresh array            algorithm.hpp:30-37
 * spb_coo_transpose  spsparse::transpose(ret, A, perm)            algorithm.hpp:46-57: new dimension k takes old
 *                    dimension perm[k] (indices AND shape); entries keep their order; result not flagged sorted
 * spb_coo_to_dense   VectorCooArray::to_dense                     VectorCooArray.hpp:313-321, with the duplicate policies
 *                    of DenseAccum (accum.hpp:110-140; the method itself uses ADD).  `dense` is a HOST array of
 *                    prod(shape) doubles, row-major, overwritten.  Out-of-bounds indices are an error.
 * spb_dense_to_coo   spsparse::to_sparse                          algorithm.hpp:433-440: every element != 0 (NaN
 *                    included) of a HOST row-major array, in storage order; result not flagged sorted */
int spb_coo_copy(spb_ctx *ctx, const spb_coo *in, spb_coo **out);
int spb_coo_transpose(spb_ctx *ctx, const spb_coo *in, const int *perm /*[rank]*/, spb_coo **out);
int spb_coo_to_dense(spb_ctx *ctx, const spb_coo *in, int policy, double *dense);
int spb_dense_to_coo(spb_ctx *ctx, int rank, const uint64_t *shape, const double *dense, spb_coo **out);

/* ---- multiply, matrix*matrix  (spsparse::multiply, multiply_sparse.hpp:152-248) ---------
 * out = C * diag(si) * op(A) * diag(sj) * op(B) * diag(sk); scale vectors may be NULL; they are
 * used as stored and must be ascending and non-repeating (xiter.hpp:146, 201), else SPB_ERR_ARG.  A and B are consolidated internally unless already
 * flagged sorted in the order the reference needs (Consolidate<>, algorithm.hpp:354-369).
 * The result is row-major sorted, unique, exact-zero sums dropped, and -- like the reference's --
 * left flagged unsorted / in edit mode. */
typedef struct {
    uint64_t products;       /* F: intermediate products a*b formed */
    uint64_t nnz_a, nnz_b;   /* after consolidation */
    uint64_t rows_a;         /* non-empty rows of op(A) */
    uint64_t rows_merge;     /* rows done by the register k-way-merge kernels */
    uint64_t rows_esc;       /* rows done by expand-sort-compress */
    uint64_t products_esc;
    uint64_t nnz_c;
    uint64_t rows_hash;      /* longer rows done by the bitmap + shared-memory hash-accumulator kernels */
    uint64_t products_hash;
    float ms_prepare;        /* consolidations of A and B, CSR build, scale densify */
    float ms_symbolic, ms_numeric, ms_total;
    /* inside ms_symbolic: register-merge count kernel; bitmap count pass of the hash bin; expand-sort-compress */
    float ms_merge_count, ms_hash_count, ms_esc;
    /* inside ms_numeric: register-merge numeric kernel; hash bin: column emit pass, window searches, accumulators */
    float ms_merge_numeric, ms_hash_emit, ms_hash_splits, ms_hash_numeric;
} spb_mm_stats;
int spb_multiply_mm(spb_ctx *ctx, double C, const spb_coo *scalei, const spb_coo *A, char transpose_A,
                    const spb_coo *scalej, const spb_coo *B, char transpose_B, const spb_coo *scalek,
                    int policy, int zero_nan, spb_coo **out, spb_mm_stats *stats /* may be NULL */);

/* Operands prepared once, multiply many times (what bench.py times as "SpGEMM only").
 * A must be consolidated with sort_order {a_row_dim, 1-a_row_dim}; B with {b_inner_dim, 1-b_inner_dim}
 * (i.e. sorted by the inner index first).  Same arithmetic and output as spb_multiply_mm. */
int spb_multiply_mm_prepared(spb_ctx *ctx, double C, const spb_coo *scalei, const spb_coo *A,
                             int a_row_dim, const spb_coo *scalej, const spb_coo *B, int b_inner_dim,
                             const spb_coo *scalek, spb_coo **out, spb_mm_stats *stats);

/* ---- multiply in row panels -----------------------------------------------------------------
 * The A-row loop of spsparse::multiply carries no state from one row to the next
 * (multiply_sparse.hpp:192-246): the product can be formed one panel -- a contiguous range of the
 * non-empty rows of op(A) -- at a time, and the panels' results, concatenated in panel order, are
 * exactly what spb_multiply_mm returns.  This is the way to products that no single array can
 * hold (>= 2^31 entries, the reference's own cap, algorithm.hpp:419; or more bytes than the GPU
 * has): R-MAT 2^24 rows A*A has 3*10^10 outputs.
 *
 * spb_mm_plan_create   consolidates A and B as spb_multiply_mm does (once), counts the intermediate
 *                      products of every row and cuts the rows into panels of about
 *                      max_products_per_panel products each (a single row is never cut).  The scale
 *                      vectors are used, not copied: they must outlive the plan.  A and B may be freed.
 * spb_mm_plan_info     which rows of C panel p holds (first/last row index), its product count, and the
 *                      shape of C (multiply_sparse.hpp:169).  panel >= n_panels: only `shape` is written.
 * spb_mm_plan_symbolic symbolic phase of one panel only: exact product count and bins, and the panel's
 *                      output count (exact, except that outputs of the register-merge and hash-accumulator bins whose
 *                      terms cancel to exactly 0 are still counted: the symbolic phase reads no values) -- no result
 *                      array is allocated.
 * spb_mm_plan_panel    the panel's rows of C, as spb_multiply_mm would have produced them. */
typedef struct spb_mm_plan spb_mm_plan;
int spb_mm_plan_create(spb_ctx *ctx, double C, const spb_coo *scalei, const spb_coo *A, char transpose_A,
                       const spb_coo *scalej, const spb_coo *B, char transpose_B, const spb_coo *scalek,
                       int policy, int zero_nan, uint64_t max_products_per_panel, spb_mm_plan **out,
                       uint64_t *n_panels, uint64_t *products);
int spb_mm_plan_info(const spb_mm_plan *plan, uint64_t panel, int32_t *first_row, int32_t *last_row,
                     uint64_t *products, uint64_t *shape /*[2]*/);
int spb_mm_plan_symbolic(spb_mm_plan *plan, uint64_t panel, spb_mm_stats *stats);
int spb_mm_plan_panel(spb_mm_plan *plan, uint64_t panel, spb_coo **out, spb_mm_stats *stats /* may be NULL */);
int spb_mm_plan_destroy(spb_mm_plan *plan);

/* ---- row-partitioned multiply on the GPUs of one node ---------------------------------------
 * One process per GPU.  The A-row loop of spsparse::multiply carries no state between rows
 * (multiply_sparse.hpp:192-246): every rank holds a block of the rows of A (blocks that tile A's rows in rank
 * order) and emits those rows of C = c * diag(si) * A * diag(sj) * B * diag(sk); the ranks' results concatenated
 * in rank order are the reference's output.  B is sharded by ITS rows (the inner index): rank r owns rows
 * [row_lo[r], row_lo[r+1]).  Every call each rank consolidates its shard of B,
 * publishes it in compressed form in a buffer the other ranks have mapped (CUDA IPC, NVLink), and fetches --
 * with loads from the peers' memory, under its own consolidate(A) -- the rows of B its block of A can
 * reference: the interval hull of the inner indices of its A entries (a banded block: its shard plus a halo; a
 * general one: all of B), or all of B when fetch_all != 0.  Sizes, offsets and the hand-shake stay on the
 * devices; the host is not involved between the kernels of a step.  The reference has no counterpart (it is
 * single-process); SURVEY.md section 8e.
 *
 * spb_rowpart_create   collective: same row_lo[n_ranks+1] (row_lo[0] = 0) and cap_entries (upper bound of the
 *                      consolidated entries of any rank's shard of B) on every rank
 * spb_rowpart_handle   64-byte handle of this rank's shard buffer; the caller all-gathers the handles of all ranks
 *                      (MPI, torch.distributed, a file -- any means) ...
 * spb_rowpart_attach   ... and hands the n_ranks handles, in rank order, to every rank
 * spb_rowpart_multiply collective: every rank calls it once per step, also when its own block is empty.  A and B
 *                      are this rank's raw blocks (any order, duplicates allowed; blocks already flagged sorted
 *                      {0,1} are used as they are), indices are GLOBAL.  No transposes: op(A) = A, op(B) = B. */
typedef struct spb_rowpart spb_rowpart;
typedef struct {
    spb_consolidate_stats a, b;   /* this rank's block of A, its shard of B */
    spb_mm_stats mm;
    uint64_t rows_fetched, entries_fetched;   /* rows / entries of B this rank fetched (own shard included) */
    float ms_consolidate_a, ms_consolidate_b;
    float ms_fetch;         /* duration of the fetch kernel on its own stream (overlaps consolidate(A)) */
    float ms_side_stream;   /* hull + wait for the peers + fetch + scale vector, on the side stream */
    float ms_fetch_wait;    /* what the multiply still had to wait for after consolidate(A) */
    float ms_total;
} spb_rowpart_stats;
int spb_rowpart_create(spb_ctx *ctx, int rank, int n_ranks, const uint64_t *row_lo, uint64_t cap_entries, spb_rowpart **out);
int spb_rowpart_handle(spb_rowpart *rp, void *handle, uint64_t handle_bytes /* >= 64 */);
int spb_rowpart_attach(spb_rowpart *rp, const void *handles /* n_ranks x handle_bytes */, uint64_t handle_bytes);
int spb_rowpart_multiply(spb_rowpart *rp, double C, const spb_coo *scalei, const spb_coo *A_block, const spb_coo *scalej,
                         const spb_coo *B_shard, const spb_coo *scalek, int policy, int zero_nan, int fetch_all,
                         spb_coo **out, spb_rowpart_stats *stats /* may be NULL */);
int spb_rowpart_destroy(spb_rowpart *rp);

/* ---- multiply, matrix*vector  (spsparse::multiply, multiply_sparse.hpp:281-365) -------- */
int spb_multiply_mv(spb_ctx *ctx, double C, const spb_coo *scalei, const spb_coo *A, char transpose_A,
                    const spb_coo *scalej, const spb_coo *V, int policy, int zero_nan, spb_coo **out);

/* ---- synthetic inputs, generated on the device (SURVEY.md Appendix C; the same arithmetic as
 *      oracle/spsparse_oracle.c:orc_gen_* and spsparse_b200/gen.py) --------------------------- */
/* config 2 family: n entries [i0, i0+n) over `ubase` distinct draws in a 2^bits x 2^bits shape. */
int spb_gen_dup_coo(spb_ctx *ctx, uint64_t seed, uint64_t i0, uint64_t n, uint64_t ubase, int bits,
                    uint64_t zero_every, spb_coo **out);
/* config 5 family: rows [r0, r1) of an m x m pentadiagonal matrix, 5 entries per row inserted in a
 * scrambled order; out-of-range diagonals are emitted as explicit 0.0 entries on the clamped column. */
int spb_gen_banded(spb_ctx *ctx, uint64_t seed, uint64_t m, uint64_t r0, uint64_t r1, spb_coo **out);
/* config 3 family: (ny*nx) x (gy*gx) bilinear-overlap matrix, 4 entries per row, scrambled. */
int spb_gen_regrid(spb_ctx *ctx, uint64_t seed, uint32_t ny, uint32_t nx, uint32_t gy, uint32_t gx,
                   spb_coo **out);
/* config 4 family: R-MAT, 2^scale rows/cols, nedges raw edges (duplicates kept). */
int spb_gen_rmat(spb_ctx *ctx, uint64_t seed, int scale, uint64_t nedges, spb_coo **out);
/* dense-support sparse vector: indices 0..dim-1 ascending, value 0.5+u01(seed+j), flagged sorted. */
int spb_gen_vector(spb_ctx *ctx, uint64_t seed, uint64_t dim, spb_coo **out);

#ifdef __cplusplus
}
#endif
#endif /* SPSPARSE_B200_H */
