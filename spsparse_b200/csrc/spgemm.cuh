// spgemm.cuh -- row-wise sparse*sparse multiply  C = c * diag(si) * op(A) * diag(sj) * op(B) * diag(sk).
//
// Replaces the loop nest of spsparse::multiply (reference slib/spsparse/multiply_sparse.hpp:192-246)
// and its Join2Xiter/Join3Xiter merge-joins (xiter.hpp:149-278, next_noincr_body.hpp:1-53).  The
// reference evaluates every (row of A) x (column of B) pair; here each non-empty row i of op(A)
// merges the rows B[j,:] of the inner indices j it holds (Gustavson).  Contract kept (SURVEY.md
// App. A M6-M10): rows/cols absent from or zero in scalei/scalek are excluded; j absent from
// scalej is excluded; every output (i,k) adds its terms (a*s)*b in ascending j starting from 0;
// it is emitted iff the sum != 0, as ((sum*C)*a_scale)*b_scale, in (i asc, k asc) order.
//
// Rows are binned by intermediate-product count:
//   short rows (<= MERGE_MAX_LISTS inner indices, <= merge_max_products products): one THREAD per
//     row runs a k-way merge of the (already column-sorted) B rows entirely in registers -- the
//     heads of the lists are compared, equal columns are summed in list (= ascending j) order.
//     A symbolic pass counts, a scan places the rows, the numeric pass repeats the merge and writes.
//   longer rows (>= hash_min_products products; wide matrices in column windows of the bitmap's size):
//     symbolic = bitmap of the products' columns, whose set bits in order are the sorted outputs;
//     numeric = shared-memory hash table column -> output rank with accumulators in rank order,
//     products added entry after entry (ascending j).
//   everything else: expand-sort-compress through global memory with the radix sort / duplicate-
//     reduce kernels of consolidate (keys (row number, k), stable => terms still in ascending j).
// Every bin is deterministic and its sums are bit-identical to the reference's.
#pragma once
#include "common.cuh"

constexpr int MERGE_MAX_LISTS = 8;
#ifndef MR_MIN_BLOCKS
#define MR_MIN_BLOCKS 1
#endif
enum { ROW_SKIP = 0, ROW_MERGE = 1, ROW_ESC = 2, ROW_HASH = 3 };

struct MMOperands {
    // op(A), consolidated, sorted by (row, inner): compressed rows
    const i32 *a_j;
    const double *a_val;
    u32 nnz_a;
    const i32 *arow_id;     // [nrows] row index i of each non-empty row
    const u32 *arow_start;  // [nrows+1]
    u32 nrows;
    // op(B), consolidated, sorted by (inner, col): dense pointer over the inner index
    const u32 *bptr;  // [nj+1]
    const i32 *b_k;
    const double *b_val;
    // dense-ified scale vectors (nullptr when the argument was NULL)
    const double *si;             // [rows of op(A)]  absent = 0 => row excluded
    const double *sj;             // [inner]
    const unsigned char *sj_mask; // [inner]          absent => term excluded
    const double *sk;             // [cols of op(B)]  absent = 0 => column excluded
    double C;
    int debug;  // experiments only (SPB_MERGE_DEBUG): 1 = skip the global stores, 2 = plain (non-streaming) stores
};

// ---- longest compressed row (picks the register-merge kernels' NLMAX) ----------------------------------
__global__ void k_row_maxlen(const u32 *__restrict__ row_start, u32 nrows, u32 *out) {
    u32 best = 0;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (u64)gridDim.x * blockDim.x)
        best = max(best, row_start[r + 1] - row_start[r]);
    best = __reduce_max_sync(SPB_FULL_MASK, best);
    if (lane_id() == 0 && best) atomicMax(out, best);
}

// ---- per A entry: number of products it forms (0 if its row or its j is excluded) -------------
__global__ void k_entry_products(MMOperands m, const i32 *__restrict__ a_row, u32 *ent_f) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < m.nnz_a; e += (u64)gridDim.x * blockDim.x) {
        i32 j = m.a_j[e];
        u32 f = m.bptr[(u32)j + 1] - m.bptr[j];
        if (m.sj_mask && !m.sj_mask[j]) f = 0;
        if (m.si && m.si[a_row[e]] == 0.0) f = 0;
        ent_f[e] = f;
    }
}

// ---- long rows only: product count per row from the per-entry prefix sums; second-level binning -----
// Long rows with at least hash_min_products products go to the bitmap + hash-accumulator kernels (ROW_HASH; only
// offered when the output columns fit the shared-memory bitmap), the rest stay with expand-sort-compress (ROW_ESC).
// stats: [0] F merged rows, [1] rows merged, [2] rows long (ESC+HASH), [3] F ESC rows, [4] F HASH rows, [5] rows HASH
// ROW_HASH rows with at most hash_small_max products go to hash_rows (k_hash_symbolic_small lists their columns by sorting them in
// shared memory, whatever the width of the matrix), the others to hash_rows_big (bitmap, column windows); stats[6] / [7] count them.
__global__ void k_esc_row_products(MMOperands m, const u64 *__restrict__ ent_off, unsigned char *row_cls, u64 *esc_f,
                                   u64 hash_min_products, u64 hash_small_max, u32 *hash_rows, u32 *hash_rows_big, ull *stats) {
    u64 f_esc = 0, f_hash = 0;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < m.nrows; r += (u64)gridDim.x * blockDim.x) {
        u64 f = 0;
        if (row_cls[r] == ROW_ESC) {
            f = ent_off[m.arow_start[r + 1]] - ent_off[m.arow_start[r]];
            if (hash_rows && f >= hash_min_products) {
                row_cls[r] = ROW_HASH;
                atomicAdd(&stats[5], 1ull);
                if (f <= hash_small_max) hash_rows[atomicAdd(&stats[6], 1ull)] = (u32)r;
                else hash_rows_big[atomicAdd(&stats[7], 1ull)] = (u32)r;
                f_hash += f;
                f = 0;
            }
        }
        esc_f[r] = f;
        f_esc += f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        f_esc += __shfl_xor_sync(SPB_FULL_MASK, f_esc, o);
        f_hash += __shfl_xor_sync(SPB_FULL_MASK, f_hash, o);
    }
    if (lane_id() == 0) {
        if (f_esc) atomicAdd(&stats[3], (ull)f_esc);
        if (f_hash) atomicAdd(&stats[4], (ull)f_hash);
    }
}

// ---- short rows: k-way merge in registers, one thread per row -----------------------------------
// The heads of up to NL column-sorted B rows live in registers; each step takes the smallest head
// column, sums every list that holds it in list (= ascending j) order and advances those lists.
// Heads are compared unsigned and an exhausted list holds MERGE_END, a value no column can take (columns are < 2^31):
// column 2^31-1 = INT32_MAX is a real column of a matrix 2^31 wide.
constexpr u32 MERGE_END = 0xffffffffu;
// Where a merge reads B from: the global arrays (k0 = j0 = 0, read-only cache loads), or -- LOCAL -- the copies a block made in
// shared memory of the stretch of B its rows reference (k0 / j0 = first entry / first row of that stretch).
struct BView {
    const i32 *k;
    const double *v;
    const u32 *p;
    u32 k0, j0;
};
template <bool LOCAL> __device__ __forceinline__ i32 bv_k(const BView &b, u32 e) { return LOCAL ? b.k[e - b.k0] : __ldg(b.k + e); }
template <bool LOCAL> __device__ __forceinline__ double bv_v(const BView &b, u32 e) { return LOCAL ? b.v[e - b.k0] : __ldg(b.v + e); }
template <bool LOCAL> __device__ __forceinline__ u32 bv_p(const BView &b, u32 j) { return LOCAL ? b.p[j - b.j0] : __ldg(b.p + j); }

template <int NL, bool LOCAL = false>
struct RowMerge {
    u32 cur[NL], end[NL];
    u32 hk[NL];   // head column, MERGE_END once the list is exhausted
    double hv[NL], as[NL];
    BView b;

    __device__ __forceinline__ void init(const MMOperands &m, u32 s, u32 len, const BView *view = nullptr) {
        if (view) b = *view;
        else { b.k = m.b_k; b.v = m.b_val; b.p = m.bptr; b.k0 = 0; b.j0 = 0; }
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            cur[l] = end[l] = 0;
            hk[l] = MERGE_END;
            hv[l] = 0.0;
            as[l] = 0.0;
            if ((u32)l < len) {
                i32 j = __ldg(m.a_j + s + l);
                double a = __ldg(m.a_val + s + l);
                bool ok = !m.sj_mask || m.sj_mask[j];
                if (ok) {
                    cur[l] = bv_p<LOCAL>(b, (u32)j);
                    end[l] = bv_p<LOCAL>(b, (u32)j + 1);
                    as[l] = m.sj ? __dmul_rn(a, __ldg(m.sj + j)) : a;  // (a*s) first, multiply_sparse.hpp:228
                    if (cur[l] < end[l]) {
                        hk[l] = (u32)bv_k<LOCAL>(b, cur[l]);
                        hv[l] = bv_v<LOCAL>(b, cur[l]);
                    }
                }
            }
        }
    }

    // Sum of everything init() loaded.  Callers compare it against an impossible value before entering
    // their merge loop: that one real consumer makes the loop-invariant registers (as[], the row scale)
    // "arrived" for ptxas.  Without it every iteration re-waits on their scoreboard slot, which by then is
    // shared with the freshly issued next-head loads -- the step then stalls a full L2 round trip on the
    // loads it only needs in the NEXT step (profiles/r01_merge_numeric_notes.md).
    __device__ __forceinline__ double touch() const {
        double t = 0.0;
#pragma unroll
        for (int l = 0; l < NL; ++l) t += as[l];
        return t;
    }

    // Next output column and its dot product; false when every list is exhausted.
    __device__ __forceinline__ bool next(const MMOperands &m, i32 &k, double &sum) {
        u32 kmin = hk[0];
#pragma unroll
        for (int l = 1; l < NL; ++l) kmin = min(kmin, hk[l]);
        if (kmin == MERGE_END) return false;
        double acc = 0.0;  // multiply_sparse.hpp:219
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            if (hk[l] == kmin) {
                acc = __dadd_rn(acc, __dmul_rn(as[l], hv[l]));
                ++cur[l];
                if (cur[l] < end[l]) {
                    hk[l] = (u32)bv_k<LOCAL>(b, cur[l]);
                    hv[l] = bv_v<LOCAL>(b, cur[l]);
                } else {
                    hk[l] = MERGE_END;
                }
            }
        }
        k = (i32)kmin;
        sum = acc;
        return true;
    }
};

// The same merge over the COLUMNS only: what the symbolic pass needs.  Three registers per list instead of seven, no loads of
// B's or A's values, no arithmetic.  It counts the distinct unmasked columns of the row; an output whose terms cancel to exactly
// 0 (dropped by the reference, multiply_sparse.hpp:238) is therefore still counted -- the numeric pass finds it and leaves a
// tombstone that the compaction pass (k_live_flags / k_compact_entries, shared with the hash bin) closes.  Rare: exact
// cancellation only.  Config 5 count pass 7.3 -> 4.3 ms, config 3 2.4 -> 1.6 ms.
template <int NL, bool LOCAL = false>
struct RowMergeK {
    u32 cur[NL], end[NL];
    u32 hk[NL];   // as in RowMerge
    BView b;
    __device__ __forceinline__ void init(const MMOperands &m, u32 s, u32 len, const BView *view = nullptr) {
        if (view) b = *view;
        else { b.k = m.b_k; b.v = m.b_val; b.p = m.bptr; b.k0 = 0; b.j0 = 0; }
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            cur[l] = end[l] = 0;
            hk[l] = MERGE_END;
            if ((u32)l < len) {
                const i32 j = __ldg(m.a_j + s + l);
                if (!m.sj_mask || m.sj_mask[j]) {
                    cur[l] = bv_p<LOCAL>(b, (u32)j);
                    end[l] = bv_p<LOCAL>(b, (u32)j + 1);
                    if (cur[l] < end[l]) hk[l] = (u32)bv_k<LOCAL>(b, cur[l]);
                }
            }
        }
    }
    __device__ __forceinline__ bool next(i32 &k) {
        u32 kmin = hk[0];
#pragma unroll
        for (int l = 1; l < NL; ++l) kmin = min(kmin, hk[l]);
        if (kmin == MERGE_END) return false;
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            if (hk[l] == kmin) {
                ++cur[l];
                hk[l] = cur[l] < end[l] ? (u32)bv_k<LOCAL>(b, cur[l]) : MERGE_END;
            }
        }
        k = (i32)kmin;
        return true;
    }
};

// keep iff sum != 0 (NaN kept, multiply_sparse.hpp:238) and the column's scale is present and non-zero
__device__ __forceinline__ bool keep_output(const MMOperands &m, i32 k, double sum, double &b_scale) {
    b_scale = 1.0;
    bool keep = (sum != 0.0);
    if (m.sk) {
        b_scale = __ldg(m.sk + k);
        keep = keep && (b_scale != 0.0);
    }
    return keep;
}

// ---- LOCAL variants of the merge kernels: the block's stretch of B in shared memory ---------------------------------------
// Matrices with row locality (banded, stencil-like: consecutive rows of A reference neighbouring rows of B) make a block's
// 128 rows read one short CONTIGUOUS stretch of B -- rows jlo..jhi of a row-sorted B are adjacent in memory.  The block copies
// that stretch (row pointers, columns, values) into shared memory once, with coalesced loads, and its merges then chase their
// list heads at shared-memory latency instead of one L2 round trip per step.  Blocks whose rows reach too far (the stretch
// does not fit) run the ordinary global-memory merge: nothing is assumed about the matrix.
constexpr int ML_JCAP = 1024;      // rows of B a block may stage
constexpr int ML_CAP_COUNT = 1536; // entries of B, count kernel (22 KB per block)
constexpr int ML_CAP_NUM = 1024;   // entries of B, numeric kernel (next to its 26 KB of output staging)
template <int CAP, int JCAP = ML_JCAP>
struct BStage {
    i32 k[CAP];
    double v[CAP];
    u32 p[JCAP + 2];
    u32 red[2][4];
};
// jlo..jhi: the inner indices of this thread's row (jlo > jhi: none).  Block-uniform result; three barriers.
template <int CAP, int JCAP>
__device__ __forceinline__ bool stage_b(const MMOperands &m, BStage<CAP, JCAP> &sm, u32 jlo, u32 jhi, BView &view) {
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    jlo = __reduce_min_sync(SPB_FULL_MASK, jlo);
    jhi = __reduce_max_sync(SPB_FULL_MASK, jhi);
    if (lane == 0) { sm.red[0][warp] = jlo; sm.red[1][warp] = jhi; }
    __syncthreads();
    u32 JLO = sm.red[0][0], JHI = sm.red[1][0];
    for (u32 w = 1; w < (blockDim.x >> 5); ++w) { JLO = min(JLO, sm.red[0][w]); JHI = max(JHI, sm.red[1][w]); }
    bool ok = JLO <= JHI && JHI - JLO < (u32)JCAP;
    if (ok)
        for (u32 t = tid; t < JHI - JLO + 2; t += blockDim.x) sm.p[t] = __ldg(m.bptr + JLO + t);
    __syncthreads();
    u32 seg0 = 0, seg1 = 0;
    if (ok) {
        seg0 = sm.p[0];
        seg1 = sm.p[JHI - JLO + 1];
        ok = seg1 - seg0 <= (u32)CAP;
    }
    if (ok)
        for (u32 t = tid; t < seg1 - seg0; t += blockDim.x) {
            sm.k[t] = ld_stream_i32(m.b_k + seg0 + t);
            sm.v[t] = ld_stream_f64(m.b_val + seg0 + t);
        }
    __syncthreads();
    view.k = sm.k; view.v = sm.v; view.p = sm.p; view.k0 = seg0; view.j0 = JLO;
    return ok;
}

// symbolic: bin the row and, for a short row, count its outputs exactly
template <int NL, bool LOCAL = false>
__device__ __forceinline__ int count_row(const MMOperands &m, u32 s, u32 len, u32 max_products, u32 &count, u64 &f, const BView *view = nullptr) {
    RowMergeK<NL, LOCAL> st;
    st.init(m, s, len, view);
    f = 0;
#pragma unroll
    for (int l = 0; l < NL; ++l) f += st.end[l] - st.cur[l];
    count = 0;
    if (f == 0) return ROW_SKIP;
    if (f > max_products) return ROW_ESC;
    i32 k;
    while (st.next(k))
        if (!m.sk || __ldg(m.sk + k) != 0.0) ++count;   // columns excluded by scalek are never outputs (:208-213)
    return ROW_MERGE;
}

// Registers: a merge of NL lists keeps 7 registers per list live (cursor, end, head column, head value, scaled A
// value).  Compiled for eight lists the kernels need 78-86 registers and run 20 warps per SM, which is what bounds
// them -- every step waits an L2 round trip for the heads it advanced.  NLMAX = the longest row of op(A) that can
// take the merge, rounded up to 2/4/6/8 (the host knows it): configs 3 and 5 (4 and 5 entries per row) get kernels
// with half the registers and twice the warps.
template <int NLMAX> struct MergeBlocks { static constexpr int value = NLMAX <= 4 ? 8 : NLMAX <= 6 ? 7 : 5; };  // (NL = 6: 72 registers = 7 blocks; at 74 the kernel loses a block and 11 % of its speed)

// stats: MC_STRIPES stripes of 8 counters, one cache line apart in pairs -- [0] F of merged rows, [1] rows merged, [2] rows
// ESC, [6] longest row of op(A) (entries); a warp adds its totals to one stripe (warps take the stripes in turn) and the host sums the
// stripes.  (One set of counters for the whole grid, one atomic per warp, made this kernel wait for the L2 atomic unit of a
// single address: 6 M atomics on one cache line in a 6.5 ms kernel.)
constexpr int MC_STRIPES = 64;
template <int NLMAX, bool LOCAL = false>
__global__ void __launch_bounds__(128, MergeBlocks<NLMAX>::value) k_merge_count(MMOperands m, u32 max_products, unsigned char *row_cls,
                                                     u32 *row_cnt, ull *stats) {
    __shared__ BStage<LOCAL ? ML_CAP_COUNT : 1, LOCAL ? ML_JCAP : 1> s_b;
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    int cls = ROW_SKIP;
    u32 c = 0;
    u64 f = 0;
    u32 s = 0, len = 0;
    bool on = false;
    if (r < m.nrows) {
        s = m.arow_start[r];
        len = m.arow_start[r + 1] - s;
        on = !m.si || m.si[m.arow_id[r]] != 0.0;  // row excluded by scalei (multiply_sparse.hpp:195)
    }
    BView view;
    bool staged = false;
    if (LOCAL) {
        u32 jlo = 0xffffffffu, jhi = 0;
        if (on && len <= (u32)MERGE_MAX_LISTS)
            for (u32 l = 0; l < len; ++l) {
                const u32 j = (u32)__ldg(m.a_j + s + l);
                jlo = min(jlo, j);
                jhi = max(jhi, j);
            }
        staged = stage_b(m, s_b, jlo, jhi, view);
        if (staged && threadIdx.x == 0) atomicAdd(&stats[(size_t)(blockIdx.x % MC_STRIPES) * 8 + 3], 1ull);   // blocks that ran from shared memory
    }
    if (r < m.nrows) {
        if (on) {
            if (len > (u32)MERGE_MAX_LISTS) cls = ROW_ESC;   // products counted later, from the per-entry prefix sums
            else if (LOCAL && staged) {
                if (len <= 2) cls = count_row<2, true>(m, s, len, max_products, c, f, &view);
                else if (NLMAX >= 4 && len <= 4) cls = count_row<(NLMAX >= 4 ? 4 : 2), true>(m, s, len, max_products, c, f, &view);
                else if (NLMAX >= 6 && len <= 6) cls = count_row<(NLMAX >= 6 ? 6 : 2), true>(m, s, len, max_products, c, f, &view);
                else if (NLMAX >= 8) cls = count_row<(NLMAX >= 8 ? 8 : 2), true>(m, s, len, max_products, c, f, &view);
            }
            else if (len <= 2) cls = count_row<2>(m, s, len, max_products, c, f);
            else if (NLMAX >= 4 && len <= 4) cls = count_row<(NLMAX >= 4 ? 4 : 2)>(m, s, len, max_products, c, f);
            else if (NLMAX >= 6 && len <= 6) cls = count_row<(NLMAX >= 6 ? 6 : 2)>(m, s, len, max_products, c, f);
            else if (NLMAX >= 8) cls = count_row<(NLMAX >= 8 ? 8 : 2)>(m, s, len, max_products, c, f);
        }
        row_cls[r] = (unsigned char)cls;
        if (cls != ROW_ESC) row_cnt[r] = c;  // ESC rows are filled by the expand-sort-compress stage
    }
    u64 f_merge = (cls == ROW_MERGE) ? f : 0;
    u32 n_merge = (cls == ROW_MERGE), n_esc = (cls == ROW_ESC);
    const u32 mylen = r < m.nrows ? m.arow_start[r + 1] - m.arow_start[r] : 0u;
    const u32 maxlen = __reduce_max_sync(SPB_FULL_MASK, mylen);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        f_merge += __shfl_xor_sync(SPB_FULL_MASK, f_merge, o);
        n_merge += __shfl_xor_sync(SPB_FULL_MASK, n_merge, o);
        n_esc += __shfl_xor_sync(SPB_FULL_MASK, n_esc, o);
    }
    if (lane_id() == 0) {
        // one stripe per warp in turn: 64 addresses share what a single one had to take
        ull *mine = stats + (size_t)((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) % MC_STRIPES) * 8;
        if (f_merge) atomicAdd(&mine[0], (ull)f_merge);
        if (n_merge) atomicAdd(&mine[1], (ull)n_merge);
        if (n_esc) atomicAdd(&mine[2], (ull)n_esc);
        if (maxlen > (u32)mine[6]) atomicMax(&mine[6], (ull)maxlen);
    }
}

// numeric: the 32 rows of a warp advance in lock step; outputs are staged per lane in shared memory and
// flushed as contiguous runs (lane l's run is written by 16 lanes at once), so C is written in full
// sectors instead of one 4/8-byte store per thread per step.
constexpr int MR_THREADS = 128;

// The symbolic pass counted the distinct unmasked columns of the row without reading a value; an output whose terms cancel to
// exactly 0 is dropped by the reference (:238).  It keeps its slot here as a TOMBSTONE (column and row index -1) -- every counted
// slot is written, in order -- and the lanes that wrote any add to *shrunk; the host then runs the compaction pass it already has
// for the hash bin.  Nothing is added to the common path but a select per stored entry (checking the rows' ranges, or counting what
// was produced, in this kernel cost 0.4-1.0 ms of its 8.9 on config 5: profiles/r02_notes.md).
template <int NL, int STAGE, bool LOCAL = false>
__device__ __forceinline__ void merge_rows_warp(const MMOperands &m, bool mine, u32 s, u32 len, i32 irow,
                                                u64 dst, i32 *sk, double *sv, i32 *c_i, i32 *c_k, double *c_v, u32 *shrunk, const BView *view = nullptr) {
    constexpr int PITCH = STAGE + 1;
    constexpr int RUNS = 32 / STAGE;  // lanes' runs written per flush iteration
    const u32 lane = lane_id();
    RowMerge<NL, LOCAL> st;
    st.init(m, s, mine ? len : 0, view);
    double a_scale = 1.0;
    if (mine && m.si) a_scale = m.si[irow];
    u32 cnt = 0;
    bool active = mine;
    u32 ndead = 0;
    if (st.touch() + a_scale + (double)dst == -1.2345678e300) active = false;  // never true; see RowMerge::touch
    for (;;) {
        if (active) {
            i32 k;
            double sum, b_scale = 1.0;
            if (!st.next(m, k, sum)) active = false;
            else {
                bool masked = false;   // columns excluded by scalek are never outputs (:208-213) and were not counted
                if (m.sk) { b_scale = __ldg(m.sk + k); masked = b_scale == 0.0; }
                if (!masked) {
                    const bool dead = !(sum != 0.0);   // :238 (NaN != 0 is kept)
                    sk[lane * PITCH + cnt] = dead ? -1 : k;
                    sv[lane * PITCH + cnt] = __dmul_rn(__dmul_rn(__dmul_rn(sum, m.C), a_scale), b_scale);  // :242
                    ++cnt;
                    ndead += dead;
                }
            }
        }
        const bool any_active = __any_sync(SPB_FULL_MASK, active);
        if (__any_sync(SPB_FULL_MASK, cnt == (u32)STAGE) || !any_active) {
            __syncwarp();
#pragma unroll 4
            for (int it = 0; it < 32 / RUNS; ++it) {
                const int l = RUNS * it + (int)(lane / STAGE);
                const u32 t = lane % STAGE;
                const u32 n_l = __shfl_sync(SPB_FULL_MASK, cnt, l);
                const u64 d_l = __shfl_sync(SPB_FULL_MASK, dst, l);
                const i32 i_l = __shfl_sync(SPB_FULL_MASK, irow, l);
                if (t < n_l && m.debug != 1) {
                    const i32 kk = sk[l * PITCH + t];
                    if (m.debug == 2) {
                        c_k[d_l + t] = kk;
                        c_v[d_l + t] = sv[l * PITCH + t];
                        c_i[d_l + t] = kk < 0 ? -1 : i_l;
                    } else {  // streaming stores: C is written once and never re-read here; keep L1/L2 for B
                        __stcs(c_k + d_l + t, kk);
                        __stcs(c_v + d_l + t, sv[l * PITCH + t]);
                        __stcs(c_i + d_l + t, kk < 0 ? -1 : i_l);
                    }
                }
            }
            dst += cnt;
            cnt = 0;
            __syncwarp();
        }
        if (!any_active) break;
    }
    if (ndead) atomicAdd(shrunk, ndead);   // rare
}

template <int NLMAX, int STAGE, bool LOCAL = false>
__global__ void __launch_bounds__(MR_THREADS, (STAGE == 16 ? (LOCAL && MergeBlocks<NLMAX>::value > 5 ? 5 : MergeBlocks<NLMAX>::value) : 1)) k_merge_numeric(MMOperands m, const unsigned char *__restrict__ row_cls,
                                                              const u64 *__restrict__ c_ptr, i32 *c_i, i32 *c_k,
                                                              double *c_v, u32 *shrunk) {
    __shared__ i32 s_k[MR_THREADS * (STAGE + 1)];
    __shared__ double s_v[MR_THREADS * (STAGE + 1)];
    __shared__ BStage<LOCAL ? ML_CAP_NUM : 1, LOCAL ? ML_JCAP : 1> s_b;
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 warp = threadIdx.x >> 5;
    const bool mine = (r < m.nrows) && (row_cls[r] == ROW_MERGE);
    u32 s = 0, len = 0;
    i32 irow = 0;
    u64 dst = 0;
    if (mine) {
        s = m.arow_start[r];
        len = m.arow_start[r + 1] - s;
        irow = m.arow_id[r];
        dst = c_ptr[r];
    }
    BView view;
    bool staged = false;
    if (LOCAL) {   // before any warp leaves: the staging has barriers
        u32 jlo = 0xffffffffu, jhi = 0;
        for (u32 l = 0; l < len; ++l) {
            const u32 j = (u32)__ldg(m.a_j + s + l);
            jlo = min(jlo, j);
            jhi = max(jhi, j);
        }
        staged = stage_b(m, s_b, jlo, jhi, view);
    }
    const u32 maxlen = __reduce_max_sync(SPB_FULL_MASK, len);
    i32 *sk = s_k + warp * 32 * (STAGE + 1);
    double *sv = s_v + warp * 32 * (STAGE + 1);
    if (maxlen == 0) return;
    if (LOCAL && staged) {
        if (maxlen <= 2) merge_rows_warp<2, STAGE, true>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk, &view);
        else if (NLMAX >= 4 && maxlen <= 4) merge_rows_warp<(NLMAX >= 4 ? 4 : 2), STAGE, true>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk, &view);
        else if (NLMAX >= 6 && maxlen <= 6) merge_rows_warp<(NLMAX >= 6 ? 6 : 2), STAGE, true>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk, &view);
        else if (NLMAX >= 8) merge_rows_warp<(NLMAX >= 8 ? 8 : 2), STAGE, true>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk, &view);
        return;
    }
    if (maxlen <= 2) merge_rows_warp<2, STAGE>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk);
    else if (NLMAX >= 4 && maxlen <= 4) merge_rows_warp<(NLMAX >= 4 ? 4 : 2), STAGE>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk);
    else if (NLMAX >= 6 && maxlen <= 6) merge_rows_warp<(NLMAX >= 6 ? 6 : 2), STAGE>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk);
    else if (NLMAX >= 8) merge_rows_warp<(NLMAX >= 8 ? 8 : 2), STAGE>(m, mine, s, len, irow, dst, sk, sv, c_i, c_k, c_v, shrunk);
}

// ---- short rows, ONE pass: merge, then place ---------------------------------------------------------------------------------
// When every row of op(A) is a register-merge row with at most STAGE outputs (banded / stencil matrices: 9 outputs per row), the
// symbolic pass is pure overhead: it runs the same merges as the numeric pass only to learn where the rows go.  Here a warp
// merges its 32 rows ONCE, keeping their outputs in its staging area, learns its place in C from a decoupled look-back over the
// warps (in row order: tiles are handed out by a ticket, so every predecessor is running or done), and writes.  C is allocated
// for STAGE outputs per row; the exact count comes back with the kernel.  A row this kernel cannot take (more than 8 inner
// indices, more than max_products products, more than STAGE outputs) raises *fail: the remaining warps skip their merges (they
// still publish, nobody may wait forever), the host throws the result away and runs the two-pass path.
// out[0] = outputs, out[1] = products, out[2] = rows merged, out[3] = longest row
template <int NL, int STAGE>
__device__ __forceinline__ bool merge_rows_stage(const MMOperands &m, bool mine, u32 s, u32 len, i32 irow, u32 max_products,
                                                 i32 *sk, double *sv, u32 &cnt, u64 &f) {
    constexpr int PITCH = STAGE + 1;
    const u32 lane = lane_id();
    RowMerge<NL> st;
    st.init(m, s, mine ? len : 0);
    f = 0;
#pragma unroll
    for (int l = 0; l < NL; ++l) f += st.end[l] - st.cur[l];
    double a_scale = 1.0;
    if (mine && m.si) a_scale = m.si[irow];
    cnt = 0;
    bool ok = f <= (u64)max_products;
    bool active = mine && ok && f != 0;
    if (st.touch() + a_scale == -1.2345678e300) active = false;  // never true; see RowMerge::touch
    while (__any_sync(SPB_FULL_MASK, active)) {
        if (active) {
            i32 k;
            double sum, b_scale;
            if (!st.next(m, k, sum)) active = false;
            else if (keep_output(m, k, sum, b_scale)) {
                if (cnt == (u32)STAGE) { ok = false; active = false; }
                else {
                    sk[lane * PITCH + cnt] = k;
                    sv[lane * PITCH + cnt] = __dmul_rn(__dmul_rn(__dmul_rn(sum, m.C), a_scale), b_scale);  // :242
                    ++cnt;
                }
            }
        }
    }
    return ok;
}

template <int NLMAX>
__global__ void __launch_bounds__(MR_THREADS, MergeBlocks<NLMAX>::value) k_merge_onepass(MMOperands m, u32 max_products, u64 *state, u32 *ticket,
                                                                                         u32 *fail, ull *out, i32 *c_i, i32 *c_k, double *c_v) {
    constexpr int STAGE = 16, PITCH = STAGE + 1, RUNS = 32 / STAGE;
    __shared__ i32 s_k[MR_THREADS * PITCH];
    __shared__ double s_v[MR_THREADS * PITCH];
    __shared__ u32 s_tile;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const u64 r = (u64)tile * MR_THREADS + threadIdx.x;
    const bool skip = *(volatile u32 *)fail != 0;   // the result is lost already: publish an empty aggregate and leave
    u32 s = 0, len = 0, cnt = 0;
    i32 irow = 0;
    u64 f = 0;
    bool bad = false, mine = false;
    if (r < m.nrows && !skip) {
        s = m.arow_start[r];
        len = m.arow_start[r + 1] - s;
        irow = m.arow_id[r];
        const bool on = !m.si || m.si[irow] != 0.0;  // row excluded by scalei (multiply_sparse.hpp:195)
        bad = on && len > (u32)MERGE_MAX_LISTS;
        mine = on && !bad;
    }
    const u32 rowlen = len;
    if (!mine) len = 0;
    const u32 maxlen = __reduce_max_sync(SPB_FULL_MASK, len);
    i32 *sk = s_k + warp * 32 * PITCH;
    double *sv = s_v + warp * 32 * PITCH;
    bool ok = true;
    if (maxlen == 0) ok = true;
    else if (maxlen <= 2) ok = merge_rows_stage<2, STAGE>(m, mine, s, len, irow, max_products, sk, sv, cnt, f);
    else if (NLMAX >= 4 && maxlen <= 4) ok = merge_rows_stage<(NLMAX >= 4 ? 4 : 2), STAGE>(m, mine, s, len, irow, max_products, sk, sv, cnt, f);
    else if (NLMAX >= 6 && maxlen <= 6) ok = merge_rows_stage<(NLMAX >= 6 ? 6 : 2), STAGE>(m, mine, s, len, irow, max_products, sk, sv, cnt, f);
    else if (NLMAX >= 8) ok = merge_rows_stage<(NLMAX >= 8 ? 8 : 2), STAGE>(m, mine, s, len, irow, max_products, sk, sv, cnt, f);
    else ok = false;   // a row longer than this build covers (the host picks NLMAX from the longest row: cannot happen)
    if (__any_sync(SPB_FULL_MASK, bad || !ok)) {
        if (lane == 0) *fail = 1u;
        cnt = 0;
    }
    // place the warp: exclusive prefix of the warps' output counts, in row order
    const u32 incl = warp_incl_scan(cnt);
    const u32 wtotal = __shfl_sync(SPB_FULL_MASK, incl, 31);
    const u32 wid = tile * (MR_THREADS / 32) + warp;
    const u64 base = lookback_exclusive(state, wid, (u64)wtotal);
    const u64 dst = base + incl - cnt;
    __syncwarp();
#pragma unroll 4
    for (int it = 0; it < 32 / RUNS; ++it) {
        const int l = RUNS * it + (int)(lane / STAGE);
        const u32 t = lane % STAGE;
        const u32 n_l = __shfl_sync(SPB_FULL_MASK, cnt, l);
        const u64 d_l = __shfl_sync(SPB_FULL_MASK, dst, l);
        const i32 i_l = __shfl_sync(SPB_FULL_MASK, irow, l);
        if (t < n_l) {
            __stcs(c_k + d_l + t, sk[l * PITCH + t]);
            __stcs(c_v + d_l + t, sv[l * PITCH + t]);
            __stcs(c_i + d_l + t, i_l);
        }
    }
    // totals: one stripe per warp in turn (see k_merge_count)
    u64 fsum = mine ? f : 0;
    u32 nm = mine && f != 0 && f <= (u64)max_products;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        fsum += __shfl_xor_sync(SPB_FULL_MASK, fsum, o);
        nm += __shfl_xor_sync(SPB_FULL_MASK, nm, o);
    }
    const u32 longest = __reduce_max_sync(SPB_FULL_MASK, rowlen);
    if (lane == 0) {
        ull *mine_s = out + 8 + (size_t)(wid % MC_STRIPES) * 8;
        if (fsum) atomicAdd(&mine_s[0], (ull)fsum);
        if (nm) atomicAdd(&mine_s[1], (ull)nm);
        if (longest > (u32)mine_s[6]) atomicMax(&mine_s[6], (ull)longest);
        if ((u64)tile * MR_THREADS + (u64)(warp + 1) * 32 >= (u64)m.nrows && (u64)tile * MR_THREADS + (u64)warp * 32 < (u64)m.nrows)
            out[0] = base + wtotal;   // the warp that holds the last row: everything before it is placed
    }
}

// ---- longer rows: shared-memory bitmap (symbolic) + shared-memory hash accumulators (numeric) ----------
// Symbolic, one block per row: every product sets the bit of its column in a shared-memory bitmap (order-free,
// so all warps work at once); scanning the bitmap yields the row's DISTINCT OUTPUT COLUMNS ALREADY IN ASCENDING
// ORDER -- no sort.  The count pass stores their number; after the rows are placed, the emit pass repeats the
// bitmap and writes the columns straight into C and cuts the row into work items of <= HASH_CAP outputs.
//
// Numeric, one block per item: the item's columns (sorted, read back from C) are inserted into a shared-memory
// hash table that maps column -> output rank; the accumulators sit in shared memory in rank order.  The A
// entries of the row are staged NT at a time (for an item that covers only part of the row, each B row is
// narrowed to the item's column range by binary search), their products are packed NT per step (prefix sums +
// search), looked up in the table and added.  Order: steps run in ascending (j, k); two products of one step that
// hit the same output (different j, same k) are serialised by a claim word per output (atomicMin of the thread
// number, lowest = smallest j first).  Every output therefore adds its terms in ascending j starting from 0 --
// the reference's order (multiply_sparse.hpp:219-236) -- and the sums are bit-identical to the reference's.
// An output whose sum is exactly 0 is dropped by the reference (:238); here it leaves a tombstone that the host
// closes afterwards (rare: exact cancellation only).
constexpr int HS_THREADS = 1024;            // symbolic (bitmap) kernel
constexpr int HS_WARPS = HS_THREADS / 32;
constexpr u32 HASH_MAX_COLS = 1572864;      // 192 KB of bitmap
constexpr u32 HS_LIST_CAP = HASH_MAX_COLS / 1024 * 3;   // sparse units: at most this many non-zero bitmap words (4608; list of u16)
constexpr int HS_LIST_PER = (HS_LIST_CAP + HS_THREADS - 1) / HS_THREADS;   // consecutive list entries per thread (5)

struct HashArgs {
    const u32 *rows;     // compressed row numbers of the ROW_HASH rows: the small ones (k_hash_symbolic_small) first
    u32 nrows;
    u32 row0;            // bitmap kernel: first row of rows[] it handles (the rows before it went to k_hash_symbolic_small)
    u32 *next;           // work counter (zeroed before every launch)
    u32 wpw;             // bitmap words per warp of the symbolic kernel (multiple of 32; HS_WARPS * wpw * 32 >= columns)
    u32 no_sparse_walk;  // SPB_HASH_SPARSE_WALK=0: every unit walks all its 32-word groups (the round-2 path, for A/B runs)
    u32 cap;             // outputs per numeric work item (HASH_CAP of the numeric kernel that will run)
    u32 n_win;           // column windows per row: the bitmap covers win_cols columns at a time (1 when they all fit)
    u32 win_cols;        // multiple of 32
    u32 *win_cnt;        // [nrows * n_win] outputs of (row, window)
    u32 *row_cnt;        // number of distinct, unmasked output columns of the row (zeroed; windows add up)
    i32 *tmp_k;          // the output columns of the hash rows, one ascending segment per (row, window), segments in no particular order
    ull *tmp_cursor;     // entries of tmp_k handed out
    u64 *seg_off;        // [nrows * n_win] where the segment of (row, window) starts in tmp_k
    u32 *win_pre;        // [nrows * n_win] outputs of the row in earlier windows (k_hash_items)
    const u32 *win_bound; // [nnz_a * (n_win - 1)] or nullptr: win_bound[e * (n_win - 1) + w - 1] = first position of the B row of A
                         // entry e whose column is >= w * win_cols (k_hash_win_bounds); nullptr: searched inside the bitmap kernel
    const u64 *c_ptr;    // emit + numeric
    i32 *c_i, *c_k;
    double *c_v;
    i32 *item_key;       // k_hash_items: first output column of every work item (the lower bound of its column window)
    u64 *items;          // emit: (index into rows[] << 32 | part), appended in any order
    u32 *n_items;
    u64 *row_split;      // emit: per ROW_HASH row cut into W > 1 items, the offset of its (W-1) x (row entries) block in split[]
    ull *split_total;    // emit: entries of split[] handed out
    const u32 *split;    // numeric: split[row_split + (p-1)*len + x] = first position of entry x's B row inside item p's window
    u32 *shrunk;         // numeric: number of outputs dropped (written as tombstones)
    ull *dbg;            // numeric, tracing only: [0] items, [1] staged chunks, [2] steps, [3] barriers between entries, [4] warp-pipelined steps, [5..9] clocks per phase
};

// ---- staged entries ---------------------------------------------------------------------------------------------
// Both kernels take the A entries of a row NT at a time: every thread looks up one entry's B row, entries without
// products are squeezed out, and the products of the chunk are numbered 0..T-1 in (entry, position) order
// (pre[x] = number of the first product of staged entry x, strictly increasing, pre[nE] = T).  Threads then take
// products, not entries -- a 13000-entry hub row and a 1-entry row cost the same per product.
//
// Entry of product p_first + lane, for a warp whose first product is p_first: a two-level 32-ary search by the whole
// warp finds the entry of p_first (from xs, an entry known to start at or before p_first), one more probe per lane
// finds the (at most 32, entries are non-empty) entry boundaries inside the warp's 32 products.
__device__ __forceinline__ u32 staged_entry(const u32 *pre, u32 nE, u32 xs, u32 p_first) {
    const u32 lane = lane_id();
    u32 idx = xs + lane * 32;
    const u32 c1 = __popc(__ballot_sync(SPB_FULL_MASK, idx < nE && pre[idx] <= p_first));
    const u32 blk = xs + (c1 ? c1 - 1 : 0) * 32;
    idx = blk + lane;
    const u32 c2 = __popc(__ballot_sync(SPB_FULL_MASK, idx < nE && pre[idx] <= p_first));
    const u32 x_first = blk + (c2 ? c2 - 1 : 0);
    idx = x_first + 1 + lane;
    const u32 d = (idx <= nE ? pre[idx] : 0xffffffffu) - p_first;
    const u32 bounds = __reduce_or_sync(SPB_FULL_MASK, d < 32 ? 1u << d : 0u);
    return x_first + __popc(bounds & (0xffffffffu >> (31 - lane)));
}

// Squeezes the (bs, len) pairs of the NT threads into st_bs/st_pre (and calls keep(slot) for the survivors);
// returns the number of staged entries and products.  Two barriers.
template <int NT, typename Keep>
__device__ __forceinline__ void stage_entries(u32 bs, u32 len, u32 *st_bs, u32 *st_pre, u32 (*wsum)[NT / 32], u32 &nE, u32 &T, Keep keep) {
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 incl = warp_incl_scan(len);
    const u32 live = __ballot_sync(SPB_FULL_MASK, len != 0);
    if (lane == 31) { wsum[0][warp] = incl; wsum[1][warp] = __popc(live); }
    __syncthreads();
    u32 pre = incl - len, slot = __popc(live & lanemask_lt());
    T = 0; nE = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) {
        const u32 t = wsum[0][w], c = wsum[1][w];
        if ((u32)w < warp) { pre += t; slot += c; }
        T += t;
        nE += c;
    }
    if (len) { st_bs[slot] = bs; st_pre[slot] = pre; keep(slot); }
    if (tid == 0) st_pre[nE] = T;
    __syncthreads();
}

__device__ __forceinline__ u32 hn_lower_bound(const i32 *__restrict__ b_k, u32 lo, u32 hi, i32 key);

// Where every column window begins in the B row of every entry of the ROW_HASH rows: one independent search per (entry,
// window boundary), hundreds of thousands in flight -- inside the bitmap kernel the same searches were two chains of
// dependent L2 round trips in front of every (row, window) unit, 45 % of its time at 2^24 columns (11 windows).
__global__ void __launch_bounds__(128) k_hash_win_bounds(MMOperands m, HashArgs a, u32 *win_bound) {
    const u32 nb = a.n_win - 1;
    for (u32 hrow = a.row0 + blockIdx.x; hrow < a.nrows; hrow += gridDim.x) {   // (the rows before row0 are listed without windows)
        const u32 r = a.rows[hrow];
        const u32 s = m.arow_start[r], len = m.arow_start[r + 1] - s;
        for (u32 t = threadIdx.x; t < len * nb; t += blockDim.x) {
            const u32 x = t / nb, w = t % nb + 1;
            const i32 j = m.a_j[s + x];
            const u64 col = (u64)w * a.win_cols;
            const u32 bs = m.bptr[j], be = m.bptr[(u32)j + 1];
            win_bound[(u64)(s + x) * nb + (w - 1)] = col <= (u64)INT32_MAX ? hn_lower_bound(m.b_k, bs, be, (i32)col) : be;
        }
    }
}

// column of output number t (ascending) of ROW_HASH row hrow: the windows' segments of tmp_k in window order
__device__ __forceinline__ i32 hash_col(const HashArgs &a, u32 hrow, u32 t) {
    const u64 u0 = (u64)hrow * a.n_win;
    if (a.n_win == 1) return a.tmp_k[a.seg_off[u0] + t];
    const u32 *pre = a.win_pre + u0;
    u32 lo = 0, hi = a.n_win;   // last window w with pre[w] <= t (empty windows share their successor's prefix: the last one holds t)
    while (hi - lo > 1) {
        const u32 mid = lo + (hi - lo) / 2;
        if (pre[mid] <= t) lo = mid; else hi = mid;
    }
    return a.tmp_k[a.seg_off[u0 + lo] + (t - pre[lo])];
}

// After the bitmap pass: per ROW_HASH row (one warp each) the prefix of its windows' counts, its work items (<= cap outputs
// each, cut by output rank over the whole row) and its block of split[] (k_hash_splits)
__global__ void __launch_bounds__(256) k_hash_items(MMOperands m, HashArgs a) {
    const u32 lane = lane_id();
    const u32 warps = gridDim.x * (blockDim.x >> 5);
    for (u32 hrow = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); hrow < a.nrows; hrow += warps) {
        const u32 r = a.rows[hrow];
        const u64 u0 = (u64)hrow * a.n_win;
        u32 run = 0;
        for (u32 w0 = 0; w0 < a.n_win; w0 += 32) {
            const u32 w = w0 + lane;
            const u32 c = w < a.n_win ? a.win_cnt[u0 + w] : 0;
            const u32 incl = warp_incl_scan(c);
            if (w < a.n_win) a.win_pre[u0 + w] = run + incl - c;
            run += __shfl_sync(SPB_FULL_MASK, incl, 31);
        }
        const u32 total = run;   // == row_cnt[r]
        const u32 n_items = (total + a.cap - 1) / a.cap;
        u32 item0 = 0;
        if (lane == 0 && n_items) {
            item0 = atomicAdd(a.n_items, n_items);
            if (n_items > 1) a.row_split[hrow] = atomicAdd(a.split_total, (ull)(n_items - 1) * (m.arow_start[r + 1] - m.arow_start[r]));
        }
        item0 = __shfl_sync(SPB_FULL_MASK, item0, 0);
        __syncwarp();   // win_pre of this row is complete (hash_col reads it)
        const u32 per = n_items ? (total + n_items - 1) / n_items : 0;
        for (u32 p = lane; p < n_items; p += 32) {
            a.items[item0 + p] = ((u64)hrow << 32) | p;
            a.item_key[item0 + p] = hash_col(a, hrow, p * per);   // looked up once here, not by every thread of k_hash_splits
        }
    }
}

// ---- symbolic: bitmap --------------------------------------------------------------------------------------------
// Matrices with more columns than the bitmap holds are handled in column windows of win_cols columns: a work unit is
// (row, window); every B row is narrowed to the window by two searches when it is staged.
// ONE pass (round 1 ran the bitmap twice, once to count and once to emit): when a (row, window)'s bitmap is complete its
// set bits are counted, a segment of that many entries is taken from the temporary column list tmp_k (an atomic cursor:
// segments land in no particular order, seg_off remembers where) and the columns are written there in ascending order.
// The rows' output counts (row_cnt) come out of the same pass; the numeric kernel later copies the columns into C.
__global__ void __launch_bounds__(HS_THREADS, 1) k_hash_symbolic(MMOperands m, HashArgs a) {
    constexpr bool EMIT = true;
    extern __shared__ u32 s_bitmap[];  // HS_WARPS * a.wpw words
    __shared__ u32 s_row, s_grab;
    __shared__ u64 s_segbase;
    __shared__ u32 s_wsum[2][HS_WARPS];
    __shared__ u32 s_bs[HS_THREADS], s_pre[HS_THREADS + 1];
    // dense units: set bits per group of 32 bitmap words (then their exclusive prefix) and the list of the non-empty groups;
    // sparse units: the list of the non-zero bitmap WORDS (same storage -- a unit takes one path or the other)
    __shared__ __align__(8) unsigned char s_walk[HASH_MAX_COLS / 1024 * 6];
    u32 *const s_gcnt = reinterpret_cast<u32 *>(s_walk);
    unsigned short *const s_glist = reinterpret_cast<unsigned short *>(s_walk + HASH_MAX_COLS / 1024 * 4);
    unsigned short *const s_list = reinterpret_cast<unsigned short *>(s_walk);
    __shared__ u32 s_summ[HASH_MAX_COLS / 1024];  // one bit per bitmap word: set by the atomicOr that found the word empty
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (u32 w = tid; w < HS_WARPS * a.wpw; w += HS_THREADS) s_bitmap[w] = 0;
    for (u32 w = tid; w < HASH_MAX_COLS / 1024; w += HS_THREADS) s_summ[w] = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_row = atomicAdd(a.next, 1u);
        __syncthreads();
        if (s_row >= (a.nrows - a.row0) * a.n_win) return;
        const u32 hrow = a.row0 + s_row / a.n_win, win = s_row % a.n_win;  // index into rows[], column window
        const u32 col0 = win * a.win_cols;                        // first column of the window
        const u32 r = a.rows[hrow];
        const u32 s = m.arow_start[r], e = m.arow_start[r + 1];
        // ---- products: bits of their columns.  Consecutive lanes hold consecutive products, i.e. (within one B row)
        //      ascending columns, so lanes that hit the same bitmap word form a contiguous run: one ATOMS per run
        //      instead of one per lane (power-law rows pack their columns densely). -------------------------------
        for (u32 c0 = s; c0 < e; c0 += HS_THREADS) {
            const u32 ent = c0 + tid;
            u32 bs = 0, len = 0;
            if (ent < e) {
                const i32 j = m.a_j[ent];
                if (!m.sj_mask || m.sj_mask[j]) {
                    bs = m.bptr[j];
                    u32 be = m.bptr[(u32)j + 1];
                    if (a.n_win > 1 && a.win_bound) {
                        const u32 *wb = a.win_bound + (u64)ent * (a.n_win - 1);
                        if (win > 0) bs = wb[win - 1];
                        if (win + 1 < a.n_win) be = wb[win];
                    } else if (a.n_win > 1 && bs < be) {
                        bs = hn_lower_bound(m.b_k, bs, be, (i32)col0);
                        if ((u64)col0 + a.win_cols <= (u64)INT32_MAX) be = hn_lower_bound(m.b_k, bs, be, (i32)(col0 + a.win_cols));
                    }
                    len = be - bs;
                }
            }
            u32 nE, T;
            if (c0 != s) __syncthreads();  // previous chunk's staging no longer read
            stage_entries<HS_THREADS>(bs, len, s_bs, s_pre, s_wsum, nE, T, [](u32) {});
            u32 xs = 0;
            for (u32 b0 = 0; b0 < T; b0 += 4 * HS_THREADS) {
                u32 k[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const u32 p0 = b0 + u * HS_THREADS;  // first product of this sub-step (block-uniform)
                    k[u] = 0xffffffffu;
                    if (p0 < T) {
                        if (s_pre[xs + 1] <= p0) xs = __shfl_sync(SPB_FULL_MASK, staged_entry(s_pre, nE, xs, p0), 0);
                        const u32 p = p0 + tid;
                        u32 x = xs;
                        if (s_pre[xs + 1] < min(p0 + (u32)HS_THREADS, T)) x = staged_entry(s_pre, nE, xs, p0 + warp * 32);
                        if (p < T) k[u] = (u32)ld_stream_i32(m.b_k + s_bs[x] + (p - s_pre[x]));
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (b0 + u * HS_THREADS >= T) break;  // block-uniform
                    const u32 word = k[u] == 0xffffffffu ? 0x7ffffffu : (k[u] - col0) >> 5;  // lanes past the end: no word
                    const u32 prev = __shfl_up_sync(SPB_FULL_MASK, word, 1);
                    const u32 heads = __ballot_sync(SPB_FULL_MASK, lane == 0 || prev != word);
                    const u32 le = 0xffffffffu >> (31 - lane);               // lanes at or below mine
                    const u32 first = 31 - __clz(heads & le);
                    const u32 above = heads & ~le;
                    const u32 last = above ? (u32)__ffs(above) - 2 : 31u;    // last lane of my run
                    u32 bits = k[u] != 0xffffffffu ? 1u << (k[u] & 31) : 0u;  // col0 is a multiple of 32
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {  // OR of the run, gathered at its first lane
                        const u32 t = __shfl_down_sync(SPB_FULL_MASK, bits, o);
                        if (lane + o <= last) bits |= t;
                    }
                    if (lane == first && bits && atomicOr(&s_bitmap[word], bits) == 0) atomicOr(&s_summ[word >> 5], 1u << (word & 31));
                }
            }
        }
        __syncthreads();
        // ---- outputs = set bits, in ascending column order.  Columns excluded by scalek are cleared first
        //      (multiply_sparse.hpp:208-213).  The bitmap is walked in groups of 32 words dealt round-robin to the warps:
        //      power-law rows pack their columns into one end of the bitmap, a contiguous stretch per warp would leave
        //      one warp with all the work. -------------------------------------------------------------------------------
        const u32 ngroups = HS_WARPS * a.wpw / 32;
        // ---- how many bitmap words hold anything (summary bits; a thread owns summary words 2t and 2t+1, which it clears) ----
        u32 n_nz, nz_before;
        u32 sw0 = 0, sw1 = 0;
        {
            if (2 * tid < ngroups) { sw0 = s_summ[2 * tid]; s_summ[2 * tid] = 0; }
            if (2 * tid + 1 < ngroups) { sw1 = s_summ[2 * tid + 1]; s_summ[2 * tid + 1] = 0; }
            const u32 c = __popc(sw0) + __popc(sw1);
            const u32 incl = warp_incl_scan(c);
            if (lane == 31) s_wsum[0][warp] = incl;
            __syncthreads();
            nz_before = incl - c;
            n_nz = 0;
#pragma unroll
            for (int w = 0; w < HS_WARPS; ++w) {
                const u32 t = s_wsum[0][w];
                if ((u32)w < warp) nz_before += t;
                n_nz += t;
            }
        }
        if (EMIT && n_nz <= HS_LIST_CAP && !a.no_sparse_walk) {
            // ---- sparse unit (a few thousand outputs in tens of thousands of words -- most units of a wide matrix): only the
            //      non-zero words are visited.  Their ordered list; then every thread takes HS_LIST_PER consecutive words of it,
            //      counts, and writes its columns behind those of the threads before it.  Walking all the 32-word groups cost
            //      the same ~45 instructions per group whether a group held one column or a thousand. ------------------------
            {
                u32 pos = nz_before;
                for (u32 t = sw0; t; t &= t - 1) s_list[pos++] = (unsigned short)(2 * tid * 32 + __ffs(t) - 1);
                for (u32 t = sw1; t; t &= t - 1) s_list[pos++] = (unsigned short)((2 * tid + 1) * 32 + __ffs(t) - 1);
            }
            __syncthreads();   // list complete; s_wsum read by everyone
            const u32 per = (n_nz + HS_THREADS - 1) / HS_THREADS;   // <= HS_LIST_PER
            const u32 l0 = tid * per;
            u32 wbits[HS_LIST_PER];
            u32 cnt = 0;
#pragma unroll
            for (int u = 0; u < HS_LIST_PER; ++u) {
                wbits[u] = 0;
                if ((u32)u < per && l0 + u < n_nz) {
                    const u32 w = s_list[l0 + u];
                    u32 bits = s_bitmap[w];
                    s_bitmap[w] = 0;
                    if (m.sk) {
                        for (u32 t = bits; t; t &= t - 1) {
                            const u32 b = __ffs(t) - 1;
                            if (m.sk[col0 + w * 32 + b] == 0.0) bits &= ~(1u << b);
                        }
                    }
                    wbits[u] = bits;
                    cnt += __popc(bits);
                }
            }
            const u32 incl = warp_incl_scan(cnt);
            if (lane == 31) s_wsum[1][warp] = incl;
            __syncthreads();
            u32 before = incl - cnt, total = 0;
#pragma unroll
            for (int w = 0; w < HS_WARPS; ++w) {
                const u32 t = s_wsum[1][w];
                if ((u32)w < warp) before += t;
                total += t;
            }
            if (tid == 0) {
                const u64 unit = (u64)hrow * a.n_win + win;
                s_segbase = total ? atomicAdd(a.tmp_cursor, (ull)total) : 0ull;
                a.seg_off[unit] = s_segbase;
                a.win_cnt[unit] = total;
                if (total) atomicAdd(&a.row_cnt[r], total);
            }
            __syncthreads();
            u64 pos = s_segbase + before;
#pragma unroll
            for (int u = 0; u < HS_LIST_PER; ++u) {
                if (!wbits[u]) continue;
                const u32 c0w = col0 + (u32)s_list[l0 + u] * 32;   // (the list stays put until the next unit)
                for (u32 t = wbits[u]; t; t &= t - 1, ++pos) a.tmp_k[pos] = (i32)(c0w + __ffs(t) - 1);
            }
            continue;
        }
        u32 mine = 0;
        for (u32 g = warp; g < ngroups; g += HS_WARPS) {
            const u32 w = g * 32 + lane;
            u32 bits = s_bitmap[w];
            if (m.sk && bits) {
                u32 live = bits;
                for (u32 t = bits; t; t &= t - 1) {
                    const u32 b = __ffs(t) - 1;
                    if (m.sk[col0 + w * 32 + b] == 0.0) live &= ~(1u << b);
                }
                if (EMIT && live != bits) s_bitmap[w] = live;
                bits = live;
            }
            if (!EMIT) s_bitmap[w] = 0;
            const u32 c = __popc(bits);
            if (EMIT) {
                const u32 gc = __reduce_add_sync(SPB_FULL_MASK, c);
                if (lane == 0) s_gcnt[g] = gc;
            } else {
                mine += c;
            }
        }
        if (!EMIT) {
            mine = __reduce_add_sync(SPB_FULL_MASK, mine);
            if (lane == 0) s_wsum[0][warp] = mine;
            __syncthreads();
            if (tid == 0) {
                u32 total = 0;
                for (int w = 0; w < HS_WARPS; ++w) total += s_wsum[0][w];
                if (a.n_win > 1) { a.win_cnt[(u64)hrow * a.n_win + win] = total; atomicAdd(&a.row_cnt[r], total); }
                else a.row_cnt[r] = total;
            }
            continue;
        }
        __syncthreads();
        // exclusive prefix of the group counts, and the list of the non-empty groups (two groups per thread)
        u32 total, n_live;
        {
            const u32 g0 = 2 * tid, g1 = 2 * tid + 1;
            const u32 v0 = g0 < ngroups ? s_gcnt[g0] : 0, v1 = g1 < ngroups ? s_gcnt[g1] : 0;
            const u32 l0 = v0 != 0, l1 = v1 != 0;
            const u32 incl = warp_incl_scan(v0 + v1), lincl = warp_incl_scan(l0 + l1);
            if (lane == 31) { s_wsum[0][warp] = incl; s_wsum[1][warp] = lincl; }
            __syncthreads();
            u32 before = incl - (v0 + v1), lbefore = lincl - (l0 + l1);
            total = 0; n_live = 0;
#pragma unroll
            for (int w = 0; w < HS_WARPS; ++w) {
                const u32 t = s_wsum[0][w], c = s_wsum[1][w];
                if ((u32)w < warp) { before += t; lbefore += c; }
                total += t;
                n_live += c;
            }
            if (g0 < ngroups) s_gcnt[g0] = before;
            if (g1 < ngroups) s_gcnt[g1] = before + v0;
            if (l0) s_glist[lbefore] = (unsigned short)g0;
            if (l1) s_glist[lbefore + l0] = (unsigned short)g1;
        }
        if (tid == 0) {
            const u64 unit = (u64)hrow * a.n_win + win;
            s_segbase = total ? atomicAdd(a.tmp_cursor, (ull)total) : 0ull;
            a.seg_off[unit] = s_segbase;
            a.win_cnt[unit] = total;
            if (total) atomicAdd(&a.row_cnt[r], total);
            s_grab = 0;
        }
        __syncthreads();
        // ---- ... and the columns are written, one non-empty group per warp at a time (grabbed from a counter: the
        //      groups of a power-law row differ in weight by orders of magnitude): the lanes hold 32 consecutive
        //      words, so their outputs are consecutive in C ------------------------------------------------------------
        const u64 base = s_segbase;
        // sparse units (a couple of outputs per group): the groups are dealt to the warps in turn, no counter; dense ones
        // (hub rows: groups of up to 1024 outputs next to groups of one) are grabbed one at a time
        const bool dealt = total <= 4 * n_live;
        for (u32 turn = warp;; turn += HS_WARPS) {
            u32 i = turn;
            if (!dealt) {
                if (lane == 0) i = atomicAdd(&s_grab, 1u);
                i = __shfl_sync(SPB_FULL_MASK, i, 0);
            }
            if (i >= n_live) break;
            const u32 g = s_glist[i];
            const u32 w = g * 32 + lane;
            u32 bits = s_bitmap[w];
            s_bitmap[w] = 0;
            const u32 c = __popc(bits);
            const u32 incl = warp_incl_scan(c);
            u64 pos = base + s_gcnt[g] + incl - c;
            for (; bits; bits &= bits - 1, ++pos) a.tmp_k[pos] = (i32)(col0 + w * 32 + __ffs(bits) - 1);
        }
    }
}

// ---- symbolic for rows of a few thousand products: sort their columns in shared memory ---------------------------------------
// The bitmap costs the same ~20 us per (row, column window) whether the row has 600 products or 60 000, and a matrix of 2^24
// columns has 11 windows per row: half of config 4's long rows have fewer than 8192 products and cost half of the bitmap
// pass for 5 % of the products.  Here a 256-thread block gathers ALL product columns of such a row into shared memory (one warp
// per B row, coalesced), sorts them (bitonic network, padded to a power of two), drops repeats and columns masked by scalek and
// writes the list -- one segment per row, filed under its first window, so that everything downstream (k_hash_items, the
// numeric kernel) reads it like any other row's.  Independent of the matrix width; six blocks per SM.
constexpr int HSM_THREADS = 256;
constexpr u32 HSM_CAP = 8192;
__global__ void __launch_bounds__(HSM_THREADS) k_hash_symbolic_small(MMOperands m, HashArgs a, u32 n_small) {
    __shared__ u32 s_key[HSM_CAP];
    __shared__ u32 s_bs[HSM_THREADS], s_pre[HSM_THREADS + 1];
    __shared__ u32 s_wsum[2][HSM_THREADS / 32];
    __shared__ u32 s_cnt[HSM_THREADS / 32];
    __shared__ u64 s_base;
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (u32 hrow = blockIdx.x; hrow < n_small; hrow += gridDim.x) {
        const u32 r = a.rows[hrow];
        const u32 s = m.arow_start[r], e = m.arow_start[r + 1];
        // ---- all product columns of the row, entry after entry ---------------------------------------------------------
        u32 T = 0;
        for (u32 c0 = s; c0 < e; c0 += HSM_THREADS) {
            const u32 ent = c0 + tid;
            u32 bs = 0, len = 0;
            if (ent < e) {
                const i32 j = m.a_j[ent];
                if (!m.sj_mask || m.sj_mask[j]) { bs = m.bptr[j]; len = m.bptr[(u32)j + 1] - bs; }
            }
            u32 nE, Tc;
            __syncthreads();   // the previous chunk's staging (and the previous row's keys) are no longer read
            stage_entries<HSM_THREADS>(bs, len, s_bs, s_pre, s_wsum, nE, Tc, [](u32) {});
            for (u32 x = warp; x < nE; x += HSM_THREADS / 32) {
                const u32 b0 = s_bs[x], p0 = T + s_pre[x], ln = s_pre[x + 1] - s_pre[x];
                for (u32 t = lane; t < ln; t += 32)
                    if (p0 + t < HSM_CAP) s_key[p0 + t] = (u32)ld_stream_i32(m.b_k + b0 + t);   // (the host only sends rows that fit)
            }
            T += Tc;
        }
        if (T > HSM_CAP) T = HSM_CAP;
        u32 P = 64;
        while (P < T) P <<= 1;
        __syncthreads();
        for (u32 t = T + tid; t < P; t += HSM_THREADS) s_key[t] = 0xffffffffu;
        __syncthreads();
        // ---- bitonic sort of s_key[0..P) ---------------------------------------------------------------------------------
        for (u32 k = 2; k <= P; k <<= 1)
            for (u32 j = k >> 1; j > 0; j >>= 1) {
                for (u32 p = tid; p < P / 2; p += HSM_THREADS) {
                    const u32 lo = ((p & ~(j - 1)) << 1) | (p & (j - 1)), hi = lo + j;
                    const u32 x = s_key[lo], y = s_key[hi];
                    if ((x > y) == ((lo & k) == 0)) { s_key[lo] = y; s_key[hi] = x; }
                }
                __syncthreads();
            }
        // ---- distinct, unmasked columns: every thread a contiguous stretch --------------------------------------------
        const u32 per = P / HSM_THREADS > 0 ? P / HSM_THREADS : 1;   // P >= 64: threads beyond P / per have nothing
        const u32 i0 = tid * per, i1 = min(P, i0 + per);
        u32 mine = 0;
        for (u32 i = i0; i < i1 && i0 < P; ++i) {
            const u32 c = s_key[i];
            if (c != 0xffffffffu && (i == 0 || s_key[i - 1] != c) && (!m.sk || m.sk[c] != 0.0)) ++mine;
        }
        const u32 incl = warp_incl_scan(mine);
        if (lane == 31) s_cnt[warp] = incl;
        __syncthreads();
        u32 before = incl - mine, total = 0;
#pragma unroll
        for (int w = 0; w < HSM_THREADS / 32; ++w) {
            if ((u32)w < warp) before += s_cnt[w];
            total += s_cnt[w];
        }
        if (tid == 0) {
            const u64 unit = (u64)hrow * a.n_win;
            s_base = total ? atomicAdd(a.tmp_cursor, (ull)total) : 0ull;
            a.seg_off[unit] = s_base;
            a.win_cnt[unit] = total;     // the other windows of the row stay 0 (zeroed by the host)
            a.row_cnt[r] = total;
        }
        __syncthreads();
        u64 pos = s_base + before;
        for (u32 i = i0; i < i1 && i0 < P; ++i) {
            const u32 c = s_key[i];
            if (c != 0xffffffffu && (i == 0 || s_key[i - 1] != c) && (!m.sk || m.sk[c] != 0.0)) a.tmp_k[pos++] = (i32)c;
        }
    }
}

// ---- numeric: hash accumulators ------------------------------------------------------------------------------------
// first position in [lo, hi) of the sorted run b_k whose column is >= key.  Four-way: three probes in flight per
// level halve the chain of dependent L2 round trips of a binary search (the staging of windowed items is
// latency-bound on exactly this chain).
__device__ __forceinline__ u32 hn_lower_bound(const i32 *__restrict__ b_k, u32 lo, u32 hi, i32 key) {
    while (hi - lo > 3) {
        const u32 q = (hi - lo) / 4;
        const u32 m1 = lo + q, m2 = lo + 2 * q, m3 = lo + 3 * q;
        const i32 v1 = __ldg(b_k + m1), v2 = __ldg(b_k + m2), v3 = __ldg(b_k + m3);
        if (v1 >= key) hi = m1;
        else if (v2 >= key) { lo = m1 + 1; hi = m2; }
        else if (v3 >= key) { lo = m2 + 1; hi = m3; }
        else lo = m3 + 1;
    }
    while (lo < hi && __ldg(b_k + lo) < key) ++lo;
    return lo;
}

// Column windows.  A row with more outputs than one item holds is cut into W items by output rank; item p covers
// the columns from its first output to just before item p+1's first output.  For every entry x of the row, the
// position in its B row where item p's window begins is found HERE, by one independent thread per (item, entry)
// -- millions of searches in flight -- instead of inside the numeric kernel, where the same searches were a chain
// of dependent L2 round trips in front of every item (29 % of its time).
__global__ void __launch_bounds__(256) k_hash_splits(MMOperands m, HashArgs a, u32 total_items, u32 *split) {
    for (u32 item = blockIdx.x; item < total_items; item += gridDim.x) {
        const u64 it = a.items[item];
        const u32 sr = (u32)(it >> 32), part = (u32)it;
        if (part == 0) continue;
        const u32 r = a.rows[sr];
        const u32 s = m.arow_start[r], len = m.arow_start[r + 1] - s;
        const u64 base = a.c_ptr[r];
        const u32 total = (u32)(a.c_ptr[r + 1] - base);
        const u32 n_items = (total + a.cap - 1) / a.cap;
        const u32 per = (total + n_items - 1) / n_items;
        const i32 key = a.item_key[item];
        u32 *dst = split + a.row_split[sr] + (u64)(part - 1) * len;
        for (u32 x = threadIdx.x; x < len; x += blockDim.x) {
            const i32 j = m.a_j[s + x];
            dst[x] = hn_lower_bound(m.b_k, m.bptr[j], m.bptr[(u32)j + 1], key);
        }
    }
}

template <int NT, int CAP, int SLOTS>
struct HashSmem {
    u32 keys[SLOTS];
    double acc[CAP];
    double st_as[NT];
    u32 st_bs[NT];
    u32 st_pre[NT + 1];
    unsigned short rank[SLOTS];
    u32 wsum[2][NT / 32];
};

// one step's products, fetched ahead of their use
struct HashStep {
    u32 k;        // column (valid lanes)
    double b;     // B value
    double as;    // scaled A value of the product's entry
    u32 x;        // staged entry of the product
    u32 x_first, x_last;  // staged entries of the step's first and last product (block-uniform)
    bool valid;
};

template <int NT, int CAP, int SLOTS>
__global__ void __launch_bounds__(NT, 1024 / NT) k_hash_numeric(MMOperands m, HashArgs a, u32 total_items) {
    extern __shared__ __align__(16) unsigned char hn_raw[];
    typedef HashSmem<NT, CAP, SLOTS> Smem;
    Smem &sm = *reinterpret_cast<Smem *>(hn_raw);
    constexpr u32 EMPTY = 0xffffffffu;
    constexpr u32 NO_ENTRY = 0xffffffffu;
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    u32 dropped = 0;
    ull n_chunks = 0, n_steps = 0, n_rounds = 0, n_done = 0, n_piped = 0;
    long long c_setup = 0, c_stage = 0, c_steps = 0, c_piped = 0, c_out = 0, t0 = 0, t1;  // tracing: clocks per phase
#define HN_TICK(acc) do { if (a.dbg) { t1 = clock64(); acc += t1 - t0; t0 = t1; } } while (0)
    // items are dealt round-robin: ~10^3 items per block average their very different sizes out, and no block ever
    // waits for a work counter
    for (u32 item = blockIdx.x; item < total_items; item += gridDim.x) {
        __syncthreads();
        if (a.dbg) t0 = clock64();
        ++n_done;
        const u64 it = a.items[item];
        const u32 sr = (u32)(it >> 32), part = (u32)it;
        const u32 r = a.rows[sr];
        const u32 s = m.arow_start[r], e = m.arow_start[r + 1];
        const u64 base = a.c_ptr[r];
        const u32 total = (u32)(a.c_ptr[r + 1] - base);
        const u32 n_items = (total + a.cap - 1) / a.cap;  // a.cap <= CAP (smaller only in tests)
        const u32 per = (total + n_items - 1) / n_items;
        const u32 o_lo = part * per, o_hi = min(o_lo + per, total);
        const u32 n_out = o_hi - o_lo;   // >= 1
        const bool windowed = n_items > 1;
        // table size: power of two >= 2 * n_out, at most SLOTS (load factor <= CAP / SLOTS)
        u32 slots = 64;
        while (slots < 2 * n_out && slots < (u32)SLOTS) slots <<= 1;
        const u32 mask = slots - 1;
        const int hshift = 32 - (31 - __clz(slots));
        // the item's columns (sorted; written by the emit pass): loads first, the table is cleared under them
        constexpr int KPT = (CAP + NT - 1) / NT;
        u32 mykey[KPT];
#pragma unroll
        for (int u = 0; u < KPT; ++u) {
            const u32 t = tid + u * NT;
            mykey[u] = t < n_out ? (u32)hash_col(a, sr, o_lo + t) : EMPTY;
        }
        // windows of the B rows (k_hash_splits): where this item starts / the next one starts
        const u32 *split_lo = nullptr, *split_hi = nullptr;
        if (windowed) {
            const u32 *rs = a.split + a.row_split[sr];
            if (part > 0) split_lo = rs + (u64)(part - 1) * (e - s);
            if (part + 1 < n_items) split_hi = rs + (u64)part * (e - s);
        }
        for (u32 t = tid; t < slots; t += NT) sm.keys[t] = EMPTY;
        for (u32 t = tid; t < n_out; t += NT) sm.acc[t] = 0.0;  // sum starts at 0 (:219)
        __syncthreads();
#pragma unroll
        for (int u = 0; u < KPT; ++u) {
            const u32 t = tid + u * NT;
            if (t < n_out) {
                u32 h = (mykey[u] * 0x9E3779B1u) >> hshift;
                while (atomicCAS(&sm.keys[h], EMPTY, mykey[u]) != EMPTY) h = (h + 1) & mask;
                sm.rank[h] = (unsigned short)t;
            }
        }
        for (u32 c0 = s; c0 < e; c0 += NT) {
            __syncthreads();  // table built / previous chunk's adds done, its staging no longer read
            if (c0 == s) HN_TICK(c_setup);
            ++n_chunks;
            // ---- stage NT entries of the row: scaled value, start and length of (the item's window of) the B row ----
            const u32 ent = c0 + tid;
            u32 bs = 0, len = 0;
            double as = 0.0;
            if (ent < e) {
                const i32 j = m.a_j[ent];
                u32 w_lo = 0, w_hi = 0;
                if (split_lo) w_lo = split_lo[ent - s];
                if (split_hi) w_hi = split_hi[ent - s];
                if (!m.sj_mask || m.sj_mask[j]) {
                    bs = split_lo ? w_lo : m.bptr[j];
                    const u32 be = split_hi ? w_hi : m.bptr[(u32)j + 1];
                    len = be - bs;
                    as = m.a_val[ent];
                    if (m.sj) as = __dmul_rn(as, m.sj[j]);  // (a*s) first, :228
                }
            }
            u32 nE, T;
            stage_entries<NT>(bs, len, sm.st_bs, sm.st_pre, sm.wsum, nE, T, [&](u32 slot) { sm.st_as[slot] = as; });
            HN_TICK(c_stage);
            // ---- the chunk's T products, NT per step, in (entry, position) order; the loads of step i+1 are issued
            //      before step i is applied.  xs = entry of the next fetch's first product (block-uniform). ------------
            u32 xs = 0;
            auto fetch = [&](u32 b0, HashStep &st) {
                const u32 end = min(b0 + (u32)NT, T);
                if (sm.st_pre[xs + 1] <= b0) xs = __shfl_sync(SPB_FULL_MASK, staged_entry(sm.st_pre, nE, xs, b0), 0);
                st.x_first = st.x_last = st.x = xs;
                const u32 p = b0 + tid;
                st.valid = p < end;
                if (sm.st_pre[xs + 1] < end) {  // more than one entry in the step
                    st.x_last = __shfl_sync(SPB_FULL_MASK, staged_entry(sm.st_pre, nE, xs, end - 1), 0);
                    st.x = staged_entry(sm.st_pre, nE, xs, b0 + warp * 32);
                }
                if (st.valid) {
                    const u32 q = sm.st_bs[st.x] + (p - sm.st_pre[st.x]);
                    st.k = (u32)ld_stream_i32(m.b_k + q);
                    st.b = ld_stream_f64(m.b_val + q);
                    st.as = sm.st_as[st.x];
                }
            };
            HashStep cur, nxt;
            nxt.valid = false; nxt.x = nxt.x_first = nxt.x_last = 0; nxt.k = 0; nxt.b = 0.0; nxt.as = 0.0;
            if (T) fetch(0, nxt);
            u32 last_x = NO_ENTRY;  // entry whose products were added last (block-uniform)
            for (u32 b0 = 0; b0 < T; b0 += NT) {
                cur = nxt;
                if (b0 + NT < T) fetch(b0 + NT, nxt);
                ++n_steps;
                bool pending = cur.valid;
                u32 rk = 0;
                double v = 0.0;
                if (pending) {
                    v = __dmul_rn(cur.as, cur.b);
                    u32 h = (cur.k * 0x9E3779B1u) >> hshift;
                    for (;;) {
                        const u32 kk = sm.keys[h];
                        if (kk == cur.k) break;
                        if (kk == EMPTY) { pending = false; break; }  // column excluded by scalek: not an output
                        h = (h + 1) & mask;
                    }
                    rk = sm.rank[h];
                }
                // Order.  The products of ONE entry have distinct columns: its threads add at once.  Two entries may
                // share an output, and the one with the smaller j must add first (reference order, :219-236):
                if (cur.x_last - cur.x_first < 32) {
                    // a few entries in the step: one after the other, a barrier wherever the entry changes
                    for (u32 xi = cur.x_first; xi <= cur.x_last; ++xi) {
                        if (last_x != xi) { __syncthreads(); ++n_rounds; }
                        last_x = xi;
                        if (pending && cur.x == xi) sm.acc[rk] = __dadd_rn(sm.acc[rk], v);
                    }
                    HN_TICK(c_steps);
                } else {
                    // many short entries: one warp after the other (ascending j across warps); inside a warp the
                    // lanes that share an output add in lane order (ascending j again)
                    ++n_piped;
                    u32 peers = 0, myrank = 0;
                    const u32 pend = __ballot_sync(SPB_FULL_MASK, pending);
                    if (pending) {
                        peers = __match_any_sync(pend, rk);
                        myrank = __popc(peers & lanemask_lt());
                    }
                    const u32 rounds = __reduce_max_sync(SPB_FULL_MASK, (u32)__popc(peers));
                    for (u32 w = 0; w < (u32)(NT / 32); ++w) {
                        __syncthreads();
                        if (warp == w) {
                            for (u32 i = 0; i < rounds; ++i) {
                                if (pending && myrank == i) sm.acc[rk] = __dadd_rn(sm.acc[rk], v);
                                __syncwarp();
                            }
                        }
                    }
                    last_x = NO_ENTRY;
                    HN_TICK(c_piped);
                }
            }
        }
        __syncthreads();
        // ---- outputs, in rank (= ascending column) order ---------------------------------------------------------------
        const i32 irow = m.arow_id[r];
        double a_scale = 1.0;
        if (m.si) a_scale = m.si[irow];
#pragma unroll
        for (int u = 0; u < KPT; ++u) {
            const u32 t = tid + u * NT;
            if (t >= n_out) break;
            const double sum = sm.acc[t];
            double b_scale = 1.0;
            if (m.sk) b_scale = m.sk[mykey[u]];
            __stcs(a.c_v + base + o_lo + t, __dmul_rn(__dmul_rn(__dmul_rn(sum, m.C), a_scale), b_scale));  // :242
            __stcs(a.c_k + base + o_lo + t, (i32)mykey[u]);
            const bool dead = !(sum != 0.0);  // :238 (NaN != 0 is kept).  Tombstone: the host closes the gaps afterwards
            __stcs(a.c_i + base + o_lo + t, dead ? -1 : irow);
            dropped += dead;
        }
        HN_TICK(c_out);
    }
#undef HN_TICK
    if (dropped) atomicAdd(a.shrunk, dropped);
    if (a.dbg && tid == 0) {
        atomicAdd(a.dbg + 0, n_done); atomicAdd(a.dbg + 1, n_chunks); atomicAdd(a.dbg + 2, n_steps); atomicAdd(a.dbg + 3, n_rounds);
        atomicAdd(a.dbg + 4, n_piped);
        atomicAdd(a.dbg + 5, (ull)c_setup); atomicAdd(a.dbg + 6, (ull)c_stage); atomicAdd(a.dbg + 7, (ull)c_steps);
        atomicAdd(a.dbg + 8, (ull)c_piped); atomicAdd(a.dbg + 9, (ull)c_out);
    }
}

// Rare: outputs of hash-accumulator rows that summed to exact zero were written as
// tombstones (row index -1).  keep[t] = 1 for live entries; after a scan of keep[], k_compact_entries moves them.
__global__ void k_live_flags(const i32 *__restrict__ c_i, u64 n, unsigned char *keep) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) keep[t] = c_i[t] >= 0;
}
__global__ void k_compact_entries(u64 n, const unsigned char *__restrict__ keep, const u64 *__restrict__ slot,
                                  const i32 *__restrict__ i_old, const i32 *__restrict__ k_old, const double *__restrict__ v_old,
                                  i32 *i_new, i32 *k_new, double *v_new) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        if (keep[t]) {
            const u64 d = slot[t];
            i_new[d] = i_old[t];
            k_new[d] = k_old[t];
            v_new[d] = v_old[t];
        }
    }
}

// ---- long rows: expand-sort-compress ------------------------------------------------------------
// chunk boundaries: rb[c] = first row whose ESC product offset >= c*chunk; pb[c] = that offset
__global__ void k_esc_chunks(const u64 *__restrict__ esc_off, u32 nrows, u64 chunk, u32 nchunks, u32 *rb, u64 *pb) {
    u32 c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > nchunks) return;
    u32 lo = 0, hi = nrows;
    if (c == nchunks) lo = nrows;
    else {
        u64 want = (u64)c * chunk;
        while (lo < hi) {
            u32 mid = lo + (hi - lo) / 2;
            if (esc_off[mid] < want) lo = mid + 1; else hi = mid;
        }
    }
    rb[c] = lo;
    pb[c] = esc_off[lo];
}

// product p of the chunk -> (key = (row number << kbits) | k, value (a*s)*b), in (row, j, k) order
__global__ void k_esc_expand(MMOperands m, const u64 *__restrict__ esc_off, const u64 *__restrict__ ent_off,
                             u32 row_lo, u32 row_hi, u64 p_lo, u64 count, int kbits, u64 *keys, double *vals) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (u64)gridDim.x * blockDim.x) {
        const u64 p = p_lo + t;
        // row: last r in [row_lo,row_hi) with esc_off[r] <= p
        u32 lo = row_lo, hi = row_hi;
        while (hi - lo > 1) {
            u32 mid = lo + (hi - lo) / 2;
            if (esc_off[mid] <= p) lo = mid; else hi = mid;
        }
        const u32 r = lo;
        const u32 s = m.arow_start[r], e_end = m.arow_start[r + 1];
        const u64 want = ent_off[s] + (p - esc_off[r]);
        u32 el = s, eh = e_end;  // last entry e with ent_off[e] <= want
        while (eh - el > 1) {
            u32 mid = el + (eh - el) / 2;
            if (ent_off[mid] <= want) el = mid; else eh = mid;
        }
        const u32 e = el;
        const i32 j = m.a_j[e];
        const u32 b = m.bptr[j] + (u32)(want - ent_off[e]);
        double as = m.a_val[e];
        if (m.sj) as = __dmul_rn(as, m.sj[j]);
        keys[t] = ((u64)(r - row_lo) << kbits) | (u64)(u32)m.b_k[b];
        vals[t] = __dmul_rn(as, m.b_val[b]);
    }
}

// compressed rows of the chunk's output: first[row] = first entry, cnt[row] = entries
__global__ void k_esc_row_spans(const i32 *__restrict__ t_row, u32 n, u32 *first, u32 *cnt) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        i32 r = t_row[t];
        if (t == 0 || t_row[t - 1] != r) first[r] = (u32)t;
    }
}
__global__ void k_esc_row_counts(const i32 *__restrict__ t_row, u32 n, const u32 *__restrict__ first, u32 *cnt) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        i32 r = t_row[t];
        if (t + 1 == n || t_row[t + 1] != r) cnt[r] = (u32)t + 1 - first[r];
    }
}
__global__ void k_esc_copy(const i32 *__restrict__ t_row, const i32 *__restrict__ t_k, const double *__restrict__ t_v,
                           u32 n, const u32 *__restrict__ first, const u64 *__restrict__ c_ptr,
                           const i32 *__restrict__ arow_id, i32 *c_i, i32 *c_k, double *c_v) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        i32 r = t_row[t];
        u64 dst = c_ptr[r] + ((u32)t - first[r]);
        c_i[dst] = arow_id[r];
        c_k[dst] = t_k[t];
        c_v[dst] = t_v[t];
    }
}

// ---- matrix * vector  (multiply_sparse.hpp:281-365): one thread per row, ascending j -----------
__global__ void k_mv_rows(MMOperands m, const double *__restrict__ v_dense, const unsigned char *__restrict__ v_mask,
                          double *row_val, unsigned char *row_keep) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < m.nrows; r += (u64)gridDim.x * blockDim.x) {
        const i32 irow = m.arow_id[r];
        double a_scale = 1.0;
        bool use = true;
        if (m.si) { a_scale = m.si[irow]; use = (a_scale != 0.0); }
        double sum = 0.0;
        if (use) {
            for (u32 e = m.arow_start[r]; e < m.arow_start[r + 1]; ++e) {
                i32 j = m.a_j[e];
                if (!v_mask[j]) continue;
                if (m.sj_mask && !m.sj_mask[j]) continue;
                double as = m.a_val[e];
                if (m.sj) as = __dmul_rn(as, m.sj[j]);
                sum = __dadd_rn(sum, __dmul_rn(as, v_dense[j]));
            }
        }
        bool keep = use && (sum != 0.0);
        row_keep[r] = keep ? 1 : 0;
        row_val[r] = __dmul_rn(__dmul_rn(sum, m.C), a_scale);
    }
}
__global__ void k_mv_emit(u32 nrows, const i32 *__restrict__ arow_id, const double *__restrict__ row_val,
                          const unsigned char *__restrict__ row_keep, const u32 *__restrict__ slot, i32 *out_i,
                          double *out_v) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (u64)gridDim.x * blockDim.x)
        if (row_keep[r]) { out_i[slot[r]] = arow_id[r]; out_v[slot[r]] = row_val[r]; }
}
