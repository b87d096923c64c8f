// csr.cuh -- row structure of a sorted COO array.
//
// k_row_heads replaces spsparse::dim_beginnings (reference slib/spsparse/algorithm.hpp:74-118): the
// compressed list of offsets where the leading sorted index changes (non-empty rows only).  The
// dense row pointer over the inner index of B (needed for row-wise SpGEMM, no reference
// counterpart -- the reference walks columns with DimBeginningsXiter instead) is built from it by
// scattering row lengths and scanning them.
#pragma once
#include "scan.cuh"

constexpr int RH_THREADS = 256;
constexpr int RH_IPT = 8;
constexpr int RH_TILE = RH_THREADS * RH_IPT;
constexpr int RH_WARPS = RH_THREADS / 32;

// Positions i where hi[i] != hi[i-1] (and i == 0), compacted in order; row_id gets hi[i].
// count[0] = number of heads.  Caller appends the sentinel.
__global__ void __launch_bounds__(RH_THREADS) k_row_heads(const i32 *__restrict__ hi, u32 n,
                                                          u32 *row_start, i32 *row_id, u32 *count,
                                                          u64 *state, u32 *ticket) {
    __shared__ u32 s_part[RH_IPT * RH_WARPS];
    __shared__ u32 s_tile;
    __shared__ u64 s_excl;
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u64 base = (u64)tile * RH_TILE;
    if (base >= n) return;
    const u32 lt = lanemask_lt();
    u32 head_bits = 0, rank[RH_IPT];
    i32 mine[RH_IPT];
#pragma unroll
    for (int k = 0; k < RH_IPT; ++k) {
        u64 i = base + (u64)k * RH_THREADS + tid;
        bool head = false;
        mine[k] = 0;
        if (i < n) {
            mine[k] = hi[i];
            head = (i == 0) || (hi[i - 1] != mine[k]);
        }
        u32 b = __ballot_sync(SPB_FULL_MASK, head);
        rank[k] = __popc(b & lt);
        if (head) head_bits |= 1u << k;
        if (lane == 0) s_part[k * RH_WARPS + warp] = __popc(b);
    }
    __syncthreads();
    if (warp == 0) {
        u32 x = s_part[2 * lane], y = s_part[2 * lane + 1];
        u32 s = warp_incl_scan(x + y);
        u32 total = __shfl_sync(SPB_FULL_MASK, s, 31);
        s_part[2 * lane] = s - x - y;
        s_part[2 * lane + 1] = s - y;
        u64 excl = lookback_exclusive(state, tile, total);
        if (lane == 0) {
            s_excl = excl;
            if (base + RH_TILE >= n) *count = (u32)(excl + total);
        }
    }
    __syncthreads();
    const u64 excl = s_excl;
#pragma unroll
    for (int k = 0; k < RH_IPT; ++k) {
        if (!((head_bits >> k) & 1u)) continue;
        u64 slot = excl + s_part[k * RH_WARPS + warp] + rank[k];
        row_start[slot] = (u32)(base + (u64)k * RH_THREADS + tid);
        if (row_id) row_id[slot] = mine[k];
    }
}

// row_start[*count] = n  (the sentinel of dim_beginnings, algorithm.hpp:95-98)
__global__ void k_row_sentinel(u32 *row_start, const u32 *count, u32 n) { row_start[*count] = n; }

// len[row_id[r]] = row_start[r+1] - row_start[r]   (len zeroed beforehand)
__global__ void k_scatter_row_len(const u32 *__restrict__ row_start, const i32 *__restrict__ row_id,
                                  const u32 *count, u32 *len) {
    const u32 nr = *count;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (u64)gridDim.x * blockDim.x)
        len[row_id[r]] = row_start[r + 1] - row_start[r];
}

// Dense pointer straight from the compressed rows: ptr[v] = offset of the first entry whose leading index is >= v, for v in
// [0, extent].  Compressed row t fills the values (id[t-1], id[t]] -- the empty rows in front of it and itself -- and the last
// one also everything behind it.  One read of the compressed rows, one write of the pointer; no zero-fill, no scan.
// A stretch longer than DP_LONG_GAP values (rows {0, 2^31-1}: one thread would write 2^31 words) is not written by its
// thread but appended to `gaps`, and k_fill_gaps writes it with the whole grid.  Such a stretch needs at least DP_LONG_GAP
// empty rows, so the caller passes gaps = nullptr when extent + 1 - nrows is smaller: every thread then writes its own.
constexpr u64 DP_LONG_GAP = 4096;
struct DpGap { u64 lo, end; u32 value; };
__device__ __forceinline__ void dp_fill(u32 *ptr, u64 lo, u64 end, u32 value, DpGap *gaps, u32 *n_gaps) {
    if (gaps && end - lo > DP_LONG_GAP) {
        gaps[atomicAdd(n_gaps, 1u)] = DpGap{lo, end, value};
        return;
    }
    for (u64 v = lo; v < end; ++v) ptr[v] = value;
}
__global__ void k_dense_ptr_from_rows(const u32 *__restrict__ row_start, const i32 *__restrict__ row_id, u32 nrows, u32 n, u64 extent, u32 *ptr,
                                      DpGap *gaps, u32 *n_gaps) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nrows; t += (u64)gridDim.x * blockDim.x) {
        const u64 hi = (u64)(u32)row_id[t];
        const u64 lo = t ? (u64)(u32)row_id[t - 1] + 1 : 0;
        dp_fill(ptr, lo, hi + 1, row_start[t], gaps, n_gaps);
        if (t + 1 == nrows) dp_fill(ptr, hi + 1, extent + 1, n, gaps, n_gaps);
    }
}
__global__ void k_fill_gaps(const DpGap *__restrict__ gaps, const u32 *n_gaps, u32 *ptr) {
    const u32 ng = *n_gaps;
    for (u32 g = 0; g < ng; ++g) {
        const DpGap d = gaps[g];
        for (u64 v = d.lo + (u64)blockIdx.x * blockDim.x + threadIdx.x; v < d.end; v += (u64)gridDim.x * blockDim.x) ptr[v] = d.value;
    }
}
__global__ void k_fill_u32(u32 *p, u64 count, u32 value) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (u64)gridDim.x * blockDim.x) p[t] = value;
}

// Same for the leading-index values lo..hi-1 only: len[1 + id - lo] = entries of that row, len[0] = entries of the
// rows below lo (so that the exclusive scan of len[] yields absolute offsets from its second element on).
__global__ void k_scatter_row_len_range(const u32 *__restrict__ row_start, const i32 *__restrict__ row_id,
                                        const u32 *count, u64 lo, u64 hi, u32 *len) {
    const u32 nr = *count;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (u64)gridDim.x * blockDim.x) {
        const u64 id = (u64)row_id[r];
        const u32 c = row_start[r + 1] - row_start[r];
        if (id < lo) atomicAdd(&len[0], c);
        else if (id < hi) len[1 + id - lo] = c;
    }
}

// Sparse scale vector -> dense values (absent = 0) and presence mask (SURVEY App. A M6-M8).
// Entries whose index is beyond `dim` can never join a row/column and are ignored.  The reference's joins walk these
// vectors as sorted lists without repeats (xiter.hpp:146, 201); one that is not leaves *bad != 0 and the call fails --
// with a repeated index the scatter below would have no defined winner.
__global__ void k_densify(const i32 *__restrict__ idx, const double *__restrict__ val, u64 n, u64 dim,
                          double *dense, unsigned char *mask, u32 *bad) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        u32 j = (u32)idx[t];
        if (t && idx[t - 1] >= idx[t]) *bad = 1u;
        if (j < dim) {
            dense[j] = val[t];
            if (mask) mask[j] = 1;
        }
    }
}
