// cons_plan.cuh -- consolidate with a fixed index pattern (spb_consolidate_plan_*): the pattern is sorted once, stably and
// with every entry kept; each later consolidate of new values over that pattern is one gather pass plus the duplicate-reduce
// of reduce_by_key.cuh.
//
// Why the result equals a fresh consolidate bit for bit: the fresh path stably sorts the KEPT entries and folds every run
// left to right.  The plan holds the stable order of ALL entries; dropping the entries the drop rule rejects from that
// sequence leaves the kept entries in the same stable order, so the reduce pass sees the same keys and values in the same
// order.  The zero_nan rule needs the first kept entry of the sorted sequence (the "leading run", algorithm.hpp:272-275):
// the fresh path finds it by key and then by position (k_first_kept_key / k_first_kept_pos); in the plan's stable order it is
// simply the first sorted position whose value is neither 0 nor NaN, and a NaN is dropped iff it sits before that position.
#pragma once
#include "radix_sort.cuh"
#include "scan.cuh"

constexpr int CP_THREADS = 256;
constexpr int CP_IPT = 16;
constexpr int CP_TILE = CP_THREADS * CP_IPT;   // 4096 sorted positions per tile
constexpr int CP_WARPS = CP_THREADS / 32;

// Plan creation: the pattern sorted with the entry numbers as payload (k_iota_bits) -> packed keys and the permutation
// narrowed to 32 bits; n_runs counts the distinct keys.
__global__ void k_plan_pack(const i32 *__restrict__ hi, const i32 *__restrict__ lo, const double *__restrict__ iota, u32 n,
                            int bits_lo, u64 *__restrict__ keys, u32 *__restrict__ perm, u32 *n_runs) {
    u32 runs = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64 k = pack_key(hi[i], lo ? lo[i] : 0, bits_lo);
        keys[i] = k;
        perm[i] = (u32)__double_as_longlong(iota[i]);
        if (i == 0 || k != pack_key(hi[i - 1], lo ? lo[i - 1] : 0, bits_lo)) ++runs;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) runs += __shfl_xor_sync(SPB_FULL_MASK, runs, o);
    if (lane_id() == 0 && runs) atomicAdd(n_runs, runs);
}

// zero_nan: *bound = the first sorted position whose value is neither 0 nor NaN (0xffffffff: none; set by the caller).
// Tiles are taken in ascending order from a ticket, and a block stops as soon as a position below its next tile has been
// found, so the work follows the length of the leading run, not n.
__global__ void __launch_bounds__(CP_THREADS) k_plan_first_kept(const u32 *__restrict__ perm, const double *__restrict__ val,
                                                                u32 n, u32 *ticket, u32 *bound) {
    __shared__ u32 s_tile;
    for (;;) {
        if (threadIdx.x == 0) {
            const u32 t = atomicAdd(ticket, 1u);
            const u64 base = (u64)t * CP_TILE;
            s_tile = (base >= n || base >= (u64)ld_relaxed_u32(bound)) ? 0xffffffffu : t;
        }
        __syncthreads();
        const u32 tile = s_tile;
        __syncthreads();   // s_tile is rewritten by the next trip
        if (tile == 0xffffffffu) return;
        const u64 base = (u64)tile * CP_TILE;
        u32 best = 0xffffffffu;
#pragma unroll 4
        for (int k = 0; k < CP_IPT; ++k) {
            const u64 p = base + (u64)k * CP_THREADS + threadIdx.x;
            if (p < n) {
                const double v = val[perm[p]];
                if (v != 0.0 && !isnan(v) && (u32)p < best) best = (u32)p;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(SPB_FULL_MASK, best, o));
        if (lane_id() == 0 && best != 0xffffffffu) atomicMin(bound, best);
    }
}

struct PlanGatherArgs {
    const u64 *keys;      // [n] sorted packed keys of the plan
    const u32 *perm;      // [n] sorted position -> entry number
    const double *val;    // [n] the new values, in entry order
    u32 n;
    const u32 *bound;     // zero_nan: NaNs at sorted positions below *bound are dropped; nullptr: no NaN is dropped
    u64 *keys_out;        // kept (key, value) pairs, compacted in sorted order
    double *vals_out;
    u32 *n_kept;          // written by the last tile
    u64 *state;           // look-back words, one per tile, zeroed
    u32 *ticket;          // zeroed
};

// One pass over the sorted positions: read the permutation and the key, gather the value, apply consolidate()'s drop rule
// (input_kept: zeros always, NaNs before the bound) and write the kept pairs compacted.  Compaction is single-pass: warp
// ballots inside the tile, a decoupled look-back across tiles -- the pass reads 4 + 8 + 8 bytes and writes at most 16 bytes
// per entry.  (Per-tile counts + a separate scan + a scatter pass would read the permutation and the gathered values twice:
// 12 bytes more per entry, and the second gather is the expensive, scattered one.)  Items are warp-striped: item k of lane l
// of warp w is position tile * 4096 + w * 512 + k * 32 + l, so every load and every store of a warp covers consecutive slots.
__global__ void __launch_bounds__(CP_THREADS) k_plan_gather(PlanGatherArgs a) {
    __shared__ u32 s_tile;
    __shared__ u32 s_wcount[CP_WARPS];
    __shared__ u64 s_wbase[CP_WARPS];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(a.ticket, 1u);   // tiles in start order: the look-back never waits for an unscheduled tile
    __syncthreads();
    const u32 tile = s_tile;
    const u64 base = (u64)tile * CP_TILE;
    if (base >= a.n) return;
    const u32 bound = a.bound ? *a.bound : 0u;
    const u64 wbase = base + (u64)warp * (32 * CP_IPT) + lane;

    u32 p[CP_IPT];
#pragma unroll
    for (int k = 0; k < CP_IPT; ++k) {
        const u64 i = wbase + (u64)k * 32;
        p[k] = i < a.n ? __ldcs(a.perm + i) : 0u;
    }
    double v[CP_IPT];
#pragma unroll
    for (int k = 0; k < CP_IPT; ++k) {
        const u64 i = wbase + (u64)k * 32;
        v[k] = i < a.n ? __ldg(a.val + p[k]) : 0.0;
    }
    u64 key[CP_IPT];
#pragma unroll
    for (int k = 0; k < CP_IPT; ++k) {
        const u64 i = wbase + (u64)k * 32;
        key[k] = i < a.n ? ld_stream_u64(a.keys + i) : 0ull;
    }
    u32 mask[CP_IPT];
    u32 wcount = 0;
#pragma unroll
    for (int k = 0; k < CP_IPT; ++k) {
        const u64 i = wbase + (u64)k * 32;
        const bool ok = i < a.n && v[k] != 0.0 && !(isnan(v[k]) && (u32)i < bound);
        mask[k] = __ballot_sync(SPB_FULL_MASK, ok);
        wcount += __popc(mask[k]);
    }
    if (lane == 0) s_wcount[warp] = wcount;
    __syncthreads();
    if (warp == 0) {
        const u32 c = lane < (u32)CP_WARPS ? s_wcount[lane] : 0u;
        const u32 incl = warp_incl_scan(c);
        const u32 total = __shfl_sync(SPB_FULL_MASK, incl, 31);
        const u64 excl = lookback_exclusive(a.state, tile, total);
        if (lane < (u32)CP_WARPS) s_wbase[lane] = excl + incl - c;
        if (lane == 0 && base + CP_TILE >= a.n) *a.n_kept = (u32)(excl + total);
    }
    __syncthreads();
    u64 out = s_wbase[warp];
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int k = 0; k < CP_IPT; ++k) {
        if ((mask[k] >> lane) & 1u) {
            const u64 o = out + __popc(mask[k] & lt);
            a.keys_out[o] = key[k];
            a.vals_out[o] = v[k];
        }
        out += __popc(mask[k]);
    }
}
