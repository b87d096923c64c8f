// mm_pattern.cuh -- multiply with a fixed operand pattern (spb_mm_pattern_*): each operand that spb_multiply_mm would
// consolidate is sorted once, with every entry kept; a run folds the new values of every run of equal indices into one slot
// per run, and the numeric kernels of spgemm.cuh read those slots.
//
// Why a fold equals consolidate(): consolidate stably sorts the KEPT entries and folds every run left to right.  The plan
// holds the stable order of ALL entries; skipping the entries the drop rule rejects leaves the kept ones of a run in the same
// order, so the fold sees the same values in the same order.  Consolidate drops zeros always, and with zero_nan the NaNs that
// precede the first kept entry of the REFERENCE's sorted sequence (input_kept, radix_sort.cuh).  For A the reference sorts as
// the plan does, so that bound is a sorted position; B is sorted by (inner, col) while the reference's order is (col, inner),
// so the plan keeps every sorted entry's position in the reference's order and the bound is a position in that order.
#pragma once
#include "common.cuh"
#include "reduce_by_key.cuh"

constexpr u32 PF_LONG_RUN = 256;   // runs longer than this are folded one warp per run (k_pattern_fold_long)

struct PatternFold {
    const u32 *perm;      // [n] sorted position -> entry number
    const u32 *off;       // [runs + 1] first sorted position of every run
    const u32 *ref_pos;   // [n] position of the sorted entry in the reference's order; nullptr: its sorted position
    const double *val;    // [n] the new values, in entry order
    const u32 *bound;     // zero_nan: a NaN at a (reference) position below *bound is dropped; nullptr: no NaN is dropped
    u32 runs;
    int policy;           // POLICY_ADD / LEAVE_ALONE / REPLACE
    double *out;          // [runs] the folded value of every run
    unsigned char *live;  // [runs] 1 where the run kept a value
    u32 *empty;           // runs left empty (zeroed by the caller)
    u32 *long_list;       // runs longer than PF_LONG_RUN, handed to k_pattern_fold_long
    u32 *long_count;      // (zeroed by the caller)
    u32 long_cap;
};

__device__ __forceinline__ bool pf_kept(const PatternFold &f, u32 bound, u32 p, double v) {
    if (v == 0.0) return false;
    if (isnan(v)) return (f.ref_pos ? f.ref_pos[p] : p) >= bound;
    return true;
}

// One thread per run, the values one after the other: ADD is acc = v0; acc += v1; ... (algorithm.hpp:279, 307-310),
// LEAVE_ALONE keeps the first kept value, REPLACE the last.  Long runs are listed for the warp kernel.
__global__ void __launch_bounds__(256) k_pattern_fold(PatternFold f) {
    const u32 bound = f.bound ? *f.bound : 0u;
    u32 empty = 0;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < f.runs; r += (u64)gridDim.x * blockDim.x) {
        const u32 s = f.off[r], e = f.off[r + 1];
        if (e - s > PF_LONG_RUN) {
            const u32 t = atomicAdd(f.long_count, 1u);
            if (t < f.long_cap) f.long_list[t] = (u32)r;
            continue;
        }
        double acc = 0.0;
        bool any = false;
        for (u32 p = s; p < e; ++p) {
            const double v = f.val[f.perm[p]];
            if (!pf_kept(f, bound, p, v)) continue;
            if (!any) { acc = v; any = true; }
            else if (f.policy == POLICY_ADD) acc = __dadd_rn(acc, v);
            else if (f.policy == POLICY_REPLACE) acc = v;
        }
        f.out[r] = acc;
        f.live[r] = any ? 1 : 0;
        empty += any ? 0u : 1u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) empty += __shfl_xor_sync(SPB_FULL_MASK, empty, o);
    if (lane_id() == 0 && empty) atomicAdd(f.empty, empty);
}

// Runs longer than PF_LONG_RUN: one warp per run.  The lanes gather 32 consecutive sorted positions at a time and the kept
// values are added one after the other in lane order, handed over by shuffles -- still the left-to-right fold.
__global__ void __launch_bounds__(256) k_pattern_fold_long(PatternFold f) {
    const u32 bound = f.bound ? *f.bound : 0u;
    u32 cnt = *f.long_count;
    if (cnt > f.long_cap) cnt = f.long_cap;
    const u32 lane = lane_id();
    const u32 warps = gridDim.x * (blockDim.x >> 5);
    for (u32 t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < cnt; t += warps) {
        const u32 r = f.long_list[t];
        const u32 s = f.off[r], e = f.off[r + 1];
        double acc = 0.0;
        bool any = false;
        for (u32 i = s; i < e; i += 32) {
            const u32 p = i + lane;
            double v = 0.0;
            bool k = false;
            if (p < e) { v = f.val[f.perm[p]]; k = pf_kept(f, bound, p, v); }
            u32 m = __ballot_sync(SPB_FULL_MASK, k);
            if (f.policy == POLICY_ADD) {
                while (m) {   // warp-uniform
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    const double x = __shfl_sync(SPB_FULL_MASK, v, l);
                    if (!any) { acc = x; any = true; }
                    else acc = __dadd_rn(acc, x);
                }
            } else if (m) {
                const int l = f.policy == POLICY_REPLACE ? 31 - __clz(m) : __ffs(m) - 1;
                const double x = __shfl_sync(SPB_FULL_MASK, v, l);
                if (f.policy == POLICY_REPLACE || !any) acc = x;
                any = true;
            }
        }
        if (lane == 0) {
            f.out[r] = acc;
            f.live[r] = any ? 1 : 0;
            if (!any) atomicAdd(f.empty, 1u);
        }
    }
}

// B flagged in the reference's order: spb_multiply_mm re-buckets it keeping every entry (zeros too), so its values are a
// pure gather through the permutation.
__global__ void k_pattern_gather(const u32 *__restrict__ perm, const double *__restrict__ val, u32 n, double *out) {
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (u64)gridDim.x * blockDim.x) out[p] = val[perm[p]];
}

// zero_nan on B: *bound = the smallest reference position of a value that is neither 0 nor NaN (0xffffffff: none; set by the
// caller).  The reference's first kept entry is that one: positions in the reference's order are its stable sort order.
__global__ void k_pattern_ref_bound(const u32 *__restrict__ perm, const u32 *__restrict__ ref_pos, const double *__restrict__ val,
                                    u32 n, u32 *bound) {
    u32 best = 0xffffffffu;
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (u64)gridDim.x * blockDim.x) {
        const double v = val[perm[p]];
        if (v != 0.0 && !isnan(v)) best = min(best, ref_pos[p]);
    }
    best = __reduce_min_sync(SPB_FULL_MASK, best);
    if (lane_id() == 0 && best != 0xffffffffu) atomicMin(bound, best);
}

// ---- plan creation ------------------------------------------------------------------------------------------------------
// The pattern sorted with the entry numbers as payload (k_iota_bits): the permutation, and a flag on the first entry of
// every run.
__global__ void k_pattern_heads(const i32 *__restrict__ hi, const i32 *__restrict__ lo, const double *__restrict__ iota, u32 n,
                                u32 *perm, unsigned char *head) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        perm[i] = (u32)__double_as_longlong(iota[i]);
        head[i] = (i == 0 || hi[i] != hi[i - 1] || lo[i] != lo[i - 1]) ? 1 : 0;
    }
}
// slot = exclusive scan of head (n + 1 entries): the run offsets and the consolidated index vectors, one entry per run
__global__ void k_pattern_runs(const i32 *__restrict__ hi, const i32 *__restrict__ lo, const unsigned char *__restrict__ head,
                               const u64 *__restrict__ slot, u32 n, u32 *off, i32 *run_hi, i32 *run_lo) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (head[i]) {
            const u64 r = slot[i];
            off[r] = (u32)i;
            run_hi[r] = hi[i];
            run_lo[r] = lo[i];
        }
        if (i == n - 1) off[slot[n]] = n;
    }
}
// ref_iota: the pattern sorted in the reference's order with the entry numbers as payload.  inv[entry] = reference position.
__global__ void k_pattern_invert(const double *__restrict__ ref_iota, u32 n, u32 *inv) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (u64)gridDim.x * blockDim.x)
        inv[(u32)__double_as_longlong(ref_iota[q])] = (u32)q;
}
__global__ void k_pattern_ref_pos(const u32 *__restrict__ perm, const u32 *__restrict__ inv, u32 n, u32 *ref_pos) {
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (u64)gridDim.x * blockDim.x) ref_pos[p] = inv[perm[p]];
}
