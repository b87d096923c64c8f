// device_array.hpp -- a COO array that STAYS on the GPU between operations, for C++ callers.
//
// The reference's templates work on host containers: every call of the drop-in layer (algorithm.hpp, multiply.hpp) uploads its
// operands and downloads its result, as the reference's signatures require.  A chain such as
//     consolidate(A) -> transpose -> multiply -> consolidate -> to_dense
// then crosses PCIe at every arrow.  DeviceCooArray<RANK> is the same chain with the arrows on the device: a move-only RAII
// owner of a `spb_coo` handle whose methods are the C-ABI kernels behind the reference routines they are named after --
//   consolidate      algorithm.hpp:251-319                 (spb_consolidate)
//   copy / transpose algorithm.hpp:30-37, 46-57            (spb_coo_copy, spb_coo_transpose: device-to-device)
//   to_dense         VectorCooArray.hpp:313-321 + the duplicate policies of DenseAccum, accum.hpp:110-140  (spb_coo_to_dense)
//   from_dense       to_sparse, algorithm.hpp:433-440      (spb_dense_to_coo)
//   dim_beginnings   algorithm.hpp:74-118                  (spb_dim_beginnings)
//   multiply         multiply_sparse.hpp:152-248, 281-365  (spb_multiply_mm, spb_multiply_mv)
// Index and value types are the C ABI's (int32, double).  Errors go through spsparse_error like everywhere else.
#pragma once

#include <utility>
#include <vector>

#include "algorithm.hpp"

namespace spsparse {
namespace b200 {

template <int RANK>
class DeviceCooArray {
    static_assert(RANK == 1 || RANK == 2, "rank 1 and 2 arrays only");
    spb_coo *h_ = nullptr;

    void info(uint64_t *shape, uint64_t *n, int *so) const {
        int rank = 0;
        uint64_t sh[2] = {0, 0}, nn = 0;
        int order[2] = {-1, -1};
        if (h_) check(spb_coo_info(h_, &rank, sh, &nn, order));
        if (shape) { shape[0] = sh[0]; shape[1] = sh[1]; }
        if (n) *n = nn;
        if (so) { so[0] = order[0]; so[1] = order[1]; }
    }

public:
    static const int rank = RANK;
    typedef int index_type;
    typedef double val_type;

    DeviceCooArray() {}
    explicit DeviceCooArray(spb_coo *adopt) : h_(adopt) {}   // takes ownership of a handle from the C ABI
    template <class IndexT, class ValT>
    explicit DeviceCooArray(VectorCooArray<IndexT, ValT, RANK> const &A) {   // upload (the sort-order flag travels with it)
        Handle t;
        upload(A, t);
        h_ = t.h;
        t.h = nullptr;
    }
    DeviceCooArray(DeviceCooArray const &) = delete;
    DeviceCooArray &operator=(DeviceCooArray const &) = delete;
    DeviceCooArray(DeviceCooArray &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    DeviceCooArray &operator=(DeviceCooArray &&o) noexcept {
        if (this != &o) { reset(); h_ = o.h_; o.h_ = nullptr; }
        return *this;
    }
    ~DeviceCooArray() { reset(); }
    void reset() {
        if (h_) spb_coo_free(default_context(), h_);
        h_ = nullptr;
    }
    spb_coo *handle() const { return h_; }
    spb_coo *release() { spb_coo *t = h_; h_ = nullptr; return t; }

    size_t size() const { uint64_t n = 0; info(nullptr, &n, nullptr); return (size_t)n; }
    std::array<size_t, RANK> shape() const {
        uint64_t sh[2];
        info(sh, nullptr, nullptr);
        std::array<size_t, RANK> out;
        for (int k = 0; k < RANK; ++k) out[k] = (size_t)sh[k];
        return out;
    }
    std::array<int, RANK> sort_order() const {   // {-1, ..} when not flagged sorted
        int so[2];
        info(nullptr, nullptr, so);
        std::array<int, RANK> out;
        for (int k = 0; k < RANK; ++k) out[k] = so[k];
        if (out[0] < 0) out.fill(-1), out[0] = -1;
        return out;
    }

    // ---- the operations, device to device ----------------------------------------------------------------------------------
    DeviceCooArray consolidate(std::array<int, RANK> const &sort_order, DuplicatePolicy policy = DuplicatePolicy::ADD,
                               bool zero_nan = false) const {
        spb_coo *r = nullptr;
        int so[2] = {sort_order[0], RANK > 1 ? sort_order[RANK - 1] : 0};
        check(spb_consolidate(default_context(), h_, so, policy_code(policy), zero_nan ? 1 : 0, &r, nullptr));
        return DeviceCooArray(r);
    }
    DeviceCooArray copy() const {
        spb_coo *r = nullptr;
        check(spb_coo_copy(default_context(), h_, &r));
        return DeviceCooArray(r);
    }
    // result.dim[k] == this->dim[perm[k]] (indices and shape); entries keep their order
    DeviceCooArray transpose(std::array<int, RANK> const &perm) const {
        spb_coo *r = nullptr;
        check(spb_coo_transpose(default_context(), h_, perm.data(), &r));
        return DeviceCooArray(r);
    }
    // row-major dense copy on the host; duplicates combine by `policy` in storage order, as DenseAccum would
    std::vector<double> to_dense(DuplicatePolicy policy = DuplicatePolicy::ADD) const {
        uint64_t sh[2];
        info(sh, nullptr, nullptr);
        size_t cells = 1;
        for (int k = 0; k < RANK; ++k) cells *= (size_t)sh[k];
        std::vector<double> dense(cells);
        check(spb_coo_to_dense(default_context(), h_, policy_code(policy), dense.data()));
        return dense;
    }
    // every element != 0 of a row-major host array, in storage order (to_sparse)
    static DeviceCooArray from_dense(std::array<size_t, RANK> const &shape, const double *dense) {
        uint64_t sh[2] = {0, 0};
        for (int k = 0; k < RANK; ++k) sh[k] = shape[k];
        spb_coo *r = nullptr;
        check(spb_dense_to_coo(default_context(), RANK, sh, dense, &r));
        return DeviceCooArray(r);
    }
    // offsets where the leading sorted index changes, plus the sentinel (the array must be flagged sorted)
    std::vector<size_t> dim_beginnings() const {
        const size_t n = size();
        std::vector<size_t> out;
        if (n == 0) return out;
        std::vector<uint64_t> buf(n + 1);
        uint64_t count = 0;
        check(spb_dim_beginnings(default_context(), h_, buf.data(), buf.size(), &count));
        out.assign(buf.begin(), buf.begin() + count);
        return out;
    }
    // entries into any accumulator (bulk copy when it is a VectorCooArray that covers the shape); sets no flag
    template <class AccumulatorT>
    void download(AccumulatorT &ret) const {
        if (h_) deliver<RANK>(ret, h_);
    }
};

// consolidate for a fixed index pattern (spb_consolidate_plan_*): the pattern of A is sorted once; consolidate(val, ...)
// returns what A-with-values-val .consolidate(sort_order, ...) would, bit for bit, with one gather pass and the
// duplicate-reduce instead of a sort.  `val` holds A.size() doubles in A's entry order, in device or host memory.  A may be
// destroyed once the plan exists.  Move-only; 12 bytes of device memory per entry.
template <int RANK>
class ConsolidatePlan {
    static_assert(RANK == 1 || RANK == 2, "rank 1 and 2 arrays only");
    spb_cons_plan *h_ = nullptr;
    size_t n_runs_ = 0;

public:
    ConsolidatePlan() {}
    ConsolidatePlan(DeviceCooArray<RANK> const &A, std::array<int, RANK> const &sort_order) {
        int so[2] = {sort_order[0], RANK > 1 ? sort_order[RANK - 1] : 0};
        uint64_t runs = 0;
        check(spb_consolidate_plan_create(default_context(), A.handle(), so, &h_, &runs));
        n_runs_ = (size_t)runs;
    }
    ConsolidatePlan(ConsolidatePlan const &) = delete;
    ConsolidatePlan &operator=(ConsolidatePlan const &) = delete;
    ConsolidatePlan(ConsolidatePlan &&o) noexcept : h_(o.h_), n_runs_(o.n_runs_) { o.h_ = nullptr; o.n_runs_ = 0; }
    ConsolidatePlan &operator=(ConsolidatePlan &&o) noexcept {
        if (this != &o) { reset(); h_ = o.h_; n_runs_ = o.n_runs_; o.h_ = nullptr; o.n_runs_ = 0; }
        return *this;
    }
    ~ConsolidatePlan() { reset(); }
    void reset() {
        if (h_) spb_consolidate_plan_destroy(h_);
        h_ = nullptr;
        n_runs_ = 0;
    }
    spb_cons_plan *handle() const { return h_; }
    size_t n_runs() const { return n_runs_; }   // distinct index tuples of the pattern

    DeviceCooArray<RANK> consolidate(const double *val, DuplicatePolicy policy = DuplicatePolicy::ADD,
                                     bool zero_nan = false) const {
        spb_coo *r = nullptr;
        check(spb_consolidate_plan_run(h_, val, policy_code(policy), zero_nan ? 1 : 0, &r, nullptr));
        return DeviceCooArray<RANK>(r);
    }
};

// multiply() for fixed operand patterns (spb_mm_pattern_*): the indices of A and B, the transpose flags, C, the scale vectors,
// the policy and zero_nan are fixed at construction; run(a_val, b_val) returns multiply() of A's and B's indices with those
// values (A.size() / B.size() doubles in entry order, device or host memory), bit for bit, without sorting or a symbolic phase.
// A, B and the scale vectors may be destroyed once the plan exists.  Move-only.
class MultiplyPattern {
    spb_mm_pattern *h_ = nullptr;
    size_t nnz_bound_ = 0;

public:
    MultiplyPattern() {}
    MultiplyPattern(double C, DeviceCooArray<1> const *scalei, DeviceCooArray<2> const &A, char transpose_A,
                    DeviceCooArray<1> const *scalej, DeviceCooArray<2> const &B, char transpose_B,
                    DeviceCooArray<1> const *scalek, DuplicatePolicy policy = DuplicatePolicy::ADD, bool zero_nan = false) {
        uint64_t bound = 0;
        check(spb_mm_pattern_create(default_context(), C, scalei ? scalei->handle() : nullptr, A.handle(), transpose_A,
                                    scalej ? scalej->handle() : nullptr, B.handle(), transpose_B,
                                    scalek ? scalek->handle() : nullptr, policy_code(policy), zero_nan ? 1 : 0, &h_, &bound));
        nnz_bound_ = (size_t)bound;
    }
    MultiplyPattern(MultiplyPattern const &) = delete;
    MultiplyPattern &operator=(MultiplyPattern const &) = delete;
    MultiplyPattern(MultiplyPattern &&o) noexcept : h_(o.h_), nnz_bound_(o.nnz_bound_) { o.h_ = nullptr; o.nnz_bound_ = 0; }
    MultiplyPattern &operator=(MultiplyPattern &&o) noexcept {
        if (this != &o) { reset(); h_ = o.h_; nnz_bound_ = o.nnz_bound_; o.h_ = nullptr; o.nnz_bound_ = 0; }
        return *this;
    }
    ~MultiplyPattern() { reset(); }
    void reset() {
        if (h_) spb_mm_pattern_destroy(h_);
        h_ = nullptr;
        nnz_bound_ = 0;
    }
    spb_mm_pattern *handle() const { return h_; }
    size_t nnz_bound() const { return nnz_bound_; }   // outputs of the full pattern: no run returns more

    DeviceCooArray<2> run(const double *a_val, const double *b_val) const {
        spb_coo *r = nullptr;
        check(spb_mm_pattern_run(h_, a_val, b_val, &r, nullptr));
        return DeviceCooArray<2>(r);
    }
};

// C * diag(scalei) * op(A) * diag(scalej) * op(B) * diag(scalek); absent scale vectors: nullptr.  Operands need not be
// consolidated (the library does what the reference's Consolidate<> does); the result is consolidated row-major.
inline DeviceCooArray<2> multiply(double C, DeviceCooArray<1> const *scalei, DeviceCooArray<2> const &A, char transpose_A,
                                  DeviceCooArray<1> const *scalej, DeviceCooArray<2> const &B, char transpose_B,
                                  DeviceCooArray<1> const *scalek, DuplicatePolicy policy = DuplicatePolicy::ADD, bool zero_nan = false) {
    spb_coo *r = nullptr;
    check(spb_multiply_mm(default_context(), C, scalei ? scalei->handle() : nullptr, A.handle(), transpose_A,
                          scalej ? scalej->handle() : nullptr, B.handle(), transpose_B, scalek ? scalek->handle() : nullptr,
                          policy_code(policy), zero_nan ? 1 : 0, &r, nullptr));
    return DeviceCooArray<2>(r);
}
inline DeviceCooArray<1> multiply(double C, DeviceCooArray<1> const *scalei, DeviceCooArray<2> const &A, char transpose_A,
                                  DeviceCooArray<1> const *scalej, DeviceCooArray<1> const &V,
                                  DuplicatePolicy policy = DuplicatePolicy::ADD, bool zero_nan = false) {
    spb_coo *r = nullptr;
    check(spb_multiply_mv(default_context(), C, scalei ? scalei->handle() : nullptr, A.handle(), transpose_A,
                          scalej ? scalej->handle() : nullptr, V.handle(), policy_code(policy), zero_nan ? 1 : 0, &r));
    return DeviceCooArray<1>(r);
}

}  // namespace b200
}  // namespace spsparse
