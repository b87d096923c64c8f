// consolidate_plan_test.cpp -- b200::ConsolidatePlan, the C++ face of spb_consolidate_plan_*: one plan over a fixed index
// pattern, several value sets, every result equal to DeviceCooArray::consolidate of the same indices and values.  Needs a
// GPU.  Built by __graft_entry__.build(), run by tests/test_gpu_consolidate_plan.py.
#include <spsparse/VectorCooArray.hpp>
#include <spsparse_b200/device_array.hpp>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>

using namespace spsparse;

static int failures = 0;
#define CHECK(cond)                                                          \
    do {                                                                     \
        if (!(cond)) { ++failures; std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

typedef VectorCooArray<int, double, 2> Mat;
typedef VectorCooArray<int, double, 1> Vec;
typedef b200::DeviceCooArray<2> DMat;
typedef b200::DeviceCooArray<1> DVec;

static bool same_bits(std::vector<double> const &a, std::vector<double> const &b) {
    return a.size() == b.size() && (a.empty() || std::memcmp(a.data(), b.data(), a.size() * sizeof(double)) == 0);
}

template <int RANK, class HostT>
static bool same_result(b200::DeviceCooArray<RANK> const &got, b200::DeviceCooArray<RANK> const &want, HostT shape_of) {
    HostT g(shape_of.shape), w(shape_of.shape);
    got.download(g);
    want.download(w);
    bool ok = g.size() == w.size() && same_bits(g.val_data(), w.val_data()) && got.sort_order() == want.sort_order();
    for (int k = 0; k < RANK; ++k) ok = ok && g.index_data(k) == w.index_data(k);
    return ok && got.dim_beginnings() == want.dim_beginnings();
}

static void test_rank2() {
    const double nan = std::numeric_limits<double>::quiet_NaN();
    const int rows[] = {2, 0, 2, 1, 0, 2, 3, 0, 2, 1};
    const int cols[] = {1, 3, 1, 0, 0, 3, 2, 3, 1, 0};
    const int n = 10;
    const std::vector<std::vector<double>> sets = {
        {4., 1.5, -1., 0.25, 2., 7., 3., 1., 0.5, 8.},          // all non-zero
        {0., 1.5, -0., 0.25, 2., 7., 3., 1., 0., 8.},           // run (2,1) emptied by zeros
        {4., 1.5, -4., 0.25, 2., 7., 3., -2.5, 0., -0.25},      // exact cancellations: explicit 0.0
        {nan, 1.5, 1., 0.25, nan, 7., 3., nan, 0.5, 8.},        // NaNs inside and after the leading run
        {0., 0., -0., 0., 0., 0., 0., 0., 0., 0.},              // everything dropped
    };
    Mat pattern({4, 4});
    for (int i = 0; i < n; ++i) pattern.add({rows[i], cols[i]}, 1.);
    for (int so = 0; so < 2; ++so) {
        const std::array<int, 2> order = so ? std::array<int, 2>{1, 0} : std::array<int, 2>{0, 1};
        b200::ConsolidatePlan<2> plan;
        {
            DMat dp(pattern);
            plan = b200::ConsolidatePlan<2>(dp, order);   // the plan outlives its input
        }
        CHECK(plan.n_runs() == 6);
        for (auto const &vals : sets) {
            Mat a({4, 4});
            for (int i = 0; i < n; ++i) a.add({rows[i], cols[i]}, vals[i]);
            DMat da(a);
            double *dval = nullptr;
            spb_coo_device_ptrs(da.handle(), nullptr, &dval);
            for (int pol = 0; pol < 3; ++pol)
                for (int zn = 0; zn < 2; ++zn) {
                    const DuplicatePolicy p = (DuplicatePolicy)pol;
                    DMat want = da.consolidate(order, p, zn != 0);
                    CHECK(same_result<2>(plan.consolidate(vals.data(), p, zn != 0), want, a));   // host values
                    CHECK(same_result<2>(plan.consolidate(dval, p, zn != 0), want, a));          // device values
                }
        }
        // moves
        b200::ConsolidatePlan<2> moved(std::move(plan));
        CHECK(plan.handle() == nullptr && moved.handle() != nullptr && moved.n_runs() == 6);
        CHECK(moved.consolidate(sets[0].data()).size() == 6);
    }
}

static void test_rank1_and_empty() {
    Vec v({8});
    const int idx[] = {5, 1, 5, 5, 0, 1};
    const double vals[] = {1., 2., 0.5, 0.25, -3., 0.};
    for (int i = 0; i < 6; ++i) v.add({idx[i]}, vals[i]);
    DVec dv(v);
    b200::ConsolidatePlan<1> plan(dv, {0});
    CHECK(plan.n_runs() == 3);
    for (int pol = 0; pol < 3; ++pol) {
        const DuplicatePolicy p = (DuplicatePolicy)pol;
        CHECK(same_result<1>(plan.consolidate(vals, p), dv.consolidate({0}, p), v));
    }
    // an empty pattern: empty results, flagged sorted
    DMat e(Mat({3, 3}));
    b200::ConsolidatePlan<2> pe(e, {0, 1});
    DMat r = pe.consolidate(nullptr);
    CHECK(pe.n_runs() == 0 && r.size() == 0 && r.sort_order()[0] == 0 && r.sort_order()[1] == 1);
    // a null value pointer for a non-empty pattern is an error
    bool threw = false;
    try { (void)plan.consolidate(nullptr); } catch (spsparse::Exception const &) { threw = true; }
    CHECK(threw);
}

int main() {
    test_rank2();
    test_rank1_and_empty();
    std::printf("consolidate_plan_test: %d failure(s)\n", failures);
    return failures ? 1 : 0;
}
