// multiply_pattern_test.cpp -- b200::MultiplyPattern, the C++ face of spb_mm_pattern_*: one plan over fixed operand patterns,
// several value sets (fast path and fallback), every result equal to b200::multiply of the same indices and values, bit for
// bit.  Needs a GPU.  Built by __graft_entry__.build(), run by tests/test_gpu_multiply_pattern.py.
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

static bool same(DMat const &got, DMat const &want, std::array<size_t, 2> shape) {
    Mat g(shape), w(shape);
    got.download(g);
    want.download(w);
    bool ok = g.size() == w.size() && got.sort_order() == want.sort_order();
    ok = ok && (g.size() == 0 || std::memcmp(g.val_data().data(), w.val_data().data(), g.size() * sizeof(double)) == 0);
    for (int k = 0; k < 2; ++k) ok = ok && g.index_data(k) == w.index_data(k);
    return ok;
}

int main() {
    const double inf = std::numeric_limits<double>::infinity();
    // A: 4 x 5, unsorted with duplicates; B: 5 x 3, unsorted with duplicates
    const int ar[] = {2, 0, 2, 1, 0, 3, 2, 1, 0};
    const int ac[] = {1, 3, 1, 0, 4, 2, 1, 0, 3};
    const int br[] = {1, 3, 0, 4, 1, 2, 3, 0};
    const int bc[] = {2, 0, 1, 2, 2, 0, 1, 1};
    const int na = 9, nb = 8;
    const std::vector<std::vector<double>> a_sets = {
        {1.5, -2., 0.25, 3., 1., -0.5, 4., 2., 0.125},
        {1.5, 0., 0.25, 0., 1., -0.5, 4., 0., 0.},       // runs (1,0) and (0,3) emptied: fallback
        {1.5, -2., -1.5, 3., 1., -0.5, 0., 2., 0.125},   // (2,1) cancels to an explicit 0.0
        {0., 0., 0., 0., 0., 0., 0., 0., 0.},            // everything dropped
    };
    const std::vector<std::vector<double>> b_sets = {
        {0.5, 2., -1., 3., 0.75, 1., -2., 4.},
        {0.5, 2., -1., 3., -0.5, inf, -2., 4.},          // (1,2) cancels; an infinity
        {0., 2., -1., 3., 0., 1., -2., 4.},              // run (1,2) emptied: fallback
    };
    Mat pa({4, 5}), pb({5, 3});
    for (int i = 0; i < na; ++i) pa.add({ar[i], ac[i]}, 1.);
    for (int i = 0; i < nb; ++i) pb.add({br[i], bc[i]}, 1.);
    Vec w({5});
    w.add({0}, 2.); w.add({1}, 0.5); w.add({3}, -1.); w.add({4}, 3.);   // index 2 absent: inner index masked
    DVec dw(w);
    for (int pol = 0; pol < 3; ++pol) {
        const DuplicatePolicy p = (DuplicatePolicy)pol;
        b200::MultiplyPattern plan;
        {
            DMat da(pa), db(pb);
            DVec dw2(w);
            plan = b200::MultiplyPattern(1.5, nullptr, da, '.', &dw2, db, '.', nullptr, p);   // the plan outlives its inputs
        }
        CHECK(plan.nnz_bound() > 0);
        for (auto const &av : a_sets)
            for (auto const &bv : b_sets) {
                Mat a({4, 5}), b({5, 3});
                for (int i = 0; i < na; ++i) a.add({ar[i], ac[i]}, av[i]);
                for (int i = 0; i < nb; ++i) b.add({br[i], bc[i]}, bv[i]);
                DMat da(a), db(b);
                DMat want = b200::multiply(1.5, nullptr, da, '.', &dw, db, '.', nullptr, p);
                CHECK(same(plan.run(av.data(), bv.data()), want, {4, 3}));   // host values
                double *dav = nullptr, *dbv = nullptr;
                spb_coo_device_ptrs(da.handle(), nullptr, &dav);
                spb_coo_device_ptrs(db.handle(), nullptr, &dbv);
                CHECK(same(plan.run(dav, dbv), want, {4, 3}));               // device values
                CHECK(plan.run(av.data(), bv.data()).size() <= plan.nnz_bound());
            }
        b200::MultiplyPattern moved(std::move(plan));
        CHECK(plan.handle() == nullptr && moved.handle() != nullptr);
    }
    // a null value pointer is an error
    {
        DMat da(pa), db(pb);
        b200::MultiplyPattern plan(1.0, nullptr, da, '.', nullptr, db, '.', nullptr);
        bool threw = false;
        try { (void)plan.run(nullptr, b_sets[0].data()); } catch (spsparse::Exception const &) { threw = true; }
        CHECK(threw);
    }
    std::printf("multiply_pattern_test: %d failure(s)\n", failures);
    return failures ? 1 : 0;
}
