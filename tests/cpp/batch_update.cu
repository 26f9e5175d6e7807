// C++-level test of stencil::cuda::GridBatch with a transition function that is not part of the
// library: radius 2, a cell of two fields, a time-dependent value and border tests on `stencil.id`.
// Every member of the batch must equal the update of the same member as a Grid, bit for bit, in
// both staging paths (TMA and cp.async), and a single member range must round-trip.
// Runner: the Catch2 stand-in of oracle/ref_harness/catch2; built by
// stencilstream_b200/tools/build_reference_tests.py (`build_own`).
#include <StencilStream/BaseTransitionFunction.hpp>
#include <StencilStream/cuda/GridBatch.hpp>
#include <StencilStream/cuda/StencilUpdate.hpp>
#include <catch2/catch_all.hpp>

#include <cstdlib>
#include <cstring>
#include <tuple>
#include <vector>

using namespace stencil;

struct TwoField {
    float u, v;
    static constexpr auto fields = std::make_tuple(&TwoField::u, &TwoField::v);
};

struct CrossRadius2 : public BaseTransitionFunction {
    using Cell = TwoField;
    using TimeDependentValue = float;
    static constexpr std::size_t stencil_radius = 2;
    float w = 0.125f;
    STST_HD float get_time_dependent_value(std::size_t i) const { return 0.001f * float(i % 7); }
    STST_HD Cell operator()(Stencil<Cell, 2, float> const &st) const {
        float s = 0.0f;
        for (std::size_t d = 0; d < 5; d++)
            s += st[sycl::id<2>(2, d)].u + st[sycl::id<2>(d, 2)].v;
        const bool edge = st.id[0] == 0 || st.id[1] + 1 == st.grid_range[1];
        Cell c = st[sycl::id<2>(2, 2)];
        c.u = w * s + st.time_dependent_value + (edge ? 1.0f : 0.0f);
        c.v = 0.5f * c.v + 0.25f * st[sycl::id<2>(0, 4)].u;
        return c;
    }
};

static void run_case(std::size_t members, std::size_t rows, std::size_t cols, std::size_t n) {
    using Update = cuda::StencilUpdate<CrossRadius2>;
    std::vector<TwoField> cells(members * rows * cols);
    unsigned state = 12345u;
    for (auto &c : cells) {
        state = state * 1664525u + 1013904223u;
        c.u = float(state >> 8) / float(1u << 24);
        c.v = float(state & 0xffu) - 128.0f;
    }
    Update::Params params{};
    params.halo_value = TwoField{0.5f, -1.0f};
    params.iteration_offset = 3;
    params.n_iterations = n;
    params.blocking = true;
    Update batch_update(params);
    cuda::GridBatch<TwoField> batch(members, rows, cols);
    batch.copy_from_host(cells.data(), cells.size());
    cuda::GridBatch<TwoField> out = batch_update(batch);
    std::vector<TwoField> got(cells.size());
    out.copy_to_host(got.data(), got.size());
    REQUIRE(batch_update.get_n_processed_cells() == n * members * rows * cols);

    for (std::size_t b = 0; b < members; b++) {
        Update single_update(params);
        cuda::Grid<TwoField> grid(rows, cols);
        grid.copy_from_host(cells.data() + b * rows * cols);
        cuda::Grid<TwoField> result = single_update(grid);
        std::vector<TwoField> want(rows * cols);
        result.copy_to_host(want.data());
        REQUIRE(std::memcmp(want.data(), got.data() + b * rows * cols, want.size() * sizeof(TwoField)) == 0);
    }

    // one member range back, and the size check
    std::vector<TwoField> part(2 * rows * cols);
    out.copy_to_host(1, 2, part.data(), part.size());
    REQUIRE(std::memcmp(part.data(), got.data() + rows * cols, part.size() * sizeof(TwoField)) == 0);
    bool threw = false;
    try {
        out.copy_to_host(members - 1, 2, part.data(), part.size());
    } catch (std::range_error const &) {
        threw = true;
    }
    REQUIRE(threw);
}

TEST_CASE("GridBatch with a user functor equals per-member grids (TMA)", "[batch]") {
    setenv("STST_TMA", "1", 1);
    run_case(6, 131, 301, 9);
}

TEST_CASE("GridBatch with a user functor equals per-member grids (cp.async)", "[batch]") {
    setenv("STST_TMA", "0", 1);
    run_case(5, 70, 97, 7);
    setenv("STST_TMA", "1", 1);
}

int main() { return catch_standin::run_all_test_cases() == 0 ? 0 : 1; }
