// Host-only probe of the small-grid rule of the launch planner (cuda/internal/Planner.hpp:
// small_grid_tile_rows) for grid batches. Compiled with g++ (no device code, no CUDA runtime call)
// and driven by tests/test_batch_planner_cpu.py.
//   usage: batch_planner <tile_h> <halo> <tile_w> <grid_h> <grid_w> <members> <slots>
#include <StencilStream/cuda/internal/Planner.hpp>

#include <cstdio>
#include <cstdlib>

int main(int argc, char **argv) {
    if (argc != 8)
        return 2;
    unsigned a[7];
    for (int i = 0; i < 7; i++)
        a[i] = unsigned(std::strtoul(argv[i + 1], nullptr, 0));
    std::printf("%u\n", stencil::cuda::internal::small_grid_tile_rows(a[0], a[1], a[2], a[3], a[4],
                                                                       a[5], a[6]));
    return 0;
}
