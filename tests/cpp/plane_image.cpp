// Host-only probe of the plane image format (cuda/internal/PlaneImage.hpp) and of the slab layout
// built on it (SlabLayout, cuda/internal/SlabUpdate.hpp). Compiled with g++ — no device code, no
// CUDA runtime call — and driven by tests/test_plane_image_cpu.py, which checks the printed layouts.
//   usage: plane_image    (one JSON object per line: every grid image, then every slab)
#include <StencilStream/cuda/internal/SlabUpdate.hpp>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <tuple>

using namespace stencil::cuda::internal;

struct MixedCell {
    double d;
    float f;
    std::int16_t h;
    std::uint8_t a, b;
    static constexpr auto fields =
        std::make_tuple(&MixedCell::d, &MixedCell::f, &MixedCell::h, &MixedCell::a, &MixedCell::b);
};
static_assert(CellLayout<MixedCell>::is_split && CellLayout<MixedCell>::n_planes == 5);

static const std::size_t widths[] = {1, 31, 1030, 16384};

static void print_list(const char *key, const std::size_t *values, std::size_t n) {
    std::printf(", \"%s\": [", key);
    for (std::size_t i = 0; i < n; i++)
        std::printf(i ? ", %zu" : "%zu", values[i]);
    std::printf("]");
}

template <typename Cell> void grid(const char *cell, std::size_t width, std::size_t rows) {
    const PlaneImage<Cell> image(width, rows);
    const std::size_t n = CellLayout<Cell>::n_planes;
    std::printf("{\"kind\": \"grid\", \"cell\": \"%s\", \"width\": %zu, \"rows\": %zu", cell, width,
                rows);
    print_list("pitch", image.pitch, n);
    print_list("offset", image.offset, n);
    std::printf(", \"bytes\": %zu}\n", image.bytes);
}

template <typename Cell>
void slab(const char *cell, std::size_t width, std::size_t owned, std::size_t ghost) {
    const SlabLayout<Cell> layout(width, owned, ghost);
    const std::size_t n = CellLayout<Cell>::n_planes;
    // The offsets are taken from real addresses inside an allocation of the slab's size.
    unsigned char *base = static_cast<unsigned char *>(std::malloc(layout.total_bytes));
    std::size_t pitch[2][max_planes], offset[2][max_planes];
    for (int b = 0; b < 2; b++) {
        const PlaneSet set = layout.planes(base, b);
        for (std::size_t i = 0; i < n; i++) {
            pitch[b][i] = std::size_t(set.pitch[i]);
            offset[b][i] = std::size_t(static_cast<unsigned char *>(set.base[i]) - base);
        }
    }
    std::free(base);
    std::printf("{\"kind\": \"slab\", \"cell\": \"%s\", \"width\": %zu, \"owned\": %zu, "
                "\"ghost\": %zu",
                cell, width, owned, ghost);
    print_list("pitch0", pitch[0], n);
    print_list("pitch1", pitch[1], n);
    print_list("offset0", offset[0], n);
    print_list("offset1", offset[1], n);
    std::printf(", \"bytes\": %zu}\n", layout.total_bytes);
}

template <typename Cell> void all(const char *cell) {
    for (std::size_t width : widths) {
        for (std::size_t rows : {0, 1, 7, 1000})
            grid<Cell>(cell, width, rows);
        slab<Cell>(cell, width, 7, 3);
        slab<Cell>(cell, width, 100, 6);
    }
}

int main() {
    all<bool>("u8");
    all<float>("f32");
    all<double>("f64");
    all<MixedCell>("mixed");
    return 0;
}
