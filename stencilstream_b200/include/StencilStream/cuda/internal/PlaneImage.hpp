/*
 * StencilStream-B200 — the plane image: the device format of a grid's cells, and the copies between
 * it and a host array of whole cells.
 *
 * A plane image of `rows` x `width` cells holds one row-major plane per `Cell::fields` entry
 * (CellLayout, Helpers.hpp). Each plane row is padded to the smallest pitch whose byte size is a
 * multiple of 128, so that every row start is 128-byte aligned and TMA-addressable. Each plane starts
 * at a multiple of 256 bytes, and all planes sit in one allocation. A grid and a grid batch
 * (GridStorage, cuda/Grid.hpp) hold one image; a row slab (SlabUpdate.hpp) holds two images of
 * owned + 2·ghost rows behind its flag words. The pitch depends on the width alone, so a row of a
 * slab and a row of a grid of the same width have the same byte size: slabs are filled from and
 * stored to a grid with one contiguous copy per plane.
 */
#pragma once
#include "Helpers.hpp"
#include "Runtime.hpp"

#include <algorithm>
#include <cstddef>
#include <stdexcept>
#include <string>

namespace stencil {
namespace cuda {
namespace internal {

/// Byte layout of a plane image of `rows` x `width` cells; a pure function of that shape.
template <typename Cell> struct PlaneImage {
    using Layout = CellLayout<Cell>;

    std::size_t pitch[max_planes];  ///< elements between consecutive rows, per plane
    std::size_t offset[max_planes]; ///< byte offset of plane i from the start of the image
    std::size_t bytes;              ///< size of the image, a multiple of 256

    /// Zero rows or columns count as one, so that an empty grid still gets planes to point at.
    PlaneImage(std::size_t width, std::size_t rows) : pitch{}, offset{}, bytes(0) {
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            const std::size_t elem = Layout::plane_bytes(i);
            // Smallest element count whose byte size is a multiple of both `elem` and 128.
            std::size_t p = std::max<std::size_t>(width, 1);
            while ((p * elem) % 128 != 0)
                p++;
            pitch[i] = p;
            offset[i] = bytes;
            bytes += (p * std::max<std::size_t>(rows, 1) * elem + 255) / 256 * 256;
        }
    }

    std::size_t row_bytes(std::size_t i) const { return pitch[i] * Layout::plane_bytes(i); }

    /// The planes of the image that starts at `base`.
    PlaneSet planes(void *base) const {
        PlaneSet set{};
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            set.base[i] = static_cast<unsigned char *>(base) + offset[i];
            set.pitch[i] = pitch[i];
        }
        return set;
    }

    /// Address of row `r` of plane `i` in `set`, an image of this layout.
    unsigned char *row(PlaneSet const &set, std::size_t i, std::size_t r) const {
        return static_cast<unsigned char *>(set.base[i]) + r * row_bytes(i);
    }
};

#if defined(__CUDACC__)

/**
 * Spread `n_rows` x `width` cells, stored as a dense row-major array of whole cells at `aos`, over the
 * planes, starting at plane row `plane_row0`. Counterpart of the reference's `scatter_kernel`
 * (cuda/StencilUpdate.hpp:294-321), but run once per host->device transfer instead of once per update.
 */
template <typename Cell>
__global__ void __launch_bounds__(256)
    scatter_cells_kernel(const Cell *__restrict__ aos, PlaneSet planes, unsigned long long width,
                         unsigned long long plane_row0, unsigned long long n_cells) {
    using L = CellLayout<Cell>;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
         idx < n_cells; idx += stride) {
        const unsigned long long r = idx / width, c = idx - r * width;
        const Cell cell = aos[idx];
        for_each_plane<Cell>([&](auto I) {
            using T = typename L::template plane_t<I>;
            static_cast<T *>(planes.base[I])[(plane_row0 + r) * planes.pitch[I] + c] =
                L::template get<I>(cell);
        });
    }
}

/// Inverse of scatter_cells_kernel; counterpart of the reference's `gather_kernel` (:408-438).
template <typename Cell>
__global__ void __launch_bounds__(256)
    gather_cells_kernel(Cell *__restrict__ aos, PlaneSet planes, unsigned long long width,
                        unsigned long long plane_row0, unsigned long long n_cells) {
    using L = CellLayout<Cell>;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
         idx < n_cells; idx += stride) {
        const unsigned long long r = idx / width, c = idx - r * width;
        Cell cell;
        for_each_plane<Cell>([&](auto I) {
            using T = typename L::template plane_t<I>;
            L::template get<I>(cell) =
                static_cast<const T *>(planes.base[I])[(plane_row0 + r) * planes.pitch[I] + c];
        });
        aos[idx] = cell;
    }
}

#endif // __CUDACC__

/**
 * Enqueue on `stream` of `device` the copy between the dense row-major array `cells` of `n_rows` x
 * `width` whole cells and plane rows [row0, row0 + n_rows) of `planes`: into the planes if
 * `to_device`, else out of them. `cells` may be any host memory: pinned memory is copied by DMA
 * directly, anything else through the runtime's staged pipeline (stst_memcpy_2d_auto).
 *
 * Cells of one plane take one strided copy. Split cells go through device staging buffers in chunks,
 * double-buffered, and scatter_cells_kernel / gather_cells_kernel convert between whole cells and
 * planes. The caller synchronises `stream` before it reuses or reads `cells`.
 */
template <typename Cell>
void transfer_cells(int device, stst_stream_t stream, PlaneSet const &planes, std::size_t width,
                    std::size_t row0, std::size_t n_rows, Cell *cells, bool to_device) {
    if (n_rows * width == 0)
        return;
    const std::size_t row_bytes = width * sizeof(Cell);
    const int kind = to_device ? /*h2d*/ 0 : /*d2h*/ 1;
    if constexpr (!CellLayout<Cell>::is_split) {
        const std::size_t pitch_bytes = planes.pitch[0] * sizeof(Cell);
        STST_RT_CHECK(stst_memcpy_2d_auto(static_cast<unsigned char *>(planes.base[0]) +
                                              row0 * pitch_bytes,
                                          pitch_bytes, cells, row_bytes, row_bytes, n_rows, kind,
                                          device, stream));
    } else {
#if defined(__CUDACC__)
        // Pageable host memory goes through the runtime's pinned staging ring, which drains at the
        // end of every call: larger device-side chunks amortise the drain.
        int pinned = 0;
        (void)stst_host_is_pinned(cells, &pinned);
        const std::size_t budget = std::size_t(pinned ? 64 : 256) << 20;
        const std::size_t chunk_rows =
            std::max<std::size_t>(1, std::min<std::size_t>(n_rows, budget / row_bytes));
        void *staging[2] = {device_alloc(device, chunk_rows * row_bytes, stream),
                            device_alloc(device, chunk_rows * row_bytes, stream)};
        select_device(device);
        const unsigned block = 256;
        std::size_t chunk = 0;
        for (std::size_t row = 0; row < n_rows; row += chunk_rows, chunk++) {
            const std::size_t rows = std::min(chunk_rows, n_rows - row);
            const std::size_t n = rows * width;
            Cell *stage = static_cast<Cell *>(staging[chunk & 1]);
            const unsigned grid =
                unsigned(std::min<std::size_t>((n + block - 1) / block, std::size_t(148) * 16));
            auto s = static_cast<cudaStream_t>(stream);
            if (to_device) {
                STST_RT_CHECK(stst_memcpy_2d_auto(stage, row_bytes, cells + row * width, row_bytes,
                                                  row_bytes, rows, kind, device, stream));
                scatter_cells_kernel<Cell><<<grid, block, 0, s>>>(stage, planes, width, row0 + row, n);
            } else {
                gather_cells_kernel<Cell><<<grid, block, 0, s>>>(stage, planes, width, row0 + row, n);
                STST_RT_CHECK(stst_memcpy_2d_auto(stage, row_bytes, cells + row * width, row_bytes,
                                                  row_bytes, rows, kind, device, stream));
            }
            const cudaError_t err = cudaGetLastError();
            if (err != cudaSuccess)
                throw std::runtime_error(
                    std::string("StencilStream-B200: layout kernel launch failed: ") +
                    cudaGetErrorString(err));
        }
        device_free(device, staging[0], stream);
        device_free(device, staging[1], stream);
#else
        throw std::runtime_error("StencilStream-B200 must be compiled with nvcc for sm_100a; "
                                 "there is no CPU fallback");
#endif
    }
}

} // namespace internal
} // namespace cuda
} // namespace stencil
