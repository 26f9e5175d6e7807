/*
 * StencilStream-B200 — per-field device operations on the plane image (PlaneImage.hpp) of a grid,
 * grid batch or slab: max-norm reductions and single-field transfers.
 *
 * The reference has no counterpart: its applications obtain such values on the host, through a
 * `GridAccessor` that migrates the WHOLE array-of-structs buffer first. Mantle convection does so
 * after every batch of pseudo-transient iterations — five max-norms over all cells
 * (reference examples/convection/convection.cpp:412-438, 88 bytes per cell over PCIe for 40 useful
 * ones) — and FDTD/convection write frames of ONE field (examples/fdtd/src/fdtd.cpp:114-166,
 * convection.cpp:460-477). Because `cuda::Grid` stores one plane per `Cell::fields` entry, both are
 * plane-local here:
 *
 *   field_requests          the requests of `FieldExtent`s (grid coordinates) on an image that holds
 *                           some of the grid's rows from some plane row on: a grid all rows from 0,
 *                           batch member m rows [0, H) from m * H, a slab its owned rows from `ghost`.
 *   reduce_max_abs_kernel   one launch evaluates up to `max_field_reductions` requests
 *                           max{ |plane[r][c]| : row_lo <= r < row_hi, c < cols } — every request
 *                           streams its sub-rectangle once with 128-bit loads; HBM-bound,
 *                           sizeof(field) bytes per cell and request.
 *   copy of one plane       a strided 2-D copy of the plane, no kernel, no other field touched.
 *
 * Comparison semantics are the reference loop's: start at -infinity, replace on `|v| > max`
 * (a NaN never replaces anything).
 */
#pragma once
#include "Helpers.hpp"
#include "Runtime.hpp"

#include <cstddef>
#include <cstdint>
#include <cstring>
#include <limits>
#include <stdexcept>
#include <type_traits>
#include <vector>

#if defined(__CUDACC__)
    #include <cuda_runtime.h>
#endif

namespace stencil {
namespace cuda {

/// B200 extension: "field `plane` (index into `Cell::fields`; 0 for scalar cells), restricted to the
/// first `rows` rows and `cols` columns of the grid" — the operand of `Grid::max_abs`.
struct FieldExtent {
    std::size_t plane;
    std::size_t rows, cols;
};

namespace internal {

inline constexpr unsigned max_field_reductions = 8;

/// One reduction: plane rows [row_lo, row_hi) (PLANE coordinates, ghosts included), columns [0, cols).
struct FieldReduceRequest {
    unsigned plane;
    unsigned row_lo, row_hi;
    unsigned cols;
};

struct FieldReduceBatch {
    unsigned n;
    FieldReduceRequest req[max_field_reductions];
};

/// Device results are kept as order-preserving integer keys of non-negative doubles so that the
/// cross-CTA combination is one 64-bit atomicMax: key = bit pattern + 1, 0 = "nothing seen".
STST_HD inline unsigned long long max_abs_key(double non_negative) {
    unsigned long long bits;
    memcpy(&bits, &non_negative, sizeof(bits));
    return bits + 1ull;
}

inline double max_abs_from_key(unsigned long long key) {
    if (key == 0)
        return -std::numeric_limits<double>::infinity();
    const unsigned long long bits = key - 1ull;
    double v;
    std::memcpy(&v, &bits, sizeof(v));
    return v;
}

/// Types a plane may hold for `reduce_max_abs`: arithmetic types, and enumerations (by their value).
template <typename T>
inline constexpr bool is_reducible_v = std::is_arithmetic_v<T> || std::is_enum_v<T>;

template <typename T> STST_HD constexpr double reducible_to_double(T const &v) {
    if constexpr (std::is_enum_v<T>)
        return double(static_cast<std::underlying_type_t<T>>(v));
    else
        return double(v);
}

/// True if plane `plane` of `Cell` holds such a type.
template <typename Cell> bool plane_is_arithmetic(std::size_t plane) {
    bool result = false;
    for_each_plane<Cell>([&](auto I) {
        if (plane == I)
            result = is_reducible_v<typename CellLayout<Cell>::template plane_t<I>>;
    });
    return result;
}

#if defined(__CUDACC__)

inline constexpr unsigned reduce_block_threads = 256;

/**
 * Grid: any number of CTAs (the launcher uses a multiple of the SM count); CTA b scans the rows
 * row_lo + b, row_lo + b + gridDim.x, ... of every request. `keys[q]` must be zero before the launch.
 */
template <typename Cell>
__global__ void __launch_bounds__(reduce_block_threads)
    reduce_max_abs_kernel(const __grid_constant__ PlaneSet planes,
                          const __grid_constant__ FieldReduceBatch batch,
                          unsigned long long *__restrict__ keys) {
    using L = CellLayout<Cell>;
    __shared__ double warp_max[reduce_block_threads / 32];

    for (unsigned q = 0; q < batch.n; q++) {
        const FieldReduceRequest rq = batch.req[q];
        double m = -1.0; // below every |v|; "nothing seen" if it survives
        for_each_plane<Cell>([&](auto I) {
            using T = typename L::template plane_t<I>;
            if constexpr (is_reducible_v<T>) {
                if (rq.plane != I)
                    return;
                constexpr unsigned V = sizeof(T) >= 16 ? 1u : unsigned(16 / sizeof(T));
                struct alignas(sizeof(T) * V) Vec {
                    T v[V];
                };
                const T *base = static_cast<const T *>(planes.base[I]);
                const unsigned long long pitch = planes.pitch[I];
                const unsigned n_vec = (rq.cols + V - 1) / V;
                for (unsigned row = rq.row_lo + blockIdx.x; row < rq.row_hi; row += gridDim.x) {
                    // rows start 128-byte aligned and are padded to 128 bytes: a vector that straddles
                    // `cols` stays inside the row's allocation
                    const Vec *rp = reinterpret_cast<const Vec *>(base + row * pitch);
                    for (unsigned i = threadIdx.x; i < n_vec; i += reduce_block_threads) {
                        const Vec x = rp[i];
#pragma unroll
                        for (unsigned j = 0; j < V; j++) {
                            if (i * V + j < rq.cols) {
                                double a = reducible_to_double(x.v[j]);
                                a = a < 0.0 ? -a : a;
                                if (a > m)
                                    m = a;
                            }
                        }
                    }
                }
            }
        });

#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double other = __shfl_xor_sync(0xffffffffu, m, o);
            if (other > m)
                m = other;
        }
        if ((threadIdx.x & 31u) == 0)
            warp_max[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (unsigned w = 1; w < reduce_block_threads / 32; w++)
                if (warp_max[w] > m)
                    m = warp_max[w];
            if (m >= 0.0)
                atomicMax(keys + q, max_abs_key(m));
        }
        __syncthreads();
    }
}

#endif // __CUDACC__

/**
 * Evaluate `requests` on `planes` (device `device`, in order on `stream`), one launch per
 * `max_field_reductions` of them, and wait for the results. result[q] = max |v| of request q,
 * -infinity if the request covers no cell.
 */
template <typename Cell>
inline std::vector<double> reduce_max_abs(int device, stst_stream_t stream, PlaneSet const &planes,
                                          std::vector<FieldReduceRequest> const &requests) {
    std::vector<double> result(requests.size());
#if defined(__CUDACC__)
    for (auto const &rq : requests) {
        if (rq.plane >= CellLayout<Cell>::n_planes || !plane_is_arithmetic<Cell>(rq.plane))
            throw std::invalid_argument("StencilStream-B200: field cannot be reduced (no such "
                                        "field, or not an arithmetic type)");
    }
    const std::size_t bytes = sizeof(unsigned long long) * max_field_reductions;
    for (std::size_t first = 0; first < requests.size(); first += max_field_reductions) {
        FieldReduceBatch batch{};
        batch.n = unsigned(std::min<std::size_t>(requests.size() - first, max_field_reductions));
        unsigned max_rows = 0;
        for (unsigned q = 0; q < batch.n; q++) {
            auto const &rq = batch.req[q] = requests[first + q];
            if (rq.row_hi > rq.row_lo && rq.cols > 0)
                max_rows = std::max(max_rows, rq.row_hi - rq.row_lo);
        }
        unsigned long long *host_keys = static_cast<unsigned long long *>(pinned_alloc(bytes));
        void *dev_keys = nullptr;
        try {
            dev_keys = device_alloc(device, bytes, stream);
            STST_RT_CHECK(stst_memset_async(dev_keys, 0, bytes, stream));
            if (max_rows > 0) {
                select_device(device);
                const unsigned ctas = std::min<unsigned>(max_rows, 148u * 8u);
                reduce_max_abs_kernel<Cell>
                    <<<ctas, reduce_block_threads, 0, static_cast<cudaStream_t>(stream)>>>(
                        planes, batch, static_cast<unsigned long long *>(dev_keys));
                if (cudaGetLastError() != cudaSuccess)
                    throw std::runtime_error("StencilStream-B200: reduction kernel launch failed");
            }
            STST_RT_CHECK(stst_memcpy_d2h_async(host_keys, dev_keys, bytes, stream));
            STST_RT_CHECK(stst_stream_synchronize(stream));
        } catch (...) {
            device_free(device, dev_keys, stream);
            pinned_free(host_keys);
            throw;
        }
        for (unsigned q = 0; q < batch.n; q++)
            result[first + q] = max_abs_from_key(host_keys[q]);
        device_free(device, dev_keys, stream);
        pinned_free(host_keys);
    }
#else
    (void)device, (void)stream, (void)planes;
    if (!requests.empty())
        throw std::runtime_error("StencilStream-B200 must be compiled with nvcc for sm_100a; "
                                 "there is no CPU fallback");
#endif
    return result;
}

/**
 * The requests that evaluate `extents` (grid coordinates: rows [0, extent.rows), columns
 * [0, extent.cols)) on an image whose plane rows from `plane_row0` on hold the grid rows
 * [row_lo, row_hi) of a grid `width` columns wide. Rows and columns outside those are not covered;
 * an extent that covers none of them gives an empty request.
 */
inline std::vector<FieldReduceRequest> field_requests(std::vector<FieldExtent> const &extents,
                                                      std::size_t width, std::size_t row_lo,
                                                      std::size_t row_hi, std::size_t plane_row0) {
    std::vector<FieldReduceRequest> requests(extents.size());
    for (std::size_t q = 0; q < extents.size(); q++) {
        const std::size_t hi = std::min(extents[q].rows, row_hi);
        requests[q].plane = unsigned(extents[q].plane);
        requests[q].row_lo = unsigned(plane_row0);
        requests[q].row_hi = unsigned(hi > row_lo ? plane_row0 + (hi - row_lo) : plane_row0);
        requests[q].cols = unsigned(std::min(extents[q].cols, width));
    }
    return requests;
}

/**
 * Copy plane rows [row_lo, row_lo + n_rows) x [0, cols) of plane `plane` into the dense row-major
 * host array `host` (to_device = false) or the other way round. In order on `stream`; the caller
 * synchronises the stream before it uses `host` (a pinned `host` is copied asynchronously).
 */
template <typename Cell>
inline void copy_plane_rows(int device, stst_stream_t stream, PlaneSet const &planes,
                            std::size_t plane, std::size_t row_lo, std::size_t n_rows,
                            std::size_t cols, void *host, bool to_device) {
    if (plane >= CellLayout<Cell>::n_planes)
        throw std::invalid_argument("StencilStream-B200: no such field");
    const std::size_t elem = CellLayout<Cell>::plane_bytes(plane);
    const std::size_t pitch_bytes = planes.pitch[plane] * elem;
    unsigned char *dev = static_cast<unsigned char *>(planes.base[plane]) + row_lo * pitch_bytes;
    // pinned host memory: one strided DMA; anything else: the runtime's staged pipeline
    STST_RT_CHECK(stst_memcpy_2d_auto(dev, pitch_bytes, host, cols * elem, cols * elem, n_rows,
                                      to_device ? 0 : 1, device, stream));
}

/// Index of the plane that stores `Cell::*Field`, for cells with a `fields` list.
template <typename Cell, auto Field> constexpr std::size_t plane_of_field() {
    static_assert(CellLayout<Cell>::is_split, "the cell type has no (complete) Cell::fields list");
    std::size_t found = CellLayout<Cell>::n_planes;
    for_each_plane<Cell>([&](auto I) {
        constexpr auto member = std::get<I>(Cell::fields);
        if constexpr (std::is_same_v<std::remove_cvref_t<decltype(member)>,
                                     std::remove_cvref_t<decltype(Field)>>) {
            if (member == Field)
                found = I;
        }
    });
    return found;
}

} // namespace internal
} // namespace cuda
} // namespace stencil
