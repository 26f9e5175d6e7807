/*
 * StencilStream-B200 — `stencil::cuda::Grid<Cell>`: a two-dimensional grid that lives in B200 HBM.
 *
 * Drop-in for the reference's `stencil::cuda::Grid` (reference StencilStream/cuda/Grid.hpp:50-188):
 * same constructors, `copy_from_buffer` / `copy_to_buffer` (throwing `std::range_error` on a size
 * mismatch), nested `GridAccessor<mode>`, `get_grid_height/width/range`, `make_similar`, and the
 * same *handle* semantics — copying a Grid yields a second reference to the same cells
 * (reference Grid.hpp:97).
 *
 * What is different underneath: the reference keeps an array-of-structs `sycl::buffer<Cell, 2>` and
 * lets the SYCL runtime migrate it. Here the device copy is a plane image (cuda/internal/PlaneImage.hpp:
 * one row-major plane per `Cell::fields` entry), allocated from the runtime's stream-ordered pool; the
 * host copy is a lazily created pinned array-of-structs mirror that only exists once host code asks
 * for a `GridAccessor` or a buffer copy. Transfers between the two are explicit (`transfer_cells`)
 * and happen at the same points where SYCL would migrate: accessor construction and the next update.
 */
#pragma once
#include "internal/FieldOps.hpp"
#include "internal/Helpers.hpp"
#include "internal/PlaneImage.hpp"
#include "internal/Runtime.hpp"

#include <sycl/sycl.hpp>

#include <algorithm>
#include <cstdlib>
#if defined(__linux__)
    #include <sys/mman.h>
#endif
#include <cstring>
#include <memory>
#include <stdexcept>
#include <vector>

namespace stencil {
namespace cuda {

namespace internal {

/// Device ordinal used by grids and updaters that were not told otherwise (env STST_DEVICE, else 0).
inline int default_device_ordinal() {
    if (const char *env = std::getenv("STST_DEVICE"))
        return std::atoi(env);
    return 0;
}

/**
 * Shared state behind all handles to one grid: the device planes, the optional pinned host
 * mirror, and which of the two currently holds the authoritative contents.
 */
template <typename Cell> class GridStorage {
  public:
    using Layout = CellLayout<Cell>;

    GridStorage(std::size_t height, std::size_t width, int device)
        : height(height), width(width), device(device), stream(default_stream(device)),
          image(width, height), planes{}, device_block(nullptr), host(nullptr),
          host_is_pinned(false), host_current(true), device_current(true) {
        if (height > 0x7fffffffull || width > 0x7fffffffull)
            throw std::range_error("StencilStream-B200 grids are limited to 2^31-1 rows/columns");
    }

    GridStorage(GridStorage const &) = delete;
    GridStorage &operator=(GridStorage const &) = delete;

    ~GridStorage() {
        device_free(device, device_block, stream);
        if (host) {
            // The mirror may still be the source/target of an in-flight copy.
            (void)stst_stream_synchronize(stream);
            if (host_is_pinned)
                pinned_free(host);
            else
                std::free(host);
        }
    }

    /// Make sure the device planes exist (contents unspecified if they had to be created).
    void allocate_device() {
        if (device_block)
            return;
        device_block = device_alloc(device, image.bytes, stream);
        planes = image.planes(device_block);
    }

    void allocate_host() {
        if (host)
            return;
        const std::size_t bytes = std::max<std::size_t>(n_cells(), 1) * sizeof(Cell);
        void *p = nullptr;
        if (stst_malloc_host(bytes, &p) == 0) {
            host_is_pinned = true;
        } else {
            // The machine refuses to pin that much memory: an ordinary (pageable) mirror still
            // works, transfers are just staged by the driver and slower.
            // 2 MiB alignment + MADV_HUGEPAGE: a fresh gigabyte image otherwise takes a page fault
            // per 4 KiB the first time a download writes it.
            constexpr std::size_t huge = std::size_t(2) << 20;
            p = std::aligned_alloc(huge, (bytes + huge - 1) / huge * huge);
            if (!p)
                throw std::bad_alloc();
#if defined(__linux__) && defined(MADV_HUGEPAGE)
            (void)madvise(p, (bytes + huge - 1) / huge * huge, MADV_HUGEPAGE);
#endif
            host_is_pinned = false;
        }
        host = static_cast<Cell *>(p);
    }

    std::size_t n_cells() const { return height * width; }

    /// Bring the device planes up to date (uploading the host mirror if that is newer).
    void require_device() {
        allocate_device();
        if (!device_current) {
            transfer(host, /*to_device=*/true);
            device_current = true;
        }
    }

    /// Bring the host mirror up to date (downloading the planes if those are newer).
    void require_host() {
        allocate_host();
        if (!host_current) {
            transfer(host, /*to_device=*/false);
            host_current = true;
        }
    }

    /// The device planes were (or are being, in stream order) overwritten.
    void device_written() {
        device_current = true;
        host_current = false;
    }

    /// The host mirror was handed out for writing.
    void host_written() {
        host_current = true;
        device_current = false;
    }

    const std::size_t height, width;
    const int device;
    const stst_stream_t stream;
    const PlaneImage<Cell> image;
    PlaneSet planes;

    /**
     * Copy between the dense row-major array of whole cells at `cells` (any host memory, see
     * transfer_cells) and the device planes: into them if `to_device`, else out of them. Returns
     * when `cells` may be reused, or holds the cells. With `n_rows`, only plane rows
     * [row0, row0 + n_rows) are copied, to or from the first n_rows rows of `cells`.
     */
    void transfer(Cell *cells, bool to_device, std::size_t row0 = 0,
                  std::size_t n_rows = ~std::size_t(0)) {
        n_rows = std::min(n_rows, height - std::min(row0, height));
        if (n_rows * width == 0)
            return;
        allocate_device();
        transfer_cells<Cell>(device, stream, planes, width, row0, n_rows, cells, to_device);
        STST_RT_CHECK(stst_stream_synchronize(stream));
    }

    /// True if the host mirror exists and is the authoritative copy (or as current as the planes).
    bool host_is_current() const { return host != nullptr && host_current; }
    bool host_mirror_is_pinned() const { return host != nullptr && host_is_pinned; }

  private:
    void *device_block;
    Cell *host;
    bool host_is_pinned;
    bool host_current, device_current;

  public:
    Cell *host_data() { return host; }
};

} // namespace internal

template <typename Cell> class Grid {
  public:
    /// Number of grid dimensions.
    static constexpr std::size_t dimensions = 2;

    /// New, uninitialised grid of `r` rows and `c` columns.
    Grid(std::size_t r, std::size_t c)
        : storage(std::make_shared<Storage>(r, c, internal::default_device_ordinal())) {}

    /// New, uninitialised grid; `range[0]` rows, `range[1]` columns.
    Grid(sycl::range<2> range) : Grid(range[0], range[1]) {}

    /// New grid with the extent and contents of `other_buffer`.
    Grid(sycl::buffer<Cell, 2> other_buffer) : Grid(other_buffer.get_range()) {
        copy_from_buffer(other_buffer);
    }

    /// A further handle to the cells of `other_grid` (no copy).
    Grid(Grid const &other_grid) = default;
    Grid &operator=(Grid const &other_grid) = default;

    /// B200 extension: new, uninitialised grid on a specific CUDA device.
    Grid(std::size_t r, std::size_t c, int cuda_device)
        : storage(std::make_shared<Storage>(r, c, cuda_device)) {}

    /// Overwrite the grid with the contents of the equally-sized `other_buffer`.
    void copy_from_buffer(sycl::buffer<Cell, 2> other_buffer) {
        if (get_grid_range() != other_buffer.get_range()) {
            throw std::range_error("The target buffer has not the same size as the grid");
        }
        sycl::host_accessor other_ac(other_buffer, sycl::read_only);
        copy_from_host(other_ac.get_pointer());
    }

    /// B200 extension: `copy_from_buffer` from a dense row-major array of height x width cells. The
    /// cells go straight to the device (no intermediate host mirror).
    void copy_from_host(const Cell *cells) {
        storage->transfer(const_cast<Cell *>(cells), /*to_device=*/true);
        storage->device_written();
    }

    /// B200 extension: `copy_to_buffer` into a dense row-major array of height x width cells.
    void copy_to_host(Cell *cells) {
        if (storage->host_is_current()) {
            STST_RT_CHECK(stst_host_memcpy(static_cast<void *>(cells), storage->host_data(),
                                           storage->n_cells() * sizeof(Cell)));
        } else {
            storage->transfer(cells, /*to_device=*/false);
        }
    }

    /// Overwrite the equally-sized `other_buffer` with the contents of the grid.
    void copy_to_buffer(sycl::buffer<Cell, 2> other_buffer) {
        if (get_grid_range() != other_buffer.get_range()) {
            throw std::range_error("The target buffer has not the same size as the grid");
        }
        sycl::host_accessor other_ac(other_buffer, sycl::write_only);
        copy_to_host(other_ac.get_pointer());
    }

    /**
     * Host-side window onto the cells. Constructing one waits for outstanding device work on the
     * grid and brings the host mirror up to date (what a `sycl::host_accessor` does implicitly in
     * the reference, Grid.hpp:145-153); a writable accessor marks the device copy stale, so the next
     * update uploads the mirror first.
     */
    template <sycl::access::mode access_mode = sycl::access::mode::read_write> class GridAccessor {
      public:
        static constexpr int dimensions = 2;
        static constexpr bool is_read_only = (access_mode == sycl::access::mode::read);
        using value_type = std::conditional_t<is_read_only, const Cell, Cell>;
        using reference = value_type &;

        /// Pointer to one row; its subscript selects the column.
        class Row {
          public:
            explicit Row(value_type *row) : row(row) {}
            reference operator[](std::size_t c) const { return row[c]; }

          private:
            value_type *row;
        };

        GridAccessor(Grid &grid) : storage(grid.storage), width(grid.get_grid_width()) {
            storage->require_host();
            if constexpr (!is_read_only)
                storage->host_written();
            data = storage->host_data();
        }

        Row operator[](std::size_t r) const { return Row(data + r * width); }
        reference operator[](sycl::id<2> id) const { return data[id[0] * width + id[1]]; }

        sycl::range<2> get_range() const { return sycl::range<2>(storage->height, storage->width); }
        value_type *get_pointer() const { return data; }
        std::size_t size() const { return storage->n_cells(); }
        std::size_t byte_size() const { return storage->n_cells() * sizeof(Cell); }

      private:
        std::shared_ptr<internal::GridStorage<Cell>> storage; // keeps `data` alive
        std::size_t width;
        value_type *data;
    };

    /// Number of rows.
    std::size_t get_grid_height() const { return storage->height; }

    /// Number of columns.
    std::size_t get_grid_width() const { return storage->width; }

    /// (rows, columns).
    sycl::range<2> get_grid_range() const { return sycl::range<2>(storage->height, storage->width); }

    /// New, uninitialised grid of the same extent (and on the same device).
    Grid make_similar() const { return Grid(storage->height, storage->width, storage->device); }

    /// B200 extension: the shared state behind this handle (used by StencilUpdate).
    internal::GridStorage<Cell> &get_storage() { return *storage; }

    /**
     * B200 extension: max-norms of single fields, evaluated on the device in ONE pass over the planes
     * involved: result[q] = max{ |cell(r, c).field_q| : r < extents[q].rows, c < extents[q].cols },
     * -infinity for an empty extent. Replaces host loops over a `GridAccessor` such as the reference's
     * convergence check in examples/convection/convection.cpp:412-438 (which first migrates the whole
     * grid to the host). Waits for pending device work on the grid.
     */
    std::vector<double> max_abs(std::vector<FieldExtent> const &extents) {
        storage->require_device();
        return internal::reduce_max_abs<Cell>(
            storage->device, storage->stream, storage->planes,
            internal::field_requests(extents, storage->width, 0, storage->height, 0));
    }

    /// B200 extension: `max_abs` of the field `Cell::*Field` over the first `rows` x `cols` cells.
    template <auto Field> double max_abs(std::size_t rows, std::size_t cols) {
        return max_abs({FieldExtent{plane_of<Field>(), rows, cols}})[0];
    }

    /// B200 extension: index of the plane that stores `Cell::*Field`.
    template <auto Field> static constexpr std::size_t plane_of() {
        return internal::plane_of_field<Cell, Field>();
    }

    /// B200 extension: size in bytes of one element of plane `plane`.
    static std::size_t plane_element_bytes(std::size_t plane) {
        if (plane >= internal::CellLayout<Cell>::n_planes)
            throw std::invalid_argument("StencilStream-B200: no such field");
        return internal::CellLayout<Cell>::plane_bytes(plane);
    }

    /**
     * B200 extension: copy ONE field of every cell into the dense row-major host array `dst`
     * (height x width elements of the field's type) — `sizeof(field)` instead of `sizeof(Cell)` bytes
     * per cell over PCIe (frame dumps: reference examples/fdtd/src/fdtd.cpp:114-166,
     * examples/convection/convection.cpp:460-477). Returns when the copy is complete.
     */
    void copy_plane_to_host(std::size_t plane, void *dst) {
        storage->require_device();
        internal::copy_plane_rows<Cell>(storage->device, storage->stream, storage->planes, plane, 0, storage->height,
                                        storage->width, dst, /*to_device=*/false);
        STST_RT_CHECK(stst_stream_synchronize(storage->stream));
    }

    /// B200 extension: overwrite ONE field of every cell from the dense host array `src`.
    void copy_plane_from_host(std::size_t plane, const void *src) {
        storage->require_device();
        internal::copy_plane_rows<Cell>(storage->device, storage->stream, storage->planes, plane, 0, storage->height,
                                        storage->width, const_cast<void *>(src), /*to_device=*/true);
        STST_RT_CHECK(stst_stream_synchronize(storage->stream));
        storage->device_written();
    }

    /// B200 extension: `copy_plane_to_host` into a buffer of the field's type.
    template <auto Field, typename T> void copy_field_to_buffer(sycl::buffer<T, 2> other_buffer) {
        constexpr std::size_t plane = plane_of<Field>();
        static_assert(std::is_same_v<T, typename internal::CellLayout<Cell>::template plane_t<plane>>,
                      "buffer element type differs from the field's type");
        if (get_grid_range() != other_buffer.get_range()) {
            throw std::range_error("The target buffer has not the same size as the grid");
        }
        sycl::host_accessor other_ac(other_buffer, sycl::write_only);
        copy_plane_to_host(plane, other_ac.get_pointer());
    }

  private:
    using Storage = internal::GridStorage<Cell>;
    std::shared_ptr<Storage> storage;
};

} // namespace cuda
} // namespace stencil
