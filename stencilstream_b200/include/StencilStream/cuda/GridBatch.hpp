/*
 * StencilStream-B200 — `stencil::cuda::GridBatch<Cell>`: B independent grids ("members") of the same
 * extent on one device, advanced together by `StencilUpdate::operator()(GridBatch &)` with one fused
 * launch per pass whatever B is (ensembles and parameter studies of small grids, which one launch
 * per member would leave launch-bound).
 *
 * Storage: the members are stacked by rows in ONE plane image (cuda/internal/PlaneImage.hpp) of
 * B * H x W cells, member b at plane rows [b * H, (b + 1) * H): the `GridStorage` of a `Grid<Cell>` of
 * that extent. Uploads, downloads and the per-field operations are the grid's own, with row offsets. The update treats
 * every member as a grid of its own: each member's neighbours outside its H x W cells read as
 * `halo_value`, so the result equals B separate grid updates, bit for bit.
 *
 * Like `Grid`, copying a GridBatch yields a second handle to the same cells. A batch has no host
 * accessor: cells move with `copy_from_host` / `copy_to_host` (whole batch or a member range).
 */
#pragma once
#include "Grid.hpp"

#include <stdexcept>
#include <vector>

namespace stencil {
namespace cuda {

template <typename Cell> class GridBatch {
  public:
    static constexpr std::size_t dimensions = 2;

    /// New, uninitialised batch of `members` grids of `rows` x `cols` cells on `cuda_device`
    /// (negative: the default device, STST_DEVICE or 0).
    GridBatch(std::size_t members, std::size_t rows, std::size_t cols, int cuda_device = -1)
        : members(members), rows(rows) {
        if (members > 0 && rows > 0x7fffffffull / members)
            throw std::range_error("StencilStream-B200 grid batches are limited to 2^31-1 rows in all");
        storage = std::make_shared<Storage>(members * rows, cols,
                                            cuda_device < 0 ? internal::default_device_ordinal()
                                                            : cuda_device);
    }

    GridBatch(GridBatch const &) = default;
    GridBatch &operator=(GridBatch const &) = default;

    /// Number of members.
    std::size_t get_members() const { return members; }

    /// Extent of one member: (rows, columns).
    sycl::range<2> get_grid_range() const { return sycl::range<2>(rows, storage->width); }

    /// New, uninitialised batch of the same member count and extent, on the same device.
    GridBatch make_similar() const { return GridBatch(members, rows, storage->width, storage->device); }

    /// Overwrite members [first_member, first_member + n_members) with the dense array `cells` of
    /// n_members x rows x cols cells; `n_cells` must be that count, else std::range_error.
    void copy_from_host(std::size_t first_member, std::size_t n_members, const Cell *cells,
                        std::size_t n_cells) {
        check_range(first_member, n_members, n_cells);
        storage->require_device();
        storage->transfer(const_cast<Cell *>(cells), /*to_device=*/true, first_member * rows,
                          n_members * rows);
        storage->device_written();
    }

    /// The whole batch from a dense array of members x rows x cols cells.
    void copy_from_host(const Cell *cells, std::size_t n_cells) {
        copy_from_host(0, members, cells, n_cells);
    }

    /// Copy members [first_member, first_member + n_members) into the dense array `cells` of
    /// n_members x rows x cols cells; `n_cells` must be that count, else std::range_error.
    void copy_to_host(std::size_t first_member, std::size_t n_members, Cell *cells,
                      std::size_t n_cells) {
        check_range(first_member, n_members, n_cells);
        storage->require_device();
        storage->transfer(cells, /*to_device=*/false, first_member * rows, n_members * rows);
    }

    /// The whole batch into a dense array of members x rows x cols cells.
    void copy_to_host(Cell *cells, std::size_t n_cells) { copy_to_host(0, members, cells, n_cells); }

    /// `Grid::max_abs` for member `member`: extents are member-local.
    std::vector<double> max_abs(std::size_t member, std::vector<FieldExtent> const &extents) {
        if (member >= members)
            throw std::range_error("StencilStream-B200: no such member in the grid batch");
        storage->require_device();
        return internal::reduce_max_abs<Cell>(
            storage->device, storage->stream, storage->planes,
            internal::field_requests(extents, storage->width, 0, rows, member * rows));
    }

    /// ONE field of every cell of every member into the dense host array `dst` (members x rows x
    /// cols elements of the field's type). Returns when the copy is complete.
    void copy_plane_to_host(std::size_t plane, void *dst) {
        storage->require_device();
        internal::copy_plane_rows<Cell>(storage->device, storage->stream, storage->planes, plane, 0,
                                        storage->height, storage->width, dst, /*to_device=*/false);
        STST_RT_CHECK(stst_stream_synchronize(storage->stream));
    }

    /// The stacked device image (members * rows x cols cells), used by StencilUpdate.
    internal::GridStorage<Cell> &get_storage() { return *storage; }

  private:
    using Storage = internal::GridStorage<Cell>;

    void check_range(std::size_t first_member, std::size_t n_members, std::size_t n_cells) const {
        if (first_member > members || n_members > members - first_member)
            throw std::range_error("StencilStream-B200: member range outside the grid batch");
        if (n_cells != n_members * rows * storage->width)
            throw std::range_error("The target buffer has not the same size as the grid batch members");
    }

    std::size_t members, rows;
    std::shared_ptr<Storage> storage;
};

} // namespace cuda
} // namespace stencil
