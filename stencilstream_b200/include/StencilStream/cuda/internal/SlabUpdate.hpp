/*
 * StencilStream-B200 — the multi-GPU partitioner: one row slab of a grid per GPU, depth-k halos
 * pushed to the neighbours over NVLink while the interior is being computed.
 *
 * The reference's cuda backend is single-device (StencilStream/cuda/StencilUpdate.hpp:83, :124-127),
 * so this component has no counterpart there; what it must preserve is the observable result of the
 * reference's generation loop (:212-273) on the whole grid. The temporal-blocking rules it relies on
 * are the reference's own for its tiled FPGA pipeline: a pass that fuses k iterations consumes a halo
 * of k * n_subiterations * radius cells (StencilStream/tiling/internal/StencilUpdateKernel.hpp:79-99).
 *
 * Decomposition. GPU g owns the global rows [row_lo, row_hi) of every plane and keeps `ghost` further
 * rows on each side, ghost = k * n_sub * r for the fusion depth k fixed at construction. A slab holds
 * two complete plane sets (ping/pong) and two 32-bit flags in ONE cudaMalloc block, so that a single
 * IPC handle (or, within a process, a peer mapping) makes all of it addressable by the neighbours.
 *
 * One pass (two launches that together advance the slab by n_gens <= k iterations), epoch e:
 *
 *   boundary stream:  wait  flag_from_up >= e+1, flag_from_down >= e+1      (ghosts of epoch e in place)
 *                     wait  interior launch of epoch e-1
 *                     sweep the top and bottom `ghost` rows of the slab in ONE launch; the kernel stores
 *                           them into the own target planes AND into the neighbours' ghost rows
 *                           (HaloPush), and its last CTA signals the neighbours:
 *                           their flag_from_{down,up} = e+2
 *   interior stream:  wait  boundary launches of epoch e-1
 *                     sweep the remaining rows (they depend on no ghost row)
 *
 * so the exchange for the next pass overlaps the interior sweep of this one, and nothing but the
 * small boundary launch ever waits for a neighbour (a slab too thin for two strips, or one built
 * without `overlap`, runs its pass as one launch, see pass()). Flags are waited for with
 * cuStreamWaitValue32 (stream-ordered, no host involvement, works across processes) and raised by the
 * boundary launch itself: every CTA fences its stores system-wide and takes an atomic ticket, the
 * holder of the last ticket stores the flags (exchange_halos(), which copies with cudaMemcpy, still
 * uses a one-thread kernel behind the copies). The flag protocol also
 * covers the write-after-read hazards of the ping/pong buffers: a neighbour can only write ghost rows
 * of buffer B in its epoch e+1 after it saw flag e+2, which is raised after this slab's epoch-e
 * boundary CTAs — the last readers of those ghost rows — have finished.
 *
 * Who provides the neighbours' addresses is not decided here: `attach()` takes raw pointers. Within a
 * process they come from another SlabUpdate (peer access enabled), across processes from
 * cudaIpcOpenMemHandle (see the stst_slab_* C ABI in include/stst_workloads.h, and
 * stencilstream_b200/sharding.py, which moves the handles with torch.distributed).
 */
#pragma once
#include "FieldOps.hpp"
#include "Helpers.hpp"
#include "Launch.hpp"
#include "PassThrough.hpp"
#include "Planner.hpp"
#include "Runtime.hpp"
#include "TileKernel.hpp"

#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace stencil {
namespace cuda {
namespace internal {

#if defined(__CUDACC__)
/// Raise a flag in (possibly remote) device memory once everything before it in the stream is done.
/// (A template only so that this header can be included in several translation units.)
template <int = 0> __global__ void raise_flag_kernel(volatile unsigned *flag, unsigned value) {
    __threadfence_system();
    *flag = value;
    __threadfence_system();
}
#endif

/// Byte layout of a slab's single device allocation; a pure function of its shape, so that a
/// neighbour can address into a mapped slab knowing only that slab's row range.
template <typename Cell> struct SlabLayout {
    using Layout = CellLayout<Cell>;
    /// [0]: flag_from_up, [1]: flag_from_down, [8]: ticket counter of the boundary launches
    static constexpr std::size_t flag_bytes = 256;
    static constexpr int ticket_word = 8;

    std::size_t width, owned_rows, ghost, buf_rows;
    std::size_t pitch[max_planes];        ///< elements between rows, per plane
    std::size_t plane_offset[2][max_planes]; ///< byte offset of plane i of buffer b
    std::size_t total_bytes;

    SlabLayout(std::size_t width, std::size_t owned_rows, std::size_t ghost)
        : width(width), owned_rows(owned_rows), ghost(ghost), buf_rows(owned_rows + 2 * ghost),
          pitch{}, plane_offset{}, total_bytes(0) {
        std::size_t offset = flag_bytes;
        for (int b = 0; b < 2; b++) {
            for (std::size_t i = 0; i < Layout::n_planes; i++) {
                const std::size_t elem = Layout::plane_bytes(i);
                std::size_t p = std::max<std::size_t>(width, 1);
                while ((p * elem) % 128 != 0)
                    p++;
                pitch[i] = p;
                plane_offset[b][i] = offset;
                const std::size_t bytes = p * buf_rows * elem;
                offset += (bytes + 255) / 256 * 256;
            }
        }
        total_bytes = offset;
    }

    PlaneSet planes(void *base, int buffer) const {
        PlaneSet set{};
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            set.base[i] = static_cast<unsigned char *>(base) + plane_offset[buffer][i];
            set.pitch[i] = pitch[i];
        }
        return set;
    }

    static unsigned *flag(void *base, int which) { return static_cast<unsigned *>(base) + which; }
};

/// Rows [lo, hi) owned by shard `index` of `count` when `rows` rows are dealt out as evenly as
/// possible (the first `rows % count` shards get one row more).
inline void partition_rows(std::size_t rows, std::size_t count, std::size_t index, std::size_t &lo,
                           std::size_t &hi) {
    const std::size_t base = rows / count, extra = rows % count;
    lo = index * base + std::min(index, extra);
    hi = lo + base + (index < extra ? 1 : 0);
}

enum class SlabSide : int { up = 0, down = 1 };

template <typename F> class SlabUpdate {
  public:
    using Cell = typename F::Cell;
    using Layout = CellLayout<Cell>;

    struct Config {
        std::size_t grid_rows, grid_cols; ///< extent of the WHOLE grid
        std::size_t row_lo, row_hi;       ///< global rows owned by this slab
        int device;
        unsigned fused_iterations; ///< upper bound for k; 0 = planner's choice. Must resolve to the
                                   ///< same k on every slab of a grid (checked by the caller).
        unsigned tile_rows;
        bool overlap; ///< boundary strips and interior in two launches (else one launch per pass)
    };

    explicit SlabUpdate(Config const &config)
        : cfg(config), plan(make_plan<F>(config.device, unsigned(config.row_hi - config.row_lo),
                                         unsigned(config.grid_cols), max_fused_iterations,
                                         config.fused_iterations, config.tile_rows)),
          ghost(std::size_t(plan.fused_iterations) * F::n_subiterations * F::stencil_radius),
          layout(config.grid_cols, config.row_hi - config.row_lo, ghost), base(nullptr), epoch(0),
          n_launches(0), interior_stream(nullptr), boundary_stream(nullptr) {
        if (cfg.row_hi <= cfg.row_lo || cfg.row_hi > cfg.grid_rows)
            throw std::invalid_argument("StencilStream-B200: illegal slab row range");
        if (cfg.grid_rows > 0x7fffffffull || cfg.grid_cols > 0x7fffffffull)
            throw std::range_error("StencilStream-B200 grids are limited to 2^31-1 rows/columns");
        const bool has_neighbour = cfg.row_lo > 0 || cfg.row_hi < cfg.grid_rows;
        if (has_neighbour && owned_rows() < ghost)
            throw std::invalid_argument(
                "StencilStream-B200: a slab must own at least k*n_sub*radius rows (its neighbour's "
                "ghost rows must come from one slab); use fewer GPUs or a smaller fused_iterations");
        // Events, streams and launches below belong to cfg.device: make it current for this thread.
        STST_RT_CHECK(stst_set_device(cfg.device));
        boundary_done = std::make_unique<Event>();
        interior_done = std::make_unique<Event>();
        STST_RT_CHECK(stst_malloc_ipc(cfg.device, layout.total_bytes, &base));
        STST_RT_CHECK(stst_stream_create(cfg.device, 0, &interior_stream));
        STST_RT_CHECK(stst_stream_create(cfg.device, 1, &boundary_stream));
        STST_RT_CHECK(stst_memset_async(base, 0, SlabLayout<Cell>::flag_bytes, interior_stream));
        STST_RT_CHECK(stst_stream_synchronize(interior_stream));
        for (int s = 0; s < 2; s++) {
            peer_base[s] = nullptr;
            peer_row_lo[s] = peer_row_hi[s] = 0;
        }
        // Fields the cell type declares constant (Cell::constant_fields) pass through from the
        // start; none of the backup / verify / repeat protocol below is needed for them.
        if (PassThrough<F>::declared())
            plan_passthrough();
    }

    SlabUpdate(SlabUpdate const &) = delete;
    SlabUpdate &operator=(SlabUpdate const &) = delete;

    ~SlabUpdate() {
        (void)stst_stream_synchronize(interior_stream);
        (void)stst_stream_synchronize(boundary_stream);
        pass_through.free_flags();
        device_free(cfg.device, backup_block, interior_stream);
        (void)stst_stream_synchronize(interior_stream);
        (void)stst_stream_destroy(interior_stream);
        (void)stst_stream_destroy(boundary_stream);
        (void)stst_free_ipc(cfg.device, base);
    }

    // ---- speculative plane pass-through on slabs ---------------------------------------------------
    //
    // Same mechanism as the single-GPU updater (PassThrough.hpp, run_tile in TileKernel.hpp): the
    // first pass observes which planes the transition function leaves unchanged, later passes leave
    // those planes in place, every pass verifies them. What differs is the repeat after a wrong
    // guess: a slab has no untouched source grid, and its neighbours have already consumed the rows it
    // pushed. The owner of the slabs therefore (1) calls backup() before run(), (2) combines
    // take_violations() of ALL slabs after it, and (3) if any slab reports one, has every slab
    // drop_passthrough(mask), restore() and run() again (sharding.py does this with one all-reduce
    // per call). Off unless enable_speculation(true).

    /// Turn detection on or off for the following run() calls (no-op for functors that cannot pass
    /// planes through or declare their constant fields). Returns whether it is on.
    bool enable_speculation(bool on) {
        detecting = on && PassThrough<F>::detected();
        return detecting;
    }

    /// Planes that currently pass through every sub-iteration.
    unsigned passthrough_planes() const {
        return (detecting || PassThrough<F>::declared()) ? pass_through.single_planes() : 0u;
    }

    /// Save the current generation (owned and ghost rows) so that restore() can return to it.
    void backup() {
        join_streams();
        // the ghost rows of the current generation are complete once the neighbours have raised
        // this epoch's flags — the same condition a pass waits for (with the NCCL transport the
        // receive that filled them is already ordered before this point by join_streams())
        for (int s = 0; s < 2 && !nccl_comm; s++) {
            if (has_side(s))
                STST_RT_CHECK(stst_stream_wait_value32_geq(interior_stream, my_flag(s),
                                                           unsigned(epoch + 1)));
        }
        const std::size_t bytes = plane_set_bytes();
        if (!backup_block)
            backup_block = device_alloc(cfg.device, bytes, interior_stream);
        STST_RT_CHECK(stst_memcpy_d2d_async(backup_block, plane_set_begin(int(epoch & 1)), bytes,
                                            interior_stream));
        fork_streams();
    }

    /// Return to the generation saved by backup(), as the *current* buffer. Every slab of the grid
    /// must do this at the same point (their ghost rows are part of what is restored).
    void restore() {
        if (!backup_block)
            throw std::logic_error("StencilStream-B200: restore() without backup()");
        join_streams();
        STST_RT_CHECK(stst_memcpy_d2d_async(plane_set_begin(int(epoch & 1)), backup_block,
                                            plane_set_bytes(), interior_stream));
        fork_streams();
    }

    /// Planes for which some pass since the last call saw a kept plane change. Waits for the slab.
    unsigned take_violations() {
        join_streams();
        const unsigned violated = pass_through.take_violations(interior_stream);
        fork_streams();
        return violated;
    }

    /// Never let `planes` pass through again.
    void drop_passthrough(unsigned planes) {
        pass_through.drop(planes);
        plan_passthrough();
    }

    // ---- topology ---------------------------------------------------------------------------------

    /// The slab's device allocation (export it with stst_ipc_get_mem_handle, or hand it to a slab
    /// of the same process).
    void *device_base() const { return base; }
    std::size_t device_bytes() const { return layout.total_bytes; }
    std::size_t owned_rows() const { return cfg.row_hi - cfg.row_lo; }
    std::size_t ghost_rows() const { return ghost; }
    bool has_up() const { return cfg.row_lo > 0; }
    bool has_down() const { return cfg.row_hi < cfg.grid_rows; }
    LaunchPlan const &get_plan() const { return plan; }
    /// The plan the next pass will use (taller tiles once planes pass through).
    LaunchPlan const &get_active_plan() const { return passthrough_planes() ? spec_plan : plan; }
    Config const &get_config() const { return cfg; }
    std::size_t get_n_launches() const { return n_launches; }
    std::size_t get_epoch() const { return epoch; }
    stst_stream_t stream() const { return interior_stream; }

    /// Make the neighbouring slab on `side`, mapped at `mapped_base` in this process and owning the
    /// global rows [row_lo, row_hi), the target of this slab's halo pushes.
    void attach(SlabSide side, void *mapped_base, std::size_t row_lo, std::size_t row_hi) {
        const int s = int(side);
        if (side == SlabSide::up ? row_hi != cfg.row_lo : row_lo != cfg.row_hi)
            throw std::invalid_argument("StencilStream-B200: attached slab is not adjacent");
        if (row_hi - row_lo < ghost)
            throw std::invalid_argument("StencilStream-B200: attached slab owns too few rows");
        peer_base[s] = mapped_base;
        peer_row_lo[s] = row_lo;
        peer_row_hi[s] = row_hi;
    }

    /**
     * Use NCCL instead of peer-mapped memory as the halo transport (north_star: "by P2P copies or NCCL
     * send/recv"): after its boundary strips a pass sends them with one grouped ncclSend/ncclRecv
     * exchange (stst_nccl_neighbor_exchange) and receives the neighbours' strips into its ghost rows.
     * The exchange itself orders the slabs — no flags, no mapped neighbour memory, no attach(). It is
     * the portable route (works wherever NCCL does, across nodes too); the default route stores
     * straight into the neighbour while sweeping and needs no extra launch. `up_rank` / `down_rank`:
     * NCCL ranks of the neighbours, negative where there is none. The communicator stays owned by the
     * caller.
     */
    void use_nccl(stst_nccl_comm_t comm, int up_rank, int down_rank) {
        if ((has_up() && up_rank < 0) || (has_down() && down_rank < 0))
            throw std::invalid_argument("StencilStream-B200: a neighbouring slab has no NCCL rank");
        nccl_comm = comm;
        nccl_rank[0] = up_rank;
        nccl_rank[1] = down_rank;
    }

    /// Forget both neighbours (after waiting for this slab's work): nothing this slab does afterwards
    /// touches their memory, so their owners may free it. Every slab of a grid detaches before any
    /// of them is destroyed (sharding.py: barrier, detach, barrier, destroy).
    void detach() {
        synchronize();
        for (int s = 0; s < 2; s++) {
            peer_base[s] = nullptr;
            peer_row_lo[s] = peer_row_hi[s] = 0;
        }
    }

    // ---- data ---------------------------------------------------------------------------------------

    /// Replace the owned rows by `cells` (dense row-major array of whole cells, owned_rows x width).
    /// Asynchronous on stream(); `cells` should be pinned and must stay valid until synchronize().
    void upload(const Cell *cells) { upload_rows(cells, 0, owned_rows()); }

    /// Replace `n_rows` owned rows starting at slab-local row `first_row` (for slabs too large to be
    /// staged in host memory at once).
    void upload_rows(const Cell *cells, std::size_t first_row, std::size_t n_rows) {
        check_row_range(first_row, n_rows);
        transfer</*to_device=*/true>(const_cast<Cell *>(cells), first_row, n_rows);
    }

    /// Copy the owned rows of the current generation into `cells`. Returns after the copy is done.
    void download(Cell *cells) { download_rows(cells, 0, owned_rows()); }

    void download_rows(Cell *cells, std::size_t first_row, std::size_t n_rows) {
        check_row_range(first_row, n_rows);
        join_streams();
        transfer</*to_device=*/false>(cells, first_row, n_rows);
        STST_RT_CHECK(stst_stream_synchronize(interior_stream));
    }

    /**
     * Max-norms of single fields over this slab's share of the extents (see Grid::max_abs): request q
     * covers the GLOBAL rows [0, rows[q]) and columns [0, cols[q]) of plane planes[q]; out[q] is the
     * maximum over the rows this slab owns (-infinity if it owns none of them). The caller combines
     * the slabs' values with `max` (an all-reduce across ranks). Waits for the slab's pending work.
     */
    void max_abs(std::size_t n, const std::size_t *planes_idx, const std::size_t *rows,
                 const std::size_t *cols, double *out) {
        join_streams();
        const PlaneSet planes = layout.planes(base, int(epoch & 1));
        for (std::size_t first = 0; first < n; first += max_field_reductions) {
            FieldReduceBatch batch{};
            batch.n = unsigned(std::min<std::size_t>(n - first, max_field_reductions));
            for (unsigned q = 0; q < batch.n; q++) {
                const std::size_t hi = std::min(rows[first + q], cfg.row_hi);
                batch.req[q].plane = unsigned(planes_idx[first + q]);
                batch.req[q].row_lo = unsigned(ghost);
                batch.req[q].row_hi = unsigned(hi > cfg.row_lo ? ghost + (hi - cfg.row_lo) : ghost);
                batch.req[q].cols = unsigned(std::min(cols[first + q], cfg.grid_cols));
            }
            select_device();
            reduce_max_abs<Cell>(cfg.device, interior_stream, planes, batch, out + first);
        }
    }

    /// Copy ONE field of `n_rows` owned rows starting at slab-local row `first_row` into the dense
    /// host array `dst` (n_rows x width elements of the field's type). Returns after the copy.
    void download_plane_rows(std::size_t plane, void *dst, std::size_t first_row,
                             std::size_t n_rows) {
        check_row_range(first_row, n_rows);
        join_streams();
        select_device();
        copy_plane_rows<Cell>(cfg.device, interior_stream, layout.planes(base, int(epoch & 1)), plane,
                              ghost + first_row, n_rows, cfg.grid_cols, dst, /*to_device=*/false);
        STST_RT_CHECK(stst_stream_synchronize(interior_stream));
    }

    /// The planes that hold the current generation, and how many ghost rows precede the owned rows
    /// in them (for copy_owned_rows_from of another slab).
    PlaneSet current_planes() const { return layout.planes(base, int(epoch & 1)); }

    /**
     * Replace the owned rows by those of another slab of the SAME grid rows, columns and cell type
     * on the same device — typically the slab of a different transition function over the same
     * cells (mantle convection alternates a pseudo-transient and a thermal update,
     * reference examples/convection/convection.cpp:405-455). Device-to-device, one copy per plane;
     * follow it with exchange_halos(). `other_*` describe the source slab's current planes, whose
     * contents must be complete (the caller synchronises the source slab first).
     */
    void copy_owned_rows_from(PlaneSet const &other_planes, std::size_t other_ghost) {
        join_streams();
        const PlaneSet mine = current_planes();
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            const std::size_t row_bytes = layout.pitch[i] * Layout::plane_bytes(i);
            STST_RT_CHECK(stst_memcpy_d2d_async(
                static_cast<unsigned char *>(mine.base[i]) + ghost * row_bytes,
                static_cast<const unsigned char *>(other_planes.base[i]) + other_ghost * row_bytes,
                owned_rows() * row_bytes, interior_stream));
        }
        fork_streams();
    }

    /**
     * Replace the owned AND the ghost rows by the corresponding rows of a whole grid whose planes
     * (same row pitch as a slab's: both are "width rounded up to 128 bytes") live on `grid_device` —
     * one contiguous device-to-device (peer) copy per plane, after `ready` (recorded on the grid's
     * stream) has fired. Because the ghost rows come along, no exchange_halos() is needed; like it,
     * this opens a fresh pair of epochs and is collective: every slab of the grid does it at the same
     * point of its sequence of operations. Used by the single-process multi-GPU path of
     * StencilUpdate (cuda/StencilUpdate.hpp, run_sharded).
     */
    void load_from_grid(PlaneSet const &grid_planes, int grid_device, stst_event_t ready) {
        join_streams();
        // The neighbours' last pass pushed into the ghost rows of the buffer that is about to be
        // overwritten: wait until those pushes have landed (the condition a pass waits for).
        // (A slab that has never run a pass or an exchange has no such pushes pending — and flags
        // that still read zero.)
        for (int s = 0; s < 2 && epoch > 0 && !nccl_comm; s++) {
            if (has_side(s))
                STST_RT_CHECK(stst_stream_wait_value32_geq(interior_stream, my_flag(s),
                                                           unsigned(epoch + 1)));
        }
        epoch += 2;
        const int cur = int(epoch & 1);
        const PlaneSet mine = layout.planes(base, cur);
        const std::size_t first = cfg.row_lo >= ghost ? cfg.row_lo - ghost : 0; // global rows copied
        const std::size_t last = std::min(cfg.grid_rows, cfg.row_hi + ghost);
        const std::size_t into = first + ghost - cfg.row_lo; // slab row that holds global row `first`
        if (ready)
            STST_RT_CHECK(stst_stream_wait_event(interior_stream, ready));
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            if (grid_planes.pitch[i] != layout.pitch[i])
                throw std::logic_error("StencilStream-B200: grid and slab row pitches differ");
            const std::size_t row_bytes = layout.pitch[i] * Layout::plane_bytes(i);
            STST_RT_CHECK(stst_memcpy_peer_async(
                static_cast<unsigned char *>(mine.base[i]) + into * row_bytes, cfg.device,
                static_cast<const unsigned char *>(grid_planes.base[i]) + first * row_bytes,
                grid_device, (last - first) * row_bytes, interior_stream));
        }
        // the ghost rows of the new epoch are in place: what the neighbours' flags would say
        for (int s = 0; s < 2; s++) {
            if (has_side(s))
                STST_RT_CHECK(stst_stream_write_value32(interior_stream, my_flag(s),
                                                        unsigned(epoch + 1)));
        }
        fork_streams();
    }

    /// Copy the owned rows of the current generation into the planes of a whole grid on
    /// `grid_device` (peer copy, one per plane) and record `done` behind the copies.
    void store_to_grid(PlaneSet const &grid_planes, int grid_device, stst_event_t done) {
        join_streams();
        const PlaneSet mine = current_planes();
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            if (grid_planes.pitch[i] != layout.pitch[i])
                throw std::logic_error("StencilStream-B200: grid and slab row pitches differ");
            const std::size_t row_bytes = layout.pitch[i] * Layout::plane_bytes(i);
            STST_RT_CHECK(stst_memcpy_peer_async(
                static_cast<unsigned char *>(grid_planes.base[i]) + cfg.row_lo * row_bytes,
                grid_device, static_cast<const unsigned char *>(mine.base[i]) + ghost * row_bytes,
                cfg.device, owned_rows() * row_bytes, interior_stream));
        }
        if (done)
            STST_RT_CHECK(stst_event_record(done, interior_stream));
        fork_streams();
    }

    /// Publish the owned boundary rows of the current buffer to the neighbours' ghost rows (needed
    /// once after upload(); afterwards every pass pushes its own boundary rows). Collective: every
    /// slab of the grid has to call it at the same point of its sequence of operations.
    void exchange_halos() {
        join_streams();
        // A fresh pair of epochs (same buffer parity): flag values raised for earlier passes must
        // not satisfy the waits of the passes that follow this exchange.
        epoch += 2;
        const int cur = int(epoch & 1);
        const PlaneSet mine = layout.planes(base, cur);
        if (nccl_comm) {
            nccl_exchange(cur);
            fork_streams();
            return;
        }
        for (int s = 0; s < 2; s++) {
            if (!has_side(s))
                continue;
            require_attached(s);
            const SlabLayout<Cell> peer(cfg.grid_cols, peer_row_hi[s] - peer_row_lo[s], ghost);
            const PlaneSet theirs = peer.planes(peer_base[s], cur);
            // rows I own next to that neighbour, and where they live in its planes
            const std::size_t my_first = (s == 0) ? ghost : ghost + owned_rows() - ghost;
            const std::size_t their_first = (s == 0) ? ghost + peer.owned_rows : 0;
            for (std::size_t i = 0; i < Layout::n_planes; i++) {
                const std::size_t row_bytes = layout.pitch[i] * Layout::plane_bytes(i);
                STST_RT_CHECK(stst_memcpy_d2d_async(
                    static_cast<unsigned char *>(theirs.base[i]) + their_first * row_bytes,
                    static_cast<const unsigned char *>(mine.base[i]) + my_first * row_bytes,
                    ghost * row_bytes, boundary_stream));
            }
            raise_flag(s, unsigned(epoch + 1));
        }
        fork_streams();
    }

    // ---- the generation loop --------------------------------------------------------------------------

    /// Enqueue `n_iterations` iterations starting at global iteration `iteration_offset`.
    void run(F const &tf, Cell const &halo_value, std::size_t iteration_offset,
             std::size_t n_iterations) {
        const std::size_t k = plan.fused_iterations;
        std::size_t iteration = iteration_offset;
        std::size_t remaining = n_iterations;
        while (remaining > 0) {
            const unsigned n_gens = unsigned(std::min(remaining, k));
            if (detecting && !pass_through.probed()) {
                // the first pass ever observes; its result tells which planes may stay in place
                const Speculation observe = pass_through.observing(cfg.device, interior_stream);
                pass(tf, halo_value, iteration, n_gens, &observe);
                join_streams();
                pass_through.read_observation(interior_stream);
                fork_streams();
                plan_passthrough();
            } else {
                const auto spec = passthrough_planes()
                                      ? pass_through.verifying(cfg.device, interior_stream)
                                      : std::nullopt;
                pass(tf, halo_value, iteration, n_gens, spec ? &*spec : nullptr);
            }
            iteration += n_gens;
            remaining -= n_gens;
        }
    }

    /// Record `event` behind everything enqueued on this slab so far (both streams).
    void record(stst_event_t event) {
        join_streams();
        STST_RT_CHECK(stst_event_record(event, interior_stream));
    }

    /// Wait until everything enqueued on this slab has finished.
    void synchronize() {
        STST_RT_CHECK(stst_stream_synchronize(boundary_stream));
        STST_RT_CHECK(stst_stream_synchronize(interior_stream));
    }

  private:
    bool has_side(int s) const { return s == 0 ? has_up() : has_down(); }

    void require_attached(int s) const {
        if (!peer_base[s])
            throw std::logic_error("StencilStream-B200: neighbouring slab not attached");
    }

    unsigned *my_flag(int s) const { return SlabLayout<Cell>::flag(base, s); }

    /// The flag INSIDE neighbour s that this slab raises: the up neighbour sees me as "down".
    unsigned *peer_flag(int s) const { return SlabLayout<Cell>::flag(peer_base[s], 1 - s); }

    void raise_flag(int s, unsigned value) {
#if defined(__CUDACC__)
        select_device();
        raise_flag_kernel<><<<1, 1, 0, static_cast<cudaStream_t>(boundary_stream)>>>(peer_flag(s),
                                                                                     value);
        if (cudaGetLastError() != cudaSuccess)
            throw std::runtime_error("StencilStream-B200: flag kernel launch failed");
        n_launches++;
#else
        (void)s, (void)value;
        throw std::runtime_error("StencilStream-B200 must be compiled with nvcc for sm_100a");
#endif
    }

    void select_device() {
#if defined(__CUDACC__)
        int current = -1;
        if (cudaGetDevice(&current) != cudaSuccess || current != cfg.device)
            cudaSetDevice(cfg.device);
#endif
    }

    /// boundary stream waits for the interior stream and vice versa
    void join_streams() {
        // Re-recording an event does not disturb waits that were enqueued on its earlier state.
        select_device();
        boundary_done->record(boundary_stream);
        STST_RT_CHECK(stst_stream_wait_event(interior_stream, boundary_done->get()));
        interior_done->record(interior_stream);
        STST_RT_CHECK(stst_stream_wait_event(boundary_stream, interior_done->get()));
    }

    void fork_streams() { join_streams(); }

    /// Plan the tiles for the planes that pass through. The fusion depth stays what the slab was
    /// built with: it fixes the ghost rows.
    void plan_passthrough() {
        spec_plan = make_plan<F>(cfg.device, unsigned(cfg.row_hi - cfg.row_lo),
                                 unsigned(cfg.grid_cols), max_fused_iterations,
                                 plan.fused_iterations, cfg.tile_rows, pass_through.single_planes());
        if (spec_plan.fused_iterations != plan.fused_iterations)
            throw std::logic_error("StencilStream-B200: pass-through changed the fusion depth");
    }

    std::size_t plane_set_bytes() const {
        return layout.plane_offset[1][0] - layout.plane_offset[0][0];
    }
    unsigned char *plane_set_begin(int buffer) const {
        return static_cast<unsigned char *>(base) + layout.plane_offset[buffer][0];
    }

    void pass(F const &tf, Cell const &halo_value, std::size_t iteration0, unsigned n_gens,
              Speculation const *spec) {
        const LaunchPlan &use_plan = (spec && !spec->probe) ? spec_plan : plan;
        const int cur = int(epoch & 1);
        const PlaneSet src = layout.planes(base, cur);
        const PlaneSet dst = layout.planes(base, cur ^ 1);

        HaloPush push{};
        push.up_row_hi = INT_MIN;
        push.down_row_lo = INT_MAX;
        for (int s = 0; s < 2 && !nccl_comm; s++) {
            if (!has_side(s))
                continue;
            require_attached(s);
            const SlabLayout<Cell> peer(cfg.grid_cols, peer_row_hi[s] - peer_row_lo[s], ghost);
            const PlaneSet theirs = peer.planes(peer_base[s], cur ^ 1);
            if (s == 0) {
                push.up = theirs;
                push.up_buf_row0 = int(peer_row_lo[s]) - int(ghost);
                push.up_row_hi = int(cfg.row_lo + ghost);
            } else {
                push.down = theirs;
                push.down_buf_row0 = int(peer_row_lo[s]) - int(ghost);
                push.down_row_lo = int(cfg.row_hi - ghost);
            }
        }
        const bool neighbours = has_up() || has_down();
        const bool pushes = neighbours && !nccl_comm; // store into mapped neighbour memory + flags

        LaunchRegion region{};
        region.device = cfg.device;
        region.grid_h = unsigned(cfg.grid_rows);
        region.grid_w = unsigned(cfg.grid_cols);
        region.buf_row0 = int(cfg.row_lo) - int(ghost);
        region.buf_rows = layout.buf_rows;

        // Everything launched in this pass reads rows written by BOTH streams in the previous pass.
        join_streams();
        for (int s = 0; s < 2 && !nccl_comm; s++) {
            if (has_side(s))
                STST_RT_CHECK(stst_stream_wait_value32_geq(boundary_stream, my_flag(s),
                                                           unsigned(epoch + 1)));
        }

        // The boundary launch raises the neighbours' flags itself (its last CTA, see HaloPush).
        if (pushes) {
            push.ticket = SlabLayout<Cell>::flag(base, SlabLayout<Cell>::ticket_word);
            push.flag_up = has_up() ? peer_flag(0) : nullptr;
            push.flag_down = has_down() ? peer_flag(1) : nullptr;
            push.flag_value = unsigned(epoch + 2);
        }

        // rows [lo, hi) and, optionally, [lo2, hi2) in ONE launch
        auto sweep = [&](std::size_t lo, std::size_t hi, std::size_t lo2, std::size_t hi2,
                         bool with_push, bool strip, stst_stream_t stream) {
            if (hi <= lo) {       // only the second range exists
                lo = lo2, hi = hi2;
                lo2 = hi2 = 0;
            }
            if (hi <= lo)
                return;
            region.out_row_lo = int(lo);
            region.out_row_hi = int(hi);
            region.out2_row_lo = int(lo2);
            region.out2_row_hi = int(hi2 > lo2 ? hi2 : lo2);
            region.tile_h = strip ? unsigned(hi - lo) : 0;
            SweepLauncher<F>::launch(use_plan, tf, halo_value, src, dst,
                                     (with_push && pushes) ? &push : nullptr, region, iteration0,
                                     n_gens, tensor_maps, stream, spec);
            n_launches++;
        };

        // How a pass is launched:
        //   overlap — both boundary strips in ONE launch on the high-priority stream (it waits for the
        //     neighbours' flags, pushes, and its last CTA raises their flags), the interior in another
        //     launch that needs no flag at all: two launches per pass. (A one-launch form whose tile
        //     rows ran boundary first was measured slower on 8 GPUs: the whole pass then waits for the
        //     neighbours' flags, FDTD 4608^2 565 vs 596, HotSpot 16384^2 5618 vs 5766
        //     GCell-updates/s, profiles/r02_pass_ab_8gpu_*.json.)
        //   no overlap, or a slab too thin for two strips — one launch in natural order, every CTA
        //     takes a ticket, the flags are raised at its very end.
        // Strips are `ghost` rows tall. Tile-high strips (no strip tile staging `ghost + 2 halo` rows
        // for `ghost` rows of output) were measured too: a boundary CTA spends ~18 us in its
        // system-scope fence and ticket whatever it computed (ncu, eight 576-row FDTD slabs: 84 strip
        // CTAs 25 us, 84 full-tile CTAs 45 us, a wave of interior tiles 22-26 us), and 576 rows are
        // 13.09 tile rows either way, so the taller strips only moved work into the launch that
        // holds its SMs longest (N = 2: 197 vs 195 GCell-updates/s; not adopted).
        const bool can_split = cfg.overlap && neighbours && owned_rows() > 2 * ghost;
        if (can_split) {
            // Two launches per pass: both boundary strips (with the halo push and the flags), then
            // the interior. (The NCCL transport needs the strips finished before it can send them.)
            const std::size_t top_hi = has_up() ? cfg.row_lo + ghost : cfg.row_lo;
            const std::size_t bottom_lo = has_down() ? cfg.row_hi - ghost : cfg.row_hi;
            sweep(cfg.row_lo, top_hi, bottom_lo, cfg.row_hi, true, true, boundary_stream);
            if (nccl_comm)
                nccl_exchange(cur ^ 1); // strips out, ghost rows of the next generation in
            sweep(top_hi, bottom_lo, 0, 0, false, false, interior_stream);
        } else {
            sweep(cfg.row_lo, cfg.row_hi, 0, 0, true, false, boundary_stream);
            if (nccl_comm)
                nccl_exchange(cur ^ 1);
        }
        epoch++;
    }

    /// Send the `ghost` owned rows next to each neighbour, receive that neighbour's into the ghost
    /// rows on the same side — all planes, both sides, one NCCL group on the boundary stream.
    void nccl_exchange(int buffer) {
        const PlaneSet mine = layout.planes(base, buffer);
        int peers[2 * max_planes];
        const void *send[2 * max_planes];
        void *recv[2 * max_planes];
        std::size_t send_bytes[2 * max_planes], recv_bytes[2 * max_planes];
        int n = 0;
        for (int s = 0; s < 2; s++) {
            if (!has_side(s))
                continue;
            const std::size_t my_first = (s == 0) ? ghost : owned_rows();        // rows I own there
            const std::size_t ghost_first = (s == 0) ? 0 : ghost + owned_rows(); // rows I receive
            for (std::size_t i = 0; i < Layout::n_planes; i++, n++) {
                const std::size_t row_bytes = layout.pitch[i] * Layout::plane_bytes(i);
                unsigned char *plane = static_cast<unsigned char *>(mine.base[i]);
                peers[n] = nccl_rank[s];
                send[n] = plane + my_first * row_bytes;
                recv[n] = plane + ghost_first * row_bytes;
                send_bytes[n] = recv_bytes[n] = ghost * row_bytes;
            }
        }
        if (n > 0)
            STST_RT_CHECK(stst_nccl_neighbor_exchange(nccl_comm, n, peers, send, send_bytes, recv,
                                                      recv_bytes, boundary_stream));
    }

    void check_row_range(std::size_t first_row, std::size_t n_rows) const {
        if (first_row > owned_rows() || n_rows > owned_rows() - first_row)
            throw std::range_error("StencilStream-B200: row range exceeds the slab");
    }

    template <bool to_device>
    void transfer(Cell *cells, std::size_t first_row, std::size_t n_rows) {
#if defined(__CUDACC__)
        select_device();
        const int cur = int(epoch & 1);
        PlaneSet planes = layout.planes(base, cur);
        const std::size_t width = cfg.grid_cols;
        const std::size_t row_bytes = std::max<std::size_t>(width * sizeof(Cell), 1);
        if (n_rows == 0)
            return;
        // pageable host memory moves through the runtime's staging ring, which drains per call:
        // larger device-side chunks amortise that (see GridStorage::rows_per_chunk)
        int pinned = 0;
        (void)stst_host_is_pinned(cells, &pinned);
        const std::size_t budget = std::size_t(pinned ? 64 : 256) << 20;
        const std::size_t chunk_rows =
            std::max<std::size_t>(1, std::min<std::size_t>(n_rows, budget / row_bytes));
        void *staging[2] = {device_alloc(cfg.device, chunk_rows * width * sizeof(Cell), interior_stream),
                            device_alloc(cfg.device, chunk_rows * width * sizeof(Cell), interior_stream)};
        std::size_t chunk = 0;
        for (std::size_t row = 0; row < n_rows; row += chunk_rows, chunk++) {
            const std::size_t rows = std::min(chunk_rows, n_rows - row);
            const std::size_t n = rows * width;
            Cell *stage = static_cast<Cell *>(staging[chunk & 1]);
            const unsigned block = 256;
            const unsigned grid =
                unsigned(std::min<std::size_t>((n + block - 1) / block, std::size_t(148) * 16));
            auto s = static_cast<cudaStream_t>(interior_stream);
            if constexpr (to_device) {
                STST_RT_CHECK(stst_memcpy_2d_auto(stage, row_bytes, cells + row * width, row_bytes,
                                                  row_bytes, rows, /*h2d*/ 0, cfg.device,
                                                  interior_stream));
                scatter_cells_kernel<Cell><<<grid, block, 0, s>>>(stage, planes, width,
                                                                  ghost + first_row + row, n);
            } else {
                gather_cells_kernel<Cell><<<grid, block, 0, s>>>(stage, planes, width,
                                                                 ghost + first_row + row, n);
                STST_RT_CHECK(stst_memcpy_2d_auto(stage, row_bytes, cells + row * width, row_bytes,
                                                  row_bytes, rows, /*d2h*/ 1, cfg.device,
                                                  interior_stream));
            }
            if (cudaGetLastError() != cudaSuccess)
                throw std::runtime_error("StencilStream-B200: layout kernel launch failed");
        }
        device_free(cfg.device, staging[0], interior_stream);
        device_free(cfg.device, staging[1], interior_stream);
#else
        (void)cells;
        throw std::runtime_error("StencilStream-B200 must be compiled with nvcc for sm_100a; "
                                 "there is no CPU fallback");
#endif
    }

    Config cfg;
    LaunchPlan plan;
    std::size_t ghost;
    SlabLayout<Cell> layout;
    void *base;
    std::size_t epoch;
    std::size_t n_launches;
    stst_stream_t interior_stream, boundary_stream;
    void *peer_base[2];
    std::size_t peer_row_lo[2], peer_row_hi[2];
    TensorMapCache<Cell> tensor_maps;
    std::unique_ptr<Event> boundary_done, interior_done;
    // plane pass-through; `detecting`: run-time detection on (enable_speculation)
    PassThrough<F> pass_through;
    bool detecting = false;
    LaunchPlan spec_plan{};
    // NCCL halo transport (use_nccl); nullptr: peer-mapped memory and flags
    stst_nccl_comm_t nccl_comm = nullptr;
    int nccl_rank[2] = {-1, -1};
    void *backup_block = nullptr;
};

} // namespace internal
} // namespace cuda
} // namespace stencil
