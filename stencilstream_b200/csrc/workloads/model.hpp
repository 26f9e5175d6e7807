/*
 * libstst_workloads — the type-erased object model behind the C ABI of include/stst_workloads.h:
 * Grid / StencilUpdate / slab holders instantiated per transition function, and the registry entry
 * that creates them. Shared by the translation units that instantiate the backend for the individual
 * workloads (workloads_<group>.cu, compiled in parallel) and by workloads.cu, which implements the
 * C entry points. Everything is in a NAMED namespace: a grid created by one workload's entry may be
 * handed to another workload's updater (convection_pt / convection_thermal share a cell type), and the
 * `dynamic_cast` in UpdateHolder::apply must see ONE GridHolder<Cell> type across translation units.
 */
#pragma once
#include <StencilStream/cuda/StencilUpdate.hpp>
#include <StencilStream/cuda/internal/SlabUpdate.hpp>
#include <stst_workloads.h>

#include "functors.hpp"

#include <algorithm>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace stst_model {

using namespace stst_workloads;
namespace sc = stencil::cuda;

/// Message of the last failure on the calling thread (one instance for the whole library).
inline thread_local std::string g_error;

inline int report(int code, std::string message) {
    g_error = std::move(message);
    return code;
}

/// The C ABI's extents as the `FieldExtent`s of Grid::max_abs and its batch and slab counterparts.
inline std::vector<sc::FieldExtent> field_extents(const stst_field_extent *extents, std::size_t n) {
    std::vector<sc::FieldExtent> list(n);
    for (std::size_t q = 0; q < n; q++)
        list[q] = sc::FieldExtent{extents[q].field, extents[q].rows, extents[q].cols};
    return list;
}

// ---- type-erased object model -------------------------------------------------------------------

struct GridBase {
    virtual ~GridBase() = default;
    const char *workload = nullptr;
    virtual std::size_t rows() const = 0;
    virtual std::size_t cols() const = 0;
    virtual std::size_t cell_bytes() const = 0;
    virtual void copy_from_host(const void *cells) = 0;
    virtual void copy_to_host(void *cells) = 0;
    virtual void sync_to_device() = 0;
    virtual void *host_accessor(int mode) = 0;
    virtual bool host_pinned() = 0;
    virtual void max_abs(const stst_field_extent *extents, std::size_t n, double *out) = 0;
    virtual std::size_t field_bytes(std::size_t field) const = 0;
    virtual void copy_field(std::size_t field, void *host, bool to_device) = 0;
    virtual GridBase *share() = 0;
    virtual GridBase *make_similar() = 0;
};

template <typename Cell> struct GridHolder final : GridBase {
    sc::Grid<Cell> grid;
    GridHolder(const char *name, sc::Grid<Cell> g) : grid(std::move(g)) { workload = name; }
    std::size_t rows() const override { return grid.get_grid_height(); }
    std::size_t cols() const override { return grid.get_grid_width(); }
    std::size_t cell_bytes() const override { return sizeof(Cell); }
    void copy_from_host(const void *cells) override {
        // copy_from_buffer semantics without the intermediate sycl::buffer
        grid.copy_from_host(static_cast<const Cell *>(cells));
    }
    void copy_to_host(void *cells) override {
        grid.copy_to_host(static_cast<Cell *>(cells));
    }
    void sync_to_device() override {
        grid.get_storage().require_device();
        sc::internal::check(stst_stream_synchronize(grid.get_storage().stream), "stream sync");
    }
    void *host_accessor(int mode) override {
        if (mode == 0) {
            typename sc::Grid<Cell>::template GridAccessor<sycl::access::mode::read> ac(grid);
            return const_cast<void *>(static_cast<const void *>(ac.get_pointer()));
        }
        typename sc::Grid<Cell>::template GridAccessor<sycl::access::mode::read_write> ac(grid);
        return static_cast<void *>(ac.get_pointer());
    }
    bool host_pinned() override { return grid.get_storage().host_mirror_is_pinned(); }
    void max_abs(const stst_field_extent *extents, std::size_t n, double *out) override {
        const std::vector<double> result = grid.max_abs(field_extents(extents, n));
        std::copy(result.begin(), result.end(), out);
    }
    std::size_t field_bytes(std::size_t field) const override {
        return sc::Grid<Cell>::plane_element_bytes(field);
    }
    void copy_field(std::size_t field, void *host, bool to_device) override {
        if (to_device)
            grid.copy_plane_from_host(field, host);
        else
            grid.copy_plane_to_host(field, host);
    }
    GridBase *share() override { return new GridHolder(workload, grid); }
    GridBase *make_similar() override { return new GridHolder(workload, grid.make_similar()); }
};

struct BatchBase {
    virtual ~BatchBase() = default;
    const char *workload = nullptr;
    virtual std::size_t members() const = 0;
    virtual std::size_t rows() const = 0;
    virtual std::size_t cols() const = 0;
    virtual std::size_t cell_bytes() const = 0;
    virtual void copy(std::size_t first_member, std::size_t n_members, void *cells, std::size_t bytes,
                      bool to_device) = 0;
    virtual void max_abs(std::size_t member, const stst_field_extent *extents, std::size_t n,
                         double *out) = 0;
    virtual std::size_t field_bytes(std::size_t field) const = 0;
    virtual void copy_field_to_host(std::size_t field, void *host) = 0;
};

template <typename Cell> struct BatchHolder final : BatchBase {
    sc::GridBatch<Cell> batch;
    BatchHolder(const char *name, sc::GridBatch<Cell> b) : batch(std::move(b)) { workload = name; }
    std::size_t members() const override { return batch.get_members(); }
    std::size_t rows() const override { return batch.get_grid_range()[0]; }
    std::size_t cols() const override { return batch.get_grid_range()[1]; }
    std::size_t cell_bytes() const override { return sizeof(Cell); }
    void copy(std::size_t first_member, std::size_t n_members, void *cells, std::size_t bytes,
              bool to_device) override {
        if (bytes % sizeof(Cell) != 0)
            throw std::range_error("The target buffer has not the same size as the grid batch members");
        if (to_device)
            batch.copy_from_host(first_member, n_members, static_cast<const Cell *>(cells),
                                 bytes / sizeof(Cell));
        else
            batch.copy_to_host(first_member, n_members, static_cast<Cell *>(cells),
                               bytes / sizeof(Cell));
    }
    void max_abs(std::size_t member, const stst_field_extent *extents, std::size_t n,
                 double *out) override {
        const std::vector<double> result = batch.max_abs(member, field_extents(extents, n));
        std::copy(result.begin(), result.end(), out);
    }
    std::size_t field_bytes(std::size_t field) const override {
        return sc::Grid<Cell>::plane_element_bytes(field);
    }
    void copy_field_to_host(std::size_t field, void *host) override {
        batch.copy_plane_to_host(field, host);
    }
};

struct UpdateBase {
    virtual ~UpdateBase() = default;
    const char *workload = nullptr;
    virtual void set_params(const stst_update_params &p) = 0;
    virtual GridBase *apply(GridBase &source) = 0;
    virtual BatchBase *apply_batch(BatchBase &source) = 0;
    virtual void stats(stst_update_stats &s) = 0;
};

template <typename F, typename ParamBlock> struct UpdateHolder final : UpdateBase {
    using Update = sc::StencilUpdate<F>;
    using Cell = typename F::Cell;
    std::unique_ptr<Update> update;

    static typename Update::Params convert(const stst_update_params &p) {
        if (p.transition_function_bytes != sizeof(ParamBlock) || p.transition_function == nullptr)
            throw std::invalid_argument("transition_function_bytes does not match the workload's "
                                        "parameter struct");
        if (p.halo_value != nullptr && p.halo_value_bytes != sizeof(Cell))
            throw std::invalid_argument("halo_value_bytes does not match the workload's cell type");
        typename Update::Params out{};
        std::memcpy(&out.transition_function.p, p.transition_function, sizeof(ParamBlock));
        if (p.halo_value != nullptr)
            std::memcpy(static_cast<void *>(&out.halo_value), p.halo_value, sizeof(Cell));
        out.iteration_offset = p.iteration_offset;
        out.n_iterations = p.n_iterations;
        out.blocking = p.blocking != 0;
        out.profiling = p.profiling != 0;
        out.cuda_device = p.cuda_device;
        out.fused_iterations = p.fused_iterations;
        out.tile_rows = p.tile_rows;
        if (p.n_cuda_devices != 0) {
            if (p.cuda_devices == nullptr)
                throw std::invalid_argument("n_cuda_devices is set but cuda_devices is null");
            out.cuda_devices.assign(p.cuda_devices, p.cuda_devices + p.n_cuda_devices);
        }
        return out;
    }

    UpdateHolder(const char *name, const stst_update_params &p)
        : update(std::make_unique<Update>(convert(p))) {
        workload = name;
    }

    void set_params(const stst_update_params &p) override { update->get_params() = convert(p); }

    GridBase *apply(GridBase &source) override {
        auto *typed = dynamic_cast<GridHolder<Cell> *>(&source);
        if (!typed)
            throw std::invalid_argument("grid belongs to a workload with a different cell type");
        sc::Grid<Cell> result = (*update)(typed->grid);
        return new GridHolder<Cell>(source.workload, result);
    }

    BatchBase *apply_batch(BatchBase &source) override {
        auto *typed = dynamic_cast<BatchHolder<Cell> *>(&source);
        if (!typed)
            throw std::invalid_argument("grid batch belongs to a workload with a different cell type");
        sc::GridBatch<Cell> result = (*update)(typed->batch);
        return new BatchHolder<Cell>(source.workload, result);
    }

    void stats(stst_update_stats &s) override {
        std::memset(&s, 0, sizeof(s));
        s.n_processed_cells = update->get_n_processed_cells();
        s.walltime = update->get_walltime();
        s.kernel_runtime = update->get_kernel_runtime();
        s.n_launches = update->get_n_launches();
        auto const &plan = update->get_last_plan();
        s.fused_iterations = plan.fused_iterations;
        s.tile_h = plan.tile_h;
        s.tile_w = plan.tile_w;
        s.block_x = plan.block_x;
        s.block_y = plan.block_y;
        s.use_tma = plan.use_tma ? 1u : 0u;
        s.smem_bytes = plan.smem_bytes;
        s.passthrough_planes = update->get_passthrough_planes();
        s.speculation_redos = update->get_n_speculation_redos();
        s.n_slabs = update->get_n_slabs();
    }
};

struct SlabBase {
    virtual ~SlabBase() = default;
    const char *workload = nullptr;
    std::vector<void *> ipc_mappings;
    virtual std::size_t cell_bytes() const = 0;
    virtual void info(stst_slab_info &out) = 0;
    virtual void *device_base() = 0;
    virtual int device() const = 0;
    virtual void attach(int side, void *mapped, std::size_t lo, std::size_t hi) = 0;
    virtual void detach() = 0;
    virtual void use_nccl(void *comm, int up_rank, int down_rank) = 0;
    virtual void upload(const void *cells, std::size_t first_row, std::size_t n_rows) = 0;
    virtual void download(void *cells, std::size_t first_row, std::size_t n_rows) = 0;
    virtual void exchange() = 0;
    virtual void max_abs(const stst_field_extent *extents, std::size_t n, double *out) = 0;
    virtual std::size_t field_bytes(std::size_t field) const = 0;
    virtual void download_field(std::size_t field, void *host, std::size_t first_row,
                                std::size_t n_rows) = 0;
    virtual void update(const stst_update_params &p) = 0;
    virtual void synchronize() = 0;
    virtual void record(void *event) = 0;
    virtual void copy_from(SlabBase &other) = 0;
    virtual sc::internal::PlaneSet current_planes() = 0;
    virtual std::size_t ghost() const = 0;
    virtual bool enable_speculation(bool on) = 0;
    virtual void backup() = 0;
    virtual void restore() = 0;
    virtual unsigned take_violations() = 0;
    virtual void drop_passthrough(unsigned planes) = 0;
};

template <typename F, typename ParamBlock> struct SlabHolder final : SlabBase {
    using Slab = sc::internal::SlabUpdate<F>;
    using Cell = typename F::Cell;
    std::unique_ptr<Slab> slab;

    SlabHolder(const char *name, typename Slab::Config const &cfg)
        : slab(std::make_unique<Slab>(cfg)) {
        workload = name;
    }
    ~SlabHolder() override {
        slab.reset();
        for (void *m : ipc_mappings)
            (void)stst_ipc_close_mem_handle(m);
    }
    std::size_t cell_bytes() const override { return sizeof(Cell); }
    void info(stst_slab_info &out) override {
        std::memset(&out, 0, sizeof(out));
        auto const &cfg = slab->get_config();
        auto const &plan = slab->get_active_plan();
        out.grid_rows = cfg.grid_rows;
        out.grid_cols = cfg.grid_cols;
        out.row_lo = cfg.row_lo;
        out.row_hi = cfg.row_hi;
        out.ghost_rows = slab->ghost_rows();
        out.device_bytes = slab->device_bytes();
        out.n_launches = slab->get_n_launches();
        out.epoch = slab->get_epoch();
        out.device = cfg.device;
        out.fused_iterations = plan.fused_iterations;
        out.tile_h = plan.tile_h;
        out.tile_w = plan.tile_w;
        out.block_x = plan.block_x;
        out.block_y = plan.block_y;
        out.use_tma = plan.use_tma ? 1u : 0u;
        out.overlap = cfg.overlap ? 1u : 0u;
        out.smem_bytes = plan.smem_bytes;
        out.passthrough_planes = slab->passthrough_planes();
    }
    void *device_base() override { return slab->device_base(); }
    int device() const override { return slab->get_config().device; }
    void attach(int side, void *mapped, std::size_t lo, std::size_t hi) override {
        slab->attach(side == 0 ? sc::internal::SlabSide::up : sc::internal::SlabSide::down, mapped,
                     lo, hi);
    }
    void use_nccl(void *comm, int up_rank, int down_rank) override {
        slab->use_nccl(comm, up_rank, down_rank);
    }
    void detach() override {
        slab->detach();
        for (void *m : ipc_mappings)
            (void)stst_ipc_close_mem_handle(m);
        ipc_mappings.clear();
    }
    void upload(const void *cells, std::size_t first_row, std::size_t n_rows) override {
        slab->upload_rows(static_cast<const Cell *>(cells), first_row, n_rows);
    }
    void download(void *cells, std::size_t first_row, std::size_t n_rows) override {
        slab->download_rows(static_cast<Cell *>(cells), first_row, n_rows);
    }
    void exchange() override { slab->exchange_halos(); }
    void max_abs(const stst_field_extent *extents, std::size_t n, double *out) override {
        const std::vector<double> result = slab->max_abs(field_extents(extents, n));
        std::copy(result.begin(), result.end(), out);
    }
    std::size_t field_bytes(std::size_t field) const override {
        return sc::Grid<Cell>::plane_element_bytes(field);
    }
    void download_field(std::size_t field, void *host, std::size_t first_row,
                        std::size_t n_rows) override {
        slab->download_plane_rows(field, host, first_row, n_rows);
    }
    void update(const stst_update_params &p) override {
        auto params = UpdateHolder<F, ParamBlock>::convert(p);
        slab->run(params.transition_function, params.halo_value, params.iteration_offset,
                  params.n_iterations);
        if (params.blocking)
            slab->synchronize();
    }
    void synchronize() override { slab->synchronize(); }
    void record(void *event) override { slab->record(event); }
    sc::internal::PlaneSet current_planes() override { return slab->current_planes(); }
    std::size_t ghost() const override { return slab->ghost_rows(); }
    void copy_from(SlabBase &other) override {
        stst_slab_info mine, theirs;
        info(mine);
        other.info(theirs);
        if (other.cell_bytes() != cell_bytes() || theirs.grid_rows != mine.grid_rows ||
            theirs.grid_cols != mine.grid_cols || theirs.row_lo != mine.row_lo ||
            theirs.row_hi != mine.row_hi)
            throw std::range_error("The source slab has not the same rows, columns or cell type");
        if (other.device() != device())
            throw std::invalid_argument("the two slabs live on different devices");
        other.synchronize(); // its current generation must be complete before it is read
        slab->copy_owned_rows_from(other.current_planes(), other.ghost());
    }
    bool enable_speculation(bool on) override { return slab->enable_speculation(on); }
    void backup() override { slab->backup(); }
    void restore() override { slab->restore(); }
    unsigned take_violations() override { return slab->take_violations(); }
    void drop_passthrough(unsigned planes) override { slab->drop_passthrough(planes); }
};

struct WorkloadEntry {
    const char *name;
    stst_workload_info info;
    GridBase *(*make_grid)(const char *, std::size_t, std::size_t, int);
    BatchBase *(*make_batch)(const char *, std::size_t, std::size_t, std::size_t, int);
    UpdateBase *(*make_update)(const char *, const stst_update_params &);
    SlabBase *(*make_slab)(const char *, std::size_t, std::size_t, std::size_t, std::size_t, int,
                           unsigned, unsigned, bool);
};

template <typename F, typename ParamBlock> WorkloadEntry make_entry(const char *name) {
    using Cell = typename F::Cell;
    WorkloadEntry e{};
    e.name = name;
    e.info.cell_bytes = sizeof(Cell);
    e.info.params_bytes = sizeof(ParamBlock);
    e.info.n_planes = sc::internal::CellLayout<Cell>::n_planes;
    e.info.stencil_radius = F::stencil_radius;
    e.info.n_subiterations = F::n_subiterations;
    e.info.bytes_per_cell_iteration = 2 * sizeof(Cell) * F::n_subiterations;
    e.make_grid = [](const char *n, std::size_t r, std::size_t c, int device) -> GridBase * {
        if (device < 0)
            device = sc::internal::default_device_ordinal();
        return new GridHolder<Cell>(n, sc::Grid<Cell>(r, c, device));
    };
    e.make_batch = [](const char *n, std::size_t members, std::size_t r, std::size_t c,
                      int device) -> BatchBase * {
        return new BatchHolder<Cell>(n, sc::GridBatch<Cell>(members, r, c, device));
    };
    e.make_update = [](const char *n, const stst_update_params &p) -> UpdateBase * {
        return new UpdateHolder<F, ParamBlock>(n, p);
    };
    e.make_slab = [](const char *n, std::size_t grid_rows, std::size_t grid_cols, std::size_t row_lo,
                     std::size_t row_hi, int device, unsigned fused, unsigned tile_rows,
                     bool overlap) -> SlabBase * {
        if (device < 0)
            device = sc::internal::default_device_ordinal();
        typename sc::internal::SlabUpdate<F>::Config cfg{grid_rows, grid_cols, row_lo, row_hi,
                                                          device,    fused,     tile_rows, overlap};
        return new SlabHolder<F, ParamBlock>(n, cfg);
    };
    return e;
}

} // namespace stst_model
