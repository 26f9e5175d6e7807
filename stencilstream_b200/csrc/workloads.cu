/*
 * libstst_workloads — the C ABI of include/stst_workloads.h over the type-erased object model of
 * workloads/model.hpp. The backend itself is instantiated for the individual transition functions in
 * workloads_<group>.cu (one translation unit per group, compiled in parallel).
 *
 * All compute goes through stencil::cuda::StencilUpdate -> fused_sweep_kernel; nothing in this
 * library computes cells on the host.
 */
#include "workloads/model.hpp"

namespace stst_model {
void register_light(std::vector<WorkloadEntry> &entries);
void register_hotspot(std::vector<WorkloadEntry> &entries);
void register_fdtd(std::vector<WorkloadEntry> &entries);
void register_convection(std::vector<WorkloadEntry> &entries);
void register_kat(std::vector<WorkloadEntry> &entries);
} // namespace stst_model

using namespace stst_model;

namespace {

const std::vector<WorkloadEntry> &registry() {
    static const std::vector<WorkloadEntry> entries = [] {
        std::vector<WorkloadEntry> list;
        register_light(list);      // conway, jacobi5, jacobi9, jacobi_r2, jacobi_r3
        register_hotspot(list);    // hotspot
        register_fdtd(list);       // fdtd
        register_convection(list); // convection_pt, convection_thermal
        register_kat(list);        // kat, kat_r2
        return list;
    }();
    return entries;
}

const WorkloadEntry *find(const char *name) {
    if (!name)
        return nullptr;
    for (auto const &e : registry())
        if (std::strcmp(e.name, name) == 0)
            return &e;
    return nullptr;
}

template <typename Fn> int guarded(Fn &&fn) {
    try {
        return fn();
    } catch (std::range_error const &e) {
        return report(STST_ERR_RANGE, e.what());
    } catch (std::invalid_argument const &e) {
        return report(STST_ERR_INVALID_ARGUMENT, e.what());
    } catch (std::exception const &e) {
        return report(STST_ERR_RUNTIME, e.what());
    } catch (...) {
        return report(STST_ERR_RUNTIME, "unknown exception");
    }
}

} // namespace

struct stst_grid {
    std::unique_ptr<GridBase> impl;
};
struct stst_update {
    std::unique_ptr<UpdateBase> impl;
};
struct stst_slab {
    std::unique_ptr<SlabBase> impl;
};
struct stst_batch {
    std::unique_ptr<BatchBase> impl;
};

#define STST_EXPORT extern "C" __attribute__((visibility("default")))

STST_EXPORT int stst_workloads_abi_version(void) { return STST_WORKLOADS_ABI_VERSION; }

STST_EXPORT const char *stst_workloads_last_error(void) { return g_error.c_str(); }

STST_EXPORT int stst_workload_count(void) { return int(registry().size()); }

STST_EXPORT const char *stst_workload_name(int index) {
    if (index < 0 || index >= int(registry().size()))
        return nullptr;
    return registry()[index].name;
}

STST_EXPORT int stst_workload_get_info(const char *workload, stst_workload_info *info) {
    const WorkloadEntry *e = find(workload);
    if (!e)
        return report(STST_ERR_UNKNOWN_WORKLOAD, std::string("unknown workload: ") +
                                                     (workload ? workload : "(null)"));
    if (!info)
        return report(STST_ERR_INVALID_ARGUMENT, "info is null");
    *info = e->info;
    return STST_OK;
}

STST_EXPORT int stst_grid_create(const char *workload, size_t rows, size_t cols, int device,
                                 stst_grid **grid) {
    const WorkloadEntry *e = find(workload);
    if (!e)
        return report(STST_ERR_UNKNOWN_WORKLOAD, std::string("unknown workload: ") +
                                                     (workload ? workload : "(null)"));
    if (!grid)
        return report(STST_ERR_INVALID_ARGUMENT, "grid is null");
    return guarded([&] {
        *grid = new stst_grid{std::unique_ptr<GridBase>(e->make_grid(e->name, rows, cols, device))};
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_share(stst_grid *grid, stst_grid **other) {
    if (!grid || !other)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *other = new stst_grid{std::unique_ptr<GridBase>(grid->impl->share())};
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_make_similar(stst_grid *grid, stst_grid **other) {
    if (!grid || !other)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *other = new stst_grid{std::unique_ptr<GridBase>(grid->impl->make_similar())};
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_destroy(stst_grid *grid) {
    delete grid;
    return STST_OK;
}

STST_EXPORT int stst_grid_shape(const stst_grid *grid, size_t *rows, size_t *cols) {
    if (!grid || !rows || !cols)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    *rows = grid->impl->rows();
    *cols = grid->impl->cols();
    return STST_OK;
}

STST_EXPORT int stst_grid_copy_from_host(stst_grid *grid, const void *cells, size_t bytes) {
    if (!grid || (!cells && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    if (bytes != grid->impl->rows() * grid->impl->cols() * grid->impl->cell_bytes())
        return report(STST_ERR_RANGE, "The target buffer has not the same size as the grid");
    return guarded([&] {
        grid->impl->copy_from_host(cells);
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_copy_to_host(stst_grid *grid, void *cells, size_t bytes) {
    if (!grid || (!cells && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    if (bytes != grid->impl->rows() * grid->impl->cols() * grid->impl->cell_bytes())
        return report(STST_ERR_RANGE, "The target buffer has not the same size as the grid");
    return guarded([&] {
        grid->impl->copy_to_host(cells);
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_sync_to_device(stst_grid *grid) {
    if (!grid)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        grid->impl->sync_to_device();
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_host_accessor(stst_grid *grid, int mode, void **cells) {
    if (!grid || !cells || mode < 0 || mode > 2)
        return report(STST_ERR_INVALID_ARGUMENT, "bad argument");
    return guarded([&] {
        *cells = grid->impl->host_accessor(mode);
        return STST_OK;
    });
}

STST_EXPORT int stst_grid_host_image_is_pinned(stst_grid *grid, int *pinned) {
    if (!grid || !pinned)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    *pinned = grid->impl->host_pinned() ? 1 : 0;
    return STST_OK;
}

STST_EXPORT int stst_grid_max_abs(stst_grid *grid, const stst_field_extent *extents, size_t n,
                                  double *out) {
    if (!grid || (n != 0 && (!extents || !out)))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        grid->impl->max_abs(extents, n, out);
        return STST_OK;
    });
}

namespace {
int grid_copy_field(stst_grid *grid, size_t field, void *host, size_t bytes, bool to_device) {
    if (!grid || (!host && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        const size_t want = grid->impl->rows() * grid->impl->cols() * grid->impl->field_bytes(field);
        if (bytes != want)
            return report(STST_ERR_RANGE, "The target buffer has not the same size as the field");
        grid->impl->copy_field(field, host, to_device);
        return STST_OK;
    });
}
} // namespace

STST_EXPORT int stst_grid_copy_field_to_host(stst_grid *grid, size_t field, void *values,
                                             size_t bytes) {
    return grid_copy_field(grid, field, values, bytes, false);
}

STST_EXPORT int stst_grid_copy_field_from_host(stst_grid *grid, size_t field, const void *values,
                                               size_t bytes) {
    return grid_copy_field(grid, field, const_cast<void *>(values), bytes, true);
}

STST_EXPORT int stst_update_create(const char *workload, const stst_update_params *params,
                                   stst_update **update) {
    const WorkloadEntry *e = find(workload);
    if (!e)
        return report(STST_ERR_UNKNOWN_WORKLOAD, std::string("unknown workload: ") +
                                                     (workload ? workload : "(null)"));
    if (!params || !update)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *update = new stst_update{std::unique_ptr<UpdateBase>(e->make_update(e->name, *params))};
        return STST_OK;
    });
}

STST_EXPORT int stst_update_set_params(stst_update *update, const stst_update_params *params) {
    if (!update || !params)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        update->impl->set_params(*params);
        return STST_OK;
    });
}

STST_EXPORT int stst_update_apply(stst_update *update, stst_grid *source, stst_grid **result) {
    if (!update || !source || !result)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *result = new stst_grid{std::unique_ptr<GridBase>(update->impl->apply(*source->impl))};
        return STST_OK;
    });
}

STST_EXPORT int stst_update_get_stats(stst_update *update, stst_update_stats *stats) {
    if (!update || !stats)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        update->impl->stats(*stats);
        return STST_OK;
    });
}

STST_EXPORT int stst_update_destroy(stst_update *update) {
    delete update;
    return STST_OK;
}

// ---- grid batches --------------------------------------------------------------------------------------

STST_EXPORT int stst_batch_create(const char *workload, size_t members, size_t rows, size_t cols,
                                  int device, stst_batch **batch) {
    const WorkloadEntry *e = find(workload);
    if (!e)
        return report(STST_ERR_UNKNOWN_WORKLOAD, std::string("unknown workload: ") +
                                                     (workload ? workload : "(null)"));
    if (!batch)
        return report(STST_ERR_INVALID_ARGUMENT, "batch is null");
    return guarded([&] {
        *batch = new stst_batch{
            std::unique_ptr<BatchBase>(e->make_batch(e->name, members, rows, cols, device))};
        return STST_OK;
    });
}

STST_EXPORT int stst_batch_destroy(stst_batch *batch) {
    delete batch;
    return STST_OK;
}

STST_EXPORT int stst_batch_shape(const stst_batch *batch, size_t *members, size_t *rows,
                                 size_t *cols) {
    if (!batch || !members || !rows || !cols)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    *members = batch->impl->members();
    *rows = batch->impl->rows();
    *cols = batch->impl->cols();
    return STST_OK;
}

STST_EXPORT int stst_batch_copy_from_host(stst_batch *batch, size_t first_member, size_t n_members,
                                          const void *cells, size_t bytes) {
    if (!batch || (!cells && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        batch->impl->copy(first_member, n_members, const_cast<void *>(cells), bytes, true);
        return STST_OK;
    });
}

STST_EXPORT int stst_batch_copy_to_host(stst_batch *batch, size_t first_member, size_t n_members,
                                        void *cells, size_t bytes) {
    if (!batch || (!cells && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        batch->impl->copy(first_member, n_members, cells, bytes, false);
        return STST_OK;
    });
}

STST_EXPORT int stst_batch_max_abs(stst_batch *batch, size_t member, const stst_field_extent *extents,
                                   size_t n, double *out) {
    if (!batch || (n != 0 && (!extents || !out)))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        batch->impl->max_abs(member, extents, n, out);
        return STST_OK;
    });
}

STST_EXPORT int stst_batch_copy_field_to_host(stst_batch *batch, size_t field, void *values,
                                              size_t bytes) {
    if (!batch || (!values && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        const size_t want = batch->impl->members() * batch->impl->rows() * batch->impl->cols() *
                            batch->impl->field_bytes(field);
        if (bytes != want)
            return report(STST_ERR_RANGE, "The target buffer has not the same size as the field");
        batch->impl->copy_field_to_host(field, values);
        return STST_OK;
    });
}

STST_EXPORT int stst_update_apply_batch(stst_update *update, stst_batch *source,
                                        stst_batch **result) {
    if (!update || !source || !result)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *result = new stst_batch{std::unique_ptr<BatchBase>(update->impl->apply_batch(*source->impl))};
        return STST_OK;
    });
}

// ---- row slabs ---------------------------------------------------------------------------------------

STST_EXPORT int stst_slab_create(const char *workload, size_t grid_rows, size_t grid_cols,
                                 size_t row_lo, size_t row_hi, int device,
                                 unsigned fused_iterations, unsigned tile_rows, int overlap,
                                 stst_slab **slab) {
    const WorkloadEntry *e = find(workload);
    if (!e)
        return report(STST_ERR_UNKNOWN_WORKLOAD, std::string("unknown workload: ") +
                                                     (workload ? workload : "(null)"));
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "slab is null");
    if (row_hi <= row_lo || row_hi > grid_rows || grid_cols == 0)
        return report(STST_ERR_INVALID_ARGUMENT, "illegal slab row range");
    return guarded([&] {
        *slab = new stst_slab{std::unique_ptr<SlabBase>(
            e->make_slab(e->name, grid_rows, grid_cols, row_lo, row_hi, device, fused_iterations,
                         tile_rows, overlap != 0))};
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_destroy(stst_slab *slab) {
    delete slab;
    return STST_OK;
}

STST_EXPORT int stst_slab_get_info(stst_slab *slab, stst_slab_info *info) {
    if (!slab || !info)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->info(*info);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_get_ipc_handle(stst_slab *slab, unsigned char handle[64]) {
    if (!slab || !handle)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        sc::internal::check(stst_ipc_get_mem_handle(slab->impl->device_base(), handle),
                            "stst_ipc_get_mem_handle");
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_attach_ipc(stst_slab *slab, int side, const unsigned char handle[64],
                                     size_t peer_row_lo, size_t peer_row_hi) {
    if (!slab || !handle || side < 0 || side > 1)
        return report(STST_ERR_INVALID_ARGUMENT, "bad argument");
    return guarded([&] {
        sc::internal::check(stst_set_device(slab->impl->device()), "stst_set_device");
        void *mapped = nullptr;
        sc::internal::check(stst_ipc_open_mem_handle(handle, &mapped), "stst_ipc_open_mem_handle");
        slab->impl->ipc_mappings.push_back(mapped);
        slab->impl->attach(side, mapped, peer_row_lo, peer_row_hi);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_attach_local(stst_slab *slab, int side, stst_slab *peer) {
    if (!slab || !peer || side < 0 || side > 1)
        return report(STST_ERR_INVALID_ARGUMENT, "bad argument");
    return guarded([&] {
        stst_slab_info theirs;
        peer->impl->info(theirs);
        if (peer->impl->device() != slab->impl->device()) {
            int can = 0;
            sc::internal::check(stst_peer_can_access(slab->impl->device(), peer->impl->device(), &can),
                                "stst_peer_can_access");
            if (!can)
                throw std::runtime_error("the two slabs' devices cannot access each other");
            sc::internal::check(stst_peer_enable(slab->impl->device(), peer->impl->device()),
                                "stst_peer_enable");
        }
        slab->impl->attach(side, peer->impl->device_base(), theirs.row_lo, theirs.row_hi);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_use_nccl(stst_slab *slab, void *nccl_comm, int up_rank, int down_rank) {
    if (!slab || !nccl_comm)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->use_nccl(nccl_comm, up_rank, down_rank);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_detach(stst_slab *slab) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->detach();
        return STST_OK;
    });
}

namespace {
int slab_copy_rows(stst_slab *slab, void *cells, size_t bytes, size_t first_row, size_t n_rows,
                   bool whole, bool to_device) {
    if (!slab || (!cells && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        stst_slab_info info;
        slab->impl->info(info);
        const size_t owned = info.row_hi - info.row_lo;
        if (whole) {
            first_row = 0;
            n_rows = owned;
        }
        if (first_row > owned || n_rows > owned - first_row ||
            bytes != n_rows * info.grid_cols * slab->impl->cell_bytes())
            return report(STST_ERR_RANGE, "The target buffer has not the same size as the slab rows");
        if (to_device)
            slab->impl->upload(cells, first_row, n_rows);
        else
            slab->impl->download(cells, first_row, n_rows);
        return STST_OK;
    });
}
} // namespace

STST_EXPORT int stst_slab_copy_from_host(stst_slab *slab, const void *cells, size_t bytes) {
    return slab_copy_rows(slab, const_cast<void *>(cells), bytes, 0, 0, true, true);
}

STST_EXPORT int stst_slab_copy_to_host(stst_slab *slab, void *cells, size_t bytes) {
    return slab_copy_rows(slab, cells, bytes, 0, 0, true, false);
}

STST_EXPORT int stst_slab_copy_rows_from_host(stst_slab *slab, size_t first_row, size_t n_rows,
                                              const void *cells, size_t bytes) {
    return slab_copy_rows(slab, const_cast<void *>(cells), bytes, first_row, n_rows, false, true);
}

STST_EXPORT int stst_slab_copy_rows_to_host(stst_slab *slab, size_t first_row, size_t n_rows,
                                            void *cells, size_t bytes) {
    return slab_copy_rows(slab, cells, bytes, first_row, n_rows, false, false);
}

STST_EXPORT int stst_slab_exchange_halos(stst_slab *slab) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->exchange();
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_max_abs(stst_slab *slab, const stst_field_extent *extents, size_t n,
                                  double *out) {
    if (!slab || (n != 0 && (!extents || !out)))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->max_abs(extents, n, out);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_copy_field_rows_to_host(stst_slab *slab, size_t field, size_t first_row,
                                                  size_t n_rows, void *values, size_t bytes) {
    if (!slab || (!values && bytes != 0))
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        stst_slab_info info;
        slab->impl->info(info);
        const size_t owned = info.row_hi - info.row_lo;
        if (first_row > owned || n_rows > owned - first_row ||
            bytes != n_rows * info.grid_cols * slab->impl->field_bytes(field))
            return report(STST_ERR_RANGE, "The target buffer has not the same size as the field rows");
        slab->impl->download_field(field, values, first_row, n_rows);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_update(stst_slab *slab, const stst_update_params *params) {
    if (!slab || !params)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->update(*params);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_copy_from_slab(stst_slab *slab, stst_slab *source) {
    if (!slab || !source)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->copy_from(*source->impl);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_enable_speculation(stst_slab *slab, int enable, int *enabled) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        const bool on = slab->impl->enable_speculation(enable != 0);
        if (enabled)
            *enabled = on ? 1 : 0;
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_backup(stst_slab *slab) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->backup();
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_restore(stst_slab *slab) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->restore();
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_take_violations(stst_slab *slab, unsigned *planes) {
    if (!slab || !planes)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        *planes = slab->impl->take_violations();
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_drop_passthrough(stst_slab *slab, unsigned planes) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->drop_passthrough(planes);
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_synchronize(stst_slab *slab) {
    if (!slab)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->synchronize();
        return STST_OK;
    });
}

STST_EXPORT int stst_slab_record_event(stst_slab *slab, void *event) {
    if (!slab || !event)
        return report(STST_ERR_INVALID_ARGUMENT, "null argument");
    return guarded([&] {
        slab->impl->record(event);
        return STST_OK;
    });
}
