/*
 * stst_workloads.h — C ABI of libstst_workloads.so: the StencilStream-B200 generation loop for a
 * fixed set of transition functions, reachable without a C++ compiler (ctypes, cgo, JNI, ...).
 *
 * The reference's boundary for this path is a C++ template API, not an ABI: user code instantiates
 * `stencil::cuda::Grid<Cell>` (reference StencilStream/cuda/Grid.hpp:50-188) and
 * `stencil::cuda::StencilUpdate<F, split>` (reference StencilStream/cuda/StencilUpdate.hpp:41-445)
 * with its own functor. The header-only backend in stencilstream_b200/include/StencilStream keeps
 * that template API. This library instantiates it for the reference's example functors and its
 * self-checking test functor, and exposes the *same object model* over C:
 *
 *   stst_grid_*        <- cuda::Grid<Cell>: ctor (Grid.hpp:66-74), copy_from_buffer / copy_to_buffer
 *                         (:109-134; size mismatch -> STST_ERR_RANGE where the reference throws
 *                         std::range_error), get_grid_height/width (:158-163), make_similar (:176)
 *   stst_update_*      <- cuda::StencilUpdate<F>: ctor from Params (StencilUpdate.hpp:54-111),
 *                         get_params() mutation (:152), operator() (:123-144),
 *                         get_n_processed_cells / get_walltime / get_kernel_runtime (:160-198)
 *
 * Cells cross this boundary as dense row-major arrays of the C structs below ("array of structs",
 * exactly the memory image of the reference's `sycl::buffer<Cell, 2>`); transition-function
 * parameters cross as the stst_*_params structs below.
 *
 * Every function returns STST_OK or a negative STST_ERR_* code; stst_workloads_last_error() returns
 * the message of the last failure on the calling thread. There is no CPU fallback: without a CUDA
 * device, grid uploads and updates fail with STST_ERR_RUNTIME.
 */
#ifndef STST_WORKLOADS_H
#define STST_WORKLOADS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STST_WORKLOADS_ABI_VERSION 3

#define STST_OK 0
#define STST_ERR_UNKNOWN_WORKLOAD (-1)
#define STST_ERR_INVALID_ARGUMENT (-2)
#define STST_ERR_RANGE (-3)   /* std::range_error in the C++ API */
#define STST_ERR_RUNTIME (-4) /* CUDA / runtime failure */

/* ---- cell types (array-of-structs images) ------------------------------------------------------ */

/* "conway": Cell = bool (1 byte, 0 or 1).  reference examples/conway/conway.cpp:35-56            */
/* "jacobi5", "jacobi9", "jacobi_r2", "jacobi_r3": Cell = float.  examples/jacobi/kernels.hpp     */

typedef struct stst_hotspot_cell { /* reference examples/hotspot/hotspot.cpp:57-62 */
    float temp;
    float power;
} stst_hotspot_cell;

typedef struct stst_fdtd_cell { /* reference examples/fdtd/src/material/CoefResolver.hpp:27-29 */
    float ex, ey, hz, hz_sum;
    float ca, cb, da, db;
} stst_fdtd_cell;

typedef struct stst_convection_cell { /* reference examples/convection/convection.cpp:36-40 */
    double T, Pt, Vx, Vy;
    double tau_xx, tau_yy, sigma_xy;
    double dVxd_tau, dVyd_tau;
    double ErrV, ErrP;
} stst_convection_cell;

typedef struct stst_kat_cell { /* reference tests/TransFuncs.hpp:36-47 */
    int32_t r, c, i_iteration, i_subiteration;
    int32_t status; /* 0 = Normal, 1 = Invalid, 2 = Halo */
} stst_kat_cell;

/* ---- transition-function parameters ------------------------------------------------------------- */

typedef struct stst_conway_params {
    int32_t reserved; /* the rule has no runtime parameters */
} stst_conway_params;

typedef struct stst_jacobi5_params { /* Jacobi5General::coef, examples/jacobi/kernels.hpp:265-271 */
    float coef[5];                   /* north, west, south, east, centre */
} stst_jacobi5_params;

typedef struct stst_jacobi9_params { /* Jacobi9General::coef, examples/jacobi/kernels.hpp:303-317 */
    float coef[3][3];
} stst_jacobi9_params;

typedef struct stst_jacobi_star_params { /* B200 addition: radius-2/3 star stencils (no reference functor) */
    float centre;
    float arm[3]; /* weight of the 4 cells at distance 1, 2, 3 (radius-2 variant ignores arm[2]) */
} stst_jacobi_star_params;

typedef struct stst_hotspot_params { /* HotspotKernel members, examples/hotspot/hotspot.cpp:67 */
    float Rx_1, Ry_1, Rz_1, Cap_1;
} stst_hotspot_params;

typedef struct stst_fdtd_params { /* Kernel<CoefResolver> members, examples/fdtd/src/Kernel.hpp:130-140 */
    float dt, t_0, tau, omega;
    uint64_t cutoff_iteration;
    uint64_t detect_iteration;
    float source_radius_squared;
    float source_r, source_c, source_distance_bound;
    float double_center_rc;
} stst_fdtd_params;

typedef struct stst_convection_pt_params { /* PseudoTransientKernel, examples/convection/convection.cpp:82-93 */
    uint64_t nx, ny;
    double roh0_g_alpha;
    double delta_eta_delta_T;
    double eta0;
    double deltaT;
    double dx, dy;
    double delta_tau_iter;
    double beta;
    double rho;
    double dampX, dampY;
    double DcT;
} stst_convection_pt_params;

typedef struct stst_convection_thermal_params { /* ThermalSolverKernel, convection.cpp:191-193 */
    uint64_t nx, ny;
    double dx, dy, dt;
    double DcT;
} stst_convection_thermal_params;

typedef struct stst_kat_params {
    int32_t reserved; /* FPGATransFunc<1> has no runtime parameters (tests/TransFuncs.hpp:55-104) */
} stst_kat_params;

/* ---- registry --------------------------------------------------------------------------------- */

typedef struct stst_workload_info {
    size_t cell_bytes;         /* sizeof(Cell)                                    */
    size_t params_bytes;       /* sizeof(stst_<name>_params)                      */
    size_t n_planes;           /* device planes per cell                          */
    size_t stencil_radius;     /* F::stencil_radius                               */
    size_t n_subiterations;    /* F::n_subiterations                              */
    size_t bytes_per_cell_iteration; /* 2 * sizeof(Cell) * n_subiterations: the reference's own
                                        traffic model, scripts/benchmark-common.jl:150-151 */
} stst_workload_info;

int stst_workloads_abi_version(void);
const char *stst_workloads_last_error(void);
int stst_workload_count(void);
const char *stst_workload_name(int index);
int stst_workload_get_info(const char *workload, stst_workload_info *info);

/* ---- grids ---------------------------------------------------------------------------------------- */

typedef struct stst_grid stst_grid;

/* New, uninitialised grid of rows x cols cells of the workload's cell type. device < 0: default. */
int stst_grid_create(const char *workload, size_t rows, size_t cols, int device, stst_grid **grid);
/* A second handle to the same cells (Grid copy constructor). */
int stst_grid_share(stst_grid *grid, stst_grid **other);
int stst_grid_make_similar(stst_grid *grid, stst_grid **other);
int stst_grid_destroy(stst_grid *grid);
int stst_grid_shape(const stst_grid *grid, size_t *rows, size_t *cols);
/* copy_from_buffer / copy_to_buffer: `bytes` must equal rows*cols*cell_bytes, else STST_ERR_RANGE. */
int stst_grid_copy_from_host(stst_grid *grid, const void *cells, size_t bytes);
int stst_grid_copy_to_host(stst_grid *grid, void *cells, size_t bytes);
/* Force the device copy to be current (uploads a pending host image); for resident-data timing. */
int stst_grid_sync_to_device(stst_grid *grid);
/*
 * GridAccessor<mode> (Grid.hpp:145-153): waits for pending device work, brings the pinned host image
 * up to date and returns a pointer to it (rows*cols cells, row-major), valid while any handle to the
 * cells exists. mode: 0 = read, 1 = write, 2 = read_write; writable modes mark the device copy stale,
 * so the next update uploads the image first.
 */
int stst_grid_host_accessor(stst_grid *grid, int mode, void **cells);
/* Whether that host image exists and is pinned (boxes cap pinnable memory; a pageable image is moved
 * through the runtime's staged pipeline, stst_memcpy_2d_staged in stst_rt.h). */
int stst_grid_host_image_is_pinned(stst_grid *grid, int *pinned);

/* ---- per-field operations (B200 extensions) ----------------------------------------------------
 *
 * The reference's applications compute max-norms and dump single fields on the host, through a
 * GridAccessor that first migrates the whole array-of-structs grid (examples/convection/
 * convection.cpp:412-438 and :460-477, examples/fdtd/src/fdtd.cpp:114-166). Grids are stored one
 * plane per field here, so both run on the planes involved only.
 * `field` is the index into the cell struct's members in declaration order (0 for scalar cells). */

typedef struct stst_field_extent {
    size_t field;
    size_t rows, cols; /* the first `rows` rows and `cols` columns of the grid */
} stst_field_extent;

/* out[q] = max |cell.field_q| over extents[q] (-inf for an empty extent); one device pass for up to
 * 8 extents. Comparison as in the reference loop: `abs(v) > max`, i.e. NaNs are never selected. */
int stst_grid_max_abs(stst_grid *grid, const stst_field_extent *extents, size_t n, double *out);
/* Dense rows x cols array of ONE field; bytes must equal rows*cols*sizeof(field), else STST_ERR_RANGE. */
int stst_grid_copy_field_to_host(stst_grid *grid, size_t field, void *values, size_t bytes);
int stst_grid_copy_field_from_host(stst_grid *grid, size_t field, const void *values, size_t bytes);

/* ---- updaters ------------------------------------------------------------------------------------ */

typedef struct stst_update stst_update;

typedef struct stst_update_params {
    const void *transition_function; /* -> stst_<workload>_params */
    size_t transition_function_bytes;
    const void *halo_value; /* -> one cell; NULL = value-initialised cell */
    size_t halo_value_bytes;
    size_t iteration_offset;
    size_t n_iterations;
    int blocking;
    int profiling;
    int cuda_device;           /* < 0: the source grid's device */
    unsigned fused_iterations; /* 0 = automatic */
    unsigned tile_rows;        /* 0 = automatic */
    /* CUDA devices to spread ONE update over (row slabs, one per entry; an ordinal may repeat);
     * n_cuda_devices == 0: the environment variable STST_DEVICES, else the source grid's device.
     * Source and result grids stay single-device grids (Params::cuda_devices of the C++ API). */
    const int *cuda_devices;
    size_t n_cuda_devices;
} stst_update_params;

typedef struct stst_update_stats {
    size_t n_processed_cells;
    double walltime;       /* seconds, host side                              */
    double kernel_runtime; /* seconds, device side (profiling only, else 0)   */
    size_t n_launches;     /* fused kernel launches so far                    */
    unsigned fused_iterations, tile_h, tile_w, block_x, block_y, use_tma;
    size_t smem_bytes;
    /* speculative plane pass-through: planes (bit i = field i) the tile sweeps currently leave in
     * place instead of copying them, and how many updates had to be repeated because one changed */
    unsigned passthrough_planes;
    size_t speculation_redos;
    size_t n_slabs; /* row slabs (GPUs) the most recent update ran on; 1 = not sharded */
} stst_update_stats;

int stst_update_create(const char *workload, const stst_update_params *params, stst_update **update);
/* Equivalent of mutating get_params(): takes effect at the next stst_update_apply. */
int stst_update_set_params(stst_update *update, const stst_update_params *params);
/* operator(): *result is a new grid handle owned by the caller; `source` is not modified. */
int stst_update_apply(stst_update *update, stst_grid *source, stst_grid **result);
int stst_update_get_stats(stst_update *update, stst_update_stats *stats);
int stst_update_destroy(stst_update *update);

/* ---- grid batches (B200 extension) ---------------------------------------------------------------
 *
 * `members` independent grids of rows x cols cells of one workload on one device, advanced together:
 * stst_update_apply_batch applies the update to every member with one fused launch per pass, and
 * each member's result equals the stst_update_apply result of that member alone, bit for bit (cells
 * outside a member read as halo_value; members never see each other). Cells cross as dense arrays of
 * n_members x rows x cols cells, member-major. A batch runs on its own device: an update whose
 * cuda_devices lists more than one device fails with STST_ERR_INVALID_ARGUMENT for a batch, and
 * STST_DEVICES is ignored. At most 65535 members. */

typedef struct stst_batch stst_batch;

/* New, uninitialised batch. device < 0: default. */
int stst_batch_create(const char *workload, size_t members, size_t rows, size_t cols, int device,
                      stst_batch **batch);
int stst_batch_destroy(stst_batch *batch);
int stst_batch_shape(const stst_batch *batch, size_t *members, size_t *rows, size_t *cols);
/* Members [first_member, first_member + n_members): bytes must equal n_members*rows*cols*cell_bytes
 * and the range must lie inside the batch, else STST_ERR_RANGE. */
int stst_batch_copy_from_host(stst_batch *batch, size_t first_member, size_t n_members,
                              const void *cells, size_t bytes);
int stst_batch_copy_to_host(stst_batch *batch, size_t first_member, size_t n_members, void *cells,
                            size_t bytes);
/* stst_grid_max_abs of member `member` (extents member-local); a member out of range: STST_ERR_RANGE. */
int stst_batch_max_abs(stst_batch *batch, size_t member, const stst_field_extent *extents, size_t n,
                       double *out);
/* ONE field of every member: bytes must equal members*rows*cols*sizeof(field), else STST_ERR_RANGE. */
int stst_batch_copy_field_to_host(stst_batch *batch, size_t field, void *values, size_t bytes);
/* operator()(GridBatch&): *result is a new batch handle owned by the caller; `source` is not
 * modified. Statistics as for a grid: n_processed_cells grows by n_iterations*members*rows*cols,
 * n_launches by one per fused pass whatever the member count. */
int stst_update_apply_batch(stst_update *update, stst_batch *source, stst_batch **result);

/* ---- row slabs: the multi-GPU partitioner --------------------------------------------------------
 *
 * No counterpart in the reference (its cuda backend drives one device,
 * StencilStream/cuda/StencilUpdate.hpp:83): a grid of grid_rows x grid_cols cells is cut into
 * contiguous row slabs, one per GPU, each slab object owning rows [row_lo, row_hi) plus
 * k * n_subiterations * radius ghost rows per side. Every fused launch stores the rows its
 * neighbours need directly into their ghost rows over NVLink (peer/IPC-mapped memory) and the slabs
 * order themselves with stream-ordered flags, so a run needs no host synchronisation and no
 * collective. The result equals the single-grid update of the whole grid.
 *
 * Protocol, identical on every slab of a grid (one slab per process, or several in one process):
 *   create -> exchange handles (get_ipc_handle/attach_ipc across processes, attach_local within one)
 *   -> copy_from_host -> exchange_halos -> update ... update -> copy_to_host.
 * exchange_halos and update are collective in the sense that every slab must issue the same sequence.
 */

typedef struct stst_slab stst_slab;

typedef struct stst_slab_info {
    size_t grid_rows, grid_cols, row_lo, row_hi;
    size_t ghost_rows;   /* k * n_subiterations * radius                         */
    size_t device_bytes; /* size of the slab's single device allocation          */
    size_t n_launches;   /* fused kernel launches so far                         */
    size_t epoch;        /* passes so far (incl. the two an exchange_halos adds) */
    int device;
    unsigned fused_iterations, tile_h, tile_w, block_x, block_y, use_tma, overlap;
    size_t smem_bytes;
    unsigned passthrough_planes; /* planes the sweeps currently leave in place (see below) */
} stst_slab_info;

/* fused_iterations: upper bound for k (0 = automatic); all slabs of a grid must end up with the same
 * k (compare stst_slab_info.fused_iterations and re-create with the minimum if they differ).
 * overlap != 0: boundary rows first on a high-priority stream, interior concurrently. */
int stst_slab_create(const char *workload, size_t grid_rows, size_t grid_cols, size_t row_lo,
                     size_t row_hi, int device, unsigned fused_iterations, unsigned tile_rows,
                     int overlap, stst_slab **slab);
int stst_slab_destroy(stst_slab *slab);
int stst_slab_get_info(stst_slab *slab, stst_slab_info *info);
/* side: 0 = the slab above (lower row indices), 1 = the slab below. */
int stst_slab_get_ipc_handle(stst_slab *slab, unsigned char handle[64]);
int stst_slab_attach_ipc(stst_slab *slab, int side, const unsigned char handle[64],
                         size_t peer_row_lo, size_t peer_row_hi);
int stst_slab_attach_local(stst_slab *slab, int side, stst_slab *peer);
/* Alternative halo transport: grouped ncclSend/ncclRecv per pass instead of stores into mapped
 * neighbour memory (no attach needed). nccl_comm: a communicator from stst_nccl_comm_init_rank
 * (include/stst_rt.h) that spans the slabs' processes; up_rank/down_rank: the neighbours' ranks in it,
 * negative where the slab has no neighbour. Every slab of a grid must use the same transport. */
int stst_slab_use_nccl(stst_slab *slab, void *nccl_comm, int up_rank, int down_rank);
/* Wait for the slab's work, then forget both neighbours and unmap their memory. Every slab of a grid
 * detaches before any of them is destroyed (a neighbour may still be pushing halo rows into it). */
int stst_slab_detach(stst_slab *slab);
/* Owned rows only: bytes must equal (row_hi-row_lo)*grid_cols*cell_bytes, else STST_ERR_RANGE.
 * copy_from_host is asynchronous when `cells` is pinned (stst_malloc_host / stst_host_register). */
int stst_slab_copy_from_host(stst_slab *slab, const void *cells, size_t bytes);
int stst_slab_copy_to_host(stst_slab *slab, void *cells, size_t bytes);
/* The same for `n_rows` owned rows starting at slab-local row `first_row` (slabs larger than what
 * the host wants to stage at once). */
int stst_slab_copy_rows_from_host(stst_slab *slab, size_t first_row, size_t n_rows,
                                  const void *cells, size_t bytes);
int stst_slab_copy_rows_to_host(stst_slab *slab, size_t first_row, size_t n_rows, void *cells,
                                size_t bytes);
/* Replace the owned rows by those of `source`: a slab of the same grid, row range and cell type on
 * the same device, usually the slab of ANOTHER workload over the same cells (convection alternates
 * "convection_pt" and "convection_thermal" updates). Device-to-device; waits for `source`; else
 * STST_ERR_RANGE. Follow it with stst_slab_exchange_halos. */
int stst_slab_copy_from_slab(stst_slab *slab, stst_slab *source);
int stst_slab_exchange_halos(stst_slab *slab);
/* As stst_grid_max_abs, extents in GLOBAL grid coordinates; out[q] covers the rows this slab owns
 * (-inf if none): combine the slabs' results with max (across processes: an all-reduce). */
int stst_slab_max_abs(stst_slab *slab, const stst_field_extent *extents, size_t n, double *out);
/* ONE field of `n_rows` owned rows from slab-local row `first_row` on. */
int stst_slab_copy_field_rows_to_host(stst_slab *slab, size_t field, size_t first_row, size_t n_rows,
                                      void *values, size_t bytes);
/* Uses transition_function, halo_value, iteration_offset, n_iterations and blocking of `params`. */
int stst_slab_update(stst_slab *slab, const stst_update_params *params);
/*
 * Speculative plane pass-through on slabs (the single-grid updater does all of this by itself, see
 * stst_update_stats.passthrough_planes). Fields the transition function never changes are left in
 * place by the tile sweeps; every pass verifies that. A slab has no untouched source grid to repeat
 * from, and its neighbours consume the rows it pushes, so the owner of the slabs drives the repeat:
 *   enable_speculation(1) once;  per update:  backup -> update -> take_violations on EVERY slab ->
 *   OR the masks together (across processes: an all-reduce) -> if non-zero: drop_passthrough(mask),
 *   restore and update again on every slab.
 */
int stst_slab_enable_speculation(stst_slab *slab, int enable, int *enabled /* may be NULL */);
int stst_slab_backup(stst_slab *slab);
int stst_slab_restore(stst_slab *slab);
int stst_slab_take_violations(stst_slab *slab, unsigned *planes);
int stst_slab_drop_passthrough(stst_slab *slab, unsigned planes);
int stst_slab_synchronize(stst_slab *slab);
/* The stream a CUDA event must be recorded on to bracket the slab's work (after join). */
int stst_slab_record_event(stst_slab *slab, void *event);

#ifdef __cplusplus
}
#endif
#endif /* STST_WORKLOADS_H */
