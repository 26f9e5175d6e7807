/*
 * StencilStream-B200 — `stencil::cuda::StencilUpdate<F, split_cell_structure>`: the generation loop.
 *
 * Drop-in for the reference's updater (reference StencilStream/cuda/StencilUpdate.hpp:41-445):
 * same template parameters, the same `Params` aggregate (field names and order are API because user
 * code uses designated initialisers; B200-only fields come last), the same methods
 * (`operator()(GridImpl&)`, `get_params`, `get_n_processed_cells`, `get_walltime`,
 * `get_kernel_runtime`) and the same observable semantics:
 *
 *   - the source grid is never modified; the result is a different allocation (for
 *     `n_iterations == 0` the result aliases the source, like the reference's non-split path, :275),
 *   - iteration i in [iteration_offset, iteration_offset + n_iterations) runs sub-iterations
 *     0 .. F::n_subiterations-1 as full-grid sweeps (:212-215),
 *   - the time-dependent value of iteration i is `transition_function.get_time_dependent_value(i)`,
 *     evaluated ON THE HOST (:224) — here once per iteration up front, shipped per launch as a
 *     kernel-parameter array (the scheme of the reference's
 *     tdv::single_pass::PrecomputeOnHostStrategy, StencilStream/tdv/SinglePassStrategies.hpp:203-264),
 *   - cells outside the grid read as `halo_value` in every sweep (:241-252),
 *   - `params` is re-read on every call (:223), calls are asynchronous unless `blocking` (:133-135),
 *   - `n_processed_cells += n_iterations * H * W`, walltime accumulates (:137-141).
 *
 * B200 extension: `operator()(GridBatch<Cell> &)` advances every member of a grid batch
 * (cuda/GridBatch.hpp) with the same parameters, one launch per fused pass for all members; the
 * result equals one grid update per member, bit for bit. It shares the generation loop, the planner
 * and plane pass-through with the grid overload. A batch runs on its own device: `cuda_devices`
 * with more than one entry throws std::invalid_argument, and STST_DEVICES does not apply.
 *
 * What is different: instead of one launch per sweep, ceil(n_iterations / k) launches of the fused,
 * shared-memory-tiled kernel in cuda/internal/TileKernel.hpp, planned by cuda/internal/Planner.hpp.
 * Fields that a transition function only passes through are no longer copied between the tile
 * buffers (cuda/internal/PassThrough.hpp): declared by the cell type (HotSpot's `power`), or detected
 * at run time (FDTD's material coefficients), verified by every launch and transparently repeated
 * without them if a launch ever sees such a field change (see `run_detected` below and run_tile in
 * TileKernel.hpp).
 * `split_cell_structure` is accepted for source compatibility; the device layout is decided by
 * `Grid<Cell>` from `Cell::fields` alone (planes whenever the cell lists its fields), so both
 * values select the same code path and produce the same results.
 */
#pragma once
#include "../Concepts.hpp"
#include "../Stencil.hpp"
#include "Grid.hpp"
#include "GridBatch.hpp"
#include "internal/Helpers.hpp"
#include "internal/Launch.hpp"
#include "internal/PassThrough.hpp"
#include "internal/Planner.hpp"
#include "internal/Runtime.hpp"
#include "internal/SlabUpdate.hpp"
#include "internal/TileKernel.hpp"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <string>
#include <vector>

namespace stencil {
namespace cuda {

template <concepts::TransitionFunction F, bool split_cell_structure = false> class StencilUpdate {
  public:
    // (public: nvcc's host-side rewriting of designated initialisers such as
    // `{.halo_value = MyCell{}}` names the aggregate's member types through these aliases)
    using Cell = typename F::Cell;
    using TDV = typename F::TimeDependentValue;

  private:
    static_assert(std::is_trivially_copyable_v<F>,
                  "transition functions are copied into kernel parameters and must be trivially "
                  "copyable");
    static_assert(std::is_trivially_copyable_v<TDV>,
                  "time-dependent values are shipped as kernel parameters and must be trivially "
                  "copyable");

  public:
    /// The grid type this updater consumes and produces.
    using GridImpl = Grid<Cell>;

    /// B200 extension: the grid batch type this updater also consumes and produces.
    using GridBatchImpl = GridBatch<Cell>;

    struct Params {
        /// The transition function instance; may carry runtime parameters.
        F transition_function;

        /// Value presented for every cell outside the grid, in every sweep.
        Cell halo_value = Cell();

        /// Iteration index of the input grid; added to the local iteration counter.
        std::size_t iteration_offset = 0;

        /// Number of iterations to compute.
        std::size_t n_iterations = 1;

        /// Kept for source compatibility (the shim's sycl::device carries no information); an update
        /// runs on the CUDA device its source grid lives on, see `cuda_device`.
        sycl::device device = sycl::device();

        /// Wait for the result before returning from `operator()`.
        bool blocking = false;

        /// Record device-side timestamps around every launch (see get_kernel_runtime()).
        bool profiling = false;

        // ---- B200 extensions (keep last: designated initialisers of reference code stay valid) ----

        /// CUDA device ordinal the update is expected to run on; negative (default): wherever the
        /// source grid lives. An update never migrates a grid: a non-negative ordinal that differs
        /// from the source grid's device makes `operator()` throw std::invalid_argument.
        int cuda_device = -1;

        /// Iterations fused per launch (temporal blocking depth k); 0 picks one automatically.
        unsigned fused_iterations = 0;

        /// Upper bound for the output tile height; 0 lets the planner fill shared memory.
        unsigned tile_rows = 0;

        /// CUDA devices to spread one update over: the grid is cut into row slabs, one per entry
        /// (an ordinal may appear more than once), each slab runs the generation loop on its device
        /// and pushes its boundary rows into its neighbours over NVLink (cuda/internal/SlabUpdate.hpp).
        /// Source and result grid stay ordinary single-device grids: the slabs are filled from the
        /// source and gathered into the result with device-to-device copies, inside `operator()`.
        /// Empty (default): the environment variable STST_DEVICES ("0,1,2,3" or "0-7"), else the
        /// device of the source grid alone. The reference's updater takes one device
        /// (reference cuda/StencilUpdate.hpp:83, :124-127); this is how a program written against
        /// it — the unmodified examples — uses a whole 8 x B200 box.
        std::vector<int> cuda_devices = {};
    };

    StencilUpdate(Params params)
        : params(params), n_processed_cells(0), walltime(0.0), n_launches(0), last_plan(),
          tensor_maps(), profile_events() {}

    StencilUpdate(StencilUpdate const &other)
        : params(other.params), n_processed_cells(other.n_processed_cells),
          walltime(other.walltime), n_launches(other.n_launches), last_plan(other.last_plan),
          tensor_maps(), profile_events(other.profile_events), pass_through(other.pass_through),
          n_spec_redos(other.n_spec_redos) {}
    StencilUpdate &operator=(StencilUpdate const &) = delete;

    /**
     * Compute `n_iterations` iterations of the source grid and return the result as a new grid.
     * The source grid is not modified.
     */
    GridImpl operator()(GridImpl &source_grid) {
        auto walltime_start = std::chrono::high_resolution_clock::now();

        GridImpl result_grid = run_simulation(source_grid);

        if (params.blocking) {
            STST_RT_CHECK(stst_stream_synchronize(source_grid.get_storage().stream));
        }

        auto walltime_end = std::chrono::high_resolution_clock::now();
        walltime += std::chrono::duration<double>(walltime_end - walltime_start).count();
        n_processed_cells +=
            params.n_iterations * source_grid.get_grid_height() * source_grid.get_grid_width();
        return result_grid;
    }

    /**
     * B200 extension: compute `n_iterations` iterations of every member of `source` and return the
     * result as a new batch (the source itself for `n_iterations == 0`); the source is not modified.
     * Semantics as for a grid, per member; `n_processed_cells` grows by n_iterations * members *
     * H * W, `get_n_launches()` by one per fused pass.
     */
    GridBatchImpl operator()(GridBatchImpl &source) {
        if (params.cuda_devices.size() > 1)
            throw std::invalid_argument("StencilStream-B200: a grid batch runs on one device; "
                                        "Params::cuda_devices lists several");
        if (source.get_members() > internal::max_batch_members)
            throw std::invalid_argument("StencilStream-B200: a grid batch holds at most " +
                                        std::to_string(internal::max_batch_members) + " members");
        auto walltime_start = std::chrono::high_resolution_clock::now();

        GridBatchImpl result = run_simulation(source);

        if (params.blocking) {
            STST_RT_CHECK(stst_stream_synchronize(source.get_storage().stream));
        }

        auto walltime_end = std::chrono::high_resolution_clock::now();
        walltime += std::chrono::duration<double>(walltime_end - walltime_start).count();
        n_processed_cells +=
            params.n_iterations * source.get_storage().height * source.get_storage().width;
        return result;
    }

    /// Live reference to the parameters; changes apply to the next call of `operator()`.
    Params &get_params() { return params; }

    /// Accumulated `n_iterations * height * width` over all calls.
    std::size_t get_n_processed_cells() const { return n_processed_cells; }

    /// Accumulated host-side time spent in `operator()` (meaningful as compute time if `blocking`).
    double get_walltime() const { return walltime; }

    /**
     * Accumulated device-side runtime in seconds of all fused launches submitted while
     * `Params::profiling` was set. Waits for those launches to finish.
     */
    double get_kernel_runtime() const {
        double seconds = 0.0;
        for (auto const &pair : profile_events) {
            STST_RT_CHECK(stst_event_synchronize(pair.second->get()));
            float ms = 0.0f;
            STST_RT_CHECK(stst_event_elapsed_ms(pair.first->get(), pair.second->get(), &ms));
            seconds += double(ms) * 1e-3;
        }
        return seconds;
    }

    /// B200 extension: number of kernel launches submitted so far.
    std::size_t get_n_launches() const { return n_launches; }

    /// B200 extension: number of row slabs (GPUs) the most recent call ran on (1: not sharded).
    std::size_t get_n_slabs() const { return shards ? shards->slabs.size() : 1; }

    /// B200 extension: the plan used by the most recent call.
    internal::LaunchPlan const &get_last_plan() const { return last_plan; }

    /// B200 extension: planes (bit i = plane i) that currently pass through every sub-iteration
    /// without being copied (speculative plane pass-through), and how many times an update had to
    /// be repeated because a launch saw such a plane change.
    unsigned get_passthrough_planes() const {
        return shards ? shards->slabs.front()->passthrough_planes() : pass_through.single_planes();
    }
    std::size_t get_n_speculation_redos() const { return n_spec_redos; }

  private:
    using PassThrough = internal::PassThrough<F>;

    /// Members of a grid batch, 0 for a grid (the launches' LaunchRegion::members).
    static unsigned members_of(GridImpl &) { return 0; }
    static unsigned members_of(GridBatchImpl &batch) { return unsigned(batch.get_members()); }

    // G: GridImpl or GridBatchImpl
    template <typename G> G run_simulation(G &source_grid) {
        constexpr bool is_batch = std::is_same_v<G, GridBatchImpl>;
        if (params.n_iterations == 0) {
            return source_grid;
        }
        if (params.cuda_device >= 0 && params.cuda_device != source_grid.get_storage().device)
            throw std::invalid_argument(
                "StencilStream-B200: Params::cuda_device is " + std::to_string(params.cuda_device) +
                " but the source grid lives on device " +
                std::to_string(source_grid.get_storage().device) +
                "; updates run where their grid is (create the grid on that device)");
        if constexpr (!is_batch) {
            const std::vector<int> devices = resolve_devices();
            if (devices.size() > 1 && source_grid.get_grid_height() > 0 &&
                source_grid.get_grid_width() > 0) {
                if (ensure_shards(source_grid, devices))
                    return run_sharded(source_grid);
            } else {
                shards.reset();
            }
        }
        auto &source = source_grid.get_storage();
        if (source.height == 0 || source.width == 0)
            return source_grid.make_similar();

        lap_start = std::chrono::high_resolution_clock::now();
        source.require_device();
        lap("require_device");

        if (PassThrough::declared()) {
            // Fields declared constant by the cell type: no observing launch and no read-back, the
            // call stays asynchronous. With STST_VERIFY_CONSTANT_FIELDS=1 the kernels' own check of
            // the kept planes is read after the last launch (one stream synchronisation) and a
            // violated declaration throws std::logic_error.
            const auto spec = pass_through.verifying(source.device, source.stream);
            const unsigned members = members_of(source_grid);
            G result = run_passes(source_grid,
                                  plan_for(source, pass_through.single_planes(), members), &*spec,
                                  params.iteration_offset, params.n_iterations);
            static const bool verify = internal::env_long("STST_VERIFY_CONSTANT_FIELDS", 0) != 0;
            if (verify) {
                const unsigned violated = pass_through.take_violations(source.stream);
                if (violated != 0)
                    throw std::logic_error(
                        "StencilStream-B200: the transition function changed a field that its cell "
                        "type lists in Cell::constant_fields (plane mask " +
                        std::to_string(violated) + ")");
            }
            return result;
        }
        if (PassThrough::detected() && !pass_through.nothing_left())
            return run_detected(source_grid);
        return run_passes(source_grid, plan_for(source, 0, members_of(source_grid)), nullptr,
                          params.iteration_offset, params.n_iterations);
    }

    /**
     * The generation loop with pass-through of DETECTED planes.
     *
     * The first launch this updater ever submits also *observes*: per sub-iteration, which planes
     * came out of the transition function different from the centre cell that went in. Planes that
     * never changed are from then on left in place by the tile sweeps instead of being copied from
     * tile buffer to tile buffer, and planes untouched in every sub-iteration need only one tile
     * buffer, so the tiles grow. Every launch still compares what the function returned for those
     * planes with what went in (for a genuinely passed-through field the compiler folds that away)
     * and reports any difference through a device flag, which is read when all launches of the call
     * have been submitted. If a launch reports a difference — the field does change after all, e.g.
     * FDTD's `hz_sum` once `iteration >= detect_iteration` — that plane is struck from the masks and
     * the WHOLE call is repeated from the (never modified) source grid. The result is therefore
     * always what the plain loop computes; the price is that such calls end with a stream
     * synchronisation even when `blocking` is false.
     */
    template <typename G> G run_detected(G &source_grid) {
        auto &source = source_grid.get_storage();
        const unsigned members = members_of(source_grid);
        // launches and profiling events of an attempt that is discarded must not be counted
        const std::size_t launches_before = n_launches;
        const std::size_t events_before = profile_events.size();
        for (;;) {
            G result = source_grid;
            std::size_t observed = 0; // iterations computed by the observing launch
            if (!pass_through.probed()) {
                const internal::Speculation observe =
                    pass_through.observing(source.device, source.stream);
                const internal::LaunchPlan plan = plan_for(source, 0, members);
                observed = std::min<std::size_t>(params.n_iterations, plan.fused_iterations);
                result = run_passes(source_grid, plan, &observe, params.iteration_offset, observed);
                pass_through.read_observation(source.stream);
            }
            const auto spec = pass_through.verifying(source.device, source.stream);
            if (observed < params.n_iterations)
                result = run_passes(result, plan_for(source, pass_through.single_planes(), members),
                                    spec ? &*spec : nullptr, params.iteration_offset + observed,
                                    params.n_iterations - observed, observed > 0);
            const unsigned violated = spec ? pass_through.take_violations(source.stream) : 0u;
            if (violated == 0)
                return result;
            // A plane believed to pass through did change: never keep it again and recompute this
            // call from the untouched source grid.
            pass_through.drop(violated);
            n_spec_redos++;
            n_launches = launches_before;
            profile_events.resize(events_before);
        }
    }

    /**
     * The generation loop: iterations [iteration, iteration + n_iterations) as launches of `plan`
     * (with `spec`, if given) from `source` through two scratch grids, the second one allocated only
     * if there is more than one launch. With `source_is_scratch` (the source is the result of an
     * earlier launch of this call) the source grid itself serves as the second scratch grid.
     */
    template <typename G>
    G run_passes(G &source, internal::LaunchPlan const &plan, internal::Speculation const *spec,
                 std::size_t iteration, std::size_t n_iterations, bool source_is_scratch = false) {
        last_plan = plan;
        const std::size_t k = plan.fused_iterations;
        const unsigned members = members_of(source);
        G swap_a = source.make_similar();
        G swap_b = source_is_scratch ? source
                   : (n_iterations > k) ? source.make_similar()
                                        : swap_a;
        swap_a.get_storage().allocate_device();
        swap_b.get_storage().allocate_device();
        lap("allocate scratch grids");

        G *pass_source = &source, *pass_target = &swap_a;
        while (n_iterations > 0) {
            const unsigned n_gens = unsigned(std::min(n_iterations, k));
            launch(plan, pass_source->get_storage(), pass_target->get_storage(), iteration, n_gens,
                   spec, members);
            iteration += n_gens;
            n_iterations -= n_gens;
            pass_source = pass_target;
            pass_target = (pass_target == &swap_a) ? &swap_b : &swap_a;
        }
        pass_source->get_storage().device_written();
        lap("submit launches");
        return *pass_source;
    }

    /// Plan for the grid `source`, or for the batch of `members` members it holds.
    internal::LaunchPlan plan_for(internal::GridStorage<Cell> const &source, unsigned single_planes,
                                  unsigned members) {
        const internal::LaunchPlan plan = internal::make_plan<F>(
            source.device, unsigned(members ? source.height / members : source.height),
            unsigned(source.width), params.n_iterations, params.fused_iterations, params.tile_rows,
            single_planes, std::max(members, 1u));
        lap("make_plan");
        return plan;
    }

    /// STST_TRACE: host time since the previous step of this call, on stderr.
    void lap(const char *what) {
        if (!std::getenv("STST_TRACE"))
            return;
        const auto now = std::chrono::high_resolution_clock::now();
        std::fprintf(stderr, "[stst] %-22s %9.3f ms\n", what,
                     std::chrono::duration<double, std::milli>(now - lap_start).count());
        lap_start = now;
    }

    // ---- one update spread over several GPUs of the box (Params::cuda_devices / STST_DEVICES) ----------

    using Slab = internal::SlabUpdate<F>;

    struct ShardSet {
        ~ShardSet() {
            // a slab may still be pushing rows into a neighbour: wait for all before freeing any
            for (auto &slab : slabs)
                if (slab)
                    slab->synchronize();
        }
        std::vector<int> devices;
        std::size_t grid_h = 0, grid_w = 0;
        unsigned fused_override = 0, tile_rows = 0;
        std::vector<std::unique_ptr<Slab>> slabs;
        std::vector<std::unique_ptr<internal::Event>> done; ///< per slab: result rows are in place
        bool speculating = false;
    };

    std::vector<int> resolve_devices() const {
        if (!params.cuda_devices.empty())
            return params.cuda_devices;
        std::vector<int> devices;
        const char *env = std::getenv("STST_DEVICES");
        if (!env || !*env)
            return devices;
        // "0,1,2,3", "0-7" or a mixture ("0-3,6,7")
        const std::string text(env);
        std::size_t pos = 0;
        while (pos < text.size()) {
            std::size_t end = text.find(',', pos);
            if (end == std::string::npos)
                end = text.size();
            const std::string item = text.substr(pos, end - pos);
            const std::size_t dash = item.find('-', 1);
            try {
                if (dash == std::string::npos) {
                    devices.push_back(std::stoi(item));
                } else {
                    const int lo = std::stoi(item.substr(0, dash)), hi = std::stoi(item.substr(dash + 1));
                    for (int d = lo; d <= hi; d++)
                        devices.push_back(d);
                }
            } catch (std::exception const &) {
                throw std::invalid_argument("StencilStream-B200: cannot parse STST_DEVICES=\"" + text +
                                            "\"");
            }
            pos = end + 1;
        }
        return devices;
    }

    /// Build (or reuse) the slabs for this grid and device list. Returns false if the grid cannot be
    /// cut that way (fewer rows per slab than the ghost depth needs): the caller then runs unsharded.
    bool ensure_shards(GridImpl &source_grid, std::vector<int> const &devices) {
        using namespace internal;
        auto &source = source_grid.get_storage();
        if (shards && shards->devices == devices && shards->grid_h == source.height &&
            shards->grid_w == source.width && shards->fused_override == params.fused_iterations &&
            shards->tile_rows == params.tile_rows)
            return true;
        shards.reset();
        int n_devices = 0;
        STST_RT_CHECK(stst_device_count(&n_devices));
        for (int d : devices)
            if (d < 0 || d >= n_devices)
                throw std::invalid_argument("StencilStream-B200: no CUDA device " + std::to_string(d) +
                                            " (cuda_devices / STST_DEVICES)");
        for (std::size_t count = std::min<std::size_t>(devices.size(), source.height); count > 1;
             count--) {
            auto set = std::make_unique<ShardSet>();
            set->devices = devices;
            set->grid_h = source.height;
            set->grid_w = source.width;
            set->fused_override = params.fused_iterations;
            set->tile_rows = params.tile_rows;
            try {
                unsigned fused = params.fused_iterations;
                for (int attempt = 0; attempt < 2; attempt++) {
                    set->slabs.clear();
                    unsigned k_min = ~0u, k_max = 0;
                    for (std::size_t i = 0; i < count; i++) {
                        typename Slab::Config cfg{};
                        cfg.grid_rows = source.height;
                        cfg.grid_cols = source.width;
                        partition_rows(source.height, count, i, cfg.row_lo, cfg.row_hi);
                        cfg.device = devices[i];
                        cfg.fused_iterations = fused;
                        cfg.tile_rows = params.tile_rows;
                        cfg.overlap = true;
                        set->slabs.push_back(std::make_unique<Slab>(cfg));
                        const unsigned k = set->slabs.back()->get_plan().fused_iterations;
                        k_min = std::min(k_min, k);
                        k_max = std::max(k_max, k);
                    }
                    if (k_min == k_max)
                        break;
                    fused = k_min; // all slabs must fuse the same depth: it fixes the ghost rows
                }
            } catch (std::invalid_argument const &) {
                continue; // a slab would own fewer rows than its neighbour's ghost depth: use fewer
            }
            // neighbours push into each other, the grid's device copies to and from every slab
            for (std::size_t i = 0; i < count; i++) {
                const int me = devices[i];
                auto allow = [&](int a, int b) {
                    if (a == b)
                        return;
                    int can = 0;
                    STST_RT_CHECK(stst_peer_can_access(a, b, &can));
                    if (!can)
                        throw std::runtime_error("StencilStream-B200: devices " + std::to_string(a) +
                                                 " and " + std::to_string(b) +
                                                 " cannot access each other's memory");
                    STST_RT_CHECK(stst_peer_enable(a, b));
                };
                if (i > 0) {
                    allow(me, devices[i - 1]);
                    auto const &up = set->slabs[i - 1]->get_config();
                    set->slabs[i]->attach(SlabSide::up, set->slabs[i - 1]->device_base(), up.row_lo,
                                          up.row_hi);
                }
                if (i + 1 < count) {
                    allow(me, devices[i + 1]);
                    auto const &down = set->slabs[i + 1]->get_config();
                    set->slabs[i]->attach(SlabSide::down, set->slabs[i + 1]->device_base(),
                                          down.row_lo, down.row_hi);
                }
                allow(me, source.device);
                allow(source.device, me);
                // (a CUDA event belongs to the device that is current when it is created, and can
                // only be recorded on that device's streams)
                STST_RT_CHECK(stst_set_device(me));
                set->done.push_back(std::make_unique<Event>());
            }
            set->speculating = PassThrough::detected();
            for (auto &slab : set->slabs)
                slab->enable_speculation(set->speculating);
            shards = std::move(set);
            return true;
        }
        return false;
    }

    /**
     * The generation loop on row slabs, one per device: fill the slabs (owned and ghost rows) from
     * the source grid, advance all of them pass by pass — the passes of the slabs are enqueued
     * round-robin, so that no device's launch queue fills up with work that waits for a neighbour
     * whose work is not enqueued yet — and gather the owned rows into the result grid. Everything is
     * stream-ordered; the result grid's stream waits for the gather. With plane pass-through active
     * the call ends by collecting the slabs' verification flags, and is repeated from the (never
     * modified) source grid if any slab saw a kept plane change.
     */
    GridImpl run_sharded(GridImpl &source_grid) {
        using namespace internal;
        auto &source = source_grid.get_storage();
        source.require_device();
        GridImpl result = source_grid.make_similar();
        auto &target = result.get_storage();
        target.allocate_device();
        STST_RT_CHECK(stst_set_device(source.device)); // `ready` and the profiling events live there
        Event ready;
        const std::size_t k = shards->slabs.front()->get_plan().fused_iterations;
        std::size_t launches_before = 0;
        for (auto &slab : shards->slabs)
            launches_before += slab->get_n_launches();

        std::shared_ptr<Event> start, stop;
        if (params.profiling) {
            start = std::make_shared<Event>(true);
            stop = std::make_shared<Event>(true);
            start->record(source.stream);
        }
        for (;;) {
            ready.record(source.stream);
            for (auto &slab : shards->slabs)
                slab->load_from_grid(source.planes, source.device, ready.get());
            std::size_t iteration = params.iteration_offset, remaining = params.n_iterations;
            while (remaining > 0) {
                const std::size_t n_gens = std::min(remaining, k);
                for (auto &slab : shards->slabs)
                    slab->run(params.transition_function, params.halo_value, iteration, n_gens);
                iteration += n_gens;
                remaining -= n_gens;
            }
            unsigned violated = 0;
            if (shards->speculating) {
                bool useful = false;
                for (auto &slab : shards->slabs) {
                    violated |= slab->take_violations();
                    useful = useful || slab->passthrough_planes() != 0;
                }
                if (violated == 0 && !useful) {
                    shards->speculating = false; // nothing left to pass through: drop the protocol
                    for (auto &slab : shards->slabs)
                        slab->enable_speculation(false);
                }
            }
            if (violated == 0)
                break;
            for (auto &slab : shards->slabs)
                slab->drop_passthrough(violated);
            n_spec_redos++;
        }
        for (std::size_t i = 0; i < shards->slabs.size(); i++) {
            shards->slabs[i]->store_to_grid(target.planes, target.device, shards->done[i]->get());
            STST_RT_CHECK(stst_stream_wait_event(target.stream, shards->done[i]->get()));
        }
        if (params.profiling) {
            stop->record(target.stream);
            profile_events.emplace_back(std::move(start), std::move(stop));
        }
        target.device_written();
        last_plan = shards->slabs.front()->get_active_plan();
        std::size_t launches_after = 0;
        for (auto &slab : shards->slabs)
            launches_after += slab->get_n_launches();
        n_launches += launches_after - launches_before;
        // leave the thread on the grid's device, as a single-device update does
        STST_RT_CHECK(stst_set_device(source.device));
        return result;
    }

    /// One fused launch over the grid in `src`, or over every member of the batch it holds.
    void launch(internal::LaunchPlan const &plan, internal::GridStorage<Cell> &src,
                internal::GridStorage<Cell> &dst, std::size_t iteration0, unsigned n_gens,
                internal::Speculation const *spec, unsigned members) {
        using namespace internal;
        const std::size_t grid_h = members ? src.height / members : src.height;
        LaunchRegion region{};
        region.device = src.device;
        region.grid_h = unsigned(grid_h);
        region.grid_w = unsigned(src.width);
        region.buf_row0 = 0;
        region.buf_rows = src.height;
        region.out_row_lo = 0;
        region.out_row_hi = int(grid_h);
        region.tile_h = 0;
        region.members = members;

        std::shared_ptr<Event> start, stop;
        if (params.profiling) {
            STST_RT_CHECK(stst_set_device(src.device)); // events belong to the current device
            start = std::make_shared<Event>(true);
            stop = std::make_shared<Event>(true);
            start->record(src.stream);
        }

        SweepLauncher<F>::launch(plan, params.transition_function, params.halo_value, src.planes,
                                 dst.planes, nullptr, region, iteration0, n_gens, tensor_maps,
                                 src.stream, spec);
        n_launches++;

        if (params.profiling) {
            stop->record(src.stream);
            profile_events.emplace_back(std::move(start), std::move(stop));
        }
    }

    Params params;
    std::size_t n_processed_cells;
    double walltime;
    std::size_t n_launches;
    internal::LaunchPlan last_plan;
    internal::TensorMapCache<Cell> tensor_maps;
    std::vector<std::pair<std::shared_ptr<internal::Event>, std::shared_ptr<internal::Event>>>
        profile_events;
    internal::PassThrough<F> pass_through;
    std::size_t n_spec_redos = 0;
    std::chrono::high_resolution_clock::time_point lap_start; ///< STST_TRACE

    // row slabs of the multi-GPU path (run_sharded); rebuilt when grid shape or device list change
    std::unique_ptr<ShardSet> shards;
};

} // namespace cuda
} // namespace stencil
