/*
 * StencilStream-B200 — host side of one fused launch: geometry, TMA descriptors, time-dependent
 * values, kernel attributes, the `<<<>>>` itself.
 *
 * Shared by the single-GPU updater (cuda/StencilUpdate.hpp) and the row-sharded one
 * (cuda/internal/SlabUpdate.hpp). The reference's counterpart is the body of the host loop in
 * StencilStream/cuda/StencilUpdate.hpp:216-263 (accessor set-up, capture of `halo_value`, the functor
 * and the host-evaluated time-dependent value, `parallel_for`).
 */
#pragma once
#include "Helpers.hpp"
#include "PassThrough.hpp"
#include "Planner.hpp"
#include "Runtime.hpp"
#include "TileKernel.hpp"

#include <climits>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>
#include <tuple>
#include <type_traits>

namespace stencil {
namespace cuda {
namespace internal {

/// Which part of which buffer one launch reads and writes.
struct LaunchRegion {
    int device;              ///< CUDA device the planes (and `stream`) live on
    unsigned grid_h, grid_w; ///< global grid extent
    int buf_row0;            ///< global row held in plane row 0 of both plane sets
    std::size_t buf_rows;    ///< rows present in the planes (slab rows incl. ghosts)
    int out_row_lo;          ///< global rows [out_row_lo, out_row_hi) are produced
    int out_row_hi;
    unsigned tile_h;         ///< output tile height for this launch (0: the plan's)
    int out2_row_lo = 0;     ///< optional second row range of the same launch (a slab's other
    int out2_row_hi = 0;     ///< boundary strip); empty unless out2_row_hi > out2_row_lo
    /// > 0: the planes hold a grid batch of this many members of grid_h x grid_w cells each, stacked
    /// by rows (fused_sweep_batch_kernel); every row range above is then member-local.
    unsigned members = 0;
};

/// Members one batch launch can hold (gridDim.y).
inline constexpr unsigned max_batch_members = 65535;

/**
 * TMA descriptors, encoded once per (plane set, box) and reused: cuTensorMapEncodeTiled costs a
 * microsecond or two per plane, which adds up for many-plane cells and short launches.
 */
template <typename Cell> class TensorMapCache {
  public:
    using Layout = CellLayout<Cell>;

    TensorMapSet const &get(PlaneSet const &planes, std::size_t width, std::size_t rows,
                            unsigned box_cols, unsigned box_rows) {
        const Key key{planes.base[0], planes.pitch[0], width, rows, box_cols, box_rows};
        auto it = cache.find(key);
        if (it != cache.end())
            return it->second;
        if (cache.size() >= 64)
            cache.clear();
        TensorMapSet maps{};
        for (std::size_t i = 0; i < Layout::n_planes; i++) {
            STST_RT_CHECK(stst_tensor_map_encode_2d(
                &maps.map[i][0], planes.base[i], int(Layout::plane_bytes(i)), width, rows,
                planes.pitch[i] * Layout::plane_bytes(i), box_cols, box_rows));
        }
        return cache.emplace(key, maps).first->second;
    }

    void clear() { cache.clear(); }

  private:
    using Key = std::tuple<void *, unsigned long long, std::size_t, std::size_t, unsigned, unsigned>;
    std::map<Key, TensorMapSet> cache;
};

template <typename F> struct SweepLauncher {
    using Cell = typename F::Cell;
    using TDV = typename F::TimeDependentValue;
    using Layout = CellLayout<Cell>;
    static constexpr int CW = column_group_width<Cell>();
    // Register window: rotated by unrolling for light-weight cells, shifted for medium ones; fat
    // cells re-read their neighbourhood from shared memory instead (see sweep_rows).
#if defined(STST_WINDOW_MODE)
    static constexpr int kMode = STST_WINDOW_MODE;
#else
    static constexpr int kMode = sizeof(Cell) <= 8    ? window_rotate
                                 : sizeof(Cell) <= 16 ? window_shift
                                                      : window_reload;
#endif

    /**
     * Enqueue one fused launch on `stream`: iterations [iteration0, iteration0 + n_gens) of `tf`
     * applied to `region` of `src`, results into `dst` (and, with `push`, into the neighbour slabs).
     */
    static void launch(LaunchPlan const &plan, F const &tf, Cell const &halo_value,
                       PlaneSet const &src, PlaneSet const &dst, HaloPush const *push,
                       LaunchRegion const &region, std::size_t iteration0, unsigned n_gens,
                       TensorMapCache<Cell> &maps_cache, stst_stream_t stream,
                       Speculation const *spec = nullptr) {
#if defined(__CUDACC__)
        constexpr unsigned n_sub = unsigned(F::n_subiterations);
        constexpr unsigned radius = unsigned(F::stencil_radius);
        if (n_gens == 0 || n_gens > plan.fused_iterations || n_gens > max_fused_iterations)
            throw std::invalid_argument("StencilStream-B200: illegal number of fused iterations");
        if (region.out_row_hi <= region.out_row_lo || region.grid_w == 0)
            return;
        const bool batch = region.members > 0;
        if (region.members > max_batch_members || (batch && (push || region.buf_row0 != 0)))
            throw std::invalid_argument("StencilStream-B200: illegal grid batch launch");

        SweepGeometry geo{};
        geo.grid_h = region.grid_h;
        geo.grid_w = region.grid_w;
        geo.buf_row0 = region.buf_row0;
        geo.buf_rows = unsigned(region.buf_rows);
        geo.out_row_lo = region.out_row_lo;
        geo.out_row_hi = region.out_row_hi;
        geo.tile_h = region.tile_h ? std::min(region.tile_h, plan.tile_h) : plan.tile_h;
        const bool second = region.out2_row_hi > region.out2_row_lo;
        geo.tile_h = std::min(geo.tile_h, unsigned(region.out_row_hi - region.out_row_lo));
        if (second)
            geo.tile_h = std::min(geo.tile_h, unsigned(region.out2_row_hi - region.out2_row_lo));
        geo.tile_w = plan.tile_w;
        geo.halo = n_gens * n_sub * radius;
        geo.hpad = plan.hpad;
        geo.n_gens = n_gens;
        geo.tiles_x = (geo.grid_w + geo.tile_w - 1) / geo.tile_w;
        geo.use_tma = plan.use_tma ? 1u : 0u;
        geo.push = push ? 1u : 0u;
        geo.inv_block_y = (1u << 24) / plan.block_y + 1u;
        constexpr unsigned all_planes =
            Layout::n_planes >= 32 ? ~0u : ((1u << Layout::n_planes) - 1u);
        unsigned single_planes = 0;
        if (spec) {
            if constexpr (speculation_capable<F>()) {
                for (unsigned q = 0; q < n_sub && q < max_spec_subiterations; q++)
                    geo.keep[q] = spec->probe ? 0u : (spec->keep[q] & all_planes);
                geo.probe = spec->probe ? 1u : 0u;
                geo.spec_flags = spec->flags;
                single_planes = spec->probe ? 0u : spec->single_planes(n_sub, all_planes);
                if (single_planes != plan.single_planes)
                    throw std::logic_error("StencilStream-B200: plan and speculation masks disagree");
            } else {
                throw std::logic_error("StencilStream-B200: speculation on an incapable functor");
            }
        }
        geo.iteration0 = iteration0;
        const unsigned out_rows = unsigned(region.out_row_hi - region.out_row_lo);
        geo.tiles_first = geo.tiles_x * ((out_rows + geo.tile_h - 1) / geo.tile_h);
        unsigned tiles_second = 0;
        if (second) {
            geo.out2_row_lo = region.out2_row_lo;
            geo.out2_row_hi = region.out2_row_hi;
            const unsigned rows2 = unsigned(region.out2_row_hi - region.out2_row_lo);
            tiles_second = geo.tiles_x * ((rows2 + geo.tile_h - 1) / geo.tile_h);
        }

        // Time-dependent values: evaluated on the host, exactly once per iteration
        // (reference cuda/StencilUpdate.hpp:224).
        TdvArray<TDV> tdvs{};
        for (unsigned g = 0; g < n_gens; g++)
            tdvs.v[g] = tf.get_time_dependent_value(iteration0 + g);

        const unsigned rows = geo.tile_h + 2 * geo.halo;
        const unsigned cols = plan.block_x * unsigned(CW);
        const std::size_t smem =
            tile_smem_bytes<Cell>(rows, cols, (n_gens * n_sub > 1) ? 2 : 1, single_planes);

        static const TensorMapSet no_maps{};
        TensorMapSet const *maps = &no_maps;
        if (plan.use_tma)
            maps = &maps_cache.get(src, region.grid_w, region.buf_rows, cols, rows);

        static const HaloPush no_push{};

        int current_device = -1;
        if (cudaGetDevice(&current_device) != cudaSuccess || current_device != region.device) {
            if (cudaSetDevice(region.device) != cudaSuccess)
                throw std::runtime_error("StencilStream-B200: cannot select CUDA device " +
                                         std::to_string(region.device));
        }

        const dim3 block(plan.block_x, plan.block_y, 1);
        const dim3 grid(geo.tiles_first + tiles_second, batch ? region.members : 1u, 1);
        auto submit = [&](auto kernel, std::size_t &configured_smem, auto batch_c) {
            if (smem > configured_smem) {
                cudaError_t err = cudaFuncSetAttribute(
                    kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
                if (err != cudaSuccess)
                    throw std::runtime_error(std::string("StencilStream-B200: cannot reserve ") +
                                             std::to_string(smem) + " bytes of shared memory: " +
                                             cudaGetErrorString(err));
                configured_smem = smem;
            }
            if constexpr (decltype(batch_c)::value)
                kernel<<<grid, block, smem, static_cast<cudaStream_t>(stream)>>>(
                    tf, halo_value, tdvs, src, dst, *maps, geo);
            else
                kernel<<<grid, block, smem, static_cast<cudaStream_t>(stream)>>>(
                    tf, halo_value, tdvs, src, dst, push ? *push : no_push, *maps, geo);
        };
        // [spec][batch][device]
        static std::size_t configured_smem_per_device[2][2][64] = {};
        auto submit_kind = [&](auto spec_c) {
            constexpr bool kSpec = decltype(spec_c)::value;
            if (batch)
                submit(fused_sweep_batch_kernel<F, CW, kMode, fixed_block_x<Cell>(),
                                                max_threads_per_cta<Cell>(), 1, kSpec>,
                       configured_smem_per_device[kSpec][1][region.device & 63], std::true_type{});
            else
                submit(fused_sweep_kernel<F, CW, kMode, fixed_block_x<Cell>(),
                                          max_threads_per_cta<Cell>(), 1, kSpec>,
                       configured_smem_per_device[kSpec][0][region.device & 63], std::false_type{});
        };
        if constexpr (speculation_capable<F>()) {
            if (spec)
                submit_kind(std::true_type{});
            else
                submit_kind(std::false_type{});
        } else {
            submit_kind(std::false_type{});
        }
        cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess)
            throw std::runtime_error(std::string("StencilStream-B200: kernel launch failed: ") +
                                     cudaGetErrorString(err));
#else
        (void)plan, (void)tf, (void)halo_value, (void)src, (void)dst, (void)push, (void)region;
        (void)iteration0, (void)n_gens, (void)maps_cache, (void)stream;
        throw std::runtime_error("StencilStream-B200 must be compiled with nvcc for sm_100a; "
                                 "there is no CPU fallback");
#endif
    }
};

} // namespace internal
} // namespace cuda
} // namespace stencil
