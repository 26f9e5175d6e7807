/*
 * StencilStream-B200 — launch planning for the fused generation loop.
 *
 * Decides, per transition function and device, how many iterations one launch fuses (k), the
 * shape of the CTA (column groups x row groups) and of its output tile, and the dynamic shared
 * memory that follows from it. The reference has nothing comparable for its cuda backend (one
 * work-item per cell, k = 1: StencilStream/cuda/StencilUpdate.hpp:209-215); the closest relative is
 * the FPGA tiling backend's compile-time tile/temporal-parallelism arithmetic
 * (StencilStream/tiling/internal/StencilUpdateKernel.hpp:79-99), whose halo rule
 * `halo = radius * n_subiterations * fused iterations` is the one used here.
 *
 * Every choice can be overridden, in this order of precedence: `StencilUpdate::Params` fields
 * (fused_iterations — an upper bound, clamped to what fits into shared memory — and tile_rows), then the environment (STST_FUSE, STST_TILE_ROWS, STST_BLOCK_Y,
 * STST_BLOCK_X, STST_TMA), then the built-in heuristic.
 */
#pragma once
#include "Helpers.hpp"
#include "Runtime.hpp"
#include "TileKernel.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <stdexcept>
#include <string>

namespace stencil {
namespace cuda {
namespace internal {

struct LaunchPlan {
    unsigned fused_iterations; ///< k: iterations per full launch
    unsigned block_x, block_y; ///< CTA shape; block_x * CW columns are staged per tile row
    unsigned tile_h, tile_w;   ///< output tile of a full (k-iteration) launch
    unsigned halo, hpad;       ///< halo depth of a full launch, and its column-aligned version
    std::size_t smem_bytes;    ///< dynamic shared memory of a full launch
    bool use_tma;
    unsigned single_planes;    ///< planes the plan assumes are never rewritten (one tile buffer)
};

inline long env_long(const char *name, long fallback) {
    const char *v = std::getenv(name);
    return (v && *v) ? std::atol(v) : fallback;
}

/// Static properties of a device, queried once (cudaGetDeviceProperties takes milliseconds and can
/// stall behind queued work, which is far too slow for a per-call query).
inline const stst_device_info &cached_device_info(int device) {
    constexpr int max_devices = 64;
    static stst_device_info infos[max_devices];
    static bool valid[max_devices] = {};
    if (device < 0 || device >= max_devices)
        throw std::invalid_argument("StencilStream-B200: device ordinal out of range");
    if (!valid[device]) {
        STST_RT_CHECK(stst_get_device_info(device, &infos[device]));
        valid[device] = true;
    }
    return infos[device];
}

/// Column-group width: 128-bit vectors of the widest plane element, at most 4 columns.
template <typename Cell> constexpr int column_group_width() {
    // Very fat cells (mantle convection: 11 doubles): one column per thread keeps the functor within
    // 128 registers, which allows 512-thread CTAs (16 warps per SM instead of 8).
    if (sizeof(Cell) > 64) {
#if defined(STST_FAT_COLUMN_GROUP_WIDTH)
        return STST_FAT_COLUMN_GROUP_WIDTH;
#else
        return 1;
#endif
    }
    const std::size_t widest = CellLayout<Cell>::max_plane_bytes();
    if (widest >= 16)
        return 1;
    if (widest >= 8)
        return 2;
    // One-byte cells (Conway's bool): 16 columns = one 128-bit access per thread and tile row;
    // measured 801 -> 867 GCell-updates/s against 4 columns (profiles/r01_s3_sweep_conway_column_groups.log).
    if (sizeof(Cell) == 1) {
#if defined(STST_BYTE_COLUMN_GROUP_WIDTH)
        return STST_BYTE_COLUMN_GROUP_WIDTH;
#else
        return 16;
#endif
    }
#if defined(STST_LIGHT_COLUMN_GROUP_WIDTH)
    if (CellLayout<Cell>::n_planes == 1 && widest == 4)
        return STST_LIGHT_COLUMN_GROUP_WIDTH;
#endif
    return 4;
}

/// Threads per CTA the sweep kernel is compiled for (`__launch_bounds__`).
template <typename Cell> constexpr int max_threads_per_cta() {
#if defined(STST_LIGHT_MAX_THREADS)
    if (sizeof(Cell) <= 8)
        return STST_LIGHT_MAX_THREADS;
#endif
    // Cells of tens of bytes (FDTD: 32) re-read their neighbourhood from shared memory and are
    // latency-bound at 8 warps per SM; their kernels need ~150 registers, which still allows 12
    // warps: 384 threads measured +3.5 % over 256 (FDTD max_grid 99.7 -> 103.3 GCell-updates/s;
    // 320: 102.8; 512 forces spills: +1 %; profiles/r02_variants_fdtd_threads.txt).
    if (sizeof(Cell) > 16 && sizeof(Cell) <= 64) {
#if defined(STST_MID_MAX_THREADS)
        return STST_MID_MAX_THREADS;
#else
        return 384;
#endif
    }
    // Very fat cells (mantle convection, 88 bytes of doubles), one column per thread: the kernel is
    // bound by the latency of dependent fp64 chains (15 divisions per cell-iteration), so warps count.
    // 640 threads (20 warps, 92 registers, no spills) measured 9.69 against 9.17 GCell-updates/s with
    // 512 (98 registers); 768 (80 registers) 8.95 (profiles/r02_variants_convection_threads.txt).
    if (sizeof(Cell) > 64 && column_group_width<Cell>() == 1) {
#if defined(STST_FAT_MAX_THREADS)
        return STST_FAT_MAX_THREADS;
#else
        return 640;
#endif
    }
    return 256;
}

/// blockDim.x the sweep kernel is compiled for, or 0 if it is a run-time choice. Cells that use
/// lane-major tiles (TileKernel.hpp) get a fixed 64 so that their sub-row offsets are immediates.
template <typename Cell> constexpr int fixed_block_x() {
    // 256 staged columns per tile row: 64 threads x 4 columns, or 32 x 8
    return lane_major_tiles<Cell, column_group_width<Cell>()>() ? 256 / column_group_width<Cell>() : 0;
}

/// Whether every plane of `Cell` can be staged by a TMA box load.
template <typename Cell> constexpr bool tma_capable() {
    using L = CellLayout<Cell>;
    constexpr int cw = column_group_width<Cell>();
    for (std::size_t i = 0; i < L::n_planes; i++) {
        const std::size_t b = L::plane_bytes(i);
        if (!(b == 1 || b == 2 || b == 4 || b == 8))
            return false;
        if ((b * cw * 32) % 16 != 0)
            return false;
    }
    return true;
}

/**
 * Granularity (in columns) of the column halo and hence of every tile's first column. It is a
 * multiple of the column-group width; with TMA staging the byte offset of a box's first column must
 * additionally be a multiple of 16 in EVERY plane (cp.async.bulk.tensor traps otherwise), which for
 * 1- and 2-byte elements is coarser than the column group.
 */
template <typename Cell> constexpr unsigned column_alignment(bool for_tma) {
    using L = CellLayout<Cell>;
    unsigned align = unsigned(column_group_width<Cell>());
    if (for_tma) {
        for (std::size_t i = 0; i < L::n_planes; i++) {
            const unsigned need = unsigned(16 / (L::plane_bytes(i) < 16 ? L::plane_bytes(i) : 16));
            align = need > align ? need : align;
        }
    }
    return align;
}

struct TileShape {
    unsigned halo, hpad, tile_h, tile_w, rows, cols;
    std::size_t smem_bytes;
    double efficiency; ///< useful cells / staged cells
    bool feasible;
};

/// Geometry of a launch that fuses `k` iterations with the given CTA shape and shared-memory budget.
template <typename Cell>
TileShape shape_for(unsigned k, unsigned n_sub, unsigned radius, unsigned cw, unsigned col_align,
                    unsigned block_x, unsigned tile_rows_override, std::size_t smem_budget,
                    unsigned grid_h, unsigned single_planes = 0) {
    TileShape s{};
    s.halo = k * n_sub * radius;
    s.hpad = (s.halo + col_align - 1) / col_align * col_align;
    s.cols = block_x * cw;
    s.feasible = false;
    if (2 * s.hpad >= s.cols)
        return s;
    s.tile_w = s.cols - 2 * s.hpad;
    const unsigned n_buffers = (k * n_sub > 1) ? 2 : 1;
    // planes in `single_planes` are never rewritten and live in the first buffer only
    const std::size_t per_row = tile_buffer_bytes<Cell>(1, s.cols) +
                                tile_buffer_bytes<Cell>(1, s.cols, single_planes) * (n_buffers - 1);
    // tile_buffer_bytes pads every plane to 128 bytes; leave a little slack for that.
    const std::size_t usable = smem_budget > 4096 ? smem_budget - 2048 : 0;
    unsigned max_rows = unsigned(std::min<std::size_t>(usable / std::max<std::size_t>(per_row, 1), 256));
    if (max_rows <= 2 * s.halo)
        return s;
    unsigned tile_h = max_rows - 2 * s.halo;
    if (tile_rows_override > 0)
        tile_h = std::min(tile_h, tile_rows_override);
    tile_h = std::min(tile_h, std::max(grid_h, 1u));
    s.tile_h = tile_h;
    s.rows = tile_h + 2 * s.halo;
    s.smem_bytes = tile_smem_bytes<Cell>(s.rows, s.cols, n_buffers, single_planes);
    s.efficiency = double(s.tile_h) * s.tile_w / (double(s.rows) * s.cols);
    s.feasible = s.smem_bytes <= smem_budget;
    return s;
}

/**
 * Small grids: with fewer CTAs than the GPU holds at once, a launch lasts as long as ONE CTA's
 * load -> sweeps -> store sequence, however few SMs take part. Shorter tiles spread the grid over
 * just under one resident set of CTAs (a second, mostly empty wave costs more than it gains:
 * 1024^2 HotSpot, 29-row tiles 166, 13-row tiles 205, 19-row tiles — 270 CTAs on 296 slots —
 * 249 GCell-updates/s; Jacobi 340 -> 408; 2048^2 and larger are unaffected;
 * profiles/r01_s3_sweep_small_grids.log). Not below twice the halo (tile efficiency).
 *
 * Returns the tile height for `members` grids of grid_h x grid_w cells launched together (a grid
 * batch): the CTAs of all members count against the `slots` resident CTAs, so a batch of many small
 * members keeps the tall tiles `tile_h` of the unshrunk plan. A result below `tile_h` asks for the
 * shorter tile. Host-only.
 */
inline unsigned small_grid_tile_rows(unsigned tile_h, unsigned halo, unsigned tile_w,
                                     unsigned grid_h, unsigned grid_w, unsigned members,
                                     unsigned slots) {
    const unsigned long long tiles_x = (std::max(grid_w, 1u) + tile_w - 1) / tile_w;
    const unsigned long long tile_columns = tiles_x * std::max(members, 1u);
    const unsigned want_tile_rows =
        unsigned(std::max<unsigned long long>(1ull, slots * 95ull / 100ull / tile_columns));
    const unsigned shrunk =
        std::max(2 * halo, (std::max(grid_h, 1u) + want_tile_rows - 1) / want_tile_rows);
    return std::min(tile_h, shrunk);
}

/**
 * Plan launches for transition function `F` on `device`.
 *
 * The heuristic models the time per cell-iteration of a k-fused launch as
 *     sqrt((HBM bytes / k)^2 + (on-chip work)^2) / efficiency
 * with on-chip work growing with the cell size, and picks the k that minimises it among the
 * feasible ones (at most `max_k`). Two CTAs per SM are targeted so that one CTA's tile staging
 * overlaps the other's sweeps.
 */
template <typename F>
LaunchPlan make_plan(int device, unsigned grid_h, unsigned grid_w, std::size_t n_iterations,
                     unsigned fused_override, unsigned tile_rows_override,
                     unsigned single_planes = 0, unsigned members = 1) {
    using Cell = typename F::Cell;
    using L = CellLayout<Cell>;
    constexpr unsigned cw = unsigned(column_group_width<Cell>());
    constexpr unsigned n_sub = unsigned(F::n_subiterations);
    constexpr unsigned radius = unsigned(F::stencil_radius);

    const stst_device_info &info = cached_device_info(device);
    const std::size_t smem_optin = std::size_t(info.max_smem_per_block_optin);
    const std::size_t smem_sm = std::size_t(info.max_smem_per_sm);

    unsigned block_x = unsigned(env_long("STST_BLOCK_X", 0));
    if (block_x == 0) {
        // 256 staged columns for small cells, narrower tiles once a cell is tens of bytes wide.
        block_x = (sizeof(Cell) <= 16 || cw == 1) ? 64 : 32;
        if (cw > 4)
            block_x = 32;
        while (block_x > 32 && block_x * cw / 2 >= std::max(grid_w, 1u) + 2 * cw)
            block_x /= 2;
    }
    block_x = std::max(32u, block_x / 32 * 32);
    if (fixed_block_x<Cell>() != 0)
        block_x = unsigned(fixed_block_x<Cell>());
    unsigned block_y = unsigned(env_long("STST_BLOCK_Y", 0));
    if (block_y == 0)
        block_y = std::max(1u, unsigned(max_threads_per_cta<Cell>()) / block_x);
    if (block_x * block_y > unsigned(max_threads_per_cta<Cell>()))
        throw std::invalid_argument("StencilStream-B200: CTA shape exceeds the compiled thread limit");

    if (fused_override == 0)
        fused_override = unsigned(env_long("STST_FUSE", 0));
    if (tile_rows_override == 0)
        tile_rows_override = unsigned(env_long("STST_TILE_ROWS", 0));
    const unsigned ctas_per_sm = unsigned(std::max(1l, env_long("STST_CTAS_PER_SM", 2)));

    const unsigned k_cap = unsigned(
        std::min<std::size_t>(std::max<std::size_t>(n_iterations, 1), max_fused_iterations));

    // Shared memory available to one CTA if `ctas_per_sm` are to be co-resident (1 KB each is
    // reserved by the hardware).
    auto budget_for = [&](unsigned ctas) {
        std::size_t per_cta = smem_sm / ctas;
        per_cta = per_cta > 1024 ? per_cta - 1024 : 0;
        return std::min(per_cta, smem_optin);
    };

    const bool want_tma = tma_capable<Cell>() && env_long("STST_TMA", 1) != 0;
    const unsigned col_align = column_alignment<Cell>(want_tma);

    auto evaluate = [&](unsigned k, unsigned ctas) {
        return shape_for<Cell>(k, n_sub, radius, cw, col_align, block_x, tile_rows_override,
                               budget_for(ctas), grid_h, single_planes);
    };

    unsigned best_k = 0;
    TileShape best{};
    // Cost model in "HBM-byte equivalents" per cell-iteration.
    const double hbm_bytes = 2.0 * double(sizeof(Cell)) * n_sub; // one read + one write / sweep
    // on-chip work per cell-iteration, fitted to measured sweeps (profiles/r01_sweep_*.log)
    // ... and with the stencil radius (window loads and functor work per cell): without this factor
    // the radius-3 star was planned at k = 3 (793 GCell-updates/s) where k = 2 runs at 839; the
    // radius-2 star must stay at k = 4 (1174; k = 3: 1142) — profiles/r02_sweep_jacobi_r{2,3}.log
    const double onchip = (0.475 * double(sizeof(Cell)) * n_sub + 0.4 * n_sub) *
                          (1.0 + 0.28 * double(radius - 1));
    if (fused_override > 0) {
        // `fused_iterations` is an upper bound: take the deepest fusion not exceeding it whose tile
        // still fits into shared memory — split between `ctas_per_sm` CTAs or given to one,
        // whichever the cost model prefers (a feasible but tiny tile must not win by default:
        // FDTD with pass-through fits k = 3 into half an SM's shared memory with 1-row tiles).
        for (unsigned k = std::min(fused_override, k_cap); k >= 1 && best_k == 0; k--) {
            double best_cost = 0.0;
            for (unsigned ctas : {ctas_per_sm, 1u}) {
                const TileShape s = evaluate(k, ctas);
                if (!s.feasible)
                    continue;
                const double solo = (ctas == 1 && ctas_per_sm > 1) ? 1.40 : 1.0;
                const double hbm = hbm_bytes / k;
                const double cost = solo * std::sqrt(hbm * hbm + onchip * onchip) / s.efficiency;
                if (best_k == 0 || cost < best_cost) {
                    best_k = k;
                    best = s;
                    best_cost = cost;
                }
            }
        }
        if (best_k == 0)
            throw std::invalid_argument(
                "StencilStream-B200: cell type too large for a shared-memory tile");
    } else {
        double best_cost = 0.0;
        // Candidates: every depth k, with the shared memory of an SM split between `ctas_per_sm`
        // co-resident CTAs (one CTA's staging overlaps the other's sweeps) or given to a single CTA
        // (taller tiles, less halo overhead — what fat cells need). Tiles that waste most of their
        // footprint on halo are not considered, unless (tiny grids) nothing else exists.
        for (double min_efficiency : {0.35, 0.0}) {
            for (unsigned ctas : {ctas_per_sm, 1u}) {
                for (unsigned k = 1; k <= k_cap; k++) {
                    const TileShape s = evaluate(k, ctas);
                    if (!s.feasible || s.efficiency < min_efficiency)
                        continue;
                    // a lone CTA per SM cannot hide its own staging and barriers: measured 16-27 %
                    // slower at equal k for light cells, hence a 40 % handicap in this model
                    const double solo = (ctas == 1 && ctas_per_sm > 1) ? 1.40 : 1.0;
                    // HBM time and on-chip time overlap only partly: 2-norm instead of max()
                    const double hbm = hbm_bytes / k;
                    // (A launch-overhead term that pushes small grids towards deep fusion was
                    // tried and made them slower — 1024^2 HotSpot 249 -> 162 GCell-updates/s: a
                    // launch over a grid of one wave of CTAs lasts as long as ONE CTA's load ->
                    // k sweeps -> store sequence, which grows with k;
                    // profiles/r01_s3_driver_hotspot_scaling_deepfusion.csv.)
                    const double cost = solo * std::sqrt(hbm * hbm + onchip * onchip) / s.efficiency;
                    if (best_k == 0 || cost < best_cost * 0.995) {
                        best_k = k;
                        best = s;
                        best_cost = cost;
                    }
                }
            }
            if (best_k != 0)
                break;
        }
        if (best_k == 0)
            throw std::invalid_argument(
                "StencilStream-B200: cell type too large for a shared-memory tile");
    }

    // Small grids (small_grid_tile_rows): shorter tiles, unless the batch fills the GPU anyway.
    if (tile_rows_override == 0 && best.tile_h > 2 * best.halo) {
        const unsigned slots = unsigned(std::max(info.sm_count, 1)) * ctas_per_sm;
        const unsigned tile_h = small_grid_tile_rows(best.tile_h, best.halo, best.tile_w, grid_h,
                                                     grid_w, members, slots);
        if (tile_h < best.tile_h) {
            const TileShape shrunk =
                shape_for<Cell>(best_k, n_sub, radius, cw, col_align, block_x, tile_h,
                                budget_for(ctas_per_sm), grid_h, single_planes);
            if (shrunk.feasible)
                best = shrunk;
        }
    }

    LaunchPlan plan{};
    plan.fused_iterations = best_k;
    plan.block_x = block_x;
    plan.block_y = block_y;
    plan.tile_h = best.tile_h;
    plan.tile_w = best.tile_w;
    plan.halo = best.halo;
    plan.hpad = best.hpad;
    plan.smem_bytes = best.smem_bytes;
    plan.use_tma = want_tma && best.cols <= 256 && best.rows <= 256;
    plan.single_planes = single_planes;
    (void)L::n_planes;
    return plan;
}

} // namespace internal
} // namespace cuda
} // namespace stencil
