/*
 * StencilStream-B200 — the generation loop as sm_100a kernels.
 *
 * This file replaces the device side of the reference's cuda backend: `aos_stencil_kernel`
 * (reference StencilStream/cuda/StencilUpdate.hpp:227-263) and `soa_stencil_kernel` (:346-393); its
 * `scatter_kernel`/`gather_kernel` pair lives in PlaneImage.hpp. The reference launches one sweep per
 * (iteration, sub-iteration), one work-item per cell, every work-item gathering its (2r+1)^2
 * neighbourhood from global memory. Here one launch advances the grid by up to
 * `max_fused_iterations` iterations:
 *
 *   1. A CTA owns an output tile of tile_h x tile_w cells and stages the tile plus a halo of
 *      d = n_gens * n_subiterations * radius cells (columns padded to the vector width) into shared
 *      memory, one dense row-major plane per cell field, either with 128-bit cp.async or with one
 *      TMA box load per plane.
 *   2. It then runs the n_gens * n_subiterations sweeps entirely in shared memory, ping-ponging
 *      between two tile buffers; the region that is still exact shrinks by `radius` per sweep
 *      (overlapped/trapezoidal temporal blocking; the rule is the reference's own for its FPGA
 *      pipeline: StencilStream/tiling/internal/StencilUpdateKernel.hpp:79-99, :240-254, :314-320).
 *      Cells outside the global grid are re-set to `halo_value` after every sweep, exactly as the
 *      reference presents them (cuda/StencilUpdate.hpp:241-252 — the halo is never evolved).
 *      Interior tiles of radius-1 single-plane rules (Jacobi) run the sweeps in pairs, two
 *      generations per pass over shared memory (sweep_pair, paired_sweeps).
 *   3. The last sweep writes its CW-wide column groups straight to HBM with 128-bit stores.
 *
 * Inside a sweep a thread owns CW adjacent columns and walks down a run of rows, holding the
 * (2r+1) x (CW+2r) window in registers: per row it issues one vector shared-memory load per plane
 * plus 2r scalar loads for the edge columns (warp shuffles are the compile-time alternative; they
 * measured slower, see load_row), builds the user-visible `Stencil` objects in registers and calls
 * the transition function CW times. Loads of neighbour
 * fields the functor never reads are dead code and disappear.
 *
 * Tiles whose halo-extended footprint lies completely inside the grid take a path without any
 * bounds logic; only border tiles pay for halo handling.
 */
#pragma once
#include "../../Stencil.hpp"
#include "Helpers.hpp"

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <type_traits>

namespace stencil {
namespace cuda {
namespace internal {

/// Where sweep_rows writes: known at compile time (two specialised loop bodies, light functors) or
/// decided by its run-time argument (one body, heavy functors: code size).
inline constexpr int store_tile = 0, store_grid = 1, store_runtime = 2;

/**
 * Lane-major tile rows. In the natural (row-major) tile layout a thread's CW = 4 columns are one
 * 128-bit vector, which is ideal for the vector load, but the two edge columns it needs from its
 * neighbours sit 16 bytes apart from lane to lane: a 4-way bank conflict, 4 wavefronts per scalar
 * load — after all other savings, half of the kernel's shared-memory traffic (ncu: 44 % of the
 * wavefronts were conflicts, the MIO pipe 77 % busy). In the lane-major layout tile row y of a plane is
 * stored as CW sub-rows of TX = blockDim.x elements, column c at `y*cols + (c % CW)*TX + c / CW`, so
 * that lane t finds its own columns at t, TX+t, 2TX+t, 3TX+t and its neighbours' edge columns at
 * 3TX+t-1 and t+1: every access is a conflict-free scalar load (10 instead of 16 wavefronts per
 * warp and row). TMA delivers tiles in natural order, so the first sweep of a launch reads natural and
 * writes lane-major; all later sweeps read and write lane-major. The price is scalar instead of vector
 * loads/stores (6 + 4 instead of 3 + 1 instructions per row and plane), so it pays where shared memory,
 * not instruction issue, is the limit: measured +8..12 % for Jacobi (one 4-byte plane; k=6: 1603
 * GCell-updates/s) but -4 % for HotSpot (two planes, only one of which is read at neighbours) —
 * profiles/r01_sweep_light_v4_lane_major.log. Hence: scalar 4-byte cells only.
 */
template <typename Cell, int CW> constexpr bool lane_major_tiles() {
#if defined(STST_NO_LANE_MAJOR)
    return false;
#else
    using L = CellLayout<Cell>;
    if (!(CW == 4 || CW == 8))
        return false;
    // ONE evolving 4-byte plane (Jacobi's float; HotSpot's `temp`), plus any number of 4-byte planes
    // the cell type declares constant (`Cell::constant_fields`: HotSpot's `power`). Declared planes
    // pass through the sweeps untouched, i.e. they are never rewritten and so can never be
    // converted: they stay in the natural layout TMA delivers and are read with one 128-bit load per
    // row (plus, if a functor does read a neighbour's constant, the natural layout's edge loads),
    // while the evolving plane gets the conflict-free lane-major rows — for HotSpot 6 + 4 instead of
    // 12 + 4 shared-memory wavefronts per row and warp.
    const unsigned constant = constant_fields_mask<Cell>();
    unsigned evolving = 0;
    for (std::size_t i = 0; i < L::n_planes; i++) {
        if (L::plane_bytes(i) != 4)
            return false;
        if (!((constant >> i) & 1u))
            evolving++;
    }
    // Measured on B200 (profiles/r02_variants_hotspot_mixed_layout.txt): HotSpot 16384^2, mixed layout
    // 779 vs natural layout 794 GCell-updates/s — the scalar loads and stores of the lane-major plane
    // cost more issue slots than the bank conflicts they remove once `power` no longer moves. So the
    // mixed layout is opt-in (-DSTST_MIXED_LANE_MAJOR); by default only single-plane cells qualify.
  #if defined(STST_MIXED_LANE_MAJOR)
    return evolving == 1;
  #else
    return L::n_planes == 1 && evolving == 1;
  #endif
#endif
}

/// Whether plane I of a lane-major kernel is stored lane-major (the evolving plane) or natural (the
/// declared-constant ones).
template <typename Cell, std::size_t I> constexpr bool plane_is_lane_major() {
    return ((constant_fields_mask<Cell>() >> I) & 1u) == 0;
}

/// Neighbourhood acquisition strategies of sweep_rows.
inline constexpr int window_shift = 0, window_rotate = 1, window_reload = 2;

/**
 * Paired sweeps (sweep_pair): interior tiles evaluate two generations per shared-memory round trip,
 * keeping the intermediate generation in registers. Per warp and tile row that is 8 loads and 4
 * stores instead of 2 x (6 + 4), and one barrier instead of two, for 6 instead of 4 functor calls in
 * the intermediate generation: it pays where the shared-memory pipe and the barriers, not the FP
 * pipe, are the limit (Jacobi). Radius 1 only (the two register windows of a wider stencil do not
 * fit), one sub-iteration (a pair is two whole iterations), no speculative pass-through.
 * Define STST_SINGLE_SWEEPS for one sweep per round trip everywhere (the A/B variant).
 */
template <typename F, int CW, int kMode, bool kSpec> constexpr bool paired_sweeps() {
#if defined(STST_SINGLE_SWEEPS)
    return false;
#else
    return lane_major_tiles<typename F::Cell, CW>() && CellLayout<typename F::Cell>::n_planes == 1 &&
           F::stencil_radius == 1 && F::n_subiterations == 1 && kMode == window_rotate && !kSpec;
#endif
}

/// Upper bound for the number of iterations fused into one launch (sizes the TDV parameter array).
inline constexpr unsigned max_fused_iterations = 16;

/// Sub-iterations per iteration up to which speculative plane pass-through is supported.
inline constexpr unsigned max_spec_subiterations = 4;

/// Geometry of one fused launch; passed by value.
struct SweepGeometry {
    unsigned grid_h, grid_w; ///< global grid extent (rows, columns)
    int buf_row0;            ///< global row held in row 0 of every plane (slab origin, ghosts incl.)
    unsigned buf_rows;       ///< rows present in every plane: [buf_row0, buf_row0 + buf_rows)
    int out_row_lo;          ///< first global row this launch has to produce
    int out_row_hi;          ///< one past the last global row this launch has to produce
    int out2_row_lo;         ///< a second row range produced by the same launch (both boundary strips of
    int out2_row_hi;         ///< a slab in one launch); empty unless out2_row_hi > out2_row_lo
    unsigned tiles_first;    ///< number of CTAs that work on the first range (the rest: the second)
    unsigned tile_h, tile_w; ///< output tile extent
    unsigned halo;           ///< d = n_gens * n_subiterations * radius
    unsigned hpad;           ///< column halo, d rounded up to a multiple of CW
    unsigned n_gens;         ///< iterations fused into this launch (>= 1)
    unsigned tiles_x;        ///< tiles per tile-row (blockIdx.x = ty * tiles_x + tx)
    unsigned use_tma;        ///< non-zero: stage tiles with TMA box loads (maps valid)
    unsigned push;           ///< non-zero: also store result rows into neighbour slabs (HaloPush valid)
    unsigned inv_block_y;    ///< floor(2^24 / blockDim.y) + 1: row split by multiply-shift, not division
    // ---- speculative plane pass-through (kernels instantiated with kSpec only; see run_tile) ----
    unsigned keep[max_spec_subiterations]; ///< per sub-iteration: planes assumed to come out unchanged
    unsigned probe;          ///< non-zero: record per sub-iteration which planes changed at all
    unsigned *spec_flags;    ///< device words [0, S): changed per sub-iteration, [S]: violated planes
    unsigned long long iteration0; ///< global index of the first fused iteration
};

template <typename TDV> struct TdvArray {
    TDV v[max_fused_iterations];
};

/// One 128-byte TMA descriptor per plane (only read when SweepGeometry::use_tma != 0).
struct alignas(64) TensorMapSet {
    unsigned char map[max_planes][128];
};

/**
 * Halo push of a row-sharded run (see SlabUpdate.hpp): while a launch writes its result rows, the
 * rows the neighbouring slabs need as ghosts for THEIR next launch are additionally stored straight
 * into the neighbours' planes — peer memory, reached over NVLink through a peer- or IPC-mapped
 * address — so that the transfer rides along with the sweep instead of following it as a copy.
 * Global rows below `up_row_hi` go to the upper neighbour, rows from `down_row_lo` on to the lower
 * one; `*_buf_row0` is the global row held in plane row 0 of that neighbour's planes.
 */
struct HaloPush {
    PlaneSet up, down;
    int up_buf_row0, down_buf_row0;
    int up_row_hi;   ///< INT_MIN if there is nothing to push upwards
    int down_row_lo; ///< INT_MAX if there is nothing to push downwards
    // Completion signal, raised by the launch itself: the CTA that finishes LAST (atomic ticket in
    // own device memory) stores `flag_value` into the neighbours' flag words once every CTA's
    // pushed rows are visible system-wide. Saves the two one-thread flag kernels (and their launch
    // latency on the critical path between neighbouring slabs) that used to follow a boundary launch.
    unsigned *ticket;      ///< device word, zero between launches; nullptr: the launch raises nothing
    unsigned *flag_up;     ///< flag word inside the upper neighbour's slab (or nullptr)
    unsigned *flag_down;   ///< flag word inside the lower neighbour's slab (or nullptr)
    unsigned flag_value;
};

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------

template <typename T, int N> struct alignas((sizeof(T) * N) % 16 == 0 ? 16
                                            : (sizeof(T) * N) % 8 == 0 ? 8
                                            : (sizeof(T) * N) % 4 == 0 ? 4
                                                                       : alignof(T)) Pack {
    T v[N];
};

template <typename T>
inline constexpr bool is_shuffleable_v = std::is_trivially_copyable_v<T> &&
                                         (sizeof(T) == 1 || sizeof(T) == 2 || sizeof(T) == 4 ||
                                          sizeof(T) == 8);

// ---- shared-memory accounting (host and device; used by the planner) ---------------------------

/// Unused bytes in front of the first and behind the last tile buffer: edge-column loads of the
/// first/last thread of a tile row reach up to `radius` elements beyond their row, and must stay
/// inside the CTA's dynamic shared memory (what they fetch there is never used for exact cells).
inline constexpr unsigned tile_guard_bytes = 128;

/// Bytes of one tile buffer (each plane padded to 128 bytes) that holds every plane except those
/// in `without_planes`.
template <typename Cell>
STST_HD inline std::size_t tile_buffer_bytes(unsigned tile_rows, unsigned tile_cols,
                                             unsigned without_planes = 0) {
    using L = CellLayout<Cell>;
    std::size_t total = 0;
    for (std::size_t i = 0; i < L::n_planes; i++) {
        if ((without_planes >> i) & 1u)
            continue;
        std::size_t b = std::size_t(tile_rows) * tile_cols * L::plane_bytes(i);
        total += (b + 127) / 128 * 128;
    }
    return total;
}

/// Dynamic shared memory of a CTA: guard, `n_buffers` tile buffers, guard. Planes in
/// `single_planes` (never rewritten, see run_tile) exist in the first buffer only.
template <typename Cell>
STST_HD inline std::size_t tile_smem_bytes(unsigned tile_rows, unsigned tile_cols,
                                           unsigned n_buffers, unsigned single_planes = 0) {
    return tile_buffer_bytes<Cell>(tile_rows, tile_cols) +
           tile_buffer_bytes<Cell>(tile_rows, tile_cols, single_planes) * (n_buffers - 1) +
           2 * tile_guard_bytes;
}

#if defined(__CUDACC__)

template <typename To, typename From> __device__ __forceinline__ To bit_cast_dev(From const &f) {
    static_assert(sizeof(To) >= sizeof(From));
    To t{};
    memcpy(&t, &f, sizeof(From));
    return t;
}

template <typename T> __device__ __forceinline__ T from_bits(unsigned long long bits) {
    T t;
    memcpy(&t, &bits, sizeof(T));
    return t;
}

/// Value of `v` held by the lane `delta` below (up) / above (down) the caller.
template <typename T> __device__ __forceinline__ T shuffle_from_lower_lane(T const &v) {
    if constexpr (sizeof(T) <= 4) {
        unsigned bits = bit_cast_dev<unsigned>(v);
        bits = __shfl_up_sync(0xffffffffu, bits, 1);
        return from_bits<T>(bits);
    } else {
        unsigned long long bits = bit_cast_dev<unsigned long long>(v);
        bits = __shfl_up_sync(0xffffffffu, bits, 1);
        return from_bits<T>(bits);
    }
}

template <typename T> __device__ __forceinline__ T shuffle_from_upper_lane(T const &v) {
    if constexpr (sizeof(T) <= 4) {
        unsigned bits = bit_cast_dev<unsigned>(v);
        bits = __shfl_down_sync(0xffffffffu, bits, 1);
        return from_bits<T>(bits);
    } else {
        unsigned long long bits = bit_cast_dev<unsigned long long>(v);
        bits = __shfl_down_sync(0xffffffffu, bits, 1);
        return from_bits<T>(bits);
    }
}

template <int Bytes>
__device__ __forceinline__ void cp_async_group(void *smem_dst, const void *gmem_src) {
    unsigned saddr = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    if constexpr (Bytes % 16 == 0) {
#pragma unroll
        for (int o = 0; o < Bytes; o += 16) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(saddr + o),
                         "l"(static_cast<const char *>(gmem_src) + o)
                         : "memory");
        }
    } else if constexpr (Bytes == 8) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(saddr), "l"(gmem_src)
                     : "memory");
    } else {
        static_assert(Bytes == 4);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(saddr), "l"(gmem_src)
                     : "memory");
    }
}

__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.wait_all;\n" ::: "memory");
}

// ---- mbarrier + TMA (cp.async.bulk.tensor) -----------------------------------------------------

__device__ __forceinline__ void mbarrier_init(unsigned long long *bar, unsigned count) {
    unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(addr), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_mbarrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}

__device__ __forceinline__ void mbarrier_arrive_expect_tx(unsigned long long *bar, unsigned bytes) {
    unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(addr), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbarrier_wait_parity(unsigned long long *bar, unsigned parity) {
    unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    unsigned done = 0;
    do {
        asm volatile("{\n"
                     ".reg .pred p;\n"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
                     "selp.u32 %0, 1, 0, p;\n"
                     "}\n"
                     : "=r"(done)
                     : "r"(addr), "r"(parity)
                     : "memory");
    } while (!done);
}

__device__ __forceinline__ void tma_load_2d(void *smem_dst, const void *tensor_map, int x, int y,
                                            unsigned long long *bar) {
    unsigned dst = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    unsigned mbar = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
                 " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(dst),
                 "l"(tensor_map), "r"(mbar), "r"(x), "r"(y)
                 : "memory");
}

// ------------------------------------------------------------------------------------------------
// shared-memory tile bookkeeping
// ------------------------------------------------------------------------------------------------

template <typename Cell> struct TileView {
    using L = CellLayout<Cell>;
    unsigned char *base;
    unsigned rows, cols; // THH, TWH
    unsigned plane_off[L::n_planes];

    __device__ __forceinline__ TileView(unsigned char *base, unsigned rows, unsigned cols)
        : base(base), rows(rows), cols(cols) {
        unsigned off = 0;
#pragma unroll
        for (unsigned i = 0; i < L::n_planes; i++) {
            plane_off[i] = off;
            unsigned b = rows * cols * unsigned(L::plane_bytes(i));
            off += (b + 127u) / 128u * 128u;
        }
    }

    /// View whose plane offsets the caller fills in (run_tile with plane pass-through).
    __device__ __forceinline__ TileView(unsigned char *base, unsigned rows, unsigned cols, int)
        : base(base), rows(rows), cols(cols) {}

    template <std::size_t I> __device__ __forceinline__ typename L::template plane_t<I> *plane() const {
        return reinterpret_cast<typename L::template plane_t<I> *>(base + plane_off[I]);
    }
};

// ------------------------------------------------------------------------------------------------
// tile staging: HBM -> shared memory
// ------------------------------------------------------------------------------------------------

/**
 * Fill tile buffer `tile` with the grid cells at global rows [gy0, gy0 + rows) and global columns
 * [gx0, gx0 + cols); positions outside the global grid receive `halo_value`.
 * Ends with a CTA-wide barrier.
 */
template <typename Cell, int CW, bool kInterior>
__device__ __forceinline__ void stage_tile(TileView<Cell> const &tile, PlaneSet const &src,
                                           TensorMapSet const &maps, SweepGeometry const &geo,
                                           Cell const &halo_value, int gy0, int gx0,
                                           unsigned long long *mbar) {
    using L = CellLayout<Cell>;
    const int c0 = int(threadIdx.x) * CW;
    const int gx = gx0 + c0;

    if (geo.use_tma) {
        // One box load per plane, issued by a single thread; out-of-grid elements arrive as zeros
        // and are patched below (border tiles only).
        if (threadIdx.x == 0 && threadIdx.y == 0) {
            unsigned total = 0;
            for_each_plane<Cell>([&](auto I) {
                total += tile.rows * tile.cols * unsigned(sizeof(typename L::template plane_t<I>));
            });
            mbarrier_arrive_expect_tx(mbar, total);
            for_each_plane<Cell>([&](auto I) {
                tma_load_2d(tile.template plane<I>(), &maps.map[I][0], gx0, gy0 - geo.buf_row0,
                            mbar);
            });
        }
        // Every thread observes the phase completion itself (the acquire that makes the
        // async-proxy writes of the TMA unit visible to it). Letting one warp poll and releasing the
        // others through bar.sync was measured too: 14 % of the convection kernel's stall samples
        // sit in this loop, but its rate moved by 1 % (9.2 -> 9.3) — nothing else could have used
        // those issue slots — so the conservative form stays.
        mbarrier_wait_parity(mbar, 0);
        if constexpr (!kInterior) {
            for (int row = int(threadIdx.y); row < int(tile.rows); row += int(blockDim.y)) {
                const int gy = gy0 + row;
                const bool row_in = gy >= 0 && gy < int(geo.grid_h);
                for_each_plane<Cell>([&](auto I) {
                    auto *s = tile.template plane<I>() + std::size_t(row) * tile.cols + c0;
#pragma unroll
                    for (int i = 0; i < CW; i++) {
                        const bool in = row_in && (gx + i) >= 0 && (gx + i) < int(geo.grid_w);
                        if (!in)
                            s[i] = L::template get<I>(halo_value);
                    }
                });
            }
            __syncthreads();
        }
        return;
    }

    for_each_plane<Cell>([&](auto I) {
        using T = typename L::template plane_t<I>;
        T *sp = tile.template plane<I>();
        const T *gp = static_cast<const T *>(src.base[I]);
        const unsigned long long pitch = src.pitch[I];
        for (int row = int(threadIdx.y); row < int(tile.rows); row += int(blockDim.y)) {
            const int gy = gy0 + row;
            T *s = sp + std::size_t(row) * tile.cols + c0;
            const T *g = gp + (long long)(gy - geo.buf_row0) * (long long)pitch + gx;
            if constexpr (kInterior) {
                if constexpr ((sizeof(T) * CW) % 16 == 0 || sizeof(T) * CW == 8 ||
                              sizeof(T) * CW == 4) {
                    cp_async_group<int(sizeof(T)) * CW>(s, g);
                } else {
                    *reinterpret_cast<Pack<T, CW> *>(s) = *reinterpret_cast<const Pack<T, CW> *>(g);
                }
            } else {
                // Inside the grid AND inside the planes that are really mapped: the last tile row of
                // a slab launch may reach below the slab's ghost rows (the tile height does not
                // divide the row range); what would be read there is never used for a stored cell.
                const bool row_in = gy >= 0 && gy < int(geo.grid_h) &&
                                    unsigned(gy - geo.buf_row0) < geo.buf_rows;
                if (row_in && gx >= 0 && gx + CW <= int(geo.grid_w)) {
                    *reinterpret_cast<Pack<T, CW> *>(s) = *reinterpret_cast<const Pack<T, CW> *>(g);
                } else {
#pragma unroll
                    for (int i = 0; i < CW; i++) {
                        const bool in = row_in && (gx + i) >= 0 && (gx + i) < int(geo.grid_w);
                        s[i] = in ? g[i] : L::template get<I>(halo_value);
                    }
                }
            }
        }
    });
    if constexpr (kInterior)
        cp_async_wait_all();
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// one sweep (one sub-iteration) over the still-exact part of a tile
// ------------------------------------------------------------------------------------------------

/**
 * Apply sub-iteration `SUB` of `tf` to tile rows [row_lo, row_hi) of `in`, writing either into the
 * tile buffer `out` or — if `to_global` — into the destination planes in HBM.
 *
 * \tparam kMode How a thread obtains the (2r+1) x (CW+2r) neighbourhood of its column group:
 *               window_shift  — keep it in registers, load one new row per step, shift by moves;
 *               window_rotate — same, but the row loop is unrolled (2r+1)-fold so that the window
 *                               rotates by register renaming (light-weight cells only: code size);
 *               window_reload — re-read all (2r+1) rows from shared memory for every output row, with
 *                               plain loads instead of shuffles. Nothing stays live between rows, so
 *                               only fields the functor really reads cost registers and loads: the
 *                               choice for fat cells (tens of bytes), where a resident window of whole
 *                               cells exceeds the register file.
 */
/// Per-thread bookkeeping of speculative plane pass-through (kSpec kernels).
struct SpecTrack {
    unsigned keep;     ///< planes this sweep must not store into the tile (they pass through)
    unsigned probe;    ///< non-zero: collect `changed`
    unsigned changed;  ///< planes whose value differed from the centre cell's in this sweep
    unsigned violated; ///< kept planes whose value differed: the speculation was wrong
};

/// Bitwise inequality of two plane values.
template <typename T> __device__ __forceinline__ bool bits_differ(T const &a, T const &b) {
    if constexpr (sizeof(T) == 1 || sizeof(T) == 2 || sizeof(T) == 4) {
        return bit_cast_dev<unsigned>(a) != bit_cast_dev<unsigned>(b);
    } else if constexpr (sizeof(T) == 8) {
        return bit_cast_dev<unsigned long long>(a) != bit_cast_dev<unsigned long long>(b);
    } else {
        const unsigned char *pa = reinterpret_cast<const unsigned char *>(&a);
        const unsigned char *pb = reinterpret_cast<const unsigned char *>(&b);
        bool d = false;
#pragma unroll
        for (unsigned i = 0; i < sizeof(T); i++)
            d |= pa[i] != pb[i];
        return d;
    }
}

/// Rows [y_begin, y_end) of the sweep rows [row_lo, row_hi) that row group threadIdx.y works on:
/// balanced to within one row, group g gets rows [n*g/G, n*(g+1)/G).
/// x / blockDim.y == (x * inv_block_y) >> 24 (64-bit product) exactly for x < 2^16 and
/// blockDim.y <= 32: the error term x / 2^24 stays below 1 / blockDim.y. A run-time integer
/// division costs ~20 instructions, twice per sweep and warp — 7 % of all instructions of the
/// Jacobi kernel before this.
__device__ __forceinline__ void row_group_rows(SweepGeometry const &geo, int row_lo, int row_hi,
                                               int &y_begin, int &y_end) {
    const unsigned n_rows = unsigned(row_hi - row_lo);
    y_begin = row_lo + int((std::uint64_t(n_rows * threadIdx.y) * geo.inv_block_y) >> 24);
    y_end = row_lo + int((std::uint64_t(n_rows * (threadIdx.y + 1u)) * geo.inv_block_y) >> 24);
}

/// Every cell an interior tile computes — exact or not — lies at least one cell inside the grid
/// (fused_sweep_kernel admits a tile to that path only if its staged footprint does). Telling the
/// compiler lets it fold the border tests functors make on `stencil.id` / `stencil.grid_range`
/// (HotSpot's adiabatic borders, reference examples/hotspot/hotspot.cpp:77-87: four compares and
/// four selects per cell) out of the interior path; border tiles keep them.
__device__ __forceinline__ void assume_inside_grid(std::size_t id_r, std::size_t id_c,
                                                   std::size_t range_r, std::size_t range_c) {
    __builtin_assume(id_r != 0);
    __builtin_assume(id_r != range_r - 1);
    __builtin_assume(id_r < range_r - 1);
    __builtin_assume(id_r + 1 < range_r);
    __builtin_assume(id_c != 0);
    __builtin_assume(id_c != range_c - 1);
    __builtin_assume(id_c < range_c - 1);
    __builtin_assume(id_c + 1 < range_c);
}

/**
 * Store the CW cells `result` of tile row `y` (global row `gy`) that thread threadIdx.x computed:
 * into the tile buffer `out`, or — if `to_global` — into the destination planes in HBM (own column
 * groups and rows of the launch only) and, with a halo push, into the neighbour slabs. Planes in
 * `keep` pass through and are not stored into the tile (`out` aliases the input for them).
 */
template <typename Cell, int CW, bool kInterior, bool kOutLaneMajor, int kTX>
__device__ __forceinline__ void
store_cells(Cell const (&result)[CW], int y, int gy, bool to_global, unsigned keep,
            TileView<Cell> const &out, PlaneSet const &dst, HaloPush const &push,
            SweepGeometry const &geo, int gx0, int out_lo, int out_hi) {
    using L = CellLayout<Cell>;
    const int cols = int(out.cols);
    const int c0 = int(threadIdx.x) * CW;
    const int tx = int(threadIdx.x), TX = kTX ? kTX : int(blockDim.x);
    if (!to_global) {
        for_each_plane<Cell>([&](auto I) {
            using T = typename L::template plane_t<I>;
            if ((keep >> I) & 1u)
                return; // passes through: `out` aliases `in` for this plane
            if constexpr (kOutLaneMajor && plane_is_lane_major<Cell, I>()) {
                T *o = out.template plane<I>() + y * cols + tx;
#pragma unroll
                for (int i = 0; i < CW; i++)
                    o[i * TX] = L::template get<I>(result[i]);
            } else {
                Pack<T, CW> q;
#pragma unroll
                for (int i = 0; i < CW; i++)
                    q.v[i] = L::template get<I>(result[i]);
                *reinterpret_cast<Pack<T, CW> *>(out.template plane<I>() + y * cols + c0) = q;
            }
        });
    } else {
        // Only the tile's own column groups are exact after the last sweep.
        const bool own_group = c0 >= int(geo.hpad) && c0 < int(geo.hpad + geo.tile_w);
        if (!own_group)
            return;
        const int gxg = gx0 + c0;
        if constexpr (!kInterior) {
            if (gy < out_lo || gy >= out_hi || gy >= int(geo.grid_h))
                return;
        }
        auto store_row = [&](PlaneSet const &planes, int buf_row0) {
            for_each_plane<Cell>([&](auto I) {
                using T = typename L::template plane_t<I>;
                T *g = static_cast<T *>(planes.base[I]) +
                       (long long)(gy - buf_row0) * (long long)planes.pitch[I] + gxg;
                if (kInterior || gxg + CW <= int(geo.grid_w)) {
                    Pack<T, CW> q;
#pragma unroll
                    for (int i = 0; i < CW; i++)
                        q.v[i] = L::template get<I>(result[i]);
                    *reinterpret_cast<Pack<T, CW> *>(g) = q;
                } else {
#pragma unroll
                    for (int i = 0; i < CW; i++) {
                        if (gxg + i < int(geo.grid_w))
                            g[i] = L::template get<I>(result[i]);
                    }
                }
            });
        };
        store_row(dst, geo.buf_row0);
        if (geo.push) {
            if (gy < push.up_row_hi)
                store_row(push.up, push.up_buf_row0);
            if (gy >= push.down_row_lo)
                store_row(push.down, push.down_buf_row0);
        }
    }
}

template <typename F, int CW, bool kInterior, int kMode, int kStore, bool kInLaneMajor,
          bool kOutLaneMajor, int kTX, bool kSpec, std::size_t SUB>
__device__ __forceinline__ void
sweep_rows(F const &tf, typename F::Cell const &halo_value,
           typename F::TimeDependentValue const &tdv, std::size_t iteration,
           TileView<typename F::Cell> const &in, TileView<typename F::Cell> const &out,
           bool to_global_arg, PlaneSet const &dst, HaloPush const &push, SweepGeometry const &geo,
           int gy0, int gx0, int row_lo, int row_hi, int out_lo, int out_hi, SpecTrack &spec) {
    using Cell = typename F::Cell;
    using TDV = typename F::TimeDependentValue;
    using L = CellLayout<Cell>;
    using StencilImpl = Stencil<Cell, F::stencil_radius, TDV>;
    constexpr int R = int(F::stencil_radius);
    constexpr int D = 2 * R + 1;
    constexpr int WC = CW + 2 * R;
    // any radius is legal (the reference's backends accept any); the unclamped edge-column loads
    // reach R elements beyond a tile row, which the guard bytes must cover
    static_assert(std::size_t(R) * L::max_plane_bytes() <= tile_guard_bytes,
                  "stencil radius times the widest field exceeds the shared-memory guard");

    const int cols = int(in.cols);
    const int c0 = int(threadIdx.x) * CW;
    const int lane = int(threadIdx.x) & 31;
    // kTX != 0: blockDim.x is known at compile time, lane-major offsets become immediates
    const int tx = int(threadIdx.x), TX = kTX ? kTX : int(blockDim.x);
    const bool to_global = kStore == store_runtime ? to_global_arg : (kStore == store_grid);

    // Split the rows of this sweep over the blockDim.y row groups (uniform per warp).
    int y_begin, y_end;
    row_group_rows(geo, row_lo, row_hi, y_begin, y_end);
    if (y_begin >= y_end)
        return;

    // window_reload may produce several output rows per step from ONE (D + rows - 1)-row window: the
    // rows share D - 1 window rows (fewer shared-memory loads), and their functor evaluations are
    // independent instruction streams the scheduler can interleave (latency-bound fat functors).
#if defined(STST_RELOAD_ROWS)
    constexpr int RPS = (kMode == window_reload) ? STST_RELOAD_ROWS : 1;
#else
    constexpr int RPS = 1;
#endif
    constexpr int DW = D + RPS - 1;
    Cell win[DW][WC];

    // Load tile row `row`, columns [c0 - R, c0 + CW + R), into `w`.
    auto load_row = [&](Cell(&w)[WC], int row) {
        for_each_plane<Cell>([&](auto I) {
            using T = typename L::template plane_t<I>;
            const T *rp = in.template plane<I>() + row * cols;
            if constexpr (kInLaneMajor && plane_is_lane_major<Cell, I>()) {
                // see lane_major_tiles(): all conflict-free scalar loads
                const T *q = rp + tx;
#pragma unroll
                for (int i = 0; i < CW; i++)
                    L::template get<I>(w[R + i]) = q[i * TX];
                // column c0 - j is element (CW - j % CW) % CW of the group ceil(j / CW) to the left,
                // column c0 + CW - 1 + j element (j - 1) % CW of the group (j - 1) / CW + 1 to the right
#pragma unroll
                for (int j = 1; j <= R; j++) {
                    L::template get<I>(w[R - j]) =
                        q[((CW - j % CW) % CW) * TX - (j + CW - 1) / CW];
                    L::template get<I>(w[R + CW - 1 + j]) = q[((j - 1) % CW) * TX + (j - 1) / CW + 1];
                }
                return;
            }
            const Pack<T, CW> p = *reinterpret_cast<const Pack<T, CW> *>(rp + c0);
#pragma unroll
            for (int i = 0; i < CW; i++)
                L::template get<I>(w[R + i]) = p.v[i];
#pragma unroll
            for (int j = 1; j <= R; j++) {
                T left, right;
                // The 2r edge columns of a thread's window belong to its lane neighbours. They can be
                // fetched by warp shuffle (plus a load for the first/last lane of the warp) or by two
                // plain scalar shared-memory loads at constant offsets from the vector load's address.
                // Measured on B200 (profiles/r01_variants_shuffle_vs_lds_cw4_vs_cw8.log): the plain
                // loads win by 17-20 % (Jacobi k=4 1154 -> 1378, HotSpot 548 -> 639 GCell-updates/s) —
                // a shuffle occupies the same MIO issue slot as an LDS, and the shuffle variant needs
                // the predicated fix-up loads on top. Define STST_EDGE_SHUFFLES for the shuffle variant.
#if defined(STST_EDGE_SHUFFLES)
                constexpr bool use_shuffles = true;
#else
                constexpr bool use_shuffles = false;
#endif
                if constexpr (is_shuffleable_v<T> && kMode != window_reload && use_shuffles) {
                    static_assert(R <= CW || sizeof(T) == 0,
                                  "edge shuffles reach one lane to each side only");
                    left = shuffle_from_lower_lane(p.v[CW - j]);
                    right = shuffle_from_upper_lane(p.v[j - 1]);
                    if (lane == 0)
                        left = rp[c0 - j];
                    if (lane == 31)
                        right = rp[c0 + CW - 1 + j];
                } else {
                    // constant offsets from the vector load's address; see tile_guard_bytes
                    left = rp[c0 - j];
                    right = rp[c0 + CW - 1 + j];
                }
                L::template get<I>(w[R - j]) = left;
                L::template get<I>(w[R + CW - 1 + j]) = right;
            }
        });
    };

    // Compute the CW cells of tile row `y` from the window whose top row sits in slot `top`.
    auto compute_row = [&](auto top_c, int y) {
        constexpr int top = decltype(top_c)::value;
        const int gy = gy0 + y;
        Cell result[CW];
#pragma unroll
        for (int i = 0; i < CW; i++) {
            const int gx = gx0 + c0 + i;
            bool in_grid = true;
            if constexpr (!kInterior) {
                in_grid = gy >= 0 && gy < int(geo.grid_h) && gx >= 0 && gx < int(geo.grid_w);
            }
            if (in_grid) {
                const std::size_t id_r = std::size_t(unsigned(gy)), id_c = std::size_t(unsigned(gx));
                const std::size_t range_r = geo.grid_h, range_c = geo.grid_w;
                if constexpr (kInterior)
                    assume_inside_grid(id_r, id_c, range_r, range_c);
                StencilImpl st(sycl::id<2>(id_r, id_c), sycl::range<2>(range_r, range_c), iteration,
                               SUB, tdv);
#pragma unroll
                for (int sr = 0; sr < D; sr++) {
#pragma unroll
                    for (int sc = 0; sc < D; sc++) {
                        st[sycl::id<2>(sr, sc)] = win[(top + sr) % DW][i + sc];
                    }
                }
                result[i] = tf(st);
            } else {
                result[i] = halo_value;
            }
        }

        if constexpr (kSpec) {
            // Which planes really changed? For a field the functor passes through untouched the
            // compiler folds the comparison away; for the others it is one compare per cell.
            for_each_plane<Cell>([&](auto I) {
                const bool kept = (spec.keep >> I) & 1u;
                if (kept || spec.probe) {
                    bool differs = false;
#pragma unroll
                    for (int i = 0; i < CW; i++) {
                        bool in_grid = true;
                        if constexpr (!kInterior) {
                            const int gx = gx0 + c0 + i;
                            in_grid = gy >= 0 && gy < int(geo.grid_h) && gx >= 0 && gx < int(geo.grid_w);
                        }
                        if (in_grid)
                            differs |= bits_differ(L::template get<I>(result[i]),
                                                   L::template get<I>(win[(top + R) % DW][R + i]));
                    }
                    if (differs) {
                        spec.changed |= 1u << I;
                        if (kept)
                            spec.violated |= 1u << I;
                    }
                }
            });
        }

        store_cells<Cell, CW, kInterior, kOutLaneMajor, kTX>(result, y, gy, to_global,
                                                             kSpec ? spec.keep : 0u, out, dst, push,
                                                             geo, gx0, out_lo, out_hi);
    };

    // Prime the window with the D-1 rows above/around the first row.
    if constexpr (kMode != window_reload) {
#pragma unroll
        for (int j = 0; j < D - 1; j++)
            load_row(win[j], y_begin - R + j);
    }

    if constexpr (kMode == window_reload) {
        int y = y_begin;
        if constexpr (RPS > 1) {
            for (; y + RPS <= y_end; y += RPS) {
#pragma unroll
                for (int j = 0; j < DW; j++)
                    load_row(win[j], y - R + j);
                [&]<int... Us>(std::integer_sequence<int, Us...>) {
                    (compute_row(std::integral_constant<int, Us>{}, y + Us), ...);
                }(std::make_integer_sequence<int, RPS>{});
            }
        }
        for (; y < y_end; y++) {
#pragma unroll
            for (int j = 0; j < D; j++)
                load_row(win[j], y - R + j);
            compute_row(std::integral_constant<int, 0>{}, y);
        }
    } else if constexpr (kMode == window_rotate) {
        // full groups of D rows without per-row guards (a guard is a branch plus a convergence
        // barrier pair per row), then one guarded group for the remaining < D rows
        int y = y_begin;
        for (; y + D <= y_end; y += D) {
            [&]<int... Us>(std::integer_sequence<int, Us...>) {
                (
                    [&] {
                        load_row(win[(Us + D - 1) % D], y + Us + R);
                        compute_row(std::integral_constant<int, Us>{}, y + Us);
                    }(),
                    ...);
            }(std::make_integer_sequence<int, D>{});
        }
        if (y < y_end) {
            [&]<int... Us>(std::integer_sequence<int, Us...>) {
                (
                    [&] {
                        if (y + Us < y_end) {
                            load_row(win[(Us + D - 1) % D], y + Us + R);
                            compute_row(std::integral_constant<int, Us>{}, y + Us);
                        }
                    }(),
                    ...);
            }(std::make_integer_sequence<int, D>{});
        }
    } else {
        for (int y = y_begin; y < y_end; y++) {
            load_row(win[D - 1], y + R);
            compute_row(std::integral_constant<int, 0>{}, y);
#pragma unroll
            for (int j = 0; j < D - 1; j++) {
#pragma unroll
                for (int i = 0; i < WC; i++)
                    win[j][i] = win[j + 1][i];
            }
        }
    }
}

/**
 * Two generations per pass over tile rows [row_lo, row_hi) of an interior tile (see paired_sweeps):
 * read generation g from `in`, evaluate generation g+1 in registers and write generation g+2 into
 * the lane-major tile buffer `out` (kStore == store_tile) or into HBM (kStore == store_grid).
 *
 * The row group that produces rows [y_begin, y_end) of g+2 loads rows y_begin-2 .. y_end+1 of g,
 * columns c0-2 .. c0+CW+1, and evaluates rows y_begin-1 .. y_end of g+1, columns c0-1 .. c0+CW:
 * the edge columns of g+1 are recomputed by both neighbouring threads (shuffles measured slower,
 * see load_row of sweep_rows), the end rows by both neighbouring row groups. Both windows rotate by
 * the same three-fold unroll as window_rotate. The rows of g read here lie inside
 * [row_lo - 2, row_hi + 2), which the previous sweep left exact; the columns reach two elements past
 * the thread's own, which stays inside the tile row in the lane-major layout and inside
 * tile_guard_bytes in the natural one — no further than the edge loads of two single sweeps.
 */
template <int V> using int_c = std::integral_constant<int, V>;

template <typename F, int CW, int kStore, bool kInLaneMajor, int kTX>
__device__ __forceinline__ void
sweep_pair(F const &tf, typename F::TimeDependentValue const &tdv1,
           typename F::TimeDependentValue const &tdv2, std::size_t iteration,
           TileView<typename F::Cell> const &in, TileView<typename F::Cell> const &out,
           PlaneSet const &dst, HaloPush const &push, SweepGeometry const &geo, int gy0, int gx0,
           int row_lo, int row_hi, int out_lo, int out_hi) {
    using Cell = typename F::Cell;
    using TDV = typename F::TimeDependentValue;
    using L = CellLayout<Cell>;
    using T = typename L::template plane_t<0>;
    using StencilImpl = Stencil<Cell, 1, TDV>;
    static_assert(L::n_planes == 1 && F::stencil_radius == 1 && CW % 2 == 0);
    constexpr int W0 = CW + 4, W1 = CW + 2; // window widths of generations g and g+1

    const int cols = int(in.cols);
    const int c0 = int(threadIdx.x) * CW;
    const int tx = int(threadIdx.x), TX = kTX ? kTX : int(blockDim.x);

    int y_begin, y_end;
    row_group_rows(geo, row_lo, row_hi, y_begin, y_end);
    if (y_begin >= y_end)
        return;

    Cell w0[3][W0]; // generation g:   row r in slot (r - y_begin + 2) % 3, column c0 - 2 + i in [i]
    Cell w1[3][W1]; // generation g+1: row r in slot (r - y_begin + 1) % 3, column c0 - 1 + i in [i]

    // Row `row` of generation g into slot S of w0.
    auto load_row = [&](auto slot_c, int row) {
        Cell(&w)[W0] = w0[decltype(slot_c)::value];
        const T *rp = in.template plane<0>() + row * cols;
        if constexpr (kInLaneMajor) {
            // own columns at tx + i*TX (lane_major_tiles); c0-2 and c0-1 are elements CW-2 and CW-1
            // of the group to the left, c0+CW and c0+CW+1 elements 0 and 1 of the group to the right
            const T *q = rp + tx;
#pragma unroll
            for (int i = 0; i < CW; i++)
                L::template get<0>(w[2 + i]) = q[i * TX];
            L::template get<0>(w[0]) = q[(CW - 2) * TX - 1];
            L::template get<0>(w[1]) = q[(CW - 1) * TX - 1];
            L::template get<0>(w[CW + 2]) = q[1];
            L::template get<0>(w[CW + 3]) = q[TX + 1];
        } else {
            // natural layout: the edge columns are 8-byte aligned pairs
            const Pack<T, CW> p = *reinterpret_cast<const Pack<T, CW> *>(rp + c0);
            const Pack<T, 2> l = *reinterpret_cast<const Pack<T, 2> *>(rp + c0 - 2);
            const Pack<T, 2> r = *reinterpret_cast<const Pack<T, 2> *>(rp + c0 + CW);
#pragma unroll
            for (int i = 0; i < CW; i++)
                L::template get<0>(w[2 + i]) = p.v[i];
            L::template get<0>(w[0]) = l.v[0];
            L::template get<0>(w[1]) = l.v[1];
            L::template get<0>(w[CW + 2]) = r.v[0];
            L::template get<0>(w[CW + 3]) = r.v[1];
        }
    };

    // `tf` for the cell at global (gy, gx) whose neighbourhood is nb(sr, sc), sr, sc in [0, 3).
    auto apply = [&](auto inside_c, auto const &nb, int gy, int gx, std::size_t it,
                     TDV const &tdv) -> Cell {
        const std::size_t id_r = std::size_t(unsigned(gy)), id_c = std::size_t(unsigned(gx));
        const std::size_t range_r = geo.grid_h, range_c = geo.grid_w;
        if constexpr (decltype(inside_c)::value)
            assume_inside_grid(id_r, id_c, range_r, range_c);
        StencilImpl st(sycl::id<2>(id_r, id_c), sycl::range<2>(range_r, range_c), it, 0, tdv);
#pragma unroll
        for (int sr = 0; sr < 3; sr++) {
#pragma unroll
            for (int sc = 0; sc < 3; sc++)
                st[sycl::id<2>(sr, sc)] = nb(sr, sc);
        }
        return tf(st);
    };

    // Row y of generation g+1 into slot S of w1, from the rows of w0 starting at slot TOP.
    auto first = [&](auto top_c, auto slot_c, int y) {
        constexpr int top = decltype(top_c)::value;
#pragma unroll
        for (int i = 0; i < W1; i++) {
            auto nb = [&](int sr, int sc) -> Cell const & { return w0[(top + sr) % 3][i + sc]; };
            const int gx = gx0 + c0 - 1 + i;
            // The edge columns c0 - 1 and c0 + CW of the first and last thread may lie on the grid's
            // border (they are never exact); all other cells are inside, as in sweep_rows.
            if (i == 0 || i == W1 - 1)
                w1[decltype(slot_c)::value][i] =
                    apply(std::false_type{}, nb, gy0 + y, gx, iteration, tdv1);
            else
                w1[decltype(slot_c)::value][i] =
                    apply(std::true_type{}, nb, gy0 + y, gx, iteration, tdv1);
        }
    };

    // Row y of generation g+2 from the rows of w1 starting at slot TOP, stored.
    auto second = [&](auto top_c, int y) {
        constexpr int top = decltype(top_c)::value;
        const int gy = gy0 + y;
        Cell result[CW];
#pragma unroll
        for (int i = 0; i < CW; i++) {
            auto nb = [&](int sr, int sc) -> Cell const & { return w1[(top + sr) % 3][i + sc]; };
            result[i] = apply(std::true_type{}, nb, gy, gx0 + c0 + i, iteration + 1, tdv2);
        }
        store_cells<Cell, CW, true, kStore == store_tile, kTX>(result, y, gy, kStore == store_grid, 0u,
                                                               out, dst, push, geo, gx0, out_lo,
                                                               out_hi);
    };

    // Output row y, with y - y_begin == U (mod 3).
    auto row_step = [&](auto u_c, int y) {
        constexpr int u = decltype(u_c)::value;
        load_row(int_c<(u + 1) % 3>{}, y + 2);
        first(int_c<(u + 2) % 3>{}, int_c<(u + 2) % 3>{}, y + 1);
        second(int_c<u>{}, y);
    };

    // Prime: generation g+1 at rows y_begin - 1 and y_begin.
    load_row(int_c<0>{}, y_begin - 2);
    load_row(int_c<1>{}, y_begin - 1);
    load_row(int_c<2>{}, y_begin);
    first(int_c<0>{}, int_c<0>{}, y_begin - 1);
    load_row(int_c<0>{}, y_begin + 1);
    first(int_c<1>{}, int_c<1>{}, y_begin);

    int y = y_begin;
    for (; y + 3 <= y_end; y += 3) {
        row_step(int_c<0>{}, y);
        row_step(int_c<1>{}, y + 1);
        row_step(int_c<2>{}, y + 2);
    }
    if (y < y_end) {
        row_step(int_c<0>{}, y);
        if (y + 1 < y_end)
            row_step(int_c<1>{}, y + 1);
    }
}

// ------------------------------------------------------------------------------------------------
// one tile: stage, run all fused sweeps, write back
// ------------------------------------------------------------------------------------------------

// kBatch: instantiated separately for fused_sweep_batch_kernel (same code), so that the batch kernel
// leaves the code generated for fused_sweep_kernel exactly as it is
template <typename F, int CW, bool kInterior, int kMode, int kTX, bool kSpec, bool kBatch = false>
__device__ __forceinline__ void
run_tile(F const &tf, typename F::Cell const &halo_value,
         TdvArray<typename F::TimeDependentValue> const &tdvs, PlaneSet const &src,
         PlaneSet const &dst, HaloPush const &push, TensorMapSet const &maps,
         SweepGeometry const &geo, unsigned char *smem, unsigned long long *mbar, int gy0,
         int gx0, int out_lo, int out_hi) {
    using Cell = typename F::Cell;
    using L = CellLayout<Cell>;
    constexpr int R = int(F::stencil_radius);
    constexpr unsigned n_sub = unsigned(F::n_subiterations);
    constexpr unsigned all_planes = (L::n_planes >= 32) ? ~0u : ((1u << L::n_planes) - 1u);

    const unsigned rows = geo.tile_h + 2 * geo.halo;
    const unsigned cols = blockDim.x * CW;
    const unsigned buffer_bytes = unsigned(tile_buffer_bytes<Cell>(rows, cols));

    TileView<Cell> buf0(smem + tile_guard_bytes, rows, cols);
    TileView<Cell> buf1(smem + tile_guard_bytes + buffer_bytes, rows, cols);

    // Speculative plane pass-through (kSpec). A sweep only stores the planes that are not in its
    // `keep` mask; a kept plane's current version simply stays where it is. `where` tracks, per
    // plane, which of the two buffers holds the current version. Planes kept in EVERY sub-iteration
    // are never rewritten and exist in the first buffer only, so the second buffer is smaller
    // (more tile rows per CTA). Every kept plane is verified against the functor's result; a
    // mismatch is reported through geo.spec_flags and the host repeats the update without
    // speculating on that plane (StencilUpdate.hpp).
    unsigned single = 0, where = 0;
    unsigned changed[n_sub] = {};
    unsigned violated = 0;
    if constexpr (kSpec) {
        static_assert(n_sub <= max_spec_subiterations);
        single = all_planes;
#pragma unroll
        for (unsigned q = 0; q < n_sub; q++)
            single &= geo.keep[q];
        unsigned off = 0;
        for_each_plane<Cell>([&](auto I) {
            if ((single >> I) & 1u) {
                buf1.plane_off[I] = buf0.plane_off[I] - buffer_bytes; // never addressed
            } else {
                buf1.plane_off[I] = off;
                off += (rows * cols * unsigned(L::plane_bytes(I)) + 127u) / 128u * 128u;
            }
        });
    }

    stage_tile<Cell, CW, kInterior>(buf0, src, maps, geo, halo_value, gy0, gx0, mbar);

    if constexpr (kInterior && paired_sweeps<F, CW, kMode, kSpec>()) {
        // Pairs of generations (sweep_pair), one barrier per pair. An odd n_gens leaves one single
        // sweep, which goes first: it also converts the natural layout TMA delivers to lane-major.
        // With an even n_gens the first pair reads the natural layout itself.
        using grid_c = std::integral_constant<int, store_grid>;
        using tile_c = std::integral_constant<int, store_tile>;
        unsigned g = 0;
        bool flip = false; // the current generation is in buf1
        if (geo.n_gens & 1u) {
            const bool last = geo.n_gens == 1;
            SpecTrack track{0u, 0u, 0u, 0u};
            auto sweep = [&](auto store_c, auto out_lm_c) {
                sweep_rows<F, CW, true, kMode, decltype(store_c)::value, false,
                           decltype(out_lm_c)::value, kTX, false, 0>(
                    tf, halo_value, tdvs.v[0], std::size_t(geo.iteration0), buf0, buf1, last, dst,
                    push, geo, gy0, gx0, R, int(rows) - R, out_lo, out_hi, track);
            };
            if (last) {
                sweep(grid_c{}, std::false_type{});
                return;
            }
            sweep(tile_c{}, std::true_type{});
            __syncthreads();
            g = 1;
            flip = true;
        }
        for (; g < geo.n_gens; g += 2) {
            const bool last = g + 2 == geo.n_gens;
            auto pair = [&](auto store_c, auto in_lm_c) {
                sweep_pair<F, CW, decltype(store_c)::value, decltype(in_lm_c)::value, kTX>(
                    tf, tdvs.v[g], tdvs.v[g + 1], std::size_t(geo.iteration0) + g,
                    flip ? buf1 : buf0, flip ? buf0 : buf1, dst, push, geo, gy0, gx0,
                    int(g + 2) * R, int(rows) - int(g + 2) * R, out_lo, out_hi);
            };
            if (g == 0) {
                if (last)
                    pair(grid_c{}, std::false_type{});
                else
                    pair(tile_c{}, std::false_type{});
            } else {
                if (last)
                    pair(grid_c{}, std::true_type{});
                else
                    pair(tile_c{}, std::true_type{});
            }
            if (!last)
                __syncthreads();
            flip = !flip;
        }
        return;
    }

    unsigned step = 0;
    for (unsigned g = 0; g < geo.n_gens; g++) {
        const std::size_t iteration = std::size_t(geo.iteration0) + g;
        const typename F::TimeDependentValue tdv = tdvs.v[g];
        [&]<std::size_t... Subs>(std::index_sequence<Subs...>) {
            (
                [&] {
                    const bool last = (g + 1 == geo.n_gens) && (Subs + 1 == n_sub);
                    const int lo = int(step + 1) * R;
                    const int hi = int(rows) - int(step + 1) * R;
                    constexpr bool kLM = lane_major_tiles<Cell, CW>() && kMode != window_reload;
                    constexpr std::size_t kSub = Subs;
                    SpecTrack track{0u, 0u, 0u, 0u};
                    auto run = [&](TileView<Cell> const &in, TileView<Cell> const &out) {
                        auto sweep = [&](auto store_c, auto in_lm_c, auto out_lm_c) {
                            sweep_rows<F, CW, kInterior, kMode, decltype(store_c)::value,
                                       decltype(in_lm_c)::value, decltype(out_lm_c)::value, kTX, kSpec,
                                       kSub>(tf, halo_value, tdv, iteration, in, out, last, dst, push,
                                             geo, gy0, gx0, lo, hi, out_lo, out_hi, track);
                        };
                        using std::false_type;
                        using std::true_type;
                        using grid_c = std::integral_constant<int, store_grid>;
                        using tile_c = std::integral_constant<int, store_tile>;
                        using runtime_c = std::integral_constant<int, store_runtime>;
                        if constexpr (kLM) {
                            // first sweep reads the TMA-staged (natural) tile, later ones lane-major
                            if (step == 0) {
                                if (last)
                                    sweep(grid_c{}, false_type{}, false_type{});
                                else
                                    sweep(tile_c{}, false_type{}, true_type{});
                            } else {
                                if (last)
                                    sweep(grid_c{}, true_type{}, false_type{});
                                else
                                    sweep(tile_c{}, true_type{}, true_type{});
                            }
                        } else if constexpr (sizeof(Cell) <= 16) {
                            if (last)
                                sweep(grid_c{}, false_type{}, false_type{});
                            else
                                sweep(tile_c{}, false_type{}, false_type{});
                        } else {
                            sweep(runtime_c{}, false_type{}, false_type{});
                        }
                    };
                    if constexpr (kSpec) {
                        track.keep = geo.keep[kSub] & all_planes;
                        track.probe = geo.probe;
                        TileView<Cell> in(smem + tile_guard_bytes, rows, cols, 0);
                        TileView<Cell> out(smem + tile_guard_bytes, rows, cols, 0);
                        for_each_plane<Cell>([&](auto I) {
                            const unsigned a = buf0.plane_off[I];
                            const unsigned b = buffer_bytes + buf1.plane_off[I];
                            const bool in_second = (where >> I) & 1u;
                            in.plane_off[I] = in_second ? b : a;
                            out.plane_off[I] = ((track.keep >> I) & 1u) ? in.plane_off[I]
                                                                         : (in_second ? a : b);
                        });
                        run(in, out);
                        where ^= ~track.keep & all_planes;
                        changed[kSub] |= track.changed;
                        violated |= track.violated;
                    } else {
                        run((step & 1u) ? buf1 : buf0, (step & 1u) ? buf0 : buf1);
                    }
                    if (!last)
                        __syncthreads();
                    step++;
                }(),
                ...);
        }(std::make_index_sequence<n_sub>{});
    }

    if constexpr (kSpec) {
        // one atomic per warp and word, and only where there is something to report
        violated = __reduce_or_sync(0xffffffffu, violated);
        const bool leader = (threadIdx.x & 31u) == 0;
        if (violated != 0 && leader)
            atomicOr(geo.spec_flags + max_spec_subiterations, violated);
        if (geo.probe) {
#pragma unroll
            for (unsigned q = 0; q < n_sub; q++) {
                const unsigned c = __reduce_or_sync(0xffffffffu, changed[q]);
                if (c != 0 && leader)
                    atomicOr(geo.spec_flags + q, c);
            }
        }
    }
}

/**
 * The fused generation-loop kernel. Grid: one CTA per output tile, blockIdx.x = ty * tiles_x + tx;
 * block: (TWH / CW, row groups), blockDim.x a multiple of 32.
 * Dynamic shared memory: two tile buffers (one if the launch consists of a single sweep).
 */
template <typename F, int CW, int kMode, int kTX, int kMaxThreads, int kMinBlocks, bool kSpec = false>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks)
    fused_sweep_kernel(const __grid_constant__ F tf,
                       const __grid_constant__ typename F::Cell halo_value,
                       const __grid_constant__ TdvArray<typename F::TimeDependentValue> tdvs,
                       const __grid_constant__ PlaneSet src, const __grid_constant__ PlaneSet dst,
                       const __grid_constant__ HaloPush push,
                       const __grid_constant__ TensorMapSet maps,
                       const __grid_constant__ SweepGeometry geo) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ unsigned long long mbar;

    if (geo.use_tma) {
        if (threadIdx.x == 0 && threadIdx.y == 0) {
            mbarrier_init(&mbar, 1);
            fence_mbarrier_init();
        }
        __syncthreads();
    }

    // Which of the (at most two) row ranges of this launch the CTA works on.
    unsigned tile_index = blockIdx.x;
    int out_lo = geo.out_row_lo, out_hi = geo.out_row_hi;
    if (tile_index >= geo.tiles_first) {
        tile_index -= geo.tiles_first;
        out_lo = geo.out2_row_lo;
        out_hi = geo.out2_row_hi;
    }
    const unsigned tx = tile_index % geo.tiles_x;
    const unsigned ty = tile_index / geo.tiles_x;
    const int tile_gy = out_lo + int(ty * geo.tile_h);
    const int tile_gx = int(tx * geo.tile_w);
    const int gy0 = tile_gy - int(geo.halo);
    const int gx0 = tile_gx - int(geo.hpad);

    // Interior: the staged footprint lies inside the grid, with at least one column to spare on
    // either side (rows: every computed row is >= radius rows away from the footprint's edge
    // anyway) — so that ALL cells the tile computes, including the never-exact outermost columns,
    // are at least one cell inside the grid (see the __builtin_assume in sweep_rows).
    const bool interior = gy0 >= 0 && tile_gy + int(geo.tile_h + geo.halo) <= int(geo.grid_h) &&
                          tile_gy + int(geo.tile_h) <= out_hi && gx0 >= 1 &&
                          tile_gx + int(geo.tile_w + geo.hpad) + 1 <= int(geo.grid_w);

    if (interior) {
        run_tile<F, CW, true, kMode, kTX, kSpec>(tf, halo_value, tdvs, src, dst, push, maps, geo, smem,
                                                 &mbar, gy0, gx0, out_lo, out_hi);
    } else {
        run_tile<F, CW, false, (kMode == window_reload ? window_reload : window_shift), kTX, kSpec>(
            tf, halo_value, tdvs, src, dst, push, maps, geo, smem, &mbar, gy0, gx0, out_lo, out_hi);
    }

    // (`blockIdx.x < gridDim.x` always holds; without that test ptxas gives FDTD's plain kernel two
    // registers more, see profiles/r02_kernel_resources.txt)
    if (geo.push && push.ticket != nullptr && blockIdx.x < gridDim.x) {
        // Every thread makes its stores (own planes and the neighbours' ghost rows) visible
        // system-wide, then the CTA takes a ticket; the holder of the last ticket knows that every
        // CTA of the launch has passed its fence (fence / relaxed atomic / fence: release and
        // acquire patterns of the PTX memory model) and raises the neighbours' flags. The launch that
        // pushes is also the only reader of this slab's ghost rows, which the neighbours overwrite
        // next.
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0 && threadIdx.y == 0) {
            const unsigned ticket = atomicAdd(push.ticket, 1u);
            if (ticket == gridDim.x - 1u) {
                __threadfence_system();
                if (push.flag_up != nullptr)
                    *reinterpret_cast<volatile unsigned *>(push.flag_up) = push.flag_value;
                if (push.flag_down != nullptr)
                    *reinterpret_cast<volatile unsigned *>(push.flag_down) = push.flag_value;
                *reinterpret_cast<volatile unsigned *>(push.ticket) = 0u; // for the next launch
                __threadfence_system();
            }
        }
    }
}

/**
 * The fused kernel over a grid batch: member b of the batch occupies plane rows [b * H, (b + 1) * H)
 * of `src` and `dst`, where H = geo.grid_h is the member extent. Grid: blockIdx.y is the member,
 * blockIdx.x = ty * tiles_x + tx the tile within it, so a launch holds at most 65535 members
 * (gridDim.y). Everything the tile code sees is member-local (`stencil.id`, `grid_range`, the
 * interior test, the halo patching and the re-imposition of `halo_value`); only addresses into the
 * planes carry the member's row offset, through buf_row0. A border tile's TMA box may reach into
 * the neighbouring members' rows: those rows lie outside [0, H) and are overwritten with
 * `halo_value` exactly like rows outside a single grid. One row range per launch, no halo push.
 * (A kernel of its own rather than a branch in fused_sweep_kernel, whose code stays as it is.)
 */
template <typename F, int CW, int kMode, int kTX, int kMaxThreads, int kMinBlocks, bool kSpec = false>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks)
    fused_sweep_batch_kernel(const __grid_constant__ F tf,
                             const __grid_constant__ typename F::Cell halo_value,
                             const __grid_constant__ TdvArray<typename F::TimeDependentValue> tdvs,
                             const __grid_constant__ PlaneSet src,
                             const __grid_constant__ PlaneSet dst,
                             const __grid_constant__ TensorMapSet maps,
                             const __grid_constant__ SweepGeometry geo) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ unsigned long long mbar;

    if (geo.use_tma) {
        if (threadIdx.x == 0 && threadIdx.y == 0) {
            mbarrier_init(&mbar, 1);
            fence_mbarrier_init();
        }
        __syncthreads();
    }

    SweepGeometry member = geo;
    member.buf_row0 = geo.buf_row0 - int(blockIdx.y * geo.grid_h);
    member.push = 0u;
    const HaloPush no_push{};

    // as in fused_sweep_kernel, member-local
    const int out_lo = geo.out_row_lo, out_hi = geo.out_row_hi;
    const unsigned tx = blockIdx.x % geo.tiles_x;
    const unsigned ty = blockIdx.x / geo.tiles_x;
    const int tile_gy = out_lo + int(ty * geo.tile_h);
    const int tile_gx = int(tx * geo.tile_w);
    const int gy0 = tile_gy - int(geo.halo);
    const int gx0 = tile_gx - int(geo.hpad);
    const bool interior = gy0 >= 0 && tile_gy + int(geo.tile_h + geo.halo) <= int(geo.grid_h) &&
                          tile_gy + int(geo.tile_h) <= out_hi && gx0 >= 1 &&
                          tile_gx + int(geo.tile_w + geo.hpad) + 1 <= int(geo.grid_w);

    if (interior) {
        run_tile<F, CW, true, kMode, kTX, kSpec, true>(tf, halo_value, tdvs, src, dst, no_push, maps,
                                                       member, smem, &mbar, gy0, gx0, out_lo, out_hi);
    } else {
        run_tile<F, CW, false, (kMode == window_reload ? window_reload : window_shift), kTX, kSpec,
                 true>(tf, halo_value, tdvs, src, dst, no_push, maps, member, smem, &mbar, gy0, gx0,
                       out_lo, out_hi);
    }
}

#endif // __CUDACC__

} // namespace internal
} // namespace cuda
} // namespace stencil
