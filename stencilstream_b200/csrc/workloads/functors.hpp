/*
 * Transition functions instantiated by libstst_workloads.so.
 *
 * These restate, for nvcc (every member __host__ __device__), the functors of the reference's
 * examples and of its self-checking unit test. The arithmetic — operand order, literal types,
 * implicit float/double promotions — follows the cited reference expressions exactly, because the
 * parity tests compare against the reference's own sources compiled for the CPU (oracle/_ref) and,
 * in the `-fmad=false` build, demand bit-identical results. The parameter blocks are the C structs
 * of include/stst_workloads.h, so that parameters cross the C ABI as plain memory.
 *
 * The unmodified reference example sources are additionally built against this backend by
 * stencilstream_b200/tools/build_reference_examples.py (drop-in check); this header is what ships.
 */
#pragma once
#include <StencilStream/BaseTransitionFunction.hpp>
#include <StencilStream/Stencil.hpp>
#include <stst_workloads.h>

#include <cstddef>
#include <tuple>

namespace stst_workloads {

using stencil::BaseTransitionFunction;
using stencil::Stencil;

// ------------------------------------------------------------------------------------------------
// Conway's Game of Life — reference examples/conway/conway.cpp:35-56
// ------------------------------------------------------------------------------------------------
struct ConwayRule : public BaseTransitionFunction {
    using Cell = bool;
    stst_conway_params p;

    STST_HD bool operator()(Stencil<bool, 1> const &st) const {
        int neighbours = 0;
#pragma unroll
        for (int dr = -1; dr <= 1; dr++) {
#pragma unroll
            for (int dc = -1; dc <= 1; dc++) {
                const bool is_centre = (dr == 0 && dc == 0);
                if (!is_centre && st[dr][dc])
                    neighbours++;
            }
        }
        return st[0][0] ? (neighbours == 2 || neighbours == 3) : (neighbours == 3);
    }
};

// ------------------------------------------------------------------------------------------------
// Jacobi — reference examples/jacobi/kernels.hpp
// ------------------------------------------------------------------------------------------------

/// Jacobi5General, kernels.hpp:236-272. Weights: north, west, south, east, centre.
struct Jacobi5Rule : public BaseTransitionFunction {
    using Cell = float;
    stst_jacobi5_params p;

    STST_HD float operator()(Stencil<float, 1> const &st) const {
        return p.coef[0] * st[-1][0] + p.coef[1] * st[0][-1] + p.coef[2] * st[1][0] +
               p.coef[3] * st[0][1] + p.coef[4] * st[0][0];
    }
};

/// Jacobi9General, kernels.hpp:274-319. Row-major accumulation starting from 0.
struct Jacobi9Rule : public BaseTransitionFunction {
    using Cell = float;
    stst_jacobi9_params p;

    STST_HD float operator()(Stencil<float, 1> const &st) const {
        float acc = 0.0f;
#pragma unroll
        for (int dr = -1; dr <= 1; dr++) {
#pragma unroll
            for (int dc = -1; dc <= 1; dc++) {
                acc += p.coef[dr + 1][dc + 1] * st[dr][dc];
            }
        }
        return acc;
    }
};

/**
 * Radius-R star ("plus"-shaped) Jacobi stencil with 4R+1 points. BASELINE.json asks for radius-2/3
 * Jacobi variants; the reference has no such functor (all of kernels.hpp is radius 1), so this one is
 * defined here and run through the reference's radius-generic cpu backend for the oracle.
 * acc = centre*c + sum_{d=1..R} arm[d-1] * (((n_d + w_d) + s_d) + e_d).
 */
template <std::size_t R> struct JacobiStarRule : public BaseTransitionFunction {
    using Cell = float;
    static constexpr std::size_t stencil_radius = R;
    stst_jacobi_star_params p;

    STST_HD float operator()(Stencil<float, R> const &st) const {
        float acc = p.centre * st[0][0];
#pragma unroll
        for (int d = 1; d <= int(R); d++) {
            acc += p.arm[d - 1] * (((st[-d][0] + st[0][-d]) + st[d][0]) + st[0][d]);
        }
        return acc;
    }
};

// ------------------------------------------------------------------------------------------------
// Rodinia HotSpot — reference examples/hotspot/hotspot.cpp:57-97
// ------------------------------------------------------------------------------------------------
struct HotspotCell {
    float temp;
    float power;
    static constexpr auto fields = std::make_tuple(&HotspotCell::temp, &HotspotCell::power);
    /// B200 extension (cuda/internal/Helpers.hpp): no HotSpot sweep ever changes the dissipated power.
    /// (The unmodified reference example has no such line and gets the same effect from the
    /// run-time detection of StencilUpdate::run_detected; FDTD below is left to that detection on
    /// purpose, so that both routes stay exercised.)
    static constexpr auto constant_fields = std::make_tuple(&HotspotCell::power);
};
static_assert(sizeof(HotspotCell) == sizeof(stst_hotspot_cell));

struct HotspotRule : public BaseTransitionFunction {
    using Cell = HotspotCell;
    stst_hotspot_params p;

    STST_HD Cell operator()(Stencil<HotspotCell, 1> const &st) const {
        const float ambient = 80.0f; // amb_temp, hotspot.cpp:55
        const float power = st[0][0].power;
        const float old = st[0][0].temp;
        float north = st[-1][0].temp;
        float south = st[1][0].temp;
        float west = st[0][-1].temp;
        float east = st[0][1].temp;

        // Adiabatic borders: the missing neighbour is replaced by the cell itself (:77-87).
        if (st.id[0] == 0) {
            north = old;
        } else if (st.id[0] == st.grid_range[0] - 1) {
            south = old;
        }
        if (st.id[1] == 0) {
            west = old;
        } else if (st.id[1] == st.grid_range[1] - 1) {
            east = old;
        }

        const float next = old + p.Cap_1 * (power + (south + north - 2.f * old) * p.Ry_1 +
                                            (east + west - 2.f * old) * p.Rx_1 +
                                            (ambient - old) * p.Rz_1);
        return HotspotCell{next, power};
    }
};

// ------------------------------------------------------------------------------------------------
// FDTD, coefficient-carrying cells — reference examples/fdtd/src/Kernel.hpp:52-141 with
// material/CoefResolver.hpp:24-68
// ------------------------------------------------------------------------------------------------
struct FdtdCell {
    float ex, ey, hz, hz_sum;
    float ca, cb, da, db;
    static constexpr auto fields =
        std::make_tuple(&FdtdCell::ex, &FdtdCell::ey, &FdtdCell::hz, &FdtdCell::hz_sum,
                        &FdtdCell::ca, &FdtdCell::cb, &FdtdCell::da, &FdtdCell::db);
};
static_assert(sizeof(FdtdCell) == sizeof(stst_fdtd_cell));

struct FdtdCoefRule {
    using Cell = FdtdCell;
    using TimeDependentValue = float;
    static constexpr std::size_t stencil_radius = 1;
    static constexpr std::size_t n_subiterations = 2;
    stst_fdtd_params p;

    /// Source wave amplitude of iteration i; evaluated on the host only (Kernel.hpp:80-84).
    STST_HD float get_time_dependent_value(std::size_t i_iteration) const {
        float current_time = i_iteration * p.dt;
        float wave_progress = (current_time - p.t_0) / p.tau;
        return sycl::cos(p.omega * current_time) * sycl::exp(-1 * wave_progress * wave_progress);
    }

    STST_HD Cell operator()(Stencil<Cell, 1, float> const &st) const {
        Cell cell = st[0][0];

        float r = st.id[0];
        float c = st.id[1];
        float source_distance_score = r * (r - 2 * p.source_r) + c * (c - 2 * p.source_c);

        // CoefResolver: the material coefficients travel with the cell (CoefResolver.hpp:60-67).
        const float ca = st[0][0].ca, cb = st[0][0].cb, da = st[0][0].da, db = st[0][0].db;

        if (st.subiteration == 0) {
            // E-field half step
            cell.ex *= ca;
            cell.ex += cb * (st[0][0].hz - st[0][-1].hz);
            cell.ey *= ca;
            cell.ey += cb * (st[-1][0].hz - st[0][0].hz);
        } else {
            // H-field half step, source injection and detection
            cell.hz *= da;
            cell.hz += db * (st[0][1].ex - st[0][0].ex + st[0][0].ey - st[1][0].ey);

            if (source_distance_score <= p.source_distance_bound &&
                st.iteration <= p.cutoff_iteration) {
                float interp_factor;
                if (p.source_radius_squared != 0) {
                    float cell_distance_squared = source_distance_score +
                                                  p.source_c * p.source_c +
                                                  p.source_r * p.source_r;
                    interp_factor = 1.0 - float(cell_distance_squared) / p.source_radius_squared;
                } else {
                    interp_factor = 1.0;
                }
                cell.hz += interp_factor * st.time_dependent_value;
            }

            if (st.iteration > p.detect_iteration) {
                cell.hz_sum += cell.hz * cell.hz;
            }
        }
        return cell;
    }
};

// ------------------------------------------------------------------------------------------------
// Mantle convection — reference examples/convection/convection.cpp:36-242
// ------------------------------------------------------------------------------------------------
struct ConvectionCell {
    double T, Pt, Vx, Vy;
    double tau_xx, tau_yy, sigma_xy;
    double dVxd_tau, dVyd_tau;
    double ErrV, ErrP;
    static constexpr auto fields = std::make_tuple(
        &ConvectionCell::T, &ConvectionCell::Pt, &ConvectionCell::Vx, &ConvectionCell::Vy,
        &ConvectionCell::tau_xx, &ConvectionCell::tau_yy, &ConvectionCell::sigma_xy,
        &ConvectionCell::dVxd_tau, &ConvectionCell::dVyd_tau, &ConvectionCell::ErrV,
        &ConvectionCell::ErrP);
};
static_assert(sizeof(ConvectionCell) == sizeof(stst_convection_cell));

/// PseudoTransientKernel, convection.cpp:76-183: three sweeps per iteration.
struct ConvectionPseudoTransientRule : public BaseTransitionFunction {
    using Cell = ConvectionCell;
    static constexpr std::size_t n_subiterations = 3;
    stst_convection_pt_params p;

    STST_HD Cell operator()(Stencil<Cell, 1> const &st) const {
        Cell next = st[0][0];
        const std::size_t x = st.id[0];
        const std::size_t y = st.id[1];
        const std::size_t nx = p.nx, ny = p.ny;

        if (st.subiteration == 0) {
            // keep the previous Vy / Pt for the error estimate (:100-108)
            if (x < nx && y < ny + 1)
                next.ErrV = st[0][0].Vy;
            if (x < nx && y < ny)
                next.ErrP = st[0][0].Pt;

            // pressure and normal/shear stresses (:110-128)
            if (x < nx && y < ny) {
                const double dVx_dx = (st[1][0].Vx - st[0][0].Vx) / p.dx;
                const double dVy_dy = (st[0][1].Vy - st[0][0].Vy) / p.dy;
                const double div_V = dVx_dx + dVy_dy;
                const double eta =
                    p.eta0 * (1.0 - p.delta_eta_delta_T * (st[0][0].T + p.deltaT / 2.0));

                next.Pt = st[0][0].Pt - p.delta_tau_iter / p.beta * div_V;
                next.tau_xx = 2.0 * eta * ((st[1][0].Vx - st[0][0].Vx) / p.dx - (1.0 / 3.0) * div_V);
                next.tau_yy = 2.0 * eta * ((st[0][1].Vy - st[0][0].Vy) / p.dy - (1.0 / 3.0) * div_V);

                if (x < nx - 1 && y < ny - 1) {
                    next.sigma_xy = eta * ((st[1][1].Vx - st[1][0].Vx) / p.dy +
                                           (st[1][1].Vy - st[0][1].Vy) / p.dx);
                }
            }
        } else if (st.subiteration == 1) {
            // momentum residuals and velocity update (:130-153)
            if (x >= 1 && y >= 1) {
                if (x < (nx + 1) - 1 && y < ny - 1) {
                    const double Rx = 1.0 / p.rho *
                                      ((st[0][0].tau_xx - st[-1][0].tau_xx) / p.dx +
                                       (st[-1][0].sigma_xy - st[-1][-1].sigma_xy) / p.dy -
                                       (st[0][0].Pt - st[-1][0].Pt) / p.dx);
                    next.dVxd_tau = p.dampX * st[0][0].dVxd_tau + Rx * p.delta_tau_iter;
                    next.Vx = st[0][0].Vx + next.dVxd_tau * p.delta_tau_iter;
                }
                if (x < nx - 1 && y < (ny + 1) - 1) {
                    const double Ry =
                        1.0 / p.rho *
                        ((st[0][0].tau_yy - st[0][-1].tau_yy) / p.dy +
                         (st[0][-1].sigma_xy - st[-1][-1].sigma_xy) / p.dx -
                         (st[0][0].Pt - st[0][-1].Pt) / p.dy +
                         p.roh0_g_alpha * ((st[0][-1].T + st[0][0].T) * 0.5));
                    next.dVyd_tau = p.dampY * st[0][0].dVyd_tau + Ry * p.delta_tau_iter;
                    next.Vy = st[0][0].Vy + next.dVyd_tau * p.delta_tau_iter;
                }
            }
        } else if (st.subiteration == 2) {
            // free-slip boundaries (:155-172)
            if (x < nx + 1 && y < ny) {
                if (y == 0)
                    next.Vx = st[0][1].Vx;
                if (y == ny - 1)
                    next.Vx = st[0][-1].Vx;
            }
            if (x < nx && y < ny + 1) {
                if (x == 0)
                    next.Vy = st[1][0].Vy;
                if (x == nx - 1)
                    next.Vy = st[-1][0].Vy;
            }
            // error estimates (:174-181)
            if (x < nx && y < ny + 1)
                next.ErrV = st[0][0].ErrV - next.Vy;
            if (x < nx && y < ny)
                next.ErrP = st[0][0].ErrP - st[0][0].Pt;
        }
        return next;
    }
};

/// ThermalSolverKernel, convection.cpp:185-242: two sweeps per iteration.
struct ConvectionThermalRule : public BaseTransitionFunction {
    using Cell = ConvectionCell;
    static constexpr std::size_t n_subiterations = 2;
    stst_convection_thermal_params p;

    STST_HD Cell operator()(Stencil<Cell, 1> const &st) const {
        Cell next = st[0][0];
        const std::size_t x = st.id[0];
        const std::size_t y = st.id[1];
        const std::size_t nx = p.nx, ny = p.ny;

        if (st.subiteration == 0) {
            if (x > 0 && y > 0 && x < nx - 1 && y < ny - 1) {
                // diffusive heat fluxes through the four faces (:206-210)
                const double qx_lo = -p.DcT * (st[0][0].T - st[-1][0].T) / p.dx;
                const double qx_hi = -p.DcT * (st[1][0].T - st[0][0].T) / p.dx;
                const double qy_lo = -p.DcT * (st[0][0].T - st[0][-1].T) / p.dy;
                const double qy_hi = -p.DcT * (st[0][1].T - st[0][0].T) / p.dy;

                // upwind advection (:215-227)
                double dT_dt = -((qx_hi - qx_lo) / p.dx + (qy_hi - qy_lo) / p.dy);
                if (st[0][0].Vx > 0)
                    dT_dt -= st[0][0].Vx * (st[0][0].T - st[-1][0].T) / p.dx;
                if (st[1][0].Vx < 0)
                    dT_dt -= st[1][0].Vx * (st[1][0].T - st[0][0].T) / p.dx;
                if (st[0][0].Vy > 0)
                    dT_dt -= st[0][0].Vy * (st[0][0].T - st[0][-1].T) / p.dy;
                if (st[0][1].Vy < 0)
                    dT_dt -= st[0][1].Vy * (st[0][1].T - st[0][0].T) / p.dy;

                next.T = st[0][0].T + dT_dt * p.dt;
            }
        } else if (st.subiteration == 1) {
            // zero-flux side walls (:233-239)
            if (x == nx - 1 && y < ny)
                next.T = st[-1][0].T;
            if (x == 0 && y < ny)
                next.T = st[1][0].T;
        }
        return next;
    }
};

// ------------------------------------------------------------------------------------------------
// Self-checking known-answer functor — reference tests/TransFuncs.hpp:30-104 (FPGATransFunc<1>)
// ------------------------------------------------------------------------------------------------
enum class KatStatus : std::int32_t { Normal = 0, Invalid = 1, Halo = 2 };

struct KatCell {
    std::int32_t r, c, i_iteration, i_subiteration;
    KatStatus status;

    STST_HD static KatCell halo() { return KatCell{0, 0, 0, 0, KatStatus::Halo}; }

    static constexpr auto fields = std::make_tuple(&KatCell::r, &KatCell::c, &KatCell::i_iteration,
                                                   &KatCell::i_subiteration, &KatCell::status);
};
static_assert(sizeof(KatCell) == sizeof(stst_kat_cell));

/**
 * Every in-grid neighbour must carry its own coordinates and the current (iteration,
 * sub-iteration); every out-of-grid neighbour must be the halo cell; the time-dependent value must
 * equal the iteration index. Any violation marks the cell Invalid, which then spreads.
 */
template <std::size_t R> struct KatRule {
    using Cell = KatCell;
    using TimeDependentValue = std::size_t;
    static constexpr std::size_t stencil_radius = R;
    static constexpr std::size_t n_subiterations = 2;
    stst_kat_params p;

    STST_HD std::size_t get_time_dependent_value(std::size_t i_iteration) const {
        return i_iteration;
    }

    STST_HD Cell operator()(Stencil<Cell, R, std::size_t> const &st) const {
        Cell next = st[0][0];
        bool ok = true;
#pragma unroll
        for (int dr = -int(R); dr <= int(R); dr++) {
#pragma unroll
            for (int dc = -int(R); dc <= int(R); dc++) {
                const Cell seen = st[dr][dc];
                const long long rr = (long long)(st.id[0]) + dr;
                const long long cc = (long long)(st.id[1]) + dc;
                const bool inside = rr >= 0 && cc >= 0 && rr < (long long)(st.grid_range[0]) &&
                                    cc < (long long)(st.grid_range[1]);
                if (inside) {
                    ok &= seen.r == rr && seen.c == cc;
                    ok &= std::size_t(seen.i_iteration) == st.iteration;
                    ok &= std::size_t(seen.i_subiteration) == st.subiteration;
                    ok &= seen.status == KatStatus::Normal;
                } else {
                    const Cell h = Cell::halo();
                    ok &= seen.r == h.r && seen.c == h.c && seen.i_iteration == h.i_iteration &&
                          seen.i_subiteration == h.i_subiteration && seen.status == h.status;
                }
            }
        }
        ok &= st.time_dependent_value == st.iteration;

        next.status = ok ? KatStatus::Normal : KatStatus::Invalid;
        if (next.i_subiteration == int(n_subiterations) - 1) {
            next.i_iteration += 1;
            next.i_subiteration = 0;
        } else {
            next.i_subiteration++;
        }
        return next;
    }
};

} // namespace stst_workloads
