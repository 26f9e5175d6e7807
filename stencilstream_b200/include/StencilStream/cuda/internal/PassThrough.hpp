/*
 * StencilStream-B200 — plane pass-through: which planes the tile sweeps leave in place, and when that
 * pays. One object per updater: the single-GPU one (cuda/StencilUpdate.hpp) and every row slab
 * (cuda/internal/SlabUpdate.hpp).
 *
 * A field that a transition function never changes (HotSpot's `power`, FDTD's material
 * coefficients) need not be copied from tile buffer to tile buffer; left in place in every
 * sub-iteration it needs only ONE tile buffer, so the tiles grow (run_tile in TileKernel.hpp). The
 * planes kept that way come from one of two sources:
 *
 *   - declared: the cell type lists them in `Cell::constant_fields` (Helpers.hpp). Nothing is
 *     observed and nothing repeated; the kernels' own check is only read on request.
 *   - detected: the first launch *observes* which planes come out of the transition function
 *     unchanged, per sub-iteration. Later launches keep those planes and *verify* that they still do
 *     not change, reporting any that did through a device word. The owner reads those words after
 *     the launches, drops the planes that changed and repeats the work from a generation it kept.
 */
#pragma once
#include "Helpers.hpp"
#include "Planner.hpp"
#include "Runtime.hpp"
#include "TileKernel.hpp"

#include <optional>

namespace stencil {
namespace cuda {
namespace internal {

/// What one launch does about pass-through (see run_tile in TileKernel.hpp).
struct Speculation {
    unsigned keep[max_spec_subiterations] = {};
    bool probe = false;          ///< the launch only observes (keep must be all-zero)
    unsigned *flags = nullptr;   ///< device: [0, S) changed per sub-iteration, [S] violated planes

    unsigned single_planes(unsigned n_sub, unsigned all_planes) const {
        unsigned m = all_planes;
        for (unsigned q = 0; q < n_sub; q++)
            m &= keep[q];
        return m;
    }
};

/// Cells with several planes, few sub-iterations and at most 64 bytes can run the pass-through
/// kernels. Larger cells run at the register limit of their CTAs, where the per-plane buffer
/// bookkeeping of those kernels spills (convection: 9.2 -> 8.2 GCell-updates/s even with four of
/// eleven fields constant in the benchmark input); their pass-through kernels are not instantiated.
template <typename F> constexpr bool speculation_capable() {
    using Layout = CellLayout<typename F::Cell>;
    return Layout::n_planes >= 2 && Layout::n_planes <= 32 &&
           F::n_subiterations <= max_spec_subiterations && sizeof(typename F::Cell) <= 64;
}

/// STST_SPECULATE=0 turns plane pass-through off, declared and detected; read once per process.
inline bool passthrough_switched_on() {
    static const bool on = env_long("STST_SPECULATE", 1) != 0;
    return on;
}

template <typename F> class PassThrough {
  public:
    using Cell = typename F::Cell;
    using Layout = CellLayout<Cell>;
    static constexpr unsigned all_planes =
        Layout::n_planes >= 32 ? ~0u : ((1u << Layout::n_planes) - 1u);
    static constexpr unsigned declared_planes = constant_fields_mask<Cell>();
    static_assert(declared_planes != ~0u || Layout::n_planes >= 32,
                  "every entry of Cell::constant_fields must also be listed in Cell::fields");

    /// Pass-through pays through the planes that need only ONE tile buffer (taller tiles) and the
    /// stores it saves; the kernels that support it carry per-plane buffer bookkeeping, which costs
    /// registers. Measured (profiles/r01_s3_sweep_speculation.log): HotSpot +11 %, FDTD +19 % with
    /// half of the cell passing through, mantle convection -11 % with one field of eleven. Below a
    /// quarter of the cell's bytes the plain kernels are used.
    static constexpr bool pays(unsigned single_planes) {
        std::size_t bytes = 0;
        for (std::size_t i = 0; i < Layout::n_planes; i++)
            if ((single_planes >> i) & 1u)
                bytes += Layout::plane_bytes(i);
        return 4 * bytes >= sizeof(Cell);
    }

    /// The keep masks are `Cell::constant_fields`: no observation, no repeat.
    static bool declared() {
        if constexpr (speculation_capable<F>() && declared_planes != 0)
            return passthrough_switched_on() && pays(declared_planes);
        else
            return false;
    }

    /// The keep masks are detected at run time (cell types that declare no constant fields).
    static bool detected() {
        if constexpr (speculation_capable<F>() && declared_planes == 0)
            return passthrough_switched_on();
        else
            return false;
    }

    PassThrough() {
        if (declared()) {
            for (unsigned q = 0; q < n_masks; q++)
                keep[q] = declared_planes;
            was_probed = true;
        }
    }
    /// What was observed about the transition function travels with a copy; the device words are
    /// per object and allocated on first use.
    PassThrough(PassThrough const &other) : was_probed(other.was_probed) {
        for (unsigned q = 0; q < n_masks; q++)
            keep[q] = other.keep[q];
    }
    PassThrough &operator=(PassThrough const &) = delete;
    ~PassThrough() {
        free_flags();
        pinned_free(host_flags);
    }

    /// Whether the keep masks are known (declared, or observed by an earlier launch).
    bool probed() const { return was_probed; }

    /// Planes kept in every sub-iteration: the planes that need one tile buffer (for make_plan).
    unsigned single_planes() const {
        unsigned m = all_planes;
        for (unsigned q = 0; q < n_masks; q++)
            m &= keep[q];
        return n_masks > 0 ? m : 0u;
    }

    /// An observation found nothing worth keeping, or every kept plane has been dropped.
    bool nothing_left() const { return was_probed && single_planes() == 0; }

    /// The Speculation of a launch that only observes which planes change.
    Speculation observing(int device, stst_stream_t stream) {
        Speculation spec{};
        spec.probe = true;
        spec.flags = device_flags(device, stream);
        return spec;
    }

    /// The Speculation of a launch that keeps the planes and verifies them; none if nothing is kept.
    std::optional<Speculation> verifying(int device, stst_stream_t stream) {
        if (single_planes() == 0)
            return std::nullopt;
        Speculation spec{};
        for (unsigned q = 0; q < n_masks; q++)
            spec.keep[q] = keep[q];
        spec.flags = device_flags(device, stream);
        return spec;
    }

    /// After an observing launch on `stream`: keep what never changed, if that pays. Waits for it.
    void read_observation(stst_stream_t stream) {
        const unsigned *changed = read_flags(stream);
        for (unsigned q = 0; q < n_masks; q++)
            keep[q] = ~changed[q] & all_planes;
        was_probed = true;
        settle();
    }

    /// Planes that a verifying launch on `stream` saw change since the last call. Waits for them.
    unsigned take_violations(stst_stream_t stream) {
        return flags ? read_flags(stream)[max_spec_subiterations] : 0u;
    }

    /// Never keep `planes` again.
    void drop(unsigned planes) {
        for (unsigned q = 0; q < n_masks; q++)
            keep[q] &= ~planes;
        settle();
    }

    /// Free the device words (in order on the stream they were allocated on).
    void free_flags() {
        device_free(flags_device, flags, flags_stream);
        flags = nullptr;
    }

  private:
    static constexpr unsigned n_masks =
        unsigned(F::n_subiterations) <= max_spec_subiterations ? unsigned(F::n_subiterations) : 0u;
    static constexpr std::size_t flag_bytes = sizeof(unsigned) * (max_spec_subiterations + 1);

    void settle() {
        if (!pays(single_planes()))
            for (unsigned q = 0; q < n_masks; q++)
                keep[q] = 0;
    }

    /// The device words on `device`, zeroed in order on `stream` when they are (re)allocated.
    unsigned *device_flags(int device, stst_stream_t stream) {
        if (flags && flags_device != device)
            free_flags();
        if (!flags) {
            flags = static_cast<unsigned *>(device_alloc(device, flag_bytes, stream));
            flags_device = device;
            flags_stream = stream;
            STST_RT_CHECK(stst_memset_async(flags, 0, flag_bytes, stream));
        }
        return flags;
    }

    /// Copy the device words to the host and zero them for the launches that follow.
    const unsigned *read_flags(stst_stream_t stream) {
        if (!host_flags)
            host_flags = static_cast<unsigned *>(pinned_alloc(flag_bytes));
        STST_RT_CHECK(stst_memcpy_d2h_async(host_flags, flags, flag_bytes, stream));
        STST_RT_CHECK(stst_stream_synchronize(stream));
        STST_RT_CHECK(stst_memset_async(flags, 0, flag_bytes, stream));
        return host_flags;
    }

    unsigned keep[max_spec_subiterations] = {}; ///< per sub-iteration: planes left in place
    bool was_probed = false;
    unsigned *flags = nullptr;                  ///< device words of the kernels' reports
    int flags_device = 0;
    stst_stream_t flags_stream = nullptr;
    unsigned *host_flags = nullptr;             ///< pinned landing zone of `flags`, allocated once
};

} // namespace internal
} // namespace cuda
} // namespace stencil
