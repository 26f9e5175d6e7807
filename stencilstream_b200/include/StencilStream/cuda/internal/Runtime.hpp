/*
 * StencilStream-B200 — C++ veneer over the C-ABI device runtime (include/stst_rt.h).
 *
 * Turns status codes into exceptions and makes a device current before a kernel launch
 * (select_device); it owns nothing else. The reference obtains the same services from the SYCL
 * runtime (sycl::queue / sycl::buffer / sycl::event; reference
 * StencilStream/cuda/StencilUpdate.hpp:124-135 and cuda/Grid.hpp:66-134).
 */
#pragma once
#include <stst_rt.h>
#if defined(__CUDACC__)
    #include <cuda_runtime.h>
#endif

#include <cstddef>
#include <stdexcept>
#include <string>

namespace stencil {
namespace cuda {
namespace internal {

/// Thrown for every failed runtime call; there is no CPU fallback behind any of them.
class runtime_error : public std::runtime_error {
  public:
    runtime_error(const char *call, int code)
        : std::runtime_error(std::string("StencilStream-B200 runtime: ") + call + " failed (" +
                             std::to_string(code) + "): " + stst_last_error()),
          code(code) {}
    int code;
};

inline void check(int status, const char *call) {
    if (status != 0)
        throw runtime_error(call, status);
}

#define STST_RT_CHECK(call) ::stencil::cuda::internal::check((call), #call)

/// Make `device` current for the calling thread if it is not: a kernel launched on a stream must be
/// launched with the stream's device current.
inline void select_device(int device) {
#if defined(__CUDACC__)
    int current = -1;
    if (cudaGetDevice(&current) != cudaSuccess || current != device) {
        if (cudaSetDevice(device) != cudaSuccess)
            throw std::runtime_error("StencilStream-B200: cannot select CUDA device " +
                                     std::to_string(device));
    }
#else
    (void)device; // code compiled without nvcc launches no kernel
#endif
}

inline stst_stream_t default_stream(int device) {
    stst_stream_t s = nullptr;
    STST_RT_CHECK(stst_default_stream(device, &s));
    return s;
}

inline void *device_alloc(int device, std::size_t bytes, stst_stream_t stream) {
    void *p = nullptr;
    STST_RT_CHECK(stst_malloc(device, bytes, stream, &p));
    return p;
}

inline void device_free(int device, void *p, stst_stream_t stream) noexcept {
    if (p)
        (void)stst_free(device, p, stream);
}

inline void *pinned_alloc(std::size_t bytes) {
    void *p = nullptr;
    STST_RT_CHECK(stst_malloc_host(bytes, &p));
    return p;
}

inline void pinned_free(void *p) noexcept {
    if (p)
        (void)stst_free_host(p);
}

/// RAII event.
class Event {
  public:
    explicit Event(bool timing = false) : ev(nullptr) {
        STST_RT_CHECK(stst_event_create(timing ? 1 : 0, &ev));
    }
    Event(Event const &) = delete;
    Event &operator=(Event const &) = delete;
    Event(Event &&o) noexcept : ev(o.ev) { o.ev = nullptr; }
    ~Event() {
        if (ev)
            (void)stst_event_destroy(ev);
    }
    void record(stst_stream_t stream) { STST_RT_CHECK(stst_event_record(ev, stream)); }
    void synchronize() { STST_RT_CHECK(stst_event_synchronize(ev)); }
    stst_event_t get() const { return ev; }

  private:
    stst_event_t ev;
};

} // namespace internal
} // namespace cuda
} // namespace stencil
