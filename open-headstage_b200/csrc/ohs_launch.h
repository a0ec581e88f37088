// ohs_launch.h — host-side launchers of the render kernel, one translation unit per transform size (ohs_render.cu is
// compiled with -DOHS_RENDER_N=128/256/512/1024/2048 so that the sizes build in parallel), and the two dispatch rules
// every launcher shares: transform size to template, and function attributes once per device.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <type_traits>

#include "ohs_kernels.cuh"

namespace ohs {

struct RenderLaunch {
    int streams_per_cta;   // G: template instantiation to run
    int device;            // for the once-per-device function attributes
    cudaStream_t stream;
    int first_stream;      // the launch renders streams [first_stream, n_streams) of RenderParams
    int variant;           // RenderSmem V: 0 throughput, 1 latency (launches of one or two blocks; N = 512, else ignored),
                           // 2 EQ-only pre-pass of the time-batched route (N = 512 only: render_launch<512>)
    size_t min_smem_bytes; // EQ-only variant: ask for at least this much dynamic shared memory (keeps other kernels' CTAs off the SM)
    bool dependent;        // programmatic dependent launch: this grid may start while the previous launch on the stream
                           // drains; the kernel waits (griddepcontrol.wait) before it touches stream state
    bool moving;           // render_kernel<N, G, V, true>: per-block HRIR sets with crossfaded transitions (variants 0 and 1)
};

// cudaSuccess, or the CUDA error of the attribute call / launch; cudaErrorInvalidConfiguration if G does not fit.
// Instantiated in ohs_render.cu, one transform size per object.
template <int N> cudaError_t render_launch(const RenderLaunch&, const RenderParams&);
// whether render_kernel<N, streams_per_cta> fits in shared memory
template <int N> bool render_fits(int streams_per_cta);

// f(std::integral_constant<int, N>{}) for the runtime transform size n = 2 * block, one of the sizes ohs_create
// accepts; `otherwise` for any other n
template <typename R, typename F> R with_transform_size(int n, R otherwise, F&& f) {
    switch (n) {
        case 128: return f(std::integral_constant<int, 128>{});
        case 256: return f(std::integral_constant<int, 256>{});
        case 512: return f(std::integral_constant<int, 512>{});
        case 1024: return f(std::integral_constant<int, 1024>{});
        case 2048: return f(std::integral_constant<int, 2048>{});
    }
    return otherwise;
}

// Function attributes are per device: a launcher keeps one static OncePerDevice per kernel and sets the kernel's
// attributes through it.  Handles on different threads may race here, hence atomic flags (setting an attribute twice
// is harmless).  Devices outside 0..63 are never set.
struct OncePerDevice {
    std::atomic<unsigned char> done[64];
    // set() (a cudaError_t) unless it has succeeded for `device` before
    template <typename F> cudaError_t run(int device, F&& set) {
        if (device < 0 || device >= 64 || done[device].load(std::memory_order_acquire)) return cudaSuccess;
        const cudaError_t e = set();
        if (e == cudaSuccess) done[device].store(1, std::memory_order_release);
        return e;
    }
};

}  // namespace ohs
