// ohs_launch.h — host-side launchers of the render kernel, one translation unit per transform size (ohs_render.cu is
// compiled with -DOHS_RENDER_N=128/256/512/1024/2048 so that the sizes build in parallel).
#pragma once

#include <cuda_runtime.h>

#include "ohs_kernels.cuh"

namespace ohs {

struct RenderLaunch {
    int streams_per_cta;   // G: template instantiation to run
    int device;            // for the once-per-device function attributes
    cudaStream_t stream;
    int first_stream;      // the launch renders streams [first_stream, n_streams) of RenderParams
    int variant;           // RenderSmem V: 0 throughput, 1 latency (launches of one or two blocks; N = 512, else ignored),
                           // 2 EQ-only pre-pass of the time-batched route (N = 512 only: render_launch_512)
    size_t min_smem_bytes; // EQ-only variant: ask for at least this much dynamic shared memory (keeps other kernels' CTAs off the SM)
    bool dependent;        // programmatic dependent launch: this grid may start while the previous launch on the stream
                           // drains; the kernel waits (griddepcontrol.wait) before it touches stream state
    bool moving;           // render_kernel<N, G, V, true>: per-block HRIR sets with crossfaded transitions (variants 0 and 1)
};

// cudaSuccess, or the CUDA error of the attribute call / launch; cudaErrorInvalidConfiguration if G does not fit
#define OHS_DECLARE_RENDER(N)                                                  \
    cudaError_t render_launch_##N(const RenderLaunch&, const RenderParams&);  \
    bool render_fits_##N(int streams_per_cta);                                 \
    int render_threads_##N(int streams_per_cta);
OHS_DECLARE_RENDER(128)
OHS_DECLARE_RENDER(256)
OHS_DECLARE_RENDER(512)
OHS_DECLARE_RENDER(1024)
OHS_DECLARE_RENDER(2048)
#undef OHS_DECLARE_RENDER

}  // namespace ohs
