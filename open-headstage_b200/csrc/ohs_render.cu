// ohs_render.cu — the render kernel's instantiations and launcher for ONE transform size; compiled once per size with
// -DOHS_RENDER_N=<128|256|512|1024|2048> (open-headstage_b200/_build.py builds the five objects in parallel).
#include <atomic>

#include "ohs_launch.h"

#ifndef OHS_RENDER_N
#error "compile with -DOHS_RENDER_N=<transform size>"
#endif

namespace ohs {
namespace {

constexpr int N = OHS_RENDER_N;

template <int G, int V, bool Moving = false> cudaError_t launch_gv(const RenderLaunch& L, const RenderParams& p) {
    using SM = RenderSmem<N, G, V>;
    if constexpr (!SM::kFits) {
        return cudaErrorInvalidConfiguration;
    } else {
        constexpr auto kernel = render_kernel<N, G, V, Moving>;
        // function attributes are per device; distinct handles may race here, so the flags are atomic (setting an
        // attribute twice is harmless)
        static std::atomic<unsigned char> attr_set[64];
        if (L.device >= 0 && L.device < 64 && !attr_set[L.device].load(std::memory_order_acquire)) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kEqOnly ? 227 * 1024 : (int)SM::kBytes);
            if (e != cudaSuccess) return e;
            e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (e != cudaSuccess) return e;
            attr_set[L.device].store(1, std::memory_order_release);
        }
        const int n = p.n_streams - L.first_stream;
        if (n <= 0) return cudaSuccess;
        RenderParams q = p;
        q.first_stream = L.first_stream;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)((n + G - 1) / G));
        cfg.blockDim = dim3((unsigned)SM::kThreads);
        cfg.dynamicSmemBytes = (SM::kEqOnly && L.min_smem_bytes > SM::kBytes) ? L.min_smem_bytes : SM::kBytes;
        cfg.stream = L.stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = L.dependent ? 1 : 0;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, kernel, q);
    }
}

// the latency variant (RenderSmem, V = 1) where it exists and fits, else the throughput variant; the EQ-only variant
// (V = 2) on request, for static launches only
template <int G> cudaError_t launch_g(const RenderLaunch& L, const RenderParams& p) {
    if constexpr (N == 512) {
        if (L.variant == 2) {
            if constexpr (RenderSmem<N, G, 2>::kFits) { if (!L.moving) return launch_gv<G, 2>(L, p); }
            return cudaErrorInvalidConfiguration;
        }
        if constexpr (RenderSmem<N, G, 1>::kFits) {
            if (L.variant == 1) return L.moving ? launch_gv<G, 1, true>(L, p) : launch_gv<G, 1>(L, p);
        }
    } else {
        if (L.variant == 2) return cudaErrorInvalidConfiguration;
    }
    return L.moving ? launch_gv<G, 0, true>(L, p) : launch_gv<G, 0>(L, p);
}

template <int G> constexpr int threads_g() {
    if constexpr (RenderSmem<N, G>::kFits) return RenderSmem<N, G>::kThreads;
    else return 0;
}

}  // namespace

#define OHS_CAT2(a, b) a##b
#define OHS_CAT(a, b) OHS_CAT2(a, b)

cudaError_t OHS_CAT(render_launch_, OHS_RENDER_N)(const RenderLaunch& L, const RenderParams& p) {
    switch (L.streams_per_cta) {
        case 1: return launch_g<1>(L, p);
        case 2: return launch_g<2>(L, p);
        case 3: return launch_g<3>(L, p);
        case 4: return launch_g<4>(L, p);
        case 5: return launch_g<5>(L, p);
        case 6: return launch_g<6>(L, p);
        case 7: return launch_g<7>(L, p);
    }
    return cudaErrorInvalidConfiguration;
}

int OHS_CAT(render_threads_, OHS_RENDER_N)(int g) {
    switch (g) {
        case 1: return threads_g<1>(); case 2: return threads_g<2>(); case 3: return threads_g<3>(); case 4: return threads_g<4>();
        case 5: return threads_g<5>(); case 6: return threads_g<6>(); case 7: return threads_g<7>();
    }
    return 0;
}

bool OHS_CAT(render_fits_, OHS_RENDER_N)(int g) { return OHS_CAT(render_threads_, OHS_RENDER_N)(g) > 0; }

}  // namespace ohs
