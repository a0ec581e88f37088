// ohs_render.cu — the render kernel's instantiations and launcher for ONE transform size; compiled once per size with
// -DOHS_RENDER_N=<128|256|512|1024|2048> (open-headstage_b200/_build.py builds the five objects in parallel).
#include "ohs_launch.h"

#ifndef OHS_RENDER_N
#error "compile with -DOHS_RENDER_N=<transform size>"
#endif

namespace ohs {
namespace {

template <int N, int G, int V, bool Moving = false> cudaError_t launch_gv(const RenderLaunch& L, const RenderParams& p) {
    using SM = RenderSmem<N, G, V>;
    if constexpr (!SM::kFits) {
        return cudaErrorInvalidConfiguration;
    } else {
        constexpr auto kernel = render_kernel<N, G, V, Moving>;
        static OncePerDevice attrs;
        const cudaError_t e = attrs.run(L.device, [] {
            const cudaError_t r = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kEqOnly ? 227 * 1024 : (int)SM::kBytes);
            return r != cudaSuccess ? r : cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        });
        if (e != cudaSuccess) return e;
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
template <int N, int G> cudaError_t launch_g(const RenderLaunch& L, const RenderParams& p) {
    if constexpr (N == 512) {
        if (L.variant == 2) {
            if constexpr (RenderSmem<N, G, 2>::kFits) { if (!L.moving) return launch_gv<N, G, 2>(L, p); }
            return cudaErrorInvalidConfiguration;
        }
        if constexpr (RenderSmem<N, G, 1>::kFits) {
            if (L.variant == 1) return L.moving ? launch_gv<N, G, 1, true>(L, p) : launch_gv<N, G, 1>(L, p);
        }
    } else {
        if (L.variant == 2) return cudaErrorInvalidConfiguration;
    }
    return L.moving ? launch_gv<N, G, 0, true>(L, p) : launch_gv<N, G, 0>(L, p);
}

}  // namespace

template <int N> cudaError_t render_launch(const RenderLaunch& L, const RenderParams& p) {
    switch (L.streams_per_cta) {
        case 1: return launch_g<N, 1>(L, p);
        case 2: return launch_g<N, 2>(L, p);
        case 3: return launch_g<N, 3>(L, p);
        case 4: return launch_g<N, 4>(L, p);
        case 5: return launch_g<N, 5>(L, p);
        case 6: return launch_g<N, 6>(L, p);
        case 7: return launch_g<N, 7>(L, p);
    }
    return cudaErrorInvalidConfiguration;
}

template <int N> bool render_fits(int g) {
    constexpr bool fits[kMaxG + 1] = {false, RenderSmem<N, 1>::kFits, RenderSmem<N, 2>::kFits, RenderSmem<N, 3>::kFits, RenderSmem<N, 4>::kFits,
                                      RenderSmem<N, 5>::kFits, RenderSmem<N, 6>::kFits, RenderSmem<N, 7>::kFits};
    return g >= 1 && g <= kMaxG && fits[g];
}

template cudaError_t render_launch<OHS_RENDER_N>(const RenderLaunch&, const RenderParams&);
template bool render_fits<OHS_RENDER_N>(int);

}  // namespace ohs
