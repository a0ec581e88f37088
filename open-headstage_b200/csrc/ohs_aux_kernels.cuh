// ohs_aux_kernels.cuh — the kernels around the fused render kernel: HRIR set-up (set_ir), the time-batched long-response
// route (history gather, per-bin convolution along time, inverse transforms), history reset and the object mixdown.
// Included by ohs_api.cu only (the non-template kernels here have external linkage); the render kernel's templates
// live in ohs_kernels.cuh and are instantiated per transform size in ohs_render.cu.
#pragma once

#include "ohs_kernels.cuh"

namespace ohs {

// Threads per transform of the stand-alone forward and inverse kernels: twice the render kernel's where that keeps the
// radix plan (8 points per thread instead of 16: same butterflies, same twiddles, bit-identical spectra), because these
// kernels are bound by memory latency and want warps, not registers
constexpr int xform_threads(int n) { return (n / fft_threads(n) >= 16) ? 2 * fft_threads(n) : fft_threads(n); }

// ---------------------------------------------------------------------------------------------------------------
// HRIR set-up: ConvolutionEngine::set_ir (src/dsp/convolution.rs:111-139) for one (set, partition) per CTA.
// ir: [set][4][pmax*B] zero-padded time-domain taps; filt: [set][pmax][N]
// ---------------------------------------------------------------------------------------------------------------
template <int N> struct SetupSmem {
    static constexpr int T = fft_threads(N);
    static constexpr int TX = xform_threads(N);   // the stand-alone forward and inverse kernels of the time-batched route
    static_assert(FftPlan<N, TX>::R1 == FftPlan<N, T>::R1 && FftPlan<N, TX>::R2 == FftPlan<N, T>::R2 && FftPlan<N, TX>::R3 == FftPlan<N, T>::R3 &&
                  FftPlan<N, TX>::R4 == FftPlan<N, T>::R4, "same radix plan, hence bit-identical transforms");
    static constexpr int NP = padded_len(N);
    static constexpr size_t kBytes = sizeof(float2) * (N + 4 * NP);
};

// first-pass loader: an impulse-response chunk of two paths as (re, im), zero-padded from B to N (:123-129)
struct IrChunk {
    const float* ha; const float* hb; int B;
    __device__ __forceinline__ float2 ld(int i) const { return i < B ? make_float2(ha[i], hb[i]) : make_float2(0.f, 0.f); }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const { a = ld(i); b = ld(i + 1); }
};

template <int N>
__global__ void __launch_bounds__(SetupSmem<N>::T) setup_filters_kernel(const float* __restrict__ ir, float4* __restrict__ filt,
                                                                      const float2* __restrict__ tw_g,
                                                                      const int* __restrict__ set_list,
                                                                      const int* __restrict__ set_parts, int pmax) {
    using SM = SetupSmem<N>;
    constexpr int B = N / 2, T = SM::T, NP = SM::NP;
    using Pl = FftPlan<N, T>;
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tw = reinterpret_cast<float2*>(smem);
    float2* a0 = tw + N;
    float2* a1 = a0 + NP;
    float2* c0 = a1 + NP;
    float2* c1 = c0 + NP;
    const int tid = threadIdx.x;
    const int part = blockIdx.x;
    const int set = set_list[blockIdx.y];
    if (part >= set_parts[set]) return;
    for (int i = tid; i < N; i += T) tw[i] = tw_g[i];
    __syncthreads();
    const float* h = ir + (size_t)set * 4 * pmax * B + (size_t)part * B;
    const size_t ps = (size_t)pmax * B;  // path stride
    auto sync = [&]() { __syncthreads(); };
    const SmemCx gl{Pl::kOutInB0 ? a0 : a1}, gr{Pl::kOutInB0 ? c0 : c1};
    // G_L = FFT(h_LSL + i h_LSR), G_R = FFT(h_RSL + i h_RSR)
    fft_run<N, T>(tid, tw, a0, a1, IrChunk{h, h + ps, B}, gl, sync, [&]() {});
    fft_run<N, T>(tid, tw, c0, c1, IrChunk{h + 2 * ps, h + 3 * ps, B}, gr, sync, [&]() {});
    __syncthreads();
    const float sc = 1.0f / (2.0f * (float)N);  // 1/2 of the real/imag split and the 1/FFT_SIZE of :280, exact power of two
    float4* dst = filt + ((size_t)set * pmax + part) * N;
    for (int k = tid; k < N; k += T) {
        const float2 l = gl.ld(k), r = gr.ld(k);
        // even bins first, odd bins behind them: the layout the convolution warps' lane-contiguous loads want
        dst[(k & 1) * (N / 2) + (k >> 1)] = make_float4((l.x + r.y) * sc, (l.y - r.x) * sc, (l.x - r.y) * sc, (l.y + r.x) * sc);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Time-batched long responses (SURVEY 8f: the offline per-bin pipeline).  The fused kernel re-reads every stream's
// delay line (P-1 spectra of 8N bytes) for every block; for a launch of K blocks with a long response that is K(P-1)
// spectrum reads per stream where K + P - 1 would do.  In this mode the render kernel only filters and transforms
// (EQ, forward FFT, spectra into the delay-line ring AND into a buffer in time order), then per bin
//     W_t[k] = sum_q  Z_{t-q}[k] A_q[k] + conj(Z_{t-q}[N-k]) C_q[k]
// is a short convolution ALONG TIME: a thread owns a bin couple (k, N-k) of one stream and TB consecutive blocks,
// keeps their TB accumulators and a sliding window of TB spectra in registers, and walks q once — one new spectrum
// value and one filter tap loaded per step for TB*16 FMAs.  A third kernel runs the inverse transforms.
// ---------------------------------------------------------------------------------------------------------------
// The time-ordered buffer is CIRCULAR in time: `cap` slots per stream, the slot of the next block (`zbase`) moves on
// by the blocks rendered, and the pmax-1 slots behind it hold the history — so consecutive time-batched sub-launches
// and calls find their history in place and nothing is copied between them.  The delay-line ring (what the
// block-by-block kernel reads) and the buffer are converted into each other only when the route changes:
// ring -> buffer (time -q, q = 1..pmax-1, goes to slot zbase - q) ...
__global__ void gather_history_kernel(const float2* __restrict__ fdl, float2* __restrict__ zlin, int N, int pmax, int head,
                                      long long zlin_stride, int zbase, int cap) {
    const int q = blockIdx.x + 1, s = blockIdx.y;
    int sl = head - q; if (sl < 0) sl += pmax;
    int zs = zbase - q; if (zs < 0) zs += cap;
    const float4* src = reinterpret_cast<const float4*>(fdl + ((size_t)s * pmax + sl) * N);
    float4* dst = reinterpret_cast<float4*>(zlin + (size_t)s * zlin_stride + (size_t)zs * N);
    for (int i = threadIdx.x; i < N / 2; i += blockDim.x) dst[i] = src[i];
}
// ... and buffer -> ring
__global__ void scatter_history_kernel(const float2* __restrict__ zlin, float2* __restrict__ fdl, int N, int pmax, int head,
                                       long long zlin_stride, int zbase, int cap) {
    const int q = blockIdx.x + 1, s = blockIdx.y;
    int sl = head - q; if (sl < 0) sl += pmax;
    int zs = zbase - q; if (zs < 0) zs += cap;
    const float4* src = reinterpret_cast<const float4*>(zlin + (size_t)s * zlin_stride + (size_t)zs * N);
    float4* dst = reinterpret_cast<float4*>(fdl + ((size_t)s * pmax + sl) * N);
    for (int i = threadIdx.x; i < N / 2; i += blockDim.x) dst[i] = src[i];
}

// Block = 4 warps = 4 streams x 32 bin couples: the four warps read the same filter taps (they hit in L1), each its own
// stream's spectra (32 couples x 8 bytes contiguous per load).  The window of TB spectra lives in shared memory, one
// 16-byte column entry per thread and slot (slot = time mod TB), so the step loop needs no unrolling over the
// window's rotation: fully unrolled it is 90 KB of code and the kernel stalls on instruction fetch.
// Two steps (partitions q and q+1) per iteration: the window value of time tau meets tap q in block tau+q and tap q+1 in
// block tau+q+1, so every value read from the shared-memory window feeds 32 FMAs instead of 16 — the per-step form
// spent as many shared-memory wavefront cycles as FMA issue cycles (16 LDS.128 per 256 FMAs per thread).  The value of
// time t0-q-1, which block t0 needs for tap q+1, is the one that has just been loaded from the time-ordered buffer and
// is still in registers.  An odd last partition runs the single step.
template <int TB, bool kDc>
__device__ __forceinline__ void bin_conv_steps(float2 (&a0)[TB], float2 (&a1)[TB], float4* win, const float4* __restrict__ f,
                                               const float2* __restrict__ z, int N, int nparts, int zslot, int cap, int f0i, int f1i,
                                               int k0, int k1) {
    // One iteration's operands: the taps of partitions q and q+1 for the thread's two bins, and the spectra of times
    // t0-q-1 and t0-q-2, which enter the window behind them.  They are loaded one iteration ahead (an iteration is ~570
    // instructions, more than a loaded HBM round trip) into the register set the other iteration does not use (the
    // loop is unrolled by two by hand: no register moves), taps through running pointers, spectra through a running slot.
    struct Ops { float4 fa0, fb0, fa1, fb1, n0, n1; };
    // `z`: the stream's circular time-ordered buffer (cap slots); `zslot`: the slot of the thread's first block t0
    const float4* pf0 = f + f0i;
    const float4* pf1 = f + f1i;
    const long long N2 = 2ll * N;
    int sz = zslot - 1; if (sz < 0) sz += cap;   // slot of time t0-q-1, walking back two slots per iteration
    auto load = [&](Ops& o, int q) {
        if (q < nparts) { o.fa0 = pf0[0]; o.fb0 = pf1[0]; }
        if (q + 1 < nparts) { o.fa1 = pf0[N]; o.fb1 = pf1[N]; }
        // the spectra loads are unconditional: a wrapped slot is always inside the stream's buffer, and a value that no
        // partition needs is never used (a conditional load here compiles to a branch that pins the load behind it)
        int s1 = sz - 1; if (s1 < 0) s1 += cap;
        const float2* zp0 = z + (long long)sz * N;
        const float2* zp1 = z + (long long)s1 * N;
        const float2 x0 = zp0[k0], y0 = zp0[k1], x1 = zp1[k0], y1 = zp1[k1];
        o.n0 = make_float4(x0.x, x0.y, y0.x, y0.y);
        o.n1 = make_float4(x1.x, x1.y, y1.x, y1.y);
        pf0 += N2; pf1 += N2;
        sz = s1 - 1; if (sz < 0) sz += cap;
    };
    auto pair_step = [&](const Ops& o, int q) {
        const int rot = (TB - (q & (TB - 1))) & (TB - 1);   // slot of time t0+tb-q is (tb + rot) mod TB
        const float4* wrot = win + rot * 128;               // every slot is stored twice, TB slots apart: no wrap in the reads
        {
            const float2 u0 = make_float2(o.n0.x, o.n0.y), u1 = make_float2(o.n0.z, o.n0.w);   // time t0-q-1, tap q+1, block t0
            mac_bin(a0[0], u0, kDc ? u0 : u1, o.fa1);
            mac_bin(a1[0], u1, kDc ? u1 : u0, o.fb1);
        }
#pragma unroll
        for (int tb = 0; tb < TB; ++tb) {
            const float4 v = wrot[tb * 128];
            const float2 u0 = make_float2(v.x, v.y), u1 = make_float2(v.z, v.w);
            mac_bin(a0[tb], u0, kDc ? u0 : u1, o.fa0);   // couple 0 = the two self-mirrored bins 0 and N/2
            mac_bin(a1[tb], u1, kDc ? u1 : u0, o.fb0);
            if (tb + 1 < TB) {
                mac_bin(a0[tb + 1], u0, kDc ? u0 : u1, o.fa1);
                mac_bin(a1[tb + 1], u1, kDc ? u1 : u0, o.fb1);
            }
        }
        // the window moves two blocks back: times t0-q-1 and t0-q-2 replace times t0+TB-1-q and t0+TB-2-q
        const int e1 = (TB - 1 + rot) & (TB - 1), e2 = (TB - 2 + rot) & (TB - 1);
        win[e1 * 128] = o.n0; win[(e1 + TB) * 128] = o.n0;
        win[e2 * 128] = o.n1; win[(e2 + TB) * 128] = o.n1;
    };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    Ops A{zero4, zero4, zero4, zero4, zero4, zero4}, B = A;
    load(A, 0);
    const int npairs = nparts >> 1;
#pragma unroll 1
    for (int p = 0; p < npairs; p += 2) {
        load(B, 2 * p + 2);
        pair_step(A, 2 * p);
        if (p + 1 < npairs) {
            load(A, 2 * p + 4);
            pair_step(B, 2 * p + 2);
        }
    }
    if (nparts & 1) {   // odd partition count: one single step (no later step reads the window)
        const int q = nparts - 1;
        const bool in_a = (npairs & 1) == 0;   // the set the last load went to
        const float4 fa = in_a ? A.fa0 : B.fa0, fb = in_a ? A.fb0 : B.fb0;
        const int rot = (TB - (q & (TB - 1))) & (TB - 1);
        const float4* wrot = win + rot * 128;
#pragma unroll
        for (int tb = 0; tb < TB; ++tb) {
            const float4 v = wrot[tb * 128];
            const float2 u0 = make_float2(v.x, v.y), u1 = make_float2(v.z, v.w);
            mac_bin(a0[tb], u0, kDc ? u0 : u1, fa);
            mac_bin(a1[tb], u1, kDc ? u1 : u0, fb);
        }
    }
}

template <int TB>
__global__ void __launch_bounds__(128, 3) bin_conv_kernel(const float2* __restrict__ zlin, float2* __restrict__ wlin,
                                                       const float4* __restrict__ filt, const int* __restrict__ stream_hrir,
                                                       const int* __restrict__ set_parts, int N, int pmax, int K, int n_streams,
                                                       long long zlin_stride, int zslot0, int cap) {
    static_assert((TB & (TB - 1)) == 0, "window slots are indexed modulo a power of two");
    extern __shared__ __align__(16) unsigned char smem[];
    float4* win = reinterpret_cast<float4*>(smem) + threadIdx.x;   // this thread's column: slot e at win[e * 128]
    const int i = blockIdx.x * 32 + (threadIdx.x & 31);   // couple index: bins (i, N-i); couple 0 is (0, N/2)
    const int t0 = blockIdx.y * TB, s = blockIdx.z * 4 + (threadIdx.x >> 5);
    if (i >= N / 2 || s >= n_streams) return;
    const int k0 = i, k1 = i ? N - i : N / 2;
    const int set = stream_hrir[s];
    const int nparts = set_parts[set];
    const float4* f = filt + (size_t)set * pmax * N;
    const int f0i = (k0 & 1) * (N / 2) + (k0 >> 1), f1i = (k1 & 1) * (N / 2) + (k1 >> 1);   // even-bins-first table layout
    const float2* z = zlin + (size_t)s * zlin_stride;   // circular: block t of this launch sits in slot (zslot0 + t) mod cap
    int zs = zslot0 + t0; if (zs >= cap) zs -= cap;
    float2 a0[TB], a1[TB];
    {
        // the window's first TB spectra: every load unconditional (blocks past the launch's last re-read that one and are
        // zeroed by a select) and issued before the first store, so that the TB round trips overlap
        float2 v0[TB], v1[TB];
        const int last = K - 1 - t0;
#pragma unroll
        for (int tb = 0; tb < TB; ++tb) {
            int sl = zs + (tb < last ? tb : last); if (sl >= cap) sl -= cap;
            v0[tb] = z[(size_t)sl * N + k0];
            v1[tb] = z[(size_t)sl * N + k1];
        }
#pragma unroll
        for (int tb = 0; tb < TB; ++tb) {
            a0[tb] = make_float2(0.f, 0.f); a1[tb] = make_float2(0.f, 0.f);
            const bool live = tb <= last;
            const float4 v = live ? make_float4(v0[tb].x, v0[tb].y, v1[tb].x, v1[tb].y) : make_float4(0.f, 0.f, 0.f, 0.f);
            win[tb * 128] = v;
            win[(tb + TB) * 128] = v;
        }
    }
    // couple 0 (bins 0 and N/2, each its own mirror) lives in lane 0 of the first couple group's warps only
    if (blockIdx.x == 0) {
        if (i == 0) bin_conv_steps<TB, true>(a0, a1, win, f, z, N, nparts, zs, cap, f0i, f1i, k0, k1);
        else bin_conv_steps<TB, false>(a0, a1, win, f, z, N, nparts, zs, cap, f0i, f1i, k0, k1);
    } else {
        bin_conv_steps<TB, false>(a0, a1, win, f, z, N, nparts, zs, cap, f0i, f1i, k0, k1);
    }
    float2* w = wlin + ((size_t)s * K) * N;
#pragma unroll
    for (int tb = 0; tb < TB; ++tb)
        if (t0 + tb < K) { w[(size_t)(t0 + tb) * N + k0] = a0[tb]; w[(size_t)(t0 + tb) * N + k1] = a1[tb]; }
}

// first-pass loader of the forward transform from global memory: the overlap-save window [previous block | current block]
// of a stream's EQ-filtered rows, z = left + i*right
struct RowWindow {
    const float* pl; const float* pr; const float* cl; const float* cr; int B;   // cl/cr already offset by -B
    __device__ __forceinline__ float2 ld(int i) const { return i < B ? make_float2(pl[i], pr[i]) : make_float2(cl[i], cr[i]); }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const {  // i even: samples i and i+1
        const float2 l = *reinterpret_cast<const float2*>((i < B ? pl : cl) + i), r = *reinterpret_cast<const float2*>((i < B ? pr : cr) + i);
        a = make_float2(l.x, r.x); b = make_float2(l.y, r.y);
    }
};

// last-pass store of the forward transform: the packed spectrum goes straight from registers to its slot of the
// time-ordered buffer
struct SpectrumStore {
    float2* zl;
    __device__ __forceinline__ void st(int i, float2 v) const { zl[i] = v; }
    __device__ __forceinline__ void st2(int i, float2 a, float2 b) const {
        *reinterpret_cast<float4*>(zl + i) = make_float4(a.x, a.y, b.x, b.y);
    }
};

// one CTA per (block, stream): forward transform of block t0 + blockIdx.x of the filtered rows `xf` (block 0's history is
// the engine's overlap-save block `prev`), same plan and rounding as the render kernel's forward transform, into slot
// (zlin_base + t) mod cap of the circular time-ordered buffer.  (The delay-line ring is not written here: it is rebuilt
// from the buffer when something needs it, scatter_history_kernel.)
template <int N>
__global__ void __launch_bounds__(SetupSmem<N>::TX) forward_kernel(const float* __restrict__ xf, long long xf_stride, int t0,
                                                                 const float* __restrict__ prev, float2* __restrict__ zlin,
                                                                 long long zlin_stride, int zlin_base, int cap,
                                                                 const float2* __restrict__ tw_g) {
    constexpr int T = SetupSmem<N>::TX, NP = SetupSmem<N>::NP, B = N / 2;
    extern __shared__ __align__(16) unsigned char smem[];
    float2* b0 = reinterpret_cast<float2*>(smem);
    float2* b1 = b0 + NP;
    const int t = t0 + blockIdx.x, s = blockIdx.y;
    const float* cl = xf + ((size_t)s * 2) * xf_stride + (size_t)t * B;
    const float* cr = cl + xf_stride;
    const float* pl = t ? cl - B : prev + (size_t)s * 2 * B;
    const float* pr = t ? cr - B : pl + B;
    int zs = zlin_base + t; if (zs >= cap) zs -= cap;
    float2* zl = zlin + (size_t)s * zlin_stride + (size_t)zs * N;
    auto sync = [&]() { __syncthreads(); };
    fft_run<N, T>(threadIdx.x, tw_g, b0, b1, RowWindow{pl, pr, cl - B, cr - B, B}, SpectrumStore{zl}, sync, [&]() {});
}

// first-pass loader of the inverse transform from global memory, with the swap of swap o FFT o swap
struct SpectrumSwapLoad {
    const float2* w;
    __device__ __forceinline__ float2 ld(int i) const { const float2 v = w[i]; return make_float2(v.y, v.x); }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const {
        const float4 v = *reinterpret_cast<const float4*>(w + i);
        a = make_float2(v.y, v.x); b = make_float2(v.w, v.z);
    }
};

// one CTA per (block, stream): inverse transform of W_t, last B samples times gain to the output rows
template <int N>
__global__ void __launch_bounds__(SetupSmem<N>::TX) inverse_kernel(const float2* __restrict__ wlin, float* __restrict__ out,
                                                                const float2* __restrict__ tw_g, const float* __restrict__ stream_gain,
                                                                int K, long long row_stride) {
    constexpr int T = SetupSmem<N>::TX, NP = SetupSmem<N>::NP, B = N / 2;
    extern __shared__ __align__(16) unsigned char smem[];
    float2* b0 = reinterpret_cast<float2*>(smem);
    float2* b1 = b0 + NP;
    const int t = blockIdx.x, s = blockIdx.y;
    const float2* w = wlin + ((size_t)s * K + t) * N;
    float* out_l = out + ((size_t)s * 2) * row_stride;
    float* out_r = out_l + row_stride;
    auto sync = [&]() { __syncthreads(); };
    fft_run<N, T>(threadIdx.x, tw_g, b0, b1, SpectrumSwapLoad{w},
                  OutputStore{out_l + (size_t)t * B - B, out_r + (size_t)t * B - B, stream_gain[s], B}, sync, [&]() {});
}

// zero a stream's convolution history (delay line + overlap-save block) for streams bound to a flagged set, or all
// streams when set_flags is null
__global__ void clear_history_kernel(float2* fdl, float2* prev, const int* stream_hrir, int n_streams,
                                     const unsigned char* set_flags, size_t fdl_per_stream, size_t prev_per_stream) {
    const int s = blockIdx.x;
    if (s >= n_streams) return;
    if (set_flags && !set_flags[stream_hrir[s]]) return;
    float2* f = fdl + (size_t)s * fdl_per_stream;
    for (size_t i = threadIdx.x; i < fdl_per_stream; i += blockDim.x) f[i] = make_float2(0.f, 0.f);
    float2* q = prev + (size_t)s * prev_per_stream;
    for (size_t i = threadIdx.x; i < prev_per_stream; i += blockDim.x) q[i] = make_float2(0.f, 0.f);
}

// Group buses (ohs_set_groups; BASELINE config 4 is the single group of every stream): bus row 2g + c is the sum over the
// streams first[g] .. first[g+1]-1 of in[s][c][n], a sequential f32 sum from +0 in stream order (deterministic).  One thread
// per four frames and bus row: grid.x over 4-frame quads, grid.y over the 2G bus rows (rows past gridDim.y loop), so that
// groups of three or four streams still fill the GPU; rows read with coalesced 16-byte loads.  A row's last, partial quad
// (EQ-only calls of any length) is summed sample by sample, touching nothing past n_frames.
__global__ void mix_streams_kernel(const float* __restrict__ in, float* __restrict__ bus, const int* __restrict__ group_first,
                                   int n_rows, size_t n_frames, size_t row_stride, size_t bus_stride) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // float4 index inside a row
    if (q * 4 >= n_frames) return;
    for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
        const int g = r >> 1, c = r & 1;
        const int s0 = group_first[g], s1 = group_first[g + 1];
        const float* row = in + ((size_t)s0 * 2 + c) * row_stride + q * 4;
        float* dst = bus + (size_t)r * bus_stride + q * 4;
        if (q * 4 + 4 <= n_frames) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int s = s0; s < s1; ++s) {
                const float4 v = *reinterpret_cast<const float4*>(row + (size_t)(s - s0) * 2 * row_stride);
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
            *reinterpret_cast<float4*>(dst) = acc;
        } else {
            for (size_t k = 0; q * 4 + k < n_frames; ++k) {
                float acc = 0.f;
                for (int s = s0; s < s1; ++s) acc += row[(size_t)(s - s0) * 2 * row_stride + k];
                dst[k] = acc;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Integer PCM in and out (ohs_process_pcm, include/ohs.h): decode q -> q * 2^-(b-1) and encode
// clamp(rint(y * 2^(b-1))) with NaN -> 0, between PCM rows and f32 rows.  One thread converts one group of frames of one
// row with 16-byte accesses: 8 frames (one uint4) of S16, 16 frames (48 bytes, three uint4) of S24.  Row starts are
// 16-byte aligned on both sides (PCM rows: pitch a multiple of the group; f32 rows: of 4 frames); a row's last group
// may be partial and is converted sample by sample, touching nothing past n_frames.  Launched without the
// programmatic-serialization attribute: a render launch after a decode starts once the decode has finished, and an
// encode after a render waits for the whole render.
// ---------------------------------------------------------------------------------------------------------------
enum PcmFormat { kPcmF32 = 0, kPcmS16 = 1, kPcmS24 = 2 };   // OHS_FMT_*

template <int Fmt> struct PcmTraits;
template <> struct PcmTraits<kPcmF32> {   // f32 rows (sizes on the host only: no kernel converts F32)
    static constexpr int kBytes = 4, kGroup = 4;
};
template <> struct PcmTraits<kPcmS16> {
    static constexpr int kBytes = 2, kGroup = 8;
    static constexpr float kDecode = 0x1p-15f, kEncode = 0x1p15f, kLo = -32768.0f, kHi = 32767.0f;
};
template <> struct PcmTraits<kPcmS24> {
    static constexpr int kBytes = 3, kGroup = 16;
    static constexpr float kDecode = 0x1p-23f, kEncode = 0x1p23f, kLo = -8388608.0f, kHi = 8388607.0f;
};

// y * 2^(b-1) (exact), round to nearest even, clamp (clamping first is the same: the bounds are integers); NaN -> 0
template <int Fmt> __device__ __forceinline__ int pcm_quantise(float y) {
    using P = PcmTraits<Fmt>;
    const float v = y * P::kEncode;
    if (v != v) return 0;
    return __float2int_rn(fminf(fmaxf(v, P::kLo), P::kHi));
}

template <int Fmt> __device__ __forceinline__ int pcm_load_one(const unsigned char* p) {
    if (Fmt == kPcmS16) return (int)*reinterpret_cast<const short*>(p);
    return (int)(((unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16)) << 8) >> 8;
}

template <int Fmt> __device__ __forceinline__ void pcm_store_one(unsigned char* p, int q) {
    if (Fmt == kPcmS16) { *reinterpret_cast<short*>(p) = (short)q; return; }
    p[0] = (unsigned char)q; p[1] = (unsigned char)(q >> 8); p[2] = (unsigned char)(q >> 16);
}

// the kGroup samples of a whole group from its kGroup * kBytes / 4 little-endian words, and back
template <int Fmt> __device__ __forceinline__ void pcm_unpack(const unsigned (&w)[PcmTraits<Fmt>::kGroup * PcmTraits<Fmt>::kBytes / 4],
                                                              int (&q)[PcmTraits<Fmt>::kGroup]) {
    constexpr int G = PcmTraits<Fmt>::kGroup, NB = PcmTraits<Fmt>::kBytes;
#pragma unroll
    for (int k = 0; k < G; ++k) {
        const int o = k * NB, i = o >> 2, s = o & 3;
        if (Fmt == kPcmS16) {
            q[k] = s ? (int)w[i] >> 16 : (int)(short)(w[i] & 0xffffu);
        } else {
            const unsigned u = (s <= 1) ? (w[i] >> (8 * s)) : __funnelshift_r(w[i], w[i + 1 < G * NB / 4 ? i + 1 : i], 8 * s);
            q[k] = (int)(u << 8) >> 8;
        }
    }
}

template <int Fmt> __device__ __forceinline__ void pcm_pack(const int (&q)[PcmTraits<Fmt>::kGroup],
                                                            unsigned (&w)[PcmTraits<Fmt>::kGroup * PcmTraits<Fmt>::kBytes / 4]) {
    constexpr int G = PcmTraits<Fmt>::kGroup, NB = PcmTraits<Fmt>::kBytes, W = G * NB / 4;
#pragma unroll
    for (int j = 0; j < W; ++j) w[j] = 0u;
#pragma unroll
    for (int k = 0; k < G; ++k) {
        const int o = k * NB, i = o >> 2, s = o & 3;
        const unsigned u = (unsigned)q[k] & (NB == 2 ? 0xffffu : 0xffffffu);
        w[i] |= u << (8 * s);
        if (8 * s + 8 * NB > 32) w[i + 1 < W ? i + 1 : i] |= u >> (32 - 8 * s);
    }
}

// in: PCM rows (pitch in bytes), out: f32 rows (pitch in floats); `groups` = groups per row
template <int Fmt>
__global__ void __launch_bounds__(256) pcm_decode_kernel(const unsigned char* __restrict__ in, size_t in_pitch, float* __restrict__ out,
                                                         size_t out_pitch, size_t n_frames, size_t groups, size_t total) {
    using P = PcmTraits<Fmt>;
    constexpr int G = P::kGroup, NB = P::kBytes, W = G * NB / 4;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t row = t / groups, f0 = (t - row * groups) * G;
        const unsigned char* src = in + row * in_pitch + f0 * NB;
        float* dst = out + row * out_pitch + f0;
        if (f0 + G <= n_frames) {
            unsigned w[W];
#pragma unroll
            for (int v = 0; v < W / 4; ++v) {
                const uint4 x = reinterpret_cast<const uint4*>(src)[v];
                w[4 * v] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w;
            }
            int q[G];
            pcm_unpack<Fmt>(w, q);
#pragma unroll
            for (int v = 0; v < G / 4; ++v)
                reinterpret_cast<float4*>(dst)[v] = make_float4((float)q[4 * v] * P::kDecode, (float)q[4 * v + 1] * P::kDecode,
                                                                (float)q[4 * v + 2] * P::kDecode, (float)q[4 * v + 3] * P::kDecode);
        } else {
            for (size_t k = 0; f0 + k < n_frames; ++k) dst[k] = (float)pcm_load_one<Fmt>(src + k * NB) * P::kDecode;
        }
    }
}

// ---- dither (ohs_set_dither, include/ohs.h) ------------------------------------------------------------------------
// The noise of row r at dither position p: x = mix64(K_r + phi * (p + 1)) with K_r = mix64(seed + phi * (r + 1)) (SplitMix64's
// increment and finaliser), d = (u1 + u2 - (2^23 - 1)) * 2^-23 from the low 23 bits of each half of x: TPDF in (-1, 1) LSB,
// exact in f32.  A stateless function of (seed, r, p), so the noise does not depend on how a render is cut into calls.
constexpr unsigned long long kDitherPhi = 0x9E3779B97F4A7C15ull;
constexpr int kShapeTaps = 9;   // OHS_MAX_SHAPE_TAPS: taps of the error-feedback filter, and history floats per row

__device__ __forceinline__ unsigned long long dither_mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ unsigned long long dither_row_key(unsigned long long seed, size_t row) {
    return dither_mix64(seed + kDitherPhi * (row + 1));
}
// the noise of the position whose phi * (p + 1) has been added to the row key
__device__ __forceinline__ float dither_noise(unsigned long long keyed) {
    const unsigned long long x = dither_mix64(keyed);
    const int u1 = (int)(x & 0x7fffffu), u2 = (int)((x >> 32) & 0x7fffffu);
    return (float)(u1 + u2 - 0x7fffff) * 0x1p-23f;
}

// flat TPDF: clamp(rint(v + d)) with v + d rounded on its own (no contraction into an FMA with the exact scaling); NaN -> 0
template <int Fmt> __device__ __forceinline__ int pcm_quantise_dithered(float y, float d) {
    using P = PcmTraits<Fmt>;
    const float v = __fmul_rn(y, P::kEncode);
    if (v != v) return 0;
    return __float2int_rn(fminf(fmaxf(__fadd_rn(v, d), P::kLo), P::kHi));
}

// Mixed encode (bus rows, ohs_process_grouped_pcm / ohs_mix_device_pcm): row r of the output is bus row 2g + c, and its f32
// samples are the group's stream rows in[(2s + c)], s = group_first[g] .. group_first[g+1]-1, summed from +0 in ascending
// stream order (mix_streams_kernel's sum, bit for bit).  group_sum1: one frame, `src` at the group's first stream row;
// the ns rows sit 2 * pitch apart.
__device__ __forceinline__ float group_sum1(const float* src, int ns, size_t pitch) {
    float acc = 0.f;
    for (int s = 0; s < ns; ++s) acc += src[(size_t)s * 2 * pitch];
    return acc;
}

// in: f32 rows (pitch in floats), out: PCM rows (pitch in bytes).  Dither: flat TPDF, the group's first frame at dither
// position pos0 + f0 (the parameters behind `total` are read only then, so the undithered kernel is the plain encode).
// Mix: `total` counts the groups of the bus rows, and a thread sums its frames of the group's stream rows into registers
// first (the f32 bus is never stored); group_first is read only then.
template <int Fmt, bool Dither = false, bool Mix = false>
__global__ void __launch_bounds__(256) pcm_encode_kernel(const float* __restrict__ in, size_t in_pitch, unsigned char* __restrict__ out,
                                                         size_t out_pitch, size_t n_frames, size_t groups, size_t total,
                                                         unsigned long long seed, unsigned long long pos0,
                                                         const int* __restrict__ group_first) {
    using P = PcmTraits<Fmt>;
    constexpr int G = P::kGroup, NB = P::kBytes, W = G * NB / 4;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t row = t / groups, f0 = (t - row * groups) * G;
        const float* src = in + row * in_pitch + f0;
        unsigned char* dst = out + row * out_pitch + f0 * NB;
        // the samples of the thread's frames: the row itself, or (Mix) the group sums, all G of them in registers
        [[maybe_unused]] float4 mixed[G / 4];
        [[maybe_unused]] int ns = 0;
        if constexpr (Mix) {
            const int g = (int)(row >> 1), s0 = group_first[g];
            ns = group_first[g + 1] - s0;
            src = in + ((size_t)s0 * 2 + (row & 1)) * in_pitch + f0;
            if (f0 + G <= n_frames) {
#pragma unroll
                for (int v = 0; v < G / 4; ++v) mixed[v] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
                for (int s = 0; s < ns; ++s) {
                    const float* r = src + (size_t)s * 2 * in_pitch;
#pragma unroll
                    for (int v = 0; v < G / 4; ++v) {
                        const float4 x = reinterpret_cast<const float4*>(r)[v];
                        mixed[v].x += x.x; mixed[v].y += x.y; mixed[v].z += x.z; mixed[v].w += x.w;
                    }
                }
            }
        }
        auto sample4 = [&](int v) -> float4 {
            if constexpr (Mix) return mixed[v];
            else return reinterpret_cast<const float4*>(src)[v];
        };
        auto sample1 = [&](size_t k) -> float {
            if constexpr (Mix) return group_sum1(src + k, ns, in_pitch);
            else return src[k];
        };
        if constexpr (Dither) {
            unsigned long long z = dither_row_key(seed, row) + kDitherPhi * (pos0 + f0 + 1);
            if (f0 + G <= n_frames) {
                int q[G];
#pragma unroll
                for (int v = 0; v < G / 4; ++v) {
                    const float4 y = sample4(v);
                    const float ys[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) { q[4 * v + j] = pcm_quantise_dithered<Fmt>(ys[j], dither_noise(z)); z += kDitherPhi; }
                }
                unsigned w[W];
                pcm_pack<Fmt>(q, w);
#pragma unroll
                for (int v = 0; v < W / 4; ++v) reinterpret_cast<uint4*>(dst)[v] = make_uint4(w[4 * v], w[4 * v + 1], w[4 * v + 2], w[4 * v + 3]);
            } else {
                for (size_t k = 0; f0 + k < n_frames; ++k, z += kDitherPhi)
                    pcm_store_one<Fmt>(dst + k * NB, pcm_quantise_dithered<Fmt>(sample1(k), dither_noise(z)));
            }
        } else if (f0 + G <= n_frames) {
            int q[G];
#pragma unroll
            for (int v = 0; v < G / 4; ++v) {
                const float4 y = sample4(v);
                q[4 * v] = pcm_quantise<Fmt>(y.x); q[4 * v + 1] = pcm_quantise<Fmt>(y.y);
                q[4 * v + 2] = pcm_quantise<Fmt>(y.z); q[4 * v + 3] = pcm_quantise<Fmt>(y.w);
            }
            unsigned w[W];
            pcm_pack<Fmt>(q, w);
#pragma unroll
            for (int v = 0; v < W / 4; ++v) reinterpret_cast<uint4*>(dst)[v] = make_uint4(w[4 * v], w[4 * v + 1], w[4 * v + 2], w[4 * v + 3]);
        } else {
            for (size_t k = 0; f0 + k < n_frames; ++k) pcm_store_one<Fmt>(dst + k * NB, pcm_quantise<Fmt>(sample1(k)));
        }
    }
}

// ---- noise-shaped encode: error feedback along each row ----------------------------------------------------------
// One frame of row r (include/ohs.h): fb = h_M e_M + ... + h_1 e_1 summed oldest first, so the loop-carried chain through
// the newest error e_1 is one multiply and one add; w = v - fb; q = clamp(rint(w + d)); e = clamp(q - w, -1.5, 1.5).
// Every operation is rounded on its own (the build contracts to FMA by default; the numpy reference does not).
struct DitherTaps { float h[kShapeTaps]; };   // h[k] = h_(k+1)

// rint of a value already clamped to the format's range.  S16: |t| <= 2^15, so t + 1.5 * 2^23 lies in [2^23, 2^24), where the
// f32 ulp is 1: the add rounds to nearest even and the subtraction is exact, two 4-cycle adds on the loop-carried chain
// instead of FRND's trip through the conversion unit.  It gives +0 where rint gives -0 (t in [-0.5, 0]); a zero of the other
// sign only ever meets nonzero values in sums (x + -0 = x + 0 = x) and gives zeros in products, so no q changes.
template <int Fmt> __device__ __forceinline__ float rint_clamped(float t) {
    if constexpr (Fmt == kPcmS16) return __fsub_rn(__fadd_rn(t, 12582912.0f), 12582912.0f);
    else return rintf(t);
}

template <int Fmt, int M>
__device__ __forceinline__ int shaped_step(float y, float d, const DitherTaps& t, float (&e)[M]) {
    using P = PcmTraits<Fmt>;
    const float v = __fmul_rn(y, P::kEncode);
    float fb = __fmul_rn(t.h[M - 1], e[M - 1]);
#pragma unroll
    for (int k = M - 2; k >= 0; --k) fb = __fadd_rn(fb, __fmul_rn(t.h[k], e[k]));
    const float w = __fsub_rn(v, fb);
    const float qf = rint_clamped<Fmt>(fminf(fmaxf(__fadd_rn(w, d), P::kLo), P::kHi));   // clamping first is the same: integer bounds
    // NaN v: q - w is NaN, and fmaxf / fminf return the other operand, so bounds of 0 give the error 0 without a select on
    // the chain (v is known a frame ahead; finite or infinite v never makes q - w NaN)
    const bool nan = v != v;
    const float en = fminf(fmaxf(__fsub_rn(qf, w), nan ? 0.f : -1.5f), nan ? 0.f : 1.5f);
#pragma unroll
    for (int k = M - 1; k > 0; --k) e[k] = e[k - 1];
    e[0] = en;
    return nan ? 0 : __float2int_rn(qf);
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The recurrence runs in order along a row, so one thread owns one row: a CTA carries 32 rows in warp 0 and walks them
// in tiles of kShapeT frames.  The f32 tiles arrive through shared memory (coalesced 16-byte cp.async, double-buffered:
// tile k+1 loads while tile k is computed); warps 1-3 hash the noise of tile k+1 into shared memory meanwhile, which keeps the
// ~25 integer instructions of a noise value out of warp 0's issue slots.  Warp 0 writes the packed integers of its row to a
// byte tile that the whole CTA stores with 16-byte stores.  Tile rows are padded by 16 bytes, so that the 16-byte
// accesses of eight lanes to eight rows (one shared-memory wavefront) fall on distinct banks.  The history e_1..e_M of a
// row is read from hist[row][0..M) at the start of a launch and written back at its end.
// Mix: the CTA's rows are bus rows, and each f32 tile holds the group sums instead of copies: warps 1-3 build
// tile k+1 (plain loads and stores to shared memory) before its noise, while warp 0 runs the recurrence on tile k, and all
// four warps build tile 0.  group_first is read only then.
constexpr int kShapeT = 64, kShapeRows = 32, kShapeThreads = 128, kShapeStages = 2;

template <int Fmt, int M, bool Mix = false>
__global__ void __launch_bounds__(kShapeThreads) pcm_encode_shaped_kernel(const float* __restrict__ in, size_t in_pitch,
                                                                        unsigned char* __restrict__ out, size_t out_pitch,
                                                                        size_t n_frames, int rows, unsigned long long seed,
                                                                        unsigned long long pos0, DitherTaps taps,
                                                                        float* __restrict__ hist, const int* __restrict__ group_first) {
    using P = PcmTraits<Fmt>;
    constexpr int G = P::kGroup, NB = P::kBytes, W = G * NB / 4;
    constexpr int T = kShapeT, R = kShapeRows, NT = kShapeThreads, IP = T + 4, OP = T * NB + 16, C4 = T / 4, C16 = T * NB / 16;
    static_assert(T % G == 0 && (IP / 4) % 8 == 1 && (OP / 16) % 2 == 1, "whole groups per tile; conflict-free 16-byte rows");
    __shared__ __align__(16) float xs[kShapeStages][R][IP];   // f32 input rows
    __shared__ __align__(16) float ds[2][R][IP];              // noise
    __shared__ __align__(16) unsigned char qs[R][OP];         // packed output rows
    __shared__ unsigned long long keys[R];
    const int tid = threadIdx.x, r0 = blockIdx.x * R, nr = min(R, rows - r0);
    const size_t n_tiles = (n_frames + T - 1) / T;
    if (tid < R) keys[tid] = dither_row_key(seed, (size_t)(r0 + tid));
    auto load = [&](size_t k) {
        if (k < n_tiles) {
            const size_t f0 = k * T;
            const int nv = (int)((min((size_t)T, n_frames - f0) + 3) / 4);   // a row's last float4 is inside its pitch
            for (int i = tid; i < R * C4; i += NT) {
                const int r = i / C4, c = i - r * C4;
                if (r < nr && c < nv) cp_async16(&xs[k % kShapeStages][r][4 * c], in + (size_t)(r0 + r) * in_pitch + f0 + 4 * c);
            }
        }
        cp_async_commit();   // an empty group past the last tile keeps the wait counts uniform
    };
    // Mix: tile k of the bus rows from the stream rows.  A thread owns up to J float4 columns and walks their streams
    // together, so that J independent 16-byte loads are in flight per stream step: one column at a time left the
    // build, not the recurrence, on the critical path.
    auto build = [&](size_t k, int i0, int step) {
        constexpr int J = (R * C4 + (NT - 32) - 1) / (NT - 32);   // columns per thread of warps 1-3 (all warps: fewer)
        const size_t f0 = k * T;
        const int nv = (int)((min((size_t)T, n_frames - f0) + 3) / 4);
        const float* src[J];
        int ns[J], nmax = 0;
        float4 acc[J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const int i = i0 + j * step, r = i / C4, c = i - r * C4;
            src[j] = in; ns[j] = 0; acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < R * C4 && r < nr && c < nv) {
                const int row = r0 + r, s0 = group_first[row >> 1];
                ns[j] = group_first[(row >> 1) + 1] - s0;
                src[j] = in + ((size_t)s0 * 2 + (row & 1)) * in_pitch + f0 + 4 * c;
            }
            nmax = max(nmax, ns[j]);
        }
#pragma unroll 2
        for (int s = 0; s < nmax; ++s) {
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (s < ns[j]) {
                    const float4 v = *reinterpret_cast<const float4*>(src[j] + (size_t)s * 2 * in_pitch);
                    acc[j].x += v.x; acc[j].y += v.y; acc[j].z += v.z; acc[j].w += v.w;
                }
        }
#pragma unroll
        for (int j = 0; j < J; ++j)
            if (ns[j]) {
                const int i = i0 + j * step, r = i / C4, c = i - r * C4;
                *reinterpret_cast<float4*>(&xs[k % kShapeStages][r][4 * c]) = acc[j];
            }
    };
    auto noise = [&](size_t k) {   // warps 1-3: the noise of tile k (every frame of it; those past n_frames go unused)
        const unsigned long long p = pos0 + k * T + 1;
        for (int i = tid - 32; i < R * C4; i += NT - 32) {
            const int r = i / C4, c = i - r * C4;
            unsigned long long z = keys[r] + kDitherPhi * (p + 4 * c);
            float4 d;
            d.x = dither_noise(z); z += kDitherPhi;
            d.y = dither_noise(z); z += kDitherPhi;
            d.z = dither_noise(z); z += kDitherPhi;
            d.w = dither_noise(z);
            *reinterpret_cast<float4*>(&ds[k & 1][r][4 * c]) = d;
        }
    };
    float e[M];
    const bool owner = tid < nr;
#pragma unroll
    for (int k = 0; k < M; ++k) e[k] = owner ? hist[(size_t)(r0 + tid) * kShapeTaps + k] : 0.f;
    if constexpr (Mix) build(0, tid, NT);
    else load(0);
    __syncthreads();   // keys (Mix: and tile 0)
    if (tid >= 32) noise(0);
    for (size_t k = 0; k < n_tiles; ++k) {
        if constexpr (!Mix) {
            load(k + 1);
            cp_async_wait<1>();   // this thread's copies of tile k have landed ...
        }
        __syncthreads();      // ... and everybody's; the noise of tile k is written
        const size_t f0 = k * T;
        const int nf = (int)min((size_t)T, n_frames - f0);
        if (owner) {
            const float4* x = reinterpret_cast<const float4*>(xs[k % kShapeStages][tid]);
            const float4* dn = reinterpret_cast<const float4*>(ds[k & 1][tid]);
            unsigned char* o = qs[tid];
            // a group's samples and noise are read one group ahead, so that the chain does not wait for shared memory
            float xc[G], dc[G];
            auto fetch = [&](int g, float (&xv)[G], float (&dv)[G]) {
#pragma unroll
                for (int v = 0; v < G / 4; ++v) {
                    const float4 a = x[g / 4 + v], b = dn[g / 4 + v];
                    xv[4 * v] = a.x; xv[4 * v + 1] = a.y; xv[4 * v + 2] = a.z; xv[4 * v + 3] = a.w;
                    dv[4 * v] = b.x; dv[4 * v + 1] = b.y; dv[4 * v + 2] = b.z; dv[4 * v + 3] = b.w;
                }
            };
            fetch(0, xc, dc);
#pragma unroll 1
            for (int g = 0; g < nf; g += G) {
                float xn[G], dnx[G];
                fetch(g + G < nf ? g + G : g, xn, dnx);
                int q[G];
                if (g + G <= nf) {
#pragma unroll
                    for (int j = 0; j < G; ++j) q[j] = shaped_step<Fmt, M>(xc[j], dc[j], taps, e);
                } else {   // the call's last, partial group: only its frames step the filter
#pragma unroll
                    for (int j = 0; j < G; ++j) q[j] = g + j < nf ? shaped_step<Fmt, M>(xc[j], dc[j], taps, e) : 0;
                }
#pragma unroll
                for (int j = 0; j < G; ++j) { xc[j] = xn[j]; dc[j] = dnx[j]; }
                unsigned w[W];
                pcm_pack<Fmt>(q, w);
#pragma unroll
                for (int v = 0; v < W / 4; ++v)
                    *reinterpret_cast<uint4*>(o + g * NB + 16 * v) = make_uint4(w[4 * v], w[4 * v + 1], w[4 * v + 2], w[4 * v + 3]);
            }
        } else if (tid >= 32 && k + 1 < n_tiles) {
            if constexpr (Mix) build(k + 1, tid - 32, NT - 32);
            noise(k + 1);
        }
        __syncthreads();   // the byte tile is complete
        const int nb = nf * NB;
        for (int i = tid; i < R * C16; i += NT) {
            const int r = i / C16, c = i - r * C16;
            if (r >= nr || 16 * c >= nb) continue;
            unsigned char* dst = out + (size_t)(r0 + r) * out_pitch + f0 * NB + 16 * c;
            const unsigned char* src = &qs[r][16 * c];
            if (16 * c + 16 <= nb) *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
            else for (int b = 0; b < nb - 16 * c; ++b) dst[b] = src[b];   // nothing past n_frames is touched
        }
        __syncthreads();   // the byte tile and this tile's input stage are free again
    }
    if (owner) {
#pragma unroll
        for (int k = 0; k < M; ++k) hist[(size_t)(r0 + tid) * kShapeTaps + k] = e[k];
    }
}

}  // namespace ohs
