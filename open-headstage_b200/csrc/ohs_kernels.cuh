// ohs_kernels.cuh — hand-written sm_100a kernels of the Open Headstage DSP hot path.
//
// One fused kernel renders, for a group of G stereo streams per CTA and K engine blocks per launch,
//     10-band DF2T biquad cascade (bit-exact)  ->  uniformly partitioned overlap-save FFT convolution against the four
//     HRIR paths  ->  ear sums  ->  output gain
// i.e. the work of reference src/lib.rs:1179-1207 (Plugin::process) over src/dsp/parametric_eq.rs:166-179 and
// src/dsp/convolution.rs:184-289, for many streams at once.
//
// Design (DESIGN.md §4 has the derivations, the measured pipe numbers and the ncu evidence behind each choice):
//   * staging warp: issues the TMA bulk copies of the input rows HBM -> shared memory (one per row, completing on an
//     mbarrier) into a ring of three stage buffers, three blocks ahead.
//   * EQ warps: band-systolic in time.  Lane l*6 + c owns bands 2l and 2l+1 of chain c = (stream, channel); at step s
//     band A filters sample s-4l with the input shuffled over from lane l-1 three steps earlier, band B filters sample
//     s-4l-1 with band A's previous output.  Every band's recurrence stays strictly sequential in the reference's
//     operation order with explicitly rounded, never-contracted ops: bit-exact.  Where several CTAs share an SM the two
//     bands of a lane run as one packed f32x2 chain (RenderSmem::kEqPacked).  The chain runs continuously across the
//     blocks of a launch.
//   * convolution warps, T = max(32, N/16) threads per stream (one warp at N = 512): left + i*right go through ONE
//     complex N = 2B point Stockham FFT in shared memory (radix 8/4/2 in registers, two adjacent butterflies per thread
//     so every shared-memory access is 128-bit), the frequency-domain delay line keeps that packed spectrum Z, and the
//     four HRIR paths are applied as
//         W[k] = sum_p  Z_{t-p}[k] * A_p[k] + conj(Z_{t-p}[N-k]) * C_p[k]
//     with A = (G_L - i G_R)/2N, C = (G_L + i G_R)/2N, G_L = FFT(h_LSL + i h_LSR), G_R = FFT(h_RSL + i h_RSR):
//     Re IFFT(W) is the left ear (LSL + RSL), Im IFFT(W) the right ear (LSR + RSR) (src/dsp/convolution.rs:229-230).
//     One forward and one inverse FFT per block instead of the reference's four and four.  The products with the
//     delay line's OLDER spectra (partitions 1..P-1) are accumulated before the wait for the block's EQ output.  With a
//     single partition at N = 512 the last forward pass, the product and the first inverse pass run in registers.
//   * the roles are decoupled by named barriers and mbarriers over a 3-slot ring of filtered blocks and the stage ring,
//     so the staging of block t+3, the EQ of block t+1 and the convolution of block t overlap, and are placed on the
//     four scheduler partitions so that their loads balance.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

namespace ohs {

constexpr int kMaxBands = 10;
// EQ warps run two bands per lane (five lanes per chain, six chains per warp) or one (ten lanes, three chains):
// RenderSmem::kEqBpl.  For config 2's seven streams per CTA two bands per lane is the one that fits: with one band per
// lane (five EQ warps) two EQ warps share a scheduler partition and the block time is the same (844 k vs 852 k
// stream-s/s) for more issue slots.
// Placement weight of an EQ warp in units of a convolution warp (RenderSmem::place).  Round 2 re-measurement on config 2
// (profiles/r02_ab_placement.txt): weight 3 -> (1, 1, 1, 4) convolution warps next to the three EQ warps, 16 warp
// slots, 128 registers per thread: 1.081 M stream-s/s; weight 4 -> (0, 1, 1, 5), 20 warp slots, 96 registers, 360
// bytes of spills in the convolution warps: 1.003 M; weight 5: 0.920 M.  (ptxas 12.9 reports 128 registers and 224 B
// of spill stores and loads for today's render_kernel<512, 7, 0>.)  Weight 1 -> (1, 1, 2, 3), 12 warp slots, 168
// registers: 0.977 M, and 0.884 M with the packed EQ step (profiles/eq_packed_f32x2_ab.txt); weight 2 places config 2
// like weight 3.
#ifndef OHS_EQ_WEIGHT
#define OHS_EQ_WEIGHT 3
#endif
constexpr int kMaxG = 7;       // streams per CTA
constexpr int kEqSkew = 4;     // steps between neighbouring lanes of the systolic chain: a shuffled value is consumed 3 steps
                               // (~90 cycles) after it was sent.  8 was better while the FFT warps were heavier; on the final
                               // kernel 4 wins (948 k vs 908 k stream-s/s: fewer live registers, shorter fill and drain)
constexpr int kEqCoefStride = 8;  // floats per (eq_set, band): b0 b1 b2 a1 a2 enabled pad pad

// kBarStream0 + g (g < 7) synchronises the threads of one stream's transform when they span several warps;
// kBarInitConv / kBarInitEq: the staging warp has initialised the mbarriers (it arrives, the other role waits)
enum NamedBarrier { kBarFull0 = 1, kBarFull1 = 2, kBarEmpty0 = 3, kBarEmpty1 = 4, kBarEq = 5, kBarConv = 6, kBarStream0 = 7,
                    kBarInitConv = 14, kBarInitEq = 15 };

struct RenderParams {
    const float* in;            // [stream][2][row_stride]
    float* out;
    long long row_stride;       // frames between the input rows
    long long out_row_stride;   // frames between the output rows (= row_stride except in the EQ pre-pass of the time-batched route)
    int n_blocks;               // K engine blocks this launch
    int tail_frames;            // frames in the last block: B, or fewer in EQ-only mode (conv_enable == 0)
    int n_streams;
    const int* stream_hrir;     // [stream] -> hrir set
    const int* stream_eq;       // [stream] -> eq set
    const float* stream_gain;   // [stream]
    const float4* filt;         // [set][pmax][even bins | odd bins] {A.re, A.im, C.re, C.im}, 1/N folded in
    const int* set_parts;       // [set] partitions in use
    float2* fdl;                // [stream][pmax][N] packed spectra ring (unused when every set has 1 partition)
    float2* prev;               // [stream][2][B] f32 planar (left row, right row): last filtered input block (overlap-save history)
    const float* eqc;           // [eq_set][kMaxBands][kEqCoefStride]
    float4* eqs;                // [stream][kMaxBands] {s1L, s1R, s2L, s2R}
    const float2* tw;           // [N] exp(-2*pi*i*m/N)
    int pmax;
    int head;                   // ring slot of this launch's first block
    int n_bands;
    int eq_enable;
    int conv_enable;
    int filt_in_smem;           // 0, or the partition count of the single shared HRIR set staged in shared memory
    int uniform_set;            // 1 when every stream is bound to HRIR set 0 (enables the TMA filter-tile pipeline)
    int first_stream;           // CTA 0 renders streams first_stream .. first_stream+G-1 (set by the launcher)
    int io_first_stream;        // the stream whose rows sit at in/out row 0 (host staging by stream range), else 0
    unsigned long long* trace;  // OHS_TRACE builds: [CTA][16] clock64 stamps of the launch's milestones, else unused
    // moving sources (render_kernel<..., true> only; DESIGN §10): the set of block t is block_set[s*block_set_stride + t],
    // or stream_hrir[s] for every block when block_set is null; from_set[s] is the set of the block before block 0
    const int* from_set;
    const int* block_set;
    long long block_set_stride;
    // operands of the EQ warps' packed biquad step (df2t_step2): kernel parameters, so that ptxas cannot fold them into
    // a contraction of the separately rounded products and sums
    float one = 1.f;
    float neg_zero = -0.f;
};

#ifdef OHS_TRACE
#define OHS_STAMP(p, slot) do { if ((p).trace) (p).trace[(size_t)blockIdx.x * 16 + (slot)] = (unsigned long long)clock64(); } while (0)
#else
#define OHS_STAMP(p, slot) do { } while (0)
#endif
#define OHS_STAMP_IF(cond, p, slot) do { if (cond) OHS_STAMP(p, slot); } while (0)

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
// complex product with the contraction pinned (one rounded product, one FMA per component): every instantiation of
// the transforms — throughput and latency variant, fused and general single-partition path — rounds identically, so
// a stream's output does not depend on how many blocks a call renders
__device__ __forceinline__ float2 cmul(float2 a, float2 w) {
    return make_float2(fmaf(a.x, w.x, -__fmul_rn(a.y, w.y)), fmaf(a.x, w.y, __fmul_rn(a.y, w.x)));
}
__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }  // a * (-i)

// shared-memory index padding of the complex ping-pong buffers: 16 bytes after every 16 float2.  Adjacent pairs stay
// contiguous and 16-byte aligned (128-bit accesses), and the strided stores of the radix passes (lane stride 16 float2
// in the first pass, 64-float2 runs in the second) land on distinct banks.
__host__ __device__ constexpr int padi(int j) { return j + 2 * (j >> 4); }
__host__ __device__ constexpr int padded_len(int n) { return n + 2 * (n >> 4); }

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// Programmatic dependent launch (sm_90+): launch_dependents lets the next launch on the stream start its CTAs (as SM
// resources free up) and run its state-independent prologue while this grid is still running; grid_dependency_wait
// blocks until every earlier grid on the stream has completed and its writes are visible.  Both are no-ops for a
// launch without the programmatic-serialization attribute.
__device__ __forceinline__ void launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// AND-reduce a predicate over the first NT threads of the CTA (the EQ warps) on their named barrier
template <int NT> __device__ __forceinline__ bool __syncthreads_and_eq(bool pred) {
    unsigned r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.and.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
                 : "=r"(r) : "r"((unsigned)pred), "r"((int)kBarEq), "r"(NT) : "memory");
    return r != 0;
}

// ---- TMA (bulk asynchronous copy) + mbarrier: input rows HBM -> shared memory, issued by ONE thread per block of rows
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, unsigned parity) {
    unsigned done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}

// ---------------------------------------------------------------------------------------------------------------
// register DFTs (forward, e^{-2 pi i rq/R}), natural order in and out.  Scalar FP32: a packed f32x2 version of the FFT
// arithmetic (FADD2 complex adds, FMUL2+FFMA2 twiddle products) was measured and is slower here (conv-only 11.1 k vs
// 8.8 k cycles per block): the packed ops hold the FP32 pipe two cycles, so only issue slots are saved, and those are
// not what the convolution warps' partition runs out of.
// ---------------------------------------------------------------------------------------------------------------
template <int R> struct Dft;
template <> struct Dft<2> {
    static __device__ __forceinline__ void run(float2 (&u)[2]) {
        const float2 t = u[0];
        u[0] = cadd(t, u[1]);
        u[1] = csub(t, u[1]);
    }
};
template <> struct Dft<4> {
    static __device__ __forceinline__ void run(float2 (&u)[4]) {
        const float2 a0 = cadd(u[0], u[2]), a1 = csub(u[0], u[2]);
        const float2 a2 = cadd(u[1], u[3]), a3 = mul_mi(csub(u[1], u[3]));
        u[0] = cadd(a0, a2); u[2] = csub(a0, a2);
        u[1] = cadd(a1, a3); u[3] = csub(a1, a3);
    }
};
template <> struct Dft<8> {
    static __device__ __forceinline__ void run(float2 (&u)[8]) {
        constexpr float c = 0.70710678118654752440f;
        float2 a[4], b[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { a[r] = cadd(u[r], u[r + 4]); b[r] = csub(u[r], u[r + 4]); }
        // b[r] *= w8^r
        b[1] = make_float2(c * (b[1].x + b[1].y), c * (b[1].y - b[1].x));
        b[2] = mul_mi(b[2]);
        b[3] = make_float2(c * (b[3].y - b[3].x), -c * (b[3].x + b[3].y));
        Dft<4>::run(a);
        Dft<4>::run(b);
#pragma unroll
        for (int q = 0; q < 4; ++q) { u[2 * q] = a[q]; u[2 * q + 1] = b[q]; }
    }
};

// ---------------------------------------------------------------------------------------------------------------
// Stockham auto-sort FFT of N complex points by T threads (each thread owns E = N/T points per pass).
// Pass with radix R after radices of product P:  butterfly i -> k = i mod P, j = (i-k)*R + k,
//   u[r] = x[i + r*N/R] * w^{k r / (P R)},  y[j + q*P] = DFT_R(u)[q].   Output in natural order.
// A thread owns ADJACENT butterflies i = tid*PER + b; with an even PER it works on pairs (i, i+1), so every shared
// memory access moves two float2 in one 128-bit instruction (half the LSU instructions of the 64-bit form) and the
// two butterflies give the in-order warp two independent dependency chains.
// ---------------------------------------------------------------------------------------------------------------
constexpr int fft_threads(int n) { return (n / 16 >= 32) ? n / 16 : 32; }

template <int N, int T> struct FftPlan {
    static constexpr int E = N / T;                 // points per thread: 16 (N >= 512), 8 (N = 256), 4 (N = 128)
    static_assert(E == 16 || E == 8 || E == 4, "points per thread");
    static constexpr int RM = E < 8 ? E : 8;       // largest radix
    static constexpr int R1 = RM, P1 = 1;
    static constexpr int P2 = R1, R2 = (N / P2 >= RM) ? RM : N / P2;
    static constexpr int P3 = P2 * R2, R3 = (P3 < N) ? ((N / P3 >= RM) ? RM : N / P3) : 1;
    static constexpr int P4 = P3 * R3, R4 = (P4 < N) ? ((N / P4 >= RM) ? RM : N / P4) : 1;
    static_assert(P4 * R4 == N, "at most four passes");
    static constexpr int kPasses = 2 + (R3 > 1) + (R4 > 1);
    // per-pass twiddle tables, laid out [r-1][k] so that lanes with consecutive k read consecutive float2 (no bank
    // conflicts; a single table indexed k*r*N/(P*R) puts 8 lanes on one bank): pass with radix R after product P
    // uses entries w^{k r / (P R)}, k < P, r = 1..R-1
    static constexpr int kTw2 = 0;
    static constexpr int kTw3 = kTw2 + (R2 - 1) * P2;
    static constexpr int kTw4 = kTw3 + (R3 > 1 ? (R3 - 1) * P3 : 0);
    static constexpr int kTwLen = kTw4 + (R4 > 1 ? (R4 - 1) * P4 : 0);
    static_assert(kTwLen <= N, "twiddle tables fit in N entries");
    static constexpr bool kOutInB0 = (kPasses % 2) == 1;  // which ping-pong buffer a full transform ends in
};

// padded complex buffer in shared memory; the *2 forms move the adjacent pair (i, i+1), i even, as one float4
struct SmemCx {
    float2* p;
    __device__ __forceinline__ float2 ld(int i) const { return p[padi(i)]; }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const {
        const float4 v = *reinterpret_cast<const float4*>(p + padi(i));
        a = make_float2(v.x, v.y); b = make_float2(v.z, v.w);
    }
    __device__ __forceinline__ void st(int i, float2 v) const { p[padi(i)] = v; }
    __device__ __forceinline__ void st2(int i, float2 a, float2 b) const {
        *reinterpret_cast<float4*>(p + padi(i)) = make_float4(a.x, a.y, b.x, b.y);
    }
};

// the loads of SmemCx over an unpadded spectrum in global memory (a delay-line slot)
struct GlobalCx {
    const float2* p;
    __device__ __forceinline__ float2 ld(int i) const { return p[i]; }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const {
        const float4 v = *reinterpret_cast<const float4*>(p + i);
        a = make_float2(v.x, v.y); b = make_float2(v.z, v.w);
    }
};

template <int N, int T, int R, int P, class Load, class Store>
__device__ __forceinline__ void fft_pass(int tid, const float2* __restrict__ tw, const Load& load, const Store& store) {
    constexpr int NB = N / R;   // butterflies in this pass
    constexpr int PER = NB / T; // per thread
    static_assert(PER >= 1, "radix larger than points per thread");
    if constexpr (PER % 2 == 0) {
#pragma unroll
        for (int b = 0; b < PER; b += 2) {
            const int i = tid * PER + b;  // even: butterflies i and i+1
            float2 u[R], v[R];
#pragma unroll
            for (int r = 0; r < R; ++r) load.ld2(i + r * NB, u[r], v[r]);
            if constexpr (P > 1) {
                const int k = i & (P - 1);  // even, and k+1 < P
#pragma unroll
                for (int r = 1; r < R; ++r) {
                    const float4 w = *reinterpret_cast<const float4*>(tw + (r - 1) * P + k);
                    u[r] = cmul(u[r], make_float2(w.x, w.y));
                    v[r] = cmul(v[r], make_float2(w.z, w.w));
                }
                Dft<R>::run(u);
                Dft<R>::run(v);
                const int j = (i - k) * R + k;
#pragma unroll
                for (int q = 0; q < R; ++q) store.st2(j + q * P, u[q], v[q]);
            } else {
                Dft<R>::run(u);
                Dft<R>::run(v);
                // first pass: each butterfly writes R consecutive outputs
#pragma unroll
                for (int q = 0; q < R; q += 2) {
                    store.st2(i * R + q, u[q], u[q + 1]);
                    store.st2((i + 1) * R + q, v[q], v[q + 1]);
                }
            }
        }
    } else {
#pragma unroll
        for (int b = 0; b < PER; ++b) {
            const int i = tid * PER + b;
            const int k = i & (P - 1);
            const int j = (i - k) * R + k;
            float2 u[R];
#pragma unroll
            for (int r = 0; r < R; ++r) u[r] = load.ld(i + r * NB);
            if constexpr (P > 1) {
#pragma unroll
                for (int r = 1; r < R; ++r) u[r] = cmul(u[r], tw[(r - 1) * P + k]);
            }
            Dft<R>::run(u);
#pragma unroll
            for (int q = 0; q < R; ++q) store.st(j + q * P, u[q]);
        }
    }
}

// Full transform.  load0 feeds the first pass, store_last receives the natural-order result, b0/b1 are the ping-pong
// buffers (padded), `sync` separates passes, `after_first` runs once the first pass has consumed its input.
template <int N, int T, class Load0, class StoreLast, class Sync, class AfterFirst>
__device__ __forceinline__ void fft_run(int tid, const float2* __restrict__ tw, float2* b0p, float2* b1p, const Load0& load0,
                                        const StoreLast& store_last, Sync sync, AfterFirst after_first) {
    using Pl = FftPlan<N, T>;
    const SmemCx b0{b0p}, b1{b1p};
    fft_pass<N, T, Pl::R1, Pl::P1>(tid, tw, load0, b0);
    after_first();
    sync();
    if constexpr (Pl::kPasses == 2) {
        fft_pass<N, T, Pl::R2, Pl::P2>(tid, tw + Pl::kTw2, b0, store_last);
    } else {
        fft_pass<N, T, Pl::R2, Pl::P2>(tid, tw + Pl::kTw2, b0, b1);
        sync();
        if constexpr (Pl::kPasses == 3) {
            fft_pass<N, T, Pl::R3, Pl::P3>(tid, tw + Pl::kTw3, b1, store_last);
        } else {
            fft_pass<N, T, Pl::R3, Pl::P3>(tid, tw + Pl::kTw3, b1, b0);
            sync();
            fft_pass<N, T, Pl::R4, Pl::P4>(tid, tw + Pl::kTw4, b0, store_last);
        }
    }
}

// host side: the per-pass tables for FftPlan<N, T>, f64-computed and rounded once (as rustfft's twiddles are)
template <int N> inline void fill_twiddles(float2* out) {
    constexpr int T = fft_threads(N);
    using Pl = FftPlan<N, T>;
    const int R[3] = {Pl::R2, Pl::R3, Pl::R4}, P[3] = {Pl::P2, Pl::P3, Pl::P4}, off[3] = {Pl::kTw2, Pl::kTw3, Pl::kTw4};
    for (int i = 0; i < N; ++i) out[i] = make_float2(1.f, 0.f);
    for (int q = 0; q < 3; ++q) {
        if (R[q] <= 1) continue;
        for (int r = 1; r < R[q]; ++r)
            for (int k = 0; k < P[q]; ++k) {
                const double a = -2.0 * 3.14159265358979323846 * (double)k * (double)r / ((double)P[q] * (double)R[q]);
                out[off[q] + (r - 1) * P[q] + k] = make_float2((float)cos(a), (float)sin(a));
            }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// shared-memory carve-up of the render kernel
// ---------------------------------------------------------------------------------------------------------------
// V = 0: the throughput variant (launches of many blocks: EQ of block t+1 overlaps the convolution of block t, so the
// roles are sized for issue-slot balance).  V = 1, N = 512: the latency variant for launches of one or two blocks (the
// reference's calling pattern, one call per host buffer), where nothing overlaps and a block's time is the EQ chain's
// latency plus the transform's: twice the threads per stream in the transforms (6.0 k instead of 9.7 k cycles for a
// lone block of config 2).  One band per lane in its EQ warps was measured too and is not faster there: five EQ
// warps put two on one scheduler partition (36 cycles per step against 34).
template <int N, int G, int V = 0> struct RenderSmem {
    // V = 2, N = 512: the EQ-only variant behind the time-batched route's EQ pre-pass (ohs_api.cu): the same staging and
    // EQ warps with one band per lane, "convolution" warps that only copy the filtered rows out, no transform buffers,
    // twiddles or filter table.  It runs beside the route's throughput-bound kernels of the previous chunk instead of in
    // front of them — but not on the same SMs: next to the per-bin kernel's FMA-saturated warps every instruction of the
    // biquad chain waits for its issue slot and the chain runs 2.5x slower (measured), which makes it the critical path
    // again.  So the production shape is G = 6 (four EQ warps, one per scheduler partition; two per partition run 1.6x
    // slower per step) with 200 KB of shared memory asked for at launch, so that each CTA OWNS its SM: 43 CTAs for
    // config 5's 256 streams.  G = 3 (38 KB, six warps) serves few streams and the un-overlapped route.
    static_assert(V == 0 || ((V == 1 || V == 2) && N == 512), "the latency and EQ-only variants exist for N = 512");
    static constexpr bool kEqOnly = (V == 2);
    static constexpr int B = N / 2;
    // convolution threads per stream (V = 0: one warp at N <= 512).  The latency variant doubles them where that keeps
    // the radix plan (N = 512: 8 points per thread, radices 8-8-8 either way), so both variants round identically.
    static constexpr int T = (V == 1 && N == 512) ? 2 * fft_threads(N) : fft_threads(N);
    static constexpr int NP = padded_len(N);
    // Bands per lane of the EQ warps.  2: five lanes per chain, six chains per warp (config 2: the issue slots of three
    // warps are what the CTA can spare).  1: ten lanes per chain, three chains per warp, half the instructions and a
    // single 12-cycle dependent chain per step — for the long blocks of N >= 1024, where a CTA holds few streams and
    // the 1024-step sequential chain per block is the floor of the launch (config 5).
#ifdef OHS_BPL1_ALL   // A/B experiments only: one band per lane for every transform size
    static constexpr int kEqBpl = 1;
#else
    static constexpr int kEqBpl = (N >= 1024 || V == 2) ? 1 : 2;
#endif
    // Two bands per lane as one packed f32x2 chain (df2t_step2) where several CTAs share an SM (N <= 256: config 3),
    // whose warps compete for issue slots: config 3 870 k against 823 k stream-s/s with the scalar pair of chains.
    // Where one CTA owns the SM (N = 512) the scalar form is faster: its two independent chains per lane hide each
    // other's latency (config 2 1.084 M against 0.988 M packed, K = 1 496 k against 480 k; DESIGN §4.5).
    static constexpr bool kEqPacked = kEqBpl == 2 && N < 512;
    // lane skew of the systolic chain in steps (= steps per unrolled iteration).  One band per lane runs a step in half
    // the time, too fast for a 3-step shuffle flight: skew 8
    static constexpr int kEqSkewSteps = (B >= 128) ? (kEqBpl == 1 ? 8 : kEqSkew) : 4;
    static constexpr int kEqCpw = 32 / (kMaxBands / kEqBpl);   // chains per EQ warp: 6 or 3
    static constexpr int kEqWarps = (2 * G + kEqCpw - 1) / kEqCpw;
    static constexpr int kEqThreads = 32 * kEqWarps;
    static constexpr int kConvWarps = G * T / 32;
    // Single-partition responses (config 2) at N = 512: the forward transform's last pass, the spectral product and the
    // inverse transform's first pass run fused in registers (conv_warps_main).  Needs one warp per stream, equal first
    // and last radices and two butterflies of the last pass per thread.
    static constexpr bool kFusedMac = !kEqOnly && (T == 32) && (FftPlan<N, T>::kPasses == 3) && (FftPlan<N, T>::R1 == FftPlan<N, T>::R3) &&
                                      (N / FftPlan<N, T>::R3 == 2 * T);
    static constexpr int kWorkers = kEqThreads + G * T;       // threads that take part in the EMPTY barriers
    static constexpr int kFullCount = kWorkers + 32;          // ... and in the FULL barriers: the staging warp listens in
    // Warp placement.  A warp's scheduler partition is (warp id mod 4) and an EQ warp carries three to four times the
    // instructions of a convolution warp, so the roles are spread to equalise the partitions' load: EQ warp w sits on
    // partition w (warp id w); each convolution warp goes to the least-loaded partition; unused warp slots exit at
    // once.  (Config 2, G = 7: partitions 0-2 hold one EQ + one convolution warp, partition 3 four convolution warps.)
    struct Placement {
        int conv_warp_id[kConvWarps > 0 ? kConvWarps : 1];
        int stager_warp_id;   // the warp that issues the input rows' TMA copies (a few instructions per block)
        int total_warps;
    };
    // Balancing pads the CTA with idle warp slots, which only pays when one CTA owns the SM (N >= 512: config 2 and the
    // long-BRIR config); smaller transforms run several CTAs per SM, which balances the partitions by itself, and
    // there the roles are packed densely.
    static constexpr bool kBalanced = (N >= 512) && V == 0;
    static constexpr int kEqWeight = OHS_EQ_WEIGHT;   // an EQ warp's load in units of a convolution warp's
    static constexpr Placement place() {
        Placement pl{};
        if (!kBalanced) {
            for (int f = 0; f < kConvWarps; ++f) pl.conv_warp_id[f] = kEqWarps + f;
            pl.stager_warp_id = kEqWarps + kConvWarps;
            pl.total_warps = kEqWarps + kConvWarps + 1;
            return pl;
        }
        int load[4] = {0, 0, 0, 0}, count[4] = {0, 0, 0, 0};
        for (int w = 0; w < kEqWarps; ++w) { load[w & 3] += kEqWeight / (kEqBpl == 1 ? 2 : 1); count[w & 3] += 1; }
        for (int f = 0; f < kConvWarps; ++f) {
            int best = 3;
            for (int q = 3; q >= 0; --q) if (load[q] < load[best]) best = q;
            pl.conv_warp_id[f] = 4 * count[best] + best;
            load[best] += 1; count[best] += 1;
        }
        int few = 0;
        for (int q = 1; q < 4; ++q) if (count[q] < count[few]) few = q;
        pl.stager_warp_id = 4 * count[few] + few;
        count[few] += 1;
        int mx = 0;
        for (int q = 0; q < 4; ++q) if (count[q] > mx) mx = count[q];
        pl.total_warps = 4 * mx;
        return pl;
    }
    static constexpr int kThreads = 32 * place().total_warps;
    template <int F> static constexpr int kConvWarpId = place().conv_warp_id[F];
    static constexpr int kStagerWarpId = place().stager_warp_id;
    static constexpr size_t kTwOff = 0;                                      // float2 tw[N]
    static constexpr size_t kZOff = kTwOff + (kEqOnly ? 0 : sizeof(float2) * N);   // float2 z[G][2][NP]
    // per-stream strides carry a 16-byte pad so that neighbouring streams sit on different banks
    // planar ring[G][3 slots][left row | pad | right row | pad]: streams 16 bytes apart in bank space, a stream's two
    // rows 64 bytes apart, so the six rows an EQ warp stores to in one instruction sit on different banks
    static constexpr int kRingRowR = B + 16;                 // offset of the right row behind the left row
    static constexpr int kRingSlot = 2 * B + 32;             // floats per slot (a multiple of 32: slots share banks)
    static constexpr int kRingStride = 3 * kRingSlot + 4;    // floats per stream
    // stage[3 buffers][G][left row | pad | right row | pad]: the 16-byte pads put the six rows an EQ warp reads (three
    // streams x two channels) on different banks
    static constexpr int kStageBufs = 3;
    static constexpr int kRowR = B + 4;              // offset of the right row behind the left row
    static constexpr int kStageStride = 2 * B + 8;   // float per stream and stage buffer
    static constexpr size_t kRingOff = kZOff + (kEqOnly ? 0 : sizeof(float2) * G * 2 * NP);
    static constexpr size_t kStageOff = kRingOff + sizeof(float) * G * kRingStride;
    // filter spectra of a shared single-set, few-partition HRIR (configs 1-3) are staged here once per launch
    static constexpr size_t kFiltSmemBytes = (N <= 512 && !kEqOnly) ? 16 * 1024 : 0;
    static constexpr size_t kFiltOff = kStageOff + sizeof(float) * kStageBufs * G * kStageStride;
    static constexpr size_t kMbarOff = kFiltOff + kFiltSmemBytes;  // uint64_t stage_full[3], filt_full[2], prologue_full
    static constexpr size_t kBytes = kMbarOff + 48;
    static constexpr bool kFits = kBytes <= 227 * 1024 && kThreads <= 1024;
    // Register budget.  Warps are allocated in groups of four; as many CTAs per SM as shared memory allows (up to
    // four) while every thread keeps at least 80 registers.
    static constexpr int kWarpsAlloc = (kThreads / 32 + 3) / 4 * 4;
    static constexpr int kBySmem = kEqOnly ? 1 : (int)((227 * 1024) / (kBytes + 1024));
    static constexpr int kByRegs = 65536 / (80 * 32 * kWarpsAlloc);
    static constexpr int kMinBlocks0 = kBySmem < kByRegs ? kBySmem : kByRegs;
    static constexpr int kMinBlocks = kMinBlocks0 < 1 ? 1 : (kMinBlocks0 > 4 ? 4 : kMinBlocks0);
    static constexpr int kMaxRegs0 = (65536 / (kMinBlocks * 32 * kWarpsAlloc)) / 8 * 8;
#ifdef OHS_REG_CAP   // A/B experiments only (tools/ab_build.py): a lower register cap changes ptxas's schedule of the EQ loop
    static constexpr int kMaxRegs1 = kMaxRegs0 > OHS_REG_CAP ? OHS_REG_CAP : kMaxRegs0;
#else
    static constexpr int kMaxRegs1 = kMaxRegs0;
#endif
    static constexpr int kMaxRegs = kMaxRegs1 > 168 ? 168 : (kMaxRegs1 < 32 ? 32 : kMaxRegs1);
};

// ---------------------------------------------------------------------------------------------------------------
// EQ warp
// ---------------------------------------------------------------------------------------------------------------
// One DF2T step, reference operation order (biquad 0.4.2 DirectForm2Transposed::run behind
// src/dsp/parametric_eq.rs:116-122):   out = s1 + b0*x;  s1 = (s2 + b1*x) - a1*out;  s2 = b2*x - a2*out
// Explicit round-to-nearest intrinsics: every product and sum is rounded separately and is never contracted into an
// FMA (Rust does not contract; the cascade's output moves by 3.8e-4 if it is).  With two bands per lane, bands A and
// B are two independent scalar chains in the same lane, which gives the in-order warp the instruction-level
// parallelism to cover the 4-cycle FP32 latency, or one packed chain (df2t_step2, RenderSmem::kEqPacked).
__device__ __forceinline__ float df2t_step(float x, float& s1, float& s2, float b0, float b1, float b2, float a1, float a2) {
    const float out = __fadd_rn(s1, __fmul_rn(b0, x));
    s1 = __fsub_rn(__fadd_rn(s2, __fmul_rn(b1, x)), __fmul_rn(a1, out));
    s2 = __fsub_rn(__fmul_rn(b2, x), __fmul_rn(a2, out));
    return out;
}
// the same step with the rounded input products b0*x, b1*x, b2*x given
__device__ __forceinline__ float df2t_step_products(float p0, float p1, float p2, float& s1, float& s2, float a1, float a2) {
    const float out = __fadd_rn(s1, p0);
    s1 = __fsub_rn(__fadd_rn(s2, p1), __fmul_rn(a1, out));
    s2 = __fsub_rn(p2, __fmul_rn(a2, out));
    return out;
}

// Packed f32x2 pairs {band A, band B} (low word = A), one FFMA2 per op pair.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { f32x2 d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi)); return d; }
__device__ __forceinline__ void unpk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
// df2t_step on two bands at once, in the same operation order and with the same rounding: every product is
// fma(b, x, -0) (= the rounded product, signed zeros included) and every sum fma(a, 1, c), with 1 and -0 run-time
// values (RenderParams::one, ::neg_zero).  ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 even under
// -fmad=false, and would do the same to these if it saw the constants.  The subtractions add the product with the
// negated a1, a2 (na1, na2): -(a1*out) rounds to exactly the negated rounded product.  Half the FP32 instructions of
// two scalar steps for the same FP32-pipe time, but one dependent chain where the scalar form has two.
__device__ __forceinline__ f32x2 df2t_step2(f32x2 x, f32x2& s1, f32x2& s2, f32x2 b0, f32x2 b1, f32x2 b2, f32x2 na1, f32x2 na2,
                                            f32x2 one, f32x2 nz) {
    const f32x2 out = fma2(fma2(b0, x, nz), one, s1);
    s1 = fma2(fma2(fma2(b1, x, nz), one, s2), one, fma2(na1, out, nz));
    s2 = fma2(fma2(b2, x, nz), one, fma2(na2, out, nz));
    return out;
}

// EQ warp `w` of the CTA.  Lane l*6 + c: chain 6w + c is one (stream, channel) pair; the lane runs bands A = 2l and
// B = 2l+1 of the 10-band cascade.  The chain is systolic in time:
//     step s:  band A filters sample s - 4l      (input: lane l-1's band-B output of step s-3, by SHFL; l = 0: the input row)
//              band B filters sample s - 4l - 1  (input: this lane's band-A output of step s-1)
// so the last band (l = 4, B) runs 17 samples behind the first.  A shuffled output is consumed three steps later, which
// covers its latency (26 cycles alone, more while the convolution warps load the shared-memory pipe).  The two bands
// of a lane are two independent dependent-chains that cover each other's 4-cycle FP32 latency, or, where
// RenderSmem::kEqPacked, one packed {A, B} chain (df2t_step2) whose band B takes the low word of the previous step's
// output pair.  Every band's recurrence is the strictly sequential reference recurrence (see df2t_step): bit-exact.
template <bool V> struct Flag { static constexpr bool value = V; };
template <int N, int G, int V>
__device__ __forceinline__ void eq_warp_main(const RenderParams& p, unsigned char* smem, int stream0, int w) {
    using SM = RenderSmem<N, G, V>;
    constexpr int B = SM::B;
    constexpr int BPL = SM::kEqBpl;                    // bands per lane
    constexpr bool kPacked = SM::kEqPacked;            // the two bands as one f32x2 chain (df2t_step2)
    constexpr int LPC = kMaxBands / BPL;               // lanes per chain
    constexpr int CPW = SM::kEqCpw;                    // chains per warp
    // lane skew in steps = steps per unrolled iteration.  One band per lane runs a step in half the time, too fast for
    // a 3-step shuffle flight: skew 8.
    constexpr int DL = SM::kEqSkewSteps;
    constexpr int NQ = DL / 4;                         // float4 input loads per iteration
    constexpr int LL = DL - 1 + (BPL - 1);             // steps a lane runs behind its left neighbour: a shuffled value is used
                                                       // DL-1 steps after it was sent, band B one step after band A
    constexpr int kOutLag = LL * (LPC - 1) + (BPL - 1);  // steps the last band runs behind the first
    constexpr int kStoreU = (kOutLag + 3) % 4;         // the last lane completes an aligned group of 4 samples when u % 4 == kStoreU
    constexpr int kLagA = (kOutLag + DL - 1) / DL * DL;  // steps of a block during which the previous block is still being finished
    constexpr int kPending = 3 - kStoreU;              // outputs computed after the last group store of an iteration
    static_assert((DL == 4 || DL == 8) && (BPL == 1 || BPL == 2) && B % DL == 0 && B >= kLagA, "systolic loop layout");
    constexpr int kCount = SM::kWorkers;
    float* ring_f = reinterpret_cast<float*>(smem + SM::kRingOff);
    float* stage = reinterpret_cast<float*>(smem + SM::kStageOff);

    const int lane = threadIdx.x & 31;
    // band-major lanes: lane = l * 6 + chain.  The six first lanes (input loads) and the six last lanes (output stores)
    // each fall into one quarter-warp, so a 128-bit shared-memory access of theirs is a single wavefront.
    const int c_raw = CPW * w + lane % CPW;  // chain index in the CTA: 2*stream + channel
    const int l = lane / CPW;
    const bool chain_ok = (lane < CPW * LPC) && (c_raw < 2 * G);
    const int c = chain_ok ? c_raw : 0;
    const int g = c >> 1, ch = c & 1;
    const int s = stream0 + g;
    const bool lane_valid = chain_ok && (s < p.n_streams);
    const bool do_eq = p.eq_enable != 0;

    // band A = 2l, band B = 2l+1
    float ab0 = 0.f, ab1 = 0.f, ab2 = 0.f, aa1 = 0.f, aa2 = 0.f, as1 = 0.f, as2 = 0.f;
    float bb0 = 0.f, bb1 = 0.f, bb2 = 0.f, ba1 = 0.f, ba2 = 0.f, bs1 = 0.f, bs2 = 0.f;
    bool en_a = false, en_b = false;
    const int band_a = BPL * l, band_b = BPL * l + 1;
    const bool has_a = lane_valid && do_eq && band_a < p.n_bands, has_b = BPL == 2 && lane_valid && do_eq && band_b < p.n_bands;
    // coefficients (constant across this handle's launches) before the wait for the previous launch, states after it
    if (has_a) {
        const float* cf = p.eqc + ((size_t)p.stream_eq[s] * kMaxBands + band_a) * kEqCoefStride;
        ab0 = cf[0]; ab1 = cf[1]; ab2 = cf[2]; aa1 = cf[3]; aa2 = cf[4]; en_a = cf[5] != 0.f;
    }
    if (has_b) {
        const float* cf = p.eqc + ((size_t)p.stream_eq[s] * kMaxBands + band_b) * kEqCoefStride;
        bb0 = cf[0]; bb1 = cf[1]; bb2 = cf[2]; ba1 = cf[3]; ba2 = cf[4]; en_b = cf[5] != 0.f;
    }
    grid_dependency_wait();
    if (has_a) {
        const float* st = reinterpret_cast<const float*>(p.eqs + (size_t)s * kMaxBands + band_a);
        as1 = st[ch]; as2 = st[2 + ch];
    }
    if (has_b) {
        const float* st = reinterpret_cast<const float*>(p.eqs + (size_t)s * kMaxBands + band_b);
        bs1 = st[ch]; bs2 = st[2 + ch];
    }
    // kPacked: coefficients and state as {A, B} pairs, a1 and a2 negated (df2t_step2)
    const f32x2 one2 = pk2(p.one, p.one), nz2 = pk2(p.neg_zero, p.neg_zero);
    const f32x2 b0p = pk2(ab0, bb0), b1p = pk2(ab1, bb1), b2p = pk2(ab2, bb2), na1p = pk2(-aa1, -ba1), na2p = pk2(-aa2, -ba2);
    f32x2 s1p = pk2(as1, bs1), s2p = pk2(as2, bs2);
    // scalar two-band lanes: band A's coefficients b0, b1, b2 in both words, for its products of two steps at once
    const f32x2 ab0d = pk2(ab0, ab0), ab1d = pk2(ab1, ab1), ab2d = pk2(ab2, ab2);
    bar_sync(kBarInitEq, 32 + SM::kEqThreads);   // the staging warp has initialised the mbarriers

    OHS_STAMP_IF(threadIdx.x == 0, p, 2);
    // Input rows: block t sits in stage buffer t % 3 once that buffer's mbarrier has completed its (t/3)-th phase.
    // The copies are TMA bulk copies issued by the staging warp (stager_warp_main), three blocks ahead, so the
    // EQ warps' critical path carries neither copy instructions nor a barrier for the buffer hand-over.  Only a ragged
    // last block (EQ-only mode) is loaded here, with plain guarded loads.
    uint64_t* stage_full = reinterpret_cast<uint64_t*>(smem + SM::kMbarOff);
    auto wait_stage = [&](int t) {
        const int nb = (t == p.n_blocks - 1) ? p.tail_frames : B;
        if (nb == B) { mbar_wait(&stage_full[t % 3], (unsigned)((t / 3) & 1)); return; }
        float* dst_base = stage + (size_t)(t % 3) * G * SM::kStageStride;  // last read three blocks ago
        for (int q = threadIdx.x; q < G * 2 * B; q += SM::kEqThreads) {
            const int row = q / B, n = q - row * B;
            const int sg = stream0 + (row >> 1);
            if (sg < p.n_streams && n < nb)
                dst_base[(row >> 1) * SM::kStageStride + (row & 1) * SM::kRowR + n] =
                    p.in[((size_t)(sg - p.io_first_stream) * 2 + (row & 1)) * p.row_stride + (size_t)t * B + n];
        }
        if (SM::kEqWarps > 1) bar_sync(kBarEq, SM::kEqThreads); else __syncwarp();
    };

    // One band per lane (BPL = 1): a chain's last lane has no right neighbour, nobody reads what it shuffles.  It
    // publishes the chain's INPUT samples there instead and the first lane takes its shuffle from it, so the choice
    // between "input sample" and "left neighbour's output" is made on the PRODUCER side, on values that are long since in
    // registers, and no lane executes a select on a fresh shuffle result (18 % of that loop's time went to waiting there:
    // profiles/r01_ncu_config5_spectra_only_render.txt).  With two bands per lane the same change was measured and does
    // not pay (config 2: 1.068 M against 1.080 M), so there the first lane keeps selecting on the consumer side.
    constexpr bool kPubInput = (BPL == 1);
    const int src_lane = (l == 0) ? (kPubInput ? lane + (LPC - 1) * CPW : lane) : lane - CPW;
    const bool first = (l == 0), pub = (l == LPC - 1), last = pub && lane_valid;  // lanes of absent streams never store
    const bool feeds = kPubInput ? pub : first;   // the lane that reads the staged input rows in the steady state
    // xsel[u]: band A's input at step u of the coming iteration, already chosen between the staged input sample (first
    // lane of a chain) and lane l-1's shuffled output.  The choice is made right behind the shuffle, an iteration ahead
    // of its use: ptxas gives a value whose only consumer lies behind the loop's back-edge the lowest priority and
    // sinks its shuffle to the end of the loop body, a few instructions ahead of the consumer (~20 stall cycles per
    // iteration in the SASS of the previous form).  yl: the last DL band-B outputs.
    float xsel[DL], yl[DL];
#pragma unroll
    for (int u = 0; u < DL; ++u) { xsel[u] = 0.f; yl[u] = 0.f; }
    float ya_prev = 0.f;   // this lane's band-A output of the previous step
    struct In { float4 q[NQ]; };
    auto in_at = [&](const In& in, int u) { const float4 v = in.q[u >> 2]; return (u & 3) == 0 ? v.x : (u & 3) == 1 ? v.y : (u & 3) == 2 ? v.z : v.w; };
    using SelNext = Flag<true>;
    using SelLater = Flag<false>;

    // DL steady-state steps (local steps i0 .. i0+DL-1): every lane holds live samples (lanes of absent streams run on
    // garbage that is never stored).  `in`: this iteration's input samples, `nx`: the next iteration's.  Whenever the
    // last lane has completed an aligned group of four output samples it stores the group with one 16-byte store at
    // dst + (first sample's index relative to the block): the caller passes the end of the previous block's ring row
    // during the first kLagA steps of a block (negative indices) and the block's own row afterwards.
    // SelLater: the block's last iteration; the next block's rows may not have landed, the raw shuffled values stay in
    // xsel and seed_inputs() completes them after the stage wait.
    auto fast_iter = [&](auto sel, const In& in, const In& nx, int i0, float* dst) {
        f32x2 pa0, pa1, pa2;   // scalar two-band lanes: band A's products b*x of steps u and u+1 (u even), low word = u
#pragma unroll
        for (int u = 0; u < DL; ++u) {
            if constexpr (BPL == 2) {
                // band A on xsel[u], band B on band A's previous output
                float y;
                if constexpr (kPacked) {
                    unpk2(df2t_step2(pk2(xsel[u], ya_prev), s1p, s2p, b0p, b1p, b2p, na1p, na2p, one2, nz2), ya_prev, y);
                } else {
                    // Band A's inputs are chosen steps ahead and its products lie off its recurrence: they are formed
                    // for two steps at once by FFMA2 against -0 (= the rounded products), one instruction for two
                    // FMULs.  xsel[u + 1] is final here: it was written one to three steps ago.
                    if (u % 2 == 0) {
                        const f32x2 x2 = pk2(xsel[u], xsel[u + 1]);
                        pa0 = fma2(ab0d, x2, nz2); pa1 = fma2(ab1d, x2, nz2); pa2 = fma2(ab2d, x2, nz2);
                    }
                    float q0, q1, q2, unused;
                    if (u % 2 == 0) { unpk2(pa0, q0, unused); unpk2(pa1, q1, unused); unpk2(pa2, q2, unused); }
                    else { unpk2(pa0, unused, q0); unpk2(pa1, unused, q1); unpk2(pa2, unused, q2); }
                    y = df2t_step(ya_prev, bs1, bs2, bb0, bb1, bb2, ba1, ba2);
                    ya_prev = df2t_step_products(q0, q1, q2, as1, as2, aa1, aa2);
                }
                const float r = __shfl_sync(0xffffffffu, y, src_lane);   // band A's input DL-1 steps from now
                if (u == 0) xsel[DL - 1] = first ? in_at(in, DL - 1) : r;
                else xsel[u - 1] = (decltype(sel)::value && first) ? in_at(nx, u - 1) : r;
                if ((u & 3) == kStoreU && last)
                    *reinterpret_cast<float4*>(dst + (i0 + u - 3 - kOutLag)) =
                        make_float4(yl[(u + DL - 3) % DL], yl[(u + DL - 2) % DL], yl[(u + DL - 1) % DL], y);
                yl[u] = y;
            } else {
                const float y = df2t_step(xsel[u], as1, as2, ab0, ab1, ab2, aa1, aa2);
                // producer-side select (see src_lane): the chain's last lane publishes the input sample instead of its output
                float v = y;
                if (u == 0) v = pub ? in_at(in, DL - 1) : y;
                else if (decltype(sel)::value) v = pub ? in_at(nx, u - 1) : y;
                xsel[(u + DL - 1) % DL] = __shfl_sync(0xffffffffu, v, src_lane);
                if ((u & 3) == kStoreU && last)
                    *reinterpret_cast<float4*>(dst + (i0 + u - 3 - kOutLag)) =
                        make_float4(yl[(u + DL - 3) % DL], yl[(u + DL - 2) % DL], yl[(u + DL - 1) % DL], y);
                yl[u] = y;
            }
        }
    };
    // DL checked steps (pipeline fill and drain, ragged blocks, disabled bands): state and outputs are committed only
    // where a band holds a live sample; a disabled band passes its input through and keeps its state
    // (src/dsp/parametric_eq.rs:118-120).  na0 = band A's sample index at the first of the steps; live samples
    // are [0, nb); the last lane stores sample by sample into dst0[n].
    auto checked_iter = [&](const In& in, const In& nx, int na0, int nb, float* dst0) {
#pragma unroll
        for (int u = 0; u < DL; ++u) {
            const int na = na0 + u, nbi = na - 1;
            const bool act_a = lane_valid && na >= 0 && na < nb, act_b = lane_valid && nbi >= 0 && nbi < nb;
            const float xa = xsel[u];
            if constexpr (BPL == 2) {
                float y;
                if constexpr (kPacked) {
                    const bool upd_a = act_a && en_a, upd_b = act_b && en_b;
                    f32x2 t1 = s1p, t2 = s2p;
                    float ya;
                    unpk2(df2t_step2(pk2(xa, ya_prev), t1, t2, b0p, b1p, b2p, na1p, na2p, one2, nz2), ya, y);
                    // commit each half of the pair on its own band's condition
                    auto commit = [&](f32x2& s, f32x2 t) {
                        float sa, sb, ta, tb;
                        unpk2(s, sa, sb); unpk2(t, ta, tb);
                        s = pk2(upd_a ? ta : sa, upd_b ? tb : sb);
                    };
                    commit(s1p, t1); commit(s2p, t2);
                    y = upd_b ? y : ya_prev;
                    ya_prev = upd_a ? ya : xa;
                } else {
                    float t1 = bs1, t2 = bs2;
                    y = df2t_step(ya_prev, t1, t2, bb0, bb1, bb2, ba1, ba2);
                    const bool upd_b = act_b && en_b;
                    bs1 = upd_b ? t1 : bs1; bs2 = upd_b ? t2 : bs2;
                    y = upd_b ? y : ya_prev;
                    t1 = as1; t2 = as2;
                    float ya = df2t_step(xa, t1, t2, ab0, ab1, ab2, aa1, aa2);
                    const bool upd_a = act_a && en_a;
                    as1 = upd_a ? t1 : as1; as2 = upd_a ? t2 : as2;
                    ya_prev = upd_a ? ya : xa;
                }
                const float r = __shfl_sync(0xffffffffu, y, src_lane);
                if (u == 0) xsel[DL - 1] = first ? in_at(in, DL - 1) : r;
                else xsel[u - 1] = first ? in_at(nx, u - 1) : r;
                if (act_b && last) dst0[nbi] = y;
                yl[u] = y;
            } else {
                float t1 = as1, t2 = as2;
                float y = df2t_step(xa, t1, t2, ab0, ab1, ab2, aa1, aa2);
                const bool upd_a = act_a && en_a;
                as1 = upd_a ? t1 : as1; as2 = upd_a ? t2 : as2;
                y = upd_a ? y : xa;
                const float v = pub ? (u == 0 ? in_at(in, DL - 1) : in_at(nx, u - 1)) : y;
                xsel[(u + DL - 1) % DL] = __shfl_sync(0xffffffffu, v, src_lane);
                if (act_a && last) dst0[na] = y;
                yl[u] = y;
            }
        }
    };
    // input samples [i, i+DL) of a staged row: zeros past the end of the block ...
    auto ld_in = [&](const float* row, int i) {
        In in;
#pragma unroll
        for (int q = 0; q < NQ; ++q)
            in.q[q] = (i + 4 * q < B) ? *reinterpret_cast<const float4*>(row + i + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        return in;
    };
    // ... or, for the steady state's look-ahead loads, whatever follows: i <= B stays inside the stream's stage rows
    // (the right row, or the 4-float pad behind it), and what is read there is never used
    // Only a chain's first lane uses the samples: the load is predicated on it (6 active lanes, conflict-free rows).
    // (NQ == 2 also reads the 16 bytes behind the pad: the next row, still inside the CTA's shared memory.)
    static_assert(SM::kRowR >= B + 4 && SM::kStageStride >= SM::kRowR + B + 4, "look-ahead load of the last iteration reads the pad");
    auto ld_fast = [&](In& in, const float* row, int i) {
        if constexpr (NQ == 1) {
            if (feeds) in.q[0] = *reinterpret_cast<const float4*>(row + i);
        } else {
            if (feeds) {
#pragma unroll
                for (int q = 0; q < NQ; ++q) in.q[q] = *reinterpret_cast<const float4*>(row + i + 4 * q);
            }
        }
    };
    // a block's first DL-1 inputs: taken from the staged row by the first lane, already in flight (shuffled) elsewhere
    auto seed_inputs = [&](const In& in0, bool keep) {
#pragma unroll
        for (int u = 0; u < DL - 1; ++u) xsel[u] = first ? in_at(in0, u) : (keep ? xsel[u] : 0.f);
    };
    // the stores of the first kLagA steps all belong to the previous block, all later ones to the block itself
    static_assert(kLagA - DL + kStoreU + (DL - 1 - kStoreU) / 4 * 4 - 3 - kOutLag < 0 && kLagA + kStoreU - 3 - kOutLag >= 0 &&
                  B - kLagA >= DL, "block = head iterations + pairs of iterations + one or two last iterations");
    constexpr bool kTwoLast = ((B - kLagA) / DL) % 2 == 0;

    // Every valid band filters and the launch is whole blocks: the chain runs continuously across the launch's blocks,
    // filling once at the start and draining once at the end.
    const bool lane_fast = !lane_valid || !do_eq || (en_a && has_a && (BPL == 1 || (en_b && has_b)));
    const bool all_fast = __all_sync(0xffffffffu, lane_fast);
    const bool continuous = do_eq && p.tail_frames == B && (SM::kEqWarps > 1 ? __syncthreads_and_eq<SM::kEqThreads>(all_fast) : all_fast);
    float* ring_c = ring_f + (size_t)g * SM::kRingStride + ch * SM::kRingRowR;  // this chain's channel row of slot 0
    if (continuous) {
        bool landed = false;  // block t's rows were already seen complete (polled during the previous block)
        int sb = 0; unsigned sphase = 0;  // stage buffer t % 3 and its phase (t / 3) & 1
        for (int t = 0; t < p.n_blocks; ++t) {
            if (!landed) mbar_wait(&stage_full[sb], sphase);
            OHS_STAMP_IF(threadIdx.x == 0 && t == 0, p, 3);
            if (t >= 2) bar_sync(kBarEmpty0 + (t & 1), kCount);  // ring slot t%3 was last read as history of block t-2
            const float* row = stage + ((size_t)sb * G + g) * SM::kStageStride + ch * SM::kRowR;
            float* dcur = ring_c + (t % 3) * SM::kRingSlot;
            In a = ld_in(row, 0), b = a;
            seed_inputs(a, true);
            // during the first kLagA steps the first band starts block t while the last band finishes block t-1
            if (t == 0) {
#pragma unroll 1
                for (int i = 0; i < kLagA; i += DL) { b = ld_in(row, i + DL); checked_iter(a, b, i - LL * l, B, dcur); a = b; }
            } else {
                float* dprev_end = ring_c + ((t + 2) % 3) * SM::kRingSlot + B;  // one past the previous block's row
#pragma unroll 1
                for (int i = 0; i < kLagA; i += DL) { ld_fast(b, row, i + DL); fast_iter(SelNext{}, a, b, i, dprev_end); a = b; }
                // the previous block is complete in the ring: release the convolution warps (the barrier orders the
                // shared-memory stores before the arrival for the threads that synchronise on it)
                bar_arrive(kBarFull0 + ((t - 1) & 1), SM::kFullCount);
            }
            // poll the next block's rows (issued two blocks ago) here, a block ahead of their use: the ~90-cycle
            // mbarrier round trip stays off the block boundary
            if (++sb == 3) { sb = 0; sphase ^= 1u; }
            landed = (t + 1 < p.n_blocks) && mbar_try_wait(&stage_full[sb], sphase);
            // the rest of the block: pairs of iterations with the inputs loaded one iteration ahead, then the last one
            ld_fast(b, row, kLagA + DL);
            int i = kLagA;
#pragma unroll 1
            for (; i + 2 * DL < B; i += 2 * DL) {
                fast_iter(SelNext{}, a, b, i, dcur);
                ld_fast(a, row, i + 2 * DL);
                fast_iter(SelNext{}, b, a, i + DL, dcur);
                ld_fast(b, row, i + 3 * DL);
            }
            if constexpr (kTwoLast) { fast_iter(SelNext{}, a, b, i, dcur); a = b; i += DL; }
            fast_iter(SelLater{}, a, a, i, dcur);
        }
        {
            // drain: the first band has no more input; flush the three outputs the last fast iteration left pending,
            // then run the remaining steps checked (sample by sample stores)
            float* dl = ring_c + ((p.n_blocks - 1) % 3) * SM::kRingSlot;
            if (last) {
#pragma unroll
                for (int e = 0; e < kPending; ++e) dl[B - kOutLag - kPending + e] = yl[DL - kPending + e];
            }
            In zero;
#pragma unroll
            for (int q = 0; q < NQ; ++q) zero.q[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            seed_inputs(zero, true);
#pragma unroll 1
            for (int i = 0; i < kOutLag; i += DL) checked_iter(zero, zero, B + i - LL * l, B, dl);
            bar_arrive(kBarFull0 + ((p.n_blocks - 1) & 1), SM::kFullCount);
            OHS_STAMP_IF(threadIdx.x == 0, p, 4);
        }
    } else {
        for (int t = 0; t < p.n_blocks; ++t) {
            wait_stage(t);
            if (t >= 2) bar_sync(kBarEmpty0 + (t & 1), kCount);
            const int slot = t % 3;
            const int nb = (t == p.n_blocks - 1) ? p.tail_frames : B;
            const float* st_base = stage + (size_t)(t % 3) * G * SM::kStageStride;
            if (!do_eq) {
                // EQ off (src/lib.rs:1179): the EQ warps only move the rows into the ring
                for (int q = threadIdx.x; q < G * 2 * B; q += SM::kEqThreads) {
                    const int gg = q / (2 * B), n = q - gg * 2 * B;  // n runs over [left row | right row]
                    ring_f[gg * SM::kRingStride + slot * SM::kRingSlot + (n < B ? n : n - B + SM::kRingRowR)] =
                        st_base[gg * SM::kStageStride + (n < B ? n : n - B + SM::kRowR)];
                }
            } else {
                // per-block chain (ragged last block and/or disabled bands): fill, run and drain inside the block
                const float* row = st_base + g * SM::kStageStride + ch * SM::kRowR;
                float* dst = ring_c + slot * SM::kRingSlot;
                In a = ld_in(row, 0), b;
                seed_inputs(a, false);
                xsel[DL - 1] = 0.f;
                ya_prev = 0.f;
#pragma unroll 1
                for (int i = 0; i < nb + kOutLag; i += DL) { b = ld_in(row, i + DL); checked_iter(a, b, i - LL * l, nb, dst); a = b; }
            }
            bar_arrive(kBarFull0 + (t & 1), SM::kFullCount);
        }
    }
    if constexpr (kPacked) { unpk2(s1p, as1, bs1); unpk2(s2p, as2, bs2); }
    if (has_a) { float* st = reinterpret_cast<float*>(p.eqs + (size_t)s * kMaxBands + band_a); st[ch] = as1; st[2 + ch] = as2; }
    if (has_b) { float* st = reinterpret_cast<float*>(p.eqs + (size_t)s * kMaxBands + band_b); st[ch] = bs1; st[2 + ch] = bs2; }
    OHS_STAMP_IF(threadIdx.x == 0, p, 8);
}

// block 0 of a launch arrives by TMA unless it is a ragged (EQ-only) last block, which the EQ warps load themselves
__device__ __forceinline__ bool first_block_by_tma(const RenderParams& p, int B) { return p.n_blocks > 1 || p.tail_frames == B; }

// ---------------------------------------------------------------------------------------------------------------
// staging warp
// ---------------------------------------------------------------------------------------------------------------
// Issues the TMA bulk copies of the input rows (HBM -> stage buffer t % 3; one copy of B*4 contiguous bytes per row by
// lane = row, lane 0 arms the buffer's mbarrier with the byte count), three blocks ahead.  Buffer t % 3 is free once
// every EQ thread has arrived at block t-3's FULL barrier (it read the rows before it arrived); the warp listens in on
// that barrier and otherwise sleeps, so neither the EQ warps nor the convolution warps carry copy instructions.  A
// ragged last block is loaded by the EQ warps themselves (eq_warp_main::wait_stage).
template <int N, int G, int V>
__device__ __forceinline__ void stager_warp_main(const RenderParams& p, unsigned char* smem, int stream0) {
    using SM = RenderSmem<N, G, V>;
    const bool conv_on = !SM::kEqOnly && p.conv_enable != 0;   // compile-time false in the EQ-only variant: its transforms are dead code
    constexpr int B = SM::B;
    const int n_str = (p.n_streams - stream0) < G ? (p.n_streams - stream0) : G;
    const int row = threadIdx.x & 31;   // 2G <= 14 rows
    auto issue = [&](int t, bool reused) {
        if (t >= p.n_blocks || (t == p.n_blocks - 1 && p.tail_frames != B)) return;
        uint64_t* full = reinterpret_cast<uint64_t*>(smem + SM::kMbarOff) + (t % 3);
        float* dst_base = reinterpret_cast<float*>(smem + SM::kStageOff) + (size_t)(t % 3) * G * SM::kStageStride;
        if (reused) fence_proxy_async();   // the async-proxy writes stay behind the generic-proxy reads ordered by the barrier
        if (row == 0) mbar_expect_tx(full, (unsigned)(n_str * 2 * B * sizeof(float)));
        if (row < 2 * n_str) {
            const float* src = p.in + ((size_t)(stream0 - p.io_first_stream + (row >> 1)) * 2 + (row & 1)) * p.row_stride + (size_t)t * B;
            tma_load_1d(dst_base + (row >> 1) * SM::kStageStride + (row & 1) * SM::kRowR, src, (unsigned)(B * sizeof(float)), full);
        }
    };
    // The CTA's prologue data also arrives by TMA, all of it in flight at once and none of it through registers.  A TMA
    // copy is a warp-uniform instruction: a warp that issues one copy per lane issues them one after the other (~70
    // cycles each), so the copies a launch's first block waits for are spread over the warps: this warp initialises
    // the mbarriers and brings in the twiddle tables and the shared filter spectra (constant across this handle's
    // launches: issued BEFORE the wait for the previous launch); each stream's convolution warp fetches that stream's
    // block-0 input rows and overlap-save history rows (conv_warps_main); blocks 1 and 2 follow from here.
    {
        uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::kMbarOff);
        const unsigned tw_bytes = SM::kEqOnly ? 0u : (unsigned)(sizeof(float2) * N);
        const unsigned filt_bytes = SM::kEqOnly ? 0u : (unsigned)(p.filt_in_smem * N * sizeof(float4));
        const unsigned hist_bytes = conv_on ? (unsigned)(n_str * 2 * B * sizeof(float)) : 0u;
        if (row == 0) {
            mbar_init(&bars[0], 1);   // stage_full[0..2]: input rows of block t in stage buffer t % 3
            mbar_init(&bars[1], 1);
            mbar_init(&bars[2], 1);
            mbar_init(&bars[3], 1);   // filt_full[0..1]: filter tiles of the long-impulse-response path
            mbar_init(&bars[4], 1);
            mbar_init(&bars[5], 1);   // prologue_full: twiddles, shared filter spectra, overlap-save history
            fence_mbar_init();
            // the byte counts the other warps' copies will complete (block 0's rows, the history rows)
            if (first_block_by_tma(p, B)) mbar_expect_tx(&bars[0], (unsigned)(n_str * 2 * B * sizeof(float)));
            mbar_expect_tx(&bars[5], tw_bytes + filt_bytes + hist_bytes);
        }
        __syncwarp();
        bar_arrive(kBarInitConv, 32 + G * SM::T);
        bar_arrive(kBarInitEq, 32 + SM::kEqThreads);
        OHS_STAMP_IF(row == 0, p, 10);
        if (row == 0) {
            if (tw_bytes) tma_load_1d(smem + SM::kTwOff, p.tw, tw_bytes, &bars[5]);
            // the fused single-partition path reads bin k at position k: its table lands in stream 0's (idle) FFT buffers
            // and the convolution warps permute it into place; every other path keeps the global even-bins-first layout
            if (filt_bytes) tma_load_1d(smem + (SM::kFusedMac && p.filt_in_smem == 1 ? SM::kZOff : SM::kFiltOff), p.filt, filt_bytes, &bars[5]);
        }
        OHS_STAMP_IF(row == 0, p, 11);
        grid_dependency_wait();
        OHS_STAMP_IF(row == 0, p, 12);
    }
    issue(1, false); issue(2, false);
    OHS_STAMP_IF(row == 0, p, 9);
    for (int t = 0; t < p.n_blocks; ++t) {   // every block: the barriers count this warp
        bar_sync(kBarFull0 + (t & 1), SM::kFullCount);
        issue(t + 3, true);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// convolution warps
// ---------------------------------------------------------------------------------------------------------------
// W[ka] += u*A[ka] + conj(pu)*C[ka]
__device__ __forceinline__ void mac_bin(float2& acc, float2 u, float2 pu, float4 f) {
    acc.x = fmaf(u.x, f.x, acc.x); acc.x = fmaf(-u.y, f.y, acc.x);
    acc.y = fmaf(u.x, f.y, acc.y); acc.y = fmaf(u.y, f.x, acc.y);
    acc.x = fmaf(pu.x, f.z, acc.x); acc.x = fmaf(pu.y, f.w, acc.x);
    acc.y = fmaf(pu.x, f.w, acc.y); acc.y = fmaf(-pu.y, f.z, acc.y);
}

// first-pass loader of the forward transform: the overlap-save window [previous block | current block] read from the
// planar ring, z = left + i*right
struct RingWindow {
    const float* xp; const float* xc; int B; int R;  // R: offset of a slot's right row
    __device__ __forceinline__ float2 ld(int i) const {
        return i < B ? make_float2(xp[i], xp[R + i]) : make_float2(xc[i - B], xc[R + i - B]);
    }
    __device__ __forceinline__ void ld2(int i, float2& a, float2& b) const {  // i even: samples i and i+1
        const float* row = i < B ? xp + i : xc + (i - B);
        const float2 l = *reinterpret_cast<const float2*>(row), r = *reinterpret_cast<const float2*>(row + R);
        a = make_float2(l.x, r.x); b = make_float2(l.y, r.y);
    }
};

// last-pass store of the inverse transform (run as swap o FFT o swap): keep the last B samples, left = Im, right = Re
// of the swapped result, times the gain; coalesced stores straight to the output rows
struct OutputStore {
    float* ol; float* orr; float gain; int B;  // ol/orr already offset by -B
    __device__ __forceinline__ void st(int i, float2 v) const {
        if (i >= B) { ol[i] = v.y * gain; orr[i] = v.x * gain; }
    }
    __device__ __forceinline__ void st2(int i, float2 a, float2 b) const {  // i even
        if (i >= B) {
            *reinterpret_cast<float2*>(ol + i) = make_float2(a.y * gain, b.y * gain);
            *reinterpret_cast<float2*>(orr + i) = make_float2(a.x * gain, b.x * gain);
        }
    }
};

// OutputStore of the moving-sources kernel.  With `blend` (second pass of a transition block) the rows already hold the
// old set's output a, written by this same thread (the last passes of the two inverse transforms map elements to
// threads identically), this pass's output is b, and out[n] = a + w[n]*(b - a) with w[n] = (2n+1)/(2B), exact in f32,
// each operation rounded on its own
struct MixStore {
    float* ol; float* orr; float gain; int B; bool blend;
    __device__ __forceinline__ float mix(float a, float b, int n) const {
        const float w = __fmul_rn((float)(2 * n + 1), __frcp_rn((float)(2 * B)));
        return __fadd_rn(a, __fmul_rn(w, __fsub_rn(b, a)));
    }
    __device__ __forceinline__ void st(int i, float2 v) const {
        if (i >= B) {
            float l = __fmul_rn(v.y, gain), r = __fmul_rn(v.x, gain);
            if (blend) { l = mix(ol[i], l, i - B); r = mix(orr[i], r, i - B); }
            ol[i] = l; orr[i] = r;
        }
    }
    __device__ __forceinline__ void st2(int i, float2 a, float2 b) const {  // i even
        if (i >= B) {
            float2 l = make_float2(__fmul_rn(a.y, gain), __fmul_rn(b.y, gain)), r = make_float2(__fmul_rn(a.x, gain), __fmul_rn(b.x, gain));
            if (blend) {
                const float2 la = *reinterpret_cast<const float2*>(ol + i), ra = *reinterpret_cast<const float2*>(orr + i);
                l = make_float2(mix(la.x, l.x, i - B), mix(la.y, l.y, i + 1 - B));
                r = make_float2(mix(ra.x, r.x, i - B), mix(ra.y, r.y, i + 1 - B));
            }
            *reinterpret_cast<float2*>(ol + i) = l;
            *reinterpret_cast<float2*>(orr + i) = r;
        }
    }
};

// M: the moving-sources instantiation (render_kernel<..., true>).  Every block may name its own set; a block whose set
// differs from the previous block's renders both sets' outputs from the one history and crossfades them (MixStore).
template <int N, int G, int V, bool M = false>
__device__ __forceinline__ void conv_warps_main(const RenderParams& p, unsigned char* smem, int stream0, int conv_index) {
    using SM = RenderSmem<N, G, V>;
    const bool conv_on = !SM::kEqOnly && p.conv_enable != 0;   // compile-time false in the EQ-only variant: its transforms are dead code
    constexpr int B = SM::B, T = SM::T, NP = SM::NP;
    constexpr int kCount = SM::kWorkers;
    using Pl = FftPlan<N, T>;
    const float2* tw = reinterpret_cast<const float2*>(smem + SM::kTwOff);
    float* ring = reinterpret_cast<float*>(smem + SM::kRingOff);

    const int ft = conv_index * 32 + (threadIdx.x & 31);
    const int g = ft / T, tid = ft - g * T;
    const int s = stream0 + g;
    const bool valid = s < p.n_streams;
    float2* b0 = reinterpret_cast<float2*>(smem + SM::kZOff) + (size_t)g * 2 * NP;
    float2* b1 = b0 + NP;
    const SmemCx zbuf{Pl::kOutInB0 ? b0 : b1};   // forward transform lands here
    const SmemCx wbuf{Pl::kOutInB0 ? b1 : b0};   // frequency-domain product goes here
    float* ring_g = ring + (size_t)g * SM::kRingStride;  // planar: slot k = [left row | right row] at k*2*B

    int nparts = 1;
    const float4* filt = p.filt;      // all partitions: resident shared-memory copy or global (generic pointer)
    const float4* filt_g = p.filt;    // the set's table in global memory
    float gain = 1.f;
    float2* fdl_s = nullptr;
    if (valid) {
        const int set = p.stream_hrir[s];
        nparts = p.set_parts[set];
        filt = p.filt_in_smem ? reinterpret_cast<const float4*>(smem + SM::kFiltOff) : p.filt + (size_t)set * p.pmax * N;
        filt_g = p.filt + (size_t)set * p.pmax * N;
        gain = SM::kEqOnly ? 1.f : p.stream_gain[s];   // the EQ pre-pass hands the filtered samples on as they are
        fdl_s = p.fdl + (size_t)s * p.pmax * N;
    }
    float* out_l = p.out + ((size_t)(s - p.io_first_stream) * 2) * p.out_row_stride;
    float* out_r = out_l + p.out_row_stride;
    auto stream_sync = [&]() { if (T > 32) bar_sync(kBarStream0 + g, T); else __syncwarp(); };
    // the delay line, the history rows and possibly the input rows are what the previous launch wrote
    grid_dependency_wait();
    int set_prev = 0;   // moving: the set of the block before block t
    if constexpr (M) { if (valid) set_prev = p.from_set[s]; }
    bar_sync(kBarInitConv, 32 + G * T);   // the staging warp has initialised the mbarriers
    // this stream's block-0 input rows and overlap-save history rows (ring slot 2): two copies each, issued here so
    // that the CTA's streams fetch theirs side by side (stager_warp_main)
    if (valid && tid < 2) {
        uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::kMbarOff);
        if (first_block_by_tma(p, B))
            tma_load_1d(reinterpret_cast<float*>(smem + SM::kStageOff) + g * SM::kStageStride + tid * SM::kRowR,
                        p.in + ((size_t)(s - p.io_first_stream) * 2 + tid) * p.row_stride, (unsigned)(B * sizeof(float)), &bars[0]);
        if (conv_on)
            tma_load_1d(ring_g + 2 * SM::kRingSlot + tid * SM::kRingRowR, reinterpret_cast<const float*>(p.prev) + ((size_t)s * 2 + tid) * B,
                        (unsigned)(B * sizeof(float)), &bars[5]);
    }
    OHS_STAMP_IF(ft == 0, p, 13);
    // twiddles, shared filter spectra and history rows have landed
    mbar_wait(reinterpret_cast<uint64_t*>(smem + SM::kMbarOff) + 5, 0u);
    OHS_STAMP_IF(ft == 0, p, 1);
    if constexpr (SM::kFusedMac && SM::kFiltSmemBytes > 0) {
        if (p.filt_in_smem == 1) {
            // even-bins-first (global layout, landed in stream 0's FFT buffers) -> natural order
            const float4* src = reinterpret_cast<const float4*>(smem + SM::kZOff);
            float4* fs = reinterpret_cast<float4*>(smem + SM::kFiltOff);
            for (int i = ft; i < N; i += G * T) fs[i] = src[(i & 1) * (N / 2) + (i >> 1)];
            bar_sync(kBarConv, G * T);
        }
    }

    constexpr int kPairs = N / 4 / T;
    // TMA filter-tile pipeline (see the block loop): needs two streams' FFT buffers as tile buffers, one shared set with
    // more partitions than fit the resident table, and every conv thread of the CTA taking part
    uint64_t* filt_full = reinterpret_cast<uint64_t*>(smem + SM::kMbarOff) + 3;
    unsigned filt_phase[2] = {0u, 0u};
    constexpr bool kTmaFilterPath = (G >= 2) && (N >= 1024);  // compiled only where long responses live (register budget)
    if (kTmaFilterPath && p.uniform_set && !valid) nparts = p.set_parts[0];  // threads of an absent stream still run the tile loop
    const bool tma_filters = kTmaFilterPath && p.uniform_set && !p.filt_in_smem && conv_on && nparts > 1;
    // one delay-line partition's worth of operands of a bin pair: Z[k], Z[k+1], Z[mirror k], Z[mirror k+1] and their filters
    struct Operands { float4 uu; float2 v0, v1; float4 f0, f1, g0, g1; };
    // a partition's filter table is stored even bins first, odd bins behind them (setup_filters_kernel): a warp's loads
    // of its bins k = 2*lane, of k+1 and of the mirror bins are each contiguous across the lanes
    auto fe = [](int j) { return j >> 1; };             // position of even bin j
    auto fo = [](int j) { return N / 2 + (j >> 1); };   // position of odd bin j
    auto load_ops = [&](const float2* zq, const float4* fq, int k, int m0, int m1) {
        Operands o;
        o.uu = *reinterpret_cast<const float4*>(zq + k);
        o.v0 = zq[m0]; o.v1 = zq[m1];
        o.f0 = fq[fe(k)]; o.f1 = fq[fo(k + 1)]; o.g0 = fq[fe(m0)]; o.g1 = fq[fo(m1)];
        return o;
    };
    auto mac_ops = [&](float2 (&acc)[4], const Operands& o, int k) {
        const float2 u0 = make_float2(o.uu.x, o.uu.y), u1 = make_float2(o.uu.z, o.uu.w);
        mac_bin(acc[0], u0, k ? o.v0 : u0, o.f0);
        mac_bin(acc[1], u1, o.v1, o.f1);
        mac_bin(acc[2], o.v0, k ? u0 : o.v0, o.g0);
        mac_bin(acc[3], o.v1, u1, o.g1);
    };

    for (int t = 0; t < p.n_blocks; ++t) {
        int slot = p.head + t;
        slot -= (slot / p.pmax) * p.pmax;
        // moving: this block's set; a transition block (set differs from the previous block's) renders the old set's
        // output as well, so its history product waits until after the forward transform
        bool trans = false;
        int set_old = set_prev;
        if constexpr (M) {
            if (valid) {
                const int set = p.block_set ? p.block_set[(size_t)s * p.block_set_stride + t] : p.stream_hrir[s];
                trans = set != set_prev;
                set_prev = set;
                nparts = p.set_parts[set];
                filt_g = p.filt + (size_t)set * p.pmax * N;
                filt = p.filt_in_smem ? reinterpret_cast<const float4*>(smem + SM::kFiltOff) : filt_g;
            }
        }
        // ---- delay-line history first.  The partitions 1..P-1 of this block's product only need spectra of EARLIER
        // blocks, so their multiply-accumulate (the HBM-heavy part of a long impulse response: P-1 tiles of 8*N bytes per
        // stream) runs BEFORE the wait for this block's EQ output and overlaps the EQ warps' sequential work.  A thread
        // owns adjacent bins (k, k+1), k even, k < N/2, and their mirror bins N-k, N-k-1 (bin 0 pairs with itself, N/2
        // rides along with it); four partitions' operands are in flight at once.
        float2 acc[kPairs][4];  // W[k], W[k+1], W[mirror(k)], W[mirror(k+1)]
#pragma unroll
        for (int m = 0; m < kPairs; ++m)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[m][e] = make_float2(0.f, 0.f);
        if constexpr (kTmaFilterPath) { if (tma_filters) {
            // Long impulse response shared by the CTA's streams (config 5): partition q's filter tile (16*N bytes, the
            // same for every stream) is brought into shared memory by ONE TMA bulk copy, double-buffered in the FFT
            // ping-pong buffers of streams 0 and 1 (idle until the forward FFT), while each thread keeps two
            // partitions' worth of its own delay-line operands in flight in registers.  Partition-outer loop: every
            // tile is read from L2 once per CTA instead of once per stream, and never through a register prefetch.
            float4* fbuf[2] = {reinterpret_cast<float4*>(smem + SM::kZOff), reinterpret_cast<float4*>(smem + SM::kZOff) + (size_t)NP};
            const float4* fsrc = p.filt;  // set 0
            constexpr unsigned kTileBytes = (unsigned)(sizeof(float4) * N);
            struct ZOps { float4 uu; float2 v0, v1; };
            ZOps zr[2][kPairs];
            auto load_z = [&](ZOps (&dst)[kPairs], int q) {
                int sl = slot - q; if (sl < 0) sl += p.pmax;
                const float2* zq = fdl_s + (size_t)sl * N;
#pragma unroll
                for (int m = 0; m < kPairs; ++m) {
                    const int k = 2 * (tid + m * T);
                    dst[m].uu = *reinterpret_cast<const float4*>(zq + k);
                    dst[m].v0 = zq[k ? N - k : N / 2];
                    dst[m].v1 = zq[N - k - 1];
                }
            };
            // the tile buffers were last touched through the generic proxy (previous block's inverse FFT)
            fence_proxy_async();
            bar_sync(kBarConv, G * T);
            if (ft == 0) {
#pragma unroll
                for (int j = 0; j < 2; ++j)
                    if (1 + j < nparts) { mbar_expect_tx(&filt_full[j], kTileBytes); tma_load_1d(fbuf[j], fsrc + (size_t)(1 + j) * N, kTileBytes, &filt_full[j]); }
            }
            if (valid) {
                load_z(zr[0], 1);
                if (2 < nparts) load_z(zr[1], 2);
            }
#pragma unroll 1
            for (int q0 = 1; q0 < nparts; q0 += 2) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int q = q0 + j;
                    if (q < nparts) {
                        mbar_wait(&filt_full[j], filt_phase[j]);
                        filt_phase[j] ^= 1u;
                        if (valid) {
                            const float4* fq = fbuf[j];
#pragma unroll
                            for (int m = 0; m < kPairs; ++m) {
                                const int k = 2 * (tid + m * T);
                                const int m0 = k ? N - k : N / 2, m1 = N - k - 1;
                                Operands o;
                                o.uu = zr[j][m].uu; o.v0 = zr[j][m].v0; o.v1 = zr[j][m].v1;
                                o.f0 = fq[fe(k)]; o.f1 = fq[fo(k + 1)]; o.g0 = fq[fe(m0)]; o.g1 = fq[fo(m1)];
                                mac_ops(acc[m], o, k);
                            }
                            if (q + 2 < nparts) load_z(zr[j], q + 2);
                        }
                        fence_proxy_async();
                        bar_sync(kBarConv, G * T);  // every conv thread is done with tile buffer j
                        if (ft == 0 && q + 2 < nparts) {
                            mbar_expect_tx(&filt_full[j], kTileBytes);
                            tma_load_1d(fbuf[j], fsrc + (size_t)(q + 2) * N, kTileBytes, &filt_full[j]);
                        }
                    }
                }
            }
        } }
        if (!tma_filters && valid && conv_on && nparts > 1 && !trans) {
#pragma unroll 1
            for (int m = 0; m < kPairs; ++m) {
                const int k = 2 * (tid + m * T);
                const int m0 = k ? N - k : N / 2, m1 = N - k - 1;
                float2 a4[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
                int q = 1;
#pragma unroll 1
                for (; q + 3 < nparts; q += 4) {
                    Operands o[4];
#pragma unroll
                    for (int jq = 0; jq < 4; ++jq) {
                        int sl = slot - (q + jq); if (sl < 0) sl += p.pmax;
                        o[jq] = load_ops(fdl_s + (size_t)sl * N, filt + (size_t)(q + jq) * N, k, m0, m1);
                    }
#pragma unroll
                    for (int jq = 0; jq < 4; ++jq) mac_ops(a4, o[jq], k);
                }
#pragma unroll 1
                for (; q < nparts; ++q) {
                    int sl = slot - q; if (sl < 0) sl += p.pmax;
                    const Operands o = load_ops(fdl_s + (size_t)sl * N, filt + (size_t)q * N, k, m0, m1);
                    mac_ops(a4, o, k);
                }
                // scatter back into the per-pair accumulators with static indices
#pragma unroll
                for (int mm = 0; mm < kPairs; ++mm)
                    if (mm == m) { acc[mm][0] = a4[0]; acc[mm][1] = a4[1]; acc[mm][2] = a4[2]; acc[mm][3] = a4[3]; }
            }
        }
        bar_sync(kBarFull0 + (t & 1), SM::kFullCount);
        OHS_STAMP_IF(ft == 0 && t == 0, p, 5);
        const int cur = t % 3, prv = (t + 2) % 3;
        const float* xc = ring_g + cur * SM::kRingSlot;
        const float* xp = ring_g + prv * SM::kRingSlot;
        const bool release = (t + 2 < p.n_blocks);
        if (!valid) {
            if (release) bar_arrive(kBarEmpty0 + (t & 1), kCount);
            continue;
        }
        if (!conv_on) {
            // EQ + gain only (StereoParametricEQ::process_block followed by the gain loop)
            const int nb = (t == p.n_blocks - 1) ? p.tail_frames : B;
            for (int n = tid; n < nb; n += T) {
                out_l[(size_t)t * B + n] = xc[n] * gain;
                out_r[(size_t)t * B + n] = xc[SM::kRingRowR + n] * gain;
            }
            if (release) bar_arrive(kBarEmpty0 + (t & 1), kCount);
            continue;
        }
        if constexpr (SM::kFusedMac) {
            // (moving: not where the delay line must carry every block's spectrum, and not in a transition block)
            if (nparts == 1 && (!M || (p.pmax == 1 && !trans))) {
                // ---- single partition: forward passes 1 and 2 through shared memory; then the last forward pass, the
                // spectral product and the first inverse pass in registers.  The last pass's butterfly i produces the
                // bins i + q*NB (q < R), exactly the inputs of the inverse transform's first-pass butterfly i, and the
                // mirror bins N - (i + q*NB) are the outputs NB-i + (R-1-q)*NB of butterfly NB-i: a thread that owns
                // butterflies i and NB-i holds every operand of W[k] = Z[k] A[k] + conj(Z[N-k]) C[k] for its 2R bins.
                // (Thread 0 owns the two self-mirrored butterflies 0 and NB/2.)  Same arithmetic in the same order as
                // the general path, a third fewer shared-memory wavefronts and two fewer synchronisations per block.
                constexpr int R = Pl::R3, NB = N / R;
                const SmemCx c0{b0}, c1{b1};
                fft_pass<N, T, Pl::R1, Pl::P1>(tid, tw, RingWindow{xp, xc, B, SM::kRingRowR}, c0);
                if (release) bar_arrive(kBarEmpty0 + (t & 1), kCount);
                stream_sync();
                fft_pass<N, T, Pl::R2, Pl::P2>(tid, tw + Pl::kTw2, c0, c1);
                stream_sync();
                const bool t0 = (tid == 0);
                const int iu = tid, iv = t0 ? NB / 2 : NB - tid;
                float2 u[R], v[R], wu[R], wv[R];
#pragma unroll
                for (int r = 0; r < R; ++r) { u[r] = c1.ld(iu + r * NB); v[r] = c1.ld(iv + r * NB); }
                const float2* tw3 = tw + Pl::kTw3;   // w^{k r / N}, k < NB
#pragma unroll
                for (int r = 1; r < R; ++r) { u[r] = cmul(u[r], tw3[(r - 1) * NB + iu]); v[r] = cmul(v[r], tw3[(r - 1) * NB + iv]); }
                Dft<R>::run(u);
                Dft<R>::run(v);
                auto product = [&](auto fld) {
#pragma unroll
                    for (int q = 0; q < R; ++q) {
                        const float2 mu = t0 ? u[(R - q) & (R - 1)] : v[R - 1 - q];
                        const float2 mv = t0 ? v[R - 1 - q] : u[R - 1 - q];
                        float2 a = make_float2(0.f, 0.f), b = make_float2(0.f, 0.f);
                        mac_bin(a, u[q], mu, fld(iu + q * NB));
                        mac_bin(b, v[q], mv, fld(iv + q * NB));
                        wu[q] = make_float2(a.y, a.x);  // swap(re, im): the inverse transform is run as swap(FFT(swap(W)))
                        wv[q] = make_float2(b.y, b.x);
                    }
                };
                if (SM::kFiltSmemBytes > 0 && p.filt_in_smem) {
                    const float4* fs = reinterpret_cast<const float4*>(smem + SM::kFiltOff);  // natural order (render_kernel)
                    product([&](int k) { return fs[k]; });
                } else {
                    product([&](int k) { return filt_g[(k & 1) * (N / 2) + (k >> 1)]; });
                }
                Dft<R>::run(wu);
                Dft<R>::run(wv);
#pragma unroll
                for (int q = 0; q < R; q += 2) { c0.st2(iu * R + q, wu[q], wu[q + 1]); c0.st2(iv * R + q, wv[q], wv[q + 1]); }
                stream_sync();
                fft_pass<N, T, Pl::R2, Pl::P2>(tid, tw + Pl::kTw2, c0, c1);
                stream_sync();
                fft_pass<N, T, Pl::R3, Pl::P3>(tid, tw + Pl::kTw3, c1, OutputStore{out_l + (size_t)t * B - B, out_r + (size_t)t * B - B, gain, B});
                continue;
            }
        }
        // ---- forward FFT of the overlap-save window [previous block | current block], z = left + i*right
        fft_run<N, T>(tid, tw, b0, b1, RingWindow{xp, xc, B, SM::kRingRowR}, zbuf, stream_sync,
                      [&]() { if (release) bar_arrive(kBarEmpty0 + (t & 1), kCount); });
        stream_sync();
        // ---- this block's spectrum: into the delay line, and its product with partition 0 on top of the history.
        // (Moving: always.  A later block may move to a set with more partitions than this one's, and a transition
        // block re-reads it after its first inverse transform.)
        if (M || nparts > 1) {
            float4* dstz = reinterpret_cast<float4*>(fdl_s + (size_t)slot * N);
#pragma unroll
            for (int e = 0; e < N / 2 / T; ++e) {
                const int i = 2 * (tid + e * T);
                float2 z0, z1;
                zbuf.ld2(i, z0, z1);
                dstz[i >> 1] = make_float4(z0.x, z0.y, z1.x, z1.y);
            }
        }
        // partition 0 of filter table fq on top of the history in acc, with this block's spectrum read from z (zbuf, or
        // moving: its delay-line slot), and the swapped product into wbuf.  The static path's table is the resident
        // shared-memory copy (plain LDS: the address space is known at compile time) or global memory; one generic
        // pointer for both would compile to generic loads
        auto mac_partition0 = [&](const auto& z, const float4* fq) {
#pragma unroll
            for (int m = 0; m < kPairs; ++m) {
                const int k = 2 * (tid + m * T);
                const int m0 = k ? N - k : N / 2, m1 = N - k - 1;
                Operands o;
                float2 u0, u1;
                z.ld2(k, u0, u1);
                o.uu = make_float4(u0.x, u0.y, u1.x, u1.y);
                o.v0 = z.ld(m0); o.v1 = z.ld(m1);
                o.f0 = fq[fe(k)]; o.f1 = fq[fo(k + 1)]; o.g0 = fq[fe(m0)]; o.g1 = fq[fo(m1)];
                mac_ops(acc[m], o, k);
                // swap(re, im): the inverse transform is run as swap(FFT(swap(W)))
                wbuf.st2(k, make_float2(acc[m][0].y, acc[m][0].x), make_float2(acc[m][1].y, acc[m][1].x));
                wbuf.st(m0, make_float2(acc[m][2].y, acc[m][2].x));
                wbuf.st(m1, make_float2(acc[m][3].y, acc[m][3].x));
            }
        };
        if constexpr (M) {
            // Partition 0 reads this block's spectrum back from its delay-line slot (the first inverse transform of a
            // transition block overwrites both FFT buffers).  A transition block runs two passes: the old set's output
            // a into the output rows, then the new set's b blended onto it (MixStore); both in the static path's
            // order, history partitions first (mac_history, the same loop as above), then partition 0.
            auto mac_history = [&](const float4* fq, int np) {
#pragma unroll 1
                for (int m = 0; m < kPairs; ++m) {
                    const int k = 2 * (tid + m * T);
                    const int m0 = k ? N - k : N / 2, m1 = N - k - 1;
                    float2 a4[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
                    int q = 1;
#pragma unroll 1
                    for (; q + 3 < np; q += 4) {
                        Operands o[4];
#pragma unroll
                        for (int jq = 0; jq < 4; ++jq) {
                            int sl = slot - (q + jq); if (sl < 0) sl += p.pmax;
                            o[jq] = load_ops(fdl_s + (size_t)sl * N, fq + (size_t)(q + jq) * N, k, m0, m1);
                        }
#pragma unroll
                        for (int jq = 0; jq < 4; ++jq) mac_ops(a4, o[jq], k);
                    }
#pragma unroll 1
                    for (; q < np; ++q) {
                        int sl = slot - q; if (sl < 0) sl += p.pmax;
                        const Operands o = load_ops(fdl_s + (size_t)sl * N, fq + (size_t)q * N, k, m0, m1);
                        mac_ops(a4, o, k);
                    }
#pragma unroll
                    for (int mm = 0; mm < kPairs; ++mm)
                        if (mm == m) { acc[mm][0] = a4[0]; acc[mm][1] = a4[1]; acc[mm][2] = a4[2]; acc[mm][3] = a4[3]; }
                }
            };
            stream_sync();
            const GlobalCx zs{fdl_s + (size_t)slot * N};
#pragma unroll 1
            for (int pass = trans ? 0 : 1; pass < 2; ++pass) {
                const float4* fq = filt_g;
                if (trans) {
                    int np = nparts;
                    if (pass == 0) { fq = p.filt + (size_t)set_old * p.pmax * N; np = p.set_parts[set_old]; }
#pragma unroll
                    for (int m = 0; m < kPairs; ++m)
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[m][e] = make_float2(0.f, 0.f);
                    if (np > 1) mac_history(fq, np);
                }
                mac_partition0(zs, fq);
                stream_sync();
                fft_run<N, T>(tid, tw, zbuf.p, wbuf.p, wbuf, MixStore{out_l + (size_t)t * B - B, out_r + (size_t)t * B - B, gain, B, trans && pass == 1},
                              stream_sync, [&]() {});
                if (pass == 0) stream_sync();   // both FFT buffers are free again
            }
            continue;
        }
        if (SM::kFiltSmemBytes > 0 && p.filt_in_smem) mac_partition0(zbuf, reinterpret_cast<const float4*>(smem + SM::kFiltOff));
        else mac_partition0(zbuf, filt_g);
        stream_sync();
        // ---- inverse FFT; keep the last B samples (overlap-save), ear sums are already inside W, apply gain
        fft_run<N, T>(tid, tw, zbuf.p, wbuf.p, wbuf, OutputStore{out_l + (size_t)t * B - B, out_r + (size_t)t * B - B, gain, B},
                      stream_sync, [&]() {});
    }
    OHS_STAMP_IF(ft == 0, p, 6);
    // overlap-save history for the next launch: the last filtered block
    if (valid && conv_on && p.n_blocks > 0) {
        const float* xc = ring_g + ((p.n_blocks - 1) % 3) * SM::kRingSlot;
        float* hl = reinterpret_cast<float*>(p.prev) + (size_t)s * 2 * B;
        for (int n = 4 * tid; n < B; n += 4 * T) {
            *reinterpret_cast<float4*>(hl + n) = *reinterpret_cast<const float4*>(xc + n);
            *reinterpret_cast<float4*>(hl + B + n) = *reinterpret_cast<const float4*>(xc + SM::kRingRowR + n);
        }
    }
    OHS_STAMP_IF(ft == 0, p, 7);
}

// which convolution warp (if any) the placement puts on hardware warp slot `warp`
template <int N, int G, int V, int... F>
__device__ __forceinline__ int find_conv_index(int warp, std::integer_sequence<int, F...>) {
    int r = -1;
    ((RenderSmem<N, G, V>::template kConvWarpId<F> == warp ? (void)(r = F) : (void)0), ...);
    return r;
}

// Moving: per-block HRIR sets with one-block crossfades (conv_warps_main<..., true>; DESIGN §10), instantiated
// separately and launched only for calls that need it, so that the static instantiations carry none of its code
template <int N, int G, int V = 0, bool Moving = false>
__global__ void __maxnreg__((RenderSmem<N, G, V>::kMaxRegs)) render_kernel(const RenderParams p) {
    using SM = RenderSmem<N, G, V>;
    extern __shared__ __align__(16) unsigned char smem[];
    const int stream0 = p.first_stream + blockIdx.x * G;
    OHS_STAMP(p, 0);
    launch_dependents();   // the next launch's CTAs may take this SM as soon as this CTA leaves it
    // No common prologue and no CTA-wide barrier: every role runs its own state-independent set-up first (the staging
    // warp initialises the mbarriers and starts the TMA copies of the constant tables, the EQ warps fetch their
    // coefficients), waits (griddepcontrol) for the previous launch only where it first touches what that launch wrote,
    // and the EQ and convolution warps wait on a named barrier for the staging warp's mbarrier initialisation.
    const int warp = threadIdx.x >> 5;
    if (warp < SM::kEqWarps) { eq_warp_main<N, G, V>(p, smem, stream0, warp); return; }
    if (warp == SM::kStagerWarpId) { stager_warp_main<N, G, V>(p, smem, stream0); return; }
    const int conv_index = find_conv_index<N, G, V>(warp, std::make_integer_sequence<int, SM::kConvWarps>{});
    if (conv_index >= 0) conv_warps_main<N, G, V, Moving>(p, smem, stream0, conv_index);  // other warp slots are placement padding
}

}  // namespace ohs
