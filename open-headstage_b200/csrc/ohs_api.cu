// ohs_api.cu — the C ABI of include/ohs.h over the kernels of ohs_kernels.cuh.
//
// Host-side state of one engine handle: the per-stream bindings (HRIR set, EQ set, gain), host copies of the
// impulse responses and EQ coefficients (uploaded lazily, on the next process call, so a burst of set_ir /
// update_band calls costs one upload — the reference recomputes all 20 biquads on every process() call,
// src/lib.rs:1180-1193), and the device-resident stream state: frequency-domain delay line, overlap-save block,
// biquad states.  No CPU fallback exists anywhere in this file: without a CUDA device ohs_create fails.
#include "../../include/ohs.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: the library itself is opened with dlopen by the first ohs_comm_* call

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "ohs_aux_kernels.cuh"
#include "ohs_launch.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define OHS_CUDA(expr)                                                                                          \
    do {                                                                                                        \
        cudaError_t _e = (expr);                                                                                \
        if (_e != cudaSuccess) return fail(OHS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                           __FILE__, __LINE__);                                                 \
    } while (0)

#define OHS_CHECK_HANDLE(h) \
    do { if (!(h)) return fail(OHS_ERR_INVALID, "null engine handle"); } while (0)

constexpr int kPipe = 3;  // staging buffers of the host-pointer path

}  // namespace

struct ohs_engine {
    ohs_config cfg{};
    int B = 0, N = 0, pmax = 1, G = 1;
    cudaStream_t stream = nullptr, h2d = nullptr, d2h = nullptr;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;
    bool timing = false, timed = false;   // ohs_enable_timing: event pair around the kernels of a process call

    // device
    int* d_stream_hrir = nullptr;
    int* d_stream_eq = nullptr;
    float* d_stream_gain = nullptr;
    float4* d_filt = nullptr;
    int* d_set_parts = nullptr;
    float2* d_fdl = nullptr;
    float2* d_prev = nullptr;
    float* d_eqc = nullptr;
    float4* d_eqs = nullptr;
    float2* d_tw = nullptr;
    float* d_ir = nullptr;
    int* d_set_list = nullptr;
    unsigned char* d_set_flags = nullptr;
    size_t filt_bytes = 0;

    // host mirrors
    std::vector<int> h_stream_hrir, h_stream_eq, h_set_parts, h_path_parts;
    std::vector<float> h_gain, h_eqc;
    std::vector<std::vector<float>> h_ir;  // [set*4 + path]
    std::vector<unsigned char> set_dirty, set_external;
    bool any_set_dirty = false, eqc_dirty = true, bind_dirty = true, gain_dirty = true;

    int head = 0;
    int eq_enable = 0, conv_enable = 1, bypass = 0;
    uint64_t launches = 0;
    // tuning switches, read from the environment ONCE at ohs_create (and settable through the API afterwards)
    int time_batch = 1;            // OHS_TIME_BATCH / ohs_set_time_batch: 0 keeps long responses on the block-by-block kernel
    size_t stage_bytes = (size_t)24 << 20;  // OHS_STAGE_MB: staging chunk of the host-pointer path
    bool dependent_launch = true;  // OHS_PDL=0 switches programmatic dependent launches off
    int latency_blocks = 2;        // OHS_LATENCY_BLOCKS: launches of up to this many blocks run the latency variant
    unsigned long long* d_trace = nullptr;  // ohs_debug_trace (OHS_TRACE builds)
    std::vector<float> h_ir_padded;         // [set][4][pmax*B] host mirror of d_ir, uploaded in one copy per commit

    // host-pointer path (grow-only buffers: *_cap is the bytes allocated per buffer, see grow_buffers)
    float* d_stage[kPipe] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_in[kPipe] = {}, ev_comp[kPipe] = {}, ev_out[kPipe] = {};
    size_t stage_cap = 0;
    // ... and its integer-PCM rows: the PCM rows of a chunk, both directions, beside d_stage
    unsigned char* d_pcm_stage[kPipe] = {nullptr, nullptr, nullptr};
    size_t pcm_stage_cap = 0;
    // ... and ohs_process_grouped_pcm's bus rows of a chunk (2 * n_groups rows), beside d_stage: f32 rows, or the packed PCM
    // rows of an integer bus (pitch round_up(n, 16) frames, never more bytes than the f32 rows of the same chunk)
    float* d_bus_stage[kPipe] = {nullptr, nullptr, nullptr};
    size_t bus_stage_cap = 0;
    // f32 rows of ohs_process_device_pcm's time chunks (decoded input, rendered in place)
    float* d_pcm_scratch = nullptr;
    size_t pcm_scratch_cap = 0;
    // dither of integer PCM output (ohs_set_dither): mode, seed and taps are configuration; the position (frames encoded
    // since ohs_set_dither) and the per-row error history are state, carried by the state blob
    int dither_mode = OHS_DITHER_OFF, dither_taps = 0;
    unsigned long long dither_seed = 0, dither_pos = 0;
    ohs::DitherTaps dither_h{};
    float* d_dither_hist = nullptr;   // [4 * n_streams][OHS_MAX_SHAPE_TAPS], allocated by ohs_set_dither: stream rows, then bus rows
    bool bus_hist_live = false;       // a bus has been encoded since ohs_set_dither, ohs_set_groups or a state import

    // listener buses (ohs_set_groups): group g holds streams h_group_first[g] .. h_group_first[g+1]-1; configuration like the
    // bindings, not state.  d_group_first is sized for n_streams groups.
    std::vector<int> h_group_first;
    int* d_group_first = nullptr;

    // time-batched long-response path: spectra in time order and frequency-domain products of one sub-launch
    float2* d_zlin = nullptr;
    float2* d_wlin = nullptr;
    size_t zlin_blocks = 0;  // blocks per sub-launch the two buffers are sized for
    // The time-ordered buffer is circular (zl_cap = pmax-1 + zlin_blocks slots per stream; zl_base = slot of the next
    // block) and carries the convolution history from one time-batched call to the next; the delay-line ring d_fdl is
    // what the block-by-block kernel and the state blob use.  At least one of the two is current at any time; they are
    // converted into each other (gather / scatter, a copy of pmax-1 spectra per stream) only when the route changes.
    int zl_base = 0, zl_cap = 0;
    bool zlin_valid = false, ring_valid = true;
    // ... and its EQ pre-pass: the EQ-filtered rows of two sub-launches (halves used alternately), written by the EQ-only
    // kernel on its own stream while the previous chunk's transforms and products run on the engine's stream
    float* d_xf = nullptr;   // [2 halves][stream][2][zlin_blocks * B]
    cudaStream_t eq_stream = nullptr;
    std::vector<cudaEvent_t> ev_eq;          // EQ pre-pass of chunk c has finished (pool, used round-robin)
    cudaEvent_t ev_fwd[2] = {nullptr, nullptr};   // forward transforms have consumed a half of d_xf
    cudaEvent_t ev_call = nullptr;           // everything enqueued on the engine's stream before this call
    size_t eq_events_used = 0;

    // FIFO adaptor (src/dsp/convolution.rs:141-182)
    std::vector<float> fifo_in, fifo_out;  // [row][cap]
    size_t fifo_cap = 0, fifo_in_len = 0, fifo_out_len = 0;

    // moving sources (DESIGN §10): ohs_move_stream_hrir targets (-1: none) applied by the next convolving block, the
    // bindings they replace (the kernel's from_set) and ohs_process_device_scheduled's per-block sets
    std::vector<int> h_move_to, h_from_set;
    bool any_move = false;
    int* d_from_set = nullptr;
    int* d_sched = nullptr;
    size_t sched_cap = 0;   // bytes
};

namespace {

using namespace ohs;

// moving: the moving-sources kernel, render_kernel<..., true> (p.from_set set, p.block_set optional)
int launch_render(ohs_engine* h, const RenderParams& p, int first_stream = 0, bool moving = false) {
    // few blocks per launch: nothing overlaps inside the launch, so the variant built for latency runs it
    const bool latency = p.n_blocks <= h->latency_blocks;
    RenderLaunch L{h->G, h->cfg.device, h->stream, first_stream, latency ? 1 : 0, 0, h->dependent_launch, moving};
    RenderParams q = p;
    q.trace = h->d_trace;
    const cudaError_t e = with_transform_size(h->N, cudaErrorInvalidValue, [&](auto n) { return render_launch<n>(L, q); });
    if (e == cudaErrorInvalidConfiguration) { cudaGetLastError(); return fail(OHS_ERR_INVALID, "%d streams per CTA do not fit for block %d", h->G, h->B); }
    if (e != cudaSuccess) return fail(OHS_ERR_CUDA, "render kernel launch failed: %s", cudaGetErrorString(e));
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

template <int N> int launch_setup_n(ohs_engine* h, int max_parts, int n_sets) {
    using SM = SetupSmem<N>;
    static OncePerDevice attrs;
    OHS_CUDA(attrs.run(h->cfg.device, [] {
        return cudaFuncSetAttribute(setup_filters_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM::kBytes);
    }));
    dim3 grid(max_parts, n_sets);
    setup_filters_kernel<N><<<grid, SM::T, SM::kBytes, h->stream>>>(h->d_ir, h->d_filt, h->d_tw, h->d_set_list, h->d_set_parts, h->pmax);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// the delay-line ring brought up to date from the time-ordered buffer (after time-batched calls), before anything reads
// or partially rewrites it
int ensure_ring(ohs_engine* h) {
    if (h->ring_valid) return OHS_OK;
    if (h->pmax > 1 && h->d_zlin) {
        scatter_history_kernel<<<dim3((unsigned)(h->pmax - 1), (unsigned)h->cfg.n_streams), 256, 0, h->stream>>>(
            h->d_zlin, h->d_fdl, h->N, h->pmax, h->head, (long long)h->zl_cap * h->N, h->zl_base, h->zl_cap);
        OHS_CUDA(cudaGetLastError());
        h->launches++;
    }
    h->ring_valid = true;
    return OHS_OK;
}

int clear_history(ohs_engine* h, bool only_flagged) {
    if (only_flagged) { const int rc = ensure_ring(h); if (rc) return rc; }
    h->ring_valid = true; h->zlin_valid = false;   // the cleared ring is the current history from here on
    clear_history_kernel<<<h->cfg.n_streams, 256, 0, h->stream>>>(h->d_fdl, h->d_prev, h->d_stream_hrir, h->cfg.n_streams,
                                                                 only_flagged ? h->d_set_flags : nullptr,
                                                                 (size_t)h->pmax * h->N, (size_t)h->B);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

int upload_bindings(ohs_engine* h) {
    if (h->bind_dirty) {
        OHS_CUDA(cudaMemcpyAsync(h->d_stream_hrir, h->h_stream_hrir.data(), sizeof(int) * h->cfg.n_streams, cudaMemcpyHostToDevice, h->stream));
        OHS_CUDA(cudaMemcpyAsync(h->d_stream_eq, h->h_stream_eq.data(), sizeof(int) * h->cfg.n_streams, cudaMemcpyHostToDevice, h->stream));
        h->bind_dirty = false;
    }
    if (h->gain_dirty) {
        OHS_CUDA(cudaMemcpyAsync(h->d_stream_gain, h->h_gain.data(), sizeof(float) * h->cfg.n_streams, cudaMemcpyHostToDevice, h->stream));
        h->gain_dirty = false;
    }
    if (h->eqc_dirty) {
        OHS_CUDA(cudaMemcpyAsync(h->d_eqc, h->h_eqc.data(), sizeof(float) * h->h_eqc.size(), cudaMemcpyHostToDevice, h->stream));
        h->eqc_dirty = false;
    }
    // pageable host sources: the async copies above are staged by the runtime before returning
    return OHS_OK;
}

int commit_filters(ohs_engine* h) {
    int rc = upload_bindings(h);
    if (rc) return rc;
    if (!h->any_set_dirty) return OHS_OK;
    // every dirty set's taps go into the host mirror, ONE copy uploads the span of dirty sets and ONE launch transforms
    // them (config 4 binds a set per stream: thousands of sets per commit)
    const int n_sets = h->cfg.n_hrir_sets;
    const size_t per_path = (size_t)h->pmax * h->B, per_set = 4 * per_path;
    if (h->h_ir_padded.size() != per_set * n_sets) h->h_ir_padded.assign(per_set * n_sets, 0.f);
    std::vector<int> list;
    int max_parts = 1, lo = n_sets, hi = -1;
    for (int s = 0; s < n_sets; ++s) {
        if (!h->set_dirty[s]) continue;
        float* dst = h->h_ir_padded.data() + (size_t)s * per_set;
        std::fill(dst, dst + per_set, 0.f);
        int parts = 1;
        for (int p = 0; p < 4; ++p) {
            const std::vector<float>& ir = h->h_ir[(size_t)s * 4 + p];
            std::copy(ir.begin(), ir.end(), dst + p * per_path);
            parts = std::max(parts, h->h_path_parts[(size_t)s * 4 + p]);
        }
        h->h_set_parts[s] = parts;
        max_parts = std::max(max_parts, parts);
        lo = std::min(lo, s); hi = std::max(hi, s);
        list.push_back(s);
    }
    OHS_CUDA(cudaMemcpyAsync(h->d_ir + (size_t)lo * per_set, h->h_ir_padded.data() + (size_t)lo * per_set,
                             sizeof(float) * per_set * (size_t)(hi - lo + 1), cudaMemcpyHostToDevice, h->stream));
    OHS_CUDA(cudaMemcpyAsync(h->d_set_parts, h->h_set_parts.data(), sizeof(int) * n_sets, cudaMemcpyHostToDevice, h->stream));
    OHS_CUDA(cudaMemcpyAsync(h->d_set_list, list.data(), sizeof(int) * list.size(), cudaMemcpyHostToDevice, h->stream));
    OHS_CUDA(cudaMemcpyAsync(h->d_set_flags, h->set_dirty.data(), n_sets, cudaMemcpyHostToDevice, h->stream));
    OHS_CUDA(cudaStreamSynchronize(h->stream));  // pageable sources (`list` is a local) must be consumed before returning
    rc = with_transform_size(h->N, (int)OHS_ERR_INVALID, [&](auto n) { return launch_setup_n<n>(h, max_parts, (int)list.size()); });
    if (rc) return rc;
    // set_ir clears the history of the streams that use the set (src/dsp/convolution.rs:135-138)
    rc = clear_history(h, true);
    if (rc) return rc;
    std::fill(h->set_dirty.begin(), h->set_dirty.end(), 0);
    h->any_set_dirty = false;
    return OHS_OK;
}

// biquad 0.4.2 Coefficients::<f32>::from_params, f32 arithmetic and libm like the crate (src/dsp/parametric_eq.rs:105-111)
int eq_design_impl(int type, float fs, float fc, float q, float gain_db, float out[5]) {
    if (2.0f * fc > fs) return fail(OHS_ERR_NYQUIST, "EQ design: 2*fc (%g) > fs (%g)", 2.0 * fc, (double)fs);
    if (q < 0.0f) return fail(OHS_ERR_NEGATIVE_Q, "EQ design: negative Q %g", (double)q);
    const float pi = 3.14159265358979323846f;
    const float omega = 2.0f * pi * fc / fs;
    const float sn = sinf(omega), cs = cosf(omega);
    const float alpha = sn / (2.0f * q);
    float b0, b1, b2, a0, a1, a2;
    bool divide = false;
    if (type == OHS_FILTER_PEAK || type == OHS_FILTER_LOWSHELF || type == OHS_FILTER_HIGHSHELF) {
        const float a = powf(10.0f, gain_db / 40.0f);
        divide = true;
        if (type == OHS_FILTER_PEAK) {
            b0 = 1.0f + alpha * a; b1 = -2.0f * cs; b2 = 1.0f - alpha * a;
            a0 = 1.0f + alpha / a; a1 = -2.0f * cs; a2 = 1.0f - alpha / a;
        } else {
            const float beta = 2.0f * alpha * sqrtf(a);
            const float ap = a + 1.0f, am = a - 1.0f;
            if (type == OHS_FILTER_LOWSHELF) {
                b0 = a * (ap - am * cs + beta); b1 = 2.0f * a * (am - ap * cs); b2 = a * (ap - am * cs - beta);
                a0 = ap + am * cs + beta; a1 = -2.0f * (am + ap * cs); a2 = ap + am * cs - beta;
            } else {
                b0 = a * (ap + am * cs + beta); b1 = -2.0f * a * (am + ap * cs); b2 = a * (ap + am * cs - beta);
                a0 = ap - am * cs + beta; a1 = 2.0f * (am - ap * cs); a2 = ap - am * cs - beta;
            }
        }
    } else {
        a0 = 1.0f + alpha; a1 = -2.0f * cs; a2 = 1.0f - alpha;
        switch (type) {
            case OHS_FILTER_LOWPASS: b0 = (1.0f - cs) * 0.5f; b1 = 1.0f - cs; b2 = (1.0f - cs) * 0.5f; break;
            case OHS_FILTER_HIGHPASS: b0 = (1.0f + cs) * 0.5f; b1 = -(1.0f + cs); b2 = (1.0f + cs) * 0.5f; break;
            case OHS_FILTER_BANDPASS: b0 = sn / 2.0f; b1 = 0.0f; b2 = -(sn / 2.0f); break;
            case OHS_FILTER_NOTCH: b0 = 1.0f; b1 = -2.0f * cs; b2 = 1.0f; break;
            case OHS_FILTER_ALLPASS: b0 = 1.0f - alpha; b1 = -2.0f * cs; b2 = 1.0f + alpha; break;
            default: return fail(OHS_ERR_INVALID, "unknown filter type %d", type);
        }
    }
    if (divide) {
        out[0] = b0 / a0; out[1] = b1 / a0; out[2] = b2 / a0; out[3] = a1 / a0; out[4] = a2 / a0;
    } else {
        const float inv = 1.0f / a0;
        out[0] = b0 * inv; out[1] = b1 * inv; out[2] = b2 * inv; out[3] = a1 * inv; out[4] = a2 * inv;
    }
    return OHS_OK;
}

int set_band_host(ohs_engine* h, int eq_set, int band, const float c[5], int enabled) {
    if (eq_set < 0 || eq_set >= h->cfg.n_eq_sets) return fail(OHS_ERR_INVALID, "eq_set %d out of range", eq_set);
    if (band < 0 || band >= h->cfg.n_bands) return OHS_OK;  // silently ignored, src/dsp/parametric_eq.rs:145
    float* dst = h->h_eqc.data() + ((size_t)eq_set * kMaxBands + band) * kEqCoefStride;
    for (int i = 0; i < 5; ++i) dst[i] = c[i];
    dst[5] = enabled ? 1.0f : 0.0f;
    h->eqc_dirty = true;
    return OHS_OK;
}

size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

// Frames per chunk of a call of n_frames: about budget_bytes of rows at bytes_per_sample, whole blocks, at least one
// block.  The cap (the call rounded up to 16 frames) only sizes allocations: callers take min(chunk, frames left), so the
// chunk boundaries are those of the uncapped rule.  The cap keeps every row pitch, round_up(n, 4) of f32 rows and
// round_up(n, 16) of PCM rows, within an allocation of chunk frames (a block is a multiple of 16 frames).
size_t chunk_frames(const ohs_engine* h, size_t n_frames, size_t budget_bytes, size_t bytes_per_sample) {
    const size_t rows = (size_t)h->cfg.n_streams * 2;
    const size_t chunk = std::max<size_t>(h->B, budget_bytes / (rows * bytes_per_sample) / h->B * h->B);
    return std::min(chunk, round_up(n_frames, 16));
}

// Grows the n buffers bufs[0..n) to `bytes` each unless `cap` (the bytes each holds) is enough already.  Work enqueued
// earlier may still use the old buffers, hence the syncs.  `cap` is 0 from the first free until every allocation has
// succeeded, so after a failed cudaMalloc the next call allocates again rather than use a freed or null buffer.
template <typename T> int grow_buffers(ohs_engine* h, T** bufs, int n, size_t& cap, size_t bytes) {
    if (bytes <= cap) return OHS_OK;
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    OHS_CUDA(cudaStreamSynchronize(h->d2h));
    cap = 0;
    for (int i = 0; i < n; ++i) {
        if (bufs[i]) OHS_CUDA(cudaFree(bufs[i]));
        bufs[i] = nullptr;
        OHS_CUDA(cudaMalloc(&bufs[i], bytes));
    }
    cap = bytes;
    return OHS_OK;
}

// ---- audio I/O: the sides of a call, their argument rules, and the PCM conversions ---------------------------------
static_assert((int)kPcmF32 == OHS_FMT_F32 && (int)kPcmS16 == OHS_FMT_S16 && (int)kPcmS24 == OHS_FMT_S24, "PcmFormat is OHS_FMT_*");
static_assert(kShapeTaps == OHS_MAX_SHAPE_TAPS, "history rows of the shaped encode");

// f(std::integral_constant<int, Fmt>{}) for the runtime sample format fmt; `otherwise` for an unknown format
template <typename R, typename F> R with_pcm_format(int fmt, R otherwise, F&& f) {
    switch (fmt) {
        case OHS_FMT_F32: return f(std::integral_constant<int, kPcmF32>{});
        case OHS_FMT_S16: return f(std::integral_constant<int, kPcmS16>{});
        case OHS_FMT_S24: return f(std::integral_constant<int, kPcmS24>{});
    }
    return otherwise;
}

int n_groups(const ohs_engine* h) { return (int)h->h_group_first.size() - 1; }

// One side of an audio call, or of a chunk's work in HBM: rows of `fmt` samples from p on, `stride` frames apart; the
// 2 * n_groups bus rows with `bus`, else the 2 * n_streams stream rows.  An input side is only read.
struct Rows {
    void* p;
    int fmt;
    size_t stride;
    bool bus = false;
    // 0 for an unknown format
    size_t sample_bytes() const { return with_pcm_format(fmt, (size_t)0, [](auto f) { return (size_t)PcmTraits<f>::kBytes; }); }
    // frames in whole 16-byte units of the format: rows start 16-byte aligned when the stride is a multiple
    size_t align_frames() const { return with_pcm_format(fmt, (size_t)0, [](auto f) { return (size_t)PcmTraits<f>::kGroup; }); }
    size_t count(const ohs_engine* h) const { return bus ? (size_t)2 * n_groups(h) : (size_t)h->cfg.n_streams * 2; }
    Rows from(size_t f0) const { return {static_cast<unsigned char*>(p) + f0 * sample_bytes(), fmt, stride, bus}; }
};

// What an audio entry point asks of its arguments beyond known formats, non-null pointers and strides >= n_frames
enum CallRule : unsigned {
    kWholeBlocks = 1,          // a render: n_frames a multiple of the engine block while the convolution is on
    kSeparate = 2,             // the output (a bus) overlaps no byte of the input, whatever the formats and layouts
    kSeparateIfConverted = 4,  // when the formats differ, the output neither is nor overlaps the input: in place needs equal formats
    kDeviceRows = 8,           // 16-byte aligned pointers, and each stride a multiple of its format's align_frames()
    kWholeQuads = 16,          // with kDeviceRows: n_frames a multiple of 4 (the mixdown)
};

// The argument check of every audio entry point, before anything is enqueued, so a rejected call leaves the engine
// untouched.  A call with several faults gets the code of the first in this order.
int check_call(const ohs_engine* h, const Rows& in, const Rows& out, size_t n_frames, unsigned rules) {
    for (const Rows* r : {&in, &out})
        if (!r->sample_bytes()) return fail(OHS_ERR_INVALID, "unknown sample format %d", r->fmt);
    if (!in.p || !out.p) return fail(OHS_ERR_INVALID, "null audio pointer");
    if ((rules & kWholeBlocks) && h->conv_enable && n_frames % (size_t)h->B)
        return fail(OHS_ERR_INVALID, "n_frames %zu is not a multiple of the engine block %d (use ohs_process_fifo)", n_frames, h->B);
    for (const Rows* r : {&in, &out})
        if (r->stride < n_frames) return fail(OHS_ERR_INVALID, "%s %zu < n_frames %zu", r->bus ? "bus_stride" : "row_stride", r->stride, n_frames);
    // the decode or copy-in of a later chunk must not read what the encode or copy-out of an earlier one has written
    const bool converted = (rules & kSeparateIfConverted) && in.fmt != out.fmt;
    if ((rules & kSeparate) || converted) {
        const uintptr_t a = (uintptr_t)in.p, b = (uintptr_t)out.p;
        const size_t na = ((in.count(h) - 1) * in.stride + n_frames) * in.sample_bytes();
        const size_t nb = ((out.count(h) - 1) * out.stride + n_frames) * out.sample_bytes();
        if ((converted && a == b) || (a < b + nb && b < a + na))
            return fail(OHS_ERR_INVALID, out.bus ? "the bus overlaps the input" : "input and output overlap; in place needs equal sample formats");
    }
    if ((rules & kDeviceRows) && ((((uintptr_t)in.p | (uintptr_t)out.p) & 15u) || in.stride % in.align_frames() ||
                                  out.stride % out.align_frames() || ((rules & kWholeQuads) && n_frames % 4)))
        return fail(OHS_ERR_ALIGNMENT, "device audio needs 16-byte aligned pointers and strides that are multiples of 4 / 8 / 16 frames "
                                       "(F32 / S16 / S24)%s", (rules & kWholeQuads) ? ", and n_frames a multiple of 4" : "");
    return OHS_OK;
}

// Grid of the decode and flat-encode kernels over `rows` rows of n frames: one thread per group of PcmTraits<Fmt>::kGroup
// frames of a row, at most 2^20 CTAs of 256 (the kernels stride over the rest)
template <int Fmt> struct GroupGrid {
    size_t groups, total;
    unsigned blocks;
    GroupGrid(size_t rows, size_t n) : groups((n + PcmTraits<Fmt>::kGroup - 1) / PcmTraits<Fmt>::kGroup), total(rows * groups),
                                       blocks((unsigned)std::min<size_t>((total + 255) / 256, (size_t)1 << 20)) {}
};

// the PCM stream rows `pcm` decoded into the f32 rows x (pitch p floats) on the engine's stream
template <int Fmt> int launch_decode(ohs_engine* h, const Rows& pcm, float* x, size_t p, size_t n_frames) {
    const GroupGrid<Fmt> g((size_t)h->cfg.n_streams * 2, n_frames);
    pcm_decode_kernel<Fmt><<<g.blocks, 256, 0, h->stream>>>(static_cast<const unsigned char*>(pcm.p), pcm.stride * PcmTraits<Fmt>::kBytes,
                                                            x, p, n_frames, g.groups, g.total);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// pcm_encode_shaped_kernel<Fmt, M, Mix> for the runtime tap count m (1..OHS_MAX_SHAPE_TAPS)
template <int Fmt, bool Mix, int M = 1>
void launch_encode_shaped(int m, cudaStream_t st, const float* f32, size_t f32_pitch, unsigned char* pcm, size_t pcm_pitch,
                          size_t n_frames, int rows, unsigned long long seed, unsigned long long pos, const DitherTaps& taps,
                          float* hist, const int* group_first) {
    if constexpr (M <= kShapeTaps) {
        if (m != M)
            return launch_encode_shaped<Fmt, Mix, M + 1>(m, st, f32, f32_pitch, pcm, pcm_pitch, n_frames, rows, seed, pos, taps, hist,
                                                         group_first);
        pcm_encode_shaped_kernel<Fmt, M, Mix><<<(rows + kShapeRows - 1) / kShapeRows, kShapeThreads, 0, st>>>(
            f32, f32_pitch, pcm, pcm_pitch, n_frames, rows, seed, pos, taps, hist, group_first);
    }
}

// the bus rows' error history: behind the 2 * n_streams stream rows, room for 2 * n_streams bus rows
float* bus_hist(const ohs_engine* h) { return h->d_dither_hist + (size_t)h->cfg.n_streams * 2 * kShapeTaps; }
size_t bus_hist_bytes(const ohs_engine* h) { return sizeof(float) * (size_t)h->cfg.n_streams * 2 * kShapeTaps; }

// The encode of the f32 stream rows x (pitch p floats) into the PCM rows `pcm` on the engine's stream, dithered as
// ohs_set_dither says, its first frame at dither position pos.  Mix: `pcm` is the 2 * n_groups bus rows, each the sum of
// its group's stream rows of x (pcm_encode_kernel / pcm_encode_shaped_kernel with Mix): dither row numbers from
// 2 * n_streams on, i.e. the key hash with the seed seed + phi * 2S, and the error history behind the streams' rows.
template <int Fmt, bool Mix>
int launch_encode(ohs_engine* h, const Rows& pcm, const float* x, size_t p, size_t n_frames, unsigned long long pos) {
    const size_t S2 = (size_t)h->cfg.n_streams * 2, rows = Mix ? (size_t)2 * n_groups(h) : S2;
    const GroupGrid<Fmt> g(rows, n_frames);
    unsigned char* q = static_cast<unsigned char*>(pcm.p);
    const size_t q_pitch = pcm.stride * PcmTraits<Fmt>::kBytes;
    const unsigned long long seed = h->dither_seed + (Mix ? kDitherPhi * S2 : 0ull);
    float* hist = h->d_dither_hist ? h->d_dither_hist + (Mix ? S2 * kShapeTaps : 0) : nullptr;
    const int* gf = Mix ? h->d_group_first : nullptr;
    if (h->dither_mode == OHS_DITHER_TPDF && h->dither_taps > 0)
        launch_encode_shaped<Fmt, Mix>(h->dither_taps, h->stream, x, p, q, q_pitch, n_frames, (int)rows, seed, pos, h->dither_h, hist, gf);
    else if (h->dither_mode == OHS_DITHER_TPDF)
        pcm_encode_kernel<Fmt, true, Mix><<<g.blocks, 256, 0, h->stream>>>(x, p, q, q_pitch, n_frames, g.groups, g.total, seed, pos, gf);
    else
        pcm_encode_kernel<Fmt, false, Mix><<<g.blocks, 256, 0, h->stream>>>(x, p, q, q_pitch, n_frames, g.groups, g.total, 0, 0, gf);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    if (Mix) h->bus_hist_live = true;
    return OHS_OK;
}

// The group buses of f32 rows on the engine's stream: 2 * n_groups rows of `bus` (ohs_mix_device, ohs_process_grouped).
// A plain launch, without the programmatic-serialization attribute: it starts once the render before it has finished.
int launch_mix(ohs_engine* h, const float* in, size_t row_stride, float* bus, size_t bus_stride, size_t n_frames) {
    const unsigned threads = 256;
    const int rows = 2 * n_groups(h);
    const dim3 grid((unsigned)(((n_frames + 3) / 4 + threads - 1) / threads), (unsigned)std::min(rows, 65535));
    mix_streams_kernel<<<grid, threads, 0, h->stream>>>(in, bus, h->d_group_first, rows, n_frames, row_stride, bus_stride);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// f32 scratch rows of ohs_process_device_pcm: whole blocks, at most 256 MiB (longer calls go through it in time chunks)
constexpr size_t kPcmScratchBytes = (size_t)256 << 20;
int ensure_pcm_scratch(ohs_engine* h, size_t frames) {
    return grow_buffers(h, &h->d_pcm_scratch, 1, h->pcm_scratch_cap, (size_t)h->cfg.n_streams * 2 * frames * sizeof(float));
}

// called once, from ohs_create (the only place the environment is consulted)
int pick_streams_per_cta(const ohs_engine* h) {
    auto fits = [h](int g) { return with_transform_size(h->N, false, [g](auto n) { return render_fits<n>(g); }); };
    if (const char* e = getenv("OHS_STREAMS_PER_CTA")) {
        const int g = atoi(e);
        if (g >= 1 && g <= kMaxG && fits(g)) return g;
    }
    cudaDeviceProp prop{};
    int sms = 148;
    if (cudaGetDeviceProperties(&prop, h->cfg.device) == cudaSuccess) sms = prop.multiProcessorCount;
    // Few streams per SM (config 2: 1024 streams -> 7 per CTA, 147 CTAs): one CTA per SM holding ceil(n_streams / SMs)
    // streams, so every SM gets the same share.  Many streams per SM (config 3: 55 per SM): CTAs of three streams, whose
    // six chains exactly fill one EQ warp, several CTAs resident per SM (measured best on config 3).
    int g = (h->cfg.n_streams + sms - 1) / sms;
    g = (g > kMaxG) ? 3 : std::max(1, g);
    while (g > 1 && !fits(g)) --g;
    return g;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
namespace {

constexpr int kTimeBatch = 8;  // consecutive blocks a bin_conv_kernel thread accumulates (TB)

template <int N> int launch_inverse(ohs_engine* h, const float2* d_w, float* d_out, int K, size_t row_stride) {
    constexpr size_t smem = sizeof(float2) * 2 * padded_len(N);
    static OncePerDevice attrs;
    if (smem > 48 * 1024)
        OHS_CUDA(attrs.run(h->cfg.device, [] { return cudaFuncSetAttribute(inverse_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); }));
    inverse_kernel<N><<<dim3(K, h->cfg.n_streams), SetupSmem<N>::TX, smem, h->stream>>>(d_w, d_out, h->d_tw, h->d_stream_gain, K,
                                                                                      (long long)row_stride);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// forward transforms of blocks [t0, t0 + k) of a sub-launch from the filtered rows xf (block 0's history: d_prev)
template <int N> int launch_forward(ohs_engine* h, const float* xf, long long xf_stride, int t0, int k, long long zstride, int zbase) {
    // zbase: the time-ordered buffer's slot of the sub-launch's block 0
    constexpr size_t smem = sizeof(float2) * 2 * padded_len(N);
    static OncePerDevice attrs;
    if (smem > 48 * 1024)
        OHS_CUDA(attrs.run(h->cfg.device, [] { return cudaFuncSetAttribute(forward_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); }));
    forward_kernel<N><<<dim3(k, h->cfg.n_streams), SetupSmem<N>::TX, smem, h->stream>>>(
        xf, xf_stride, t0, reinterpret_cast<const float*>(h->d_prev), h->d_zlin, zstride, zbase, h->zl_cap, h->d_tw);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// Long responses, many blocks per call (SURVEY 8f).  Per sub-launch of up to `zlin_blocks` blocks:
//   (0) EQ pre-pass: the EQ-only variant of the render kernel (a thin CTA per three streams: two EQ warps, 38 KB) filters
//       the input rows into d_xf on its OWN stream.  The biquad chain is strictly sequential — 1024 steps per block at
//       the chain's latency, with most of the SM idle — while everything below is throughput-bound and independent of
//       later input, so the pre-pass of chunk c+1 runs beside the transforms and products of chunk c;
//   (1) delay-line history into the time-ordered buffer (once per sub-launch);
//   and per chunk (8, 8, 16, 32 blocks in a call's first sub-launch, so that only the first 8 blocks' EQ is exposed; the
//   whole sub-launch afterwards, when the pre-pass is running ahead anyway):
//   (2) forward transforms (spectra to the ring and to the time-ordered buffer), (3) the per-bin convolution along time,
//   (4) the inverse transforms.
// The delay-line ring, the overlap-save block and the EQ state end up exactly where the block-by-block path leaves
// them, so the two can be mixed freely between calls.

// Blocks per sub-launch a call of n_blocks needs on the time-batched route: as many as the 2 GiB budget holds, at most
// 64 and at most n_blocks.  0: the call runs the block-by-block kernel (the route is off or does not apply, or fewer
// than kTimeBatch blocks fit the budget).  Decided before anything is enqueued.
size_t time_batch_blocks(const ohs_engine* h, int n_blocks) {
    if (!h->time_batch || !h->conv_enable || h->pmax < 8 || n_blocks < kTimeBatch || h->cfg.n_streams > 65535)   // (grid.y = stream)
        return 0;
    const size_t S = (size_t)h->cfg.n_streams, N = (size_t)h->N, hist = (size_t)h->pmax - 1;
    const size_t budget = (size_t)2 << 30;
    // per block: a spectrum and a product (8N bytes each) and the filtered rows in both halves of d_xf (2 * 2 * 4B = 8N)
    const size_t per_block = 3 * S * N * sizeof(float2), fixed = S * hist * N * sizeof(float2);
    size_t kc = fixed < budget ? (budget - fixed) / per_block : 0;
    kc = std::min<size_t>(std::min<size_t>(kc, 64), (size_t)n_blocks);
    return kc < (size_t)kTimeBatch ? 0 : kc;
}

// Scratch of the time-batched route for sub-launches of kc = time_batch_blocks(...) blocks, grow-only (ohs_prepare
// calls this ahead of time so that no allocation happens inside a timed call)
int ensure_time_batch_scratch(ohs_engine* h, size_t kc) {
    const size_t S = (size_t)h->cfg.n_streams, N = (size_t)h->N, hist = (size_t)h->pmax - 1;
    if (kc > h->zlin_blocks) {
        { const int rc = ensure_ring(h); if (rc) return rc; }   // the history moves to the ring before its buffer goes
        h->zlin_valid = false;
        OHS_CUDA(cudaStreamSynchronize(h->stream));
        if (h->eq_stream) OHS_CUDA(cudaStreamSynchronize(h->eq_stream));
        if (h->d_zlin) OHS_CUDA(cudaFree(h->d_zlin));
        if (h->d_wlin) OHS_CUDA(cudaFree(h->d_wlin));
        if (h->d_xf) OHS_CUDA(cudaFree(h->d_xf));
        h->d_zlin = h->d_wlin = nullptr; h->d_xf = nullptr; h->zlin_blocks = 0;
        OHS_CUDA(cudaMalloc(&h->d_zlin, S * (hist + kc) * N * sizeof(float2)));
        OHS_CUDA(cudaMalloc(&h->d_wlin, S * kc * N * sizeof(float2)));
        OHS_CUDA(cudaMalloc(&h->d_xf, 2 * S * 2 * kc * (size_t)h->B * sizeof(float)));
        h->zlin_blocks = kc;
        h->zl_cap = (int)(hist + kc); h->zl_base = (int)hist;
    }
    if (!h->eq_stream) {
        int lo = 0, hi = 0;
        OHS_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        OHS_CUDA(cudaStreamCreateWithPriority(&h->eq_stream, cudaStreamNonBlocking, hi));   // its thin CTAs go first
        OHS_CUDA(cudaEventCreateWithFlags(&h->ev_fwd[0], cudaEventDisableTiming));
        OHS_CUDA(cudaEventCreateWithFlags(&h->ev_fwd[1], cudaEventDisableTiming));
        OHS_CUDA(cudaEventCreateWithFlags(&h->ev_call, cudaEventDisableTiming));
    }
    return OHS_OK;
}

// the per-bin convolution of the k blocks from slot zslot0 of the circular time-ordered buffer on, products to `w`
// ([stream][k][N])
int launch_bin_conv(ohs_engine* h, int zslot0, float2* w, int k, long long zstride) {
    const size_t S = (size_t)h->cfg.n_streams, N = (size_t)h->N;
    const dim3 blk(128);
    const unsigned gx = (unsigned)((N / 2 + 31) / 32), gz = (unsigned)((S + 3) / 4);
    static OncePerDevice attrs;
    OHS_CUDA(attrs.run(h->cfg.device, [] {
        return cudaFuncSetAttribute(bin_conv_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * 16 * 128 * sizeof(float4)));
    }));
    // 16 blocks per thread (half the spectrum and filter traffic per FMA) from 16 blocks per launch on: measured faster
    // than 8 at K = 16 (0.529 vs 0.560 ms), 32, 64 and 128 on config 5
    if (k >= 16)
        bin_conv_kernel<16><<<dim3(gx, (unsigned)((k + 15) / 16), gz), blk, 2 * 16 * 128 * sizeof(float4), h->stream>>>(
            h->d_zlin, w, h->d_filt, h->d_stream_hrir, h->d_set_parts, (int)N, h->pmax, k, (int)S, zstride, zslot0, h->zl_cap);
    else
        bin_conv_kernel<kTimeBatch><<<dim3(gx, (unsigned)((k + kTimeBatch - 1) / kTimeBatch), gz), blk, 2 * kTimeBatch * 128 * sizeof(float4), h->stream>>>(
            h->d_zlin, w, h->d_filt, h->d_stream_hrir, h->d_set_parts, (int)N, h->pmax, k, (int)S, zstride, zslot0, h->zl_cap);
    OHS_CUDA(cudaGetLastError());
    h->launches++;
    return OHS_OK;
}

// EQ pre-pass of `frames` frames of every stream on the EQ stream: rows in (stride in_stride) -> rows out (stride out_stride)
int launch_eq_prepass(ohs_engine* h, const RenderParams& base, const float* d_in, long long in_stride, float* d_out, long long out_stride,
                      size_t frames) {
    constexpr int kB = 256;   // the EQ-only variant exists for N = 512; the chain does not care how its rows are cut into blocks
    RenderParams q = base;
    q.in = d_in; q.out = d_out; q.row_stride = in_stride; q.out_row_stride = out_stride;
    q.n_blocks = (int)((frames + kB - 1) / kB);
    q.tail_frames = (int)(frames - (size_t)(q.n_blocks - 1) * kB);
    q.conv_enable = 0; q.eq_enable = 1; q.filt_in_smem = 0;
    q.trace = nullptr;
    // Shape of the pre-pass (RenderSmem, V = 2).  Many streams, run beside the previous chunk's kernels: six per CTA — four
    // EQ warps, one per scheduler partition — and 200 KB of shared memory asked for, so that each CTA OWNS its SM: next to
    // the per-bin kernel's FMA-saturated warps every instruction of the biquad chain waits for its issue slot and the
    // chain, the route's critical path, runs 2.5x slower (measured; config 5 at 256 blocks per call: 4.95 ms with 43 SMs
    // owned, 5.65 ms with thin CTAs of three streams sharing 86 SMs, 5.82 ms with twelve streams = two EQ warps per
    // partition on 22 SMs).  Fewer than twelve streams: thin CTAs of three.
    const bool own_sm = h->cfg.n_streams >= 12;
    // no programmatic dependent launch here: the next chunk's CTAs, started early, would sit on SMs of their own (they
    // cannot share one with this chunk's) and take them from the transforms of the chunk before
    RenderLaunch L{own_sm ? 6 : 3, h->cfg.device, h->eq_stream, 0, 2, own_sm ? (size_t)200 << 10 : 0, false};
    const cudaError_t e = render_launch<512>(L, q);
    if (e != cudaSuccess) return fail(OHS_ERR_CUDA, "EQ pre-pass launch failed: %s", cudaGetErrorString(e));
    h->launches++;
    return OHS_OK;
}

// the time-batched route for a call that needs sub-launches of `fit` = time_batch_blocks(h, p.n_blocks) blocks
int process_time_batched(ohs_engine* h, RenderParams p, size_t fit, const float* d_in, float* d_out, size_t row_stride) {
    const size_t S = (size_t)h->cfg.n_streams, N = (size_t)h->N, hist = (size_t)h->pmax - 1, B = (size_t)h->B;
    { const int rc = ensure_time_batch_scratch(h, fit); if (rc) return rc; }
    // sub-launches as long as the scratch allows: after a longer call, more than this call's own fit
    const size_t kc = h->zlin_blocks;
    const long long zstride = (long long)((hist + kc) * N);
    const long long xstride = (long long)(kc * B);               // frames between the rows of a half of d_xf
    const size_t xhalf = S * 2 * kc * B;                         // floats per half
    const int total = p.n_blocks;
    const bool eq_on = p.eq_enable != 0;
    const int n_sub = (total + (int)kc - 1) / (int)kc;
    // chunks of sub-launch j: (first block inside the sub-launch, blocks).  The EQ pre-pass of a chunk runs beside the
    // transforms of the chunk before it, so what a call cannot hide is the pre-pass of its first chunk and the transforms of
    // its last: the first sub-launch ramps up (16, 16, 32), the last one ramps down (32, 16, 16), everything between goes
    // in the largest pieces.  (Chunks of 8 were measured and lose: the per-bin kernel's 8-block form takes 128 us per
    // chunk against 187 us for 16 blocks; config 5 at 64 blocks per call: 1.39 ms with 16-16-16-16, 1.50 ms with
    // 8-8-16-16-8-8, 1.61 ms un-overlapped.)  With the EQ off there is nothing to overlap: one chunk per sub-launch.
    auto chunks_of = [&](int j, std::vector<std::pair<int, int>>& out) {
        out.clear();
        const int k = std::min<int>((int)kc, total - j * (int)kc);
        if (!eq_on) { out.emplace_back(0, k); return; }
        std::vector<int> head, tail;
        int rest = k;
        if (j == 0) for (int c : {16, 16, 32}) if (rest >= 2 * c) { head.push_back(c); rest -= c; }
        if (j == n_sub - 1) for (int c : {16, 16, 32}) if (rest >= 2 * c) { tail.push_back(c); rest -= c; }
        int at = 0;
        for (int c : head) { out.emplace_back(at, c); at += c; }
        if (rest > 0) { out.emplace_back(at, rest); at += rest; }
        for (size_t i = tail.size(); i-- > 0;) { out.emplace_back(at, tail[i]); at += tail[i]; }
    };
    std::vector<std::vector<std::pair<int, int>>> chunks(n_sub);
    std::vector<std::vector<cudaEvent_t>> done_ev(n_sub);
    for (int j = 0; j < n_sub; ++j) chunks_of(j, chunks[j]);
    auto next_event = [&](cudaEvent_t* ev) -> int {
        if (h->eq_events_used == h->ev_eq.size()) {
            cudaEvent_t e;
            OHS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->ev_eq.push_back(e);
        }
        *ev = h->ev_eq[h->eq_events_used++];
        return OHS_OK;
    };
    h->eq_events_used = 0;
    // enqueue the EQ pre-pass of sub-launch j (its chunks back to back on the EQ stream, an event behind each)
    auto enqueue_eq = [&](int j) -> int {
        float* xf = h->d_xf + (size_t)(j & 1) * xhalf;
        if (j >= 2) OHS_CUDA(cudaStreamWaitEvent(h->eq_stream, h->ev_fwd[j & 1], 0));   // sub-launch j-2's transforms have read this half
        for (const auto& c : chunks[j]) {
            const size_t f0 = ((size_t)j * kc + c.first) * B;
            int rc = launch_eq_prepass(h, p, d_in + f0, (long long)row_stride, xf + (size_t)c.first * B, xstride, (size_t)c.second * B);
            if (rc) return rc;
            cudaEvent_t ev;
            rc = next_event(&ev);
            if (rc) return rc;
            OHS_CUDA(cudaEventRecord(ev, h->eq_stream));
            done_ev[j].push_back(ev);
        }
        return OHS_OK;
    };
    if (eq_on) {
        // the EQ stream starts behind everything already enqueued on the engine's stream (EQ state, input rows)
        OHS_CUDA(cudaEventRecord(h->ev_call, h->stream));
        OHS_CUDA(cudaStreamWaitEvent(h->eq_stream, h->ev_call, 0));
        for (int j = 0; j < std::min(2, n_sub); ++j) { const int rc = enqueue_eq(j); if (rc) return rc; }
    }
    for (int j = 0; j < n_sub; ++j) {
        const int k = std::min<int>((int)kc, total - j * (int)kc);
        if (!h->zlin_valid) {
            // the route changes here (first call, or block-by-block calls since the last time-batched one): the ring's
            // history goes behind the next block's slot; between time-batched sub-launches and calls nothing is copied
            gather_history_kernel<<<dim3((unsigned)hist, (unsigned)S), 256, 0, h->stream>>>(h->d_fdl, h->d_zlin, (int)N, h->pmax, h->head, zstride,
                                                                                        h->zl_base, h->zl_cap);
            OHS_CUDA(cudaGetLastError());
            h->launches++;
            h->zlin_valid = true;
        }
        const int zb = h->zl_base;   // slot of this sub-launch's block 0
        // filtered rows of this sub-launch: a half of d_xf (with the EQ off, a copy of the input rows: the transforms read
        // a block's predecessor too, which an in-place call has overwritten with output by then)
        float* xf = h->d_xf + (size_t)(j & 1) * xhalf;
        if (!eq_on)
            OHS_CUDA(cudaMemcpy2DAsync(xf, (size_t)xstride * sizeof(float), d_in + (size_t)j * kc * B, row_stride * sizeof(float),
                                       (size_t)k * B * sizeof(float), S * 2, cudaMemcpyDeviceToDevice, h->stream));
        float* out_j = d_out + (size_t)j * kc * B;
        for (size_t ci = 0; ci < chunks[j].size(); ++ci) {
            const int c0 = chunks[j][ci].first, ck = chunks[j][ci].second;
            if (eq_on) OHS_CUDA(cudaStreamWaitEvent(h->stream, done_ev[j][ci], 0));
            float2* w = h->d_wlin + S * (size_t)c0 * N;
            const int rc = with_transform_size(h->N, (int)OHS_ERR_INVALID, [&](auto n) {
                int r = launch_forward<n>(h, xf, xstride, c0, ck, zstride, zb);
                if (!r) r = launch_bin_conv(h, (zb + c0) % h->zl_cap, w, ck, zstride);
                return r ? r : launch_inverse<n>(h, w, out_j + (size_t)c0 * B, ck, row_stride);
            });
            if (rc) return rc;
        }
        // overlap-save history of the next sub-launch or call: this one's last filtered block
        OHS_CUDA(cudaMemcpy2DAsync(h->d_prev, B * sizeof(float), xf + (size_t)(k - 1) * B, (size_t)xstride * sizeof(float), B * sizeof(float),
                                   S * 2, cudaMemcpyDeviceToDevice, h->stream));
        if (eq_on) {
            OHS_CUDA(cudaEventRecord(h->ev_fwd[j & 1], h->stream));
            if (j + 2 < n_sub) { const int rc = enqueue_eq(j + 2); if (rc) return rc; }
        }
        h->head = (int)(((size_t)h->head + k) % (size_t)h->pmax);
        h->zl_base = (zb + k) % h->zl_cap;
        h->ring_valid = false;   // the spectra of these blocks exist in the time-ordered buffer only (ensure_ring)
    }
    return OHS_OK;
}

}  // namespace

extern "C" {

int ohs_abi_version(void) { return OHS_ABI_VERSION; }
const char* ohs_last_error(void) { return g_last_error.c_str(); }

int ohs_eq_design(int filter_type, float fs, float fc, float q, float gain_db, float out[5]) {
    if (!out) return fail(OHS_ERR_INVALID, "null output");
    return eq_design_impl(filter_type, fs, fc, q, gain_db, out);
}

int ohs_create(const ohs_config* cfg, ohs_engine** out) {
    if (!cfg || !out) return fail(OHS_ERR_INVALID, "null argument");
    *out = nullptr;
    const int B = cfg->block;
    if (!(B == 64 || B == 128 || B == 256 || B == 512 || B == 1024)) return fail(OHS_ERR_INVALID, "block must be 64, 128, 256, 512 or 1024 (got %d)", B);
    if (cfg->n_streams < 1) return fail(OHS_ERR_INVALID, "n_streams must be >= 1");
    if (cfg->n_bands < 0 || cfg->n_bands > OHS_MAX_BANDS) return fail(OHS_ERR_INVALID, "n_bands must be 0..%d", OHS_MAX_BANDS);
    if (cfg->n_hrir_sets < 1 || cfg->n_eq_sets < 1) return fail(OHS_ERR_INVALID, "need at least one HRIR set and one EQ set");
    if (cfg->max_taps < 1) return fail(OHS_ERR_INVALID, "max_taps must be >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(OHS_ERR_NO_DEVICE, "no CUDA device available; this engine has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(OHS_ERR_INVALID, "device %d out of range (%d devices)", cfg->device, ndev);
    OHS_CUDA(cudaSetDevice(cfg->device));

    ohs_engine* h = new ohs_engine();
    h->cfg = *cfg;
    h->B = B;
    h->N = 2 * B;
    h->pmax = (cfg->max_taps + B - 1) / B;
    h->G = pick_streams_per_cta(h);
    if (const char* e = getenv("OHS_TIME_BATCH")) h->time_batch = atoi(e) != 0;
    if (const char* e = getenv("OHS_STAGE_MB")) { const long mb = atol(e); if (mb >= 1 && mb <= 4096) h->stage_bytes = (size_t)mb << 20; }
    if (const char* e = getenv("OHS_PDL")) h->dependent_launch = atoi(e) != 0;
    if (const char* e = getenv("OHS_LATENCY_BLOCKS")) h->latency_blocks = atoi(e);
    const int S = cfg->n_streams;
    const size_t per_path = (size_t)h->pmax * B;

    h->h_stream_hrir.assign(S, 0);
    h->h_group_first = {0, S};
    h->h_move_to.assign(S, -1);
    h->h_stream_eq.assign(S, 0);
    h->h_gain.assign(S, 1.0f);
    h->h_set_parts.assign(cfg->n_hrir_sets, 1);
    h->h_path_parts.assign((size_t)cfg->n_hrir_sets * 4, 1);
    h->h_ir.assign((size_t)cfg->n_hrir_sets * 4, std::vector<float>());
    h->set_dirty.assign(cfg->n_hrir_sets, 0);
    h->set_external.assign(cfg->n_hrir_sets, 0);
    h->h_eqc.assign((size_t)cfg->n_eq_sets * kMaxBands * kEqCoefStride, 0.f);
    {
        // BiquadFilter::new: PeakingEQ(0 dB) @ 20 Hz, Q 0.707, disabled (src/dsp/parametric_eq.rs:63-76)
        float c[5] = {1.f, 0.f, 0.f, 0.f, 0.f};
        if (2.0f * 20.0f <= cfg->sample_rate) eq_design_impl(OHS_FILTER_PEAK, cfg->sample_rate, 20.0f, 0.707f, 0.0f, c);
        for (int e = 0; e < cfg->n_eq_sets; ++e)
            for (int b = 0; b < kMaxBands; ++b) {
                float* dst = h->h_eqc.data() + ((size_t)e * kMaxBands + b) * kEqCoefStride;
                for (int i = 0; i < 5; ++i) dst[i] = c[i];
            }
    }

#define OHS_TRY(expr)                                   \
    do {                                                \
        cudaError_t _e = (expr);                        \
        if (_e != cudaSuccess) {                        \
            fail(OHS_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
            ohs_destroy(h);                             \
            return OHS_ERR_CUDA;                        \
        }                                               \
    } while (0)
    OHS_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    OHS_TRY(cudaStreamCreateWithFlags(&h->h2d, cudaStreamNonBlocking));
    OHS_TRY(cudaStreamCreateWithFlags(&h->d2h, cudaStreamNonBlocking));
    OHS_TRY(cudaEventCreate(&h->ev_k0));
    OHS_TRY(cudaEventCreate(&h->ev_k1));
    for (int i = 0; i < kPipe; ++i) {
        OHS_TRY(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
        OHS_TRY(cudaEventCreateWithFlags(&h->ev_comp[i], cudaEventDisableTiming));
        OHS_TRY(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
    }
    h->filt_bytes = sizeof(float4) * (size_t)cfg->n_hrir_sets * h->pmax * h->N;
    OHS_TRY(cudaMalloc(&h->d_stream_hrir, sizeof(int) * S));
    OHS_TRY(cudaMalloc(&h->d_from_set, sizeof(int) * S));
    OHS_TRY(cudaMalloc(&h->d_group_first, sizeof(int) * ((size_t)S + 1)));
    OHS_TRY(cudaMalloc(&h->d_stream_eq, sizeof(int) * S));
    OHS_TRY(cudaMalloc(&h->d_stream_gain, sizeof(float) * S));
    OHS_TRY(cudaMalloc(&h->d_filt, h->filt_bytes));
    OHS_TRY(cudaMalloc(&h->d_set_parts, sizeof(int) * cfg->n_hrir_sets));
    OHS_TRY(cudaMalloc(&h->d_set_list, sizeof(int) * cfg->n_hrir_sets));
    OHS_TRY(cudaMalloc(&h->d_set_flags, cfg->n_hrir_sets));
    OHS_TRY(cudaMalloc(&h->d_fdl, sizeof(float2) * (size_t)S * h->pmax * h->N));
    OHS_TRY(cudaMalloc(&h->d_prev, sizeof(float2) * (size_t)S * B));
    OHS_TRY(cudaMalloc(&h->d_eqc, sizeof(float) * h->h_eqc.size()));
    OHS_TRY(cudaMalloc(&h->d_eqs, sizeof(float4) * (size_t)S * kMaxBands));
    OHS_TRY(cudaMalloc(&h->d_tw, sizeof(float2) * h->N));
    OHS_TRY(cudaMalloc(&h->d_ir, sizeof(float) * (size_t)cfg->n_hrir_sets * 4 * per_path));
    OHS_TRY(cudaMemsetAsync(h->d_filt, 0, h->filt_bytes, h->stream));  // default IR = silence (src/dsp/convolution.rs:44-65)
    OHS_TRY(cudaMemsetAsync(h->d_fdl, 0, sizeof(float2) * (size_t)S * h->pmax * h->N, h->stream));
    OHS_TRY(cudaMemsetAsync(h->d_prev, 0, sizeof(float2) * (size_t)S * B, h->stream));
    OHS_TRY(cudaMemsetAsync(h->d_eqs, 0, sizeof(float4) * (size_t)S * kMaxBands, h->stream));
    OHS_TRY(cudaMemsetAsync(h->d_ir, 0, sizeof(float) * (size_t)cfg->n_hrir_sets * 4 * per_path, h->stream));
    {
        std::vector<float2> tw(h->N);
        with_transform_size(h->N, false, [&](auto n) { fill_twiddles<n>(tw.data()); return true; });
        OHS_TRY(cudaMemcpyAsync(h->d_tw, tw.data(), sizeof(float2) * h->N, cudaMemcpyHostToDevice, h->stream));
        OHS_TRY(cudaMemcpyAsync(h->d_set_parts, h->h_set_parts.data(), sizeof(int) * cfg->n_hrir_sets, cudaMemcpyHostToDevice, h->stream));
        OHS_TRY(cudaMemcpyAsync(h->d_group_first, h->h_group_first.data(), sizeof(int) * 2, cudaMemcpyHostToDevice, h->stream));
        OHS_TRY(cudaStreamSynchronize(h->stream));
    }
#undef OHS_TRY
    *out = h;
    return OHS_OK;
}

int ohs_destroy(ohs_engine* h) {
    if (!h) return OHS_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->eq_stream) { cudaStreamSynchronize(h->eq_stream); cudaStreamDestroy(h->eq_stream); }
    for (cudaEvent_t e : h->ev_eq) cudaEventDestroy(e);
    for (cudaEvent_t e : {h->ev_fwd[0], h->ev_fwd[1], h->ev_call}) if (e) cudaEventDestroy(e);
    void* ptrs[] = {h->d_stream_hrir, h->d_stream_eq, h->d_stream_gain, h->d_filt, h->d_set_parts, h->d_set_list, h->d_set_flags,
                    h->d_fdl, h->d_prev, h->d_eqc, h->d_eqs, h->d_tw, h->d_ir, h->d_stage[0], h->d_stage[1], h->d_stage[2],
                    h->d_zlin, h->d_wlin, h->d_xf, h->d_from_set, h->d_sched, h->d_pcm_stage[0], h->d_pcm_stage[1],
                    h->d_pcm_stage[2], h->d_pcm_scratch, h->d_dither_hist, h->d_group_first, h->d_bus_stage[0],
                    h->d_bus_stage[1], h->d_bus_stage[2]};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (int i = 0; i < kPipe; ++i) {
        if (h->ev_in[i]) cudaEventDestroy(h->ev_in[i]);
        if (h->ev_comp[i]) cudaEventDestroy(h->ev_comp[i]);
        if (h->ev_out[i]) cudaEventDestroy(h->ev_out[i]);
    }
    if (h->ev_k0) cudaEventDestroy(h->ev_k0);
    if (h->ev_k1) cudaEventDestroy(h->ev_k1);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->h2d) cudaStreamDestroy(h->h2d);
    if (h->d2h) cudaStreamDestroy(h->d2h);
    delete h;
    return OHS_OK;
}

// ---- HRIR ---------------------------------------------------------------------------------------------------
int ohs_set_ir(ohs_engine* h, int hrir_set, int path, const float* ir, size_t len) {
    OHS_CHECK_HANDLE(h);
    if (hrir_set < 0 || hrir_set >= h->cfg.n_hrir_sets) return fail(OHS_ERR_INVALID, "hrir_set %d out of range", hrir_set);
    if (path < 0 || path > 3) return fail(OHS_ERR_INVALID, "path %d out of range", path);
    if (len > 0 && !ir) return fail(OHS_ERR_INVALID, "null impulse response");
    if (len > (size_t)h->pmax * h->B) return fail(OHS_ERR_INVALID, "impulse response of %zu taps exceeds max_taps capacity %d", len, h->pmax * h->B);
    std::vector<float>& dst = h->h_ir[(size_t)hrir_set * 4 + path];
    dst.assign(ir, ir + len);
    // ir.chunks(BLOCK_SIZE).count(), or one silent partition for an empty slice (src/dsp/convolution.rs:114-132)
    h->h_path_parts[(size_t)hrir_set * 4 + path] = len == 0 ? 1 : (int)((len + h->B - 1) / h->B);
    h->set_dirty[hrir_set] = 1;
    h->set_external[hrir_set] = 0;
    h->any_set_dirty = true;
    return OHS_OK;
}

int ohs_num_partitions(ohs_engine* h, int hrir_set, int path, int* out) {
    OHS_CHECK_HANDLE(h);
    if (!out || hrir_set < 0 || hrir_set >= h->cfg.n_hrir_sets || path < 0 || path > 3) return fail(OHS_ERR_INVALID, "bad argument");
    *out = h->h_path_parts[(size_t)hrir_set * 4 + path];
    return OHS_OK;
}

int ohs_bind_stream_hrir(ohs_engine* h, int stream, int hrir_set) {
    OHS_CHECK_HANDLE(h);
    if (hrir_set < 0 || hrir_set >= h->cfg.n_hrir_sets) return fail(OHS_ERR_INVALID, "hrir_set %d out of range", hrir_set);
    if (stream != OHS_ALL && (stream < 0 || stream >= h->cfg.n_streams)) return fail(OHS_ERR_INVALID, "stream %d out of range", stream);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    if (stream == OHS_ALL) std::fill(h->h_stream_hrir.begin(), h->h_stream_hrir.end(), hrir_set);
    else h->h_stream_hrir[stream] = hrir_set;
    if (stream == OHS_ALL) std::fill(h->h_move_to.begin(), h->h_move_to.end(), -1);   // a hard bind cancels a pending move
    else h->h_move_to[stream] = -1;
    h->bind_dirty = true;
    // a re-bound stream starts from empty history, like a ConvolutionEngine that was just given its IRs
    if (stream == OHS_ALL) {
        int rc = upload_bindings(h);
        if (rc) return rc;
        return clear_history(h, false);
    }
    { const int rc = ensure_ring(h); if (rc) return rc; }
    h->zlin_valid = false;
    OHS_CUDA(cudaMemsetAsync(h->d_fdl + (size_t)stream * h->pmax * h->N, 0, sizeof(float2) * (size_t)h->pmax * h->N, h->stream));
    OHS_CUDA(cudaMemsetAsync(h->d_prev + (size_t)stream * h->B, 0, sizeof(float2) * (size_t)h->B, h->stream));
    return OHS_OK;
}

int ohs_move_stream_hrir(ohs_engine* h, int stream, int hrir_set) {
    OHS_CHECK_HANDLE(h);
    if (hrir_set < 0 || hrir_set >= h->cfg.n_hrir_sets) return fail(OHS_ERR_INVALID, "hrir_set %d out of range", hrir_set);
    if (stream != OHS_ALL && (stream < 0 || stream >= h->cfg.n_streams)) return fail(OHS_ERR_INVALID, "stream %d out of range", stream);
    const int lo = stream == OHS_ALL ? 0 : stream, hi = stream == OHS_ALL ? h->cfg.n_streams : stream + 1;
    for (int s = lo; s < hi; ++s) h->h_move_to[s] = hrir_set == h->h_stream_hrir[s] ? -1 : hrir_set;   // back to the binding: no move
    h->any_move = std::any_of(h->h_move_to.begin(), h->h_move_to.end(), [](int v) { return v >= 0; });
    return OHS_OK;
}

int ohs_commit_filters(ohs_engine* h) {
    OHS_CHECK_HANDLE(h);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    return commit_filters(h);
}

int ohs_filter_table(ohs_engine* h, void** dev_ptr, size_t* bytes) {
    OHS_CHECK_HANDLE(h);
    if (!dev_ptr || !bytes) return fail(OHS_ERR_INVALID, "null output");
    *dev_ptr = h->d_filt;
    *bytes = h->filt_bytes;
    return OHS_OK;
}

int ohs_mark_filters_external(ohs_engine* h, int hrir_set, int partitions) {
    OHS_CHECK_HANDLE(h);
    if (hrir_set < 0 || hrir_set >= h->cfg.n_hrir_sets) return fail(OHS_ERR_INVALID, "hrir_set %d out of range", hrir_set);
    if (partitions < 1 || partitions > h->pmax) return fail(OHS_ERR_INVALID, "partitions %d out of range 1..%d", partitions, h->pmax);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    h->set_dirty[hrir_set] = 0;
    h->set_external[hrir_set] = 1;
    h->h_set_parts[hrir_set] = partitions;
    for (int p = 0; p < 4; ++p) h->h_path_parts[(size_t)hrir_set * 4 + p] = partitions;
    h->any_set_dirty = false;
    for (unsigned char d : h->set_dirty) h->any_set_dirty |= d != 0;
    OHS_CUDA(cudaMemcpyAsync(h->d_set_parts, h->h_set_parts.data(), sizeof(int) * h->cfg.n_hrir_sets, cudaMemcpyHostToDevice, h->stream));
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    return OHS_OK;
}

// ---- EQ -----------------------------------------------------------------------------------------------------
int ohs_eq_update_band(ohs_engine* h, int eq_set, int band, int filter_type, float fc, float q, float gain_db, int enabled) {
    OHS_CHECK_HANDLE(h);
    if (band < 0 || band >= h->cfg.n_bands) {
        if (eq_set < 0 || eq_set >= h->cfg.n_eq_sets) return fail(OHS_ERR_INVALID, "eq_set %d out of range", eq_set);
        return OHS_OK;
    }
    float c[5];
    int rc = eq_design_impl(filter_type, h->cfg.sample_rate, fc, q, gain_db, c);
    if (rc) return rc;
    return set_band_host(h, eq_set, band, c, enabled);
}

int ohs_eq_set_band(ohs_engine* h, int eq_set, int band, const float coeffs[5], int enabled) {
    OHS_CHECK_HANDLE(h);
    if (!coeffs) return fail(OHS_ERR_INVALID, "null coefficients");
    return set_band_host(h, eq_set, band, coeffs, enabled);
}

int ohs_bind_stream_eq(ohs_engine* h, int stream, int eq_set) {
    OHS_CHECK_HANDLE(h);
    if (eq_set < 0 || eq_set >= h->cfg.n_eq_sets) return fail(OHS_ERR_INVALID, "eq_set %d out of range", eq_set);
    if (stream != OHS_ALL && (stream < 0 || stream >= h->cfg.n_streams)) return fail(OHS_ERR_INVALID, "stream %d out of range", stream);
    if (stream == OHS_ALL) std::fill(h->h_stream_eq.begin(), h->h_stream_eq.end(), eq_set);
    else h->h_stream_eq[stream] = eq_set;
    h->bind_dirty = true;
    return OHS_OK;
}

int ohs_eq_reset(ohs_engine* h) {
    OHS_CHECK_HANDLE(h);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    OHS_CUDA(cudaMemsetAsync(h->d_eqs, 0, sizeof(float4) * (size_t)h->cfg.n_streams * kMaxBands, h->stream));
    return OHS_OK;
}

int ohs_eq_frequency_response(ohs_engine* h, int eq_set, float sample_rate, const float* freqs, float* out, size_t n) {
    OHS_CHECK_HANDLE(h);
    if (eq_set < 0 || eq_set >= h->cfg.n_eq_sets || !freqs || !out) return fail(OHS_ERR_INVALID, "bad argument");
    const float fs = sample_rate > 0.0f ? sample_rate : h->cfg.sample_rate;
    for (size_t i = 0; i < n; ++i) {
        float rr = 1.0f, ri = 0.0f;
        for (int b = 0; b < h->cfg.n_bands; ++b) {
            const float* c = h->h_eqc.data() + ((size_t)eq_set * kMaxBands + b) * kEqCoefStride;
            if (c[5] == 0.0f) continue;
            const float w = 2.0f * 3.14159265358979323846f * freqs[i] / fs;
            const float c1 = cosf(w), s1 = sinf(w), c2 = cosf(2.0f * w), s2 = sinf(2.0f * w);
            const float nr = c[0] + c[1] * c1 + c[2] * c2, ni = c[1] * s1 + c[2] * s2;
            const float dr = 1.0f + c[3] * c1 + c[4] * c2, di = c[3] * s1 + c[4] * s2;
            const float den = dr * dr + di * di;
            const float hr = (nr * dr + ni * di) / den, hi = (ni * dr - nr * di) / den;
            const float tr = rr * hr - ri * hi, ti = rr * hi + ri * hr;
            rr = tr; ri = ti;
        }
        out[i] = hypotf(rr, ri);
    }
    return OHS_OK;
}

// ---- switches -----------------------------------------------------------------------------------------------
int ohs_set_eq_enable(ohs_engine* h, int enable) { OHS_CHECK_HANDLE(h); h->eq_enable = enable ? 1 : 0; return OHS_OK; }
int ohs_set_conv_enable(ohs_engine* h, int enable) { OHS_CHECK_HANDLE(h); h->conv_enable = enable ? 1 : 0; return OHS_OK; }
int ohs_set_bypass(ohs_engine* h, int bypass) { OHS_CHECK_HANDLE(h); h->bypass = bypass ? 1 : 0; return OHS_OK; }

int ohs_set_dither(ohs_engine* h, int mode, uint64_t seed, const float* shape, int n_taps) {
    OHS_CHECK_HANDLE(h);
    if (mode != OHS_DITHER_OFF && mode != OHS_DITHER_TPDF) return fail(OHS_ERR_INVALID, "unknown dither mode %d", mode);
    if (n_taps < 0 || n_taps > OHS_MAX_SHAPE_TAPS) return fail(OHS_ERR_INVALID, "n_taps %d outside 0..%d", n_taps, OHS_MAX_SHAPE_TAPS);
    if (mode == OHS_DITHER_OFF && n_taps) return fail(OHS_ERR_INVALID, "noise-shaping taps need OHS_DITHER_TPDF");
    if (n_taps && !shape) return fail(OHS_ERR_INVALID, "null shape with %d taps", n_taps);
    for (int k = 0; k < n_taps; ++k)
        if (!std::isfinite(shape[k])) return fail(OHS_ERR_INVALID, "shape[%d] is not finite", k);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    const size_t hist_bytes = sizeof(float) * (size_t)h->cfg.n_streams * 4 * OHS_MAX_SHAPE_TAPS;   // stream rows, then bus rows (G <= S)
    if (mode != OHS_DITHER_OFF && !h->d_dither_hist) OHS_CUDA(cudaMalloc(&h->d_dither_hist, hist_bytes));
    // on the engine's stream: ordered after every encode enqueued before
    if (h->d_dither_hist) OHS_CUDA(cudaMemsetAsync(h->d_dither_hist, 0, hist_bytes, h->stream));
    h->dither_mode = mode;
    h->dither_seed = seed;
    h->dither_taps = n_taps;
    h->dither_h = DitherTaps{};
    for (int k = 0; k < n_taps; ++k) h->dither_h.h[k] = shape[k];
    h->dither_pos = 0;
    h->bus_hist_live = false;
    return OHS_OK;
}

int ohs_set_gain(ohs_engine* h, int stream, float gain) {
    OHS_CHECK_HANDLE(h);
    if (stream != OHS_ALL && (stream < 0 || stream >= h->cfg.n_streams)) return fail(OHS_ERR_INVALID, "stream %d out of range", stream);
    if (stream == OHS_ALL) std::fill(h->h_gain.begin(), h->h_gain.end(), gain);
    else h->h_gain[stream] = gain;
    h->gain_dirty = true;
    return OHS_OK;
}

int ohs_conv_reset(ohs_engine* h) {
    OHS_CHECK_HANDLE(h);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    h->head = 0;
    return clear_history(h, false);
}

int ohs_set_time_batch(ohs_engine* h, int enable) { OHS_CHECK_HANDLE(h); h->time_batch = enable ? 1 : 0; return OHS_OK; }

int ohs_streams_per_cta(ohs_engine* h, int* out) {
    OHS_CHECK_HANDLE(h);
    if (!out) return fail(OHS_ERR_INVALID, "null output");
    *out = h->G;
    return OHS_OK;
}

int ohs_prepare(ohs_engine* h, size_t n_frames, int host_io) {
    OHS_CHECK_HANDLE(h);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    int rc = commit_filters(h);
    if (rc) return rc;
    size_t per_launch = n_frames;
    if (host_io) {
        // the widest chunk of ohs_process_pcm over every format pair: S16 has the most frames per chunk, which size the
        // f32 slots; the PCM slots hold the larger of the S16 and S24 rows
        const size_t rows = (size_t)h->cfg.n_streams * 2;
        per_launch = chunk_frames(h, n_frames, h->stage_bytes, 2);
        const size_t pcm_bytes = rows * std::max(per_launch * 2, chunk_frames(h, n_frames, h->stage_bytes, 3) * 3);
        // ohs_process_grouped_pcm's bus rows: its chunks are those of F32 output, and an integer bus's packed rows
        // (round_up(n, 16) frames of at most 3 bytes) fit in the f32 rows' bytes
        const size_t bus_bytes = (size_t)2 * n_groups(h) * chunk_frames(h, n_frames, h->stage_bytes, sizeof(float)) * sizeof(float);
        if ((rc = grow_buffers(h, h->d_stage, kPipe, h->stage_cap, rows * per_launch * sizeof(float))) ||
            (rc = grow_buffers(h, h->d_pcm_stage, kPipe, h->pcm_stage_cap, pcm_bytes)) ||
            (rc = grow_buffers(h, h->d_bus_stage, kPipe, h->bus_stage_cap, bus_bytes)))
            return rc;
    } else if (n_frames) {
        rc = ensure_pcm_scratch(h, chunk_frames(h, n_frames, kPcmScratchBytes, sizeof(float)));   // ohs_process_device_pcm
        if (rc) return rc;
    }
    const size_t tb = time_batch_blocks(h, (int)((per_launch + h->B - 1) / h->B));
    if (tb && (rc = ensure_time_batch_scratch(h, tb))) return rc;
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    return OHS_OK;
}

int ohs_debug_trace(ohs_engine* h, unsigned long long* d_stamps) {
    OHS_CHECK_HANDLE(h);
#ifdef OHS_TRACE
    h->d_trace = d_stamps;
    return OHS_OK;
#else
    (void)d_stamps;
    return fail(OHS_ERR_INVALID, "this library was built without -DOHS_TRACE");
#endif
}

// ---- processing ---------------------------------------------------------------------------------------------
}  // extern "C"

namespace {

// A multi-set engine with a delay line where some stream is bound to a one-partition set: render_kernel does not put
// that stream's spectra into the delay line (it never reads them), but a later move to a longer set needs them, so
// such calls run the moving-sources kernel, which writes every block's.  Same outputs, more delay-line traffic.
bool needs_full_ring(const ohs_engine* h) {
    if (h->pmax == 1 || h->cfg.n_hrir_sets == 1) return false;
    for (int set : h->h_stream_hrir) if (h->h_set_parts[set] == 1) return true;
    return false;
}

// ohs_process_device, and ohs_process_device_scheduled with `sets` (validated by the caller)
int process_device_impl(ohs_engine* h, const float* d_in, float* d_out, size_t n_frames, size_t row_stride, const int32_t* sets,
                        size_t sets_stride) {
    if (n_frames == 0) return OHS_OK;
    if (h->bypass) {  // master_bypass: buffer untouched, no state advances (src/lib.rs:1169)
        if (d_in != d_out)
            OHS_CUDA(cudaMemcpy2DAsync(d_out, row_stride * sizeof(float), d_in, row_stride * sizeof(float), n_frames * sizeof(float),
                                       (size_t)h->cfg.n_streams * 2, cudaMemcpyDeviceToDevice, h->stream));
        return OHS_OK;
    }
    int rc = commit_filters(h);
    if (rc) return rc;
    RenderParams p{};
    p.in = d_in; p.out = d_out; p.row_stride = p.out_row_stride = (long long)row_stride;
    p.n_blocks = (int)((n_frames + h->B - 1) / h->B);
    p.tail_frames = (int)(n_frames - (size_t)(p.n_blocks - 1) * h->B);
    p.n_streams = h->cfg.n_streams;
    p.stream_hrir = h->d_stream_hrir; p.stream_eq = h->d_stream_eq; p.stream_gain = h->d_stream_gain;
    p.filt = h->d_filt; p.set_parts = h->d_set_parts; p.fdl = h->d_fdl; p.prev = h->d_prev;
    p.eqc = h->d_eqc; p.eqs = h->d_eqs; p.tw = h->d_tw;
    p.pmax = h->pmax; p.head = h->head; p.n_bands = h->cfg.n_bands;
    p.eq_enable = h->eq_enable && h->cfg.n_bands > 0; p.conv_enable = h->conv_enable;
    p.uniform_set = (h->cfg.n_hrir_sets == 1) ? 1 : 0;
    // one HRIR set shared by every stream and small enough: the kernel keeps its spectra in shared memory
    p.filt_in_smem = 0;
    if (h->cfg.n_hrir_sets == 1 && h->N <= 512 && (size_t)h->h_set_parts[0] * h->N * sizeof(float4) <= 16 * 1024)
        p.filt_in_smem = h->h_set_parts[0];
    // moving sources: does this call carry a transition (set of a block != set of the block before)?  Pending moves
    // apply only to convolving calls, after the commit above has cleared the streams bound to re-committed sets.
    const size_t S = (size_t)h->cfg.n_streams, K = (size_t)p.n_blocks;
    bool transition = false;
    if (sets) {
        for (size_t s = 0; s < S && !transition; ++s) {
            int prev = h->h_stream_hrir[s];
            for (size_t t = 0; t < K; ++t) {
                const int cur = sets[s * sets_stride + t];
                if (cur != prev) { transition = true; break; }
                prev = cur;
            }
        }
        if (transition) {
            rc = grow_buffers(h, &h->d_sched, 1, h->sched_cap, sizeof(int) * S * K);
            if (rc) return rc;
            OHS_CUDA(cudaMemcpy2DAsync(h->d_sched, sizeof(int) * K, sets, sizeof(int) * sets_stride, sizeof(int) * K, S,
                                       cudaMemcpyHostToDevice, h->stream));
            p.block_set = h->d_sched; p.block_set_stride = (long long)K;
        }
        p.from_set = h->d_stream_hrir;   // block 0 compares with the binding
        std::fill(h->h_move_to.begin(), h->h_move_to.end(), -1);   // the schedule supersedes pending moves
        h->any_move = false;
        for (size_t s = 0; s < S; ++s) {
            const int last = sets[s * sets_stride + K - 1];
            if (last != h->h_stream_hrir[s]) { h->h_stream_hrir[s] = last; h->bind_dirty = true; }   // uploaded by the next call
        }
    } else if (h->any_move && h->conv_enable) {
        h->h_from_set = h->h_stream_hrir;
        for (size_t s = 0; s < S; ++s)
            if (h->h_move_to[s] >= 0) { h->h_stream_hrir[s] = h->h_move_to[s]; h->h_move_to[s] = -1; }
        h->any_move = false;
        h->bind_dirty = true;
        transition = true;
        rc = upload_bindings(h);
        if (rc) return rc;
        OHS_CUDA(cudaMemcpyAsync(h->d_from_set, h->h_from_set.data(), sizeof(int) * S, cudaMemcpyHostToDevice, h->stream));
        p.from_set = h->d_from_set;
    }
    // (off by default: an event between two launches keeps the second from starting while the first drains)
    if (h->timing) OHS_CUDA(cudaEventRecord(h->ev_k0, h->stream));
    // long responses over many blocks: convolve along time per bin instead of re-reading the delay line every block
    // (one set per stream and call: a call with a transition runs the block-by-block kernel)
    const size_t tb = transition ? 0 : time_batch_blocks(h, p.n_blocks);
    if (tb) {
        rc = process_time_batched(h, p, tb, d_in, d_out, row_stride);
        if (rc) return rc;
    } else {
        if (h->conv_enable) { rc = ensure_ring(h); if (rc) return rc; }   // the kernel reads and extends the delay-line ring
        const bool moving = transition || (h->conv_enable && needs_full_ring(h));
        if (moving && !p.from_set) p.from_set = h->d_stream_hrir;
        rc = launch_render(h, p, 0, moving);
        if (rc) return rc;
        if (h->conv_enable) {
            h->head = (int)(((size_t)h->head + p.n_blocks) % (size_t)h->pmax);
            h->zlin_valid = false;
        }
    }
    if (h->timing) { OHS_CUDA(cudaEventRecord(h->ev_k1, h->stream)); h->timed = true; }
    return OHS_OK;
}

// One chunk of f32 stream rows x (pitch p floats, n frames, at frame f0 of the call) in HBM: the PCM input side decoded
// into x (an f32 input side is x already), x rendered in place when `render`, then x encoded into the PCM output rows,
// mixed into the f32 bus, or mixed and encoded into the PCM bus (an f32 output side that is not a bus is x itself).  An
// encode's first frame is at dither position dither_pos + f0: the position moves once per call, at the call's exit.
int chunk_step(ohs_engine* h, const Rows& in, float* x, size_t p, size_t n, size_t f0, bool render, const Rows& out) {
    int rc = with_pcm_format(in.fmt, (int)OHS_ERR_INVALID, [&](auto f) {
        if constexpr (f == kPcmF32) return (int)OHS_OK;
        else return launch_decode<f>(h, in, x, p, n);
    });
    if (!rc && render) rc = process_device_impl(h, x, x, n, p, nullptr, 0);
    if (rc) return rc;
    const unsigned long long pos = h->dither_pos + f0;
    return with_pcm_format(out.fmt, (int)OHS_ERR_INVALID, [&](auto f) {
        if constexpr (f == kPcmF32) return out.bus ? launch_mix(h, x, p, static_cast<float*>(out.p), out.stride, n) : (int)OHS_OK;
        else return out.bus ? launch_encode<f, true>(h, out, x, p, n, pos) : launch_encode<f, false>(h, out, x, p, n, pos);
    });
}

// include/ohs.h: a call with integer output (the output format, or a bus call's bus format) moves the dither position on
// by n_frames, bypassed or not; F32 output and F32 buses leave it
bool moves_dither(const Rows& out) { return out.fmt != OHS_FMT_F32; }

// ohs_process_device_pcm past validation with at least one side an integer format, and the mixdowns (out.bus: the f32
// input rows mixed into the bus, never rendered)
int process_device_io(ohs_engine* h, const Rows& in, const Rows& out, size_t n_frames) {
    if (n_frames == 0) return OHS_OK;
    const size_t rows = (size_t)h->cfg.n_streams * 2, bi = in.sample_bytes();
    const bool render = !h->bypass && !out.bus;
    if (h->bypass && !out.bus && in.fmt == out.fmt) {   // nothing to convert: the rows as they are
        if (in.p != out.p)
            OHS_CUDA(cudaMemcpy2DAsync(out.p, out.stride * bi, in.p, in.stride * bi, n_frames * bi, rows, cudaMemcpyDeviceToDevice, h->stream));
    } else {
        // the f32 rows the call works in, chosen once: the input rows when there is nothing to decode or render, the output
        // rows (decoded into, rendered in place) for F32 output, else the scratch rows, in time chunks
        const Rows* whole = in.fmt == OHS_FMT_F32 && !render ? &in : out.fmt == OHS_FMT_F32 && !out.bus ? &out : nullptr;
        const size_t chunk = whole ? n_frames : chunk_frames(h, n_frames, kPcmScratchBytes, sizeof(float));
        int rc;
        if (!whole && (rc = ensure_pcm_scratch(h, chunk))) return rc;
        float* x = whole ? static_cast<float*>(whole->p) : h->d_pcm_scratch;
        for (size_t f0 = 0; f0 < n_frames; f0 += chunk) {
            const size_t n = std::min(chunk, n_frames - f0), p = whole ? whole->stride : round_up(n, 4);
            if (!whole && in.fmt == OHS_FMT_F32)
                OHS_CUDA(cudaMemcpy2DAsync(x, p * bi, in.from(f0).p, in.stride * bi, n * bi, rows, cudaMemcpyDeviceToDevice, h->stream));
            if ((rc = chunk_step(h, in.from(f0), x, p, n, f0, render, out.from(f0)))) return rc;
        }
    }
    if (moves_dither(out)) h->dither_pos += n_frames;
    return OHS_OK;
}

}  // namespace

extern "C" {

int ohs_process_device(ohs_engine* h, const float* d_in, float* d_out, size_t n_frames, size_t row_stride) {
    return ohs_process_device_pcm(h, d_in, OHS_FMT_F32, d_out, OHS_FMT_F32, n_frames, row_stride);
}

int ohs_process_device_scheduled(ohs_engine* h, const float* d_in, float* d_out, size_t n_frames, size_t row_stride,
                                 const int32_t* sets, size_t sets_stride) {
    OHS_CHECK_HANDLE(h);
    const int rc = check_call(h, {const_cast<float*>(d_in), OHS_FMT_F32, row_stride}, {d_out, OHS_FMT_F32, row_stride}, n_frames,
                              kWholeBlocks | kDeviceRows);
    if (rc) return rc;
    if (!sets) return fail(OHS_ERR_INVALID, "null schedule");
    if (!h->conv_enable) return fail(OHS_ERR_INVALID, "a schedule needs the convolution enabled");
    const size_t K = n_frames / (size_t)h->B;
    if (sets_stride < K) return fail(OHS_ERR_INVALID, "sets_stride %zu < %zu blocks", sets_stride, K);
    for (size_t s = 0; s < (size_t)h->cfg.n_streams; ++s)
        for (size_t t = 0; t < K; ++t) {
            const int v = sets[s * sets_stride + t];
            if (v < 0 || v >= h->cfg.n_hrir_sets) return fail(OHS_ERR_INVALID, "schedule: stream %zu block %zu names hrir_set %d out of range", s, t, v);
        }
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    return process_device_impl(h, d_in, d_out, n_frames, row_stride, sets, sets_stride);
}

int ohs_process_device_pcm(ohs_engine* h, const void* d_in, int in_format, void* d_out, int out_format, size_t n_frames, size_t row_stride) {
    OHS_CHECK_HANDLE(h);
    const Rows in{const_cast<void*>(d_in), in_format, row_stride}, out{d_out, out_format, row_stride};
    const int rc = check_call(h, in, out, n_frames, kWholeBlocks | kSeparateIfConverted | kDeviceRows);
    if (rc) return rc;
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    if (in_format == OHS_FMT_F32 && out_format == OHS_FMT_F32)
        return process_device_impl(h, static_cast<const float*>(d_in), static_cast<float*>(d_out), n_frames, row_stride, nullptr, 0);
    return process_device_io(h, in, out, n_frames);
}

int ohs_sync(ohs_engine* h) {
    OHS_CHECK_HANDLE(h);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    return OHS_OK;
}

int ohs_cuda_stream(ohs_engine* h, void** stream) {
    OHS_CHECK_HANDLE(h);
    if (!stream) return fail(OHS_ERR_INVALID, "null output");
    *stream = (void*)h->stream;
    return OHS_OK;
}

int ohs_launch_count(ohs_engine* h, uint64_t* out) {
    OHS_CHECK_HANDLE(h);
    if (!out) return fail(OHS_ERR_INVALID, "null output");
    *out = h->launches;
    return OHS_OK;
}

int ohs_enable_timing(ohs_engine* h, int enable) { OHS_CHECK_HANDLE(h); h->timing = enable != 0; if (!enable) h->timed = false; return OHS_OK; }

int ohs_last_kernel_ms(ohs_engine* h, float* ms) {
    OHS_CHECK_HANDLE(h);
    if (!ms) return fail(OHS_ERR_INVALID, "null output");
    if (!h->timed) return fail(OHS_ERR_INVALID, "no timed process call yet (ohs_enable_timing first)");
    OHS_CUDA(cudaEventSynchronize(h->ev_k1));
    OHS_CUDA(cudaEventElapsedTime(ms, h->ev_k0, h->ev_k1));
    return OHS_OK;
}

int ohs_mix_device(ohs_engine* h, const float* d_in, float* d_bus, size_t n_frames, size_t row_stride, size_t bus_stride) {
    return ohs_mix_device_pcm(h, d_in, d_bus, OHS_FMT_F32, n_frames, row_stride, bus_stride);
}

int ohs_mix_device_pcm(ohs_engine* h, const float* d_in, void* d_bus, int bus_format, size_t n_frames, size_t row_stride,
                       size_t bus_stride) {
    OHS_CHECK_HANDLE(h);
    const Rows in{const_cast<float*>(d_in), OHS_FMT_F32, row_stride}, bus{d_bus, bus_format, bus_stride, true};
    const int rc = check_call(h, in, bus, n_frames, kDeviceRows | kWholeQuads);
    if (rc) return rc;
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    return process_device_io(h, in, bus, n_frames);
}

int ohs_set_groups(ohs_engine* h, const int32_t* first, int n_groups) {
    OHS_CHECK_HANDLE(h);
    const int S = h->cfg.n_streams;
    if (!first) return fail(OHS_ERR_INVALID, "null group offsets");
    if (n_groups < 1 || n_groups > S) return fail(OHS_ERR_INVALID, "n_groups %d outside 1..%d", n_groups, S);
    if (first[0] != 0 || first[n_groups] != S)
        return fail(OHS_ERR_INVALID, "group offsets must run from 0 to n_streams %d (got %d .. %d)", S, first[0], first[n_groups]);
    for (int g = 0; g < n_groups; ++g)
        if (first[g + 1] <= first[g]) return fail(OHS_ERR_INVALID, "group %d is empty or the offsets decrease (%d, %d)", g, first[g], first[g + 1]);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    std::vector<int> v(first, first + n_groups + 1);
    // on the engine's stream: mixes enqueued before still read the old offsets (a pageable source is staged before returning)
    OHS_CUDA(cudaMemcpyAsync(h->d_group_first, v.data(), sizeof(int) * v.size(), cudaMemcpyHostToDevice, h->stream));
    // a new partition makes the old bus rows' error history meaningless: zeroed, in the same order as the offsets
    if (h->d_dither_hist) OHS_CUDA(cudaMemsetAsync(bus_hist(h), 0, bus_hist_bytes(h), h->stream));
    h->bus_hist_live = false;
    h->h_group_first.swap(v);
    return OHS_OK;
}

int ohs_num_groups(ohs_engine* h, int* out) {
    OHS_CHECK_HANDLE(h);
    if (!out) return fail(OHS_ERR_INVALID, "null output");
    *out = n_groups(h);
    return OHS_OK;
}

// ---- collectives ----------------------------------------------------------------------------------------------
namespace {
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

const NcclApi* nccl_api() {
    static NcclApi api;
    static std::atomic<int> state{0};   // 0 untried, 1 ready, -1 failed
    static std::atomic_flag busy = ATOMIC_FLAG_INIT;
    if (state.load(std::memory_order_acquire) == 0) {
        while (busy.test_and_set(std::memory_order_acquire)) {}
        if (state.load(std::memory_order_relaxed) == 0) {
            // a process that already holds an NCCL (e.g. torch's bundled one) gets that one back by SONAME
            void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
            if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
            bool ok = lib != nullptr;
            auto sym = [&](const char* name) { void* p = lib ? dlsym(lib, name) : nullptr; ok = ok && p; return p; };
            api.lib = lib;
            api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
            api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
            api.Reduce = (decltype(api.Reduce))sym("ncclReduce");
            api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
            api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
            api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
            state.store(ok ? 1 : -1, std::memory_order_release);
        }
        busy.clear(std::memory_order_release);
    }
    return state.load(std::memory_order_acquire) == 1 ? &api : nullptr;
}

#define OHS_NCCL(api, expr)                                                                                          \
    do {                                                                                                             \
        ncclResult_t _r = (expr);                                                                                    \
        if (_r != ncclSuccess) return fail(OHS_ERR_NCCL, "%s failed: %s", #expr, (api)->GetErrorString(_r));          \
    } while (0)
}  // namespace

struct ohs_comm {
    ncclComm_t comm = nullptr;
    int world = 1, rank = 0, device = 0;
};

int ohs_comm_unique_id(void* id128) {
    static_assert(sizeof(ncclUniqueId) == OHS_COMM_ID_BYTES, "ncclUniqueId size");
    if (!id128) return fail(OHS_ERR_INVALID, "null output");
    const NcclApi* api = nccl_api();
    if (!api) return fail(OHS_ERR_NCCL, "libnccl.so.2 could not be opened: %s", dlerror() ? dlerror() : "symbol missing");
    ncclUniqueId id;
    OHS_NCCL(api, api->GetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
    return OHS_OK;
}

int ohs_comm_create(ohs_comm** out, int world, int rank, int device, const void* id128) {
    if (!out || !id128) return fail(OHS_ERR_INVALID, "null argument");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world) return fail(OHS_ERR_INVALID, "rank %d outside world %d", rank, world);
    const NcclApi* api = nccl_api();
    if (!api) return fail(OHS_ERR_NCCL, "libnccl.so.2 could not be opened");
    OHS_CUDA(cudaSetDevice(device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ohs_comm* c = new ohs_comm();
    c->world = world; c->rank = rank; c->device = device;
    ncclResult_t r = api->CommInitRank(&c->comm, world, id, rank);
    if (r != ncclSuccess) { delete c; return fail(OHS_ERR_NCCL, "ncclCommInitRank failed: %s", api->GetErrorString(r)); }
    *out = c;
    return OHS_OK;
}

int ohs_comm_destroy(ohs_comm* c) {
    if (!c) return OHS_OK;
    const NcclApi* api = nccl_api();
    if (api && c->comm) { cudaSetDevice(c->device); api->CommDestroy(c->comm); }
    delete c;
    return OHS_OK;
}

int ohs_broadcast_hrir(ohs_engine* h, ohs_comm* c, int root) {
    OHS_CHECK_HANDLE(h);
    if (!c) return fail(OHS_ERR_INVALID, "null communicator");
    if (root < 0 || root >= c->world) return fail(OHS_ERR_INVALID, "root %d outside world %d", root, c->world);
    if (c->device != h->cfg.device) return fail(OHS_ERR_INVALID, "communicator is on device %d, engine on %d", c->device, h->cfg.device);
    const NcclApi* api = nccl_api();
    if (!api) return fail(OHS_ERR_NCCL, "libnccl.so.2 could not be opened");
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    const int n_sets = h->cfg.n_hrir_sets;
    if (c->rank == root) {
        int rc = commit_filters(h);
        if (rc) return rc;
    } else {
        int rc = upload_bindings(h);
        if (rc) return rc;
    }
    OHS_NCCL(api, api->GroupStart());
    OHS_NCCL(api, api->Broadcast(h->d_filt, h->d_filt, h->filt_bytes / sizeof(float), ncclFloat32, root, c->comm, h->stream));
    OHS_NCCL(api, api->Broadcast(h->d_set_parts, h->d_set_parts, (size_t)n_sets, ncclInt32, root, c->comm, h->stream));
    OHS_NCCL(api, api->GroupEnd());
    if (c->rank != root) {
        OHS_CUDA(cudaMemcpyAsync(h->h_set_parts.data(), h->d_set_parts, sizeof(int) * n_sets, cudaMemcpyDeviceToHost, h->stream));
        OHS_CUDA(cudaStreamSynchronize(h->stream));
        for (int s = 0; s < n_sets; ++s) {
            const int parts = h->h_set_parts[s];
            if (parts < 1 || parts > h->pmax) return fail(OHS_ERR_INVALID, "received partition count %d for HRIR set %d (capacity %d)", parts, s, h->pmax);
            for (int p = 0; p < 4; ++p) h->h_path_parts[(size_t)s * 4 + p] = parts;
            h->set_dirty[s] = 0;
            h->set_external[s] = 1;
        }
        h->any_set_dirty = false;
        // a freshly received response starts from empty history, like set_ir (src/dsp/convolution.rs:135-138)
        int rc = clear_history(h, false);
        if (rc) return rc;
        h->head = 0;
    }
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    return OHS_OK;
}

int ohs_reduce_bus(ohs_engine* h, ohs_comm* c, float* d_bus, size_t n_floats, int root) {
    OHS_CHECK_HANDLE(h);
    if (!c || !d_bus) return fail(OHS_ERR_INVALID, "null argument");
    if (root < 0 || root >= c->world) return fail(OHS_ERR_INVALID, "root %d outside world %d", root, c->world);
    const NcclApi* api = nccl_api();
    if (!api) return fail(OHS_ERR_NCCL, "libnccl.so.2 could not be opened");
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    OHS_NCCL(api, api->Reduce(d_bus, d_bus, n_floats, ncclFloat32, ncclSum, root, c->comm, h->stream));
    return OHS_OK;
}

int ohs_host_alloc(void** p, size_t bytes) {
    if (!p) return fail(OHS_ERR_INVALID, "null output");
    OHS_CUDA(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
    return OHS_OK;
}

int ohs_host_free(void* p) {
    if (p) OHS_CUDA(cudaFreeHost(p));
    return OHS_OK;
}

}  // extern "C"

namespace {

// Host-pointer flavour: time chunks are staged through three slots in HBM; copy-in, kernels and copy-out of consecutive
// chunks overlap on three CUDA streams.  Integer PCM crosses the link as PCM and is converted in HBM.  Per chunk: copy-in
// (PCM rows into the slot's PCM buffer, or f32 rows straight into its f32 buffer), chunk_step on the f32 buffer, and
// copy-out of the step's output side: the PCM buffer, the f32 buffer, or for a bus (ohs_process_grouped_pcm) the slot's
// bus rows, so that only those 2 * n_groups rows cross back.  ohs_process is the F32 -> F32 case.
int process_host_chunks(ohs_engine* h, const Rows& in, const Rows& out, size_t n_frames) {
    int rc = OHS_OK;
    const size_t rows = (size_t)h->cfg.n_streams * 2, bi = in.sample_bytes();
    const bool pcm_in = in.fmt != OHS_FMT_F32, int_out = out.fmt != OHS_FMT_F32, pcm_out = int_out && !out.bus;
    const size_t bo = out.bus ? sizeof(float) : out.sample_bytes();   // a bus call's stream rows stay f32
    // about stage_bytes per copy of the wider side's rows: 24 MiB by default, measured best on PCIe Gen5 x16 with both
    // directions busy (tools/e2e_probe.py)
    const size_t chunk = chunk_frames(h, n_frames, h->stage_bytes, std::max(bi, bo));
    if ((rc = grow_buffers(h, h->d_stage, kPipe, h->stage_cap, rows * chunk * sizeof(float))) ||
        (rc = grow_buffers(h, h->d_pcm_stage, kPipe, h->pcm_stage_cap, rows * chunk * std::max(pcm_in ? bi : 0, pcm_out ? bo : 0))) ||
        (out.bus && (rc = grow_buffers(h, h->d_bus_stage, kPipe, h->bus_stage_cap, out.count(h) * chunk * sizeof(float)))))
        return rc;
    if (!h->bypass) {
        rc = commit_filters(h);
        if (rc) return rc;
    }
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    size_t done = 0;
    int idx = 0;
    bool used[kPipe] = {false, false, false};
    while (done < n_frames) {
        const size_t n = std::min(chunk, n_frames - done);
        const size_t pitch = round_up(n, 4), pcm_pitch = round_up(n, 16);   // 16-byte aligned rows in every format
        const int b = idx % kPipe;
        float* x = h->d_stage[b];
        void* q = h->d_pcm_stage[b];
        // the step's sides in the slot; an integer bus is packed rows of pcm_pitch frames in the bus buffer
        const Rows si{pcm_in ? q : x, in.fmt, pcm_in ? pcm_pitch : pitch};
        const Rows so{out.bus ? h->d_bus_stage[b] : pcm_out ? q : x, out.fmt, int_out ? pcm_pitch : pitch, out.bus};
        const size_t ob = so.sample_bytes();
        if (used[b]) OHS_CUDA(cudaStreamWaitEvent(h->h2d, h->ev_out[b], 0));  // buffers free once their copy-out finished
        OHS_CUDA(cudaMemcpy2DAsync(si.p, si.stride * bi, in.from(done).p, in.stride * bi, n * bi, rows, cudaMemcpyHostToDevice, h->h2d));
        OHS_CUDA(cudaEventRecord(h->ev_in[b], h->h2d));
        OHS_CUDA(cudaStreamWaitEvent(h->stream, h->ev_in[b], 0));
        if ((rc = chunk_step(h, si, x, pitch, n, done, !h->bypass, so))) return rc;
        OHS_CUDA(cudaEventRecord(h->ev_comp[b], h->stream));
        OHS_CUDA(cudaStreamWaitEvent(h->d2h, h->ev_comp[b], 0));
        OHS_CUDA(cudaMemcpy2DAsync(out.from(done).p, out.stride * ob, so.p, so.stride * ob, n * ob, so.count(h), cudaMemcpyDeviceToHost,
                                   h->d2h));
        OHS_CUDA(cudaEventRecord(h->ev_out[b], h->d2h));
        used[b] = true;
        done += n;
        ++idx;
    }
    OHS_CUDA(cudaStreamSynchronize(h->d2h));
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    return OHS_OK;
}

// ohs_process_pcm and ohs_process_grouped_pcm past validation
int process_host_impl(ohs_engine* h, const Rows& in, const Rows& out, size_t n_frames) {
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    if (n_frames == 0) return OHS_OK;
    if (h->bypass && !out.bus && in.fmt == out.fmt) {   // nothing to convert: the rows as they are
        const size_t rows = (size_t)h->cfg.n_streams * 2, bytes = in.sample_bytes();
        if (in.p != out.p)
            for (size_t r = 0; r < rows; ++r)
                memcpy(static_cast<unsigned char*>(out.p) + r * out.stride * bytes, static_cast<const unsigned char*>(in.p) + r * in.stride * bytes,
                       n_frames * bytes);
    } else if (const int rc = process_host_chunks(h, in, out, n_frames)) {
        return rc;
    }
    if (moves_dither(out)) h->dither_pos += n_frames;
    return OHS_OK;
}

}  // namespace

extern "C" {

int ohs_process_pcm(ohs_engine* h, const void* in, int in_format, void* out, int out_format, size_t n_frames, size_t row_stride) {
    OHS_CHECK_HANDLE(h);
    const Rows src{const_cast<void*>(in), in_format, row_stride}, dst{out, out_format, row_stride};
    const int rc = check_call(h, src, dst, n_frames, kWholeBlocks | kSeparateIfConverted);
    if (rc) return rc;
    return process_host_impl(h, src, dst, n_frames);
}

int ohs_process_grouped_pcm(ohs_engine* h, const void* in, int in_format, void* bus, int bus_format, size_t n_frames, size_t row_stride,
                            size_t bus_stride) {
    OHS_CHECK_HANDLE(h);
    const Rows src{const_cast<void*>(in), in_format, row_stride}, dst{bus, bus_format, bus_stride, true};
    const int rc = check_call(h, src, dst, n_frames, kWholeBlocks | kSeparate);
    if (rc) return rc;
    return process_host_impl(h, src, dst, n_frames);
}

int ohs_process_grouped(ohs_engine* h, const void* in, int in_format, float* bus, size_t n_frames, size_t row_stride,
                        size_t bus_stride) {
    return ohs_process_grouped_pcm(h, in, in_format, bus, OHS_FMT_F32, n_frames, row_stride, bus_stride);
}

int ohs_process(ohs_engine* h, const float* in, float* out, size_t n_frames, size_t row_stride) {
    return ohs_process_pcm(h, in, OHS_FMT_F32, out, OHS_FMT_F32, n_frames, row_stride);
}

// The reference's FIFO adaptation around whole engine blocks (src/dsp/convolution.rs:141-182): append the host block,
// run every complete engine block, hand back n frames if that many are ready, else silence (and keep what is queued).
int ohs_process_fifo(ohs_engine* h, const float* in, float* out, size_t n_frames, size_t row_stride) {
    OHS_CHECK_HANDLE(h);
    int rc = check_call(h, {const_cast<float*>(in), OHS_FMT_F32, row_stride}, {out, OHS_FMT_F32, row_stride}, n_frames, 0);
    if (rc) return rc;
    const size_t rows = (size_t)h->cfg.n_streams * 2;
    if (h->bypass) {
        if (in != out) for (size_t r = 0; r < rows; ++r) memcpy(out + r * row_stride, in + r * row_stride, n_frames * sizeof(float));
        return OHS_OK;
    }
    const size_t need = std::max(h->fifo_in_len, h->fifo_out_len) + n_frames + (size_t)h->B;
    if (need > h->fifo_cap) {
        const size_t cap = std::max(need, h->fifo_cap * 2);
        std::vector<float> ni(rows * cap, 0.f), no(rows * cap, 0.f);
        for (size_t r = 0; r < rows; ++r) {
            if (h->fifo_in_len) memcpy(&ni[r * cap], &h->fifo_in[r * h->fifo_cap], h->fifo_in_len * sizeof(float));
            if (h->fifo_out_len) memcpy(&no[r * cap], &h->fifo_out[r * h->fifo_cap], h->fifo_out_len * sizeof(float));
        }
        h->fifo_in.swap(ni); h->fifo_out.swap(no); h->fifo_cap = cap;
    }
    const size_t cap = h->fifo_cap;
    for (size_t r = 0; r < rows; ++r) memcpy(&h->fifo_in[r * cap + h->fifo_in_len], in + r * row_stride, n_frames * sizeof(float));
    h->fifo_in_len += n_frames;
    const size_t whole = (h->fifo_in_len / h->B) * h->B;
    if (whole) {
        // EQ runs inside the engine on the same whole blocks; in the reference the EQ sees the host buffer before the
        // FIFO (src/lib.rs:1194-1199) — per-sample filtering, so the result is identical.
        std::vector<float> tmp(rows * whole);
        for (size_t r = 0; r < rows; ++r) memcpy(&tmp[r * whole], &h->fifo_in[r * cap], whole * sizeof(float));
        rc = ohs_process(h, tmp.data(), tmp.data(), whole, whole);
        if (rc) return rc;
        for (size_t r = 0; r < rows; ++r) {
            memcpy(&h->fifo_out[r * cap + h->fifo_out_len], &tmp[r * whole], whole * sizeof(float));
            memmove(&h->fifo_in[r * cap], &h->fifo_in[r * cap + whole], (h->fifo_in_len - whole) * sizeof(float));
        }
        h->fifo_in_len -= whole;
        h->fifo_out_len += whole;
    }
    if (h->fifo_out_len >= n_frames) {
        for (size_t r = 0; r < rows; ++r) {
            memcpy(out + r * row_stride, &h->fifo_out[r * cap], n_frames * sizeof(float));
            memmove(&h->fifo_out[r * cap], &h->fifo_out[r * cap + n_frames], (h->fifo_out_len - n_frames) * sizeof(float));
        }
        h->fifo_out_len -= n_frames;
    } else {
        for (size_t r = 0; r < rows; ++r) memset(out + r * row_stride, 0, n_frames * sizeof(float));  // :176-181
    }
    return OHS_OK;
}

// ---- state export / import ----------------------------------------------------------------------------------
// blob = StateHeader | delay line | overlap-save blocks | biquad states | FIFO residue (input rows, output rows)
//        [ | dither position (uint64) | error history float[2S][OHS_MAX_SHAPE_TAPS] ]  when flags has kStateDither
//        [ | n_groups (int32) | 0 (int32) | bus error history float[2G][OHS_MAX_SHAPE_TAPS] ]  when flags has kStateBus
namespace {
struct StateHeader {
    uint32_t magic;      // 'OHSS'
    int32_t abi, n_streams, n_bands, pmax, block, head, flags;
    uint64_t fifo_in_len, fifo_out_len, total_bytes;
};
constexpr uint32_t kStateMagic = 0x5353484Fu;
constexpr int32_t kStateDither = 1;   // the dither section follows the FIFO residue
constexpr int32_t kStateBus = 2;      // the bus section follows the dither section (dither on and a bus encoded)
size_t dither_state_bytes(const ohs_engine* h) { return sizeof(uint64_t) + sizeof(float) * (size_t)h->cfg.n_streams * 2 * OHS_MAX_SHAPE_TAPS; }
size_t bus_state_floats(int groups) { return (size_t)groups * 2 * OHS_MAX_SHAPE_TAPS; }
size_t state_need(const ohs_engine* h, size_t fifo_in, size_t fifo_out, bool dither) {
    const size_t S = h->cfg.n_streams;
    return sizeof(StateHeader) + sizeof(float2) * S * h->pmax * h->N + sizeof(float2) * S * h->B + sizeof(float4) * S * kMaxBands +
           sizeof(float) * S * 2 * (fifo_in + fifo_out) + (dither ? dither_state_bytes(h) : 0);
}
// the blob carries the bus rows' history only while it means something: dither on and a bus encoded since it was zeroed
bool bus_state(const ohs_engine* h) { return h->dither_mode != OHS_DITHER_OFF && h->bus_hist_live; }
size_t bus_state_bytes(int groups) { return 2 * sizeof(int32_t) + sizeof(float) * bus_state_floats(groups); }
}  // namespace

int ohs_state_bytes(ohs_engine* h, size_t* bytes) {
    OHS_CHECK_HANDLE(h);
    if (!bytes) return fail(OHS_ERR_INVALID, "null output");
    *bytes = state_need(h, h->fifo_in_len, h->fifo_out_len, h->dither_mode != OHS_DITHER_OFF) + (bus_state(h) ? bus_state_bytes(n_groups(h)) : 0);
    return OHS_OK;
}

int ohs_state_export(ohs_engine* h, void* host_buf, size_t bytes) {
    OHS_CHECK_HANDLE(h);
    const bool dither = h->dither_mode != OHS_DITHER_OFF, bus = bus_state(h);
    const int G = n_groups(h);
    const size_t need = state_need(h, h->fifo_in_len, h->fifo_out_len, dither) + (bus ? bus_state_bytes(G) : 0);
    if (!host_buf || bytes < need) return fail(OHS_ERR_INVALID, "state buffer too small (%zu < %zu)", bytes, need);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    int rc = commit_filters(h);
    if (rc) return rc;
    rc = ensure_ring(h);   // the blob carries the delay-line ring
    if (rc) return rc;
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    unsigned char* p = (unsigned char*)host_buf;
    const size_t S = h->cfg.n_streams;
    StateHeader hdr{kStateMagic, OHS_ABI_VERSION, h->cfg.n_streams, kMaxBands, h->pmax, h->B, h->head,
                    (dither ? kStateDither : 0) | (bus ? kStateBus : 0),
                    (uint64_t)h->fifo_in_len, (uint64_t)h->fifo_out_len, (uint64_t)need};
    memcpy(p, &hdr, sizeof(hdr)); p += sizeof(hdr);
    const size_t n0 = sizeof(float2) * S * h->pmax * h->N, n1 = sizeof(float2) * S * h->B, n2 = sizeof(float4) * S * kMaxBands;
    OHS_CUDA(cudaMemcpy(p, h->d_fdl, n0, cudaMemcpyDeviceToHost)); p += n0;
    OHS_CUDA(cudaMemcpy(p, h->d_prev, n1, cudaMemcpyDeviceToHost)); p += n1;
    OHS_CUDA(cudaMemcpy(p, h->d_eqs, n2, cudaMemcpyDeviceToHost)); p += n2;
    // what ohs_process_fifo has queued (src/dsp/convolution.rs:73-76 input_buffer / output_buffer), row by row
    for (size_t r = 0; r < S * 2; ++r) { memcpy(p, h->fifo_in.data() + r * h->fifo_cap, h->fifo_in_len * sizeof(float)); p += h->fifo_in_len * sizeof(float); }
    for (size_t r = 0; r < S * 2; ++r) { memcpy(p, h->fifo_out.data() + r * h->fifo_cap, h->fifo_out_len * sizeof(float)); p += h->fifo_out_len * sizeof(float); }
    if (dither) {
        const uint64_t pos = h->dither_pos;
        memcpy(p, &pos, sizeof(pos)); p += sizeof(pos);
        OHS_CUDA(cudaMemcpy(p, h->d_dither_hist, dither_state_bytes(h) - sizeof(pos), cudaMemcpyDeviceToHost));
        p += dither_state_bytes(h) - sizeof(pos);
    }
    if (bus) {
        const int32_t head[2] = {G, 0};
        memcpy(p, head, sizeof(head)); p += sizeof(head);
        OHS_CUDA(cudaMemcpy(p, bus_hist(h), sizeof(float) * bus_state_floats(G), cudaMemcpyDeviceToHost));
    }
    return OHS_OK;
}

int ohs_state_import(ohs_engine* h, const void* host_buf, size_t bytes) {
    OHS_CHECK_HANDLE(h);
    if (!host_buf || bytes < sizeof(StateHeader)) return fail(OHS_ERR_INVALID, "state blob too small for its header");
    const unsigned char* p = (const unsigned char*)host_buf;
    StateHeader hdr;
    memcpy(&hdr, p, sizeof(hdr)); p += sizeof(hdr);
    if (hdr.magic != kStateMagic || hdr.abi != OHS_ABI_VERSION) return fail(OHS_ERR_INVALID, "not a state blob of ABI version %d", OHS_ABI_VERSION);
    if (hdr.n_streams != h->cfg.n_streams || hdr.n_bands != kMaxBands || hdr.pmax != h->pmax || hdr.block != h->B)
        return fail(OHS_ERR_INVALID, "state blob geometry (%d streams, %d partitions, block %d) does not match this engine (%d, %d, %d)",
                    hdr.n_streams, hdr.pmax, hdr.block, h->cfg.n_streams, h->pmax, h->B);
    if (hdr.head < 0 || hdr.head >= h->pmax) return fail(OHS_ERR_INVALID, "state blob ring head %d outside 0..%d", hdr.head, h->pmax - 1);
    const size_t limit = (size_t)1 << 32;
    if (hdr.fifo_in_len > limit || hdr.fifo_out_len > limit) return fail(OHS_ERR_INVALID, "state blob FIFO lengths are implausible");
    if (hdr.flags & ~(kStateDither | kStateBus)) return fail(OHS_ERR_INVALID, "state blob has unknown flags 0x%x", (unsigned)hdr.flags);
    const bool dither = (hdr.flags & kStateDither) != 0, bus = (hdr.flags & kStateBus) != 0;
    if (bus && !dither) return fail(OHS_ERR_INVALID, "state blob carries bus dither history without dither state");
    if (dither != (h->dither_mode != OHS_DITHER_OFF))
        return fail(OHS_ERR_INVALID, dither ? "state blob carries dither state but this engine's dither is off"
                                            : "state blob carries no dither state but this engine dithers (ohs_set_dither first)");
    size_t need = state_need(h, (size_t)hdr.fifo_in_len, (size_t)hdr.fifo_out_len, dither);
    const int G = n_groups(h);
    if (bus) {
        int32_t head[2] = {0, 0};
        if (bytes >= need + sizeof(head)) memcpy(head, (const unsigned char*)host_buf + need, sizeof(head));
        if (head[0] != G || head[1] != 0)
            return fail(OHS_ERR_INVALID, "state blob's bus history is for %d groups, this engine has %d", head[0], G);
        need += bus_state_bytes(G);
    }
    if (hdr.total_bytes != need || bytes != need) return fail(OHS_ERR_INVALID, "state blob is %zu bytes, header says %llu, geometry needs %zu", bytes, (unsigned long long)hdr.total_bytes, need);
    OHS_CUDA(cudaSetDevice(h->cfg.device));
    int rc = commit_filters(h);  // pending set_ir would otherwise clear the imported history later
    if (rc) return rc;
    OHS_CUDA(cudaStreamSynchronize(h->stream));
    const size_t S = h->cfg.n_streams;
    const size_t n0 = sizeof(float2) * S * h->pmax * h->N, n1 = sizeof(float2) * S * h->B, n2 = sizeof(float4) * S * kMaxBands;
    h->head = hdr.head;
    h->ring_valid = true; h->zlin_valid = false;
    OHS_CUDA(cudaMemcpy(h->d_fdl, p, n0, cudaMemcpyHostToDevice)); p += n0;
    OHS_CUDA(cudaMemcpy(h->d_prev, p, n1, cudaMemcpyHostToDevice)); p += n1;
    OHS_CUDA(cudaMemcpy(h->d_eqs, p, n2, cudaMemcpyHostToDevice)); p += n2;
    const size_t fi = (size_t)hdr.fifo_in_len, fo = (size_t)hdr.fifo_out_len;
    const size_t cap = std::max(fi, fo) + (size_t)h->B;
    h->fifo_in.assign(S * 2 * cap, 0.f); h->fifo_out.assign(S * 2 * cap, 0.f); h->fifo_cap = cap;
    for (size_t r = 0; r < S * 2; ++r) { memcpy(h->fifo_in.data() + r * cap, p, fi * sizeof(float)); p += fi * sizeof(float); }
    for (size_t r = 0; r < S * 2; ++r) { memcpy(h->fifo_out.data() + r * cap, p, fo * sizeof(float)); p += fo * sizeof(float); }
    h->fifo_in_len = fi; h->fifo_out_len = fo;
    if (dither) {
        uint64_t pos;
        memcpy(&pos, p, sizeof(pos)); p += sizeof(pos);
        OHS_CUDA(cudaMemcpy(h->d_dither_hist, p, dither_state_bytes(h) - sizeof(pos), cudaMemcpyHostToDevice));
        p += dither_state_bytes(h) - sizeof(pos);
        h->dither_pos = pos;
        // the bus rows' history: the blob's, or zeros for a blob written before any bus encode
        if (bus) OHS_CUDA(cudaMemcpy(bus_hist(h), p + 2 * sizeof(int32_t), sizeof(float) * bus_state_floats(G), cudaMemcpyHostToDevice));
        else OHS_CUDA(cudaMemset(bus_hist(h), 0, bus_hist_bytes(h)));
    }
    h->bus_hist_live = bus;
    return OHS_OK;
}

}  // extern "C"
