/*
 * ohs.h — C ABI of the B200-native Open Headstage DSP engine (libohs_cuda.so).
 *
 * This is the drop-in boundary for ONE path of KiloHertzian/Open-Headstage: the DSP core that
 * `Plugin::process` runs per host buffer (reference src/lib.rs:1156-1211):
 *
 *     10-band parametric EQ  ->  4-path binaural partitioned convolution  ->  output gain
 *     (src/dsp/parametric_eq.rs)   (src/dsp/convolution.rs)                   (src/lib.rs:1202-1207)
 *
 * re-posed as a batched renderer: one engine handle owns `n_streams` independent stereo chains (each the
 * equivalent of one reference `ConvolutionEngine` + one `StereoParametricEQ`), resident in HBM, processed
 * together by hand-written sm_100a kernels.  Plain pointers and sizes only; no C++/torch types.
 *
 * Every entry point cites the reference interface it replaces.  The Rust-side binding a maintainer of the
 * reference would add (extern "C" block, wrapper structs with the reference's method names, build.rs
 * additions) is in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 (OHS_OK) or a negative ohs_status; ohs_last_error() gives the message of the
 *     last failure on the calling thread.  Nothing throws or aborts across the boundary (the reference
 *     panics on bad EQ parameters, src/dsp/parametric_eq.rs:111; here that is OHS_ERR_INVALID).
 *   - audio is planar f32: in/out[(stream*2 + channel) * row_stride + frame], channel 0 = left, 1 = right
 *     (reference: `let [left, right] = buffer.as_slice()`, src/lib.rs:1175).
 *   - one handle = one CUDA stream; a handle is not re-entrant (the reference API is `&mut self`); distinct
 *     handles are independent.
 *   - there is no CPU fallback: if no CUDA device is usable, ohs_create fails.
 *   - the environment is read once, in ohs_create: OHS_STREAMS_PER_CTA (1..7, which render-kernel instantiation the
 *     handle uses; default: chosen from n_streams and the SM count), OHS_TIME_BATCH (0 = ohs_set_time_batch(h, 0)),
 *     OHS_STAGE_MB (staging chunk of the host-pointer path, default 24), OHS_PDL (0 = no programmatic dependent launches),
 *     OHS_LATENCY_BLOCKS (launches of up to this many blocks run the render kernel's latency variant, default 2).
 */
#ifndef OHS_H
#define OHS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OHS_ABI_VERSION 2

typedef enum ohs_status {
    OHS_OK = 0,
    OHS_ERR_INVALID = -1,     /* bad argument (null handle, index out of range, unsupported block size, ...) */
    OHS_ERR_CUDA = -2,        /* a CUDA runtime call failed; message holds cudaGetErrorString */
    OHS_ERR_NO_DEVICE = -3,   /* no usable CUDA device (no CPU fallback exists) */
    OHS_ERR_NYQUIST = -4,     /* EQ design: 2*fc > fs  (biquad Errors::OutsideNyquist) */
    OHS_ERR_NEGATIVE_Q = -5,  /* EQ design: q < 0      (biquad Errors::NegativeQ) */
    OHS_ERR_ALIGNMENT = -6,   /* device/host audio pointer or row stride not 16-byte aligned */
    OHS_ERR_NCCL = -7         /* libnccl could not be opened, or an NCCL call failed; message holds ncclGetErrorString */
} ohs_status;

/* src/dsp/convolution.rs:26-33  enum ConvolutionPath { Lsl, Lsr, Rsl, Rsr }
 * (L/R speaker -> l/r ear; out_l = Lsl + Rsl, out_r = Lsr + Rsr, :229-230) */
typedef enum ohs_path { OHS_PATH_LSL = 0, OHS_PATH_LSR = 1, OHS_PATH_RSL = 2, OHS_PATH_RSR = 3 } ohs_path;

/* src/dsp/parametric_eq.rs:25-35  enum FilterType (declaration order) */
typedef enum ohs_filter_type {
    OHS_FILTER_PEAK = 0, OHS_FILTER_LOWSHELF = 1, OHS_FILTER_HIGHSHELF = 2, OHS_FILTER_LOWPASS = 3,
    OHS_FILTER_HIGHPASS = 4, OHS_FILTER_BANDPASS = 5, OHS_FILTER_NOTCH = 6, OHS_FILTER_ALLPASS = 7
} ohs_filter_type;

#define OHS_ALL (-1)        /* "every stream" for the per-stream setters */
#define OHS_MAX_BANDS 10    /* NUM_EQ_BANDS, src/lib.rs:40 */

/* Replaces the compile-time constants and constructor arguments of the reference:
 *   BLOCK_SIZE / FFT_SIZE (src/dsp/convolution.rs:22-23), NUM_EQ_BANDS (src/lib.rs:40),
 *   StereoParametricEQ::new(num_bands, sample_rate) (src/dsp/parametric_eq.rs:132). */
typedef struct ohs_config {
    int32_t n_streams;    /* independent stereo chains held by this engine (>= 1) */
    int32_t block;        /* engine block B in frames: 64, 128, 256, 512 or 1024; FFT size is 2*B */
    int32_t max_taps;     /* longest impulse response set_ir will be given; sizes the delay line: P = ceil(max_taps/B) */
    int32_t n_bands;      /* EQ bands per channel, 0..OHS_MAX_BANDS */
    int32_t n_hrir_sets;  /* distinct 4-path HRIR sets (>= 1); every stream starts bound to set 0 */
    int32_t n_eq_sets;    /* distinct EQ coefficient sets (>= 1); every stream starts bound to set 0 */
    int32_t device;       /* CUDA device ordinal */
    float sample_rate;    /* Hz; used by ohs_eq_update_band */
} ohs_config;

typedef struct ohs_engine ohs_engine;

/* ---- lifecycle ------------------------------------------------------------------------------------------ */
/* ConvolutionEngine::new (src/dsp/convolution.rs:87-108) + StereoParametricEQ::new (src/dsp/parametric_eq.rs:132-142)
 * for n_streams chains: every path's IR is silence (one all-zero partition, :44-65), every band is
 * PeakingEQ(0 dB)@20 Hz Q 0.707 and disabled (:63-76), gain 1, eq_enable 0 (src/lib.rs:433-434), bypass 0. */
int ohs_create(const ohs_config* cfg, ohs_engine** out);
int ohs_destroy(ohs_engine* h);
int ohs_abi_version(void);
const char* ohs_last_error(void);

/* ---- HRIR set-up ------------------------------------------------------------------------------------------ */
/* ConvolutionEngine::set_ir(path, &[f32]) (src/dsp/convolution.rs:111-139).  The IR is cut into B-frame chunks,
 * each zero-padded to 2B and transformed on the GPU; len == 0 gives one silent partition (:114-118).
 * As in the reference (:135-138) the convolution history of every stream bound to `hrir_set` is cleared.
 * (Difference, documented in DESIGN.md: the reference clears only the history of the one path; here the delay
 * line is shared by the four paths, so all four restart.  Identical whenever IRs are set before streaming.) */
int ohs_set_ir(ohs_engine* h, int hrir_set, int path, const float* ir, size_t len);
/* ir_fft_partitions.len() of that path, as asserted by the reference test (src/dsp/convolution.rs:395-399). */
int ohs_num_partitions(ohs_engine* h, int hrir_set, int path, int* out);
/* Which HRIR set a stream (or OHS_ALL) convolves with; clears that stream's convolution history. */
int ohs_bind_stream_hrir(ohs_engine* h, int stream, int hrir_set);
/* ---- moving sources (an extension: the reference reads its speaker angles and never applies them) -------------
 * A stream changes HRIR sets WITHOUT losing its history, crossfaded over one engine block.  Every stream has a set
 * set(t) for every block t it convolves; block t is a transition when set(t) != set(t-1) (for a call's first block,
 * set(t-1) is the binding before the call).  With y_X[t] the output block t of a stream bound to set X since its
 * history began (gain included, exactly what the engine renders without moves):
 *   non-transition block:  out[t] = y_set(t)[t]
 *   transition block:      a = y_set(t-1)[t], b = y_set(t)[t], w[n] = (2n+1)/(2B), n = 0..B-1,
 *                          out[t][n] = a[n] + w[n]*(b[n] - a[n]), each operation rounded on its own in f32
 * A switch never touches history (EQ state, overlap-save block, delay line): after its transition block a moved
 * stream is bit-identical to one bound to the target set from the start.  Sets with different partition counts mix
 * freely.  Pending moves and schedules are configuration, like bindings: they are not part of the state blob.
 *
 * Per-buffer form (head tracking, host automation): records a pending target for `stream` (or OHS_ALL).  The next
 * engine block that stream convolves crossfades from its binding to the target (ohs_process_device, the first chunk
 * of ohs_process, the first whole engine block ohs_process_fifo renders, possibly in a later call); the binding is
 * the target from then on.  Moving to the binding, or back to it before any call, is a no-op; ohs_bind_stream_hrir
 * cancels the move (and clears the history, as always).  Bypassed calls and calls with the convolution disabled
 * leave the move pending.  The commit of set_ir work at the start of a call clears the streams BOUND to re-committed
 * sets before moves apply: write the new direction into a spare set, then move to it, and nothing is cleared. */
int ohs_move_stream_hrir(ohs_engine* h, int stream, int hrir_set);
/* Device-resident filter spectra of all sets, for a caller-side NCCL broadcast (SURVEY.md §8e): pointer and byte
 * size of the table the render kernel reads.  ohs_commit_filters uploads pending set_ir work first; after an
 * external overwrite (broadcast receive) call ohs_mark_filters_external so pending host IRs do not overwrite it. */
int ohs_commit_filters(ohs_engine* h);
int ohs_filter_table(ohs_engine* h, void** dev_ptr, size_t* bytes);
int ohs_mark_filters_external(ohs_engine* h, int hrir_set, int partitions);

/* ---- EQ --------------------------------------------------------------------------------------------------- */
/* biquad 0.4.2 Coefficients::<f32>::from_params as called by BiquadFilter::update_coeffs
 * (src/dsp/parametric_eq.rs:86-114).  Pure host function; out = {b0, b1, b2, a1, a2} normalised by a0. */
int ohs_eq_design(int filter_type, float fs, float fc, float q, float gain_db, float out[5]);
/* StereoParametricEQ::update_band_coeffs(band_idx, sample_rate, &BandConfig) (src/dsp/parametric_eq.rs:144-164):
 * same coefficients and `enabled` for left and right, filter state kept.  band >= n_bands is ignored (returns OK)
 * exactly like the reference (:145).  Uses cfg.sample_rate. */
int ohs_eq_update_band(ohs_engine* h, int eq_set, int band, int filter_type, float fc, float q, float gain_db, int enabled);
/* Same, with the five coefficients supplied as data. */
int ohs_eq_set_band(ohs_engine* h, int eq_set, int band, const float coeffs[5], int enabled);
/* Bind a stream (or OHS_ALL) to an EQ set from its next call on.  The stream's biquad state is kept: the new set's bands
 * continue from the state the old set's bands left, as if update_band_coeffs had been called on every band. */
int ohs_bind_stream_eq(ohs_engine* h, int stream, int eq_set);
/* StereoParametricEQ::reset_all_bands_state (src/dsp/parametric_eq.rs:181-188; Plugin::reset src/lib.rs:1152-1154). */
int ohs_eq_reset(ohs_engine* h);
/* StereoParametricEQ::calculate_frequency_response(sample_rate, frequencies) (src/dsp/parametric_eq.rs:191-209):
 * |product over the enabled bands of `eq_set` of H(e^{j 2 pi f / sample_rate})|; sample_rate <= 0 means cfg.sample_rate. */
int ohs_eq_frequency_response(ohs_engine* h, int eq_set, float sample_rate, const float* freqs, float* out, size_t n);

/* ---- chain switches (Plugin::process, src/lib.rs:1169-1207) ------------------------------------------------- */
int ohs_set_eq_enable(ohs_engine* h, int enable);          /* params.eq_enable (:1179) */
int ohs_set_conv_enable(ohs_engine* h, int enable);        /* 0 = EQ/gain only: StereoParametricEQ::process_block alone */
int ohs_set_bypass(ohs_engine* h, int bypass);             /* params.master_bypass (:1169): output = input, state untouched */
int ohs_set_gain(ohs_engine* h, int stream, float gain);   /* output_gain, one value per call (:1202-1207); stream or OHS_ALL */
/* Clears convolution history (as a fresh ConvolutionEngine with the same IRs would have). */
int ohs_conv_reset(ohs_engine* h);
/* 0 keeps long responses on the block-by-block kernel (see ohs_process_device); default 1. */
int ohs_set_time_batch(ohs_engine* h, int enable);
/* Streams each CTA of the render kernel carries for this handle (which instantiation render_kernel<2*block, G> runs). */
int ohs_streams_per_cta(ohs_engine* h, int* out);
/* Set-up that would otherwise happen lazily inside the first process call of that size: uploads pending set_ir /
 * EQ / binding work and allocates the scratch (time-batched route, f32 rows of ohs_process_device_pcm) and, for
 * host_io != 0, the staging buffers that calls of n_frames frames need (of ohs_process and ohs_process_pcm alike).  Optional; lets a caller keep allocation out of a timed or real-time region, the
 * way Plugin::initialize (src/lib.rs:1124-1150) allocates before process() runs. */
int ohs_prepare(ohs_engine* h, size_t n_frames, int host_io);

/* ---- processing ------------------------------------------------------------------------------------------- */
/* The per-block process call: EQ (if enabled) -> convolution -> gain for every stream, n_frames frames each
 * (ConvolutionEngine::process_block src/dsp/convolution.rs:141 + StereoParametricEQ::process_block
 * src/dsp/parametric_eq.rs:166 + gain loop src/lib.rs:1202-1207).  n_frames must be a multiple of B: whole engine
 * blocks, i.e. the zero-latency case of the reference's FIFO (host block = multiple of BLOCK_SIZE).
 * in == out (in place) is allowed.  row_stride = frames between consecutive (stream, channel) rows (>= n_frames).
 * Device flavour: pointers are device memory on cfg.device; the call only enqueues on the engine's stream.
 * Long responses (>= 8 partitions) rendered >= 8 blocks per call take a time-batched route (EQ pre-pass on a second
 * stream of the handle, one chunk ahead of: forward transforms, a per-bin convolution along time, inverse transforms;
 * up to 2 GiB of scratch, allocated on first use or by ohs_prepare) with the same results within round-off and the
 * same state afterwards; the call is still ordered on the engine's stream alone; ohs_set_time_batch(h, 0) disables
 * it. */
int ohs_process_device(ohs_engine* h, const float* d_in, float* d_out, size_t n_frames, size_t row_stride);
/* ohs_process_device with a per-block set schedule (offline rendering of moving sources, definition above the
 * ohs_move_stream_hrir declaration): `sets` is HOST memory [n_streams][sets_stride], block t < n_frames/B of stream s
 * convolves with set sets[s*sets_stride + t].  Validated before anything is enqueued: a null pointer, sets_stride <
 * n_frames/B, a set out of range or the convolution disabled return OHS_ERR_INVALID with the engine untouched.  Pending
 * moves are superseded (block 0 compares with the binding); afterwards every stream is bound to its last column.  A
 * call with a transition runs the block-by-block kernel (long responses included: the time-batched route convolves
 * one set per stream and call); a schedule without one renders exactly like ohs_process_device.  Bypass behaves as
 * there and leaves the bindings unchanged. */
int ohs_process_device_scheduled(ohs_engine* h, const float* d_in, float* d_out, size_t n_frames, size_t row_stride,
                                 const int32_t* sets, size_t sets_stride);
/* Host flavour: pointers are host memory (pinned memory from ohs_host_alloc gives full PCIe speed); the call
 * stages time chunks through HBM with copies overlapped against the kernels and returns when `out` is complete. */
int ohs_process(ohs_engine* h, const float* in, float* out, size_t n_frames, size_t row_stride);
/* Arbitrary host-block length for ONE-call-per-host-buffer use: the reference's input/output FIFO adaptation
 * (src/dsp/convolution.rs:141-182) including the zero-filled output while fewer than n frames are ready. */
int ohs_process_fifo(ohs_engine* h, const float* in, float* out, size_t n_frames, size_t row_stride);

/* ---- integer PCM in and out (an extension: the reference processes f32 only) ------------------------------------
 * 16- and 24-bit audio converted on the GPU, so the host flavour moves 2 or 3 bytes per sample over PCIe instead of 4.
 * Layout as above: rows are (stream*2 + channel), row_stride counts FRAMES for both buffers, and row r of a buffer starts
 * at byte r * row_stride * bytes_per_sample(its format).
 *   decode   S16: q -> q * 2^-15        S24: q -> q * 2^-23        (both exact in f32)
 *   render   exactly what ohs_process / ohs_process_device do with the decoded rows (EQ, convolution, gain, the
 *            time-batched route, pending moves, state); the engine state afterwards is the state after the f32 call on
 *            the decoded input
 *   encode   b = 16 / 24:  v = y * 2^(b-1) in f32 (exact for finite y), rounded to nearest with ties to even, clamped to
 *            [-2^(b-1), 2^(b-1) - 1]; NaN -> 0, +-inf -> the clamp bounds; dithered as ohs_set_dither says (below), off by
 *            default
 * so out == encode(render(decode(in))) bit for bit.  OHS_FMT_F32 on a side means no conversion on that side; F32 -> F32
 * is ohs_process / ohs_process_device.  Bypass: out = encode(decode(in)) (equal formats: the bytes unchanged), state
 * untouched.  Checked before anything is enqueued (OHS_ERR_INVALID, engine untouched): an unknown format, n_frames not
 * a multiple of B while the convolution is on, row_stride < n_frames, and in == out or overlapping byte ranges when the
 * formats differ (in place needs equal formats).  Device flavour: OHS_ERR_ALIGNMENT unless both pointers are 16-byte
 * aligned and row_stride is a multiple of 4 / 8 / 16 frames for every format involved (F32 / S16 / S24).
 * The host flavour cuts calls into chunks of about OHS_STAGE_MB per copy of the wider side's rows, so S16 chunks hold
 * twice the frames of ohs_process's; the block-by-block kernel renders alike however a call is cut, the time-batched
 * route within round-off.  The device flavour decodes through f32 scratch rows of the engine (up to 256 MiB, allocated
 * on first use or by ohs_prepare; longer calls go through them in time chunks of whole blocks), except that a call with
 * f32 output decodes into the output rows and renders them in place.
 * Not provided: a PCM form of ohs_process_fifo or of ohs_process_device_scheduled, a clip counter, S32 and F64. */
typedef enum ohs_sample_format {
    OHS_FMT_F32 = 0,   /* float, as everywhere else in this API */
    OHS_FMT_S16 = 1,   /* int16_t, little-endian */
    OHS_FMT_S24 = 2    /* packed 3-byte little-endian two's complement (WAV/FLAC 24-bit), 3 bytes per sample */
} ohs_sample_format;
/* host memory; the same contract as ohs_process */
int ohs_process_pcm(ohs_engine* h, const void* in, int in_format, void* out, int out_format, size_t n_frames, size_t row_stride);
/* device memory; the same contract as ohs_process_device */
int ohs_process_device_pcm(ohs_engine* h, const void* d_in, int in_format, void* d_out, int out_format, size_t n_frames,
                           size_t row_stride);

/* ---- dither of integer PCM output (an extension) -----------------------------------------------------------------
 * TPDF dither, optionally with error-feedback noise shaping, for every encode to S16 or S24 by ohs_process_pcm and
 * ohs_process_device_pcm, bypassed F32 -> S16 or S24 -> S16 calls included, and for the integer buses of
 * ohs_process_grouped_pcm and ohs_mix_device_pcm (their rows numbered from 2 * n_streams on, below at ohs_set_groups).
 * F32 output is never dithered.  Exact to the bit (numpy reference: signals.pcm_encode_dithered).  Row r =
 * 2*stream + channel; b = 16 / 24; lo, hi = the clamp bounds.
 *   position  a 64-bit counter p: ohs_set_dither sets it to 0; every successful call with an integer OUTPUT format moves it
 *             on by n_frames (bypassed ones too); frame f of a call has position p0 + f.  So the noise does not depend on
 *             how a render is cut into calls or into the chunks of a call.
 *   noise     mix64(z) = SplitMix64's finaliser: z ^= z >> 30; z *= 0xBF58476D1CE4E5B9; z ^= z >> 27;
 *             z *= 0x94D049BB133111EB; z ^= z >> 31 (all uint64, wrapping), phi = 0x9E3779B97F4A7C15,
 *             K_r = mix64(seed + phi * (r + 1)), x = mix64(K_r + phi * (p + 1)),
 *             u1 = x & (2^23 - 1), u2 = (x >> 32) & (2^23 - 1), d = (u1 + u2 - (2^23 - 1)) * 2^-23:
 *             exact in f32, in (-1, 1) LSB, triangular (TPDF), variance 1/6 LSB^2
 *   flat      (n_taps = 0)  v = y * 2^(b-1);  q = clamp(rint_even(v + d), lo, hi), v + d rounded in f32;  NaN -> 0
 *   shaped    (n_taps = M)  taps h_1..h_M, per-row error history e_1..e_M (most recent first, zero after ohs_set_dither):
 *             fb = h_M*e_M, then + h_(M-1)*e_(M-1), ..., + h_1*e_1 (oldest term first), w = v - fb,
 *             q = clamp(rint_even(w + d), lo, hi), e = clamp(q - w, -1.5, 1.5) becomes e_1 and the others move one back;
 *             every product and sum rounded on its own in f32.  NaN v: q = 0, e = 0; +-inf clamps as without dither.
 *             So q = v + (1 - H(z)) e with H(z) = sum h_k z^-k: the white dither-plus-rounding error (1/4 LSB^2) shaped
 *             by |1 - H|^2.  Without clipping |q - w| < 1.5 always; the clamp of e acts only on clipped samples and keeps
 *             the loop from winding up there.
 * Seed, mode and taps are configuration, like bindings; the position and the error history are state and travel in the
 * state blob.  An equal-format bypass copies bytes and encodes nothing: the position moves on, the history stays.
 * Several GPUs: each rank numbers its rows from 0, so give every rank a seed of its own. */
#define OHS_DITHER_OFF 0       /* round and clamp only (the default) */
#define OHS_DITHER_TPDF 1      /* TPDF dither, noise-shaped when n_taps > 0 */
#define OHS_MAX_SHAPE_TAPS 9
/* Sets mode, seed and taps (shape[0..n_taps) = h_1..h_M, copied), resets the position to 0 and zeroes the history, on the
 * engine's stream (ordered after earlier calls).  Allocates the history (4 * n_streams * OHS_MAX_SHAPE_TAPS floats: stream
 * rows, then the bus rows of ohs_set_groups) for
 * OHS_DITHER_TPDF; process calls never allocate for dither.  OHS_ERR_INVALID with the engine untouched: an unknown mode,
 * n_taps outside 0..OHS_MAX_SHAPE_TAPS, taps with OHS_DITHER_OFF, a null shape with n_taps > 0, a non-finite tap. */
int ohs_set_dither(ohs_engine* h, int mode, uint64_t seed, const float* shape, int n_taps);

int ohs_sync(ohs_engine* h);
/* The engine's cudaStream_t (as void*) so callers can order their own work / NCCL calls against it. */
int ohs_cuda_stream(ohs_engine* h, void** stream);
/* Kernel launches issued by this handle since creation (bench.py's gpu_launches evidence). */
int ohs_launch_count(ohs_engine* h, uint64_t* out);
/* Elapsed device time (ms) of the kernels of the most recent ohs_process_device call made while timing was enabled;
 * blocks until they are done.  Timing is off by default: it brackets every call with two CUDA events, which keeps
 * back-to-back per-block calls from overlapping their launch with the previous call's tail. */
int ohs_enable_timing(ohs_engine* h, int enable);
int ohs_last_kernel_ms(ohs_engine* h, float* ms);

/* ---- listener buses: groups of streams mixed into one binaural bus each (an extension) ------------------------------
 * A 5.1 or 7.1 file is 3 or 4 speaker pairs, one stream each (sofa.wire_speakers wires a pair to its own HRIR set); a
 * listener's object scene is its sources, two mono sources per stream (below).  Either way a group of streams is summed
 * into one stereo bus.  Partition the streams into n_groups contiguous groups: group g holds streams
 * first[g] .. first[g+1]-1.  first is HOST memory with n_groups + 1 entries: first[0] == 0, strictly increasing,
 * first[n_groups] == n_streams, 1 <= n_groups <= n_streams.  Default (and after ohs_create): one group holding every
 * stream.  Like bindings, groups are configuration: not part of the state blob, and they change no stream's rendering.
 * OHS_ERR_INVALID with the engine untouched for anything else.  The offsets are uploaded once, here, on the engine's
 * stream (mixes enqueued before use the old ones).
 * Bus layout everywhere: row 2*g + c (c 0 = left, 1 = right) at bus + (2*g + c) * bus_stride, and with f = first[g]
 *   bus[g][c][n] = ((((+0) + y[f][c][n]) + y[f+1][c][n]) + y[f+2][c][n]) + ...
 * in ascending stream order, every addition rounded to f32 (numpy reference: signals.mix_groups).  Starting from +0
 * differs from starting with y[f] only where every term is -0: the bus is +0 there.
 * Integer buses (ohs_process_grouped_pcm, ohs_mix_device_pcm): bus row 2*g + c is encoded exactly as ohs_process_pcm
 * encodes a stream row, from the f32 bus above, and dithered as ohs_set_dither says with these rules of its own:
 *   row number  bus row 2*g + c has dither row number 2*n_streams + 2*g + c, so K = mix64(seed + phi * (2S + 2g + c + 1)):
 *               its noise never repeats a stream row's (the same keys as stream rows 2g + c under the seed seed + phi * 2S)
 *   position    the engine's one position p: every successful call with an integer bus format moves it on by n_frames
 *               (bypassed ones too), frame f of the call at p0 + f; calls with an F32 bus leave it alone
 *   history     every bus row has its own e_1..e_M, zeroed by ohs_set_dither and by ohs_set_groups (on the engine's stream,
 *               ordered like the offsets), carried by the state blob (flags bit 1)
 * Not provided: grouped forms of ohs_process_fifo and ohs_process_device_scheduled (on the device, compose
 * ohs_process_device_scheduled with ohs_mix_device or ohs_mix_device_pcm), non-contiguous groups, and a mix fused into the
 * render kernel (DESIGN §13, §14). */
int ohs_set_groups(ohs_engine* h, const int32_t* first, int n_groups);
/* The group count in force (bus rows = 2 * *out). */
int ohs_num_groups(ohs_engine* h, int* out);

/* Object mixdown (BASELINE config 4; an extension — the reference has no multi-source mode): sums the rendered
 * streams of each group (ohs_set_groups; by default one group of every stream) into its stereo bus, 2 * n_groups rows
 * of the layout above: d_bus[(2*g + c) * bus_stride + n] = sum over s in group g of d_in[(s*2 + c) * row_stride + n].
 * Two mono sources ride in one stereo stream: source A as the left input with paths (LSL, LSR) = its (left-ear,
 * right-ear) HRIRs, source B as the right input with (RSL, RSR); the engine's output is already their binaural mix
 * (src/dsp/convolution.rs:229-230).  n_frames must be a multiple of 4; pointers 16-byte aligned.  Enqueues on the
 * engine's stream; the bus padding is not touched.  The per-GPU buses are then summed with NCCL (parallel.reduce_bus, or
 * ohs_reduce_bus over all 2 * n_groups * bus_stride floats: per-listener buses reduce across GPUs the same way). */
int ohs_mix_device(ohs_engine* h, const float* d_in, float* d_bus, size_t n_frames, size_t row_stride, size_t bus_stride);
/* Host memory.  Renders exactly what ohs_process_pcm(h, in, in_format, <rows>, OHS_FMT_F32, n_frames, row_stride) renders,
 * cut into the same chunks (so the time-batched route too is bit-identical), and returns only the group buses:
 * bus (host, f32) [2*n_groups][bus_stride], each chunk's buses mixed on the GPU so that only they cross PCIe back.
 * Engine state afterwards == state after that ohs_process_pcm call (pending moves, EQ-only mode, gains and bindings
 * behave as there).  Bypass: bus = mix(decode(in)), state untouched.  The dither position does not move (no integer
 * output).  Checked before anything is enqueued (OHS_ERR_INVALID, engine untouched): the argument rules of
 * ohs_process_pcm with F32 output (an unknown format, n_frames not a multiple of B while the convolution is on,
 * row_stride < n_frames), a null bus, bus_stride < n_frames, a bus that overlaps the input bytes.  ohs_prepare(h, n, 1)
 * also allocates the bus staging. */
int ohs_process_grouped(ohs_engine* h, const void* in, int in_format, float* bus, size_t n_frames, size_t row_stride,
                        size_t bus_stride);
/* ohs_process_grouped with the buses delivered in bus_format (OHS_FMT_F32: exactly ohs_process_grouped).  Host memory;
 * bus row r at byte r * bus_stride * bytes(bus_format).  Renders what ohs_process_grouped renders, in the same chunks, and
 * leaves the same engine state, plus the dither position and bus history of an integer bus (above): each chunk's buses are
 * mixed, dithered and encoded in one launch on the GPU, and only the 2 or 3 bytes per bus sample cross PCIe back.  Bypass:
 * bus = encode(mix(decode(in))), dithered, and the position moves on.  OHS_ERR_INVALID with the engine untouched: the
 * argument rules of ohs_process_grouped, an unknown bus format, and a bus whose bytes overlap the input. */
int ohs_process_grouped_pcm(ohs_engine* h, const void* in, int in_format, void* bus, int bus_format, size_t n_frames,
                            size_t row_stride, size_t bus_stride);
/* Device memory: f32 stream rows -> the group buses in bus_format, one launch on the engine's stream (no f32 bus in
 * between).  OHS_FMT_F32 is exactly ohs_mix_device.  An integer bus takes the alignment rules of ohs_mix_device plus
 * bus_stride a multiple of 8 (S16) or 16 (S24) frames, else OHS_ERR_ALIGNMENT; an unknown format is OHS_ERR_INVALID.  The
 * rendered rows usually come from ohs_process_device on the same engine, which leaves the position alone. */
int ohs_mix_device_pcm(ohs_engine* h, const float* d_in, void* d_bus, int bus_format, size_t n_frames, size_t row_stride,
                       size_t bus_stride);

/* ---- multi-GPU collectives (SURVEY.md 8e) -------------------------------------------------------------------------
 * Streams shard across GPUs with no data-path collective; NCCL is used for exactly two things, both available here so
 * that a host without Python has the N > 1 path: one HRIR spectra table for the whole job (set_ir runs on one rank
 * only) and, for the object mixdown (config 4), the sum of the per-GPU stereo buses.  libnccl.so.2 is opened at run
 * time (dlopen) by the first ohs_comm_* call; a process that never calls them does not need NCCL.
 * One rank obtains the 128-byte id (ncclGetUniqueId) and ships it to the others by any means (the reference has no
 * multi-process mode; under torchrun parallel.create_comm ships it with torch.distributed). */
typedef struct ohs_comm ohs_comm;
#define OHS_COMM_ID_BYTES 128
int ohs_comm_unique_id(void* id128);
int ohs_comm_create(ohs_comm** out, int world, int rank, int device, const void* id128);   /* ncclCommInitRank */
int ohs_comm_destroy(ohs_comm* c);
/* Rank `root` uploads its pending set_ir work and broadcasts the device-resident spectra table and the per-set partition
 * counts on the engine's stream; the other ranks' sets are marked as externally filled (ohs_mark_filters_external).
 * Returns after the stream has drained. */
int ohs_broadcast_hrir(ohs_engine* h, ohs_comm* c, int root);
/* In-place ncclReduce(sum) of d_bus[n_floats] onto rank `root`, enqueued on the engine's stream (after ohs_mix_device). */
int ohs_reduce_bus(ohs_engine* h, ohs_comm* c, float* d_bus, size_t n_floats, int root);

/* pinned host memory helpers */
int ohs_host_alloc(void** p, size_t bytes);
int ohs_host_free(void* p);

/* Debug builds only (-DOHS_TRACE): d_stamps[CTA][16] receives clock64 stamps of the render kernel's milestones
 * (tools/trace_k1.py); a regular build returns OHS_ERR_INVALID. */
int ohs_debug_trace(ohs_engine* h, unsigned long long* d_stamps);

/* ---- state export / import (chunked offline renders resume bit-exactly; SURVEY.md §5.4) ----------------------
 * The blob holds a self-describing header (geometry, ring head, flags, byte count), the delay line, the overlap-save
 * blocks, the biquad states and whatever ohs_process_fifo has queued, and while dither is on (flags bit 0) the dither
 * position (uint64) and error history (float[2 * n_streams][OHS_MAX_SHAPE_TAPS]) behind them; with dither off the blob
 * is what it was before dither existed.  Flags bit 1, only while dither is on and a bus has been encoded since the last
 * ohs_set_dither, ohs_set_groups or import: int32 n_groups, int32 0, float[2 * n_groups][OHS_MAX_SHAPE_TAPS] (the bus
 * rows' history) behind the dither section.  Import rejects a blob whose geometry, size, ring head or dither flag does
 * not match this engine, bit 1 without bit 0 or with another group count, and then leaves the engine untouched; a blob
 * without bit 1 zeroes the bus rows' history.  ohs_state_bytes is the size an export would need NOW (it grows with the FIFO). */
int ohs_state_bytes(ohs_engine* h, size_t* bytes);
int ohs_state_export(ohs_engine* h, void* host_buf, size_t bytes);
int ohs_state_import(ohs_engine* h, const void* host_buf, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* OHS_H */
