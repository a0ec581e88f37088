"""Seeded synthetic inputs for the BASELINE.json configs (SURVEY.md §8d): pink-noise streams, synthetic HRIR/BRIR
sets and the "typical" AutoEQ-like 10-band preset.  Pure numpy; used by bench.py, smoke() and the tests so that
the GPU path, the oracle and the CPU baseline all see identical bits."""
from __future__ import annotations

import numpy as np

# FilterType order of the reference (src/dsp/parametric_eq.rs:25-35)
PEAK, LOWSHELF, HIGHSHELF, LOWPASS, HIGHPASS, BANDPASS, NOTCH, ALLPASS = range(8)

# (type, fc Hz, Q, gain dB) — AutoEQ-like preset, every band enabled (SURVEY.md §8d)
EQ_PRESET_TYPICAL = [
    (LOWSHELF, 105.0, 0.7, 6.5),
    (PEAK, 60.0, 1.2, -3.0),
    (PEAK, 200.0, 0.9, -4.1),
    (PEAK, 800.0, 1.4, 2.2),
    (PEAK, 1800.0, 2.0, -2.5),
    (PEAK, 3200.0, 3.0, 4.0),
    (PEAK, 5500.0, 4.0, -5.0),
    (PEAK, 7400.0, 5.0, 3.1),
    (PEAK, 9800.0, 2.5, -2.0),
    (HIGHSHELF, 10000.0, 0.7, -4.0),
]

# Q=10 peaks at the bottom of the band, +-16 dB: the worst case for f32 DF2T round-off
EQ_PRESET_HARSH = [
    (PEAK, 20.0, 10.0, 16.0), (PEAK, 25.0, 10.0, -16.0), (PEAK, 30.0, 10.0, 16.0), (PEAK, 35.0, 10.0, -16.0),
    (PEAK, 40.0, 10.0, 16.0), (LOWSHELF, 50.0, 0.7, 12.0), (HIGHSHELF, 8000.0, 0.7, -12.0), (NOTCH, 1000.0, 8.0, 0.0),
    (ALLPASS, 500.0, 0.7, 0.0), (PEAK, 12000.0, 6.0, 9.0),
]


def pink_noise(n_frames: int, seed: int) -> np.ndarray:
    """White N(0,1) from default_rng(seed), shaped 1/sqrt(f) in the rFFT domain, peak-normalised to 1.0 (full scale)."""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal(n_frames)
    spec = np.fft.rfft(w)
    f = np.arange(spec.size, dtype=np.float64)
    f[0] = 1.0
    spec /= np.sqrt(f)
    spec[0] = 0.0
    x = np.fft.irfft(spec, n=n_frames)
    x /= np.max(np.abs(x))
    return x.astype(np.float32)


def stream_inputs(n_streams: int, n_frames: int, base_seed: int = 1000, unique: int | None = None) -> np.ndarray:
    """x[stream, channel, frame]; seed = base_seed + 2*stream + channel.  `unique` < n_streams tiles that many
    distinct streams (bench-only shortcut to keep host-side generation short; parity tests use unique streams)."""
    u = n_streams if unique is None else min(unique, n_streams)
    base = np.empty((u, 2, n_frames), np.float32)
    for s in range(u):
        for c in range(2):
            base[s, c] = pink_noise(n_frames, base_seed + 2 * s + c)
    if u == n_streams:
        return base
    reps = (n_streams + u - 1) // u
    return np.ascontiguousarray(np.tile(base, (reps, 1, 1))[:n_streams])


def synthetic_hrir_set(taps: int, decay: float, seed: int = 7) -> np.ndarray:
    """[4, taps] (LSL, LSR, RSL, RSR): default_rng(seed) N(0,1) * exp(-n/decay), each path unit-L2."""
    rng = np.random.default_rng(seed)
    n = np.arange(taps, dtype=np.float64)
    h = rng.standard_normal((4, taps)) * np.exp(-n / decay)
    h /= np.sqrt(np.sum(h * h, axis=1, keepdims=True))
    return h.astype(np.float32)


def pack_s24(q) -> np.ndarray:
    """int32 samples in [-2^23, 2^23) -> packed 3-byte little-endian two's complement (WAV/FLAC 24-bit): the last axis
    grows threefold, uint8."""
    q = np.asarray(q, dtype=np.int32)
    b = q.astype("<i4").view(np.uint8).reshape(q.shape + (4,))[..., :3]
    return np.ascontiguousarray(b).reshape(q.shape[:-1] + (3 * q.shape[-1],))


def unpack_s24(b) -> np.ndarray:
    """Packed 24-bit bytes (last axis 3n) -> int32 samples, sign-extended."""
    b = np.asarray(b, dtype=np.uint8)
    t = b.reshape(b.shape[:-1] + (b.shape[-1] // 3, 3)).astype(np.int32)
    v = t[..., 0] | (t[..., 1] << 8) | (t[..., 2] << 16)
    return (v ^ 0x800000) - 0x800000


# PCM formats of ohs_process_pcm (include/ohs.h): bits per sample
PCM_BITS = {1: 16, 2: 24}


def pcm_decode(q, fmt: int) -> np.ndarray:
    """q * 2^-(b-1) as float32 (exact); q: int samples (S16) or int32 samples (S24, unpacked)."""
    return (np.asarray(q).astype(np.float32) * np.float32(2.0 ** (1 - PCM_BITS[fmt]))).astype(np.float32)


def pcm_encode(y, fmt: int) -> np.ndarray:
    """The encode of include/ohs.h: v = y * 2^(b-1) in f32, round to nearest even, clamp to [-2^(b-1), 2^(b-1) - 1],
    NaN -> 0.  int16 for S16, int32 (unpacked) for S24."""
    b = PCM_BITS[fmt]
    v = np.asarray(y, dtype=np.float32) * np.float32(2.0 ** (b - 1))
    with np.errstate(invalid="ignore"):
        r = np.clip(np.rint(v), -(2.0 ** (b - 1)), 2.0 ** (b - 1) - 1)
    r = np.where(np.isnan(v), np.float32(0.0), r)
    return r.astype(np.int16 if fmt == 1 else np.int32)


# Dither of integer PCM output (include/ohs.h, ohs_set_dither), exact to the bit: uint64 arithmetic wraps like C's
_PHI = np.uint64(0x9E3779B97F4A7C15)


def _mix64(z):
    """SplitMix64's finaliser on uint64 arrays."""
    z = np.asarray(z, np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def tpdf_noise(seed: int, rows, position: int, n: int) -> np.ndarray:
    """The dither noise d of rows `rows` (r = 2*stream + channel) at positions position .. position + n - 1: float32
    [len(rows), n], multiples of 2^-23 in (-1, 1)."""
    r = np.atleast_1d(np.asarray(rows, np.uint64))
    p = np.uint64(position) + np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        key = _mix64(np.uint64(seed) + _PHI * (r + np.uint64(1)))
        x = _mix64(key[:, None] + _PHI * (p[None, :] + np.uint64(1)))
    u1 = (x & np.uint64(0x7FFFFF)).astype(np.int64)
    u2 = ((x >> np.uint64(32)) & np.uint64(0x7FFFFF)).astype(np.int64)
    return ((u1 + u2 - 0x7FFFFF).astype(np.float32) * np.float32(2.0 ** -23)).astype(np.float32)


def _shape_rows(v, d, h, e, lo, hi):
    """The error-feedback recurrence on float32 rows v[R, n] with noise d[R, n], taps h[M] and history e[R, M] (most recent
    first, updated in place).  Returns (q as float32, q - w before the error clamp)."""
    m = len(h)
    q = np.empty_like(v)
    raw = np.empty_like(v)
    lo, hi, lim = np.float32(lo), np.float32(hi), np.float32(1.5)
    with np.errstate(invalid="ignore"):
        for i in range(v.shape[1]):
            fb = h[m - 1] * e[:, m - 1]
            for k in range(m - 2, -1, -1):
                fb = fb + h[k] * e[:, k]
            w = v[:, i] - fb
            qf = np.clip(np.rint(w + d[:, i]), lo, hi)
            err = qf - w
            nan = np.isnan(v[:, i])
            q[:, i] = np.where(nan, np.float32(0.0), qf)
            raw[:, i] = np.where(nan, np.float32(0.0), err)
            e[:, 1:] = e[:, :-1]
            e[:, 0] = np.where(nan, np.float32(0.0), np.clip(err, -lim, lim))
    return q, raw


def pcm_encode_dithered(y, fmt: int, seed: int, position: int, shape=(), state=None, first_row: int = 0):
    """The dithered encode of include/ohs.h (ohs_set_dither): y[..., n] float32 rows, row r = first_row + the flat index over
    the leading axes (2*stream + channel for [S, 2, n]; the buses of a grouped call, mix_groups(y, first), start at
    first_row = 2 * n_streams), frame f at dither position position + f.  shape = (h_1, ..., h_M) noise-shapes; `state` is
    the error history [rows, M] (most recent first, None = zeros after ohs_set_dither).
    Returns (q, state): int16 for S16, int32 (unpacked) for S24, and the history after the last frame."""
    b = PCM_BITS[fmt]
    y = np.asarray(y, dtype=np.float32)
    v = (y.reshape(-1, y.shape[-1]) * np.float32(2.0 ** (b - 1))).astype(np.float32)
    rows, n = v.shape
    d = tpdf_noise(seed, first_row + np.arange(rows), position, n)
    lo, hi = -(2.0 ** (b - 1)), 2.0 ** (b - 1) - 1
    h = np.asarray(shape, np.float32).ravel()
    e = np.zeros((rows, h.size), np.float32) if state is None else np.array(state, np.float32).reshape(rows, h.size)
    if h.size == 0:
        with np.errstate(invalid="ignore"):
            q = np.clip(np.rint(v + d), lo, hi)
        q = np.where(np.isnan(v), np.float32(0.0), q)
    else:
        q, _ = _shape_rows(v, d, h, e, lo, hi)
    return q.astype(np.int16 if fmt == 1 else np.int32).reshape(y.shape), e


def mix_groups(y, first) -> np.ndarray:
    """The group buses of include/ohs.h (ohs_set_groups): y[S, 2, n] float32 rendered streams, group g = streams
    first[g] .. first[g+1]-1.  Returns float32 [G, 2, n]: each group's rows summed from +0 in ascending stream order, every
    addition rounded to f32 (a sequential sum; np.sum adds pairwise)."""
    y = np.asarray(y, dtype=np.float32)
    first = [int(f) for f in first]
    out = np.zeros((len(first) - 1,) + y.shape[1:], np.float32)
    for g in range(len(first) - 1):
        for s in range(first[g], first[g + 1]):
            out[g] = out[g] + y[s]
    return out


# BASELINE.json configs -> engine parameters (SURVEY.md §8d table)
CONFIGS = {
    1: dict(name="cfg1: 1 stereo stream, 48 kHz, SOFA 200-tap HRIR, block 512", n_streams=1, fs=48000.0, block=512, taps=200),
    2: dict(name="cfg2: 1024 stereo streams, 48 kHz, 256-tap HRIR, block 256, 10-band PEQ", n_streams=1024, fs=48000.0,
            block=256, taps=256, decay=40.0),
    3: dict(name="cfg3: 65536 stereo streams (8192/GPU), 48 kHz, 512-tap HRIR, block 128", n_streams=8192, fs=48000.0,
            block=128, taps=512, decay=80.0),
    5: dict(name="cfg5: 2048 stereo streams (256/GPU), 96 kHz, 48000-tap BRIR, partition 1024", n_streams=256, fs=96000.0,
            block=1024, taps=48000, decay=0.15 * 96000.0),
}
