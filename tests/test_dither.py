"""Dither of integer PCM output (include/ohs.h: ohs_set_dither).  The CPU tests check the numpy reference
(signals.tpdf_noise, signals.pcm_encode_dithered) against the definition and against what dither is for; the GPU tests run
twin engines as test_pcm_io.py does: one renders f32 and its output is encoded by the reference, the other renders through
the PCM entry points with dither on, and the bytes must be equal."""

import numpy as np
import pytest
from scipy import signal as sps

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S

gpu = pytest.mark.gpu
F32, S16, S24 = ohs.FMT_F32, ohs.FMT_S16, ohs.FMT_S24
NAME = {F32: "f32", S16: "s16", S24: "s24"}
BYTES = {F32: 4, S16: 2, S24: 3}
FS = 48000.0
LSB = 2.0 ** -15

# (1 - z^-1)^2: second-order highpass shaping
H2 = (2.0, -1.0)
# 9-tap F-weighted error-feedback filter for 44.1 kHz from R. A. Wannamaker, "Psychoacoustically Optimal Noise Shaping",
# J. Audio Eng. Soc. 40(7/8), 1992 (the set SoX ships as "f-weighted")
H9 = (2.412, -3.370, 3.937, -4.174, 3.353, -2.205, 1.281, -0.569, 0.0847)
SHAPES = {"flat": (), "m1": (0.5,), "m2": H2, "m9": H9}


def shaped_error_psd(h, f, fs):
    """1/4 |1 - H(e^jw)|^2 per Hz, one-sided (the white dither-plus-rounding error of power 1/4 LSB^2, shaped)."""
    z = np.exp(-2j * np.pi * np.asarray(f) / fs)
    one_minus_h = 1.0 - sum(hk * z ** (k + 1) for k, hk in enumerate(h))
    return 0.25 * np.abs(one_minus_h) ** 2 * 2.0 / fs


# ---- CPU: the noise ----------------------------------------------------------------------------------------------
def test_mix64_is_splitmix64():
    # SplitMix64 seeded with 0: its first three outputs are mix64(phi), mix64(2 phi), mix64(3 phi)
    phi = np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        got = [int(S._mix64(phi * np.uint64(k))) for k in (1, 2, 3)]
    assert got == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]


def test_noise_is_tpdf_and_deterministic():
    d = S.tpdf_noise(7, np.arange(8), 12345, 125000)
    assert d.dtype == np.float32 and d.shape == (8, 125000)
    k = d.astype(np.float64) * 2.0 ** 23
    assert np.array_equal(k, np.round(k)) and np.abs(k).max() <= 2 ** 23 - 1   # multiples of 2^-23 in (-1, 1)
    assert abs(d.mean()) < 3e-3 and abs(d.var() - 1 / 6) < 2e-3
    hist, _ = np.histogram(d, bins=20, range=(-1, 1))
    tri = 1 - np.abs(np.linspace(-0.95, 0.95, 20))
    assert np.allclose(hist / hist.sum(), tri / tri.sum(), atol=2e-3)   # triangular
    assert np.array_equal(d, S.tpdf_noise(7, np.arange(8), 12345, 125000))
    # a stateless function of (seed, row, position): any window of positions, any subset of rows
    assert np.array_equal(S.tpdf_noise(7, [5, 2], 12345 + 1000, 77), d[[5, 2], 1000:1077])


def test_noise_uncorrelated_across_rows_seeds_and_lags():
    d = S.tpdf_noise(1, np.arange(4), 0, 1 << 18).astype(np.float64)
    e = S.tpdf_noise(2, np.arange(4), 0, 1 << 18).astype(np.float64)
    lim = 5 / np.sqrt(1 << 18)
    c = np.corrcoef(np.vstack([d, e]))
    assert np.abs(c - np.eye(8)).max() < lim
    for lag in (1, 2, 3):
        assert abs(np.corrcoef(d[0, lag:], d[0, :-lag])[0, 1]) < lim


# ---- CPU: the encode -------------------------------------------------------------------------------------------
def test_one_shaped_step_by_hand():
    seed, pos = 11, 40
    d = S.tpdf_noise(seed, [0], pos, 1)[0, 0]
    y = np.array([[100.3 * LSB]], np.float32)
    q, e = S.pcm_encode_dithered(y, S16, seed, pos, shape=H2, state=np.array([[0.25, -0.5]], np.float32))
    f32 = np.float32
    v = f32(y[0, 0]) * f32(32768)
    fb = f32(f32(-1.0) * f32(-0.5)) + f32(f32(2.0) * f32(0.25))   # oldest term first: 0.5 + 0.5
    w = f32(v - fb)
    qq = np.rint(f32(w + d))
    assert int(q[0, 0]) == int(qq) and q.dtype == np.int16
    assert e.tolist() == [[float(f32(qq - w)), 0.25]]
    # NaN: q = 0 and a zero error; +-inf: the clamp bounds
    y = np.array([[np.nan, np.inf, -np.inf]], np.float32)
    q, e = S.pcm_encode_dithered(y, S16, seed, pos, shape=H2)
    assert q.tolist() == [[0, 32767, -32768]] and np.isfinite(e).all() and np.abs(e).max() <= 1.5


def test_flat_dither_by_definition():
    y = (0.3 * np.sin(np.arange(3000) * 0.01)).astype(np.float32).reshape(2, 1500)
    d = S.tpdf_noise(5, [0, 1], 99, 1500)
    for fmt, b in ((S16, 16), (S24, 24)):
        q, _ = S.pcm_encode_dithered(y, fmt, 5, 99)
        v = y * np.float32(2.0 ** (b - 1))
        assert np.array_equal(q, np.clip(np.rint(v + d), -(2 ** (b - 1)), 2 ** (b - 1) - 1).astype(q.dtype))


def test_shaped_error_bounded_and_recovers_after_clipping():
    n = 6000
    t = np.arange(n)
    quiet = (0.001 * np.sin(2 * np.pi * 1000 * t / FS)).astype(np.float32)[None].repeat(4, 0)
    v = quiet * np.float32(32768)
    for h in (H2, H9):
        hf = np.asarray(h, np.float32)
        _, raw = S._shape_rows(v.copy(), S.tpdf_noise(3, np.arange(4), 0, n), hf, np.zeros((4, len(h)), np.float32), -32768, 32767)
        assert np.abs(raw).max() < 1.5
    # a clipped burst at 1.5x full scale, then silence: the output returns to shaped noise of a few LSB
    burst = (1.5 * np.sin(2 * np.pi * 100 * t[:4000] / FS)).astype(np.float32)
    y = np.concatenate([burst, np.zeros(4000, np.float32)])[None]
    q, e = S.pcm_encode_dithered(y, S16, 3, 0, shape=H2)
    assert q[0, :4000].max() == 32767 and q[0, :4000].min() == -32768
    assert np.abs(q[0, -2000:]).max() <= 6          # |(1 - z^-1)^2 e| <= 4 * 1.5
    assert np.abs(e).max() <= 1.5


@pytest.mark.parametrize("h", [H2, H9], ids=["second_order", "wannamaker9"])
def test_error_spectrum_follows_the_shaping_filter(h):
    rows, n = 8, 1 << 15
    t = np.arange(n)
    y = (0.01 * np.sin(2 * np.pi * 997 * t / FS)).astype(np.float32)[None].repeat(rows, 0)
    q, _ = S.pcm_encode_dithered(y, S16, 17, 0, shape=h)
    err = q.astype(np.float64) - y.astype(np.float64) * 32768
    f, p = sps.welch(err, fs=FS, nperseg=2048, axis=-1)
    p = p.mean(axis=0)
    want = shaped_error_psd(h, f, FS)
    edges = np.linspace(0, FS / 2, 9)
    for lo, hi in zip(edges[:-1], edges[1:]):
        sel = (f >= lo) & (f < hi) & (f > 0)
        db = 10 * np.log10(p[sel].mean() / want[sel].mean())
        assert abs(db) < 1.0, (lo, hi, db)


def test_what_dither_buys():
    n, rows = 1 << 16, 8
    t = np.arange(n)
    k = 1000   # whole cycles in the window: every harmonic falls on a bin
    sine = np.sin(2 * np.pi * k * t / n)
    y = (0.25 * LSB * sine).astype(np.float32)[None].repeat(rows, 0)
    assert not S.pcm_encode(y, S16).any()                      # below 1/2 LSB the undithered encode deletes it
    q, _ = S.pcm_encode_dithered(y, S16, 1, 0)
    basis = np.stack([sine, np.cos(2 * np.pi * k * t / n)], 1)
    amp = np.linalg.lstsq(np.tile(basis, (rows, 1)), q.astype(np.float64).ravel(), rcond=None)[0]
    assert abs(np.hypot(*amp) - 0.25) < 0.05 * 0.25
    # 1.3 LSB: harmonics stand above the noise undithered, not dithered
    y = (1.3 * LSB * sine).astype(np.float32)[None].repeat(rows, 0)
    spec = lambda q: (np.abs(np.fft.rfft(q.astype(np.float64), axis=-1)) ** 2).mean(0)   # noqa: E731
    harm = [3 * k, 5 * k, 7 * k]
    plain = spec(S.pcm_encode(y, S16))
    floor = np.median(plain[1:])
    assert all(plain[m] > 1e4 * max(floor, 1e-9) for m in harm)
    dith = spec(S.pcm_encode_dithered(y, S16, 2, 0)[0])
    floor = np.median(dith[1:])
    assert all(dith[m] < 4 * floor for m in harm)
    assert dith[k] > 1e3 * floor                                # the tone itself is kept


def test_set_dither_null_handle_without_a_device():
    lib = ohs.load_library()
    assert lib.ohs_set_dither(None, ohs.DITHER_TPDF, 1, None, 0) == -1


# ---- GPU helpers -------------------------------------------------------------------------------------------------
def make_engine(n_streams, block=256, taps=256, clip=True, odd=True):
    """Config 2 shape: 256-tap HRIR, block 256, 10-band PEQ; every third stream driven past full scale, and with `odd`
    stream 1 renders +-inf (gain inf) and stream 2 NaN (gain NaN)."""
    e = ohs.Engine(n_streams, block, taps, sample_rate=FS)
    e.set_hrir_set(S.synthetic_hrir_set(taps, taps / 6.0, seed=5))
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True)
    e.set_gain(0.5)
    if clip:
        for s in range(0, n_streams, 3):
            e.set_gain(6.0, s)
    if odd and n_streams > 2:
        e.set_gain(float("inf"), 1)
        e.set_gain(float("nan"), 2)
    return e


def inputs(n_streams, n, seed=0, unique=64):
    return (0.9 * S.stream_inputs(n_streams, n, base_seed=3000 + seed, unique=unique)).astype(np.float32)


def to_format(x, fmt):
    if fmt == F32:
        return x, x
    q = S.pcm_encode(x, fmt)
    return (q if fmt == S16 else S.pack_s24(q)), S.pcm_decode(q, fmt)


def as_bytes(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(a.shape[0], a.shape[1], -1)


class Reference:
    """The reference encode with the engine's dither state: position and error history carried from call to call."""

    def __init__(self, fmt, seed, shape):
        self.fmt, self.seed, self.shape, self.pos, self.state = fmt, seed, shape, 0, None

    def __call__(self, y):
        q, self.state = S.pcm_encode_dithered(y, self.fmt, self.seed, self.pos, self.shape, self.state)
        self.pos += y.shape[-1]
        return as_bytes(q if self.fmt == S16 else S.pack_s24(q))


def dev_f32(e, x, n):
    import torch

    d = torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()
    torch.cuda.synchronize()   # the engine runs on its own stream
    e.process_device(d.data_ptr(), d.data_ptr(), n)
    e.sync()
    return d.cpu().numpy()


def dev_pcm(e, buf, fi, fo, n, in_place=False):
    import torch

    d_in = torch.from_numpy(as_bytes(buf).copy()).cuda()
    d_out = d_in if in_place else torch.zeros((buf.shape[0], 2, n * BYTES[fo]), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # the engine runs on its own stream
    e.process_device_pcm(d_in.data_ptr(), fi, d_out.data_ptr(), fo, n)
    e.sync()
    return d_out.cpu().numpy()


def render(e, buf, fi, fo, n, flavour):
    return as_bytes(e.process_pcm(buf, fo)) if flavour == "host" else dev_pcm(e, buf, fi, fo, n)


def twin_call(a, b, ref, x, fmt, flavour):
    n = x.shape[2]
    buf, dec = to_format(x, fmt)
    y = a.process(dec) if flavour == "host" else dev_f32(a, dec, n)
    want = ref(y)
    got = render(b, buf, fmt, fmt, n, flavour)
    assert got.tobytes() == want.tobytes(), (NAME[fmt], flavour)
    return got


# ---- GPU: bit-exact against the reference ------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
@pytest.mark.parametrize("shape", list(SHAPES), ids=str)
@pytest.mark.parametrize("fmt", [S16, S24], ids=lambda f: NAME[f])
def test_dithered_encode_config2(fmt, shape, flavour):
    n_streams, n = 1024, 256 * 8
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_dither(ohs.DITHER_TPDF, seed=0x5EED + fmt, shape=SHAPES[shape])
    ref = Reference(fmt, 0x5EED + fmt, SHAPES[shape])
    got = twin_call(a, b, ref, inputs(n_streams, n), fmt, flavour)
    q = got.view(np.int16) if fmt == S16 else S.unpack_s24(got)
    full = 32767 if fmt == S16 else 2 ** 23 - 1
    assert q.max() == full and q.min() == -full - 1
    assert not q[2].any()                                   # the NaN stream encodes to zeros
    twin_call(a, b, ref, inputs(n_streams, n, seed=1), fmt, flavour)   # position and history carry over


@gpu
def test_same_bytes_however_the_render_is_cut(monkeypatch):
    """One long call, host chunks of one block (OHS_STAGE_MB=1) and of 24, K = 1 device calls, and a device call longer than
    the 256 MiB of f32 scratch (128 + 8 blocks): the same bytes, equal to the reference on the first 8 streams."""
    n_streams, blocks = 1024, 136
    n = 256 * blocks
    x = inputs(n_streams, n, unique=16)
    buf, dec = to_format(x, S16)

    def dithered(env=None):
        if env:
            monkeypatch.setenv("OHS_STAGE_MB", env)
        else:
            monkeypatch.delenv("OHS_STAGE_MB", raising=False)
        e = make_engine(n_streams)
        e.set_dither(ohs.DITHER_TPDF, seed=9, shape=H2)
        return e

    outs = {"host_1mb_chunks": as_bytes(dithered("1").process_pcm(buf, S16)),
            "host_default_chunks": as_bytes(dithered().process_pcm(buf, S16)),
            "device_longer_than_scratch": dev_pcm(dithered(), buf, S16, S16, n)}
    import torch

    e = dithered()
    d_in = torch.from_numpy(as_bytes(buf).copy()).cuda()
    d_out = torch.zeros_like(d_in)
    for t in range(blocks):
        rows_in = d_in[:, :, t * 512:(t + 1) * 512].contiguous()
        rows_out = torch.zeros_like(rows_in)
        torch.cuda.synchronize()   # torch's stream and the engine's are ordered by hand
        e.process_device_pcm(rows_in.data_ptr(), S16, rows_out.data_ptr(), S16, 256)
        e.sync()
        d_out[:, :, t * 512:(t + 1) * 512] = rows_out
    outs["device_one_block_calls"] = d_out.cpu().numpy()
    first = outs["host_default_chunks"].tobytes()
    for k, v in outs.items():
        assert v.tobytes() == first, k
    a = make_engine(n_streams)
    y = dev_f32(a, dec, n)
    want = Reference(S16, 9, H2)(y[:8])
    assert outs["host_default_chunks"][:8].tobytes() == want.tobytes()


@gpu
@pytest.mark.parametrize("shape", ["flat", "m9"], ids=str)
def test_state_export_mid_render(shape):
    n_streams, n = 256, 256 * 6
    a, b = make_engine(n_streams), make_engine(n_streams)
    plain = make_engine(n_streams).state_export()
    for e in (a, b):
        e.set_dither(ohs.DITHER_TPDF, seed=77, shape=SHAPES[shape])
    q1, _ = to_format(inputs(n_streams, n), S24)
    q2, _ = to_format(inputs(n_streams, n, seed=1), S24)
    a.process_pcm(q1, S24)
    b.process_pcm(q1, S24)
    blob = b.state_export()
    assert len(blob) == len(plain) + 8 + 72 * n_streams
    c = make_engine(n_streams)
    with pytest.raises(ohs.OhsError):
        c.state_import(blob)                     # this engine's dither is off
    d = make_engine(n_streams)
    d.set_dither(ohs.DITHER_TPDF, seed=77, shape=SHAPES[shape])
    with pytest.raises(ohs.OhsError):
        d.state_import(plain)                    # a blob without dither state
    c.set_dither(ohs.DITHER_TPDF, seed=77, shape=SHAPES[shape])
    c.state_import(blob)
    want = as_bytes(a.process_pcm(q2, S24)).tobytes()
    assert as_bytes(c.process_pcm(q2, S24)).tobytes() == want
    # the rejected import left d as it was: a fresh dithered engine renders the first call
    fresh = make_engine(n_streams)
    fresh.set_dither(ohs.DITHER_TPDF, seed=77, shape=SHAPES[shape])
    assert as_bytes(d.process_pcm(q1, S24)).tobytes() == as_bytes(fresh.process_pcm(q1, S24)).tobytes()


# ---- GPU: semantics ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_off_bypass_f32_output_and_in_place(flavour):
    n_streams, n = 64, 256 * 3
    x = inputs(n_streams, n)
    buf16, dec16 = to_format(x, S16)
    # OFF after TPDF: undithered bytes again
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_dither(ohs.DITHER_TPDF, seed=3, shape=H2)
    b.set_dither(ohs.DITHER_OFF)
    y = a.process(dec16)
    assert render(b, buf16, S16, S16, n, flavour).tobytes() == as_bytes(S.pcm_encode(y, S16)).tobytes()
    # an equal-format bypass copies bytes and moves the position on; a dithered F32 -> S16 bypass is the reference
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_dither(ohs.DITHER_TPDF, seed=4, shape=H9)
    ref = Reference(S16, 4, H9)
    b.set_bypass(True)
    assert render(b, buf16, S16, S16, n, flavour).tobytes() == as_bytes(buf16).tobytes()
    ref.pos += n
    xf = 1.7 * x
    assert render(b, xf, F32, S16, n, flavour).tobytes() == ref(xf).tobytes()
    b.set_bypass(False)
    twin_call(a, b, ref, x, S16, flavour)
    # F32 output is never dithered (and does not move the position)
    c = make_engine(n_streams)
    c.set_dither(ohs.DITHER_TPDF, seed=4, shape=H9)
    assert render(c, buf16, S16, F32, n, flavour).tobytes() == as_bytes(make_engine(n_streams).process(dec16)).tobytes()


@gpu
def test_in_place_equal_formats():
    n_streams, n = 256, 256 * 5
    x = inputs(n_streams, n)
    buf, dec = to_format(x, S24)
    want = Reference(S24, 6, H2)(make_engine(n_streams).process(dec)).tobytes()
    b, c = make_engine(n_streams), make_engine(n_streams)
    for e in (b, c):
        e.set_dither(ohs.DITHER_TPDF, seed=6, shape=H2)
    assert dev_pcm(b, buf, S24, S24, n, in_place=True).tobytes() == want
    host = np.ascontiguousarray(buf).copy()
    assert ohs.load_library().ohs_process_pcm(c._h, host.ctypes.data, S24, host.ctypes.data, S24, n, n) == 0
    assert as_bytes(host).tobytes() == want


@gpu
def test_launch_count_unchanged_by_dither():
    n_streams, n = 1024, 256 * 4
    buf, _ = to_format(inputs(n_streams, n), S16)
    counts = []
    for shape in (None, (), H2, H9):
        e = make_engine(n_streams)
        if shape is not None:
            e.set_dither(ohs.DITHER_TPDF, seed=1, shape=shape)
        dev_pcm(e, buf, S16, S16, n)   # set-up launches
        c0 = e.launch_count()
        dev_pcm(e, buf, S16, S24, n)
        e.process_pcm(buf, S16)
        counts.append(e.launch_count() - c0)
    assert len(set(counts)) == 1, counts


@gpu
def test_rejected_set_dither_leaves_the_engine_untouched():
    lib = ohs.load_library()
    n_streams, n = 64, 256 * 2
    buf, dec = to_format(inputs(n_streams, n), S16)
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_dither(ohs.DITHER_TPDF, seed=8, shape=H2)
    ref = Reference(S16, 8, H2)
    twin_call(a, b, ref, inputs(n_streams, n), S16, "host")
    taps = np.array([0.5, np.nan, 0.1], np.float32)
    p = taps.ctypes.data_as(ohs.engine._f32p)
    assert lib.ohs_set_dither(b._h, 2, 1, None, 0) == -1                 # unknown mode
    assert lib.ohs_set_dither(b._h, -1, 1, None, 0) == -1
    assert lib.ohs_set_dither(b._h, ohs.DITHER_TPDF, 1, p, 10) == -1     # more than 9 taps
    assert lib.ohs_set_dither(b._h, ohs.DITHER_TPDF, 1, p, -1) == -1
    assert lib.ohs_set_dither(b._h, ohs.DITHER_OFF, 1, p, 1) == -1       # taps with mode OFF
    assert lib.ohs_set_dither(b._h, ohs.DITHER_TPDF, 1, None, 2) == -1   # null shape
    assert lib.ohs_set_dither(b._h, ohs.DITHER_TPDF, 1, p, 2) == -1      # a NaN tap
    taps[1] = np.inf
    assert lib.ohs_set_dither(b._h, ohs.DITHER_TPDF, 1, p, 3) == -1
    twin_call(a, b, ref, inputs(n_streams, n, seed=1), S16, "host")
