"""Integer PCM in and out (include/ohs.h: ohs_process_pcm, ohs_process_device_pcm).  The definition is
out = encode(render(decode(in))) bit for bit, so every GPU case runs twin engines: one fed decode(in) through the f32
entry point with its output quantised by the numpy reference (signals.pcm_encode), the other fed `in` through the PCM entry point.
Outputs must be bit-identical, and so must a follow-up f32 call on both (equal state)."""

import numpy as np
import pytest

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S
from oracle import oracle as O

gpu = pytest.mark.gpu
F32, S16, S24 = ohs.FMT_F32, ohs.FMT_S16, ohs.FMT_S24
FMTS = [F32, S16, S24]
NAME = {F32: "f32", S16: "s16", S24: "s24"}
BYTES = {F32: 4, S16: 2, S24: 3}
FS = 48000.0


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_s24_pack_round_trip():
    q = np.array([[-2 ** 23, 2 ** 23 - 1, -1, 0, 1, 0x7F, 0x80, 0xFF, 0x100, -0x80, -0x81, -0x800000 + 1, 0x123456, -0x123456]], np.int32)
    b = S.pack_s24(q)
    assert b.dtype == np.uint8 and b.shape == (1, 3 * q.shape[1])
    assert list(b[0, :6]) == [0x00, 0x00, 0x80, 0xFF, 0xFF, 0x7F]          # little-endian, two's complement
    assert list(b[0, 6:9]) == [0xFF, 0xFF, 0xFF]                            # -1
    back = S.unpack_s24(b)
    assert back.dtype == np.int32 and np.array_equal(back, q)              # sign extension
    rng = np.random.default_rng(1)
    r = rng.integers(-2 ** 23, 2 ** 23, size=(3, 2, 999)).astype(np.int32)
    assert np.array_equal(S.unpack_s24(S.pack_s24(r)), r)


def test_reference_quantiser_by_hand():
    lsb16, lsb24 = 2.0 ** -15, 2.0 ** -23
    y = np.array([0.5 * lsb16, 1.5 * lsb16, 2.5 * lsb16, -0.5 * lsb16, -1.5 * lsb16, 1.0, -1.0, 1 - 2 ** -16, -0.0,
                  np.inf, -np.inf, np.nan, 0.49 * lsb16, 3.0], np.float32)
    assert S.pcm_encode(y, S16).tolist() == [0, 2, 2, 0, -2, 32767, -32768, 32767, 0, 32767, -32768, 0, 0, 32767]
    assert S.pcm_encode(y, S16).dtype == np.int16
    y24 = np.array([0.5 * lsb24, 1.5 * lsb24, -0.5 * lsb24, -1.5 * lsb24, 1.0, -1.0, 1 - 2 ** -16, -0.0, np.inf, -np.inf, np.nan],
                   np.float32)
    assert S.pcm_encode(y24, S24).tolist() == [0, 2, 0, -2, 2 ** 23 - 1, -2 ** 23, 2 ** 23 - 2 ** 7, 0, 2 ** 23 - 1, -2 ** 23, 0]
    # decode is exact and encode inverts it
    q = np.arange(-32768, 32768, dtype=np.int16)
    assert np.array_equal(S.pcm_encode(S.pcm_decode(q, S16), S16), q)
    assert S.pcm_decode(np.int16(-32768), S16) == -1.0
    q24 = np.array([-2 ** 23, -1, 0, 1, 2 ** 23 - 1], np.int32)
    assert np.array_equal(S.pcm_encode(S.pcm_decode(q24, S24), S24), q24)


def test_null_handle_without_a_device():
    lib = ohs.load_library()
    for fn in (lib.ohs_process_pcm, lib.ohs_process_device_pcm):
        assert fn(None, None, S16, None, S16, 256, 256) == -1
        assert fn(None, None, 7, None, S16, 256, 256) == -1


def test_python_format_selection_without_a_device():
    e = ohs.Engine.__new__(ohs.Engine)
    e.n_streams = 1
    with pytest.raises(ValueError):
        e.process_pcm(np.zeros((1, 2, 8), np.int32), S16)            # int32 is not a PCM dtype here
    with pytest.raises(ValueError):
        e.process_pcm(np.zeros((1, 2, 8), np.uint8), S16)            # packed 24-bit needs 3n bytes
    with pytest.raises(ValueError):
        e.process_pcm(np.zeros((1, 2, 9), np.int16), 5)              # unknown output format


# ---- GPU helpers ------------------------------------------------------------------------------------------------
def to_format(x, fmt):
    """f32 rows -> (the buffer as the API takes it in `fmt`, its decode)."""
    if fmt == F32:
        return x, x
    q = S.pcm_encode(x, fmt)
    return (q if fmt == S16 else S.pack_s24(q)), S.pcm_decode(q, fmt)


def encode(y, fmt):
    """The reference encode of f32 rows into the API's buffer form of `fmt`."""
    if fmt == F32:
        return np.ascontiguousarray(y, np.float32)
    q = S.pcm_encode(y, fmt)
    return q if fmt == S16 else S.pack_s24(q)


def as_bytes(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(a.shape[0], a.shape[1], -1)


def make_engine(n_streams, block=256, taps=256, n_sets=1, eq=True, clip=True, seed=5):
    """Config 2 shape by default: 256-tap HRIR, block 256, 10-band PEQ; with `clip` every third stream's gain drives its
    output well past full scale."""
    e = ohs.Engine(n_streams, block, taps, n_hrir_sets=n_sets, sample_rate=FS)
    for k in range(n_sets):
        e.set_hrir_set(S.synthetic_hrir_set(taps, taps / 6.0, seed=seed + k), hrir_set=k)
    if eq:
        e.eq_set_preset(S.EQ_PRESET_TYPICAL)
        e.set_eq_enable(True)
    e.set_gain(0.5)
    if clip:
        for s in range(0, n_streams, 3):
            e.set_gain(6.0, s)
    return e


def inputs(n_streams, n, seed=0, unique=64):
    return (0.9 * S.stream_inputs(n_streams, n, base_seed=3000 + seed, unique=unique)).astype(np.float32)


def dev_f32(e, x, n, rs):
    import torch

    d_in = torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()
    d_out = torch.zeros_like(d_in)
    e.process_device(d_in.data_ptr(), d_out.data_ptr(), n, rs)
    e.sync()
    return d_out.cpu().numpy()[:, :, :n]


def dev_pcm(e, buf, fi, fo, n, rs, in_place=False):
    """One ohs_process_device_pcm call; returns the output rows' first n frames as bytes [S, 2, n * BYTES[fo]]."""
    import torch

    d_in = torch.from_numpy(as_bytes(buf).copy()).cuda()
    d_out = d_in if in_place else torch.zeros((buf.shape[0], 2, rs * BYTES[fo]), dtype=torch.uint8, device="cuda")
    e.process_device_pcm(d_in.data_ptr(), fi, d_out.data_ptr(), fo, n, rs)
    e.sync()
    return d_out.cpu().numpy()[:, :, :n * BYTES[fo]]


def twin_call(a, b, x, fi, fo, flavour, n=None, rs=None):
    """a: f32 entry point on decode(in), quantised by the reference; b: the PCM entry point on in.  Asserts bit equality."""
    n = x.shape[2] if n is None else n
    rs = x.shape[2] if rs is None else rs
    buf, dec = to_format(x, fi)
    if flavour == "host":
        assert rs == x.shape[2]
        want = encode(a.process(dec), fo)
        got = b.process_pcm(buf, fo)
    else:
        want = encode(dev_f32(a, dec, n, rs), fo)
        got = dev_pcm(b, buf, fi, fo, n, rs)
    assert got.tobytes() == as_bytes(want).tobytes(), (NAME[fi], NAME[fo], flavour)
    return got


def same_state(a, b, z):
    """A follow-up f32 call on both twins: equal state gives bit-identical output."""
    ya, yb = a.process(z), b.process(z)
    assert ya.tobytes() == yb.tobytes()


# ---- GPU: every format pair at config 2 width --------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
@pytest.mark.parametrize("fo", FMTS, ids=lambda f: "to_" + NAME[f])
@pytest.mark.parametrize("fi", FMTS, ids=lambda f: "from_" + NAME[f])
def test_every_format_pair_config2(fi, fo, flavour):
    n_streams, n = 1024, 256 * 8
    a, b = make_engine(n_streams), make_engine(n_streams)
    x = inputs(n_streams, n)
    got = twin_call(a, b, x, fi, fo, flavour)
    if fo != F32:   # the clipped streams reach the bounds
        full = 32767 if fo == S16 else 2 ** 23 - 1
        q = got.view(np.int16) if fo == S16 else S.unpack_s24(got)
        assert q.max() == full and q.min() == -full - 1
    twin_call(a, b, inputs(n_streams, n, seed=1), fi, fo, flavour)   # a second call continues from the first one's state
    same_state(a, b, inputs(n_streams, 512, seed=2))


@gpu
def test_launch_count_adds_the_conversions():
    import torch

    n_streams, n = 1024, 256 * 4
    a, b = make_engine(n_streams), make_engine(n_streams)
    x = inputs(n_streams, n)
    buf, dec = to_format(x, S16)
    for _ in range(2):   # the second round has no set-up launches
        a0, b0 = a.launch_count(), b.launch_count()
        dev_f32(a, dec, n, n)
        dev_pcm(b, buf, S16, S24, n, n)
    assert b.launch_count() - b0 == a.launch_count() - a0 + 2
    torch.cuda.synchronize()


# ---- GPU: the host pipeline over several chunks, call shapes and routes ------------------------------------------
@gpu
@pytest.mark.parametrize("fi,fo", [(S16, S16), (S24, S24), (S16, F32), (F32, S24), (S24, S16)], ids=lambda f: NAME[f])
def test_host_pipeline_several_chunks(fi, fo, monkeypatch):
    """OHS_STAGE_MB=1 and 64 streams: chunks of 16 (S16) / 10 (S24) / 8 (F32) blocks, 37 blocks per call, so the
    last chunk is ragged and every pipeline slot is reused."""
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    n_streams, n = 64, 256 * 37
    a, b = make_engine(n_streams), make_engine(n_streams)
    twin_call(a, b, inputs(n_streams, n), fi, fo, "host")
    twin_call(a, b, inputs(n_streams, n, seed=1), fi, fo, "host")
    same_state(a, b, inputs(n_streams, 1024, seed=2))


@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_eq_only_ragged_tail_s24(flavour, monkeypatch):
    """EQ-only mode takes any n_frames: 3109 = 12 blocks + 37 frames, so S24's last 16-frame group is partial (5 frames);
    the device flavour with row_stride 3120 > n_frames.  On the host, OHS_STAGE_MB=1 cuts the call into a chunk of 10
    blocks and a ragged one of 549 frames."""
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    n_streams, n = 64, 256 * 12 + 37
    rs = n if flavour == "host" else 3120
    a, b = make_engine(n_streams), make_engine(n_streams)
    for e in (a, b):
        e.set_conv_enable(False)
    for fo in (S24, S16, F32):
        twin_call(a, b, inputs(n_streams, rs, seed=fo), S24, fo, flavour, n, rs)
    same_state(a, b, inputs(n_streams, 333, seed=9))


@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_one_and_two_block_calls(flavour):
    """K = 1 and K = 2 calls run the latency variant of the render kernel."""
    n_streams = 1024
    a, b = make_engine(n_streams), make_engine(n_streams)
    for i, k in enumerate([1, 2, 1, 1, 2]):
        twin_call(a, b, inputs(n_streams, 256 * k, seed=i), S16, S24 if i % 2 else S16, flavour)
    same_state(a, b, inputs(n_streams, 256, seed=7))


@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_three_partition_response(flavour):
    n_streams = 256
    a, b = make_engine(n_streams, taps=3 * 256 - 5), make_engine(n_streams, taps=3 * 256 - 5)
    for i in range(3):
        twin_call(a, b, inputs(n_streams, 256 * 6, seed=i), S24, S16, flavour)
    same_state(a, b, inputs(n_streams, 512, seed=5))


@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_time_batched_route(flavour):
    """9 partitions at block 128 and 40 blocks per call: the time-batched route (EQ pre-pass on the handle's second
    stream, ordered behind the decode on the engine's stream).  Both calls fit one chunk in either flavour."""
    n_streams, block, taps = 5, 128, 1100
    a, b = (make_engine(n_streams, block=block, taps=taps) for _ in range(2))
    for i in range(2):
        twin_call(a, b, inputs(n_streams, block * 40, seed=i, unique=5), S16, S16, flavour)
    same_state(a, b, inputs(n_streams, block * 3, seed=4, unique=5))


@gpu
def test_device_calls_longer_than_the_scratch():
    """256 MiB of f32 scratch rows hold 128 blocks of config 2's 1024 streams; a call of 136 blocks goes through them in
    two time chunks (128 + 8 blocks), each decoded, rendered in place and encoded."""
    n_streams, n = 1024, 256 * 136
    a, b = make_engine(n_streams), make_engine(n_streams)
    twin_call(a, b, inputs(n_streams, n, unique=16), S16, S24, "device")
    same_state(a, b, inputs(n_streams, 512, seed=3))


@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_pending_move_applied_by_a_pcm_call(flavour):
    n_streams = 64
    a, b = make_engine(n_streams, n_sets=2), make_engine(n_streams, n_sets=2)
    twin_call(a, b, inputs(n_streams, 256 * 4), S16, S16, flavour)
    for e in (a, b):
        e.move_stream_hrir(ohs.OHS_ALL, 1)
    twin_call(a, b, inputs(n_streams, 256 * 4, seed=1), S16, S16, flavour)
    same_state(a, b, inputs(n_streams, 512, seed=2))


# ---- GPU: bypass, in place, rejected calls -----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("flavour", ["host", "device"])
def test_bypass(flavour):
    """Equal formats copy the bytes unchanged; different ones give encode(decode(in)); the state is untouched."""
    n_streams, n = 64, 256 * 3
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_bypass(True)
    x = 1.7 * inputs(n_streams, n)   # past full scale: an F32 input is clamped on the way to S16
    for fi, fo in ((S16, S16), (S24, S24), (S24, S16), (S16, S24), (F32, S16), (S24, F32)):
        buf, dec = to_format(x, fi)
        got = b.process_pcm(buf, fo) if flavour == "host" else dev_pcm(b, buf, fi, fo, n, n)
        want = buf if fi == fo else encode(dec, fo)
        assert as_bytes(got).tobytes() == as_bytes(want).tobytes(), (NAME[fi], NAME[fo])
    b.set_bypass(False)
    same_state(a, b, inputs(n_streams, 512, seed=2))


@gpu
def test_in_place_equal_formats():
    import torch

    n_streams, n = 256, 256 * 5
    a, b, c = make_engine(n_streams), make_engine(n_streams), make_engine(n_streams)
    x = inputs(n_streams, n)
    buf, dec = to_format(x, S24)
    want = as_bytes(encode(a.process(dec), S24)).tobytes()
    assert dev_pcm(b, buf, S24, S24, n, n, in_place=True).tobytes() == want
    host = np.ascontiguousarray(buf).copy()
    lib = ohs.load_library()
    assert lib.ohs_process_pcm(c._h, host.ctypes.data, S24, host.ctypes.data, S24, n, n) == 0
    assert host.tobytes() == want
    torch.cuda.synchronize()
    z = inputs(n_streams, 512, seed=2)
    ya, yb, yc = a.process(z), b.process(z), c.process(z)   # one follow-up call each: equal state, equal output
    assert ya.tobytes() == yb.tobytes() == yc.tobytes()


@gpu
def test_rejected_calls_leave_the_engine_untouched():
    import torch

    lib = ohs.load_library()
    n_streams, n = 64, 256 * 2
    a, b = make_engine(n_streams), make_engine(n_streams)
    x = inputs(n_streams, n)
    q16, _ = to_format(x, S16)
    host = np.zeros(n_streams * 2 * n * 4 + 64, np.uint8)
    d = torch.zeros(n_streams * 2 * n * 4 + 64, dtype=torch.uint8, device="cuda")
    hp, dp = host.ctypes.data, d.data_ptr()
    for fn, p in ((lib.ohs_process_pcm, hp), (lib.ohs_process_device_pcm, dp)):
        assert fn(b._h, p, 3, p + 32768, S16, n, n) == -1                  # unknown formats
        assert fn(b._h, p, S16, p + 32768, -1, n, n) == -1
        assert fn(b._h, p, S16, p, S24, n, n) == -1                        # in place across formats
        assert fn(b._h, p, S16, p + 32, S24, n, n) == -1                   # overlapping byte ranges
        assert fn(b._h, p + 32, S24, p, S16, n, n) == -1
        assert fn(b._h, p, S16, p + 32768, S16, n - 16, n) == -1           # not whole blocks with the convolution on
        assert fn(b._h, p, S16, p + 32768, S16, n, n - 8) == -1            # row_stride < n_frames
    # device rows must start 16-byte aligned in their format
    big = n_streams * 2 * (n + 16)
    assert lib.ohs_process_device_pcm(b._h, dp + 2, S16, dp + big * 4, S16, n, n) == -6
    assert lib.ohs_process_device_pcm(b._h, dp, S16, dp + big * 2, S24, n, n + 4) == -6     # 4 frames: F32 only
    assert lib.ohs_process_device_pcm(b._h, dp, S24, dp + big * 3, S24, n, n + 8) == -6     # 8: not S24
    assert lib.ohs_process_device_pcm(b._h, dp, F32, dp + big * 4, F32, n, n + 2) == -6
    torch.cuda.synchronize()
    twin_call(a, b, x, S16, S16, "device")
    same_state(a, b, inputs(n_streams, 512, seed=2))


# ---- GPU: against the oracle -------------------------------------------------------------------------------------
@gpu
def test_s16_within_one_lsb_of_the_quantised_oracle():
    n_streams, block, taps, n = 4, 256, 256, 256 * 6
    h = S.synthetic_hrir_set(taps, taps / 6.0, seed=5)
    coeffs = np.stack([ohs.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    e = ohs.Engine(n_streams, block, taps, sample_rate=FS)
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(4.0)
    q, dec = to_format(inputs(n_streams, n, unique=4), S16)
    got = e.process_pcm(q, S16).astype(np.int32)
    ref, _ = O.render_batch(dec, block, h, coeffs, [1] * 10, True, 4.0, n_threads=4)
    want = S.pcm_encode(ref, S16).astype(np.int32)
    assert np.max(np.abs(got - want)) <= 1
    assert np.any(np.abs(want) == 32767) or np.any(want == -32768)   # gain 4 clips somewhere
