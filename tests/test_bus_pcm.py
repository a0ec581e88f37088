"""Integer PCM listener buses (include/ohs.h: ohs_process_grouped_pcm, ohs_mix_device_pcm; DESIGN §14).  A bus row is
encoded exactly as a stream row, from the f32 bus of ohs_set_groups, with dither row numbers from 2 * n_streams on.  So
the GPU cases run twin engines: A renders with ohs_process_pcm(..., F32), its rows are mixed by signals.mix_groups and
encoded by signals.pcm_encode_dithered(..., first_row=2S); B renders the same input into integer buses.  The bytes must be
equal, call after call."""
import os
import re
import struct

import numpy as np
import pytest

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S

gpu = pytest.mark.gpu
F32, S16, S24 = ohs.FMT_F32, ohs.FMT_S16, ohs.FMT_S24
NAME = {F32: "f32", S16: "s16", S24: "s24"}
BYTES = {F32: 4, S16: 2, S24: 3}
FS = 48000.0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_ALIGNMENT = -1, -6
PHI = 0x9E3779B97F4A7C15
H2 = (2.0, -1.0)
H9 = (2.412, -3.370, 3.937, -4.174, 3.353, -2.205, 1.281, -0.569, 0.0847)
# None: dither off; (): flat TPDF; taps: noise-shaped
MODES = {"off": None, "flat": (), "m1": (0.5,), "m2": H2, "m9": H9}


def mixed_groups(n_streams, sizes=(1, 2, 3, 4, 7)):
    first, k = [0], 0
    while first[-1] < n_streams:
        first.append(min(n_streams, first[-1] + sizes[k % len(sizes)]))
        k += 1
    return first


def layout(name, n_streams):
    """7.1: four speaker pairs per file; 5.1: three, the last group one stream; mixed: sizes 1, 2, 3, 4, 7."""
    if name == "7.1":
        return list(range(0, n_streams + 1, 4))
    if name == "5.1":
        assert n_streams % 3 == 1
        return list(range(0, n_streams, 3)) + [n_streams]
    return mixed_groups(n_streams)


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_symbols_are_declared_and_bound():
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ohs.h")).read(), flags=re.S)
    lib = ohs.load_library()
    bound = {s[0] for s in ohs.SYMBOLS}
    for name in ("ohs_process_grouped_pcm", "ohs_mix_device_pcm"):
        assert re.search(r"\b%s\s*\(" % name, hdr), name
        assert name in bound and hasattr(lib, name), name


def test_null_handle_and_unknown_bus_format_without_a_device():
    lib = ohs.load_library()
    for fmt in (S16, S24, F32, 7, -1):
        assert lib.ohs_process_grouped_pcm(None, None, S16, None, fmt, 256, 256, 256) == ERR_INVALID
        assert lib.ohs_mix_device_pcm(None, None, None, fmt, 256, 256, 256) == ERR_INVALID


def test_python_argument_checks_without_a_device():
    e = ohs.Engine.__new__(ohs.Engine)
    e.n_streams = 2
    with pytest.raises(ValueError):
        e.process_grouped(np.zeros((2, 2, 8), np.int16), bus_format=3)      # unknown bus format
    with pytest.raises(ValueError):
        e.process_grouped(np.zeros((2, 2, 8), np.int32), bus_format=S16)    # not a PCM input dtype
    with pytest.raises(ValueError):
        e.process_grouped(np.zeros((3, 2, 8), np.int16), bus_format=S24)    # wrong stream count


@pytest.mark.parametrize("mode", ["flat", "m2", "m9"])
@pytest.mark.parametrize("fmt", [S16, S24], ids=lambda f: NAME[f])
def test_first_row_is_a_window_of_a_larger_encode(fmt, mode):
    rng = np.random.default_rng(11)
    rows, k, n = 12, 37, 300
    y = (0.4 * rng.standard_normal((k + rows, n))).astype(np.float32)
    y[k + 3, ::7] = 2.0                  # clipped samples
    y[k + 5, 10] = np.nan
    state = (0.3 * rng.standard_normal((k + rows, len(MODES[mode])))).astype(np.float32)
    whole, e_whole = S.pcm_encode_dithered(y, fmt, 99, 1234, MODES[mode], state)
    part, e_part = S.pcm_encode_dithered(y[k:], fmt, 99, 1234, MODES[mode], state[k:], first_row=k)
    assert part.tobytes() == whole[k:].tobytes()
    assert e_part.tobytes() == e_whole[k:].tobytes()
    # first_row=0 is the default: every existing result is unchanged
    assert S.pcm_encode_dithered(y, fmt, 99, 1234, MODES[mode], state, first_row=0)[0].tobytes() == whole.tobytes()


@pytest.mark.parametrize("seed", [0, 1, 0x5EED, 2 ** 64 - 1, 2 ** 64 - PHI])
@pytest.mark.parametrize("n_streams", [1, 7, 1024, 8191])
def test_bus_keys_are_stream_keys_under_an_offset_seed(seed, n_streams):
    """Bus row 2g + c has dither row number 2S + 2g + c: the same noise as row 2g + c under the seed seed + phi * 2S (mod 2^64),
    which is what the kernels are given."""
    rows = np.arange(2 * min(n_streams, 40))
    offset = (seed + PHI * 2 * n_streams) % 2 ** 64
    a = S.tpdf_noise(seed, 2 * n_streams + rows, 77, 64)
    b = S.tpdf_noise(offset, rows, 77, 64)
    assert a.tobytes() == b.tobytes()
    assert not np.array_equal(a, S.tpdf_noise(seed, rows, 77, 64))   # never a stream row's noise


# ---- GPU helpers -------------------------------------------------------------------------------------------------
def make_engine(n_streams, first, block=256, taps=256, mode=None, seed=0x5EED, odd=True):
    """Config 2 shape: 256-tap HRIR, block 256, 10-band PEQ; every third stream driven past full scale, and with `odd`
    stream 1 renders +-inf (gain inf) and stream 4 NaN (gain NaN), in different groups of every layout here."""
    e = ohs.Engine(n_streams, block, taps, sample_rate=FS)
    e.set_hrir_set(S.synthetic_hrir_set(taps, taps / 6.0, seed=5))
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True)
    e.set_gain(0.5)
    for s in range(0, n_streams, 3):
        e.set_gain(6.0, s)
    if odd and n_streams > 4:
        e.set_gain(float("inf"), 1)
        e.set_gain(float("nan"), 4)
    if first is not None:
        e.set_groups(first)
    if mode is not None:
        e.set_dither(ohs.DITHER_TPDF, seed=seed, shape=mode)
    return e


def inputs(n_streams, n, seed=0, unique=64):
    return (0.9 * S.stream_inputs(n_streams, n, base_seed=5000 + seed, unique=min(unique, n_streams))).astype(np.float32)


def to_format(x, fmt):
    if fmt == F32:
        return x, x
    q = S.pcm_encode(x, fmt)
    return (q if fmt == S16 else S.pack_s24(q)), S.pcm_decode(q, fmt)


def as_bytes(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(a.shape[0], a.shape[1], -1)


class BusReference:
    """The reference encode of a grouped call's buses: rows numbered from 2S, position and error history carried."""

    def __init__(self, fmt, n_streams, first, mode, seed=0x5EED):
        self.fmt, self.first, self.mode, self.seed = fmt, first, mode, seed
        self.first_row, self.pos, self.state = 2 * n_streams, 0, None

    def encode(self, bus):
        if self.mode is None:
            q = S.pcm_encode(bus, self.fmt)
        else:
            q, self.state = S.pcm_encode_dithered(bus, self.fmt, self.seed, self.pos, self.mode, self.state, first_row=self.first_row)
        self.pos += bus.shape[-1]
        return as_bytes(q if self.fmt == S16 else S.pack_s24(q))

    def __call__(self, y):
        return self.encode(S.mix_groups(y, self.first))


def twin_call(a, b, ref, buf, fmt):
    want = ref(a.process_pcm(buf, F32))
    got = as_bytes(b.process_grouped(buf, bus_format=fmt))
    assert got.shape == want.shape
    assert got.tobytes() == want.tobytes()
    return got


def device_grouped(e, dec, fmt, n, k_blocks=None, block=256):
    """ohs_process_device + ohs_mix_device_pcm on the decoded input: one call, or calls of k_blocks blocks each."""
    import torch

    d = torch.from_numpy(np.ascontiguousarray(dec)).cuda()
    G = e.n_groups
    bus = torch.zeros((G, 2, n * BYTES[fmt]), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # the engine runs on its own stream
    step = n if k_blocks is None else k_blocks * block
    for f0 in range(0, n, step):
        m = min(step, n - f0)
        e.process_device(d.data_ptr() + 4 * f0, d.data_ptr() + 4 * f0, m, row_stride=n)
        e.mix_device(d.data_ptr() + 4 * f0, bus.data_ptr() + BYTES[fmt] * f0, m, row_stride=n, bus_stride=n, bus_format=fmt)
    e.sync()
    return bus.cpu().numpy()


# ---- GPU: bit-exact against the reference ------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("lay", ["7.1", "5.1", "mixed"])
@pytest.mark.parametrize("mode", list(MODES), ids=str)
@pytest.mark.parametrize("fmt", [S16, S24], ids=lambda f: NAME[f])
def test_grouped_integer_buses_config2(fmt, mode, lay):
    """1024 streams (1021 for 5.1, so its last group holds one stream), 8 blocks per call, two calls: position and history
    carry over.  The clipped, +-inf and NaN streams sit in the first groups."""
    n_streams = 1021 if lay == "5.1" else 1024
    first = layout(lay, n_streams)
    n = 256 * 8
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=MODES[mode])
    ref = BusReference(fmt, n_streams, first, MODES[mode])
    for i in range(2):
        buf, _ = to_format(inputs(n_streams, n, seed=i), S16 if i == 0 else fmt)
        got = twin_call(a, b, ref, buf, fmt)
    q = got.view(np.int16) if fmt == S16 else S.unpack_s24(got)
    full = 32767 if fmt == S16 else 2 ** 23 - 1
    assert q.max() == full and q.min() == -full - 1
    g_nan = next(g for g in range(len(first) - 1) if first[g] <= 4 < first[g + 1])
    assert not q[g_nan].any()                                     # the NaN stream's group encodes to zeros


@gpu
@pytest.mark.parametrize("fmt,mode", [(S16, "m2"), (S24, "m9"), (S16, "flat")], ids=["s16-m2", "s24-m9", "s16-flat"])
def test_same_bytes_however_the_render_is_cut(fmt, mode, monkeypatch):
    """One host call, host chunks of one block (OHS_STAGE_MB=1), one device call of ohs_process_device + ohs_mix_device_pcm,
    and K = 1 device calls: the same bytes, equal to the reference."""
    n_streams, n = 1024, 256 * 8
    first = layout("7.1", n_streams)
    buf, dec = to_format(inputs(n_streams, n), fmt)

    def engine():
        return make_engine(n_streams, first, mode=MODES[mode])

    outs = {"host": as_bytes(engine().process_grouped(buf, bus_format=fmt))}
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    outs["host_one_block_chunks"] = as_bytes(engine().process_grouped(buf, bus_format=fmt))
    monkeypatch.delenv("OHS_STAGE_MB")
    outs["device_one_call"] = device_grouped(engine(), dec, fmt, n)
    outs["device_k1_calls"] = device_grouped(engine(), dec, fmt, n, k_blocks=1)
    want = BusReference(fmt, n_streams, first, MODES[mode])(make_engine(n_streams, None).process_pcm(buf, F32))
    for k, v in outs.items():
        assert v.tobytes() == want.tobytes(), k


@gpu
@pytest.mark.parametrize("mode", ["off", "flat", "m2"], ids=str)
@pytest.mark.parametrize("fmt", [S16, S24], ids=lambda f: NAME[f])
def test_eq_only_ragged_frames_leave_the_padding(fmt, mode, monkeypatch):
    """EQ-only mode takes any n_frames: 3109 = 12 blocks + 37 frames, so the last group of the encode is partial; with
    OHS_STAGE_MB=1 the call is cut into chunks of 8 blocks and a ragged one.  Nothing past n_frames of a bus row is written."""
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    n_streams, n, bs = 64, 256 * 12 + 37, 256 * 12 + 37 + 27
    first = mixed_groups(n_streams)
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=MODES[mode])
    for e in (a, b):
        e.set_conv_enable(False)
    ref = BusReference(fmt, n_streams, first, MODES[mode])
    G = len(first) - 1
    for i in range(2):
        buf, _ = to_format(inputs(n_streams, n, seed=i), S24)
        want = ref(a.process_pcm(buf, F32))
        out = np.empty((G, 2, bs * (3 if fmt == S24 else 1)), np.uint8 if fmt == S24 else np.int16)
        out.view(np.uint8)[...] = 0x5A
        got = as_bytes(b.process_grouped(buf, out=out, bus_stride=bs, bus_format=fmt))
        assert got.tobytes() == want.tobytes()
        assert (as_bytes(out)[:, :, n * BYTES[fmt]:] == 0x5A).all()


# ---- GPU: semantics ----------------------------------------------------------------------------------------------
@gpu
def test_bypass_encodes_the_mixed_input_and_moves_the_position():
    n_streams, n = 64, 256 * 3
    first = mixed_groups(n_streams)
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=H2)
    ref = BusReference(S16, n_streams, first, H2)
    b.set_bypass(True)
    before = b.state_export()
    x = 1.7 * inputs(n_streams, n)
    for fi in (F32, S16, S24):
        buf, dec = to_format(x, fi)
        got = as_bytes(b.process_grouped(buf, bus_format=S16))
        assert got.tobytes() == ref(dec).tobytes(), NAME[fi]
    b.set_bypass(False)
    after = b.state_export()
    assert len(after) == len(before) + 8 + 72 * (len(first) - 1)   # a bus has been encoded: the blob carries its history
    header, pos = 56, len(before) - 8 - 72 * n_streams              # the dither section: position, then the stream history
    assert after[header:pos] == before[header:pos]                  # the render state is untouched
    assert struct.unpack_from("<Q", after, pos)[0] == 3 * n         # the position moved on
    buf, _ = to_format(inputs(n_streams, n, seed=1), S16)
    twin_call(a, b, ref, buf, S16)


@gpu
def test_grouped_and_per_stream_calls_share_the_position():
    n_streams, n = 64, 256 * 4
    first = mixed_groups(n_streams)
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=H9)
    ref = BusReference(S16, n_streams, first, H9)
    buf, _ = to_format(inputs(n_streams, n), S16)
    twin_call(a, b, ref, buf, S16)
    buf2, _ = to_format(inputs(n_streams, n, seed=1), S16)
    y = a.process_pcm(buf2, F32)
    q, _ = S.pcm_encode_dithered(y, S16, 0x5EED, n, H9)   # stream rows from 0, at position n, zero stream history
    assert as_bytes(b.process_pcm(buf2, S16)).tobytes() == as_bytes(q).tobytes()
    ref.pos += n
    buf3, _ = to_format(inputs(n_streams, n, seed=2), S16)
    twin_call(a, b, ref, buf3, S16)


@gpu
def test_set_groups_zeroes_the_bus_history():
    n_streams, n = 64, 256 * 4
    first = mixed_groups(n_streams)
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=H2)
    ref = BusReference(S24, n_streams, first, H2)
    buf, _ = to_format(inputs(n_streams, n), S24)
    twin_call(a, b, ref, buf, S24)
    assert np.abs(ref.state).max() > 0.1
    b.set_groups(first)
    ref.state = None
    buf, _ = to_format(inputs(n_streams, n, seed=1), S24)
    twin_call(a, b, ref, buf, S24)


@gpu
@pytest.mark.parametrize("mode", ["flat", "m9"], ids=str)
def test_state_export_mid_render(mode):
    n_streams, n = 256, 256 * 6
    first = layout("7.1", n_streams)
    G = len(first) - 1
    q1, _ = to_format(inputs(n_streams, n), S24)
    q2, _ = to_format(inputs(n_streams, n, seed=1), S24)
    dithered = make_engine(n_streams, first, mode=MODES[mode]).state_export()
    b = make_engine(n_streams, first, mode=MODES[mode])
    b.process_grouped(q1, bus_format=S24)
    blob = b.state_export()
    assert len(blob) == len(dithered) + 8 + 72 * G
    assert struct.unpack_from("<i", blob, 28)[0] == 3 and struct.unpack_from("<i", dithered, 28)[0] == 1
    assert struct.unpack_from("<ii", blob, len(dithered)) == (G, 0)
    want = as_bytes(b.process_grouped(q2, bus_format=S24)).tobytes()
    c = make_engine(n_streams, first, mode=MODES[mode])
    c.state_import(blob)
    assert as_bytes(c.process_grouped(q2, bus_format=S24)).tobytes() == want
    # another group count: rejected, the engine untouched (it renders as a fresh engine does)
    other = mixed_groups(n_streams)
    d = make_engine(n_streams, other, mode=MODES[mode])
    with pytest.raises(ohs.OhsError):
        d.state_import(blob)
    fresh = make_engine(n_streams, other, mode=MODES[mode])
    assert as_bytes(d.process_grouped(q1, bus_format=S24)).tobytes() == as_bytes(fresh.process_grouped(q1, bus_format=S24)).tobytes()
    # bit 1 without bit 0: rejected by an engine whose dither is off
    bad = bytearray(blob)
    struct.pack_into("<i", bad, 28, 2)
    e = make_engine(n_streams, first)
    plain = e.state_export()
    with pytest.raises(ohs.OhsError):
        e.state_import(bytes(bad))
    assert e.state_export() == plain
    # a blob exported before any bus encode has the old format; importing it zeroes the bus history
    p = make_engine(n_streams, first, mode=MODES[mode])
    p.process_pcm(q1, S24)
    old = p.state_export()
    assert len(old) == len(dithered) and struct.unpack_from("<i", old, 28)[0] == 1
    r = make_engine(n_streams, first, mode=MODES[mode])
    r.process_grouped(q2, bus_format=S24)
    r.state_import(old)
    assert r.state_export() == old
    assert as_bytes(r.process_grouped(q2, bus_format=S24)).tobytes() == as_bytes(p.process_grouped(q2, bus_format=S24)).tobytes()


@gpu
def test_f32_bus_through_the_new_call_is_process_grouped():
    lib = ohs.load_library()
    n_streams, n = 64, 256 * 4
    first = mixed_groups(n_streams)
    a, b = make_engine(n_streams, first, mode=H2), make_engine(n_streams, first, mode=H2)
    G = len(first) - 1
    for i in range(2):
        buf, _ = to_format(inputs(n_streams, n, seed=i), S16)
        want = np.zeros((G, 2, n), np.float32)
        assert lib.ohs_process_grouped(a._h, buf.ctypes.data, S16, want.ctypes.data, n, n, n) == 0
        got = b.process_grouped(buf, bus_format=F32)
        assert got.dtype == np.float32 and np.ascontiguousarray(got).tobytes() == want.tobytes()
    assert a.state_export() == b.state_export()   # the position has not moved, and no bus history is carried


@gpu
def test_launch_counts():
    """A grouped integer call issues as many launches as a grouped F32 call (one mix or mix-encode per chunk), and
    ohs_mix_device_pcm is one launch in every mode."""
    import torch

    n_streams, n = 1024, 256 * 4
    first = layout("7.1", n_streams)
    buf, _ = to_format(inputs(n_streams, n), S16)
    y = torch.zeros((n_streams, 2, n), dtype=torch.float32, device="cuda")
    bus = torch.zeros((len(first) - 1, 2, 4 * n), dtype=torch.uint8, device="cuda")   # room for an F32 bus
    counts = set()
    for mode in MODES.values():
        for fmt in (F32, S16, S24):
            e = make_engine(n_streams, first, mode=mode)
            e.process_grouped(buf, bus_format=fmt)   # set-up launches
            c0 = e.launch_count()
            e.process_grouped(buf, bus_format=fmt)
            counts.add(e.launch_count() - c0)
            torch.cuda.synchronize()
            c0 = e.launch_count()
            e.mix_device(y.data_ptr(), bus.data_ptr(), n, bus_format=fmt)
            assert e.launch_count() - c0 == 1
            e.sync()
    assert len(counts) == 1, counts


@gpu
def test_rejected_calls_leave_the_engine_untouched():
    import torch

    lib = ohs.load_library()
    n_streams, n = 16, 256 * 2
    first = [0, 3, 4, 9, 16]
    G = len(first) - 1
    a, b = make_engine(n_streams, None), make_engine(n_streams, first, mode=H2)
    ref = BusReference(S16, n_streams, first, H2)
    buf, _ = to_format(inputs(n_streams, n), S16)
    twin_call(a, b, ref, buf, S16)
    blob = b.state_export()
    q = np.ascontiguousarray(buf)
    bus = np.zeros((G, 2, n), np.int16)
    qp, bp = q.ctypes.data, bus.ctypes.data
    h = b._h
    assert lib.ohs_process_grouped_pcm(h, qp, S16, bp, 3, n, n, n) == ERR_INVALID            # unknown bus format
    assert lib.ohs_process_grouped_pcm(h, qp, S16, bp, -1, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped_pcm(h, qp, 5, bp, S16, n, n, n) == ERR_INVALID            # unknown input format
    assert lib.ohs_process_grouped_pcm(h, qp, S16, None, S16, n, n, n) == ERR_INVALID        # null bus
    assert lib.ohs_process_grouped_pcm(h, None, S16, bp, S16, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped_pcm(h, qp, S16, bp, S16, n, n, n - 8) == ERR_INVALID      # short bus_stride
    assert lib.ohs_process_grouped_pcm(h, qp, S16, bp, S16, n - 16, n, n) == ERR_INVALID     # not whole blocks
    assert lib.ohs_process_grouped_pcm(h, qp, S16, bp, S16, n, n - 8, n) == ERR_INVALID      # row_stride < n_frames
    # overlaps are measured in the bus's bytes: an S24 bus of 2G rows spans 3 * 2G * n bytes, an S16 one 2 * 2G * n
    big = np.zeros(3 * 2 * G * n + 2 * n_streams * n * 2, np.uint8)
    bp2 = big.ctypes.data
    assert lib.ohs_process_grouped_pcm(h, bp2 + 2 * 2 * G * n + 2, S16, bp2, S24, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped_pcm(h, qp, S16, qp + 64, S16, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped_pcm(h, qp + 64, S16, qp, S24, n, n, n) == ERR_INVALID
    # the device call
    y = torch.zeros((n_streams, 2, n), dtype=torch.float32, device="cuda")
    dbus = torch.zeros((G, 2, 3 * n + 64), dtype=torch.uint8, device="cuda")
    yp, dp = y.data_ptr(), dbus.data_ptr()
    assert lib.ohs_mix_device_pcm(h, yp, dp, 3, n, n, n) == ERR_INVALID                    # unknown bus format
    assert lib.ohs_mix_device_pcm(h, yp, None, S16, n, n, n) == ERR_INVALID                # null bus
    assert lib.ohs_mix_device_pcm(h, yp, dp, S16, n, n, n + 4) == ERR_ALIGNMENT            # bus_stride not 8 frames
    assert lib.ohs_mix_device_pcm(h, yp, dp, S24, n, n, n + 8) == ERR_ALIGNMENT            # bus_stride not 16 frames
    assert lib.ohs_mix_device_pcm(h, yp, dp + 2, S16, n, n, n) == ERR_ALIGNMENT            # misaligned bus
    assert lib.ohs_mix_device_pcm(h, yp, dp, S16, n - 2, n, n) == ERR_ALIGNMENT            # n_frames not 4 frames
    assert lib.ohs_mix_device_pcm(h, yp, dp, S16, n, n, n - 8) == ERR_INVALID              # bus_stride < n_frames
    assert lib.ohs_mix_device_pcm(h, yp, dp, S16, n, n - 4, n) == ERR_INVALID              # row_stride < n_frames
    assert lib.ohs_mix_device_pcm(h, yp, dp, F32, n, n, n + 2) == ERR_ALIGNMENT            # F32: ohs_mix_device's rules
    b.sync()
    assert b.state_export() == blob
    assert not bus.any() and not dbus.cpu().numpy().any() and not big.any()
    buf, _ = to_format(inputs(n_streams, n, seed=1), S16)
    twin_call(a, b, ref, buf, S16)
