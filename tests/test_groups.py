"""Listener buses (include/ohs.h: ohs_set_groups, ohs_process_grouped, grouped ohs_mix_device).  Every bus is defined bit
for bit against calls that already exist, so the GPU cases run twin engines: A renders with ohs_process_pcm(..., F32) and
its rows are mixed by the numpy reference (signals.mix_groups); B renders the same input with ohs_process_grouped.  The
buses must be byte-identical, and so must the state blobs and a follow-up plain call on both."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S
from oracle import oracle as O

gpu = pytest.mark.gpu
F32, S16, S24 = ohs.FMT_F32, ohs.FMT_S16, ohs.FMT_S24
NAME = {F32: "f32", S16: "s16", S24: "s24"}
FS = 48000.0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = np.int32(0x7FA5A5A5)   # a signalling-NaN bit pattern no render or mix produces
ERR_INVALID = -1


def mixed_groups(n_streams, sizes=(1, 2, 3, 4, 7)):
    """Group offsets with sizes cycling through `sizes`, the last group the remainder."""
    first, k = [0], 0
    while first[-1] < n_streams:
        first.append(min(n_streams, first[-1] + sizes[k % len(sizes)]))
        k += 1
    return first


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_symbols_are_declared_and_bound():
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ohs.h")).read(), flags=re.S)
    lib = ohs.load_library()
    bound = {s[0] for s in ohs.SYMBOLS}
    for name in ("ohs_set_groups", "ohs_num_groups", "ohs_process_grouped", "ohs_mix_device"):
        assert re.search(r"\b%s\s*\(" % name, hdr), name
        assert name in bound and hasattr(lib, name), name


def test_mix_groups_is_an_explicit_sequential_sum():
    rng = np.random.default_rng(3)
    n_streams, n = 23, 37
    y = (rng.standard_normal((n_streams, 2, n)) * np.exp2(rng.integers(-20, 20, (n_streams, 2, n)))).astype(np.float32)
    y[5:7, :, :4] = -0.0                    # a group of negative zeros only sums to +0 (the sum starts from +0)
    first = [0, 1, 3, 5, 7, 11, 18, 23]
    got = S.mix_groups(y, first)
    assert got.dtype == np.float32 and got.shape == (7, 2, n)
    for g in range(7):
        for c in range(2):
            for i in range(n):
                acc = np.float32(0.0)
                for s in range(first[g], first[g + 1]):
                    acc = np.float32(acc + y[s, c, i])
                assert got[g, c, i].tobytes() == acc.tobytes(), (g, c, i)
    assert not np.signbit(got[3, :, :4]).any()
    # one group of every stream is the config 4 mixdown
    one = np.zeros((2, n), np.float32)
    for s in range(n_streams):
        one = (one + y[s]).astype(np.float32)
    assert S.mix_groups(y, [0, n_streams])[0].tobytes() == one.tobytes()


def test_null_handle_without_a_device():
    lib = ohs.load_library()
    first = (C.c_int32 * 2)(0, 1)
    assert lib.ohs_set_groups(None, first, 1) == ERR_INVALID
    n = C.c_int()
    assert lib.ohs_num_groups(None, C.byref(n)) == ERR_INVALID
    assert lib.ohs_process_grouped(None, None, S16, None, 256, 256, 256) == ERR_INVALID
    assert lib.ohs_process_grouped(None, None, 7, None, 256, 256, 256) == ERR_INVALID


def test_python_argument_checks_without_a_device():
    e = ohs.Engine.__new__(ohs.Engine)
    e.n_streams = 2
    with pytest.raises(ValueError):
        e.process_grouped(np.zeros((2, 2, 8), np.int32))           # not a PCM dtype
    with pytest.raises(ValueError):
        e.process_grouped(np.zeros((3, 2, 8), np.float32))         # wrong stream count
    with pytest.raises(ValueError):
        e.set_groups([0])                                          # no group at all


# ---- GPU helpers ------------------------------------------------------------------------------------------------
def make_engine(n_streams, block=256, taps=256, n_sets=3, eq=True, seed=5):
    """Config 2 shape: 256-tap HRIRs, block 256, 10-band PEQ; `n_sets` HRIR sets bound s % n_sets, per-stream gains."""
    e = ohs.Engine(n_streams, block, taps, n_hrir_sets=n_sets, sample_rate=FS)
    for k in range(n_sets):
        e.set_hrir_set(S.synthetic_hrir_set(taps - 17 * k, (taps - 17 * k) / 6.0, seed=seed + k), hrir_set=k)
    for s in range(n_streams):
        if n_sets > 1:
            e.bind_stream_hrir(s, s % n_sets)
        e.set_gain(float((0.25, 0.5, -0.75, 1.5, 0.0)[s % 5]), s)
    if eq:
        e.eq_set_preset(S.EQ_PRESET_TYPICAL)
        e.set_eq_enable(True)
    return e


def inputs(n_streams, n, seed=0, unique=64):
    return (0.9 * S.stream_inputs(n_streams, n, base_seed=4000 + seed, unique=min(unique, n_streams))).astype(np.float32)


def to_format(x, fmt):
    """f32 rows -> (the buffer as the API takes it in `fmt`, its decode)."""
    if fmt == F32:
        return x, x
    q = S.pcm_encode(x, fmt)
    return (q if fmt == S16 else S.pack_s24(q)), S.pcm_decode(q, fmt)


def twin_call(a, b, buf, first, bus_out=None):
    """A: ohs_process_pcm(buf, F32) mixed by the reference; B: ohs_process_grouped(buf).  Asserts equal bytes."""
    want = S.mix_groups(a.process_pcm(buf, F32), first)
    got = b.process_grouped(buf, out=bus_out)
    assert got.shape == want.shape
    assert np.ascontiguousarray(got).tobytes() == want.tobytes()
    return got


def same_state(a, b, z):
    assert a.state_export() == b.state_export()
    ya, yb = a.process(z), b.process(z)
    assert ya.tobytes() == yb.tobytes()


def twins(n_streams, first, **kw):
    a, b = make_engine(n_streams, **kw), make_engine(n_streams, **kw)
    b.set_groups(first)
    return a, b


# ---- 1. config 2 width, mixed group sizes, every input format -------------------------------------------------------
@gpu
@pytest.mark.parametrize("fi", [F32, S16, S24], ids=lambda f: NAME[f])
def test_grouped_equals_pcm_render_config2(fi):
    n_streams, n = 1024, 256 * 8
    first = mixed_groups(n_streams)
    assert first[-4:] == [1020, 1021, 1023, 1024]   # 60 rounds of (1, 2, 3, 4, 7), then 1, 2 and a remainder of 1
    a, b = twins(n_streams, first)
    for i in range(2):   # the second call continues from the first one's state
        buf, _ = to_format(inputs(n_streams, n, seed=i), fi)
        got = twin_call(a, b, buf, first)
        assert np.abs(got).max() > 0.01
    same_state(a, b, inputs(n_streams, 512, seed=7))


# ---- 2. several chunks, pageable and pinned host memory ---------------------------------------------------------------
@gpu
@pytest.mark.parametrize("fi", [F32, S16, S24], ids=lambda f: NAME[f])
@pytest.mark.parametrize("memory", ["pageable", "pinned"])
def test_several_chunks(fi, memory, monkeypatch):
    """OHS_STAGE_MB=1 and 64 streams: chunks of 8 blocks (F32 rows decide, whatever the input format), 37 blocks per call,
    so the last chunk is ragged and every pipeline slot is reused."""
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    n_streams, n = 64, 256 * 37
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    G = len(first) - 1
    for i in range(2):
        buf, _ = to_format(inputs(n_streams, n, seed=i), fi)
        if memory == "pageable":
            twin_call(a, b, buf, first)
        else:
            pin_in = ohs.PinnedBuffer(buf.shape, buf.dtype)
            pin_bus = ohs.PinnedBuffer((G, 2, n), np.float32)
            pin_in.array[...] = buf
            twin_call(a, b, pin_in.array, first, bus_out=pin_bus.array)
            pin_in.free(); pin_bus.free()
    same_state(a, b, inputs(n_streams, 1024, seed=2))


@gpu
def test_padded_bus_stride_leaves_the_padding():
    n_streams, n, bs = 64, 256 * 5, 256 * 5 + 12
    first = mixed_groups(n_streams, (4,))
    a, b = twins(n_streams, first)
    buf, _ = to_format(inputs(n_streams, n), S16)
    out = np.empty((len(first) - 1, 2, bs), np.float32)
    out.view(np.int32)[...] = SENTINEL
    want = S.mix_groups(a.process_pcm(buf, F32), first)
    got = b.process_grouped(buf, out=out, bus_stride=bs)
    assert np.ascontiguousarray(got).tobytes() == want.tobytes()
    assert (out[:, :, n:].view(np.int32) == SENTINEL).all()
    with pytest.raises(ValueError):   # an `out` of the wrong shape for the groups in force
        b.process_grouped(buf, out=np.empty((len(first) - 2, 2, bs), np.float32), bus_stride=bs)


@gpu
def test_group_count_is_read_from_the_library():
    """Engine.n_groups follows ohs_set_groups made on the raw handle, so process_grouped shapes its buses right."""
    lib = ohs.load_library()
    n_streams = 16
    a, b = twins(n_streams, [0, 16])
    assert a.n_groups == 1 and b.n_groups == 1
    first = [0, 2, 5, 16]
    assert lib.ohs_set_groups(b._h, (C.c_int32 * 4)(*first), 3) == 0
    assert b.n_groups == 3
    buf, _ = to_format(inputs(n_streams, 512), S16)
    assert twin_call(a, b, buf, first).shape == (3, 2, 512)


# ---- 3. the time-batched route ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("fi", [F32, S16], ids=lambda f: NAME[f])
def test_time_batched_route(fi):
    """9 partitions at block 128 and 40 blocks per call: the time-batched route.  Same chunks, so still bit-exact."""
    n_streams, block, taps = 12, 128, 1100
    first = [0, 1, 3, 7, 12]
    a, b = twins(n_streams, first, block=block, taps=taps, n_sets=2)
    for i in range(2):
        buf, _ = to_format(inputs(n_streams, block * 40, seed=i), fi)
        twin_call(a, b, buf, first)
    same_state(a, b, inputs(n_streams, block * 3, seed=4))


# ---- 4. semantics ----------------------------------------------------------------------------------------------------
@gpu
def test_bypass_mixes_the_decoded_input_and_keeps_the_state():
    n_streams, n = 64, 256 * 3
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    b.set_bypass(True)
    before = b.state_export()
    x = 1.7 * inputs(n_streams, n)
    for fi in (F32, S16, S24):
        buf, dec = to_format(x, fi)
        got = b.process_grouped(buf)
        assert np.ascontiguousarray(got).tobytes() == S.mix_groups(dec, first).tobytes(), NAME[fi]
    assert b.state_export() == before
    b.set_bypass(False)
    same_state(a, b, inputs(n_streams, 512, seed=2))


@gpu
def test_eq_only_ragged_frames(monkeypatch):
    """EQ-only mode takes any n_frames: 3109 = 12 blocks + 37 frames, so the mix's last quad is partial (1 frame); with
    OHS_STAGE_MB=1 the call is cut into chunks of 8 blocks and a ragged one."""
    monkeypatch.setenv("OHS_STAGE_MB", "1")
    n_streams, n = 64, 256 * 12 + 37
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    for e in (a, b):
        e.set_conv_enable(False)
    for fi in (S24, F32, S16):
        buf, _ = to_format(inputs(n_streams, n, seed=fi), fi)
        twin_call(a, b, buf, first)
    same_state(a, b, inputs(n_streams, 333, seed=9))


@gpu
def test_pending_move_applies_as_in_the_pcm_call():
    n_streams = 64
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    buf, _ = to_format(inputs(n_streams, 256 * 4), S16)
    twin_call(a, b, buf, first)
    for e in (a, b):
        e.move_stream_hrir(ohs.OHS_ALL, 2)
    buf, _ = to_format(inputs(n_streams, 256 * 4, seed=1), S16)
    twin_call(a, b, buf, first)
    same_state(a, b, inputs(n_streams, 512, seed=2))


@gpu
def test_dither_position_does_not_move():
    """With dither on, the state blob carries the dither position.  A's F32-output call does not move it, and B's grouped
    call must leave the same blob."""
    n_streams = 64
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    for e in (a, b):
        e.set_dither(ohs.DITHER_TPDF, seed=11, shape=(2.0, -1.0))
    buf, _ = to_format(inputs(n_streams, 256 * 4), S24)
    twin_call(a, b, buf, first)
    assert a.state_export() == b.state_export()
    # an integer-output call on both afterwards encodes at the same position
    z, _ = to_format(inputs(n_streams, 512, seed=3), S16)
    assert a.process_pcm(z, S16).tobytes() == b.process_pcm(z, S16).tobytes()


# ---- 5. ohs_mix_device with groups -----------------------------------------------------------------------------------
def padded(x, stride, pad_bits):
    buf = np.empty(x.shape[:-1] + (stride,), np.float32)
    buf.view(np.int32)[...] = pad_bits
    buf[..., :x.shape[-1]] = x
    return buf


@gpu
@pytest.mark.parametrize("n_frames", [4, 1028, 3 * 1024 + 4])
@pytest.mark.parametrize("n_streams,first", [(7, None), (1023, "mixed"), (1024, "quads"), (5, [0, 1, 2, 3, 4, 5])])
def test_mix_device_groups(n_streams, first, n_frames):
    """Padded row and bus strides, NaN in the input padding, the bus padding untouched; first=None is the default group
    (today's config 4 mixdown, a sequential f32 sum from +0 over every stream)."""
    import torch

    if first == "mixed":
        first = mixed_groups(n_streams)
    elif first == "quads":
        first = list(range(0, n_streams + 1, 4))
    rng = np.random.default_rng(n_streams * 7 + n_frames)
    x = (rng.standard_normal((n_streams, 2, n_frames)) * np.exp2(rng.integers(-10, 10, (n_streams, 2, n_frames)))).astype(np.float32)
    x[:, :, :4] = -0.0
    row_stride, bus_stride = n_frames + 12, n_frames + 8
    e = ohs.Engine(n_streams, 256, 1, n_bands=0)
    if first is not None:
        e.set_groups(first)
    G = 1 if first is None else len(first) - 1
    src = torch.from_numpy(padded(x, row_stride, np.float32(np.nan).view(np.int32))).cuda()
    bus = torch.from_numpy(padded(np.zeros((G, 2, n_frames), np.float32), bus_stride, SENTINEL)).cuda()
    e.mix_device(src.data_ptr(), bus.data_ptr(), n_frames, row_stride=row_stride, bus_stride=bus_stride)
    e.sync()
    got = bus.cpu().numpy()
    want = S.mix_groups(x, [0, n_streams] if first is None else first)
    assert got[:, :, :n_frames].tobytes() == want.tobytes()
    assert not np.signbit(got[:, :, :4]).any()                 # every term -0: the bus is +0
    assert (got[:, :, n_frames:].view(np.int32) == SENTINEL).all()


@gpu
def test_groups_change_no_stream_rendering():
    """Groups are configuration: the device render and the state blob do not see them."""
    import torch

    n_streams, n = 64, 256 * 4
    a, b = make_engine(n_streams), make_engine(n_streams)
    b.set_groups(mixed_groups(n_streams))
    x = torch.from_numpy(inputs(n_streams, n)).cuda()
    ya, yb = torch.empty_like(x), torch.empty_like(x)
    a.process_device(x.data_ptr(), ya.data_ptr(), n)
    b.process_device(x.data_ptr(), yb.data_ptr(), n)
    a.sync(); b.sync()
    assert ya.cpu().numpy().tobytes() == yb.cpu().numpy().tobytes()
    assert a.state_export() == b.state_export()


# ---- 6. a 7.1 layout from the CIPIC fixture ---------------------------------------------------------------------------
# (left, right) speakers of each pair, plugin UI azimuths (negative = left): front, centre + LFE, side, back
LAYOUT_71 = [(-30.0, 30.0), (0.0, 0.0), (-90.0, 90.0), (-135.0, 135.0)]


@gpu
def test_surround_71_against_the_oracle(cipic):
    from open_headstage_b200 import sofa

    hr = sofa.from_arrays(cipic["ir"], cipic["pos"], float(cipic["fs"]))
    n_files, pairs, block, gain = 6, len(LAYOUT_71), 256, 0.25
    n_streams, n = n_files * pairs, 256 * 12
    e = ohs.Engine(n_streams, block, hr.filter_length, n_hrir_sets=pairs, sample_rate=FS)
    idx = []
    for k, (az_l, az_r) in enumerate(LAYOUT_71):
        idx.append(sofa.wire_speakers(e, hr, sofa.ui_azimuth_to_sofa(az_l), 0.0, sofa.ui_azimuth_to_sofa(az_r), 0.0, hrir_set=k))
    for s in range(n_streams):
        e.bind_stream_hrir(s, s % pairs)      # stream s is pair s % pairs of file s // pairs
    e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(gain)
    first = list(range(0, n_streams + 1, pairs))
    e.set_groups(first)
    x = S.stream_inputs(n_streams, n, base_seed=1900)
    bus = e.process_grouped(S.pcm_encode(x, S16))
    dec = S.pcm_decode(S.pcm_encode(x, S16), S16)
    coeffs = np.stack([O.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    ref = np.zeros((n_streams, 2, n), np.float64)
    for k, (il, ir_) in enumerate(idx):
        irs = [hr.ir[il, 0], hr.ir[il, 1], hr.ir[ir_, 0], hr.ir[ir_, 1]]
        y, _ = O.render_batch(dec[k::pairs], block, irs, coeffs, [1] * 10, True, gain, n_threads=8)
        ref[k::pairs] = y
    want = ref.reshape(n_files, pairs, 2, n).sum(axis=1)
    assert bus.shape == (n_files, 2, n)
    assert float(np.max(np.abs(bus - want))) <= 1e-5
    assert np.abs(bus).max() > 0.05


# ---- 7. rejections -----------------------------------------------------------------------------------------------------
@gpu
def test_rejected_calls_leave_the_engine_untouched():
    lib = ohs.load_library()
    n_streams, n = 16, 256 * 2
    first = [0, 3, 4, 9, 16]
    a, b = twins(n_streams, first)
    blob = b.state_export()

    def groups(vals, count):
        arr = (C.c_int32 * len(vals))(*vals)
        return lib.ohs_set_groups(b._h, arr, count)

    assert groups([1, 16], 1) == ERR_INVALID                   # first[0] != 0
    assert groups([0, 15], 1) == ERR_INVALID                   # does not end at n_streams
    assert groups([0, 5, 5, 16], 3) == ERR_INVALID             # an empty group
    assert groups([0, 9, 4, 16], 3) == ERR_INVALID             # decreasing
    assert groups([0, 16], 0) == ERR_INVALID                   # no group
    assert groups(list(range(18)), 17) == ERR_INVALID          # more groups than streams
    assert lib.ohs_set_groups(b._h, None, 1) == ERR_INVALID
    x = inputs(n_streams, n)
    q = np.ascontiguousarray(S.pcm_encode(x, S16))
    G = len(first) - 1
    bus = np.zeros((G, 2, n), np.float32)
    qp, bp = q.ctypes.data, bus.ctypes.data
    assert lib.ohs_process_grouped(b._h, qp, 3, bp, n, n, n) == ERR_INVALID            # unknown format
    assert lib.ohs_process_grouped(b._h, qp, -1, bp, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped(b._h, qp, S16, None, n, n, n) == ERR_INVALID         # null bus
    assert lib.ohs_process_grouped(b._h, None, S16, bp, n, n, n) == ERR_INVALID
    assert lib.ohs_process_grouped(b._h, qp, S16, bp, n, n, n - 4) == ERR_INVALID       # short bus_stride
    assert lib.ohs_process_grouped(b._h, qp, S16, bp, n - 16, n, n) == ERR_INVALID      # not whole blocks
    assert lib.ohs_process_grouped(b._h, qp, S16, bp, n, n - 8, n) == ERR_INVALID       # row_stride < n_frames
    assert lib.ohs_process_grouped(b._h, qp, S16, qp + 64, n, n, n) == ERR_INVALID      # the bus overlaps the input
    assert lib.ohs_process_grouped(b._h, qp + 64, S16, qp, n, n, n) == ERR_INVALID
    assert b.state_export() == blob
    assert not bus.any()
    # one stream per group: the 2G bus rows have exactly the input's layout, and still the bus may not be the input
    c = make_engine(4)
    c.set_groups([0, 1, 2, 3, 4])
    blob_c = c.state_export()
    x4 = inputs(4, n)
    keep = x4.tobytes()
    assert lib.ohs_process_grouped(c._h, x4.ctypes.data, F32, x4.ctypes.data, n, n, n) == ERR_INVALID
    assert c.state_export() == blob_c and x4.tobytes() == keep
    # the groups set before the rejected calls are still in force
    twin_call(a, b, q, first)
    same_state(a, b, inputs(n_streams, 512, seed=2))


# ---- 8. launch count -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("stage_mb,n_streams,blocks,chunks", [(None, 1024, 4, 1), ("1", 64, 37, 5)])
def test_one_extra_launch_per_chunk(stage_mb, n_streams, blocks, chunks, monkeypatch):
    if stage_mb:
        monkeypatch.setenv("OHS_STAGE_MB", stage_mb)
    first = mixed_groups(n_streams)
    a, b = twins(n_streams, first)
    buf, _ = to_format(inputs(n_streams, 256 * blocks), S16)
    for _ in range(2):   # the second round has no set-up launches
        a0, b0 = a.launch_count(), b.launch_count()
        twin_call(a, b, buf, first)
    assert b.launch_count() - b0 == a.launch_count() - a0 + chunks
