"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C ABI, against the CPU oracle
on identical seeded inputs.

Bars (BASELINE.json north_star):
  * EQ stage: BIT-EXACT against the oracle's sequential f32 DF2T cascade.
  * convolution / whole chain: max abs error <= 1e-5 of full scale (inputs peak-normalised to 1.0), EQ compared from
    the same zero state.
"""
import numpy as np
import pytest
import scipy.signal as sps

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5  # north_star: max abs error <= 1e-5 full scale (-100 dBFS)
FS = 48000.0


def preset_coeffs(preset, fs=FS):
    return np.stack([ohs.eq_design(t, fs, fc, q, g) for (t, fc, q, g) in preset])


def oracle_render(x, block, irs, coeffs=None, enabled=None, gain=1.0, host_block=None):
    eq_on = coeffs is not None
    if coeffs is None:
        coeffs, enabled = np.zeros((1, 5), np.float32), [0]
    y, _ = O.render_batch(x, block, irs, coeffs, enabled, eq_on, gain, host_block=host_block, n_threads=8)
    return y


# ------------------------------------------------------------------------------------------------------------
# the reference's own unit tests, replayed through the mirror objects on the GPU
# ------------------------------------------------------------------------------------------------------------
def test_ref_identity_ir_passthrough():
    """src/dsp/convolution.rs:317-347"""
    e = ohs.ConvolutionEngine(512)
    e.set_ir(ohs.LSL, [1.0]); e.set_ir(ohs.LSR, [0.0]); e.set_ir(ohs.RSL, [0.0]); e.set_ir(ohs.RSR, [1.0])
    i = np.arange(512, dtype=np.float32)
    in_l = np.sin(i * np.float32(0.1)).astype(np.float32)
    in_r = np.sin(i * np.float32(-0.1)).astype(np.float32)
    e.process_block(in_l, in_r)
    out_l, out_r = e.process_block(in_l, in_r)
    assert np.max(np.abs(out_l - in_l)) < 1e-3 and np.max(np.abs(out_r - in_r)) < 1e-3
    assert np.max(np.abs(out_l - in_l)) < 1e-6  # and far inside the reference's own tolerance


def test_ref_delay_ir():
    """src/dsp/convolution.rs:349-383"""
    e = ohs.ConvolutionEngine(512)
    ir = np.zeros(6, np.float32); ir[5] = 1.0
    e.set_ir(ohs.LSL, ir); e.set_ir(ohs.LSR, [0.0]); e.set_ir(ohs.RSL, [0.0]); e.set_ir(ohs.RSR, [0.0])
    in_l = np.arange(1024, dtype=np.float32)
    out_l, out_r = e.process_block(in_l, np.zeros(1024, np.float32))
    expected = np.zeros_like(in_l); expected[5:] = in_l[:-5]
    assert np.max(np.abs(out_l[5:] - expected[5:])) < 1e-3
    assert np.max(np.abs(out_r)) < 1e-3


def test_ref_long_ir_partitioning():
    """src/dsp/convolution.rs:385-421"""
    e = ohs.ConvolutionEngine(512)
    ir = np.zeros(768, np.float32); ir[0] = 1.0; ir[-1] = 0.5
    e.set_ir(ohs.LSL, ir)
    assert e.num_partitions(ohs.LSL) == 2
    in_l = np.zeros(1536, np.float32); in_l[0] = 1.0
    out_l, _ = e.process_block(in_l, np.zeros_like(in_l))
    expected = np.zeros_like(in_l); expected[0] = 1.0; expected[767] = 0.5
    assert np.max(np.abs(out_l[:768] - expected[:768])) < 1e-3


def test_ref_biquad_passthrough_when_disabled():
    """src/dsp/parametric_eq.rs:218-225 (assert_eq: exact)"""
    q = ohs.StereoParametricEQ(1, FS)
    l, r = q.process_block([0.5], [0.5])
    assert l[0] == np.float32(0.5) and r[0] == np.float32(0.5)


def test_ref_biquad_processes_when_enabled():
    """src/dsp/parametric_eq.rs:227-238"""
    q = ohs.StereoParametricEQ(1, FS)
    q.update_band_coeffs(0, FS, ohs.BandConfig(ohs.LOWPASS, 1000.0, 0.707, 0.0, True))
    l, _ = q.process_block([0.5], [0.5])
    assert l[0] != np.float32(0.5)
    ql = O.StereoParametricEQ(1, FS)
    ql.update_band_coeffs(0, FS, O.LOWPASS, 1000.0, 0.707, 0.0, True)
    assert l[0] == ql.process_block([0.5], [0.5])[0][0]


# ------------------------------------------------------------------------------------------------------------
# EQ: bit-exact
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("preset_name", ["typical", "harsh"])
@pytest.mark.parametrize("n_streams,block,n_frames", [(1, 256, 4096), (7, 128, 3000), (4, 512, 5120), (3, 64, 1000), (2, 1024, 5000), (5, 1024, 8192)])
def test_eq_bit_exact(preset_name, n_streams, block, n_frames):
    preset = S.EQ_PRESET_TYPICAL if preset_name == "typical" else S.EQ_PRESET_HARSH
    coeffs = preset_coeffs(preset)
    x = S.stream_inputs(n_streams, n_frames, base_seed=50)
    e = ohs.Engine(n_streams, block, 1)
    e.set_conv_enable(False); e.set_eq_enable(True)
    for b in range(10):
        e.eq_set_band(b, coeffs[b], True)
    y = e.process(x)
    for s in range(n_streams):
        q = O.StereoParametricEQ(10, FS)
        for b in range(10):
            q.set_band_raw(b, coeffs[b], True)
        l, r = q.process_block(x[s, 0], x[s, 1])
        assert y[s, 0].tobytes() == l.tobytes(), "stream %d left differs (max %g)" % (s, np.max(np.abs(y[s, 0] - l)))
        assert y[s, 1].tobytes() == r.tobytes()
    assert np.isfinite(y).all()


def test_eq_state_carries_across_calls_and_resets():
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    x = S.stream_inputs(2, 2000, base_seed=70)
    e = ohs.Engine(2, 256, 1)
    e.set_conv_enable(False); e.set_eq_enable(True)
    for b in range(10):
        e.eq_set_band(b, coeffs[b], b != 4)  # one band disabled: exact skip, state untouched (:118-120)
    whole = e.process(x)
    e.eq_reset()
    parts = np.concatenate([e.process(x[:, :, a:a + 333]) for a in range(0, 2000, 333)], axis=2)
    assert parts.tobytes() == whole.tobytes()
    q = O.StereoParametricEQ(10, FS)
    for b in range(10):
        q.set_band_raw(b, coeffs[b], b != 4)
    l, r = q.process_block(x[1, 0], x[1, 1])
    assert whole[1, 0].tobytes() == l.tobytes() and whole[1, 1].tobytes() == r.tobytes()


def test_eq_disabled_engine_switch_is_exact_passthrough():
    x = S.stream_inputs(2, 512, base_seed=80)
    e = ohs.Engine(2, 256, 1)
    e.set_conv_enable(False); e.set_eq_enable(False)
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    assert e.process(x).tobytes() == x.tobytes()


def test_eq_sets_bound_per_stream():
    ca, cb = preset_coeffs(S.EQ_PRESET_TYPICAL), preset_coeffs(S.EQ_PRESET_HARSH)
    x = S.stream_inputs(5, 1024, base_seed=90)
    e = ohs.Engine(5, 256, 1, n_eq_sets=2)
    e.set_conv_enable(False); e.set_eq_enable(True)
    for b in range(10):
        e.eq_set_band(b, ca[b], True, eq_set=0)
        e.eq_set_band(b, cb[b], True, eq_set=1)
    for s in (1, 3):
        e.bind_stream_eq(s, 1)
    y = e.process(x)
    for s in range(5):
        q = O.StereoParametricEQ(10, FS)
        c = cb if s in (1, 3) else ca
        for b in range(10):
            q.set_band_raw(b, c[b], True)
        l, _ = q.process_block(x[s, 0], x[s, 1])
        assert y[s, 0].tobytes() == l.tobytes()


# ------------------------------------------------------------------------------------------------------------
# convolution: <= 1e-5 against the oracle (and against f64 truth)
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("block,taps,n_streams,n_blocks", [
    (64, 200, 2, 20), (128, 512, 5, 16), (256, 256, 7, 12), (256, 100, 3, 8), (512, 200, 2, 10), (512, 1500, 4, 9),
    (1024, 5000, 2, 8), (1024, 1024, 1, 5),
])
def test_conv_parity(block, taps, n_streams, n_blocks):
    h = S.synthetic_hrir_set(taps, taps / 6.0, seed=11)
    n = block * n_blocks
    x = S.stream_inputs(n_streams, n, base_seed=200)
    e = ohs.Engine(n_streams, block, taps, n_bands=0)
    e.set_hrir_set(h)
    for p in range(4):
        assert e.num_partitions(p) == -(-taps // block)
    y = e.process(x)
    ref = oracle_render(x, block, h)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err
    # f64 truth for stream 0
    h64 = h.astype(np.float64)
    tl = (sps.fftconvolve(x[0, 0].astype(np.float64), h64[0]) + sps.fftconvolve(x[0, 1].astype(np.float64), h64[2]))[:n]
    assert np.max(np.abs(y[0, 0] - tl)) <= TOL


@pytest.mark.parametrize("block,taps,n_streams,bands", [(256, 900, 4, 0), (256, 256, 9, 10), (128, 512, 5, 10), (64, 100, 3, 10), (512, 200, 2, 10)])
def test_conv_block_at_a_time_equals_one_long_call(block, taps, n_streams, bands):
    """K = 1 launches (the per-block API: the latency variant of the render kernel, one band per EQ lane, two warps per
    stream in the N = 512 transforms), K = 2 launches and one K = 12 launch (the throughput variant) walk the same
    state: identical bits, multi-partition and single-partition (fused in registers in the throughput variant)."""
    h = S.synthetic_hrir_set(taps, taps / 6.0, seed=3)
    x = S.stream_inputs(n_streams, block * 12, base_seed=300)

    def engine():
        e = ohs.Engine(n_streams, block, taps, n_bands=bands); e.set_hrir_set(h)
        if bands:
            e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
        return e

    whole = engine().process(x)
    for k in (1, 2, 3):
        b = engine()
        parts = np.concatenate([b.process(x[:, :, i:i + k * block]) for i in range(0, x.shape[2], k * block)], axis=2)
        assert whole.tobytes() == parts.tobytes(), k


def test_default_ir_is_silence_and_empty_ir_mutes():
    x = S.stream_inputs(2, 1024, base_seed=310)
    e = ohs.Engine(2, 256, 256, n_bands=0)
    assert not e.process(x).any()                 # ConvolutionPathData::new: zeros (:46-48)
    e.set_ir(ohs.LSL, [1.0]); e.set_ir(ohs.RSR, [1.0])
    assert np.max(np.abs(e.process(x) - x)) < 1e-6
    e.set_ir(ohs.LSL, []); e.set_ir(ohs.RSR, [])  # empty slice -> one silent partition (:114-118)
    assert e.num_partitions(ohs.LSL) == 1
    assert not e.process(x).any()


def test_set_ir_clears_history():
    """set_ir re-creates the ring and zeroes the overlap (:135-138): output restarts as from a fresh engine."""
    h = S.synthetic_hrir_set(700, 100.0, seed=5)
    x = S.stream_inputs(2, 2048, base_seed=320)
    e = ohs.Engine(2, 256, 700, n_bands=0); e.set_hrir_set(h)
    e.process(x)
    e.set_hrir_set(h)
    again = e.process(x)
    fresh = ohs.Engine(2, 256, 700, n_bands=0); fresh.set_hrir_set(h)
    assert again.tobytes() == fresh.process(x).tobytes()


def test_hrir_sets_bound_per_stream_and_ear_routing():
    """out_l = LSL + RSL, out_r = LSR + RSR (:229-230); streams pick their set."""
    ha = S.synthetic_hrir_set(256, 40.0, seed=7)
    hb = S.synthetic_hrir_set(300, 60.0, seed=8)
    x = S.stream_inputs(6, 256 * 6, base_seed=330)
    e = ohs.Engine(6, 256, 300, n_bands=0, n_hrir_sets=2)
    e.set_hrir_set(ha, 0); e.set_hrir_set(hb, 1)
    for s in (0, 2, 5):
        e.bind_stream_hrir(s, 1)
    y = e.process(x)
    for s in range(6):
        ref = oracle_render(x[s:s + 1], 256, hb if s in (0, 2, 5) else ha)
        assert np.max(np.abs(y[s] - ref[0])) <= TOL
    # ear routing with one-hot paths
    e2 = ohs.Engine(1, 256, 8, n_bands=0)
    e2.set_ir(ohs.LSR, [0.0, 1.0])  # left speaker -> right ear, delayed by one sample
    y2 = e2.process(x[:1, :, :512])
    # left + i*right share one complex FFT, so the silent ear carries round-off cross-talk (~1e-8), not exact zero
    assert np.max(np.abs(y2[0, 0])) < 1e-6
    assert np.max(np.abs(y2[0, 1, 1:] - x[0, 0, :511])) < 1e-6


# ------------------------------------------------------------------------------------------------------------
# the whole chain (EQ -> conv -> gain), BASELINE configs at oracle-sized extents
# ------------------------------------------------------------------------------------------------------------
def test_config1_single_stream_sofa_10s(cipic):
    """cfg 1: one stereo stream, 48 kHz, 10 s pink noise, bundled CIPIC HRIRs (30 deg / 330 deg), 10-band PEQ, block 512."""
    ir = cipic["ir"]
    irs = [ir[308, 0], ir[308, 1], ir[908, 0], ir[908, 1]]
    n = 938 * 512  # 10 s = 480 000 frames, zero-padded to whole blocks
    x = np.zeros((1, 2, n), np.float32)
    x[0, 0, :480000] = S.pink_noise(480000, 1)
    x[0, 1, :480000] = S.pink_noise(480000, 2)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    e = ohs.Engine(1, 512, 200)
    e.set_hrir_set(irs)
    for b in range(10):
        e.eq_set_band(b, coeffs[b], True)
    e.set_eq_enable(True); e.set_gain(0.5)
    y = e.process(x)
    ref = oracle_render(x, 512, irs, coeffs, [1] * 10, 0.5)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err
    assert np.abs(y).max() > 0.1


@pytest.mark.parametrize("cfg,n_streams,seconds", [(2, 48, 1.0), (3, 40, 0.5)])
def test_config2_3_chain_parity(cfg, n_streams, seconds):
    c = S.CONFIGS[cfg]
    block, taps = c["block"], c["taps"]
    h = S.synthetic_hrir_set(taps, c["decay"])
    n = int(seconds * c["fs"]) // block * block
    x = S.stream_inputs(n_streams, n)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL, c["fs"])
    e = ohs.Engine(n_streams, block, taps, sample_rate=c["fs"])
    e.set_hrir_set(h)
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True); e.set_gain(0.5)
    y = e.process(x)
    ref = oracle_render(x, block, h, coeffs, [1] * 10, 0.5)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err


@pytest.mark.parametrize("time_batch", ["1", "0"])
def test_config5_long_brir_parity(time_batch, monkeypatch):
    """cfg 5: 48 000-tap BRIR per path, partition 1024, 96 kHz (47 partitions); 3 streams x 60 blocks, through the
    time-batched route and through the block-by-block kernel (TMA filter tiles: 3 streams = two per CTA)."""
    monkeypatch.setenv("OHS_TIME_BATCH", time_batch)
    monkeypatch.setenv("OHS_STREAMS_PER_CTA", "2")
    c = S.CONFIGS[5]
    h = S.synthetic_hrir_set(c["taps"], c["decay"])
    n = 1024 * 60
    x = S.stream_inputs(3, n)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL, c["fs"])
    e = ohs.Engine(3, 1024, c["taps"], sample_rate=c["fs"])
    e.set_hrir_set(h)
    assert e.num_partitions(0) == 47
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True); e.set_gain(0.5)
    y = np.concatenate([e.process(x[:, :, :1024 * 25]), e.process(x[:, :, 1024 * 25:])], axis=2)
    ref = oracle_render(x, 1024, h, coeffs, [1] * 10, 0.5)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err


def test_bypass_gain_and_order():
    h = S.synthetic_hrir_set(256, 40.0)
    x = S.stream_inputs(3, 1024, base_seed=400)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    e = ohs.Engine(3, 256, 256)
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True)
    e.set_bypass(True)
    assert e.process(x).tobytes() == x.tobytes()          # src/lib.rs:1169 buffer untouched, no state advance
    e.set_bypass(False)
    e.set_gain(0.5); e.set_gain(0.25, stream=1)
    y = e.process(x)
    for s, g in ((0, 0.5), (1, 0.25), (2, 0.5)):
        ref = oracle_render(x[s:s + 1], 256, h, coeffs, [1] * 10, g)
        assert np.max(np.abs(y[s] - ref[0])) <= TOL


@pytest.mark.parametrize("n", [100, 256, 512, 700])
def test_fifo_semantics_match_reference(n):
    """src/dsp/convolution.rs:141-182: zero-filled output while starved, latency 512 - n afterwards."""
    h = S.synthetic_hrir_set(300, 50.0, seed=9)
    x = S.stream_inputs(1, n * 9, base_seed=500)
    g = ohs.ConvolutionEngine(512)
    o = O.ConvolutionEngine(512)
    for p in range(4):
        g.set_ir(p, h[p]); o.set_ir(p, h[p])
    for i in range(9):
        seg = x[0, :, i * n:(i + 1) * n]
        gl, gr = g.process_block(seg[0], seg[1])
        ol, orr = o.process_block(seg[0], seg[1])
        assert (not gl.any()) == (not ol.any())
        assert np.max(np.abs(gl - ol)) <= TOL and np.max(np.abs(gr - orr)) <= TOL


def test_state_export_import_resumes_bit_exactly():
    h = S.synthetic_hrir_set(1000, 200.0, seed=4)
    x = S.stream_inputs(3, 256 * 10, base_seed=600)

    def make():
        e = ohs.Engine(3, 256, 1000)
        e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
        return e

    a = make()
    whole = a.process(x)
    b = make()
    first = b.process(x[:, :, :256 * 4])
    blob = b.state_export()
    c = make()
    c.state_import(blob)
    second = c.process(x[:, :, 256 * 4:])
    assert np.concatenate([first, second], axis=2).tobytes() == whole.tobytes()


def test_device_pointers_stride_and_in_place():
    import torch

    h = S.synthetic_hrir_set(256, 40.0)
    x = S.stream_inputs(5, 256 * 8, base_seed=700)
    e = ohs.Engine(5, 256, 256)
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
    want = e.process(x)
    e.conv_reset(); e.eq_reset()
    stride = 256 * 8 + 64
    buf = torch.zeros((5, 2, stride), dtype=torch.float32, device="cuda")
    buf[:, :, :256 * 8] = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    n0 = e.launch_count()
    e.enable_timing(True)
    e.process_device(buf.data_ptr(), buf.data_ptr(), 256 * 8, stride)  # in place, padded rows
    e.sync()
    assert e.launch_count() == n0 + 1
    assert e.last_kernel_ms() > 0
    got = buf[:, :, :256 * 8].cpu().numpy()
    assert got.tobytes() == want.tobytes()
    assert not buf[:, :, 256 * 8:].any()


def test_errors_are_codes_not_crashes():
    e = ohs.Engine(2, 256, 256)
    with pytest.raises(ohs.OhsError):
        e.process(np.zeros((2, 2, 100), np.float32))      # not whole blocks -> use process_fifo
    with pytest.raises(ohs.OhsError):
        e.set_ir(0, np.zeros(300, np.float32))            # longer than max_taps capacity
    with pytest.raises(ohs.OhsError):
        e.set_ir(4, [1.0])
    with pytest.raises(ohs.OhsError):
        e.eq_update_band(0, ohs.PEAK, 30000.0, 1.0, 0.0)   # the reference would panic (parametric_eq.rs:111)
    e.eq_update_band(99, ohs.PEAK, 1000.0, 1.0, 0.0)       # out-of-range band silently ignored (:145)


def test_full_size_config2_properties():
    """BASELINE config 2 at full width (1024 streams): batch position must not matter — sampled streams equal the same
    stream rendered alone, bit for bit — and those sampled streams meet the oracle tolerance."""
    c = S.CONFIGS[2]
    h = S.synthetic_hrir_set(c["taps"], c["decay"])
    n = 256 * 40
    x = S.stream_inputs(1024, n, unique=64)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    e = ohs.Engine(1024, 256, 256)
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
    y = e.process(x)
    assert np.isfinite(y).all()
    # tiled inputs -> tiled outputs
    assert y[:64].tobytes() == y[64:128].tobytes() == y[960:1024].tobytes()
    for s in (0, 1, 2, 63):
        solo = ohs.Engine(1, 256, 256)
        solo.set_hrir_set(h); solo.eq_set_preset(S.EQ_PRESET_TYPICAL); solo.set_eq_enable(True); solo.set_gain(0.5)
        assert solo.process(x[s:s + 1]).tobytes() == y[s:s + 1].tobytes()
    ref = oracle_render(x[:8], 256, h, coeffs, [1] * 10, 0.5)
    assert np.max(np.abs(y[:8] - ref)) <= TOL
    # linearity of the convolution stage (EQ off): render(a) + render(b) == render(a + b) within round-off
    lin = ohs.Engine(1024, 256, 256, n_bands=0); lin.set_hrir_set(h)
    ya = lin.process(x); lin.conv_reset()
    yb = lin.process(x[::-1].copy()); lin.conv_reset()
    yab = lin.process(x + x[::-1])
    assert np.max(np.abs(ya + yb - yab)) <= TOL


def test_cpp_mirror_replays_reference_unit_tests():
    """open-headstage_b200/host/dsp.hpp: the C++ host mirror (reference type and method names over the C ABI) runs the
    reference's five unit tests (ref_unit_tests.cpp) on the GPU."""
    import subprocess

    binary = ohs.build_host_tests()
    r = subprocess.run([binary], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "PASSED" in r.stdout and "FAIL" not in r.stdout


def test_config4_object_mixdown(cipic):
    """BASELINE config 4 in miniature (one rank): 24 mono sources, each with its own direction from the bundled CIPIC set
    (idx = source*37 mod 1250), mixed to one stereo bus, EQ + gain applied once on the bus.  Config 4 has no reference
    behaviour (the reference has no multi-source mode); the definition is checked against an f64 evaluation."""
    import torch
    from open_headstage_b200 import parallel as P

    n_src, block, n = 24, 256, 256 * 12
    ir = cipic["ir"]
    hr = np.stack([ir[(s * 37) % 1250] for s in range(n_src)]).astype(np.float32)  # [n_src, 2, 200]
    src = np.stack([S.pink_noise(n, 4000 + s) for s in range(n_src)]) / np.float32(64.0)
    bus = P.render_object_mix(ohs, src, hr, block, FS, eq_preset=None, gain=0.5).cpu().numpy()
    truth = np.zeros((2, n))
    for s in range(n_src):
        for ear in range(2):
            truth[ear] += sps.fftconvolve(src[s].astype(np.float64), hr[s, ear].astype(np.float64))[:n]
    truth *= 0.5
    assert np.max(np.abs(bus - truth)) <= TOL
    assert np.abs(bus).max() > 1e-3
    # with the bus EQ: compare against the oracle's EQ run on the un-equalised GPU bus (EQ stage is bit-exact)
    raw = P.render_object_mix(ohs, src, hr, block, FS, eq_preset=None, gain=1.0).cpu().numpy()
    eqd = P.render_object_mix(ohs, src, hr, block, FS, eq_preset=S.EQ_PRESET_TYPICAL, gain=1.0).cpu().numpy()
    q = O.StereoParametricEQ(10, FS)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    for b in range(10):
        q.set_band_raw(b, coeffs[b], True)
    l, r = q.process_block(raw[0], raw[1])
    assert eqd[0].tobytes() == l.tobytes() and eqd[1].tobytes() == r.tobytes()


@pytest.mark.parametrize("block,taps,n_streams,g", [(512, 1500, 5, 2), (1024, 5000, 5, 2), (512, 2100, 7, 3), (1024, 9000, 3, 2)])
def test_long_shared_ir_tma_filter_tiles(block, taps, n_streams, g, monkeypatch):
    """The long-impulse-response path (N >= 1024, one shared HRIR set, >= 2 streams per CTA): filter tiles arrive by TMA
    bulk copy into the idle FFT buffers, delay-line operands are register-pipelined.  Odd stream counts leave an absent
    stream in the last CTA.  Launches of several blocks and block-at-a-time launches must agree with the oracle."""
    monkeypatch.setenv("OHS_STREAMS_PER_CTA", str(g))
    h = S.synthetic_hrir_set(taps, taps / 5.0, seed=21)
    n = block * 9
    x = S.stream_inputs(n_streams, n, base_seed=900)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    e = ohs.Engine(n_streams, block, taps)
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
    y = np.concatenate([e.process(x[:, :, :block * 4]), e.process(x[:, :, block * 4:block * 5]), e.process(x[:, :, block * 5:])], axis=2)
    ref = oracle_render(x, block, h, coeffs, [1] * 10, 0.5)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err


def test_repeated_runs_are_bit_identical():
    """Race evidence without a sanitizer (closed on this pool): the warp-specialised kernel (named barriers, mbarriers,
    TMA staging, shuffles) must be deterministic — twenty renders of the same input from the same state are bit-identical."""
    h = S.synthetic_hrir_set(700, 100.0, seed=5)
    x = S.stream_inputs(23, 256 * 10, base_seed=950)
    outs = []
    for _ in range(20):
        e = ohs.Engine(23, 256, 700)
        e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
        outs.append(e.process(x).tobytes())
    assert len(set(outs)) == 1


# ------------------------------------------------------------------------------------------------------------
# launch lengths around the three-buffer input staging (1..7 blocks), every EQ path: the continuous systolic chain,
# the per-block chain (a disabled band), EQ only with a ragged tail, EQ off
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_blocks", [1, 2, 3, 4, 5, 7])
@pytest.mark.parametrize("mode", ["chain", "chain_disabled_band", "eq_only_ragged", "conv_only"])
def test_short_launches_every_path(n_blocks, mode):
    block, taps, n_streams = 256, 300, 9   # 9 streams -> one stream per CTA (G = ceil(9 / #SM) = 1), nine full CTAs; partial
    # last CTAs and G = 2..7 are covered by test_every_streams_per_cta_variant below
    n = block * n_blocks - (57 if mode == "eq_only_ragged" else 0)
    x = S.stream_inputs(n_streams, n, base_seed=900 + n_blocks)
    h = S.synthetic_hrir_set(taps, 50.0, seed=5)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    enabled = [1] * 10
    e = ohs.Engine(n_streams, block, taps)
    e.set_hrir_set(h)
    if mode == "chain_disabled_band":
        enabled[3] = 0
    for b in range(10):
        e.eq_set_band(b, coeffs[b], bool(enabled[b]))
    if mode == "eq_only_ragged":
        e.set_conv_enable(False); e.set_eq_enable(True)
        y = e.process(x)
        for s in range(n_streams):
            q = O.StereoParametricEQ(10, FS)
            for b in range(10):
                q.set_band_raw(b, coeffs[b], True)
            l, r = q.process_block(x[s, 0], x[s, 1])
            assert y[s, 0].tobytes() == l.tobytes() and y[s, 1].tobytes() == r.tobytes()
        return
    if mode == "conv_only":
        e.set_eq_enable(False)
        ref = oracle_render(x, block, h)
    else:
        e.set_eq_enable(True)
        ref = oracle_render(x, block, h, coeffs, enabled)
    # two calls: the second starts from the first one's state
    half = (n_blocks // 2) * block
    y = np.concatenate([e.process(x[:, :, :half]), e.process(x[:, :, half:])], axis=2) if half else e.process(x)
    err = float(np.max(np.abs(y - ref)))
    assert err <= TOL, err


# ------------------------------------------------------------------------------------------------------------
# long responses over many blocks: the time-batched path (per-bin convolution along time) against the oracle, against
# the block-by-block kernel, and interleaved with it (the delay-line ring must end up identical)
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("block,taps,n_streams,n_blocks", [(512, 5000, 3, 24), (1024, 9000, 2, 19), (128, 1500, 5, 40), (128, 1100, 3, 150),
                                                           (256, 2100, 9, 11), (64, 600, 2, 17)])
def test_time_batched_long_response(block, taps, n_streams, n_blocks, monkeypatch):
    h = S.synthetic_hrir_set(taps, taps / 5.0, seed=21)
    n = block * n_blocks
    x = S.stream_inputs(n_streams, n, base_seed=1200)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    ref = oracle_render(x, block, h, coeffs, [1] * 10, 0.7)

    def engine():
        e = ohs.Engine(n_streams, block, taps)
        e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.7)
        return e

    monkeypatch.setenv("OHS_TIME_BATCH", "1")
    y_batched = engine().process(x)
    assert float(np.max(np.abs(y_batched - ref))) <= TOL
    monkeypatch.setenv("OHS_TIME_BATCH", "0")
    y_blocks = engine().process(x)
    assert float(np.max(np.abs(y_blocks - ref))) <= TOL
    assert float(np.max(np.abs(y_blocks - y_batched))) <= 2e-6
    # batched call, then block-by-block calls, then a batched call again on the same engine
    e = engine()
    cut1, cut2 = 16 * block, 16 * block + 2 * block
    e.set_time_batch(True)
    parts = [e.process(x[:, :, :cut1])]
    e.set_time_batch(False)
    parts.append(e.process(x[:, :, cut1:cut2]))
    e.set_time_batch(True)
    if cut2 < n:
        parts.append(e.process(x[:, :, cut2:]))
    y_mixed = np.concatenate(parts, axis=2)
    assert float(np.max(np.abs(y_mixed - ref))) <= TOL


@pytest.mark.parametrize("case", ["in_place", "eq_off", "disabled_band", "ragged_prepass", "own_sm"])
def test_time_batched_pipeline_variants(case):
    """The time-batched route's EQ pre-pass pipeline through ohs_process_device: several sub-launches and chunks per call
    (calls of 16 and 134 blocks, the second in sub-launches of 16+16+32, 64 and 6 blocks), in place; the EQ off (the
    transforms read a copy of the input rows); a disabled band (the pre-pass leaves its continuous chain); block 64 with
    a chunk that is not a whole number of the pre-pass's 256-frame rows; 14 streams, which select the pre-pass's
    production shape (render_kernel<512,6,2>: six streams per CTA on an SM of its own, here two full CTAs and a partial
    one).  Each against the oracle, and two fresh engines fed the same calls bit-identical: the pre-pass runs on a stream
    of its own, and a missing wait between it and the engine's stream would let the transforms read rows it has not
    written yet."""
    import torch

    block, taps, n_streams, n_blocks = {"in_place": (128, 1500, 5, 150), "eq_off": (128, 1100, 4, 70), "disabled_band": (256, 2100, 4, 30),
                                        "ragged_prepass": (64, 600, 3, 27), "own_sm": (128, 1100, 14, 80)}[case]
    h = S.synthetic_hrir_set(taps, taps / 5.0, seed=23)
    n = block * n_blocks
    x = S.stream_inputs(n_streams, n, base_seed=1250)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    enabled = [1] * 10
    if case == "disabled_band":
        enabled[4] = 0
    ref = oracle_render(x, block, h, None if case == "eq_off" else coeffs, None if case == "eq_off" else enabled, 0.7)
    outs = []
    for _ in range(2):
        e = ohs.Engine(n_streams, block, taps)
        e.set_hrir_set(h); e.set_gain(0.7)
        if case != "eq_off":
            for b in range(10):
                e.eq_set_band(b, coeffs[b], bool(enabled[b]))
            e.set_eq_enable(True)
        buf = torch.from_numpy(x).cuda()
        dst = buf if case == "in_place" else torch.empty_like(buf)
        # two calls: the second starts from the first one's state (ring head, overlap-save block, EQ state)
        cut = 16 * block
        e.process_device(buf.data_ptr(), dst.data_ptr(), cut, row_stride=n)
        e.process_device(buf.data_ptr() + 4 * cut, dst.data_ptr() + 4 * cut, n - cut, row_stride=n)
        e.sync()
        outs.append(dst.cpu().numpy())
    assert float(np.max(np.abs(outs[0] - ref))) <= TOL, case
    assert np.array_equal(outs[0], outs[1])


def test_time_batched_history_stays_in_the_circular_buffer():
    """Consecutive time-batched calls keep their convolution history in the circular time-ordered buffer (no copy
    between calls; the buffer wraps several times here); the delay-line ring is rebuilt from it only when something needs
    it: a state export, a block-by-block call.  Five time-batched calls, export, import into a fresh engine, four blocks
    block by block there, and two more on the first engine: all against the oracle."""
    block, taps, n_streams = 128, 1100, 4
    calls = [24, 16, 40, 8, 24]
    n_blocks = sum(calls) + 4
    h = S.synthetic_hrir_set(taps, taps / 5.0, seed=27)
    x = S.stream_inputs(n_streams, block * n_blocks, base_seed=1270)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    ref = oracle_render(x, block, h, coeffs, [1] * 10, 0.7)

    def engine():
        e = ohs.Engine(n_streams, block, taps)
        e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.7)
        return e

    e = engine()
    e.prepare(40 * block)            # scratch for the largest call: 8 history slots + 40 = 48 slots, 112 blocks go through
    parts, at = [], 0
    for k in calls:
        parts.append(e.process(x[:, :, at * block:(at + k) * block])); at += k
    blob = e.state_export()
    f = engine()
    f.state_import(blob)
    tail_f = f.process(x[:, :, at * block:])                       # 4 blocks: block by block on the importing engine
    tail_e = np.concatenate([e.process(x[:, :, at * block:(at + 2) * block]), e.process(x[:, :, (at + 2) * block:])], axis=2)
    y = np.concatenate(parts + [tail_e], axis=2)
    assert float(np.max(np.abs(y - ref))) <= TOL
    assert np.array_equal(tail_f, tail_e)


def test_time_batched_mixed_hrir_sets(monkeypatch):
    """Two HRIR sets on one engine, a long one (10 partitions) and a single-partition one, streams bound alternately:
    the time-batched route renders both kinds (a single-partition stream has no delay line of its own)."""
    block, n_streams, n_blocks = 512, 5, 20
    h_long = S.synthetic_hrir_set(5000, 900.0, seed=31)
    h_short = S.synthetic_hrir_set(300, 60.0, seed=32)
    x = S.stream_inputs(n_streams, block * n_blocks, base_seed=1300)
    refs = {0: oracle_render(x, block, h_long), 1: oracle_render(x, block, h_short)}
    for mode in ("1", "0"):
        monkeypatch.setenv("OHS_TIME_BATCH", mode)
        e = ohs.Engine(n_streams, block, 5000, n_bands=0, n_hrir_sets=2)
        e.set_hrir_set(h_long, hrir_set=0); e.set_hrir_set(h_short, hrir_set=1)
        for s in range(n_streams):
            e.bind_stream_hrir(s, s % 2)
        y = e.process(x)
        for s in range(n_streams):
            err = float(np.max(np.abs(y[s] - refs[s % 2][s])))
            assert err <= TOL, (mode, s, err)


# ------------------------------------------------------------------------------------------------------------
# every render-kernel instantiation production can select: render_kernel<2*block, G>, G = 1..7 streams per CTA
# (G = ceil(n_streams / #SM) up to 7, else 3 — csrc/ohs_api.cu pick_streams_per_cta), each with a partial last CTA,
# a single-partition and a multi-partition response, the whole chain, two calls (state carried), K = 1 launches
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("g", [1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("block", [64, 128, 256, 512, 1024])
def test_every_streams_per_cta_variant(block, g, monkeypatch):
    monkeypatch.setenv("OHS_STREAMS_PER_CTA", str(g))
    n_streams = 2 * g + 1 if g > 1 else 3          # g > 1: two full CTAs and a last CTA holding ONE stream
    n_blocks = 6
    x = S.stream_inputs(n_streams, block * n_blocks, base_seed=1500 + g)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    for taps in (block, 2 * block + block // 2):    # P = 1 (fused single-partition path at N = 512) and P = 3
        h = S.synthetic_hrir_set(taps, taps / 5.0, seed=41)
        e = ohs.Engine(n_streams, block, taps)
        if e.streams_per_cta() != g:
            assert g > 1   # G = 1 always fits
            pytest.skip("render_kernel<%d,%d> does not fit in shared memory; production never selects it" % (2 * block, g))
        e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
        ref = oracle_render(x, block, h, coeffs, [1] * 10, 0.5)
        y = np.concatenate([e.process(x[:, :, :4 * block]), e.process(x[:, :, 4 * block:5 * block]), e.process(x[:, :, 5 * block:])], axis=2)
        err = float(np.max(np.abs(y - ref)))
        assert err <= TOL, (taps, err)
        # EQ stage alone through the same instantiation: bit-exact
        q = ohs.Engine(n_streams, block, 1)
        assert q.streams_per_cta() == g
        q.set_conv_enable(False); q.set_eq_enable(True)
        for b in range(10):
            q.eq_set_band(b, coeffs[b], True)
        yq = q.process(x)
        s = n_streams - 1                            # the lone stream of the partial CTA
        o = O.StereoParametricEQ(10, FS)
        for b in range(10):
            o.set_band_raw(b, coeffs[b], True)
        l, r = o.process_block(x[s, 0], x[s, 1])
        assert yq[s, 0].tobytes() == l.tobytes() and yq[s, 1].tobytes() == r.tobytes()


@pytest.mark.parametrize("cfg,n_streams,expect_g,n_blocks", [(3, 1210, 3, 24), (2, 1024, 7, 16), (2, 600, 5, 16), (3, 300, 3, 24)])
def test_production_instantiations_at_width(cfg, n_streams, expect_g, n_blocks):
    """The instantiation the host picks BY ITSELF at production widths: config 3 (block 128, 512 taps, P = 4) beyond
    7 streams per SM -> render_kernel<256,3>, dense role packing, several CTAs per SM, partial last CTA (1210 = 403*3+1);
    config 2 (1024 streams -> <512,7>, 600 -> <512,5>).  Sampled streams against the oracle, every stream against its
    tiled twin."""
    c = S.CONFIGS[cfg]
    block, taps = c["block"], c["taps"]
    h = S.synthetic_hrir_set(taps, c["decay"])
    n = block * n_blocks
    unique = 10
    x = S.stream_inputs(n_streams, n, unique=unique)
    coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL)
    e = ohs.Engine(n_streams, block, taps)
    assert e.streams_per_cta() == expect_g, e.streams_per_cta()
    e.set_hrir_set(h); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
    y = np.concatenate([e.process(x[:, :, :n // 2]), e.process(x[:, :, n // 2:])], axis=2)
    ref = oracle_render(x[:unique], block, h, coeffs, [1] * 10, 0.5)
    assert float(np.max(np.abs(y[:unique] - ref))) <= TOL
    # tiled inputs -> tiled outputs, bit for bit, wherever the stream sits (CTA, slot in the CTA, SM)
    for s in range(unique, n_streams):
        assert y[s].tobytes() == y[s % unique].tobytes(), s


# ------------------------------------------------------------------------------------------------------------
# small rows: magnitude response helper, SOFA wiring and AutoEQ ingestion driven into the real engine, the
# multi-partition table hand-over of the broadcast path, state-blob validation
# ------------------------------------------------------------------------------------------------------------
def test_eq_frequency_response_product_function():
    """ohs_eq_frequency_response (src/dsp/parametric_eq.rs:191-209) against the oracle's restatement and against an
    independent f64 evaluation (scipy freqz) of the same coefficients; disabled bands are skipped; sample_rate honoured."""
    freqs = np.geomspace(20.0, 20000.0, 64).astype(np.float32)
    for fs in (48000.0, 44100.0):
        e = ohs.Engine(1, 256, 1, sample_rate=fs)
        o = O.StereoParametricEQ(10, fs)
        coeffs = preset_coeffs(S.EQ_PRESET_TYPICAL, fs)
        for b in range(10):
            e.eq_set_band(b, coeffs[b], b != 6)
            o.set_band_raw(b, coeffs[b], b != 6)
        got = e.eq_frequency_response(freqs, sample_rate=fs)
        want = o.calculate_frequency_response(fs, freqs)
        assert np.max(np.abs(got / want - 1.0)) <= 1e-6
        truth = np.ones(freqs.size)
        for b in range(10):
            if b == 6:
                continue
            c = coeffs[b].astype(np.float64)
            _, hh = sps.freqz([c[0], c[1], c[2]], [1.0, c[3], c[4]], worN=freqs.astype(np.float64), fs=fs)
            truth *= np.abs(hh)
        assert np.max(np.abs(got / truth - 1.0)) <= 2e-3   # f32 evaluation, as in the reference (cancellation at low f)
        # the mirror object passes its sample_rate argument through (reference signature)
        m = ohs.StereoParametricEQ(10, 48000.0)
        for b in range(10):
            m.update_band_coeffs(b, fs, ohs.BandConfig(*S.EQ_PRESET_TYPICAL[b], b != 6))
        assert np.max(np.abs(m.calculate_frequency_response(fs, freqs) / want - 1.0)) <= 1e-6
    assert e.eq_frequency_response(freqs, sample_rate=0.0).tobytes() == e.eq_frequency_response(freqs, sample_rate=44100.0).tobytes()


def test_sofa_wiring_and_autoeq_into_the_real_engine(cipic):
    """SURVEY 8f rows 1 and 4 end to end: SOFA directions -> four set_ir calls, AutoEQ CSV -> update_band_coeffs, on the
    GPU engine, against the oracle given the same indices and the same parsed bands."""
    from open_headstage_b200 import autoeq, sofa

    hr = sofa.from_arrays(cipic["ir"], cipic["pos"], float(cipic["fs"]))
    e = ohs.Engine(2, 512, 200, sample_rate=FS)
    il, ir_ = sofa.wire_speakers(e, hr, sofa.ui_azimuth_to_sofa(-30.0), 0.0, sofa.ui_azimuth_to_sofa(30.0), 0.0)
    assert (il, ir_) == (308, 908)
    csv_text = "Filter-Type,Fc,Q,Gain\n" + "\n".join(
        "%s,%g,%g,%g" % ({S.LOWSHELF: "LS", S.PEAK: "PK", S.HIGHSHELF: "HS"}[t], fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL) + "\n"
    bands = autoeq.parse_autoeq_csv(csv_text)
    assert len(bands) == 10
    autoeq.apply_to_engine(e, bands)
    e.set_eq_enable(True); e.set_gain(0.5)
    x = S.stream_inputs(2, 512 * 12, base_seed=1700)
    y = e.process(x)
    ir = cipic["ir"]
    irs = [ir[308, 0], ir[308, 1], ir[908, 0], ir[908, 1]]
    coeffs = np.stack([O.eq_design(b.filter_type, FS, b.frequency, b.q, b.gain) for b in bands])
    ref = oracle_render(x, 512, irs, coeffs, [1] * 10, 0.5)
    assert float(np.max(np.abs(y - ref))) <= TOL
    assert np.abs(y).max() > 0.05


def test_filter_table_handover_multi_partition():
    """What a broadcast receiver does (parallel.broadcast_filters): engine B never sees the impulse responses, it gets
    engine A's device-resident spectra table plus A's per-set partition counts — for a response LONGER than one block
    (ADVICE r1: the count used to be lost)."""
    import torch
    from open_headstage_b200 import parallel as P

    block, taps = 256, 900   # 4 partitions
    h = S.synthetic_hrir_set(taps, 150.0, seed=3)
    x = S.stream_inputs(3, block * 8, base_seed=1800)
    a = ohs.Engine(3, block, taps, n_bands=0); a.set_hrir_set(h); a.commit_filters(); a.sync()
    b = ohs.Engine(3, block, taps, n_bands=0)
    counts = P.set_partition_counts(a, [0])
    assert counts == [4]
    pa, na = a.filter_table(); pb, nb = b.filter_table()
    assert na == nb
    ta = torch.as_tensor(P.DeviceMemory(pa, na), device="cuda:0"); tb = torch.as_tensor(P.DeviceMemory(pb, nb), device="cuda:0")
    assert ta.data_ptr() == pa and tb.data_ptr() == pb
    tb.copy_(ta); torch.cuda.synchronize()
    P.apply_received_partition_counts(b, [0], counts, is_src=False)
    assert b.num_partitions(0) == 4
    assert b.process(x).tobytes() == a.process(x).tobytes()
    with pytest.raises(RuntimeError):
        P.apply_received_partition_counts(b, [0], [0], is_src=False)
    # world size 1: the public call is a no-op broadcast that still validates the counts
    P.broadcast_filters(a)


def test_state_blob_validation_and_fifo_residue():
    import struct

    h = S.synthetic_hrir_set(600, 100.0, seed=4)
    x = S.stream_inputs(2, 1000, base_seed=1900)

    def make(n_streams=2, taps=600):
        e = ohs.Engine(n_streams, 256, taps)
        e.set_hrir_set(h[:, :taps]); e.eq_set_preset(S.EQ_PRESET_TYPICAL); e.set_eq_enable(True); e.set_gain(0.5)
        return e

    # FIFO residue travels with the blob: ragged host blocks, export in the middle, resume on a fresh engine
    a = make()
    whole = np.concatenate([a.process_fifo(x[:, :, i:i + 100]) for i in range(0, 1000, 100)], axis=2)
    b = make()
    first = np.concatenate([b.process_fifo(x[:, :, i:i + 100]) for i in range(0, 400, 100)], axis=2)
    blob = b.state_export()
    c = make()
    c.state_import(blob)
    second = np.concatenate([c.process_fifo(x[:, :, i:i + 100]) for i in range(400, 1000, 100)], axis=2)
    assert np.concatenate([first, second], axis=2).tobytes() == whole.tobytes()
    # a corrupt ring head, a truncated blob, a padded blob and a blob from another geometry are all rejected
    magic, abi, n_streams, n_bands, pmax, block, head, _ = struct.unpack_from("<I7i", blob, 0)
    assert (n_streams, pmax, block) == (2, 3, 256) and 0 <= head < pmax
    for bad_head in (-1, pmax, 1 << 20):
        bad = bytearray(blob); struct.pack_into("<i", bad, 24, bad_head)
        with pytest.raises(ohs.OhsError):
            c.state_import(bytes(bad))
    with pytest.raises(ohs.OhsError):
        c.state_import(blob[:-4])
    with pytest.raises(ohs.OhsError):
        c.state_import(blob + b"\0\0\0\0")
    with pytest.raises(ohs.OhsError):
        make(n_streams=3).state_import(blob)
    with pytest.raises(ohs.OhsError):
        make(taps=256).state_import(blob)
    with pytest.raises(ohs.OhsError):
        c.state_import(b"\0" * len(blob))
    with pytest.raises(ValueError):
        c.process(np.zeros((2, 2, 256), np.float32), out=np.zeros((2, 2, 256), np.float64))


def test_c_abi_collectives_single_rank():
    """ohs_comm_* / ohs_broadcast_hrir / ohs_reduce_bus on a one-rank NCCL communicator: the calls a multi-GPU host makes,
    exercised on the single GPU the test box has (the N = 2..8 runs of bench.py use the same entry points)."""
    import torch
    from open_headstage_b200 import parallel as P

    comm = P.create_comm(ohs, 0)
    assert (comm.world, comm.rank) == (1, 0)
    h = S.synthetic_hrir_set(700, 100.0, seed=5)
    x = S.stream_inputs(3, 256 * 6, base_seed=2100)
    a = ohs.Engine(3, 256, 700, n_bands=0); a.set_hrir_set(h)
    want = a.process(x)
    b = ohs.Engine(3, 256, 700, n_bands=0); b.set_hrir_set(h)
    P.broadcast_filters(b, src=0, comm=comm)            # root: commit + broadcast to itself
    assert b.process(x).tobytes() == want.tobytes()
    bus = torch.arange(2 * 1024, dtype=torch.float32, device="cuda").reshape(2, 1024).contiguous()
    keep = bus.clone()
    b.reduce_bus(comm, bus.data_ptr(), bus.numel(), 0); b.sync()
    assert torch.equal(bus, keep)                        # sum over one rank
    with pytest.raises(ohs.OhsError):
        b.broadcast_hrir(comm, 3)                        # root outside the communicator
    comm.close()
