"""Moving sources (include/ohs.h, DESIGN §10): a stream changes HRIR sets without losing its history, crossfaded over
one engine block.  The definition is a blend of two static renders, so everything that checks static renders checks
it: twin streams in the same engine (bit-exact), the oracle (<= 1e-5) and an f64 evaluation (CPU tests below)."""
import ctypes as C

import numpy as np
import pytest
import scipy.signal as sps

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S
from oracle import oracle as O

gpu = pytest.mark.gpu
TOL = 1e-5
FS = 48000.0


# ---- the definition ---------------------------------------------------------------------------------------------
def crossfade(a, b, block):
    """out[n] = a[n] + w[n]*(b[n] - a[n]), w[n] = (2n+1)/(2B), each f32 operation rounded on its own."""
    w = ((2 * np.arange(block) + 1) / (2.0 * block)).astype(np.float32)
    a = a.astype(np.float32)
    return a + w * (b.astype(np.float32) - a)


def assemble(static, sets, bound, block):
    """static[set] = y of one stream [2, n] bound to that set from the start; sets[t] = set of block t; bound = the
    binding before block 0.  Returns the moving stream's output by the definition (f32 blend)."""
    out = np.empty_like(static[sets[0]])
    prev = bound
    for t, cur in enumerate(sets):
        sl = slice(t * block, (t + 1) * block)
        out[:, sl] = static[cur][:, sl] if cur == prev else crossfade(static[prev][:, sl], static[cur][:, sl], block)
        prev = cur
    return out


def oracle_moving(x, block, set_irs, sets, bound, coeffs=None, gain=1.0):
    """One stream x[2, n] through the oracle, one static render per set involved, blended per block."""
    eq = coeffs is not None
    c = coeffs if eq else np.zeros((1, 5), np.float32)
    used = set(int(v) for v in sets) | {int(bound)}
    static = {k: O.render_batch(x[None], block, set_irs[k], c, [1] * len(c), eq, gain)[0][0] for k in used}
    return assemble(static, [int(v) for v in sets], int(bound), block)


def f64_moving(x, block, set_irs, sets, bound, gain):
    """f64 truth (no EQ): the whole input convolved with each set (out_l = x_l*LSL + x_r*RSL, out_r = x_l*LSR +
    x_r*RSR), times gain, blended per block in f64."""
    n = x.shape[1]
    xd = x.astype(np.float64)
    static = {}
    for k in set(int(v) for v in sets) | {int(bound)}:
        h = [np.asarray(i, np.float64) for i in set_irs[k]]
        yl = sps.fftconvolve(xd[0], h[0])[:n] + sps.fftconvolve(xd[1], h[2])[:n]
        yr = sps.fftconvolve(xd[0], h[1])[:n] + sps.fftconvolve(xd[1], h[3])[:n]
        static[k] = np.stack([yl, yr]) * gain
    w = (2 * np.arange(block) + 1) / (2.0 * block)
    out = np.empty((2, n))
    prev = int(bound)
    for t, cur in enumerate(int(v) for v in sets):
        sl = slice(t * block, (t + 1) * block)
        a, b = static[prev][:, sl], static[cur][:, sl]
        out[:, sl] = b if cur == prev else a + w * (b - a)
        prev = cur
    return out


def two_sets(block, seed=3):
    """set 0: one partition (block - 7 taps); set 1: three partitions (2*block + 5 taps)."""
    return [S.synthetic_hrir_set(block - 7, block / 6.0, seed=seed), S.synthetic_hrir_set(2 * block + 5, block / 2.0, seed=seed + 1)]


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_symbols_declared_and_bound():
    lib = ohs.load_library()
    bound = {s[0] for s in ohs.SYMBOLS}
    for name in ("ohs_move_stream_hrir", "ohs_process_device_scheduled"):
        assert name in bound and hasattr(lib, name)


def test_null_handle_and_bad_arguments_without_a_device():
    lib = ohs.load_library()
    sets = (C.c_int32 * 4)()
    assert lib.ohs_move_stream_hrir(None, 0, 0) == -1
    assert lib.ohs_move_stream_hrir(None, ohs.OHS_ALL, 1) == -1
    assert lib.ohs_process_device_scheduled(None, None, None, 256, 256, C.cast(sets, C.c_void_p), 1) == -1
    assert lib.ohs_process_device_scheduled(None, None, None, 0, 0, None, 0) == -1


@pytest.mark.parametrize("case", ["one_to_three", "three_to_one", "random"])
def test_reference_blend_matches_f64(case):
    block, k = 64, 14
    set_irs = two_sets(block)
    x = S.stream_inputs(1, block * k, base_seed=77)[0]
    if case == "one_to_three":
        sets, bound = [0] * 5 + [1] * 9, 0
    elif case == "three_to_one":
        sets, bound = [1] * 6 + [0] * 8, 1
    else:
        sets, bound = list(np.random.default_rng(5).integers(0, 2, k)), 1
    y = oracle_moving(x, block, set_irs, sets, bound, gain=0.7)
    truth = f64_moving(x, block, set_irs, sets, bound, 0.7)
    assert np.max(np.abs(y - truth)) <= TOL


# ---- GPU helpers ------------------------------------------------------------------------------------------------
def torch_dev():
    import torch

    return torch


def make_engine(n_streams, block, set_irs, max_taps=None, coeffs=None, gain=1.0, time_batch=True):
    e = ohs.Engine(n_streams, block, max_taps or max(len(s[0]) for s in set_irs), n_hrir_sets=len(set_irs))
    for k, irs in enumerate(set_irs):
        e.set_hrir_set(irs, hrir_set=k)
    if coeffs is not None:
        for b in range(len(coeffs)):
            e.eq_set_band(b, coeffs[b], True)
        e.set_eq_enable(True)
    e.set_gain(gain)
    e.set_time_batch(time_batch)
    return e


def run(e, x, sched=None, in_place=False):
    """One device call on x[stream, 2, n]; returns the output as numpy."""
    torch = torch_dev()
    d_in = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    d_out = d_in if in_place else torch.empty_like(d_in)
    torch.cuda.synchronize()
    e.process_device(d_in.data_ptr(), d_out.data_ptr(), x.shape[2], hrir_schedule=sched)
    e.sync()
    return d_out.cpu().numpy()


def twin_layout(n_streams, n_sets, x_groups):
    """Streams in groups of 1 + n_sets: the moving stream, then one twin bound to each set; a group shares its input
    rows.  Streams past the last whole group are bound to set 0 and fed group 0's input."""
    g = 1 + n_sets
    n_groups = n_streams // g
    idx = np.minimum(np.arange(n_streams) // g, n_groups - 1)
    idx[n_groups * g:] = 0
    return n_groups, x_groups[idx]


def twin_schedule(n_streams, n_sets, moving_sets):
    """[n_streams, K]: the moving stream of group i follows moving_sets[i], twin j stays on set j, the rest on 0."""
    g = 1 + n_sets
    k = moving_sets.shape[1]
    sched = np.zeros((n_streams, k), np.int32)
    for i in range(moving_sets.shape[0]):
        sched[g * i] = moving_sets[i]
        for j in range(n_sets):
            sched[g * i + 1 + j] = j
    return sched


def bind_twins(e, n_streams, n_sets):
    g = 1 + n_sets
    for i in range(n_streams // g):
        for j in range(1, n_sets):
            e.bind_stream_hrir(g * i + 1 + j, j)


def check_twins(y, moving_sets, bound, n_sets, block):
    g = 1 + n_sets
    for i in range(moving_sets.shape[0]):
        static = {j: y[g * i + 1 + j] for j in range(n_sets)}
        want = assemble(static, list(moving_sets[i]), int(bound[i]), block)
        assert np.array_equal(y[g * i].view(np.uint32), want.view(np.uint32)), "group %d" % i


# ---- GPU: twins, oracle -----------------------------------------------------------------------------------------
# (block, streams, EQ, in place): stream counts that select one, three and seven streams per CTA, with partial last CTAs
TWIN_CASES = [(64, 7, True, False), (128, 302, False, True), (256, 1000, True, False), (512, 20, False, False),
              (512, 301, True, True), (1024, 9, True, False), (256, 5, False, True)]


@gpu
@pytest.mark.parametrize("block,n_streams,eq,in_place", TWIN_CASES)
def test_twins_bit_exact_and_oracle(block, n_streams, eq, in_place):
    rng = np.random.default_rng(block + n_streams)
    set_irs = two_sets(block)
    coeffs = np.stack([ohs.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL]) if eq else None
    k1, k2 = 6, 7
    n_groups = n_streams // 3
    xg = S.stream_inputs(max(n_groups, 1), block * (k1 + k2), base_seed=900 + block)
    n_groups, x = twin_layout(n_streams, 2, xg)
    e = make_engine(n_streams, block, set_irs, coeffs=coeffs, gain=0.625)
    bind_twins(e, n_streams, 2)
    # moving streams: first group 0 -> 1 at block 3 and back at 10 (crossing the call boundary), the others random
    mv = rng.integers(0, 2, (n_groups, k1 + k2)).astype(np.int32)
    mv[0] = [0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0]
    sched = twin_schedule(n_streams, 2, mv)
    bound = np.zeros(n_groups, np.int32)
    y1 = run(e, x[:, :, :k1 * block], sched[:, :k1], in_place)
    y2 = run(e, x[:, :, k1 * block:], sched[:, k1:], in_place)
    y = np.concatenate([y1, y2], axis=2)
    check_twins(y, mv, bound, 2, block)
    for i in sorted({0, n_groups - 1}):
        want = oracle_moving(x[3 * i], block, set_irs, mv[i], 0, coeffs, 0.625)
        assert np.max(np.abs(y[3 * i] - want)) <= TOL


@gpu
def test_config2_width_random_schedule():
    """1024 streams, B 256, two 256-tap sets, K = 192: streams without a transition are bit-identical to an
    unscheduled call, and a schedule without any transition changes nothing."""
    block, n, k = 256, 1024, 192
    set_irs = [S.synthetic_hrir_set(256, 40.0, seed=11), S.synthetic_hrir_set(256, 40.0, seed=12)]
    coeffs = np.stack([ohs.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    x = S.stream_inputs(n, block * k, unique=64)
    bound = (np.arange(n) % 2).astype(np.int32)
    rng = np.random.default_rng(2)
    sched = np.repeat(bound[:, None], k, axis=1)
    movers = rng.choice(n, n // 2, replace=False)
    for s in movers:
        t0 = int(rng.integers(1, k))
        sched[s, t0:] = 1 - bound[s]

    def engine():
        e = make_engine(n, block, set_irs, coeffs=coeffs, gain=0.5)
        for s in range(n):
            if bound[s]:
                e.bind_stream_hrir(s, 1)
        return e

    plain = run(engine(), x)
    e = engine()
    same = run(e, x, np.repeat(bound[:, None], k, axis=1))
    assert np.array_equal(same.view(np.uint32), plain.view(np.uint32))
    e = engine()
    y = run(e, x, sched)
    still = np.setdiff1d(np.arange(n), movers)
    assert np.array_equal(y[still].view(np.uint32), plain[still].view(np.uint32))
    for s in movers[:3]:
        want = oracle_moving(x[s], block, set_irs, sched[s], bound[s], coeffs, 0.5)
        assert np.max(np.abs(y[s] - want)) <= TOL


# ---- GPU: per-call moves ----------------------------------------------------------------------------------------
def per_call_engine(block, n_streams=3):
    set_irs = two_sets(block)
    return make_engine(n_streams, block, set_irs, gain=0.75), set_irs


@gpu
@pytest.mark.parametrize("k", [1, 2])
def test_per_call_moves_short_calls(k):
    """K = 1 and K = 2 calls (latency variant at B 256): moves before some calls; stream 0 moves, 1 and 2 are twins."""
    block, calls = 256, 10
    e, _ = per_call_engine(block)
    e.bind_stream_hrir(2, 1)
    xg = S.stream_inputs(1, block * k * calls, base_seed=31)
    x = np.repeat(xg, 3, axis=0)
    moves = {2: 1, 5: 0, 6: 1, 9: 0}   # call index -> target of stream 0
    cur, sets, ys = 0, [], []
    for c in range(calls):
        if c in moves:
            e.move_stream_hrir(0, moves[c])
            cur = moves[c]
        sets += [cur] * k
        ys.append(run(e, x[:, :, c * k * block:(c + 1) * k * block]))
    y = np.concatenate(ys, axis=2)
    want = assemble({0: y[1], 1: y[2]}, sets, 0, block)
    assert np.array_equal(y[0].view(np.uint32), want.view(np.uint32))


@gpu
def test_process_host_flavour_with_moves():
    block = 128
    e, _ = per_call_engine(block)
    e.bind_stream_hrir(2, 1)
    x = np.repeat(S.stream_inputs(1, block * 12, base_seed=32), 3, axis=0)
    y1 = e.process(x[:, :, :block * 5])
    e.move_stream_hrir(0, 1)
    y2 = e.process(x[:, :, block * 5:])
    y = np.concatenate([y1, y2], axis=2)
    want = assemble({0: y[1], 1: y[2]}, [0] * 5 + [1] * 7, 0, block)
    assert np.array_equal(y[0].view(np.uint32), want.view(np.uint32))


def fifo_positions(host, calls, block):
    """Which rendered frame each output frame of ohs_process_fifo carries (-1: the zero fill), and the engine blocks
    rendered before each call (the reference's FIFO, src/dsp/convolution.rs:141-182)."""
    pos, before = [], []
    queued_in = rendered = out_len = 0
    out_start = 0
    for _ in range(calls):
        before.append(rendered // block)
        queued_in += host
        whole = queued_in // block * block
        queued_in -= whole
        rendered += whole
        out_len += whole
        if out_len >= host:
            pos += list(range(out_start, out_start + host))
            out_start += host
            out_len -= host
        else:
            pos += [-1] * host
    return np.array(pos), before


@gpu
@pytest.mark.parametrize("host", [100, 700])
def test_process_fifo_crossfade_lands_on_the_first_block_rendered(host):
    block, calls = 256, 14
    e, _ = per_call_engine(block)
    e.bind_stream_hrir(2, 1)
    x = np.repeat(S.stream_inputs(1, host * calls, base_seed=33), 3, axis=0)
    pos, before = fifo_positions(host, calls, block)
    move_call = 4
    ys = []
    for c in range(calls):
        if c == move_call:
            e.move_stream_hrir(0, 1)
        ys.append(e.process_fifo(x[:, :, c * host:(c + 1) * host]))
    y = np.concatenate(ys, axis=2)
    t_move = before[move_call]
    valid = pos >= 0
    assert np.array_equal(y[:, :, ~valid], np.zeros_like(y[:, :, ~valid]))
    n_rendered = pos[valid].max() + 1 if valid.any() else 0
    n_blocks = n_rendered // block
    # rendered frames in order (the FIFO hands them back contiguously)
    r = np.zeros((3, 2, n_blocks * block), np.float32)
    keep = valid & (pos < n_blocks * block)
    r[:, :, pos[keep]] = y[:, :, keep]
    sets = [0 if t < t_move else 1 for t in range(n_blocks)]
    assert n_blocks > t_move
    want = assemble({0: r[1], 1: r[2]}, sets, 0, block)
    assert np.array_equal(r[0].view(np.uint32), want.view(np.uint32))


# ---- GPU: long responses ----------------------------------------------------------------------------------------
@gpu
def test_long_response_transition_leaves_the_time_batched_route_only_when_needed():
    block, k = 128, 16
    set_irs = [S.synthetic_hrir_set(8 * block - 3, 300.0, seed=21), S.synthetic_hrir_set(12 * block, 500.0, seed=22)]
    n = 12
    xg = S.stream_inputs(4, block * 3 * k, base_seed=41)
    _, x = twin_layout(n, 2, xg)
    sched = twin_schedule(n, 2, np.zeros((4, k), np.int32))

    def engine():
        e = make_engine(n, block, set_irs, max_taps=12 * block, gain=0.8)
        bind_twins(e, n, 2)
        return e

    # no transition: the time-batched route (more than one launch), bit-identical to a plain call
    a, b = engine(), engine()
    l0 = a.launch_count()
    ya = run(a, x[:, :, :k * block], sched)
    assert a.launch_count() - l0 > 1
    yb = run(b, x[:, :, :k * block])
    assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    # a transition call: the block-by-block kernel, twins bit-exact, oracle
    mv = np.array([[0] * 5 + [1] * 11, [1] * 16, [1] * 3 + [0] * 13, [0] * 8 + [1] * 8], np.int32)
    sched2 = twin_schedule(n, 2, mv)
    l_batched = a.launch_count() - l0
    l0 = a.launch_count()
    y2 = run(a, x[:, :, k * block:2 * k * block], sched2)
    assert a.launch_count() - l0 < l_batched   # the render kernel (after the delay line is brought up to date)
    check_twins(y2, mv, np.zeros(4, np.int32), 2, block)
    # and the same call on an engine that never takes the time-batched route: twins bit-exact there too
    c = engine()
    c.set_time_batch(False)
    run(c, x[:, :, :k * block], sched)
    yc = run(c, x[:, :, k * block:2 * k * block], sched2)
    check_twins(yc, mv, np.zeros(4, np.int32), 2, block)
    full = np.concatenate([ya, y2], axis=2)
    for i in range(4):
        want = oracle_moving(x[3 * i, :, :2 * k * block], block, set_irs, np.concatenate([np.zeros(k, np.int32), mv[i]]), 0, None, 0.8)
        assert np.max(np.abs(full[3 * i] - want)) <= TOL


# ---- GPU: semantics ---------------------------------------------------------------------------------------------
def sem_engine(block=128, n=4):
    set_irs = two_sets(block)
    return make_engine(n, block, set_irs, gain=0.9), set_irs


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@gpu
def test_move_to_bound_set_is_a_noop_and_bind_cancels():
    block = 128
    x = S.stream_inputs(4, block * 8, base_seed=51)
    a, _ = sem_engine(block)
    b, _ = sem_engine(block)
    run(a, x[:, :, :block * 4]); run(b, x[:, :, :block * 4])
    a.move_stream_hrir(1, 0)                  # already bound there
    a.move_stream_hrir(2, 1); a.move_stream_hrir(2, 0)   # and back before any call
    assert same_bits(run(a, x[:, :, block * 4:]), run(b, x[:, :, block * 4:]))
    c, _ = sem_engine(block)
    d, _ = sem_engine(block)
    run(c, x[:, :, :block * 4]); run(d, x[:, :, :block * 4])
    c.move_stream_hrir(3, 1); c.bind_stream_hrir(3, 1)   # the hard bind wins: history cleared, no crossfade
    d.bind_stream_hrir(3, 1)
    assert same_bits(run(c, x[:, :, block * 4:]), run(d, x[:, :, block * 4:]))


@gpu
def test_set_ir_on_the_spare_set_then_move_clears_nothing():
    block = 128
    x = S.stream_inputs(4, block * 8, base_seed=52)
    ref, set_irs = sem_engine(block)
    t = make_engine(4, block, [set_irs[0], S.synthetic_hrir_set(50, 10.0, seed=99)], max_taps=3 * block, gain=0.9)
    run(ref, x[:, :, :block * 4]); run(t, x[:, :, :block * 4])
    t.set_hrir_set(set_irs[1], hrir_set=1)   # the new direction goes into the spare set ...
    t.move_stream_hrir(ohs.OHS_ALL, 1)   # ... and every stream moves to it
    ref.move_stream_hrir(ohs.OHS_ALL, 1)
    assert same_bits(run(t, x[:, :, block * 4:]), run(ref, x[:, :, block * 4:]))


@gpu
def test_bypass_and_conv_off_keep_the_move_pending():
    block = 128
    x = S.stream_inputs(4, block * 6, base_seed=53)
    a, _ = sem_engine(block)
    b, _ = sem_engine(block)
    run(a, x[:, :, :block * 2]); run(b, x[:, :, :block * 2])
    a.move_stream_hrir(0, 1); b.move_stream_hrir(0, 1)
    a.set_bypass(True)
    assert same_bits(run(a, x[:, :, block * 2:block * 3]), x[:, :, block * 2:block * 3])
    a.set_bypass(False)
    a.set_conv_enable(False)
    run(a, x[:, :, block * 2:block * 3])     # EQ off: gain only, no state advances
    a.set_conv_enable(True)
    ya, yb = run(a, x[:, :, block * 3:]), run(b, x[:, :, block * 3:])
    assert same_bits(ya, yb)
    # and the move did happen: stream 0 crossfades in the first block
    c, _ = sem_engine(block)
    run(c, x[:, :, :block * 2])
    yc = run(c, x[:, :, block * 3:])
    assert not same_bits(ya[0], yc[0])


@gpu
def test_all_streams_move_like_a_schedule():
    block = 256
    x = S.stream_inputs(4, block * 6, base_seed=54)
    a, _ = sem_engine(block)
    b, _ = sem_engine(block)
    run(a, x[:, :, :block * 2]); run(b, x[:, :, :block * 2])
    a.move_stream_hrir(ohs.OHS_ALL, 1)
    ya = run(a, x[:, :, block * 2:])
    yb = run(b, x[:, :, block * 2:], np.ones((4, 4), np.int32))
    assert same_bits(ya, yb)


@gpu
def test_state_export_import_between_scheduled_calls():
    block, k = 128, 6
    x = S.stream_inputs(4, block * 2 * k, base_seed=55)
    rng = np.random.default_rng(9)
    s1 = rng.integers(0, 2, (4, k)).astype(np.int32)
    s2 = rng.integers(0, 2, (4, k)).astype(np.int32)
    a, _ = sem_engine(block)
    run(a, x[:, :, :block * k], s1)
    blob = a.state_export()
    ya = run(a, x[:, :, block * k:], s2)
    b, _ = sem_engine(block)
    for s in range(4):
        b.bind_stream_hrir(s, int(s1[s, -1]))   # bindings are configuration, not state
    b.state_import(blob)
    yb = run(b, x[:, :, block * k:], s2)
    assert same_bits(ya, yb)


@gpu
def test_rejected_schedule_leaves_the_engine_untouched():
    block, k = 128, 4
    x = S.stream_inputs(4, block * 3 * k, base_seed=56)
    a, _ = sem_engine(block)
    b, _ = sem_engine(block)
    good = np.ones((4, k), np.int32)
    run(a, x[:, :, :block * k], good); run(b, x[:, :, :block * k], good)
    bad = np.zeros((4, k), np.int32)
    bad[2, 1] = 2   # out of range (two sets)
    with pytest.raises(ohs.OhsError):
        run(a, x[:, :, block * k:2 * block * k], bad)
    a.move_stream_hrir(1, 0); b.move_stream_hrir(1, 0)
    with pytest.raises(ohs.OhsError):   # too few columns
        run(a, x[:, :, block * k:2 * block * k], good[:, :k - 1])
    a.set_conv_enable(False)
    with pytest.raises(ohs.OhsError):   # convolution disabled
        run(a, x[:, :, block * k:2 * block * k], good)
    a.set_conv_enable(True)
    assert same_bits(run(a, x[:, :, block * k:]), run(b, x[:, :, block * k:]))
