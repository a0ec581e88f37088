"""Every stream renders as if it were alone.  A CTA of the render kernel holds G <= 7 streams, and they share its shared
memory: EQ warps of six chains, one staging warp, FFT buffers that the long-response path reuses as filter tiles, and
the time-batched route's scratch.  A stream's output must depend only on its own input, its own state and its own
bindings (HRIR set, EQ set, gain), whatever its neighbours carry.

Routes, forced the way the other GPU tests force them:
  R1  throughput render_kernel<2B, G, 0>: calls of >= 3 blocks with a partial last CTA, G in {2, 3, 7} at B = 256 (two
      bands per EQ lane) and G = 2 at B = 1024 (one band per lane; <2048, 3> and <2048, 7> do not fit in shared
      memory), single-partition sets (fused path) and multi-partition sets
  R2  latency render_kernel<512, G, 1>: calls of one and two blocks
  R3  EQ-only mode (convolution off) with a ragged last block
  R4  the time-batched route (P >= 8, >= 8 blocks per call), its EQ pre-pass on its own stream, on CTAs of six streams
      that own their SM (>= 12 streams) and on thin CTAs of three
  R5  render_kernel<N, G, V, true>, the moving-sources kernel, which a multi-set engine with a delay line runs when some
      stream is bound to a one-partition set
Bindings derive from s % U and the inputs tile with period U, U prime to G, so that twin streams (same input, same
bindings) sit in different CTAs and different slots; every CTA holds streams with different bindings.

Bars: the oracle (oracle/ohs_oracle.c) at TOL for the chain, bit-exact for the EQ stage, bit-identical between twins
and between renders that differ only outside the stream or the row being checked."""
import dataclasses

import numpy as np
import pytest

import open_headstage_b200 as ohs
from open_headstage_b200 import signals as S
from oracle import oracle as O

gpu = pytest.mark.gpu
TOL = 1e-5
FS = 48000.0
GAINS = (0.5, 1.0, 0.25, -0.75, 2.0, 0.0)
ERR_ALIGNMENT = -6   # OHS_ERR_ALIGNMENT


def preset_coeffs(preset):
    return np.stack([O.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in preset]).astype(np.float32)


def eq_sets():
    """The three EQ sets: typical, harsh, and typical with band 6 disabled (a CTA holding that set leaves the continuous
    chain for the per-block one while the other CTAs of the launch stay on it)."""
    typ, harsh = preset_coeffs(S.EQ_PRESET_TYPICAL), preset_coeffs(S.EQ_PRESET_HARSH)
    return [(typ, [1] * 10), (harsh, [1] * 10), (typ, [1] * 6 + [0] + [1] * 3)]


def binding(u):
    """(HRIR set, EQ set, gain) of binding class u: neighbouring classes differ in HRIR set."""
    return u % 3, (u + u // 3) % 3, GAINS[u % 6]


def layout(n_streams, g):
    """(CTA, slot) of every stream when the render kernel holds g streams per CTA."""
    return [(s // g, s % g) for s in range(n_streams)]


def check_layout(n_streams, g, u, lone=True):
    """Every class of twins spans several CTAs and several slots, every CTA of two or more streams mixes HRIR sets, EQ
    sets and gains, and (lone) the last CTA holds one stream."""
    where = layout(n_streams, g)
    for k in range(min(u, n_streams - u)):
        twins = [where[s] for s in range(k, n_streams, u)]
        assert len({w[0] for w in twins}) == len(twins) and len({w[1] for w in twins}) > 1, (n_streams, g, u, k)
    for c in range((n_streams + g - 1) // g):
        members = [binding(s % u) for s in range(c * g, min(n_streams, (c + 1) * g))]
        if len(members) > 1:
            for k in range(3):
                assert len({m[k] for m in members}) > 1, (n_streams, g, u, c, k)
    assert n_streams % g == 1 or not lone


def seq_sum_f32(rows):
    """rows[s] summed in stream order, each addition rounded to f32 (np.sum adds pairwise)."""
    acc = np.zeros(rows.shape[1:], np.float32)
    for r in rows:
        acc = (acc + r).astype(np.float32)
    return acc


def hrir_sets(block, parts, seed=61):
    """One HRIR set per entry of `parts`, with that many partitions of `block`; tap counts all differ."""
    out = []
    for k, p in enumerate(parts):
        taps = (p - 1) * block + block // 3 + 7 * k
        out.append(S.synthetic_hrir_set(taps, taps / 5.0, seed=seed + k))
    return out


@dataclasses.dataclass(frozen=True)
class Route:
    block: int
    n_streams: int
    u: int                        # binding / input period
    parts: tuple                  # partitions of the three HRIR sets
    calls: tuple                  # frames of each call
    g: int = 0                    # OHS_STREAMS_PER_CTA (0: the engine picks)
    conv: bool = True
    host: bool = False            # ohs_process instead of ohs_process_device

    @property
    def n(self):
        return sum(self.calls)

    @property
    def pre_g(self):
        """streams per CTA of the kernel that holds the EQ chains: the render kernel, or the time-batched pre-pass"""
        if min(self.parts) >= 8:
            return 6 if self.n_streams >= 12 else 3
        return self.g


def _r1(g, block, parts, host=False):
    n = 16 if g == 3 else 15
    return Route(block, n, 11, parts, (3 * block, 4 * block), g=g, host=host)


ROUTES = {
    "r1_g2_b256_p1": _r1(2, 256, (1, 1, 1)),
    "r1_g3_b256_p1": _r1(3, 256, (1, 1, 1)),
    "r1_g7_b256_p1": _r1(7, 256, (1, 1, 1)),
    "r1_g2_b256_p3": _r1(2, 256, (3, 2, 4)),
    "r1_g3_b256_p3_host": _r1(3, 256, (3, 2, 4), host=True),
    "r1_g7_b256_p3": _r1(7, 256, (3, 2, 4)),
    "r1_g2_b1024_p1": _r1(2, 1024, (1, 1, 1)),
    "r1_g2_b1024_p3": _r1(2, 1024, (3, 2, 4)),
    "r2_g3_k1_k2": Route(256, 16, 11, (3, 2, 4), (256, 512, 256, 512), g=3),
    "r3_b256_ragged": Route(256, 16, 11, (1, 1, 1), (700, 3 * 256 + 13), g=3, conv=False),
    "r3_b1024_ragged": Route(1024, 15, 11, (1, 1, 1), (1500, 2 * 1024 + 29), g=2, conv=False),
    "r4_own_sm": Route(128, 16, 11, (8, 9, 11), (16 * 128, 12 * 128)),
    "r4_thin": Route(128, 8, 5, (8, 9, 11), (16 * 128, 12 * 128)),
    "r5_moving": Route(256, 16, 11, (1, 3, 2), (3 * 256, 4 * 256), g=3),
}
CONV_ROUTES = [k for k, r in ROUTES.items() if r.conv]
ISOLATION_ROUTES = ["r1_g3_b256_p3_host", "r1_g2_b1024_p3", "r1_g2_b256_p1", "r2_g3_k1_k2", "r3_b256_ragged", "r4_own_sm",
                    "r4_thin", "r5_moving"]


def configure(monkeypatch, route):
    if route.g:
        monkeypatch.setenv("OHS_STREAMS_PER_CTA", str(route.g))


def make_engine(route, n_bands=10, eq=True, sets=None, bind=True):
    sets = sets if sets is not None else hrir_sets(route.block, route.parts)
    e = ohs.Engine(route.n_streams, route.block, max(len(h[0]) for h in sets), n_bands=n_bands, n_hrir_sets=3, n_eq_sets=3)
    if route.g and e.streams_per_cta() != route.g:
        pytest.skip("render_kernel<%d,%d> does not fit in shared memory; production never selects it" % (2 * route.block, route.g))
    for k, h in enumerate(sets):
        e.set_hrir_set(h, hrir_set=k)
    for k, (c, en) in enumerate(eq_sets()):
        for b in range(n_bands):
            e.eq_set_band(b, c[b], bool(en[b]), eq_set=k)
    if bind:
        for s in range(route.n_streams):
            hs, es, g = binding(s % route.u)
            e.bind_stream_hrir(s, hs); e.bind_stream_eq(s, es); e.set_gain(g, stream=s)
    e.set_eq_enable(eq)
    e.set_conv_enable(route.conv)
    return e


def render(e, route, x, calls=None):
    """x through `route`'s calls: ohs_process (host flavour) or ohs_process_device on unpadded device rows."""
    calls = calls or route.calls
    if route.host:
        out, at = [], 0
        for c in calls:
            out.append(e.process(x[:, :, at:at + c])); at += c
        return np.concatenate(out, axis=2)
    import torch

    n = x.shape[2]
    stride = (n + 3) // 4 * 4   # device rows start 16-byte aligned
    src = torch.zeros((x.shape[0], 2, stride), dtype=torch.float32, device="cuda")
    src[:, :, :n] = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    dst = torch.empty_like(src)
    at = 0
    for c in calls:
        e.process_device(src.data_ptr() + 4 * at, dst.data_ptr() + 4 * at, c, row_stride=stride); at += c
    e.sync()
    return dst[:, :, :n].cpu().numpy()


def inputs(route, seed=0, scale=1.0):
    return (np.float32(scale) * S.stream_inputs(route.n_streams, route.n, base_seed=5000 + 37 * seed, unique=route.u)).astype(np.float32)


def oracle_stream(x1, route, u, sets, n_bands=10, eq=True):
    """One stream x1[2, n] through the reference chain with binding class u's HRIR set, EQ set and gain."""
    hs, es, g = binding(u)
    c, en = eq_sets()[es]
    if not route.conv:
        q = O.StereoParametricEQ(n_bands, FS)
        for b in range(n_bands):
            q.set_band_raw(b, c[b], en[b])
        l, r = q.process_block(x1[0], x1[1]) if eq else (x1[0], x1[1])
        return np.stack([l, r]).astype(np.float32) * np.float32(g)
    if not eq or n_bands == 0:
        c, en = np.zeros((1, 5), np.float32), [0]
    else:
        c, en = c[:n_bands], en[:n_bands]
    return O.render_batch(x1[None], route.block, sets[hs], c, en, eq, g)[0][0]


def assert_twins(y, u):
    for s in range(u, y.shape[0]):
        assert y[s].tobytes() == y[s % u].tobytes(), "stream %d differs from its twin %d" % (s, s % u)


def assert_oracle(y, x, route, sets, n_bands=10, eq=True):
    """Every binding class and the lone stream of the partial last CTA against the oracle run on that stream alone: bit
    for bit in EQ-only mode (the EQ stage and one f32 multiply by the gain), within TOL with the convolution on."""
    for s in sorted(set(range(route.u)) | {route.n_streams - 1}):
        ref = oracle_stream(x[s], route, s % route.u, sets, n_bands, eq)
        if route.conv:
            err = float(np.max(np.abs(y[s] - ref)))
            assert err <= TOL, (s, err)
        else:
            assert y[s].tobytes() == ref.tobytes(), "stream %d (max %g)" % (s, np.max(np.abs(y[s] - ref)))


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_binding_layout_mixes_every_cta():
    for name, r in ROUTES.items():
        check_layout(r.n_streams, r.pre_g, r.u, lone=r.pre_g == r.g)
        assert r.n_streams > r.u and all(c % 4 == 0 for c in r.calls[:-1]), name
        if r.conv:
            assert all(c % r.block == 0 for c in r.calls), name
    check_layout(1024, 7, 11, lone=False)
    # the routes the names promise: multi-partition sets distinct, P >= 8 for R4, a one-partition set beside longer ones in R5
    assert len(set(ROUTES["r1_g3_b256_p3_host"].parts)) == 3 and min(ROUTES["r1_g3_b256_p3_host"].parts) > 1
    assert min(ROUTES["r4_own_sm"].parts) >= 8 and ROUTES["r4_own_sm"].calls[-1] >= 8 * 128
    assert 1 in ROUTES["r5_moving"].parts and max(ROUTES["r5_moving"].parts) > 1
    for r in ROUTES.values():
        sets = hrir_sets(r.block, r.parts)
        assert [-(-len(h[0]) // r.block) for h in sets] == list(r.parts)
        assert len({len(h[0]) for h in sets}) == 3


def test_sequential_sum_is_stream_order():
    rng = np.random.default_rng(3)
    rows = (rng.standard_normal((1023, 64)) * np.exp2(rng.integers(-12, 12, (1023, 64)))).astype(np.float32)
    want = np.zeros(64, np.float32)
    for s in range(rows.shape[0]):
        for i in range(64):
            want[i] = np.float32(want[i] + rows[s, i])
    assert seq_sum_f32(rows).tobytes() == want.tobytes()
    # the check tells stream order from the pairwise order of np.sum and from summing streams in pairs
    assert seq_sum_f32(rows).tobytes() != np.sum(np.ascontiguousarray(rows.T), axis=1, dtype=np.float32).tobytes()
    assert seq_sum_f32(rows).tobytes() != seq_sum_f32(np.concatenate([rows[0:-1:2] + rows[1::2], rows[-1:]])).tobytes()


@pytest.mark.parametrize("scale_exp", [-126, -135])
@pytest.mark.parametrize("preset", ["typical", "harsh"])
def test_oracle_keeps_subnormals(scale_exp, preset):
    """The subnormal GPU check below means something only if the reference output is subnormal: a flush to zero on both
    sides would agree too."""
    c = preset_coeffs(S.EQ_PRESET_HARSH if preset == "harsh" else S.EQ_PRESET_TYPICAL)
    x = (S.stream_inputs(1, 4096, base_seed=77)[0] * np.float32(2.0 ** scale_exp)).astype(np.float32)
    assert np.count_nonzero(x) > 4000   # 2^-135 x is still subnormal, not zero
    q = O.StereoParametricEQ(10, FS)
    for b in range(10):
        q.set_band_raw(b, c[b], True)
    l, _ = q.process_block(x[0], x[1])
    sub = np.count_nonzero((l != 0) & (np.abs(l) < np.finfo(np.float32).tiny))
    assert sub > 0.85 * l.size, sub


def test_oracle_power_of_two_scaling():
    """The reference chain commutes with 2^k exactly (every operation is +, -, * or fma on normal values): the
    definition the GPU scaling test holds the engine to."""
    r = ROUTES["r1_g3_b256_p3_host"]
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r)[:2]
    for u in (1, 3):
        y = oracle_stream(x[u % 2], r, u, sets)
        for k in (-20, 20):
            assert oracle_stream(np.ldexp(x[u % 2], k).astype(np.float32), r, u, sets).tobytes() == np.ldexp(y, k).astype(np.float32).tobytes()


# ---- 1. heterogeneous bindings against the oracle ---------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", list(ROUTES))
def test_heterogeneous_bindings(name, monkeypatch):
    r = ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r)
    y = render(make_engine(r, sets=sets), r, x)
    assert np.isfinite(y).all()
    assert_twins(y, r.u)
    assert_oracle(y, x, r, sets)


@gpu
def test_heterogeneous_bindings_config2_width():
    """Config 2 at full width: 1024 streams, block 256, 256-tap sets -> render_kernel<512, 7> chosen by the engine."""
    r = Route(256, 1024, 11, (1, 1, 1), (8 * 256, 8 * 256))
    sets = [S.synthetic_hrir_set(t, 40.0, seed=70 + k) for k, t in enumerate((256, 200, 150))]
    x = inputs(r)
    e = make_engine(r, sets=sets)
    assert e.streams_per_cta() == 7
    y = render(e, r, x)
    assert_twins(y, r.u)
    assert_oracle(y, x, r, sets)


# ---- 2. changes between calls ------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["r1_g3_b256_p3_host", "r1_g2_b1024_p3", "r3_b256_ragged", "r4_own_sm"])
def test_changes_between_calls(name, monkeypatch):
    """Between two calls: one band of EQ set 1 gets new coefficients, stream 4 moves from EQ set 2 to EQ set 0, stream 7
    gets a new gain.  The oracle makes the same changes at the same block, one chain per stream.  ohs_bind_stream_eq
    keeps the stream's biquad state (include/ohs.h), as update_band_coeffs does in the reference: the oracle's rebound
    chain only gets new coefficients.  Bit-exact in EQ-only mode, within TOL with the convolution."""
    r = ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r)
    c1 = r.calls[0]
    band, new_c = 3, O.eq_design(S.PEAK, FS, 900.0, 2.0, 5.0)
    rebound, regained, new_gain = 4, 7, -1.5
    assert binding(rebound % r.u)[1] == 2
    e = make_engine(r, sets=sets)
    first = render(e, r, x[:, :, :c1], calls=(c1,))
    e.eq_set_band(band, new_c, True, eq_set=1)
    e.bind_stream_eq(rebound, 0)
    e.set_gain(new_gain, stream=regained)
    second = render(e, r, x[:, :, c1:], calls=r.calls[1:])
    y = np.concatenate([first, second], axis=2)
    for s in range(r.n_streams):
        hs, es, g = binding(s % r.u)
        q = O.StereoParametricEQ(10, FS)
        c, en = eq_sets()[es]
        for b in range(10):
            q.set_band_raw(b, c[b], en[b])
        conv = O.ConvolutionEngine(r.block)
        for p in range(4):
            conv.set_ir(p, sets[hs][p])
        out = []
        for k, (a, b) in enumerate(((0, c1), (c1, r.n))):
            if k == 1:
                if es == 1:
                    q.set_band_raw(band, new_c, True)
                if s == rebound:
                    c0, en0 = eq_sets()[0]
                    for bb in range(10):
                        q.set_band_raw(bb, c0[bb], en0[bb])
                if s == regained:
                    g = new_gain
            if r.conv:
                out.append(np.stack(O.chain_process(conv, q, True, False, g, x[s, 0, a:b], x[s, 1, a:b])))
            else:
                l, rr = q.process_block(x[s, 0, a:b], x[s, 1, a:b])
                out.append(np.stack([l, rr]) * np.float32(g))
        ref = np.concatenate(out, axis=1)
        if r.conv:
            assert float(np.max(np.abs(y[s] - ref))) <= TOL, s
        else:
            assert y[s].tobytes() == ref.tobytes(), s
    # the state is kept, not reset: the rebound stream's second call differs from a chain restarted at the change
    if not r.conv:
        q = O.StereoParametricEQ(10, FS)
        c0, en0 = eq_sets()[0]
        for b in range(10):
            q.set_band_raw(b, c0[b], en0[b])
        fresh = np.stack(q.process_block(x[rebound, 0, c1:], x[rebound, 1, c1:])) * np.float32(binding(rebound % r.u)[2])
        assert fresh.tobytes() != y[rebound, :, c1:].tobytes()


# ---- 3. band counts ----------------------------------------------------------------------------------------------
BAND_ROUTES = {
    "eq_only_b256": Route(256, 16, 11, (1, 1, 1), (700, 3 * 256 + 13), g=3, conv=False),
    "eq_only_b1024": Route(1024, 15, 11, (1, 1, 1), (1500, 2 * 1024 + 29), g=2, conv=False),
    "r1": ROUTES["r1_g3_b256_p3_host"],
    "r2": ROUTES["r2_g3_k1_k2"],
    "r4": ROUTES["r4_own_sm"],
}


@gpu
@pytest.mark.parametrize("n_bands", [1, 2, 5, 9])
@pytest.mark.parametrize("name", list(BAND_ROUTES))
def test_band_counts(name, n_bands, monkeypatch):
    """Fewer than ten bands: odd counts leave a lane half used (two bands per lane at B <= 512), and every CTA leaves
    the continuous chain.  EQ-only bit-exact against StereoParametricEQ(n_bands), the chain within TOL."""
    r = BAND_ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=n_bands)
    y = render(make_engine(r, n_bands=n_bands, sets=sets), r, x)
    assert_twins(y, r.u)
    assert_oracle(y, x, r, sets, n_bands=n_bands)


@gpu
@pytest.mark.parametrize("n_bands", [1, 2, 5, 9])
def test_band_counts_state_export_import(n_bands, monkeypatch):
    r = ROUTES["r1_g3_b256_p3_host"]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=20 + n_bands)
    c1 = r.calls[0]
    whole = render(make_engine(r, n_bands=n_bands, sets=sets), r, x)
    a = make_engine(r, n_bands=n_bands, sets=sets)
    first = render(a, r, x[:, :, :c1], calls=(c1,))
    b = make_engine(r, n_bands=n_bands, sets=sets)
    b.state_import(a.state_export())
    second = render(b, r, x[:, :, c1:], calls=r.calls[1:])
    assert np.concatenate([first, second], axis=2).tobytes() == whole.tobytes()


# ---- 4. isolation ------------------------------------------------------------------------------------------------
def poison(x, route, t0):
    """A NaN at one sample of a stream in the middle of a CTA and +Inf in another stream, both in block t0."""
    g = route.g or route.pre_g
    m, k = g + g // 2, 2
    y = x.copy()
    y[m, 0, t0 * route.block + route.block // 2 + 3] = np.nan
    y[k, 1, t0 * route.block + 5] = np.inf
    return y, (m, k)


@gpu
@pytest.mark.parametrize("name", ISOLATION_ROUTES)
def test_nonfinite_input_stays_in_its_stream(name, monkeypatch):
    r = ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=3)
    xp, bad = poison(x, r, 1)
    clean = render(make_engine(r, sets=sets), r, x)
    dirty = render(make_engine(r, sets=sets), r, xp)
    for s in range(r.n_streams):
        if s in bad:
            assert not np.isfinite(dirty[s]).all() or binding(s % r.u)[2] == 0.0, s
        else:
            assert dirty[s].tobytes() == clean[s].tobytes(), "stream %d changed by a non-finite sample in streams %s" % (s, bad)


RECOVERY_ROUTES = {
    "r1": ROUTES["r1_g3_b256_p3_host"],
    "r1_b1024": ROUTES["r1_g2_b1024_p3"],
    "r4": Route(128, 16, 11, (8, 9, 11), (12 * 128, 8 * 128, 12 * 128)),
    "r5": ROUTES["r5_moving"],
}


@gpu
@pytest.mark.parametrize("handover", ["same_engine", "state_export_import"])
@pytest.mark.parametrize("name", list(RECOVERY_ROUTES))
def test_nan_recovery_with_eq_off(name, handover, monkeypatch):
    """With the EQ off a NaN in block t0 reaches the spectra of blocks t0 and t0 + 1 and nothing else: the stream is
    finite again from block t0 + P + 1 on (P: its set's partitions), when both overlap-save and the reference's
    overlap-add have forgotten it, and matches the oracle fed the same input.  Later recovery would mean a history slot
    multiplied by a zero filter, or a slot never overwritten."""
    if handover == "state_export_import" and name in ("r1_b1024", "r5"):
        pytest.skip("one engine hand-over per route family is enough")
    r = RECOVERY_ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=4)
    t0 = 1
    xp, (m, k) = poison(x, r, t0)
    e = make_engine(r, eq=False, sets=sets)
    if handover == "same_engine":
        y = render(e, r, xp)
    else:
        c1 = r.calls[0]
        first = render(e, r, xp[:, :, :c1], calls=(c1,))
        f = make_engine(r, eq=False, sets=sets)
        f.state_import(e.state_export())
        y = np.concatenate([first, render(f, r, xp[:, :, c1:], calls=r.calls[1:])], axis=2)
    for s in (m, k):
        hs, _, g = binding(s % r.u)
        start = (t0 + r.parts[hs] + 1) * r.block
        assert start < r.n
        assert np.isfinite(y[s, :, start:]).all(), (s, r.parts[hs], np.flatnonzero(~np.isfinite(y[s, 0]))[-1:] // r.block)
        ref = oracle_stream(xp[s], r, s % r.u, sets, eq=False)
        assert float(np.max(np.abs(y[s, :, start:] - ref[:, start:]))) <= TOL, s
        if g != 0.0:
            assert not np.isfinite(y[s, :, t0 * r.block:(t0 + 1) * r.block]).all()   # the poison did arrive


@gpu
@pytest.mark.parametrize("name", ["r1_g3_b256_p3_host", "r1_g2_b1024_p3", "r1_g7_b256_p1", "r4_own_sm", "r5_moving"])
def test_nan_tap_stays_in_its_hrir_set(name, monkeypatch):
    r = ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    bad_sets = [h.copy() for h in sets]
    bad_sets[1][2, 3] = np.nan   # set 1, path RSL, tap 3
    x = inputs(r, seed=5)
    clean = render(make_engine(r, sets=sets), r, x)
    dirty = render(make_engine(r, sets=bad_sets), r, x)
    for s in range(r.n_streams):
        hs, _, g = binding(s % r.u)
        if hs == 1:
            assert not np.isfinite(dirty[s, 0]).all(), s
        else:
            assert dirty[s].tobytes() == clean[s].tobytes(), s


SENTINEL = np.int32(0x7FA5A5A5)   # a signalling-NaN bit pattern no render produces


def padded(x, stride, pad_bits):
    """x[S, 2, n] in rows of `stride` floats, the padding filled with the int32 bit pattern pad_bits (or random bytes)."""
    buf = np.empty(x.shape[:2] + (stride,), np.float32)
    if pad_bits is None:
        buf.view(np.uint8)[...] = np.random.default_rng(9).integers(0, 256, buf.view(np.uint8).shape, dtype=np.uint8)
    else:
        buf.view(np.int32)[...] = pad_bits
    buf[:, :, :x.shape[2]] = x
    return buf


def device_render_padded(e, x, stride, calls, in_pad, out_pad, in_place=False):
    import torch

    src = torch.from_numpy(padded(x, stride, in_pad)).cuda()
    dst = src if in_place else torch.from_numpy(padded(np.zeros_like(x), stride, out_pad)).cuda()
    at = 0
    for c in calls:
        e.process_device(src.data_ptr() + 4 * at, dst.data_ptr() + 4 * at, c, row_stride=stride); at += c
    e.sync()
    return dst.cpu().numpy()


PAD_ROUTES = {
    "r1_k1": (ROUTES["r1_g3_b256_p3_host"], (256,) * 7),
    "r1_k3": (ROUTES["r1_g3_b256_p3_host"], (3 * 256, 3 * 256, 256)),
    "r3_ragged": (ROUTES["r3_b256_ragged"], None),
    "r4": (ROUTES["r4_own_sm"], None),
    "r5": (ROUTES["r5_moving"], None),
}


@gpu
@pytest.mark.parametrize("in_place", [False, True])
@pytest.mark.parametrize("name", list(PAD_ROUTES))
def test_row_padding_is_neither_read_nor_written(name, in_place, monkeypatch):
    """Input rows padded with NaN, output rows padded with a sentinel: outputs bit-identical to a render with zero
    padding, and the sentinel (in place: the NaN padding) comes back untouched."""
    r, calls = PAD_ROUTES[name]
    calls = calls or r.calls
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=6)
    stride = ((r.n + 4 + 3) // 4) * 4 + 8
    want = device_render_padded(make_engine(r, sets=sets), x, stride, calls, 0, 0, in_place)
    got = device_render_padded(make_engine(r, sets=sets), x, stride, calls, np.float32(np.nan).view(np.int32) | 0x5A5A,
                               SENTINEL, in_place)
    assert got[:, :, :r.n].tobytes() == want[:, :, :r.n].tobytes()
    pad = got[:, :, r.n:].view(np.int32)
    assert (pad == ((np.float32(np.nan).view(np.int32) | 0x5A5A) if in_place else SENTINEL)).all()


@gpu
@pytest.mark.parametrize("fmt_in,fmt_out,conv", [(ohs.FMT_S16, ohs.FMT_F32, False), (ohs.FMT_S24, ohs.FMT_F32, False),
                                                  (ohs.FMT_S16, ohs.FMT_S16, True), (ohs.FMT_S24, ohs.FMT_S24, True),
                                                  (ohs.FMT_S16, ohs.FMT_S24, False)])
def test_pcm_row_padding(fmt_in, fmt_out, conv, monkeypatch):
    """ohs_process_device_pcm on padded rows: random bytes in the input padding, a sentinel in the output padding.  In
    EQ-only mode n_frames is not a multiple of the S16 group (8) or the S24 group (16), so the decode's partial last group
    lands next to the output padding."""
    import torch

    r = ROUTES["r3_b256_ragged"] if not conv else ROUTES["r1_g3_b256_p3_host"]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    n = 3 * 256 - 57 if not conv else 3 * 256
    stride = 3 * 256 + 32
    x = (0.9 * inputs(r, seed=7)[:, :, :n]).astype(np.float32)
    q = S.pcm_encode(x, fmt_in)
    nb_in = 2 if fmt_in == ohs.FMT_S16 else 3
    nb_out = {ohs.FMT_F32: 4, ohs.FMT_S16: 2, ohs.FMT_S24: 3}[fmt_out]
    raw = q.astype("<i2").view(np.uint8) if fmt_in == ohs.FMT_S16 else S.pack_s24(q)
    rng = np.random.default_rng(11)
    outs = []
    for dirty in (False, True):
        ib = np.zeros((r.n_streams, 2, stride * nb_in), np.uint8)
        if dirty:
            ib[...] = rng.integers(0, 256, ib.shape, dtype=np.uint8)
        ib[:, :, :n * nb_in] = raw.reshape(r.n_streams, 2, -1)
        ob = np.full((r.n_streams, 2, stride * nb_out), 0xA5 if dirty else 0, np.uint8)
        e = make_engine(r, sets=sets)
        di, do = torch.from_numpy(ib).cuda(), torch.from_numpy(ob).cuda()
        e.process_device_pcm(di.data_ptr(), fmt_in, do.data_ptr(), fmt_out, n, row_stride=stride)
        e.sync()
        outs.append(do.cpu().numpy())
    assert outs[1][:, :, :n * nb_out].tobytes() == outs[0][:, :, :n * nb_out].tobytes()
    assert (outs[1][:, :, n * nb_out:] == 0xA5).all()


# ---- 5. numeric edges --------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scale_exp", [-126, -135])
@pytest.mark.parametrize("block", [256, 1024])
@pytest.mark.parametrize("chain", ["continuous", "per_block"])
def test_subnormal_inputs_eq_bit_exact(block, chain, scale_exp):
    """EQ-only on inputs scaled into and below the normal range: bit-exact against the oracle, which keeps subnormals
    (test_oracle_keeps_subnormals).  A library built to flush subnormals to zero fails here."""
    c = preset_coeffs(S.EQ_PRESET_HARSH)
    en = [1] * 10 if chain == "continuous" else [1] * 4 + [0] + [1] * 5
    n = 3 * block + 37
    x = (S.stream_inputs(5, n, base_seed=88) * np.float32(2.0 ** scale_exp)).astype(np.float32)
    e = ohs.Engine(5, block, 1)
    e.set_conv_enable(False); e.set_eq_enable(True)
    for b in range(10):
        e.eq_set_band(b, c[b], bool(en[b]))
    y = e.process(x)
    for s in range(5):
        q = O.StereoParametricEQ(10, FS)
        for b in range(10):
            q.set_band_raw(b, c[b], en[b])
        l, r = q.process_block(x[s, 0], x[s, 1])
        assert y[s, 0].tobytes() == l.tobytes() and y[s, 1].tobytes() == r.tobytes(), s


@gpu
@pytest.mark.parametrize("k", [-20, 20])
@pytest.mark.parametrize("name", ["r1_g3_b256_p3_host", "r1_g2_b1024_p3", "r1_g2_b256_p1", "r2_g3_k1_k2", "r3_b256_ragged",
                                  "r4_own_sm", "r5_moving"])
def test_power_of_two_scaling_is_exact(name, k, monkeypatch):
    """render(2^k x) == 2^k render(x) bit for bit: every operation of the chain is +, -, * or fma on normal values, and
    binary rounding does not depend on scale.  Anything that depends on absolute level (an added constant, a clamp, an
    epsilon, a flush) breaks it."""
    r = ROUTES[name]
    configure(monkeypatch, r)
    sets = hrir_sets(r.block, r.parts)
    x = inputs(r, seed=8)
    y = render(make_engine(r, sets=sets), r, x)
    ys = render(make_engine(r, sets=sets), r, np.ldexp(x, k).astype(np.float32))
    assert ys.tobytes() == np.ldexp(y, k).astype(np.float32).tobytes()


# ---- 6. mix_streams_kernel ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_frames", [4, 1028, 3 * 1024 + 4])
@pytest.mark.parametrize("n_streams", [1, 5, 7, 1023])
def test_mix_is_a_sequential_f32_sum(n_streams, n_frames):
    """ohs_mix_device: bus[c] = in[0][c] + in[1][c] + ... in stream order, each addition rounded to f32; padded row and
    bus strides, NaN in the input padding, the bus padding left untouched."""
    import torch

    rng = np.random.default_rng(n_streams * 7 + n_frames)
    x = (rng.standard_normal((n_streams, 2, n_frames)) * np.exp2(rng.integers(-10, 10, (n_streams, 2, n_frames)))).astype(np.float32)
    row_stride, bus_stride = n_frames + 12, n_frames + 8
    src = torch.from_numpy(padded(x, row_stride, np.float32(np.nan).view(np.int32))).cuda()
    bus = torch.from_numpy(padded(np.zeros((1, 2, n_frames), np.float32), bus_stride, SENTINEL)[0]).cuda()
    e = ohs.Engine(n_streams, 256, 1, n_bands=0)
    e.mix_device(src.data_ptr(), bus.data_ptr(), n_frames, row_stride=row_stride, bus_stride=bus_stride)
    e.sync()
    got = bus.cpu().numpy()
    for c in range(2):
        assert got[c, :n_frames].tobytes() == seq_sum_f32(x[:, c]).tobytes(), c
    assert (got[:, n_frames:].view(np.int32) == SENTINEL).all()
    with pytest.raises(ohs.OhsError) as err:
        e.mix_device(src.data_ptr(), bus.data_ptr(), n_frames + 2, row_stride=row_stride, bus_stride=bus_stride)
    assert err.value.code == ERR_ALIGNMENT
