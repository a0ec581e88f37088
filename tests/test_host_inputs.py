"""Host-side rows next to the hot path (SURVEY.md §8f): HRIR selection/wiring and AutoEQ CSV ingestion.  CPU only."""
import numpy as np
import pytest

from open_headstage_b200 import autoeq, sofa


def test_nearest_neighbour_selection_matches_survey_indices(cipic):
    h = sofa.from_arrays(cipic["ir"], cipic["pos"], float(cipic["fs"]))
    assert h.filter_length == 200
    assert h.nearest(30.0, 0.0) == 308     # left speaker (SURVEY.md Q3)
    assert h.nearest(330.0, 0.0) == 908    # right speaker
    assert h.nearest(0.0, 0.0) == 608
    assert h.nearest(-30.0, 0.0) == 908    # azimuth wraps
    assert sofa.ui_azimuth_to_sofa(-30.0) == 30.0 and sofa.ui_azimuth_to_sofa(30.0) == 330.0
    l, r = h.get_hrtf_irs(30.0, 0.0)
    assert np.array_equal(l, cipic["ir"][308, 0]) and np.array_equal(r, cipic["ir"][308, 1])
    # every measurement is its own nearest neighbour: selection is an exact index lookup
    for i in range(0, 1250, 97):
        assert h.nearest(float(cipic["pos"][i, 0]), float(cipic["pos"][i, 1])) == i


def test_wire_speakers_calls_set_ir_for_the_four_paths(cipic):
    calls = []

    class FakeEngine:
        def set_ir(self, path, ir, hrir_set=0):
            calls.append((path, np.asarray(ir).copy(), hrir_set))

    h = sofa.from_arrays(cipic["ir"], cipic["pos"], 44100.0)
    il, ir_ = sofa.wire_speakers(FakeEngine(), h, sofa.ui_azimuth_to_sofa(-30.0), 0.0, sofa.ui_azimuth_to_sofa(30.0), 0.0)
    assert (il, ir_) == (308, 908)
    assert [c[0] for c in calls] == [0, 1, 2, 3]
    assert np.array_equal(calls[0][1], cipic["ir"][308, 0]) and np.array_equal(calls[3][1], cipic["ir"][908, 1])


@pytest.fixture(scope="module")
def cipic_sofa(cipic, tmp_path_factory):
    """The reference's bundled CIPIC subject 003 file, rebuilt from tests/golden/cipic003_hrir.npz (what its two datasets
    decode to, see tests/golden/make_sofa_fixture.py): full size, M = 1250 x R = 2 x N = 200, as byte-shuffled f64 zlib
    streams among unrelated bytes."""
    path = tmp_path_factory.mktemp("sofa") / "subject_003.sofa"
    write_sofa_datasets(path, cipic["pos"], cipic["ir"], np.random.default_rng(3))
    return str(path)


def test_load_sofa_reads_the_bundled_file_without_hdf5(cipic, cipic_sofa):
    """The bundled CIPIC data at full size, read back exactly.  The file is cipic_sofa's rebuild: the real file's HDF5
    byte layout around the two datasets is not exercised."""
    h = sofa.load_sofa(cipic_sofa)
    assert h.ir.shape == (1250, 2, 200)
    assert np.array_equal(h.ir, cipic["ir"]) and np.array_equal(h.position, cipic["pos"])


def test_parse_autoeq_csv():
    text = "Filter-Type,Fc,Q,Gain\nLS,105,0.7,6.5\nPK,60,1.2,-3.0\nHS,10000,0.7,-4.0\n"
    bands = autoeq.parse_autoeq_csv(text)
    assert [(b.filter_type, b.frequency, b.q, b.gain, b.enabled) for b in bands] == [
        (autoeq.LOWSHELF, 105.0, 0.7, 6.5, True), (autoeq.PEAK, 60.0, 1.2, -3.0, True), (autoeq.HIGHSHELF, 10000.0, 0.7, -4.0, True)]
    with pytest.raises(ValueError):
        autoeq.parse_autoeq_csv("Filter-Type,Fc,Q,Gain\nLP,100,0.7,0\n")   # src/autoeq_parser.rs:48

    applied = []

    class FakeEngine:
        def eq_update_band(self, *a):
            applied.append(a)

    autoeq.apply_to_engine(FakeEngine(), bands)
    assert applied[0] == (0, autoeq.LOWSHELF, 105.0, 0.7, 6.5, True, 0) and len(applied) == 3


# ------------------------------------------------------------------------------------------------------------
# the same host-side rows in C++ (open-headstage_b200/host/sofa.hpp, autoeq.hpp): SURVEY 8f rows 1 and 4 as specified
# ------------------------------------------------------------------------------------------------------------
import json  # noqa: E402
import subprocess  # noqa: E402
import zlib  # noqa: E402

import open_headstage_b200 as ohs  # noqa: E402


def write_sofa_like(path, m=24, n=32, seed=3):
    """A small seeded HRIR set written by write_sofa_datasets."""
    rng = np.random.default_rng(seed)
    az = np.array([0, 15, 30, 45, 60, 90, 120, 150, 180, 210, 240, 270, 300, 315, 330, 345] + [30, 330, 0, 90, 270, 180, 45, 315], np.float64)[:m]
    el = np.array([0.0] * 16 + [30.0] * 8)[:m]
    pos = np.stack([az, el, np.ones(m)], axis=1)
    ir = (rng.standard_normal((m, 2, n)) * np.exp(-np.arange(n) / 6.0)).astype(np.float32).astype(np.float64)  # f32-representable
    write_sofa_datasets(path, pos, ir, rng)
    return pos.astype(np.float32), ir.astype(np.float32)


def write_sofa_datasets(path, pos, ir, rng):
    """A file with the two datasets the readers look for, stored the way HDF5 stores them in a SimpleFreeFieldHRIR file
    (f64, byte-shuffled, zlib) between unrelated bytes — including stray 0x78 bytes and a decoy zlib stream."""
    pos, ir = np.asarray(pos, np.float64), np.asarray(ir, np.float64)
    shuffle = lambda a: np.ascontiguousarray(a).view(np.uint8).reshape(-1, 8).T.copy().tobytes()  # noqa: E731
    junk = rng.integers(0, 256, 5000, dtype=np.uint8).tobytes()
    decoy = zlib.compress(b"not a dataset" * 40)
    with open(path, "wb") as f:
        f.write(b"\x89HDF\r\n\x1a\n" + junk[:700] + b"\x78\x9c" + junk[700:1500] + decoy + zlib.compress(shuffle(pos), 6) + junk[1500:2600] + b"\x78"
                + zlib.compress(shuffle(ir), 9) + junk[2600:])


def run_tool(*args):
    tool = ohs.build_host_inputs_tool()
    return subprocess.run([tool, *[str(a) for a in args]], capture_output=True, text=True, timeout=120)


def weighted(v):
    v = np.asarray(v, np.float32).ravel().astype(np.float64)
    return float(np.sum(v * ((np.arange(v.size) % 7) + 1)))


def test_cpp_sofa_reader_matches_python_reader(tmp_path):
    path = str(tmp_path / "tiny.sofa")
    pos, ir = write_sofa_like(path)
    h = sofa.load_sofa(path, n_measurements=24, n_taps=32)
    assert np.array_equal(h.ir, ir) and np.array_equal(h.position, pos)
    for (azl, ell, azr, elr) in [(30, 0, 330, 0), (29, 2, 331, -3), (44, 31, 316, 28), (-30, 0, 390, 0)]:
        r = run_tool("sofa", path, 24, 32, azl, ell, azr, elr)
        assert r.returncode == 0, r.stderr
        d = json.loads(r.stdout)
        assert (d["M"], d["N"]) == (24, 32)
        assert d["left_index"] == h.nearest(azl, ell) and d["right_index"] == h.nearest(azr, elr)
        assert abs(d["ir_checksum"] - weighted(ir)) <= 1e-9 * max(1.0, abs(weighted(ir)))       # every tap, bit for bit
        assert abs(d["pos_checksum"] - weighted(pos)) <= 1e-9 * abs(weighted(pos))
        assert abs(d["left_l_checksum"] - weighted(h.get_hrtf_irs(azl, ell)[0])) <= 1e-12 + 1e-9 * abs(d["left_l_checksum"])
        assert abs(d["right_r_checksum"] - weighted(h.get_hrtf_irs(azr, elr)[1])) <= 1e-12 + 1e-9 * abs(d["right_r_checksum"])
        assert d["ui_minus30"] == 30.0 and d["ui_plus30"] == 330.0
    assert run_tool("sofa", path, 25, 32, 0, 0, 0, 0).returncode == 1          # wrong shape: datasets not found
    assert run_tool("sofa", str(tmp_path / "missing.sofa"), 24, 32, 0, 0, 0, 0).returncode == 1


def test_cpp_sofa_reader_reads_the_bundled_file(cipic, cipic_sofa):
    """As test_load_sofa_reads_the_bundled_file_without_hdf5, through the C++ reader: the real file's HDF5 byte layout
    is not exercised."""
    r = run_tool("sofa", cipic_sofa, 1250, 200, 30, 0, 330, 0)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout)
    assert (d["M"], d["N"], d["left_index"], d["right_index"]) == (1250, 200, 308, 908)     # SURVEY.md 8c indices
    assert abs(d["ir_checksum"] - weighted(cipic["ir"])) <= 1e-9 * abs(weighted(cipic["ir"]))
    assert abs(d["left_l_checksum"] - weighted(cipic["ir"][308, 0])) <= 1e-9


def test_cpp_autoeq_parser_matches_python_parser(tmp_path):
    text = "Filter-Type,Fc,Q,Gain\nLS,105,0.7,6.5\nPK,60,1.2,-3.0\nPK,5500,4.0,-5\nHS,10000,0.7,-4.0\n"
    p = tmp_path / "eq.csv"
    p.write_text(text)
    r = run_tool("autoeq", p)
    assert r.returncode == 0, r.stderr
    got = json.loads(r.stdout)
    want = autoeq.parse_autoeq_csv(text)
    f32 = lambda v: float(np.float32(v))  # noqa: E731  (the tool prints f32 values with 9 significant digits: they round-trip)
    assert [(g["enabled"], g["filter_type"], f32(g["frequency"]), f32(g["q"]), f32(g["gain"])) for g in got] == \
        [(b.enabled, b.filter_type, f32(b.frequency), f32(b.q), f32(b.gain)) for b in want]
    # columns by name, in any order
    q = tmp_path / "eq2.csv"
    q.write_text("Gain,Q,Filter-Type,Fc\n6.5,0.7,LS,105\n")
    g = json.loads(run_tool("autoeq", q).stdout)[0]
    assert (g["enabled"], g["filter_type"], f32(g["frequency"]), f32(g["q"]), f32(g["gain"])) == (True, 1, 105.0, f32(0.7), 6.5)
    bad = tmp_path / "bad.csv"
    bad.write_text("Filter-Type,Fc,Q,Gain\nLP,100,0.7,0\n")
    r = run_tool("autoeq", bad)
    assert r.returncode == 1 and "Unsupported filter type: LP" in r.stderr     # src/autoeq_parser.rs:48


@pytest.mark.gpu
def test_cpp_host_inputs_drive_the_real_engine(tmp_path):
    """SOFA file -> C++ reader -> wire_speakers -> four set_ir; AutoEQ CSV -> C++ parser -> update_band_coeffs; then the
    chain on the GPU through the C++ mirror objects — against the oracle given the same indices and bands."""
    from open_headstage_b200 import signals as S
    from oracle import oracle as O

    path = str(tmp_path / "tiny.sofa")
    pos, ir = write_sofa_like(path)
    csv_path = tmp_path / "eq.csv"
    csv_path.write_text("Filter-Type,Fc,Q,Gain\n" + "\n".join(
        "%s,%g,%g,%g" % ({S.LOWSHELF: "LS", S.PEAK: "PK", S.HIGHSHELF: "HS"}[t], fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL) + "\n")
    n = 512 * 6
    out = tmp_path / "out.f32"
    x = S.stream_inputs(1, n, base_seed=2300)[0]
    x.astype("<f4").tofile(tmp_path / "in.f32")
    r = run_tool("render", path, 24, 32, csv_path, tmp_path / "in.f32", out)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout)
    h = sofa.from_arrays(ir, pos, 44100.0)
    assert (d["left_index"], d["right_index"], d["bands"]) == (h.nearest(30.0, 0.0), h.nearest(330.0, 0.0), 10)
    y = np.fromfile(out, "<f4").reshape(2, n)
    irs = [ir[d["left_index"], 0], ir[d["left_index"], 1], ir[d["right_index"], 0], ir[d["right_index"], 1]]
    coeffs = np.stack([O.eq_design(t, 48000.0, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    ref, _ = O.render_batch(x[None], 512, irs, coeffs, [1] * 10, True, 1.0, n_threads=1)
    assert float(np.max(np.abs(y - ref[0]))) <= 1e-5
    assert np.abs(y).max() > 0.05
