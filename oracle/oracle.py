"""ctypes binding of the CPU oracle (oracle/ohs_oracle.c).

TEST INFRASTRUCTURE ONLY — see oracle/ohs_oracle.h.  Importable from tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py; never from the product package.

Mirrors the reference's Rust API one to one:
  ConvolutionEngine   -> src/dsp/convolution.rs:68-234
  StereoParametricEQ  -> src/dsp/parametric_eq.rs:125-210
  chain_process       -> src/lib.rs:1169-1207
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libohs_oracle.so")

LSL, LSR, RSL, RSR = 0, 1, 2, 3
PEAK, LOWSHELF, HIGHSHELF, LOWPASS, HIGHPASS, BANDPASS, NOTCH, ALLPASS = range(8)

_f32p = C.POINTER(C.c_float)


def build(force: bool = False) -> str:
    """Compile the oracle with gcc (oracle/Makefile).  Building the checker is not using it."""
    src = os.path.join(_HERE, "ohs_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < max(
        os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "ohs_oracle.h"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "libohs_oracle.so"])
    return _LIB_PATH


def build_native(out_dir: str) -> str:
    """The same source built -march=native into out_dir on the machine that will TIME it — the CPU-baseline legs of
    bench.py only; the parity tests keep the portable build in oracle/.  out_dir is the caller's: the source tree may
    be read-only where the benchmark runs."""
    out = os.path.join(out_dir, "libohs_oracle_native.so")
    src = os.path.join(_HERE, "ohs_oracle.c")
    subprocess.check_call(["gcc", "-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=gnu11", "-shared",
                           "-o", out, src, "-lm", "-lpthread"], cwd=out_dir)
    return out


_lib = None
_lib_path = _LIB_PATH


def use_library(path: str) -> None:
    """Bind this module to another build of the oracle (build_native()), loaded now: if it does not load, the module
    stays bound to the library it had."""
    global _lib, _lib_path
    if path != _lib_path:
        old = _lib, _lib_path
        _lib, _lib_path = None, path
        try:
            lib()
        except Exception:
            _lib, _lib_path = old
            raise


def lib():
    global _lib
    if _lib is None:
        if _lib_path == _LIB_PATH and not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_lib_path)
        L.oracle_conv_new.restype = C.c_void_p
        L.oracle_conv_new.argtypes = [C.c_int]
        L.oracle_conv_free.argtypes = [C.c_void_p]
        L.oracle_conv_set_ir.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_size_t]
        L.oracle_conv_num_partitions.argtypes = [C.c_void_p, C.c_int]
        L.oracle_conv_process_block.argtypes = [C.c_void_p, _f32p, _f32p, _f32p, _f32p, C.c_size_t]
        L.oracle_eq_design.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, _f32p]
        L.oracle_eq_new.restype = C.c_void_p
        L.oracle_eq_new.argtypes = [C.c_int, C.c_float]
        L.oracle_eq_free.argtypes = [C.c_void_p]
        L.oracle_eq_update_band.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]
        L.oracle_eq_set_band_raw.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int]
        L.oracle_eq_process_block.argtypes = [C.c_void_p, _f32p, _f32p, C.c_size_t]
        L.oracle_eq_reset.argtypes = [C.c_void_p]
        L.oracle_eq_frequency_response.argtypes = [C.c_void_p, C.c_float, _f32p, _f32p, C.c_size_t]
        L.oracle_eq_get_state.argtypes = [C.c_void_p, _f32p]
        L.oracle_chain_process.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, _f32p, _f32p, C.c_size_t]
        L.oracle_render_batch.restype = C.c_double
        L.oracle_render_batch.argtypes = [
            C.c_int, C.c_int, C.c_int, C.POINTER(_f32p), C.POINTER(C.c_size_t), C.c_int, _f32p, C.POINTER(C.c_int),
            C.c_int, C.c_float, _f32p, _f32p, C.c_size_t, C.c_size_t,
        ]
        _lib = L
    return _lib


def _p(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_f32p)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def eq_design(filter_type: int, fs: float, fc: float, q: float, gain_db: float) -> np.ndarray:
    """biquad 0.4.2 Coefficients::<f32>::from_params -> [b0, b1, b2, a1, a2] (src/dsp/parametric_eq.rs:105-111)."""
    out = np.zeros(5, np.float32)
    rc = lib().oracle_eq_design(filter_type, fs, fc, q, gain_db, _p(out))
    if rc:
        raise ValueError({-1: "OutsideNyquist", -2: "NegativeQ", -3: "bad filter type"}[rc])
    return out


class ConvolutionEngine:
    """src/dsp/convolution.rs ConvolutionEngine with a run-time block size (reference: BLOCK_SIZE = 512)."""

    def __init__(self, block: int = 512):
        self.block = block
        self._h = lib().oracle_conv_new(block)
        if not self._h:
            raise ValueError("block must be a power of two")

    def __del__(self):
        if getattr(self, "_h", None):
            lib().oracle_conv_free(self._h)
            self._h = None

    def set_ir(self, path: int, ir) -> int:
        ir = _f32(ir)
        return lib().oracle_conv_set_ir(self._h, path, _p(ir) if ir.size else None, ir.size)

    def num_partitions(self, path: int) -> int:
        return lib().oracle_conv_num_partitions(self._h, path)

    def process_block(self, in_l, in_r):
        in_l, in_r = _f32(in_l), _f32(in_r)
        out_l = np.zeros_like(in_l)
        out_r = np.zeros_like(in_r)
        lib().oracle_conv_process_block(self._h, _p(in_l), _p(in_r), _p(out_l), _p(out_r), in_l.size)
        return out_l, out_r


class StereoParametricEQ:
    """src/dsp/parametric_eq.rs StereoParametricEQ."""

    def __init__(self, num_bands: int = 10, fs: float = 48000.0):
        self.num_bands = num_bands
        self._h = lib().oracle_eq_new(num_bands, fs)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().oracle_eq_free(self._h)
            self._h = None

    def update_band_coeffs(self, band: int, fs: float, filter_type: int, fc: float, q: float, gain_db: float, enabled: bool):
        rc = lib().oracle_eq_update_band(self._h, band, fs, filter_type, fc, q, gain_db, int(enabled))
        if rc:
            raise ValueError("from_params would panic in the reference (rc=%d)" % rc)

    def set_band_raw(self, band: int, coeffs, enabled: bool):
        c = _f32(coeffs)
        lib().oracle_eq_set_band_raw(self._h, band, _p(c), int(enabled))

    def process_block(self, left, right):
        """In place in the reference; returns the processed copies here."""
        l, r = _f32(left).copy(), _f32(right).copy()
        lib().oracle_eq_process_block(self._h, _p(l), _p(r), l.size)
        return l, r

    def reset_all_bands_state(self):
        lib().oracle_eq_reset(self._h)

    def calculate_frequency_response(self, fs: float, freqs):
        f = _f32(freqs)
        out = np.zeros_like(f)
        lib().oracle_eq_frequency_response(self._h, fs, _p(f), _p(out), f.size)
        return out

    def state(self) -> np.ndarray:
        s = np.zeros((self.num_bands, 2, 2), np.float32)
        lib().oracle_eq_get_state(self._h, _p(s))
        return s


def chain_process(conv: ConvolutionEngine, eq: StereoParametricEQ | None, eq_enable: bool, bypass: bool, gain: float, left, right):
    """Plugin::process (src/lib.rs:1169-1207) on one host buffer; returns (left, right)."""
    l, r = _f32(left).copy(), _f32(right).copy()
    lib().oracle_chain_process(conv._h, eq._h if eq is not None else None, int(eq_enable), int(bypass), gain, _p(l), _p(r), l.size)
    return l, r


def render_batch(x: np.ndarray, block: int, irs, band_coeffs, band_enabled, eq_enable: bool, gain: float,
                 host_block: int | None = None, n_threads: int = 1):
    """Render x[stream, channel, frame] through one independent reference chain per stream (same IRs/EQ/gain for all).

    Returns (y, seconds) with seconds = slowest thread's time inside its process loops.
    """
    x = _f32(x)
    n_streams, n_ch, n_frames = x.shape
    assert n_ch == 2
    y = np.zeros_like(x)
    irs = [_f32(i) for i in irs]
    ir_ptrs = (_f32p * 4)(*[_p(i) if i.size else None for i in irs])
    ir_len = (C.c_size_t * 4)(*[i.size for i in irs])
    bc = _f32(band_coeffs).reshape(-1, 5)
    be = (C.c_int * bc.shape[0])(*[int(b) for b in band_enabled])
    secs = lib().oracle_render_batch(n_streams, n_threads, block, ir_ptrs, ir_len, bc.shape[0], _p(bc), be, int(eq_enable),
                                     gain, _p(x), _p(y), n_frames, host_block or block)
    return y, secs
