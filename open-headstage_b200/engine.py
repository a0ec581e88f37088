"""ctypes binding of include/ohs.h plus Python mirrors of the reference's two DSP objects.

`Engine` is the batched handle (n_streams chains).  `ConvolutionEngine` and `StereoParametricEQ` keep the reference's
method names and argument meaning (src/dsp/convolution.rs:87,111,141; src/dsp/parametric_eq.rs:132,144,166,181) over
a one-stream engine, so parity tests read like the reference's own unit tests.  Everything computes on the GPU through
libohs_cuda.so; if the library or a CUDA device is missing these raise — there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import _build

OHS_ALL = -1
ABI_VERSION = 2   # OHS_ABI_VERSION of include/ohs.h this binding was written against
LSL, LSR, RSL, RSR = 0, 1, 2, 3
PEAK, LOWSHELF, HIGHSHELF, LOWPASS, HIGHPASS, BANDPASS, NOTCH, ALLPASS = range(8)
FMT_F32, FMT_S16, FMT_S24 = 0, 1, 2   # ohs_sample_format
DITHER_OFF, DITHER_TPDF = 0, 1        # OHS_DITHER_*
MAX_SHAPE_TAPS = 9                    # OHS_MAX_SHAPE_TAPS

_f32p = C.POINTER(C.c_float)


class OhsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("ohs error %d: %s" % (code, msg))
        self.code = code


class _Config(C.Structure):
    _fields_ = [("n_streams", C.c_int32), ("block", C.c_int32), ("max_taps", C.c_int32), ("n_bands", C.c_int32),
                ("n_hrir_sets", C.c_int32), ("n_eq_sets", C.c_int32), ("device", C.c_int32), ("sample_rate", C.c_float)]


# every symbol include/ohs.h declares: (name, restype, argtypes)
_VP = C.c_void_p
SYMBOLS = [
    ("ohs_create", C.c_int, [C.POINTER(_Config), C.POINTER(_VP)]),
    ("ohs_destroy", C.c_int, [_VP]),
    ("ohs_abi_version", C.c_int, []),
    ("ohs_last_error", C.c_char_p, []),
    ("ohs_set_ir", C.c_int, [_VP, C.c_int, C.c_int, _f32p, C.c_size_t]),
    ("ohs_num_partitions", C.c_int, [_VP, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("ohs_bind_stream_hrir", C.c_int, [_VP, C.c_int, C.c_int]),
    ("ohs_move_stream_hrir", C.c_int, [_VP, C.c_int, C.c_int]),
    ("ohs_commit_filters", C.c_int, [_VP]),
    ("ohs_filter_table", C.c_int, [_VP, C.POINTER(_VP), C.POINTER(C.c_size_t)]),
    ("ohs_mark_filters_external", C.c_int, [_VP, C.c_int, C.c_int]),
    ("ohs_eq_design", C.c_int, [C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, _f32p]),
    ("ohs_eq_update_band", C.c_int, [_VP, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]),
    ("ohs_eq_set_band", C.c_int, [_VP, C.c_int, C.c_int, _f32p, C.c_int]),
    ("ohs_bind_stream_eq", C.c_int, [_VP, C.c_int, C.c_int]),
    ("ohs_eq_reset", C.c_int, [_VP]),
    ("ohs_eq_frequency_response", C.c_int, [_VP, C.c_int, C.c_float, _f32p, _f32p, C.c_size_t]),
    ("ohs_set_eq_enable", C.c_int, [_VP, C.c_int]),
    ("ohs_set_conv_enable", C.c_int, [_VP, C.c_int]),
    ("ohs_set_bypass", C.c_int, [_VP, C.c_int]),
    ("ohs_set_gain", C.c_int, [_VP, C.c_int, C.c_float]),
    ("ohs_conv_reset", C.c_int, [_VP]),
    ("ohs_set_time_batch", C.c_int, [_VP, C.c_int]),
    ("ohs_streams_per_cta", C.c_int, [_VP, C.POINTER(C.c_int)]),
    ("ohs_prepare", C.c_int, [_VP, C.c_size_t, C.c_int]),
    ("ohs_debug_trace", C.c_int, [_VP, _VP]),
    ("ohs_process_device", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_size_t]),
    ("ohs_process_device_scheduled", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_size_t, _VP, C.c_size_t]),
    ("ohs_process", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_size_t]),
    ("ohs_process_fifo", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_size_t]),
    ("ohs_process_pcm", C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_size_t, C.c_size_t]),
    ("ohs_process_device_pcm", C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_size_t, C.c_size_t]),
    ("ohs_set_dither", C.c_int, [_VP, C.c_int, C.c_uint64, _f32p, C.c_int]),
    ("ohs_sync", C.c_int, [_VP]),
    ("ohs_cuda_stream", C.c_int, [_VP, C.POINTER(_VP)]),
    ("ohs_launch_count", C.c_int, [_VP, C.POINTER(C.c_uint64)]),
    ("ohs_enable_timing", C.c_int, [_VP, C.c_int]),
    ("ohs_last_kernel_ms", C.c_int, [_VP, C.POINTER(C.c_float)]),
    ("ohs_mix_device", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_size_t, C.c_size_t]),
    ("ohs_set_groups", C.c_int, [_VP, _VP, C.c_int]),
    ("ohs_num_groups", C.c_int, [_VP, C.POINTER(C.c_int)]),
    ("ohs_process_grouped", C.c_int, [_VP, _VP, C.c_int, _VP, C.c_size_t, C.c_size_t, C.c_size_t]),
    ("ohs_process_grouped_pcm", C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t]),
    ("ohs_mix_device_pcm", C.c_int, [_VP, _VP, _VP, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t]),
    ("ohs_comm_unique_id", C.c_int, [_VP]),
    ("ohs_comm_create", C.c_int, [C.POINTER(_VP), C.c_int, C.c_int, C.c_int, _VP]),
    ("ohs_comm_destroy", C.c_int, [_VP]),
    ("ohs_broadcast_hrir", C.c_int, [_VP, _VP, C.c_int]),
    ("ohs_reduce_bus", C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_int]),
    ("ohs_host_alloc", C.c_int, [C.POINTER(_VP), C.c_size_t]),
    ("ohs_host_free", C.c_int, [_VP]),
    ("ohs_state_bytes", C.c_int, [_VP, C.POINTER(C.c_size_t)]),
    ("ohs_state_export", C.c_int, [_VP, _VP, C.c_size_t]),
    ("ohs_state_import", C.c_int, [_VP, _VP, C.c_size_t]),
]

_lib = None


def load_library(build: bool = True):
    """dlopen libohs_cuda.so (building it in-tree first if it is missing or stale and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build and _build.is_stale():
        try:
            _build.build_library()
        except Exception as e:
            if not os.path.exists(path):
                raise
            import warnings

            warnings.warn("libohs_cuda.so is older than its sources and could not be rebuilt (%s); loading the stale library" % e,
                          RuntimeWarning, stacklevel=2)
    if not os.path.exists(path):
        raise OhsError(-3, "libohs_cuda.so is missing and could not be built; there is no CPU fallback")
    L = C.CDLL(path)
    L.ohs_abi_version.restype = C.c_int
    got = L.ohs_abi_version()
    if got != ABI_VERSION:
        raise OhsError(-1, "libohs_cuda.so has ABI version %d, this binding expects %d (rebuild the library)" % (got, ABI_VERSION))
    for name, res, args in SYMBOLS:
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise OhsError(rc, load_library().ohs_last_error().decode())


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _pcm_input(x, n_streams: int):
    """The input of process_pcm / process_grouped: (contiguous array, ohs_sample_format, frames), the format from the dtype."""
    x = np.asarray(x)
    if x.ndim != 3 or x.shape[0] != n_streams or x.shape[1] != 2:
        raise ValueError("x must be [n_streams, 2, frames], got %s" % (x.shape,))
    if x.dtype == np.int16:
        fmt, n = FMT_S16, x.shape[2]
    elif x.dtype == np.float32:
        fmt, n = FMT_F32, x.shape[2]
    elif x.dtype == np.uint8 and x.shape[2] % 3 == 0:
        fmt, n = FMT_S24, x.shape[2] // 3
    else:
        raise ValueError("process_pcm takes int16, float32 or packed 24-bit uint8 [S, 2, 3n] input, got %s %s" % (x.dtype, x.shape))
    return np.ascontiguousarray(x), fmt, n


def _pcm_rows(shape, fmt: int):
    """The (shape, dtype) of PCM rows [*shape, n] in `fmt`: int16 [.., n] (S16), packed uint8 [.., 3n] (S24), float32 (F32)."""
    if fmt == FMT_F32:
        return tuple(shape), np.dtype(np.float32)
    if fmt == FMT_S16:
        return tuple(shape), np.dtype(np.int16)
    if fmt == FMT_S24:
        return tuple(shape[:-1]) + (3 * shape[-1],), np.dtype(np.uint8)
    raise ValueError("unknown sample format %r" % (fmt,))


def eq_design(filter_type: int, fs: float, fc: float, q: float, gain_db: float) -> np.ndarray:
    """Host-side RBJ design identical to biquad 0.4.2 from_params (src/dsp/parametric_eq.rs:105-111)."""
    out = np.zeros(5, np.float32)
    _check(load_library().ohs_eq_design(filter_type, fs, fc, q, gain_db, out.ctypes.data_as(_f32p)))
    return out


COMM_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the C ABI (one rank calls it and ships the 128 bytes to the others)."""
    buf = C.create_string_buffer(COMM_ID_BYTES)
    _check(load_library().ohs_comm_unique_id(buf))
    return buf.raw


class Comm:
    """ohs_comm: an NCCL communicator owned by the C ABI library (ohs_broadcast_hrir / ohs_reduce_bus)."""

    def __init__(self, world: int, rank: int, device: int, unique_id: bytes):
        assert len(unique_id) == COMM_ID_BYTES
        self._L = load_library()
        self.world, self.rank, self.device = world, rank, device
        self._c = _VP()
        _check(self._L.ohs_comm_create(C.byref(self._c), world, rank, device, unique_id))

    def close(self):
        if getattr(self, "_c", None):
            self._L.ohs_comm_destroy(self._c)
            self._c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PinnedBuffer:
    """cudaHostAlloc'd array (ohs_host_alloc) viewed as numpy; float32 unless another dtype is given."""

    def __init__(self, shape, dtype=np.float32):
        self.shape = tuple(int(s) for s in shape)
        dtype = np.dtype(dtype)
        n = int(np.prod(self.shape))
        self._ptr = _VP()
        _check(load_library().ohs_host_alloc(C.byref(self._ptr), n * dtype.itemsize))
        raw = np.ctypeslib.as_array(C.cast(self._ptr, C.POINTER(C.c_uint8)), shape=(n * dtype.itemsize,))
        self.array = raw.view(dtype).reshape(self.shape)

    def free(self):
        if self._ptr:
            self.array = None
            load_library().ohs_host_free(self._ptr)
            self._ptr = _VP()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One ohs_engine handle: n_streams independent EQ -> 4-path convolution -> gain chains resident on one GPU."""

    def __init__(self, n_streams: int, block: int, max_taps: int, n_bands: int = 10, n_hrir_sets: int = 1,
                 n_eq_sets: int = 1, device: int = 0, sample_rate: float = 48000.0):
        self._L = load_library()
        self.n_streams, self.block, self.max_taps, self.n_bands = n_streams, block, max_taps, n_bands
        self.n_hrir_sets, self.n_eq_sets, self.device = n_hrir_sets, n_eq_sets, device
        self.sample_rate = sample_rate
        cfg = _Config(n_streams, block, max_taps, n_bands, n_hrir_sets, n_eq_sets, device, sample_rate)
        self._h = _VP()
        _check(self._L.ohs_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            self._L.ohs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- HRIR
    def set_ir(self, path: int, ir, hrir_set: int = 0):
        ir = _f32(ir).ravel()
        _check(self._L.ohs_set_ir(self._h, hrir_set, path, ir.ctypes.data_as(_f32p) if ir.size else None, ir.size))

    def set_hrir_set(self, irs, hrir_set: int = 0):
        for p in range(4):
            self.set_ir(p, irs[p], hrir_set)

    def num_partitions(self, path: int, hrir_set: int = 0) -> int:
        out = C.c_int()
        _check(self._L.ohs_num_partitions(self._h, hrir_set, path, C.byref(out)))
        return out.value

    def bind_stream_hrir(self, stream: int, hrir_set: int):
        _check(self._L.ohs_bind_stream_hrir(self._h, stream, hrir_set))

    def move_stream_hrir(self, stream: int, hrir_set: int):
        """Moving source: the stream's next convolved block crossfades to `hrir_set`, history kept (ohs.h)."""
        _check(self._L.ohs_move_stream_hrir(self._h, stream, hrir_set))

    def commit_filters(self):
        _check(self._L.ohs_commit_filters(self._h))

    def filter_table(self):
        p, n = _VP(), C.c_size_t()
        _check(self._L.ohs_filter_table(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def mark_filters_external(self, hrir_set: int, partitions: int):
        _check(self._L.ohs_mark_filters_external(self._h, hrir_set, partitions))

    def broadcast_hrir(self, comm: "Comm", root: int = 0):
        """One HRIR spectra table for the whole job: rank `root` has called set_ir, everybody receives (C ABI, NCCL)."""
        _check(self._L.ohs_broadcast_hrir(self._h, comm._c, root))

    def reduce_bus(self, comm: "Comm", d_bus: int, n_floats: int, root: int = 0):
        """In-place NCCL sum of the per-GPU buses onto `root`, on the engine's stream (config 4)."""
        _check(self._L.ohs_reduce_bus(self._h, comm._c, d_bus, n_floats, root))

    # ---- EQ
    def eq_update_band(self, band: int, filter_type: int, fc: float, q: float, gain_db: float, enabled: bool = True, eq_set: int = 0):
        _check(self._L.ohs_eq_update_band(self._h, eq_set, band, filter_type, fc, q, gain_db, int(enabled)))

    def eq_set_band(self, band: int, coeffs, enabled: bool = True, eq_set: int = 0):
        c = _f32(coeffs)
        _check(self._L.ohs_eq_set_band(self._h, eq_set, band, c.ctypes.data_as(_f32p), int(enabled)))

    def eq_set_preset(self, preset, eq_set: int = 0, enabled: bool = True):
        for i, (t, fc, q, g) in enumerate(preset):
            self.eq_update_band(i, t, fc, q, g, enabled, eq_set)

    def bind_stream_eq(self, stream: int, eq_set: int):
        _check(self._L.ohs_bind_stream_eq(self._h, stream, eq_set))

    def eq_reset(self):
        _check(self._L.ohs_eq_reset(self._h))

    def eq_frequency_response(self, freqs, eq_set: int = 0, sample_rate: float = 0.0) -> np.ndarray:
        f = _f32(freqs)
        out = np.zeros_like(f)
        _check(self._L.ohs_eq_frequency_response(self._h, eq_set, sample_rate, f.ctypes.data_as(_f32p), out.ctypes.data_as(_f32p), f.size))
        return out

    # ---- switches
    def set_eq_enable(self, on: bool):
        _check(self._L.ohs_set_eq_enable(self._h, int(on)))

    def set_conv_enable(self, on: bool):
        _check(self._L.ohs_set_conv_enable(self._h, int(on)))

    def set_bypass(self, on: bool):
        _check(self._L.ohs_set_bypass(self._h, int(on)))

    def set_gain(self, gain: float, stream: int = OHS_ALL):
        _check(self._L.ohs_set_gain(self._h, stream, gain))

    def conv_reset(self):
        _check(self._L.ohs_conv_reset(self._h))

    def set_time_batch(self, on: bool):
        _check(self._L.ohs_set_time_batch(self._h, int(on)))

    def streams_per_cta(self) -> int:
        out = C.c_int()
        _check(self._L.ohs_streams_per_cta(self._h, C.byref(out)))
        return out.value

    def prepare(self, n_frames: int, host_io: bool = False):
        """Upload pending set-up and allocate scratch/staging for calls of n_frames, outside any timed region."""
        _check(self._L.ohs_prepare(self._h, n_frames, int(host_io)))

    def debug_trace(self, d_stamps: int):
        _check(self._L.ohs_debug_trace(self._h, d_stamps))

    # ---- processing
    def process(self, x, out=None) -> np.ndarray:
        """Host flavour.  x[stream, channel, frame] float32; returns the rendered array (or fills `out`)."""
        x = _f32(x)
        assert x.ndim == 3 and x.shape[0] == self.n_streams and x.shape[1] == 2, x.shape
        if out is None:
            y = np.empty_like(x)
        else:
            y = out
            if not (isinstance(y, np.ndarray) and y.dtype == np.float32 and y.shape == x.shape and y.flags["C_CONTIGUOUS"]
                    and y.flags["WRITEABLE"]):
                raise ValueError("out must be a writeable C-contiguous float32 array of shape %s" % (x.shape,))
        _check(self._L.ohs_process(self._h, x.ctypes.data, y.ctypes.data, x.shape[2], x.shape[2]))
        return y

    def process_pcm(self, x, out_format: int, out=None) -> np.ndarray:
        """Host flavour with integer PCM (ohs_process_pcm).  The input format follows the dtype: int16 [S, 2, n] is S16,
        float32 [S, 2, n] is F32, uint8 [S, 2, 3n] is packed S24 (signals.pack_s24).  Returns int16 [S, 2, n] for
        FMT_S16, uint8 [S, 2, 3n] for FMT_S24, float32 [S, 2, n] for FMT_F32 (or fills `out`, e.g. a PinnedBuffer's array)."""
        x, fmt, n = _pcm_input(x, self.n_streams)
        want = _pcm_rows((self.n_streams, 2, n), out_format)
        if out is None:
            y = np.empty(*want)
        else:
            y = out
            if not (isinstance(y, np.ndarray) and (y.shape, y.dtype) == want and y.flags["C_CONTIGUOUS"] and y.flags["WRITEABLE"]):
                raise ValueError("out must be a writeable C-contiguous %s array of shape %s" % (want[1], want[0]))
        _check(self._L.ohs_process_pcm(self._h, x.ctypes.data, fmt, y.ctypes.data, out_format, n, n))
        return y

    def set_groups(self, first):
        """Listener buses (ohs_set_groups): group g holds streams first[g] .. first[g+1]-1, first[0] = 0, strictly increasing,
        first[-1] = n_streams.  Used by process_grouped and mix_device."""
        f = np.ascontiguousarray(np.asarray(first, dtype=np.int32).ravel())
        if f.size < 2:
            raise ValueError("first needs n_groups + 1 >= 2 entries, got %d" % f.size)
        _check(self._L.ohs_set_groups(self._h, f.ctypes.data, f.size - 1))

    @property
    def n_groups(self) -> int:
        """The group count in force, read from the library (ohs_num_groups)."""
        n = C.c_int()
        _check(self._L.ohs_num_groups(self._h, C.byref(n)))
        return n.value

    def process_grouped(self, x, out=None, bus_stride: int | None = None, bus_format: int = FMT_F32) -> np.ndarray:
        """Host flavour returning only the group buses (ohs_process_grouped_pcm): renders what process_pcm(x, FMT_F32) renders
        and returns the buses [n_groups, 2, n] in `bus_format`: float32 (FMT_F32), int16 (FMT_S16) or packed uint8
        [n_groups, 2, 3n] (FMT_S24), the integer ones dithered as set_dither says (the input format follows the dtype, as in
        process_pcm).  `out`: a writeable C-contiguous array of that dtype and shape [n_groups, 2, bus_stride] (3 * bus_stride
        bytes per row for S24; e.g. a PinnedBuffer's); the first n frames of each of its rows are written and returned as a
        view."""
        x, fmt, n = _pcm_input(x, self.n_streams)
        _pcm_rows((n,), bus_format)   # an unknown format is refused before the library is asked for the group count
        bs = n if bus_stride is None else int(bus_stride)
        want = _pcm_rows((self.n_groups, 2, bs), bus_format)
        if out is None:
            y = np.empty(*want)
        else:
            y = out
            if not (isinstance(y, np.ndarray) and (y.shape, y.dtype) == want and y.flags["C_CONTIGUOUS"] and y.flags["WRITEABLE"]):
                raise ValueError("out must be a writeable C-contiguous %s array of shape %s" % (want[1], want[0]))
        _check(self._L.ohs_process_grouped_pcm(self._h, x.ctypes.data, fmt, y.ctypes.data, bus_format, n, n, bs))
        return y[:, :, :_pcm_rows((n,), bus_format)[0][0]]

    def process_device_pcm(self, d_in: int, in_format: int, d_out: int, out_format: int, n_frames: int, row_stride: int | None = None):
        """Device flavour of process_pcm on raw device pointers; row_stride counts frames for both buffers."""
        _check(self._L.ohs_process_device_pcm(self._h, d_in, in_format, d_out, out_format, n_frames,
                                              n_frames if row_stride is None else row_stride))

    def set_dither(self, mode: int, seed: int = 0, shape=()):
        """Dither of integer PCM output (ohs_set_dither): DITHER_OFF or DITHER_TPDF, noise-shaped by the error-feedback taps
        `shape` = (h_1, ..., h_M), M <= MAX_SHAPE_TAPS.  Resets the dither position and error history."""
        h = _f32(shape).ravel()
        _check(self._L.ohs_set_dither(self._h, mode, seed, h.ctypes.data_as(_f32p) if h.size else None, h.size))

    def process_fifo(self, x) -> np.ndarray:
        x = _f32(x)
        assert x.ndim == 3 and x.shape[0] == self.n_streams and x.shape[1] == 2, x.shape
        y = np.empty_like(x)
        _check(self._L.ohs_process_fifo(self._h, x.ctypes.data, y.ctypes.data, x.shape[2], x.shape[2]))
        return y

    def process_device(self, d_in: int, d_out: int, n_frames: int, row_stride: int | None = None, hrir_schedule=None):
        """Device flavour: raw device pointers (e.g. torch.Tensor.data_ptr()); enqueues on the engine's stream.
        hrir_schedule: optional int32 array [n_streams, n_blocks >= n_frames / block], the HRIR set of every block of
        every stream (moving sources, ohs_process_device_scheduled); afterwards each stream is bound to its last column."""
        rs = n_frames if row_stride is None else row_stride
        if hrir_schedule is None:
            _check(self._L.ohs_process_device(self._h, d_in, d_out, n_frames, rs))
            return
        sched = np.ascontiguousarray(hrir_schedule, dtype=np.int32)
        if sched.ndim != 2 or sched.shape[0] != self.n_streams:
            raise ValueError("hrir_schedule must be [n_streams, n_blocks], got %s" % (sched.shape,))
        _check(self._L.ohs_process_device_scheduled(self._h, d_in, d_out, n_frames, rs, sched.ctypes.data, sched.shape[1]))

    def mix_device(self, d_in: int, d_bus: int, n_frames: int, row_stride: int | None = None, bus_stride: int | None = None,
                   bus_format: int = FMT_F32):
        """Sum the rendered streams of each group (set_groups; by default one group of every stream, the config 4 object
        mixdown) into its stereo bus: 2 * n_groups rows [n_groups][2][bus_stride] at d_bus, in `bus_format`
        (ohs_mix_device_pcm: an integer bus is dithered as set_dither says, in the same launch)."""
        _check(self._L.ohs_mix_device_pcm(self._h, d_in, d_bus, bus_format, n_frames, n_frames if row_stride is None else row_stride,
                                          n_frames if bus_stride is None else bus_stride))

    def sync(self):
        _check(self._L.ohs_sync(self._h))

    def cuda_stream(self) -> int:
        s = _VP()
        _check(self._L.ohs_cuda_stream(self._h, C.byref(s)))
        return s.value or 0

    def launch_count(self) -> int:
        n = C.c_uint64()
        _check(self._L.ohs_launch_count(self._h, C.byref(n)))
        return n.value

    def enable_timing(self, on: bool = True):
        _check(self._L.ohs_enable_timing(self._h, int(on)))

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        _check(self._L.ohs_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    # ---- state
    def state_export(self) -> bytes:
        n = C.c_size_t()
        _check(self._L.ohs_state_bytes(self._h, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        _check(self._L.ohs_state_export(self._h, buf, n.value))
        return buf.raw

    def state_import(self, blob: bytes):
        _check(self._L.ohs_state_import(self._h, blob, len(blob)))


# ---------------------------------------------------------------------------------------------------------------
# Mirrors of the reference's objects (one stereo stream each)
# ---------------------------------------------------------------------------------------------------------------
@dataclass
class BandConfig:
    """src/dsp/parametric_eq.rs:37-44"""
    filter_type: int
    center_freq: float
    q: float
    gain_db: float
    enabled: bool


class ConvolutionEngine:
    """src/dsp/convolution.rs ConvolutionEngine::{new, set_ir, process_block}; block = BLOCK_SIZE (:22, 512 there)."""

    def __init__(self, block: int = 512, max_taps: int = 4096, device: int = 0):
        self._e = Engine(1, block, max_taps, n_bands=0, device=device)
        self.block = block

    def set_ir(self, path: int, ir_data):
        self._e.set_ir(path, ir_data)

    def num_partitions(self, path: int) -> int:
        return self._e.num_partitions(path)

    def process_block(self, input_left, input_right):
        """Any host-block length, with the reference's FIFO/zero-fill semantics (:141-182)."""
        x = np.stack([_f32(input_left), _f32(input_right)])[None]
        y = self._e.process_fifo(x)
        return y[0, 0], y[0, 1]


class StereoParametricEQ:
    """src/dsp/parametric_eq.rs StereoParametricEQ::{new, update_band_coeffs, process_block, reset_all_bands_state}."""

    def __init__(self, num_bands: int, initial_sample_rate: float, device: int = 0):
        self._e = Engine(1, 256, 1, n_bands=num_bands, device=device, sample_rate=initial_sample_rate)
        self._e.set_conv_enable(False)
        self._e.set_eq_enable(True)
        self.num_bands = num_bands

    def update_band_coeffs(self, band_idx: int, sample_rate: float, config: BandConfig):
        c = eq_design(config.filter_type, sample_rate, config.center_freq, config.q, config.gain_db)
        self._e.eq_set_band(band_idx, c, config.enabled)

    def process_block(self, input_left, input_right):
        """In place in the reference (:166); returns the filtered copies."""
        x = np.stack([_f32(input_left), _f32(input_right)])[None]
        y = self._e.process(x)
        return y[0, 0], y[0, 1]

    def reset_all_bands_state(self):
        self._e.eq_reset()

    def calculate_frequency_response(self, sample_rate: float, frequencies):
        return self._e.eq_frequency_response(frequencies, sample_rate=sample_rate)
