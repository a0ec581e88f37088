"""open-headstage_b200 — B200-native (sm_100a) engine for the Open Headstage DSP hot path: 10-band parametric EQ ->
4-path binaural partitioned convolution -> output gain, batched over many independent stereo streams.

The compute path is the hand-written CUDA in csrc/ behind the C ABI of include/ohs.h (libohs_cuda.so, built in-tree
by _build.build_library()).  This package is the thin host side: a ctypes binding, Python mirrors of the
reference's `ConvolutionEngine` / `StereoParametricEQ`, and the seeded synthetic inputs of the BASELINE configs.
"""
from . import autoeq, parallel, signals, sofa  # noqa: F401
from ._build import build_host_inputs_tool, build_host_tests, build_library  # noqa: F401
from .engine import (  # noqa: F401
    ALLPASS, BANDPASS, DITHER_OFF, DITHER_TPDF, FMT_F32, FMT_S16, FMT_S24, HIGHPASS, HIGHSHELF, LOWPASS, LOWSHELF, LSL, LSR, MAX_SHAPE_TAPS, NOTCH, OHS_ALL, PEAK, RSL, RSR, SYMBOLS,
    BandConfig, Comm, ConvolutionEngine, Engine, OhsError, PinnedBuffer, StereoParametricEQ, comm_unique_id, eq_design, load_library,
)
