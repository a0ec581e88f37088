#!/usr/bin/env python
"""bench.py — stereo stream-seconds rendered per second on B200 (BASELINE.json metric).

Headline workload (N = 1 and, weak-scaled, every rank at N > 1): BASELINE config 2 — 1024 independent stereo streams,
48 kHz, one shared 256-tap 4-path HRIR set, engine block 256, 10-band parametric EQ ("typical" preset), gain 0.5.
A step is one pass of the fused EQ -> 4-path convolution -> gain kernel over one batch: every stream advances by
FRAMES_PER_STEP frames (192 engine blocks = 1.024 s of audio) in ONE kernel launch.

  value        device-resident throughput: inputs already in HBM, CUDA events on the engine's stream, max over ranks
  sustained    the same launch repeated back to back for >= 3 s with clocks and power sampled throughout
  per_block_api  K = 1: one launch per engine block (the reference's calling pattern, SURVEY 8d's judged figure)
  e2e          the same work through the host-pointer C-ABI call (ohs_process) with pinned HOST buffers: H2D and D2H
               copies inside the timed region; copy_ceiling = the same bytes as bare concurrent copies on every rank
  roofline     algorithmic HBM bytes of one launch (SURVEY.md 8d formula) / average launch duration, against the
               measured copy bandwidth in MEASURED_PEAKS.json
  configs      BASELINE configs 3, 4 and 5 at one GPU's share of their full extent: throughput, roofline by the
               config's own formula, and max abs error of >= 8 sampled streams against the CPU oracle (config 4: the
               reduced bus against an f64 evaluation)
  cpu_baseline / --impl reference
               the CPU restatement of the reference (oracle/, the reference itself is Rust and cannot be built here),
               one stream per thread over all host cores, on the stated workload
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import _bootstrap  # noqa: E402

METRIC = "stereo stream-seconds rendered/sec"
UNIT = "stream-s/s"
N_STREAMS = 1024
BLOCK = 256
TAPS = 256
FS = 48000.0
BLOCKS_PER_STEP = int(os.environ.get("OHS_BENCH_BLOCKS", "192"))  # override only to keep ncu replays short
FRAMES_PER_STEP = BLOCK * BLOCKS_PER_STEP  # 49152 frames = 1.024 s
GAIN = 0.5
UNIQUE_STREAMS = 128  # distinct pink-noise streams generated on the host, tiled to N_STREAMS
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
FP32_FMA_TFLOPS_MEASURED = 70.88  # tools/microbench/fp32_pipes.cu on this pool's B200 (profiles/r01_fp32_pipes_microbench.jsonl)
SUSTAINED_SECONDS = float(os.environ.get("OHS_BENCH_SUSTAINED_S", "3.0"))
DUMP_STREAMS = min(128, 64_000_000 // (2 * FRAMES_PER_STEP * 4))  # --dump-outputs: 50 MB at the default step, never above 64 MB


def algorithmic_bytes_per_stream(k_blocks: int, block: int = BLOCK, parts: int = 1) -> int:
    """SURVEY.md §8d / BASELINE.md §3: bytes(K) for one stream through K blocks of one launch."""
    s = 8 * (block + 1)
    return 16 * block * k_blocks + 2 * s * ((parts - 1) + min(k_blocks, parts - 1)) + 16 * block + 320


def algorithmic_flops_per_stream_block(block: int = BLOCK, parts: int = 1) -> float:
    n = 2 * block
    return 4 * (2.5 * n * np.log2(n)) + 4 * parts * (block + 1) * 8 + 4 * block + 2 * block + 2 * 10 * 9 * block


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the render kernel, per launch, from the committed ncu capture of
    this same command (profiles/ncu_render_summary.json); None until a capture exists."""
    p = os.path.join(ROOT, "profiles", "ncu_render_summary.json")
    try:
        d = json.load(open(p))
        if d.get("frames_per_step") == FRAMES_PER_STEP and d.get("n_streams") == N_STREAMS:
            return float(d["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 100):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", str(period_ms)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for i, nme in enumerate(names):
                    if r[3 + i].strip().lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


def workload_arrays(signals, eq_design):
    """The headline workload's HRIR set and EQ coefficients; eq_design is the product's or the oracle's design function
    (bit-identical, tests/test_abi.py) so that each arm maps only its own library."""
    h = signals.synthetic_hrir_set(TAPS, 40.0)
    coeffs = np.stack([eq_design(t, FS, fc, q, g) for (t, fc, q, g) in signals.EQ_PRESET_TYPICAL])
    return h, coeffs


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": "cfg2: %d independent stereo streams per GPU, 48 kHz, 256-tap HRIRs (4 paths), block 256, 10-band PEQ, gain" % N_STREAMS,
        "n_streams_per_gpu": N_STREAMS, "n_streams_total": N_STREAMS * n_gpus, "block": BLOCK, "taps": TAPS, "partitions": 1,
        "sample_rate": FS, "eq_bands": 10, "frames_per_step": FRAMES_PER_STEP, "blocks_per_launch": BLOCKS_PER_STEP,
        "audio_seconds_per_step_per_stream": FRAMES_PER_STEP / FS,
        "l2": "inputs larger than L2: %.0f MB in + %.0f MB out per step per GPU" % ((N_STREAMS * 2 * FRAMES_PER_STEP * 4 / 1e6,) * 2),
        "parallelism": "streams sharded across GPUs, no data-path collective (NCCL only broadcasts the HRIR spectra at set-up)",
    }


# --------------------------------------------------------------------------------------------------------------
# reference arm: the CPU restatement of the reference's algorithm, all host threads.  Maps ONLY oracle/ (the product
# library is never loaded here: signals is pure numpy, the EQ design is the oracle's own).
# --------------------------------------------------------------------------------------------------------------
def native_oracle():
    """The oracle built -march=native on the box it is timed on, in a temporary directory that is gone once the library
    is mapped (the benchmark writes nothing into the tree); falls back to the portable build of oracle/."""
    from oracle import oracle as O

    try:
        with tempfile.TemporaryDirectory(prefix="ohs_oracle_") as d:
            O.use_library(O.build_native(d))  # loaded before the directory goes: the mapping outlives the file
        return O, "gcc -O3 -march=native -ffp-contract=off (built on this box)"
    except Exception as e:  # no compiler on the box: the portable library
        return O, "portable x86-64-v3 build (native build failed: %s)" % (str(e)[:80],)


def pocketfft_conv_bound(signals, cores: int, n_streams: int, n_blocks: int):
    """Sanity bound (SURVEY 8d): the reference's transform work per block — four forward and four inverse complex
    N-point FFTs and the full-spectrum products — on scipy's pocketfft in complex64, batched over streams on all
    cores.  Convolution only (no EQ, no FIFO); a bound on what an optimised CPU FFT would make of that stage."""
    try:
        import scipy.fft as sfft
    except Exception:
        return None
    n = 2 * BLOCK
    h = signals.synthetic_hrir_set(TAPS, 40.0)
    hf = sfft.fft(np.pad(h, ((0, 0), (0, n - TAPS))).astype(np.complex64), axis=1)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n_streams, 2, n_blocks, BLOCK)).astype(np.float32)
    t0 = time.perf_counter()
    pad = np.zeros((n_streams, 4, n_blocks, n), np.complex64)
    pad[:, 0, :, :BLOCK] = x[:, 0]; pad[:, 1, :, :BLOCK] = x[:, 0]; pad[:, 2, :, :BLOCK] = x[:, 1]; pad[:, 3, :, :BLOCK] = x[:, 1]
    spec = sfft.fft(pad, axis=3, workers=cores)
    spec *= hf[None, :, None, :]
    y = sfft.ifft(spec, axis=3, workers=cores)
    out = y.real[..., :BLOCK]
    out[:, :, 1:] += y.real[:, :, :-1, BLOCK:]
    dt = time.perf_counter() - t0
    return {"value": n_streams * n_blocks * BLOCK / FS / dt, "unit": UNIT, "what": "convolution stage only: 4+4 complex %d-point FFTs and "
            "full-spectrum products per block in scipy pocketfft complex64, %d workers (no EQ)" % (n, cores)}


def cpu_reference_run(signals, steps: int, warmup: int, n_streams: int, seconds_per_stream: float):
    O, build = native_oracle()
    cores = os.cpu_count() or 1
    h, coeffs = workload_arrays(signals, O.eq_design)
    n = int(round(seconds_per_stream * FS)) // BLOCK * BLOCK
    x = signals.stream_inputs(n_streams, n, unique=min(n_streams, 16))
    for _ in range(max(0, warmup)):
        O.render_batch(x[: min(n_streams, 4 * cores)], BLOCK, h, coeffs, [1] * 10, True, GAIN, n_threads=cores)
    dt = 0.0
    for _ in range(steps):
        # seconds = slowest thread's time inside its per-stream process loops (engine construction, set_ir and the
        # input copy are outside, as they would be for a long-running reference instance)
        dt += O.render_batch(x, BLOCK, h, coeffs, [1] * 10, True, GAIN, n_threads=cores)[1]
    value = steps * n_streams * (n / FS) / dt
    sample = "%d streams x %.3f s of audio per step, %d step(s), one stream per thread at a time on %d threads; restated CPU baseline (not rustfft), %s" % (
        n_streams, n / FS, steps, cores, build)
    return value, cores, sample, dt / steps * 1e3


def run_reference(args, signals):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step is the stated config: 1024 streams x 1.024 s of audio (about 0.4 s of CPU work per step on 16 cores)
    steps = args.steps
    value, cores, sample, ms = cpu_reference_run(signals, steps, min(args.warmup, 1), N_STREAMS, FRAMES_PER_STEP / FS)
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    bound = pocketfft_conv_bound(signals, cores, 256, 48)
    if bound:
        cpu["pocketfft_conv_only"] = bound
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (seeded pink noise, synthetic 256-tap HRIR set)", "config": workload_config(1),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json((line))


# --------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, pkg):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.pkg, self.args = torch, dist, pkg, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.comm = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            # the data path's two collectives (spectra broadcast, config-4 bus reduce) go through the C ABI's own NCCL
            # communicator; torch.distributed is plumbing (rendezvous, barriers, max-over-ranks)
            self.comm = pkg.parallel.create_comm(pkg, self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, stream, fn, reps: int) -> float:
        """ms per repetition: barrier + synchronize on both sides, CUDA events on `stream`, max over ranks."""
        torch = self.torch
        torch.cuda.synchronize(); self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        self.barrier()
        return ms / reps


def copy_ceiling(ctx: Ctx, x_host, y_host, d_in, d_out, reps: int = 3):
    """The same bytes as one e2e step as bare copies: pinned host -> device and device -> pinned host at once on two
    streams, on every rank at the same time.  GB/s each way per GPU (what ohs_process could reach with free kernels)."""
    torch = ctx.torch
    hx, hy = torch.from_numpy(x_host), torch.from_numpy(y_host)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        with torch.cuda.stream(s1):
            d_in.copy_(hx, non_blocking=True)
        with torch.cuda.stream(s2):
            hy.copy_(d_out, non_blocking=True)
        s1.synchronize(); s2.synchronize()

    once()
    torch.cuda.synchronize(); ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    dt = ctx.max_over_ranks(time.perf_counter() - t0) / reps
    ctx.barrier()
    return x_host.nbytes / dt / 1e9


def parity_vs_oracle(ctx: Ctx, y_dev, x_host_sample, sample_idx, block, h, coeffs, gain):
    """max |gpu - oracle| over the sampled streams (first engine call from zero state)."""
    from oracle import oracle as O

    ref, _ = O.render_batch(x_host_sample, block, h, coeffs, [1] * 10, True, gain, n_threads=min(8, os.cpu_count() or 1))
    got = y_dev[sample_idx].cpu().numpy()
    return float(np.max(np.abs(got - ref)))


def run_stream_config(ctx: Ctx, cfg_id: int, k_blocks: int, reps: int, also_blocks=()):
    """BASELINE config 3 or 5: one GPU's share of the streams, K blocks per call, device-resident; parity of 8 sampled
    streams (first call, zero state) against the oracle; roofline by the config's own bytes(K) formula."""
    torch, pkg = ctx.torch, ctx.pkg
    S = pkg.signals
    c = S.CONFIGS[cfg_id]
    n_streams, block, taps, fs = c["n_streams"], c["block"], c["taps"], c["fs"]
    parts = -(-taps // block)
    h = S.synthetic_hrir_set(taps, c["decay"])
    coeffs = np.stack([pkg.eq_design(t, fs, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    eng = pkg.Engine(n_streams, block, taps, device=ctx.local, sample_rate=fs)
    if ctx.rank == 0 or ctx.world == 1:
        eng.set_hrir_set(h)
    if ctx.world > 1:
        pkg.parallel.broadcast_filters(eng, src=0, comm=ctx.comm)   # the spectra table of the whole job comes from rank 0
    for b in range(10):
        eng.eq_set_band(b, coeffs[b], True)
    eng.set_eq_enable(True); eng.set_gain(GAIN)
    n = block * k_blocks
    unique = 16
    x_host = S.stream_inputs(n_streams, n, base_seed=7000 + 1000 * cfg_id + 100000 * ctx.rank, unique=unique)
    d_in = torch.from_numpy(x_host).to(ctx.dev)
    d_out = torch.empty_like(d_in)
    eng.prepare(n)                                       # scratch of the time-batched route: outside the timed region
    stream = torch.cuda.ExternalStream(eng.cuda_stream(), device=ctx.dev)
    torch.cuda.synchronize()
    # parity: first call from zero state; 8 sampled streams spread over the CTAs (tiled inputs: stream s = base[s % 16])
    eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n)
    eng.sync()
    sample = np.array([0, 1, n_streams // 7, n_streams // 3 + 1, n_streams // 2, (2 * n_streams) // 3 + 2, n_streams - 2, n_streams - 1])
    err = parity_vs_oracle(ctx, d_out, x_host[sample], torch.from_numpy(sample).to(ctx.dev), block, h, coeffs, GAIN)
    launches0 = eng.launch_count()
    for _ in range(2):
        eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n)
    ms = ctx.timed(stream, lambda: eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n), reps)
    launches = (eng.launch_count() - launches0) // (reps + 2)
    peak, _ = hbm_peak()
    bytes_per_call = algorithmic_bytes_per_stream(k_blocks, block, parts) * n_streams
    value = n_streams * ctx.world * (n / fs) / (ms * 1e-3)
    route = ("time-batched (EQ pre-pass on its own SMs beside the previous chunk's forward transforms, per-bin convolution along time, "
             "inverse transforms)") if (parts >= 8 and k_blocks >= 8) else "fused render kernel"
    out = {"workload": c["name"], "n_streams_per_gpu": n_streams, "block": block, "taps": taps, "partitions": parts, "sample_rate": fs,
           "blocks_per_call": k_blocks, "route": route, "kernel_launches_per_call": int(launches), "streams_per_cta": eng.streams_per_cta(),
           "value": value, "unit": UNIT, "ms_per_call": ms,
           "roofline": {"bound": "hbm", "achieved": bytes_per_call / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": bytes_per_call / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_call": int(bytes_per_call),
                        "note": "bytes(K=%d) of SURVEY.md 8d for this config" % k_blocks},
           "parity_max_abs": ctx.max_over_ranks(err), "parity_streams_sampled": int(sample.size), "parity_bar": 1e-5}
    # the other side of north_star's roofline ("the slower of FLOPs at FP32 peak and bytes at HBM bandwidth"), per GPU
    flops_per_call = algorithmic_flops_per_stream_block(block, parts) * k_blocks * n_streams
    t_hbm, t_fp32 = bytes_per_call / (peak * 1e9), flops_per_call / (FP32_FMA_TFLOPS_MEASURED * 1e12)
    out["roofline_fp32"] = {"achieved_tflops": flops_per_call / (ms * 1e-3) / 1e12, "peak_tflops_fma_measured": FP32_FMA_TFLOPS_MEASURED,
                            "frac": flops_per_call / (ms * 1e-3) / 1e12 / FP32_FMA_TFLOPS_MEASURED,
                            "flops_per_stream_block": algorithmic_flops_per_stream_block(block, parts)}
    out["binding_roofline"] = {"bound": "fp32" if t_fp32 > t_hbm else "hbm", "frac": max(t_fp32, t_hbm) / (ms * 1e-3),
                               "note": "time the slower roofline allows / measured time, per GPU"}
    if "time-batched" in route:
        # SURVEY.md 8d, restructuring note: the offline pipeline is reported against its OWN byte formula, 16 B + 8 S per
        # stream-block (audio in and out, one spectrum written, read and its product written and read), not bytes(K)
        own = (16 * block + 8 * 8 * (block + 1)) * k_blocks * n_streams
        out["roofline_pipeline"] = {"bound": "hbm", "achieved": own / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": own / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_call": int(own),
                                    "formula": "(16*B + 8*S) per stream-block, S = 8*(B+1)",
                                    "measured_dram_bytes_per_stream_block": 99900,
                                    "measured_note": "ncu launch list of a serialised 64-block call (profiles/r02_ncu_launches_config5_time_batched_k64.csv): "
                                                     "1.64 GB read + written per 64 blocks of 256 streams"}
    # the same engine with fewer blocks per call (the EQ pre-pass of a call's first chunk and the transforms of its last are
    # not overlapped, so short calls pay more per block)
    for kb in also_blocks:
        n2 = block * kb
        for _ in range(2):
            eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n2, row_stride=n)
        ms2 = ctx.timed(stream, lambda: eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n2, row_stride=n), reps)
        out["at_%d_blocks_per_call" % kb] = {"value": n_streams * ctx.world * (n2 / fs) / (ms2 * 1e-3), "unit": UNIT, "ms_per_call": ms2}
    del eng, d_in, d_out
    torch.cuda.empty_cache()
    return out


def run_single_stream_config(ctx: Ctx, reps: int):
    """BASELINE config 1 (the reference's own CPU-runnable case): ONE stereo stream, 48 kHz, 10 s of pink noise, the
    bundled CIPIC HRIRs (speakers at +-30 degrees: measurements 308 and 908 of tests/golden/cipic003_hrir.npz, 200 taps),
    10-band PEQ, block 512.  One stream cannot fill a GPU: what is reported is latency — the per-block API (one call per
    512-frame host buffer, the plugin's calling pattern) against the 10.67 ms such a buffer lasts — and the whole 10 s in
    one call; parity of the full render against the oracle.  Rank 0 only (the config does not shard)."""
    torch, pkg = ctx.torch, ctx.pkg
    S = pkg.signals
    fix = os.path.join(ROOT, "tests", "golden", "cipic003_hrir.npz")
    if ctx.rank != 0 or not os.path.exists(fix):
        ctx.barrier()
        return None
    from oracle import oracle as O

    block, fs = 512, 48000.0
    ir = np.load(fix)["ir"]
    irs = [ir[308, 0], ir[308, 1], ir[908, 0], ir[908, 1]]
    n_blocks = 938                      # 10 s = 480 000 frames, zero-padded to whole blocks
    n = n_blocks * block
    x = np.zeros((1, 2, n), np.float32)
    x[0, 0, :480000] = S.pink_noise(480000, 1)
    x[0, 1, :480000] = S.pink_noise(480000, 2)
    coeffs = np.stack([pkg.eq_design(t, fs, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])
    eng = pkg.Engine(1, block, 200, device=ctx.local, sample_rate=fs)
    eng.set_hrir_set(irs)
    for b in range(10):
        eng.eq_set_band(b, coeffs[b], True)
    eng.set_eq_enable(True); eng.set_gain(GAIN)
    d_in = torch.from_numpy(x).to(ctx.dev)
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.ExternalStream(eng.cuda_stream(), device=ctx.dev)
    torch.cuda.synchronize()
    eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n)       # first call from zero state: the parity run
    eng.sync()
    ref, _ = O.render_batch(x, block, irs, coeffs, [1] * 10, True, GAIN, n_threads=1)
    err = float(np.max(np.abs(d_out.cpu().numpy() - ref)))

    def whole():
        eng.process_device(d_in.data_ptr(), d_out.data_ptr(), n)

    def per_block(k=64):
        for t in range(k):
            eng.process_device(d_in.data_ptr() + 4 * t * block, d_out.data_ptr() + 4 * t * block, block, row_stride=n)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, r):
        fn()
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(r):
                fn()
            e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / r

    ms_whole = timed(whole, reps)
    ms_block = timed(per_block, reps) / 64
    # one call per host buffer WITH the host waiting for the result (what a real-time caller sees)
    t0 = time.perf_counter()
    for t in range(64):
        eng.process_device(d_in.data_ptr() + 4 * t * block, d_out.data_ptr() + 4 * t * block, block, row_stride=n)
        eng.sync()
    ms_sync = (time.perf_counter() - t0) * 1e3 / 64
    buffer_ms = block / fs * 1e3
    out = {"workload": S.CONFIGS[1]["name"], "block": block, "taps": 200, "sample_rate": fs, "seconds": 10.0,
           "whole_render_ms": ms_whole, "value": (n / fs) / (ms_whole * 1e-3), "unit": UNIT,
           "per_block_api": {"us_per_block_device": ms_block * 1e3, "us_per_block_with_host_sync": ms_sync * 1e3,
                             "host_buffer_ms": buffer_ms, "real_time_factor": buffer_ms / ms_sync},
           "note": "one stream = one CTA: latency, not roofline (SURVEY.md 8d); the whole render is bound by the sequential biquad chain "
                   "(480 000 steps)",
           "parity_max_abs": err, "parity_bar": 1e-5, "parity_extent": "all 938 blocks against the oracle"}
    del eng, d_in, d_out
    ctx.barrier()
    return out


def run_object_config(ctx: Ctx, reps: int):
    """BASELINE config 4: 512 mono sources per GPU, each with its own direction from the bundled CIPIC set, 10 s at
    48 kHz, binaurally mixed to one stereo bus; ncclReduce of the per-GPU buses and the bus EQ + gain on rank 0 are
    INSIDE the timed region, all set-up outside.  Parity: the reduced bus against an f64 evaluation of the definition
    over the first 19 blocks of every source (later blocks run the same code on the same state layout)."""
    torch, pkg, dist = ctx.torch, ctx.pkg, ctx.dist
    S, P = pkg.signals, pkg.parallel
    import scipy.signal as sps

    n_src, block, fs, seconds = 512, 256, 48000.0, 10.0
    n = int(seconds * fs) // block * block
    ir = np.load(os.path.join(ROOT, "tests", "golden", "cipic003_hrir.npz"))["ir"]
    first = n_src * ctx.rank                                   # global source index of this rank's first source
    hr = np.stack([ir[((first + s) * 37) % 1250] for s in range(n_src)]).astype(np.float32)   # [n_src, 2, 200]
    base = np.stack([S.pink_noise(n, 4000 + u) for u in range(8)]) / np.float32(64.0)
    sign = lambda s: np.float32(1.0 if ((first + s) // 8) % 2 == 0 else -1.0)  # noqa: E731
    d_base = torch.from_numpy(base).to(ctx.dev)
    src = torch.empty((n_src, n), dtype=torch.float32, device=ctx.dev)
    for s in range(n_src):
        src[s] = d_base[s % 8] * float(sign(s))
    t_setup = time.perf_counter()
    mixer = P.ObjectMixer(pkg, hr, block, fs, n, eq_preset=S.EQ_PRESET_TYPICAL, gain=GAIN, device=ctx.local, dst=0, comm=ctx.comm)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup
    # parity on the first 19 blocks (4864 frames): f64 truth of this rank's sources, summed over ranks like the bus
    m = 19 * block
    bus = mixer.render(src, apply_post=False)   # the raw reduced bus: the bus EQ is bit-exact by itself (tests) but f32
    torch.cuda.synchronize()                    # EQ round-off (2e-4 against f64) would mask the mix's own error
    truth = np.zeros((2, m))
    for s in range(n_src):
        xs = (base[s % 8][:m] * sign(s)).astype(np.float64)
        for ear in range(2):
            truth[ear] += sps.fftconvolve(xs, hr[s, ear].astype(np.float64))[:m]
    t_truth = torch.from_numpy(truth).to(ctx.dev)
    if ctx.world > 1:
        dist.reduce(t_truth, dst=0, op=dist.ReduceOp.SUM)
    err = float((bus[:, :m].double() - t_truth).abs().max().item()) if ctx.rank == 0 else 0.0
    cur = torch.cuda.current_stream(ctx.dev)
    launches0 = mixer.engine.launch_count()

    def once():
        mixer.reset()
        mixer.render(src)

    once()
    ms = ctx.timed(cur, once, reps)
    launches = (mixer.engine.launch_count() - launches0) // (reps + 1)
    peak, _ = hbm_peak()
    total_src = n_src * ctx.world
    value = total_src * (n / fs) / (ms * 1e-3)
    n_blocks = n // block
    # SURVEY 8d, per mono source and block: 1 024 B of input + the HRIR spectra once (4 112 B) ; 15 632 flop
    bytes_algo = n_src * (1024 * n_blocks + 4112)
    flops = n_src * 15632.0 * n_blocks
    out = {"workload": "cfg4: %d mono sources per GPU (4096 over 8 GPUs), own CIPIC direction each, 10 s at 48 kHz, one stereo bus; "
                       "ncclReduce + bus EQ + gain inside the timed region" % n_src,
           "n_sources_per_gpu": n_src, "n_sources_total": total_src, "block": block, "taps": 200, "seconds": n / fs,
           "value": value, "unit": "source-s/s", "ms_per_render": ms, "setup_s_outside_timed_region": t_setup,
           "kernel_launches_per_render": int(launches), "streams_per_cta": mixer.engine.streams_per_cta(),
           "roofline": {"bound": "fp32", "achieved_tflops": flops / (ms * 1e-3) / 1e12, "peak_tflops_fma_measured": FP32_FMA_TFLOPS_MEASURED,
                        "frac": flops / (ms * 1e-3) / 1e12 / FP32_FMA_TFLOPS_MEASURED,
                        "hbm_achieved_gbs": bytes_algo / (ms * 1e-3) / 1e9, "hbm_frac": bytes_algo / (ms * 1e-3) / 1e9 / peak,
                        "note": "per GPU; SURVEY.md 8d: 15 632 flop and 1 024 B per mono source and block (FP32-bound config)"},
           "parity_max_abs": ctx.max_over_ranks(err), "parity_against": "f64 evaluation of the reduced bus (before the bus EQ), first %d frames of all %d sources" % (m, total_src),
           "parity_bar": 1e-5}
    del mixer, src
    torch.cuda.empty_cache()
    return out


def dump_outputs(out_dir: str, torch, d_out):
    """What the headline step hands its caller: y[stream, channel, frame] of the last timed step, float32.  The whole step
    is 400 MB, so a fixed sample of DUMP_STREAMS streams (seed 0, sorted, spread over the batch) is written.  The inputs,
    the warm-up and the step count fix the engine's state, so equal arguments give equal outputs on one build."""
    idx = np.sort(np.random.default_rng(0).choice(N_STREAMS, DUMP_STREAMS, replace=False))
    y = d_out[torch.from_numpy(idx).to(d_out.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "y.npy"), y)


def run_gpu(args, pkg):
    ctx = Ctx(args, pkg)
    torch, dist = ctx.torch, ctx.dist
    world, rank, local = ctx.world, ctx.rank, ctx.local

    h, coeffs = workload_arrays(pkg.signals, pkg.eq_design)
    eng = pkg.Engine(N_STREAMS, BLOCK, TAPS, device=local, sample_rate=FS)
    if rank == 0 or world == 1:
        eng.set_hrir_set(h)
        eng.commit_filters()
        eng.sync()
    if world > 1:
        # one HRIR spectra table for the whole job: rank 0 transforms the IRs, NCCL broadcasts the spectra
        pkg.parallel.broadcast_filters(eng, src=0, comm=ctx.comm)
    for b in range(10):
        eng.eq_set_band(b, coeffs[b], True)
    eng.set_eq_enable(True)
    eng.set_gain(GAIN)

    x_host = pkg.PinnedBuffer((N_STREAMS, 2, FRAMES_PER_STEP))
    y_host = pkg.PinnedBuffer((N_STREAMS, 2, FRAMES_PER_STEP))
    x_host.array[...] = pkg.signals.stream_inputs(N_STREAMS, FRAMES_PER_STEP, base_seed=1000 + 100000 * rank, unique=UNIQUE_STREAMS)
    d_in = torch.from_numpy(x_host.array).cuda()
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.ExternalStream(eng.cuda_stream(), device=ctx.dev)
    eng.prepare(FRAMES_PER_STEP, host_io=True)   # staging buffers of the host-pointer path: outside every timed region
    torch.cuda.synchronize()
    step = lambda: eng.process_device(d_in.data_ptr(), d_out.data_ptr(), FRAMES_PER_STEP)  # noqa: E731

    # ---- device-resident arm ---------------------------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = eng.launch_count()
    ms_per_step = ctx.timed(stream, step, args.steps)
    launches = eng.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, d_out)
    stream_seconds_per_step = N_STREAMS * world * FRAMES_PER_STEP / FS
    value = stream_seconds_per_step / (ms_per_step * 1e-3)

    if args.device_only:
        if rank == 0:
            emit_json(({"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": ms_per_step, "gpu_launches": int(launches),
                              "note": "device-only run (profiling helper)"}))
        return

    # ---- sustained leg: the same launch back to back for >= 3 s, clocks and power sampled throughout ------------
    sus_reps = max(args.steps, int(SUSTAINED_SECONDS * 1e3 / ms_per_step) + 1)
    sus_sampler = ClockSampler(local, period_ms=200) if rank == 0 else None
    sus_ms = ctx.timed(stream, step, sus_reps)
    sus_clocks = sus_sampler.stop() if sus_sampler else None
    sus_value = stream_seconds_per_step / (sus_ms * 1e-3)

    # ---- per-block API (K = 1): one launch per engine block, state round-trips through HBM every launch ----------
    k1_blocks = 128
    k1_step = [0]

    def k1():
        off = (k1_step[0] % BLOCKS_PER_STEP) * BLOCK * 4
        k1_step[0] += 1
        eng.process_device(d_in.data_ptr() + off, d_out.data_ptr() + off, BLOCK, FRAMES_PER_STEP)

    for _ in range(16):
        k1()
    k1_ms = ctx.timed(stream, k1, k1_blocks)

    # ---- end-to-end arm: host buffers through ohs_process ----------------------------------------------------------
    e2e_steps = max(2, min(args.steps, 10))
    eng.process(x_host.array, out=y_host.array)  # warm-up
    torch.cuda.synchronize(); ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.process(x_host.array, out=y_host.array)
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    ctx.barrier()
    e2e_value = e2e_steps * stream_seconds_per_step / e2e_s
    checksum = float(np.abs(y_host.array[0, 0, :4096]).sum())
    ceiling_gbs = copy_ceiling(ctx, x_host.array, y_host.array, d_in, d_out)
    e2e_gbs = x_host.array.nbytes * e2e_steps / e2e_s / 1e9

    # ---- the other BASELINE configs at one GPU's share of their full extent ---------------------------------------
    configs = {}
    if not args.no_configs:
        del d_in, d_out
        torch.cuda.empty_cache()
        c1 = run_single_stream_config(ctx, reps=3)
        if c1 is not None:
            configs["cfg1"] = c1
        configs["cfg3"] = run_stream_config(ctx, 3, 128, reps=5)
        configs["cfg5"] = run_stream_config(ctx, 5, 512, reps=3, also_blocks=(64, 256))
        configs["cfg4"] = run_object_config(ctx, reps=3)

    if rank == 0:
        peak, peak_src = hbm_peak()
        bytes_per_launch = algorithmic_bytes_per_stream(BLOCKS_PER_STEP) * N_STREAMS
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        flops_per_launch = algorithmic_flops_per_stream_block() * BLOCKS_PER_STEP * N_STREAMS
        k1_bytes = algorithmic_bytes_per_stream(1) * N_STREAMS
        agree = abs(sus_value / value - 1.0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (seeded pink noise, %d unique streams tiled to %d; synthetic 256-tap HRIR set; AutoEQ-like 10-band preset)"
                    % (UNIQUE_STREAMS, N_STREAMS),
            "config": workload_config(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(x_host.array.nbytes), "d2h_bytes_per_step": int(y_host.array.nbytes),
                    "steps": e2e_steps, "api": "ohs_process (host pointers, pinned), 3-stage H2D/kernel/D2H pipeline",
                    "gbs_each_way_per_gpu": e2e_gbs, "copy_ceiling_gbs": ceiling_gbs, "frac_of_copy_ceiling": e2e_gbs / ceiling_gbs,
                    "copy_ceiling_note": "bare pinned H2D + D2H of the same buffers at once, on all %d rank(s) at the same time; GB/s each way per GPU "
                                         "(aggregate %.1f GB/s each way)" % (world, ceiling_gbs * world)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "sustained": {"value": sus_value, "unit": UNIT, "seconds": sus_ms * sus_reps * 1e-3, "launches": sus_reps, "ms_per_step": sus_ms,
                          "sm_mhz_median": (sus_clocks or {}).get("sm_mhz"), "power_w_max": (sus_clocks or {}).get("power_w_max"),
                          "samples": (sus_clocks or {}).get("samples"), "reasons": (sus_clocks or {}).get("reasons"),
                          "vs_value": sus_value / value,
                          "note": ("agrees with the %d-step figure within %.1f %%" % (args.steps, 100 * agree)) if agree <= 0.03 else
                                  ("differs from the %d-step figure by %.1f %%: the sustained figure is the honest one for long renders" % (args.steps, 100 * agree))},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic_bytes(), "peak_source": peak_src, "kernel": "ohs::render_kernel<512,7,0>",
                         "algorithmic_bytes_per_launch": int(bytes_per_launch),
                         "note": "K=%d blocks per launch; formula bytes(K) of SURVEY.md 8d" % BLOCKS_PER_STEP},
            "roofline_fp32": {"achieved_tflops": flops_per_launch / (ms_per_step * 1e-3) / 1e12,
                              "peak_tflops_fma_measured": FP32_FMA_TFLOPS_MEASURED,
                              "frac": flops_per_launch / (ms_per_step * 1e-3) / 1e12 / FP32_FMA_TFLOPS_MEASURED,
                              "note": "per GPU; the bit-exact EQ forbids FMA contraction, so its 180 flop/frame cost 180 FP32-pipe slots"},
            "per_block_api": {"blocks_per_launch": 1, "launches_timed": k1_blocks, "ms_per_launch": k1_ms,
                              "value": N_STREAMS * world * (BLOCK / FS) / (k1_ms * 1e-3), "unit": UNIT,
                              "roofline_achieved_gbs": k1_bytes / (k1_ms * 1e-3) / 1e9, "roofline_frac": k1_bytes / (k1_ms * 1e-3) / 1e9 / peak,
                              "kernel": "ohs::render_kernel<512,7,1> (latency variant), programmatic dependent launches"},
            "configs": configs,
            "checksum": checksum,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample, _ = cpu_reference_run(pkg.signals, 1, 1, 16 * (os.cpu_count() or 1), 10.24)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        emit_json((line))
    ctx.barrier()
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner to fd 1
    when NCCL_DEBUG is set), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, help="timed steps (default 50; 40 with --impl reference, whose steps take seconds on the CPU)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs 3/4/5 legs")
    ap.add_argument("--device-only", action="store_true", help="only the device-resident arm (used under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's output for %d streams (a fixed sample; rank 0's streams "
                         "when several GPUs run) to DIR/y.npy" % DUMP_STREAMS)
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 40 if args.impl == "reference" else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        # signals only (pure numpy): the product library is never mapped by this arm
        import importlib.util

        spec = importlib.util.spec_from_file_location("ohs_signals", os.path.join(ROOT, "open-headstage_b200", "signals.py"))
        signals = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(signals)
        run_reference(args, signals)
    else:
        run_gpu(args, _bootstrap.load_package())


if __name__ == "__main__":
    main()
