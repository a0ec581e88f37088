"""Integer PCM in and out (DESIGN §11): end-to-end throughput of ohs_process_pcm against ohs_process on BASELINE config 2
(1024 streams x 1.024 s per step, pinned host buffers from ohs_host_alloc), one JSON line per result into
<out>/pcm_io.jsonl, the card's name, power limit and max SM clock read in the same run.

  arms       F32->F32 (bench.py's e2e arm), S16->S16, S24->S24, S16->F32, each on its own engine; after a warm-up the
             arms take turns, --steps-per-turn steps at a time, until each has --steps timed steps.  Per arm:
             stream-s/s, GB/s each way, and the bare-copy ceiling of the same bytes (pinned H2D and D2H at once on two
             streams, measured in the same run) with the fraction of it reached
  parity     for each PCM arm, 8 sampled streams of a first call from zero state against the F32 path on the decoded
             input, quantised by the reference encode (signals.pcm_encode): bit for bit
  kernels    the decode and encode kernels alone (bypassed ohs_process_device_pcm calls, which run exactly one of them)
             over 403 MB of f32 rows, CUDA events over many launches, against a device-to-device cudaMemcpyAsync of
             the same f32 bytes
  trace      torch.profiler over two steps of the F32 and the S16 arm: device time of the H2D and D2H copies and of the
             kernels, per step

    python tools/bench_pcm.py --out /tmp/pcm
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import _bootstrap  # noqa: E402

pkg = _bootstrap.load_package()
S = pkg.signals
import torch  # noqa: E402

F32, S16, S24 = pkg.FMT_F32, pkg.FMT_S16, pkg.FMT_S24
NAME = {F32: "F32", S16: "S16", S24: "S24"}
BYTES = {F32: 4, S16: 2, S24: 3}
FS = 48000.0
GAIN = 0.5
N_STREAMS, BLOCK, TAPS = 1024, 256, 256
FRAMES = 192 * BLOCK   # 1.024 s per step, as bench.py
ARMS = [(F32, F32), (S16, S16), (S24, S24), (S16, F32)]
SAMPLE = np.array([0, 1, 146, 341, 512, 683, 1022, 1023])


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def engine():
    c = S.CONFIGS[2]
    e = pkg.Engine(N_STREAMS, BLOCK, TAPS, sample_rate=FS)
    e.set_hrir_set(S.synthetic_hrir_set(TAPS, c["decay"]))
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True)
    e.set_gain(GAIN)
    e.prepare(FRAMES, host_io=True)
    return e


def buffer_of(fmt, n=FRAMES):
    return pkg.PinnedBuffer((N_STREAMS, 2, n * (3 if fmt == S24 else 1)), {F32: np.float32, S16: np.int16, S24: np.uint8}[fmt])


def to_format(x, fmt):
    """f32 rows -> (PCM buffer contents, their decode)."""
    if fmt == F32:
        return x, x
    q = S.pcm_encode(x, fmt)
    return (q if fmt == S16 else S.pack_s24(q)), S.pcm_decode(q, fmt)


def encode(y, fmt):
    if fmt == F32:
        return y
    q = S.pcm_encode(y, fmt)
    return q if fmt == S16 else S.pack_s24(q)


def copy_ceiling_s(bytes_in, bytes_out, reps=5):
    """Seconds for bytes_in pinned host -> device and bytes_out device -> pinned host at once on two streams."""
    hi = pkg.PinnedBuffer((bytes_in,), np.uint8)
    ho = pkg.PinnedBuffer((bytes_out,), np.uint8)
    di = torch.empty(bytes_in, dtype=torch.uint8, device="cuda")
    do = torch.empty(bytes_out, dtype=torch.uint8, device="cuda")
    thi, tho = torch.from_numpy(hi.array), torch.from_numpy(ho.array)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        with torch.cuda.stream(s1):
            di.copy_(thi, non_blocking=True)
        with torch.cuda.stream(s2):
            tho.copy_(do, non_blocking=True)
        s1.synchronize(); s2.synchronize()

    once()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    dt = (time.perf_counter() - t0) / reps
    del di, do
    hi.free(); ho.free()
    return dt


def e2e(out, args):
    x = (0.9 * S.stream_inputs(N_STREAMS, FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    arms = []
    for fi, fo in ARMS:
        xin, yout = buffer_of(fi), buffer_of(fo)
        xin.array[...] = to_format(x, fi)[0]
        e = engine()
        if (fi, fo) == (F32, F32):
            step = lambda e=e, xin=xin, yout=yout: e.process(xin.array, out=yout.array)  # noqa: E731
        else:
            step = lambda e=e, xin=xin, yout=yout, fo=fo: e.process_pcm(xin.array, fo, out=yout.array)  # noqa: E731
        for _ in range(args.warmup):
            step()
        arms.append({"fi": fi, "fo": fo, "engine": e, "in": xin, "out": yout, "step": step, "times": []})
    # the arms take turns so that drift of the host or the link spreads over all of them alike
    while min(len(a["times"]) for a in arms) < args.steps:
        for a in arms:
            for _ in range(args.steps_per_turn):
                t0 = time.perf_counter()
                a["step"]()
                a["times"].append(time.perf_counter() - t0)
    base = None
    for a in arms:
        fi, fo = a["fi"], a["fo"]
        t = np.array(a["times"])
        sec = float(np.median(t))
        bin_, bout = N_STREAMS * 2 * FRAMES * BYTES[fi], N_STREAMS * 2 * FRAMES * BYTES[fo]
        ceil_s = copy_ceiling_s(bin_, bout)
        line = {"arm": "%s->%s" % (NAME[fi], NAME[fo]), "api": "ohs_process" if fi == fo == F32 else "ohs_process_pcm",
                "n_streams": N_STREAMS, "frames_per_step": FRAMES, "steps_timed": int(len(t)),
                "s_per_step_median": sec, "s_per_step_min": float(t.min()), "s_per_step_max": float(t.max()),
                "value": N_STREAMS * FRAMES / FS / sec, "unit": "stream-s/s",
                "h2d_bytes_per_step": bin_, "d2h_bytes_per_step": bout,
                "h2d_gbs": bin_ / sec / 1e9, "d2h_gbs": bout / sec / 1e9,
                "copy_ceiling_s": ceil_s, "copy_ceiling_h2d_gbs": bin_ / ceil_s / 1e9, "copy_ceiling_d2h_gbs": bout / ceil_s / 1e9,
                "frac_of_copy_ceiling": ceil_s / sec}
        if base is None:
            base = line["value"]
        line["vs_f32_arm"] = line["value"] / base
        if (fi, fo) != (F32, F32):
            line["parity_vs_quantised_f32"] = parity(fi, fo, x)
        out(line)
    for a in arms:
        a["in"].free(); a["out"].free()
        a["engine"].close()


def parity(fi, fo, x):
    """First call from zero state on fresh engines: the PCM arm against the F32 path on decode(in), quantised."""
    buf, dec = to_format(x, fi)
    ref, dut = engine(), engine()
    want = encode(ref.process(dec)[SAMPLE], fo)
    got = dut.process_pcm(buf, fo)[SAMPLE]
    bad = sum(int(np.ascontiguousarray(got[i]).tobytes() != np.ascontiguousarray(want[i]).tobytes()) for i in range(len(SAMPLE)))
    ref.close(); dut.close()
    return {"streams_sampled": int(len(SAMPLE)), "bit_exact_mismatches": bad}


def kernels(out, reps=50):
    """Decode / encode alone: a bypassed ohs_process_device_pcm with one integer side and one f32 side runs exactly one
    conversion kernel (decode into f32 output rows, or encode from f32 input rows)."""
    e = engine()
    e.set_bypass(True)
    stream = torch.cuda.ExternalStream(e.cuda_stream())
    n_f32 = N_STREAMS * 2 * FRAMES
    d_f32 = torch.zeros(n_f32, dtype=torch.float32, device="cuda")
    d_f32b = torch.zeros_like(d_f32)
    d_pcm = torch.zeros(n_f32 * 3, dtype=torch.uint8, device="cuda")

    def timed(fn, stream):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    f32_bytes = n_f32 * 4
    for fmt in (S16, S24):
        pcm_bytes = n_f32 * BYTES[fmt]
        for what, fi, fo, a, b in (("decode", fmt, F32, d_pcm, d_f32), ("encode", F32, fmt, d_f32, d_pcm)):
            launches0 = e.launch_count()
            sec = timed(lambda: e.process_device_pcm(a.data_ptr(), fi, b.data_ptr(), fo, FRAMES), stream)
            out({"kernel": "pcm_%s_kernel<%s>" % (what, NAME[fmt]), "f32_bytes": f32_bytes, "pcm_bytes": pcm_bytes,
                 "launches_per_call": (e.launch_count() - launches0) / (reps + 3),
                 "ms": sec * 1e3, "gbs_read_plus_written": (f32_bytes + pcm_bytes) / sec / 1e9})
    with torch.cuda.stream(stream):
        sec = timed(lambda: d_f32b.copy_(d_f32), stream)
    out({"kernel": "device-to-device cudaMemcpyAsync of the f32 bytes", "f32_bytes": f32_bytes, "ms": sec * 1e3,
         "gbs_read_plus_written": 2 * f32_bytes / sec / 1e9})
    e.close()


def trace(out, outdir):
    """torch.profiler over two steps of the F32 and the S16 arm: where each step's device time goes."""
    from torch.profiler import ProfilerActivity, profile

    x = (0.9 * S.stream_inputs(N_STREAMS, FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    for fi, fo in ((F32, F32), (S16, S16)):
        xin, yout = buffer_of(fi), buffer_of(fo)
        xin.array[...] = to_format(x, fi)[0]
        e = engine()
        step = (lambda: e.process(xin.array, out=yout.array)) if fi == F32 else (lambda: e.process_pcm(xin.array, fo, out=yout.array))
        step()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            t0 = time.perf_counter()
            for _ in range(2):
                step()
            wall = (time.perf_counter() - t0) / 2
        path = os.path.join(outdir, "pcm_trace_%s.json" % NAME[fi])
        prof.export_chrome_trace(path)
        cat = {"h2d_ms": 0.0, "d2h_ms": 0.0, "kernel_ms": 0.0}
        names = {}
        with open(path) as f:
            events = json.load(f)["traceEvents"]
        for ev in events:
            kind, n, ms = ev.get("cat", ""), ev.get("name", ""), ev.get("dur", 0) / 1e3
            if kind == "gpu_memcpy" and "HtoD" in n:
                cat["h2d_ms"] += ms
            elif kind == "gpu_memcpy" and "DtoH" in n:
                cat["d2h_ms"] += ms
            elif kind == "kernel":
                cat["kernel_ms"] += ms
                key = n.split("<")[0].split("(")[0].replace("void ", "")
                names[key] = names.get(key, 0.0) + ms
        out({"trace": "%s->%s" % (NAME[fi], NAME[fo]), "wall_ms_per_step": wall * 1e3,
             **{k: v / 2 for k, v in cat.items()}, "kernels_ms_per_step": {k: v / 2 for k, v in names.items()},
             "note": "device time summed per category and divided by the 2 steps; copies and kernels overlap"})
        xin.free(); yout.free(); e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--steps-per-turn", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="e2e,kernels,trace")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    fh = open(os.path.join(args.out, "pcm_io.jsonl"), "w")

    def out(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        fh.write(s + "\n")
        fh.flush()

    out({"card": card(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
         "workload": "BASELINE config 2: %d streams, block %d, %d-tap HRIR, 10-band PEQ, gain %.1f, %d frames (1.024 s) per step"
                     % (N_STREAMS, BLOCK, TAPS, GAIN, FRAMES)})
    legs = {"e2e": lambda: e2e(out, args), "kernels": lambda: kernels(out), "trace": lambda: trace(out, args.out)}
    for name in args.only.split(","):
        legs[name]()
    out({"card_after": card()})
    fh.close()


if __name__ == "__main__":
    main()
