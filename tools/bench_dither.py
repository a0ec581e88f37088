"""Dithered PCM output (DESIGN §12): what TPDF dither and noise shaping cost on BASELINE config 2 (1024 streams x 1.024 s
per step), the card's name, power limit and max SM clock read in the same run.  Writes <out>/dither_n1.json (a list of
records) and prints one JSON line per record.

  host     ohs_process_pcm S16->S16 with dither off, flat TPDF, shaped M = 2 and shaped M = 9, and S24->S24 off and shaped
           M = 2, each arm on its own engine with pinned buffers; after a warm-up the arms take turns, --steps-per-turn
           steps at a time, until each has --steps timed steps
  kernels  the encode kernel alone over 403 MB of f32 rows (a bypassed F32 -> S16 / S24 ohs_process_device_pcm call runs
           exactly one encode): plain, flat TPDF, shaped M = 2 and M = 9; CUDA events over many launches, arms alternating
  device   ohs_process_device_pcm S16->S16 on resident buffers, dither off against shaped M = 2 and M = 9, CUDA events,
           arms alternating
  trace    torch.profiler over two host steps of S16->S16 off and shaped M = 9: device time of copies and kernels per step

    python tools/bench_dither.py --out /tmp/dither
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench_pcm as B  # noqa: E402  (package loading, config-2 engine, pinned buffers, card query)

pkg, S, torch = B.pkg, B.S, B.torch
F32, S16, S24 = B.F32, B.S16, B.S24
H2 = (2.0, -1.0)
# Wannamaker's 9-tap F-weighted set (J. Audio Eng. Soc. 40(7/8), 1992), as in tests/test_dither.py
H9 = (2.412, -3.370, 3.937, -4.174, 3.353, -2.205, 1.281, -0.569, 0.0847)
DITHERS = {"off": None, "tpdf": (), "shaped_m2": H2, "shaped_m9": H9}


def engine(dither):
    e = B.engine()
    if dither is not None:
        e.set_dither(pkg.DITHER_TPDF, seed=1, shape=dither)
    return e


def host(out, args):
    x = (0.9 * S.stream_inputs(B.N_STREAMS, B.FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    arms = []
    for fmt, names in ((S16, ("off", "tpdf", "shaped_m2", "shaped_m9")), (S24, ("off", "shaped_m2"))):
        for name in names:
            xin, yout = B.buffer_of(fmt), B.buffer_of(fmt)
            xin.array[...] = B.to_format(x, fmt)[0]
            e = engine(DITHERS[name])
            step = lambda e=e, xin=xin, yout=yout, fmt=fmt: e.process_pcm(xin.array, fmt, out=yout.array)  # noqa: E731
            for _ in range(args.warmup):
                step()
            arms.append({"fmt": fmt, "dither": name, "engine": e, "in": xin, "out": yout, "step": step, "times": []})
    while min(len(a["times"]) for a in arms) < args.steps:
        for a in arms:
            for _ in range(args.steps_per_turn):
                t0 = time.perf_counter()
                a["step"]()
                a["times"].append(time.perf_counter() - t0)
    base = {}
    for a in arms:
        t = np.array(a["times"])
        sec = float(np.median(t))
        base.setdefault(a["fmt"], sec)
        out({"leg": "host", "arm": "%s->%s" % (B.NAME[a["fmt"]], B.NAME[a["fmt"]]), "dither": a["dither"],
             "api": "ohs_process_pcm", "steps_timed": int(len(t)), "s_per_step_median": sec, "s_per_step_min": float(t.min()),
             "s_per_step_max": float(t.max()), "value": B.N_STREAMS * B.FRAMES / B.FS / sec, "unit": "stream-s/s",
             "time_vs_dither_off": sec / base[a["fmt"]]})
        a["in"].free(); a["out"].free(); a["engine"].close()


def timed_alternating(arms, reps, rounds):
    """arms: {name: (engine, fn)}.  CUDA events on the engine's stream around `reps` calls of fn, the arms taking turns for
    `rounds` rounds: (median, min, max) ms per call."""
    for _, fn in arms.values():
        for _ in range(3):
            fn()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, (e, fn) in arms.items():
            stream = torch.cuda.ExternalStream(e.cuda_stream())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            e1.synchronize()
            res[k].append(e0.elapsed_time(e1) / reps)
    return {k: (float(np.median(v)), float(np.min(v)), float(np.max(v))) for k, v in res.items()}


def kernels(out):
    n_f32 = B.N_STREAMS * 2 * B.FRAMES
    d_f32 = torch.from_numpy((0.9 * S.stream_inputs(B.N_STREAMS, B.FRAMES, base_seed=7000, unique=16)).ravel()).cuda()
    d_pcm = torch.zeros(n_f32 * 3, dtype=torch.uint8, device="cuda")
    for fmt in (S16, S24):
        engines = {k: engine(v) for k, v in DITHERS.items()}
        for e in engines.values():
            e.set_bypass(True)
        launches0 = {k: e.launch_count() for k, e in engines.items()}
        arms = {k: (e, lambda e=e: e.process_device_pcm(d_f32.data_ptr(), F32, d_pcm.data_ptr(), fmt, B.FRAMES)) for k, e in engines.items()}
        times = timed_alternating(arms, 20, 5)
        for k, ms in times.items():
            kernel = {"off": "pcm_encode_kernel<%s>", "tpdf": "pcm_encode_kernel<%s, dither>"}.get(k, "pcm_encode_shaped_kernel<%s, M>")
            out({"leg": "kernels", "kernel": kernel % B.NAME[fmt], "dither": k, "f32_bytes": n_f32 * 4, "pcm_bytes": n_f32 * B.BYTES[fmt],
                 "launches_per_call": (engines[k].launch_count() - launches0[k]) / (3 + 20 * 5), "ms_median": ms[0], "ms_min": ms[1],
                 "ms_max": ms[2], "gbs_read_plus_written": n_f32 * (4 + B.BYTES[fmt]) / (ms[0] * 1e-3) / 1e9})
        for e in engines.values():
            e.close()


def device(out):
    x = (0.9 * S.stream_inputs(B.N_STREAMS, B.FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    q = torch.from_numpy(np.ascontiguousarray(S.pcm_encode(x, S16))).cuda()
    names = ("off", "shaped_m2", "shaped_m9")
    engines = {k: engine(DITHERS[k]) for k in names}
    bufs = {k: torch.empty_like(q) for k in names}
    for e in engines.values():
        e.prepare(B.FRAMES)
    arms = {k: (engines[k], lambda e=engines[k], o=bufs[k]: e.process_device_pcm(q.data_ptr(), S16, o.data_ptr(), S16, B.FRAMES))
            for k in names}
    times = timed_alternating(arms, 5, 6)
    base = times["off"][0]
    for k in names:
        ms = times[k][0]
        out({"leg": "device", "arm": "S16->S16", "dither": k, "api": "ohs_process_device_pcm", "ms_per_step_median": ms,
             "value": B.N_STREAMS * B.FRAMES / B.FS / (ms * 1e-3), "unit": "stream-s/s", "time_vs_dither_off": ms / base})
    for e in engines.values():
        e.close()


def trace(out, outdir):
    from torch.profiler import ProfilerActivity, profile

    x = (0.9 * S.stream_inputs(B.N_STREAMS, B.FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    for name in ("off", "shaped_m9"):
        xin, yout = B.buffer_of(S16), B.buffer_of(S16)
        xin.array[...] = B.to_format(x, S16)[0]
        e = engine(DITHERS[name])
        step = lambda: e.process_pcm(xin.array, S16, out=yout.array)  # noqa: E731
        step()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(2):
                step()
        path = os.path.join(outdir, "dither_trace_%s.json" % name)
        prof.export_chrome_trace(path)
        cat, names = {"h2d_ms": 0.0, "d2h_ms": 0.0, "kernel_ms": 0.0}, {}
        with open(path) as f:
            events = json.load(f)["traceEvents"]
        for ev in events:
            kind, n, ms = ev.get("cat", ""), ev.get("name", ""), ev.get("dur", 0) / 1e3
            if kind == "gpu_memcpy":
                cat["h2d_ms" if "HtoD" in n else "d2h_ms"] += ms
            elif kind == "kernel":
                cat["kernel_ms"] += ms
                key = n.split("(")[0].replace("void ", "")
                names[key] = names.get(key, 0.0) + ms
        out({"leg": "trace", "arm": "S16->S16", "dither": name, **{k: v / 2 for k, v in cat.items()},
             "kernels_ms_per_step": {k: v / 2 for k, v in names.items()},
             "note": "device time summed per category over 2 steps, halved; copies and kernels overlap"})
        xin.free(); yout.free(); e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--steps-per-turn", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="host,kernels,device,trace")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    records = []

    def out(obj):
        print(json.dumps(obj), flush=True)
        records.append(obj)

    out({"card": B.card(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
         "workload": "BASELINE config 2: %d streams, block %d, %d-tap HRIR, 10-band PEQ, gain %.1f, %d frames (1.024 s) per step"
                     % (B.N_STREAMS, B.BLOCK, B.TAPS, B.GAIN, B.FRAMES)})
    legs = {"host": lambda: host(out, args), "kernels": lambda: kernels(out), "device": lambda: device(out),
            "trace": lambda: trace(out, args.out)}
    for name in args.only.split(","):
        legs[name]()
    out({"card_after": B.card()})
    with open(os.path.join(args.out, "dither_n1.json"), "w") as f:
        json.dump(records, f, indent=1)


if __name__ == "__main__":
    main()
