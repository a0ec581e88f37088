"""Listener buses (DESIGN §13): what returning only the group buses buys on BASELINE config 2 streams (1024 streams x 1.024 s
per step, pinned host buffers from ohs_host_alloc), the card's name, power limit and max SM clock read in the same run.
Writes <out>/groups_n1.json (a list of records) and prints one JSON line per record.

  parity   before any timing: ohs_process_grouped on fresh engines against ohs_process_pcm(..., F32) mixed by
           signals.mix_groups, every group of every layout timed below, F32 and S16 input: bit for bit (the run stops
           otherwise)
  engines  config 2 with one HRIR set per speaker pair, as a surround file is wired (4 sets for 7.1, 3 for 5.1; stream s
           bound to set s % pairs); the per-stream arms and the device leg use the 7.1 wiring
  host     256 7.1 groups (4 streams each): ohs_process_grouped with F32 and S16 input against per-stream output through
           ohs_process (F32 -> F32) and ohs_process_pcm (S16 -> S16); 5.1 groups (3 streams each; 1024 = 341 * 3 + 1, so the
           last group holds one stream): ohs_process_grouped with F32 and S16 input.  Each arm on its own engine; after a
           warm-up the arms take turns, each turn a window of consecutive steps of at least --window seconds, until each arm
           has --turns turns.  Per arm: stream-s/s, link GB/s each way, and the bare-copy ceiling of the same bytes (pinned
           H2D and D2H at once on two streams, at least --window seconds of copies, measured in the same run)
  device   device-resident: ohs_process_device alone, ohs_process_device followed by the grouped ohs_mix_device of the 256
           7.1 groups, and that mix alone; CUDA events over windows of at least --window seconds, the arms alternating

    python tools/bench_groups.py --out /tmp/groups
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
F32, S16 = B.F32, B.S16
N, FRAMES = B.N_STREAMS, B.FRAMES
LAYOUTS = {"7.1": list(range(0, N + 1, 4)), "5.1": list(range(0, N, 3)) + [N]}
PAIRS = {"7.1": 4, "5.1": 3}   # speaker pairs per file: one HRIR set each, stream s bound to set s % pairs


def engine(pairs):
    """Config 2 engine (bench_pcm.engine) with one 256-tap HRIR set per speaker pair, wired as a surround file is."""
    c = S.CONFIGS[2]
    e = pkg.Engine(N, B.BLOCK, B.TAPS, n_hrir_sets=pairs, sample_rate=B.FS)
    for k in range(pairs):
        e.set_hrir_set(S.synthetic_hrir_set(B.TAPS, c["decay"], seed=7 + k), hrir_set=k)
    for s in range(N):
        e.bind_stream_hrir(s, s % pairs)
    e.eq_set_preset(S.EQ_PRESET_TYPICAL)
    e.set_eq_enable(True)
    e.set_gain(B.GAIN)
    e.prepare(FRAMES, host_io=True)
    return e


def grouped_engine(layout):
    first = LAYOUTS[layout]
    e = engine(PAIRS[layout])
    e.set_groups(first)
    e.prepare(FRAMES, host_io=True)   # the bus staging too
    return e


def parity(out, x):
    for layout, first in LAYOUTS.items():
        for fmt in (F32, S16):
            buf = B.to_format(x, fmt)[0]
            a, b = engine(PAIRS[layout]), grouped_engine(layout)
            want = S.mix_groups(a.process_pcm(buf, F32), first)
            got = b.process_grouped(buf)
            ok = got.tobytes() == want.tobytes()
            out({"leg": "parity", "layout": layout, "in": B.NAME[fmt], "groups": len(first) - 1, "bit_exact": ok})
            if not ok:
                raise SystemExit("ohs_process_grouped differs from ohs_process_pcm + signals.mix_groups (%s, %s)" % (layout, B.NAME[fmt]))
            a.close(); b.close()


def copy_ceiling_s(bytes_in, bytes_out, window):
    """Seconds for bytes_in pinned host -> device and bytes_out device -> pinned host at once on two streams, averaged over
    a window of at least `window` seconds."""
    hi, ho = pkg.PinnedBuffer((bytes_in,), np.uint8), pkg.PinnedBuffer((bytes_out,), np.uint8)
    di, do = torch.empty(bytes_in, dtype=torch.uint8, device="cuda"), torch.empty(bytes_out, dtype=torch.uint8, device="cuda")
    thi, tho = torch.from_numpy(hi.array), torch.from_numpy(ho.array)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        with torch.cuda.stream(s1):
            di.copy_(thi, non_blocking=True)
        with torch.cuda.stream(s2):
            tho.copy_(do, non_blocking=True)
        s1.synchronize(); s2.synchronize()

    once()
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < window:
        once()
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    del di, do
    hi.free(); ho.free()
    return dt


def host(out, x, args):
    G71, G51 = len(LAYOUTS["7.1"]) - 1, len(LAYOUTS["5.1"]) - 1
    # (name, layout or None, input format, output format for per-stream arms, bytes in, bytes out per step)
    specs = [("grouped 7.1 F32 in", "7.1", F32, None, N * 2 * FRAMES * 4, G71 * 2 * FRAMES * 4),
             ("grouped 7.1 S16 in", "7.1", S16, None, N * 2 * FRAMES * 2, G71 * 2 * FRAMES * 4),
             ("per-stream ohs_process F32->F32", None, F32, F32, N * 2 * FRAMES * 4, N * 2 * FRAMES * 4),
             ("per-stream ohs_process_pcm S16->S16", None, S16, S16, N * 2 * FRAMES * 2, N * 2 * FRAMES * 2),
             ("grouped 5.1 F32 in", "5.1", F32, None, N * 2 * FRAMES * 4, G51 * 2 * FRAMES * 4),
             ("grouped 5.1 S16 in", "5.1", S16, None, N * 2 * FRAMES * 2, G51 * 2 * FRAMES * 4)]
    arms = []
    for name, layout, fi, fo, bin_, bout in specs:
        xin = B.buffer_of(fi)
        xin.array[...] = B.to_format(x, fi)[0]
        if layout:
            e = grouped_engine(layout)
            yout = pkg.PinnedBuffer((len(LAYOUTS[layout]) - 1, 2, FRAMES), np.float32)
            step = lambda e=e, xin=xin, yout=yout: e.process_grouped(xin.array, out=yout.array)  # noqa: E731
        else:
            e = engine(PAIRS["7.1"])
            yout = B.buffer_of(fo)
            step = (lambda e=e, xin=xin, yout=yout: e.process(xin.array, out=yout.array)) if fi == F32 else \
                (lambda e=e, xin=xin, yout=yout, fo=fo: e.process_pcm(xin.array, fo, out=yout.array))  # noqa: E731
        for _ in range(args.warmup):
            step()
        arms.append({"name": name, "layout": layout, "engine": e, "in": xin, "out": yout, "step": step, "bytes_in": bin_,
                     "bytes_out": bout, "turns": []})
    for _ in range(args.turns):
        for a in arms:
            k, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < args.window:
                a["step"]()
                k += 1
            a["turns"].append((time.perf_counter() - t0) / k)
    for a in arms:
        t = np.array(a["turns"])
        sec = float(np.median(t))
        ceil = copy_ceiling_s(a["bytes_in"], a["bytes_out"], args.window)
        out({"leg": "host", "arm": a["name"], "layout": a["layout"], "turns": len(t), "window_s_min": args.window,
             "s_per_step_median": sec, "s_per_step_min": float(t.min()), "s_per_step_max": float(t.max()),
             "value": N * FRAMES / B.FS / sec, "unit": "stream-s/s",
             "bytes_in_per_step": a["bytes_in"], "bytes_out_per_step": a["bytes_out"],
             "h2d_gbs": a["bytes_in"] / sec / 1e9, "d2h_gbs": a["bytes_out"] / sec / 1e9,
             "link_gbs": (a["bytes_in"] + a["bytes_out"]) / sec / 1e9,
             "copy_ceiling_s": ceil, "fraction_of_copy_ceiling": ceil / sec})
        a["in"].free(); a["out"].free(); a["engine"].close()


def device(out, x, args):
    first = LAYOUTS["7.1"]
    G = len(first) - 1
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.empty_like(d_in)
    bus = torch.empty((G, 2, FRAMES), dtype=torch.float32, device="cuda")
    e = grouped_engine("7.1")
    e.prepare(FRAMES)
    render = lambda: e.process_device(d_in.data_ptr(), d_out.data_ptr(), FRAMES)  # noqa: E731
    mix = lambda: e.mix_device(d_out.data_ptr(), bus.data_ptr(), FRAMES)  # noqa: E731
    arms = {"render": render, "render+mix": lambda: (render(), mix()), "mix": mix}
    stream = torch.cuda.ExternalStream(e.cuda_stream())

    def window(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    reps = {}
    for k, fn in arms.items():   # warm-up, then as many calls as fill a window
        for _ in range(3):
            fn()
        ms = window(fn, 10)
        reps[k] = max(10, int(args.window * 1e3 / ms) + 1)
    res = {k: [] for k in arms}
    for _ in range(args.turns):
        for k, fn in arms.items():
            res[k].append(window(fn, reps[k]))
    # the mix's own bytes: every stream row read once, the bus rows written once
    mix_bytes = (N + G) * 2 * FRAMES * 4
    base = float(np.median(res["render"]))
    for k, v in res.items():
        ms = float(np.median(v))
        rec = {"leg": "device", "arm": k, "layout": "7.1", "groups": G, "reps_per_window": reps[k], "ms_per_step_median": ms,
               "ms_min": float(np.min(v)), "ms_max": float(np.max(v)), "time_vs_render": ms / base}
        if k == "mix":
            rec["gbs_read_plus_written"] = mix_bytes / (ms * 1e-3) / 1e9
        else:
            rec["value"], rec["unit"] = N * FRAMES / B.FS / (ms * 1e-3), "stream-s/s"
        out(rec)
    e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--turns", type=int, default=4)
    ap.add_argument("--window", type=float, default=0.5, help="seconds of each timed window")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="parity,host,device")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    records = []

    def out(obj):
        print(json.dumps(obj), flush=True)
        records.append(obj)

    out({"card": B.card(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
         "workload": "BASELINE config 2 streams: %d streams, block %d, %d-tap HRIR, 10-band PEQ, gain %.1f, %d frames (1.024 s) "
                     "per step; 7.1 = groups of 4 streams and 4 HRIR sets, 5.1 = groups of 3 and 3 HRIR sets, stream s bound to set "
                     "s %% pairs; the per-stream arms and the device leg use the 7.1 wiring" % (N, B.BLOCK, B.TAPS, B.GAIN, FRAMES)})
    x = (0.9 * S.stream_inputs(N, FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    legs = {"parity": lambda: parity(out, x), "host": lambda: host(out, x, args), "device": lambda: device(out, x, args)}
    for name in args.only.split(","):
        legs[name]()
    out({"card_after": B.card()})
    with open(os.path.join(args.out, "groups_n1.json"), "w") as f:
        json.dump(records, f, indent=1)


if __name__ == "__main__":
    main()
