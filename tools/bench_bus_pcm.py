"""Integer PCM listener buses (DESIGN §14): what mixing, dithering and encoding each group's bus in one GPU pass buys on
BASELINE config 2 streams wired as 7.1 files (1024 streams in 256 groups of 4, 1.024 s per step, pinned host buffers), the
card's name, power limit and max SM clock read in the same run.  Writes <out>/bus_pcm_n1.json (a list of records) and
prints one JSON line per record.

  parity   before any timing, on fresh engines and 16 blocks per call: every host arm's ohs_process_grouped_pcm against
           ohs_process_pcm(..., F32) mixed by signals.mix_groups and encoded by signals.pcm_encode_dithered(...,
           first_row=2S); ohs_process_device + ohs_mix_device_pcm against the host call; and, at the full step, the fused
           mix-encode against the unfused pair below in every dither mode: bit for bit (the run stops otherwise)
  host     7.1 groups, S16 input: F32 bus; S16 bus with dither off, TPDF, shaped M = 2 and M = 9; S24 input -> S24 bus off
           and shaped M = 2.  Each arm on its own engine; after a warm-up the arms take turns, each turn a window of
           consecutive steps of at least --window seconds, until each arm has --turns turns.  Per arm: ms per step,
           stream-s/s, link GB/s each way, and the bare-copy ceiling of the arm's own bytes (pinned H2D and D2H at once)
  device   device-resident, CUDA events over windows of at least --window seconds, the arms alternating:
           ohs_process_device + ohs_mix_device (F32 bus) against ohs_process_device + ohs_mix_device_pcm (S16 bus) in each
           dither mode; and the fused mix-encode alone against the unfused pair, ohs_mix_device into an f32 bus and then a
           bypassed F32 -> S16 ohs_process_device_pcm on an engine of n_streams = G (exactly one encode of the 2G bus
           rows; its seed is seed + phi * 2S, so its rows get the bus rows' noise), ordered after the mix with CUDA events

    python tools/bench_bus_pcm.py --out /tmp/bus_pcm
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench_groups as BG  # noqa: E402  (7.1 engines, the copy ceiling)
import bench_pcm as B  # noqa: E402  (package loading, pinned buffers, card query)

pkg, S, torch = B.pkg, B.S, B.torch
F32, S16, S24 = B.F32, B.S16, B.S24
N, FRAMES = B.N_STREAMS, B.FRAMES
FIRST = BG.LAYOUTS["7.1"]
G = len(FIRST) - 1
SEED = 0x5EED
PHI = 0x9E3779B97F4A7C15
H2 = (2.0, -1.0)
H9 = (2.412, -3.370, 3.937, -4.174, 3.353, -2.205, 1.281, -0.569, 0.0847)   # Wannamaker's 9-tap F-weighted set
MODES = {"off": None, "tpdf": (), "shaped_m2": H2, "shaped_m9": H9}
# (name, input format, bus format, dither mode)
HOST_ARMS = [("S16 in, F32 bus", S16, F32, "off"),
             ("S16 in, S16 bus, dither off", S16, S16, "off"),
             ("S16 in, S16 bus, TPDF", S16, S16, "tpdf"),
             ("S16 in, S16 bus, shaped M=2", S16, S16, "shaped_m2"),
             ("S16 in, S16 bus, shaped M=9", S16, S16, "shaped_m9"),
             ("S24 in, S24 bus, dither off", S24, S24, "off"),
             ("S24 in, S24 bus, shaped M=2", S24, S24, "shaped_m2")]


def engine(mode, seed=SEED):
    e = BG.grouped_engine("7.1")
    if MODES[mode] is not None:
        e.set_dither(pkg.DITHER_TPDF, seed=seed, shape=MODES[mode])
    return e


def reference(y, fmt, mode):
    """The bytes of the buses of rendered rows y under the bus definition (first call after ohs_set_dither)."""
    bus = S.mix_groups(y, FIRST)
    if fmt == F32:
        return bus.tobytes()
    if MODES[mode] is None:
        q = S.pcm_encode(bus, fmt)
    else:
        q, _ = S.pcm_encode_dithered(bus, fmt, SEED, 0, MODES[mode], first_row=2 * N)
    return (q if fmt == S16 else S.pack_s24(q)).tobytes()


def parity(out, x):
    n = 16 * B.BLOCK
    xs = np.ascontiguousarray(x[:, :, :n])
    for name, fi, fo, mode in HOST_ARMS:
        buf, dec = B.to_format(xs, fi)
        a, b, c = BG.engine(BG.PAIRS["7.1"]), engine(mode), engine(mode)
        want = reference(a.process_pcm(buf, F32), fo, mode)
        got = np.ascontiguousarray(b.process_grouped(buf, bus_format=fo)).tobytes()
        d = torch.from_numpy(dec).cuda()
        dbus = torch.zeros((G, 2, n * B.BYTES[fo]), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        c.process_device(d.data_ptr(), d.data_ptr(), n)
        c.mix_device(d.data_ptr(), dbus.data_ptr(), n, bus_format=fo)
        c.sync()
        dev = dbus.cpu().numpy().tobytes()
        ok = got == want and dev == want
        out({"leg": "parity", "arm": name, "frames": n, "host_bit_exact": got == want, "device_bit_exact": dev == want})
        if not ok:
            raise SystemExit("integer buses differ from the reference (%s)" % name)
        for e in (a, b, c):
            e.close()


class Device:
    """Rendered rows of the 7.1 engine in HBM, and the bus arms over them."""

    def __init__(self, x):
        self.d_in = torch.from_numpy(x).cuda()
        self.d_out = torch.empty_like(self.d_in)
        self.bus32 = torch.empty((G, 2, FRAMES), dtype=torch.float32, device="cuda")
        self.bus16 = torch.empty((G, 2, FRAMES), dtype=torch.int16, device="cuda")
        self.bus16b = torch.empty((G, 2, FRAMES), dtype=torch.int16, device="cuda")
        self.engines = {m: engine(m) for m in MODES}
        for e in self.engines.values():
            e.prepare(FRAMES)
        # the encode engine of the unfused pair: 2G rows, bypassed, seeded so that its row r is bus row r
        self.enc = {}
        for m in MODES:
            e = pkg.Engine(G, B.BLOCK, B.TAPS, sample_rate=B.FS)
            e.set_bypass(True)
            if MODES[m] is not None:
                e.set_dither(pkg.DITHER_TPDF, seed=(SEED + PHI * 2 * N) % 2 ** 64, shape=MODES[m])
            self.enc[m] = e
        e0 = self.engines["off"]
        torch.cuda.synchronize()
        e0.process_device(self.d_in.data_ptr(), self.d_out.data_ptr(), FRAMES)
        e0.sync()

    def render(self, m):
        self.engines[m].process_device(self.d_in.data_ptr(), self.d_out.data_ptr(), FRAMES)

    def mix_f32(self, m):
        self.engines[m].mix_device(self.d_out.data_ptr(), self.bus32.data_ptr(), FRAMES)

    def fused(self, m):
        self.engines[m].mix_device(self.d_out.data_ptr(), self.bus16.data_ptr(), FRAMES, bus_format=S16)

    def unfused(self, m):
        e, enc = self.engines[m], self.enc[m]
        s_mix, s_enc = torch.cuda.ExternalStream(e.cuda_stream()), torch.cuda.ExternalStream(enc.cuda_stream())
        self.mix_f32(m)
        ev = torch.cuda.Event()
        ev.record(s_mix)
        s_enc.wait_event(ev)
        enc.process_device_pcm(self.bus32.data_ptr(), F32, self.bus16b.data_ptr(), S16, FRAMES)
        ev2 = torch.cuda.Event()
        ev2.record(s_enc)
        s_mix.wait_event(ev2)

    def window(self, m, fn, reps):
        stream = torch.cuda.ExternalStream(self.engines[m].cuda_stream())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    def close(self):
        for e in list(self.engines.values()) + list(self.enc.values()):
            e.close()


def device(out, x, args):
    dv = Device(x)
    # parity of the fused and the unfused mix-encode at the full step, each mode from a fresh position
    for m in MODES:
        dv.fused(m)
        dv.unfused(m)
        dv.engines[m].sync()
        same = torch.equal(dv.bus16, dv.bus16b)
        out({"leg": "parity", "arm": "fused vs unfused mix-encode, %s" % m, "frames": FRAMES, "bit_exact": bool(same)})
        if not same:
            raise SystemExit("the fused mix-encode differs from the unfused pair (%s)" % m)
    arms = {"render + mix F32": ("off", lambda: (dv.render("off"), dv.mix_f32("off")))}
    for m in MODES:
        arms["render + mix S16 %s" % m] = (m, lambda m=m: (dv.render(m), dv.fused(m)))
    for m in MODES:
        arms["fused mix-encode S16 %s" % m] = (m, lambda m=m: dv.fused(m))
        arms["unfused mix F32 + encode S16 %s" % m] = (m, lambda m=m: dv.unfused(m))
    reps = {}
    for k, (m, fn) in arms.items():   # warm-up, then as many calls as fill a window
        for _ in range(3):
            fn()
        ms = dv.window(m, fn, 10)
        reps[k] = max(10, int(args.window * 1e3 / ms) + 1)
    res = {k: [] for k in arms}
    for _ in range(args.turns):
        for k, (m, fn) in arms.items():
            res[k].append(dv.window(m, fn, reps[k]))
    # HBM bytes each arm needs: the stream rows read once, the bus written once (S16: 2 bytes); the unfused pair also writes
    # and re-reads the f32 bus
    rows_in, bus32, bus16 = N * 2 * FRAMES * 4, G * 2 * FRAMES * 4, G * 2 * FRAMES * 2
    need = {"fused": rows_in + bus16, "unfused": rows_in + 2 * bus32 + bus16}
    base = float(np.median(res["render + mix F32"]))
    for k, v in res.items():
        ms = float(np.median(v))
        rec = {"leg": "device", "arm": k, "layout": "7.1", "groups": G, "reps_per_window": reps[k], "turns": len(v),
               "ms_per_step_median": ms, "ms_min": float(np.min(v)), "ms_max": float(np.max(v))}
        if k.startswith("render"):
            rec.update(value=N * FRAMES / B.FS / (ms * 1e-3), unit="stream-s/s", time_vs_render_mix_f32=ms / base)
        else:
            kind = "fused" if k.startswith("fused") else "unfused"
            rec.update(hbm_bytes=need[kind], hbm_gbs=need[kind] / (ms * 1e-3) / 1e9)
        out(rec)
    for m in MODES:
        f = float(np.median(res["fused mix-encode S16 %s" % m]))
        u = float(np.median(res["unfused mix F32 + encode S16 %s" % m]))
        out({"leg": "device", "arm": "fused / unfused, %s" % m, "time_ratio": f / u, "saved_ms_per_step": u - f,
             "bytes_saved_per_step": need["unfused"] - need["fused"]})
    dv.close()


def host(out, x, args):
    arms = []
    for name, fi, fo, mode in HOST_ARMS:
        xin = B.buffer_of(fi)
        xin.array[...] = B.to_format(x, fi)[0]
        e = engine(mode)
        shape = (G, 2, FRAMES * (3 if fo == S24 else 1))
        yout = pkg.PinnedBuffer(shape, {F32: np.float32, S16: np.int16, S24: np.uint8}[fo])
        step = lambda e=e, xin=xin, yout=yout, fo=fo: e.process_grouped(xin.array, out=yout.array, bus_format=fo)  # noqa: E731
        for _ in range(args.warmup):
            step()
        arms.append({"name": name, "in_format": B.NAME[fi], "bus_format": B.NAME[fo], "dither": mode, "engine": e, "in": xin,
                     "out": yout, "step": step, "bytes_in": N * 2 * FRAMES * B.BYTES[fi], "bytes_out": G * 2 * FRAMES * B.BYTES[fo],
                     "turns": []})
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
        ceil = BG.copy_ceiling_s(a["bytes_in"], a["bytes_out"], args.window)
        out({"leg": "host", "arm": a["name"], "in": a["in_format"], "bus": a["bus_format"], "dither": a["dither"], "layout": "7.1",
             "turns": len(t), "window_s_min": args.window, "ms_per_step_median": sec * 1e3, "ms_per_step_min": float(t.min()) * 1e3,
             "ms_per_step_max": float(t.max()) * 1e3, "value": N * FRAMES / B.FS / sec, "unit": "stream-s/s",
             "bytes_in_per_step": a["bytes_in"], "bytes_out_per_step": a["bytes_out"],
             "h2d_gbs": a["bytes_in"] / sec / 1e9, "d2h_gbs": a["bytes_out"] / sec / 1e9,
             "copy_ceiling_ms": ceil * 1e3, "fraction_of_copy_ceiling": ceil / sec})
        a["in"].free(); a["out"].free(); a["engine"].close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--turns", type=int, default=4)
    ap.add_argument("--window", type=float, default=0.5, help="seconds of each timed window")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="parity,device,host")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    records = []

    def out(obj):
        print(json.dumps(obj), flush=True)
        records.append(obj)

    out({"card": B.card(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
         "workload": "BASELINE config 2 streams wired as 7.1 files: %d streams in %d groups of 4, 4 HRIR sets (stream s bound to set "
                     "s %% 4), block %d, %d-tap HRIR, 10-band PEQ, gain %.1f, %d frames (1.024 s) per step; dither seed 0x%X"
                     % (N, G, B.BLOCK, B.TAPS, B.GAIN, FRAMES, SEED)})
    x = (0.9 * S.stream_inputs(N, FRAMES, base_seed=7000, unique=16)).astype(np.float32)
    legs = {"parity": lambda: parity(out, x), "host": lambda: host(out, x, args), "device": lambda: device(out, x, args)}
    for name in args.only.split(","):
        legs[name]()
    out({"card_after": B.card()})
    with open(os.path.join(args.out, "bus_pcm_n1.json"), "w") as f:
        json.dump(records, f, indent=1)


if __name__ == "__main__":
    main()
