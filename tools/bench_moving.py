"""Moving sources benchmark (DESIGN §10): workloads W1-W7, device-resident, one JSON line each, plus the card's name and
power limit read in the same run, into <out>/moving_sources.jsonl.  Every timed window is >= 0.5 s after a warm-up;
sampled streams are checked against twins (engines bound statically to each set, rendered from the same zero state)
by the definition in include/ohs.h, bit for bit, and W5 against the oracle.

    python tools/bench_moving.py --out /tmp/moving
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

FS = 48000.0
GAIN = 0.5
COEFFS = np.stack([pkg.eq_design(t, FS, fc, q, g) for (t, fc, q, g) in S.EQ_PRESET_TYPICAL])


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(eng, fn, min_s=0.5):
    """Seconds per call: warm-up, then enough calls for a window of >= min_s, CUDA events on the engine's stream."""
    stream = torch.cuda.ExternalStream(eng.cuda_stream())
    for _ in range(2):
        fn()
    eng.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        s = e0.elapsed_time(e1) * 1e-3
        if s >= min_s:
            return s / reps, reps, s
        reps = max(reps * 2, int(reps * min_s / max(s, 1e-6) * 1.2) + 1)


def engine(n, block, set_irs, bound=None, eq=True, time_batch=True, max_taps=None):
    e = pkg.Engine(n, block, max_taps or max(len(p) for irs in set_irs for p in irs), n_hrir_sets=len(set_irs), sample_rate=FS)
    for k, irs in enumerate(set_irs):
        e.set_hrir_set(irs, hrir_set=k)
    if eq:
        for b in range(10):
            e.eq_set_band(b, COEFFS[b], True)
        e.set_eq_enable(True)
    e.set_gain(GAIN)
    e.set_time_batch(time_batch)
    if bound is not None:
        for s in np.nonzero(bound)[0]:
            e.bind_stream_hrir(int(s), int(bound[s]))
    return e


def crossfade(a, b, block):
    w = ((2 * np.arange(block) + 1) / (2.0 * block)).astype(np.float32)
    return a + w * (b - a)


def assemble(static, sets, bound, block):
    out = np.empty_like(static[int(sets[0])])
    prev = int(bound)
    for t, cur in enumerate(int(v) for v in sets):
        sl = slice(t * block, (t + 1) * block)
        out[:, sl] = static[cur][:, sl] if cur == prev else crossfade(static[prev][:, sl], static[cur][:, sl], block)
        prev = cur
    return out


def run_once(e, d_in, d_out, n, sched=None):
    e.process_device(d_in.data_ptr(), d_out.data_ptr(), n, hrir_schedule=sched)
    e.sync()
    return d_out


def twin_parity(make, d_in, n, block, sched, bound, sample, n_sets=2):
    """Bit-exact check of sampled streams of a first scheduled call (zero state) against static engines of each set."""
    d_out = torch.empty_like(d_in)
    y = run_once(make(bound), d_in, d_out, n, sched)[sample].cpu().numpy()
    static = {}
    for k in range(n_sets):
        static[k] = run_once(make(np.full(len(bound), k)), d_in, d_out, n)[sample].cpu().numpy()
    bad = 0
    for i, s in enumerate(sample):
        want = assemble({k: static[k][i] for k in static}, sched[s], bound[s], block)
        bad += int(not np.array_equal(y[i].view(np.uint32), want.view(np.uint32)))
    return {"streams_sampled": int(len(sample)), "bit_exact_mismatches": bad}


def rate(n_streams, frames, sec):
    return n_streams * frames / FS / sec


def w1_to_w4(out):
    block, n, k = 256, 1024, 192
    set_irs = [S.synthetic_hrir_set(256, 40.0, seed=11), S.synthetic_hrir_set(256, 40.0, seed=12)]
    frames = block * k
    x = S.stream_inputs(n, frames, unique=16)
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.empty_like(d_in)
    bound = (np.arange(n) % 2).astype(np.int32)
    t = np.arange(k)
    s_ = np.arange(n)[:, None]
    static = np.repeat(bound[:, None], k, axis=1).astype(np.int32)
    every8 = (bound[:, None] ^ (((t[None, :] + s_) // 8) & 1)).astype(np.int32)   # staggered by stream
    every1 = (bound[:, None] ^ ((t[None, :] + 1) & 1)).astype(np.int32)
    make = lambda b: engine(n, block, set_irs, b)  # noqa: E731
    sample = np.array([0, 1, 333, 700, 1022, 1023])
    res = {}
    for name, sched, note in (("W1", None, "static bindings, ohs_process_device"),
                              ("W2", static, "scheduled call, no transition"),
                              ("W3", every8, "a transition every 8th block per stream, staggered by stream"),
                              ("W4", every1, "a transition every block on every stream")):
        e = make(bound)
        e.prepare(frames)
        sec, reps, window = timed(e, lambda: e.process_device(d_in.data_ptr(), d_out.data_ptr(), frames, hrir_schedule=sched))
        line = {"workload": name, "what": note, "n_streams": n, "block": block, "taps": 256, "hrir_sets": 2, "blocks_per_call": k,
                "ms_per_call": sec * 1e3, "value": rate(n, frames, sec), "unit": "stream-s/s", "calls_timed": reps, "window_s": window}
        if sched is not None:
            line["transitions_per_call"] = int(np.sum(sched[:, 1:] != sched[:, :-1]) + np.sum(sched[:, 0] != sched[:, -1]))
            line["parity_vs_twins"] = twin_parity(make, d_in, frames, block, sched, bound, sample)
        res[name] = line
        out(line)
        del e
    res["W3"]["vs_W1"] = res["W3"]["value"] / res["W1"]["value"]
    res["W4"]["vs_W1"] = res["W4"]["value"] / res["W1"]["value"]
    out({"workload": "W3/W4 vs W1", "W3_over_W1": res["W3"]["vs_W1"], "W4_over_W1": res["W4"]["vs_W1"], "W2_over_W1": res["W2"]["value"] / res["W1"]["value"]})


def w5(out):
    """512 one-source streams, the 1250 CIPIC measurements as sets, circular trajectories at 0.5 rev/s with per-stream
    phase, nearest measurement per block, 10 s in one call."""
    from oracle import oracle as O

    d = np.load(os.path.join(ROOT, "tests", "golden", "cipic003_hrir.npz"))
    ir, pos = d["ir"], d["pos"]
    az, el = np.radians(pos[:, 0]), np.radians(pos[:, 1])
    dirs = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], axis=1)
    block, n = 256, 512
    k = int(10 * FS) // block
    frames = block * k
    set_irs = [[ir[m, 0], ir[m, 1], np.zeros(0, np.float32), np.zeros(0, np.float32)] for m in range(len(ir))]
    tc = (np.arange(k) + 0.5) * block / FS
    phase = np.arange(n) / n * 2 * np.pi
    th = 2 * np.pi * 0.5 * tc[None, :] + phase[:, None]
    target = np.stack([np.cos(th), np.sin(th), np.zeros_like(th)], axis=-1)   # horizontal circle
    sched = np.argmax(target @ dirs.T, axis=-1).astype(np.int32)              # nearest measurement per block
    x = np.zeros((n, 2, frames), np.float32)
    base = np.stack([S.pink_noise(frames, 6000 + u) for u in range(8)])
    for s in range(n):
        x[s, 0] = base[s % 8]
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.empty_like(d_in)
    e = pkg.Engine(n, block, 200, n_hrir_sets=len(ir), sample_rate=FS)
    for m, irs in enumerate(set_irs):
        e.set_hrir_set(irs, hrir_set=m)
    for s in range(n):
        e.bind_stream_hrir(s, int(sched[s, -1]))   # steady state: each call continues where the last one ended
    e.set_gain(GAIN)
    e.prepare(frames)
    sec, reps, window = timed(e, lambda: e.process_device(d_in.data_ptr(), d_out.data_ptr(), frames, hrir_schedule=sched))
    # parity: a fresh engine's first call against the oracle blend, two streams, first 96 blocks
    f = pkg.Engine(n, block, 200, n_hrir_sets=len(ir), sample_rate=FS)
    for m, irs in enumerate(set_irs):
        f.set_hrir_set(irs, hrir_set=m)
    for s in range(n):
        f.bind_stream_hrir(s, int(sched[s, 0]))
    f.set_gain(GAIN)
    kk = 96
    y = run_once(f, d_in[:, :, :kk * block].contiguous(), torch.empty_like(d_in[:, :, :kk * block]).contiguous(), kk * block, sched[:, :kk])
    y = y.cpu().numpy()
    err = 0.0
    for s in (0, 311):
        used = sorted(set(sched[s, :kk].tolist()))
        st = {m: O.render_batch(x[s:s + 1, :, :kk * block], block, set_irs[m], np.zeros((1, 5), np.float32), [0], False, GAIN)[0][0] for m in used}
        err = max(err, float(np.max(np.abs(y[s] - assemble(st, sched[s, :kk], sched[s, 0], block)))))
    out({"workload": "W5", "what": "512 one-source streams, 1250 CIPIC measurements as sets, circular trajectories at 0.5 rev/s, "
                                   "nearest measurement per block, 10 s in one call",
         "n_streams": n, "block": block, "taps": 200, "hrir_sets": len(ir), "blocks_per_call": k,
         "transitions_per_call": int(np.sum(sched[:, 1:] != sched[:, :-1]) + np.sum(sched[:, 0] != sched[:, -1])),
         "ms_per_call": sec * 1e3, "value": rate(n, frames, sec), "unit": "source-s/s", "calls_timed": reps, "window_s": window,
         "parity_vs_oracle_max_abs": err, "parity_streams": 2, "parity_blocks": kk, "parity_bar": 1e-5})


def w6(out):
    """K = 1 calls: per-buffer latency with ohs_move_stream_hrir(OHS_ALL, ...) before every call against none."""
    for n, block, taps in ((1024, 256, 256), (1, 512, 200)):
        set_irs = [S.synthetic_hrir_set(taps, 40.0, seed=11), S.synthetic_hrir_set(taps, 40.0, seed=12)]
        x = S.stream_inputs(n, block * 64, unique=16)
        d_in = torch.from_numpy(x).cuda()
        d_out = torch.empty_like(d_in)
        for mode in ("static", "move_every_call"):
            e = engine(n, block, set_irs)
            e.prepare(block)
            state = {"i": 0}

            def call():
                i = state["i"] = state["i"] + 1
                if mode != "static":
                    e.move_stream_hrir(pkg.OHS_ALL, i & 1)
                o = (i % 64) * block
                e.process_device(d_in.data_ptr() + 4 * o, d_out.data_ptr() + 4 * o, block, row_stride=block * 64)

            sec, reps, window = timed(e, call)
            out({"workload": "W6", "mode": mode, "n_streams": n, "block": block, "taps": taps, "hrir_sets": 2, "blocks_per_call": 1,
                 "us_per_call": sec * 1e6, "value": rate(n, block, sec), "unit": "stream-s/s", "calls_timed": reps, "window_s": window,
                 "note": "back-to-back calls, CUDA events around the loop (host work of the move included)"})
            del e


def w7(out):
    """256 streams, two 48 000-tap sets at B 1024, 512 blocks per call, one move per 64 blocks per stream."""
    block, n, k, taps = 1024, 256, 512, 48000
    set_irs = [S.synthetic_hrir_set(taps, 9000.0, seed=31), S.synthetic_hrir_set(taps, 9000.0, seed=32)]
    frames = block * k
    x = S.stream_inputs(n, frames, unique=16)
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.empty_like(d_in)
    bound = (np.arange(n) % 2).astype(np.int32)
    t = np.arange(k)
    sched = (bound[:, None] ^ (((t[None, :] + 8 * np.arange(n)[:, None]) // 64) & 1)).astype(np.int32)
    for name, sc, tb in (("time-batched, static", None, True), ("block-by-block, static (set_time_batch(False))", None, False),
                         ("moving, one move per 64 blocks", sched, True)):
        e = engine(n, block, set_irs, bound, time_batch=tb)
        e.prepare(frames)
        sec, reps, window = timed(e, lambda: e.process_device(d_in.data_ptr(), d_out.data_ptr(), frames, hrir_schedule=sc))
        line = {"workload": "W7", "mode": name, "n_streams": n, "block": block, "taps": taps, "partitions": 47, "blocks_per_call": k,
                "ms_per_call": sec * 1e3, "value": rate(n, frames, sec), "unit": "stream-s/s", "calls_timed": reps, "window_s": window}
        if sc is not None:
            line["parity_vs_twins"] = twin_parity(lambda b: engine(n, block, set_irs, b, time_batch=False), d_in, frames, block, sc, bound,
                                                  np.array([0, 1, 130, 255]))
        out(line)
        del e
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--only", default="W1,W5,W6,W7")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "moving_sources.jsonl")
    fh = open(path, "w")

    def out(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        fh.write(s + "\n")
        fh.flush()

    out({"card": card(), "time": time.strftime("%Y-%m-%d %H:%M:%S")})
    legs = {"W1": w1_to_w4, "W5": w5, "W6": w6, "W7": w7}
    for name in args.only.split(","):
        legs[name](out)
    out({"card_after": card()})
    fh.close()


if __name__ == "__main__":
    main()
