#!/usr/bin/env python
"""What the max-hold / min-hold / average traces cost (DESIGN 3.8), on the GPU.

bench.py's cfg2 configuration (uint8 IQ, mode fast, pipelined batches, 512 frames per
step, EMA 0.3) timed with the traces off and on, legs alternated in one process over
the same K steps, with CUDA events on the engine's stream; the rows of the last step
of every leg must be the same bit for bit.  Then the latency of one peak query, host
to host, at W = 256 (cfg2's rows) and W = 65536 (cfg3's rows, crop=None).  The card's
name, power limit and maximum SM clock are read in the same run.

    python tests/tools/trace_overhead.py [--steps 40] [--reps 5] [--out profiles/trace_overhead.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [v.strip() for v in q.stdout.strip().split(",")]
        out.update(power_limit_w=float(pl), sm_max_mhz=float(clk))
    except Exception as exc:                   # the numbers are still worth having without it
        out["query_error"] = repr(exc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "trace_overhead.jsonl"))
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU timings")
    from pypanadapter_b200 import synth
    from pypanadapter_b200.engine import ZoomPSD

    w, F, K = synth.CFG2, args.frames, args.steps
    info = card()
    eng = ZoomPSD(0)
    eng.set_option("pipeline", 1)
    eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                  f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode="fast")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    W = eng.row_width
    d_in = torch.from_numpy(synth.make_frames(w, F, distinct=min(F, 8))).cuda()
    d_rows = torch.empty((F, W), dtype=torch.float32, device="cuda")

    def leg(on):
        eng.traces_enable(on)
        eng.reset_ema()
        for _ in range(args.warmup):
            eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
        eng.join()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(K):
            eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
        eng.join()
        b.record(stream)
        b.synchronize()
        rows = d_rows.cpu().numpy()
        if on:
            assert eng.trace_count == (args.warmup + K) * F
        return a.elapsed_time(b) / K, rows

    ms = {False: [], True: []}
    rows = {}
    for _rep in range(args.reps):
        for on in (False, True):
            t, r = leg(on)
            ms[on].append(t)
            if on in rows:
                assert np.array_equal(rows[on], r)
            rows[on] = r
    assert np.array_equal(rows[False], rows[True]), "traces changed the rows"
    off, on = float(np.median(ms[False])), float(np.median(ms[True]))
    rec = {"what": "cfg2 fast pipelined, ms per step, traces off vs on", "card": info, "frames": F,
           "steps": K, "reps": args.reps, "ms_off": ms[False], "ms_on": ms[True], "median_off": off,
           "median_on": on, "overhead_pct": 100.0 * (on - off) / off,
           "input_gsps_off": F * w.frame_len / (off * 1e-3) / 1e9, "input_gsps_on": F * w.frame_len / (on * 1e-3) / 1e9}

    # per-launch device time of the update, from the engine's own profile (class 18 = finalisation)
    eng.set_profiling(True)
    eng.profile()
    for on_ in (False, True):
        eng.traces_enable(on_)
        for _ in range(10):
            eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
        eng.join()
        p = eng.profile().get("finalize", (0.0, 0))
        rec["finalize_ms_per_step_%s" % ("on" if on_ else "off")] = p[0] / 10
        rec["finalize_launches_per_step_%s" % ("on" if on_ else "off")] = p[1] / 10
    eng.set_profiling(False)

    # peak query latency, host to host
    def peaks_latency(e, kind, k, d, n_calls=200):
        for _ in range(10):
            e.trace_peaks(kind, k=k, distance=d)
        ts = []
        for _ in range(n_calls):
            t0 = time.perf_counter()
            e.trace_peaks(kind, k=k, distance=d)
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        return {"median_us": float(np.median(ts)), "p90_us": float(np.percentile(ts, 90))}

    lat = {}
    for k in (8, 64):
        lat["W=256 max k=%d d=3" % k] = peaks_latency(eng, "max", k, 3)
        lat["W=256 avg k=%d d=3" % k] = peaks_latency(eng, "avg", k, 3)
    eng.traces_enable(False)
    w3 = synth.CFG3
    e3 = ZoomPSD(0)
    e3.configure(w3.fs, w3.fft_size, w3.fft_ratio, w3.frame_len, w3.window, crop=w3.crop, mode="exact")
    e3.traces_enable(True)
    e3.process(synth.make_frames(w3, 4))
    assert e3.row_width == 65536
    for k in (8, 64):
        lat["W=65536 max k=%d d=3" % k] = peaks_latency(e3, "max", k, 3)
        lat["W=65536 max k=%d d=50" % k] = peaks_latency(e3, "max", k, 50)
    rec["peaks_latency"] = lat
    rec["peaks_cfg3_max_k2"] = [(int(p["column"]), float(p["freq_hz"])) for p in e3.trace_peaks("max", k=2)]
    e3.close()
    eng.close()
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
