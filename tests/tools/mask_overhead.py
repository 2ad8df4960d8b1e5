#!/usr/bin/env python
"""What the frequency-mask trigger costs (DESIGN 3.10), on the GPU.

bench.py's cfg2 configuration (uint8 IQ, mode fast, pipelined batches, 512 frames per
step, EMA 0.3) timed with the mask off and on, legs alternated in one process over the
same K steps, with CUDA events on the engine's stream, in two configurations:

  quiet   a line 20 dB above the highest value of any row: no row violates (no capture)
  bursts  5 seeded frames of the 512 (1 %) carry a tone burst; the line is the clean rows'
          per-column maximum plus the margin that about 5 rows of a step pass; 256 capture
          slots, the log reset every leg

The rows of the last step of every leg must be the same bit for bit with the mask off and
on.  Then the check + log's own device time at cfg3's width (crop=None, W = 65536, 16
frames per step), from the engine's profile (class 18 with the mask off and on), and the
host-to-host latency of mask_events (64 events) and of one cfg2 capture.  The card's name,
power limit and maximum SM clock are read in the same run.

    python tests/tools/mask_overhead.py [--steps 40] [--reps 5] [--out profiles/mask_overhead.jsonl]
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.tools.trace_overhead import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mask_overhead.jsonl"))
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
    host = synth.make_frames(w, F, distinct=min(F, 8))
    d_clean = torch.from_numpy(host).cuda()
    rng = np.random.default_rng(2026)
    burst_at = np.sort(rng.choice(F, size=max(1, F // 100), replace=False))
    wb = dataclasses.replace(w, tones=w.tones + ((1200.0, 0.2),))     # inside the 12.5 kHz row
    noisy = host.copy()
    for i in burst_at:
        noisy[i] = synth.make_frame(wb, int(i))
    d_burst = torch.from_numpy(noisy).cuda()
    d_rows = torch.empty((F, W), dtype=torch.float32, device="cuda")

    def step(d_in):
        eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())

    # the lines, from the clean rows (EMA settled)
    eng.reset_ema()
    for _ in range(4):
        step(d_clean)
    eng.join()
    clean = d_rows.cpu().numpy()
    quiet_line = np.float32(np.nanmax(clean[np.isfinite(clean)]) + 20.0)
    # the burst line: the clean rows' per-column maximum plus a margin that only as many rows of a
    # burst step pass as there are burst frames (the EMA carries a burst into the rows after it)
    cmax = np.max(clean, axis=0)
    eng.reset_ema()
    for _ in range(4):
        step(d_burst)
    eng.join()
    over = np.sort(np.max(d_rows.cpu().numpy() - cmax, axis=1))[::-1]
    nb = len(burst_at)
    margin = 0.5 * (over[nb - 1] + over[nb])
    burst_line = (cmax + np.float32(margin)).astype(np.float32)

    def leg(d_in, arm):
        if arm is None:
            eng.mask_disable()
        else:
            arm()
        eng.reset_ema()
        for _ in range(args.warmup):
            step(d_in)
        eng.join()
        if arm is not None:
            eng.mask_reset()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(K):
            step(d_in)
        eng.join()
        b.record(stream)
        b.synchronize()
        rows = d_rows.cpu().numpy()
        counts = eng.mask_counts if arm is not None else None
        return a.elapsed_time(b) / K, rows, counts

    configs = {
        "quiet": (d_clean, lambda: eng.mask_enable(quiet_line, max_events=4096)),
        "bursts": (d_burst, lambda: eng.mask_enable(burst_line, max_events=4096, capture=256)),
    }
    rec = {"what": "cfg2 fast pipelined, ms per step, frequency mask off vs on", "card": info, "frames": F,
           "steps": K, "reps": args.reps, "burst_frames": burst_at.tolist(), "burst_margin_db": float(margin)}
    for name, (d_in, arm) in configs.items():
        ms = {False: [], True: []}
        rows, counts = {}, None
        for _rep in range(args.reps):
            for on in (False, True):
                t, r, c = leg(d_in, arm if on else None)
                ms[on].append(t)
                if on in rows:
                    assert np.array_equal(rows[on], r, equal_nan=True)
                rows[on] = r
                counts = c if on else counts
        assert np.array_equal(rows[False], rows[True], equal_nan=True), "the mask changed the rows"
        off, on = float(np.median(ms[False])), float(np.median(ms[True]))
        rec[name] = {"ms_off": ms[False], "ms_on": ms[True], "median_off": off, "median_on": on,
                     "overhead_pct": 100.0 * (on - off) / off,
                     "input_gsps_off": F * w.frame_len / (off * 1e-3) / 1e9,
                     "input_gsps_on": F * w.frame_len / (on * 1e-3) / 1e9,
                     "rows_checked_last_leg": counts[0], "events_last_leg": counts[1],
                     "events_per_step": counts[1] / K}
    assert rec["quiet"]["events_last_leg"] == 0

    # latency, host to host: 64 events, one cfg2 capture (frame_len uint8 IQ samples)
    eng.mask_enable(burst_line, max_events=4096, capture=16)
    eng.reset_ema()
    for _ in range(40):
        step(d_burst)
        eng.join()
        if eng.mask_counts[1] >= 64:
            break
    assert eng.mask_counts[1] >= 64, eng.mask_counts

    def latency(fn, n_calls=100):
        for _ in range(10):
            fn()
        ts = []
        for _ in range(n_calls):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        return {"median_us": float(np.median(ts)), "p90_us": float(np.percentile(ts, 90))}

    rec["latency"] = {"mask_events 64": latency(lambda: eng.mask_events(0, 64)),
                      "mask_capture cfg2 (%d bytes)" % (2 * w.frame_len): latency(lambda: eng.mask_capture(3))}
    eng.mask_disable()

    # cfg3's rows: crop=None, W = 65536, 16 frames of 2^20 samples per step
    w3 = synth.CFG3
    e3 = ZoomPSD(0)
    e3.configure(w3.fs, w3.fft_size, w3.fft_ratio, w3.frame_len, w3.window, crop=w3.crop, mode="exact")
    assert e3.row_width == 65536
    F3, n3 = 16, 10
    d_in3 = torch.from_numpy(synth.make_frames(w3, F3, distinct=4)).cuda()
    d_rows3 = torch.empty((F3, e3.row_width), dtype=torch.float32, device="cuda")
    e3.set_stream(stream.cuda_stream)

    def step3():
        e3.process_device(d_in3.data_ptr(), F3, d_rows3.data_ptr())

    for _ in range(3):
        step3()
    e3.set_profiling(True)
    e3.profile()
    line3 = np.float32(400.0)
    for on in (False, True):
        if on:
            e3.mask_enable(line3)
        k0 = e3.counters()["kernels"]
        for _ in range(n3):
            step3()
        e3.synchronize()
        p = e3.profile().get("finalize", (0.0, 0))
        key = "on" if on else "off"
        rec["cfg3_W65536_16frames_finalize_ms_per_step_%s" % key] = p[0] / n3
        rec["cfg3_W65536_16frames_launches_per_step_%s" % key] = (e3.counters()["kernels"] - k0) / n3
    e3.set_profiling(False)
    rec["cfg3_W65536_16frames_check_log_ms_per_step"] = (rec["cfg3_W65536_16frames_finalize_ms_per_step_on"]
                                                         - rec["cfg3_W65536_16frames_finalize_ms_per_step_off"])
    e3.close()
    eng.close()
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
