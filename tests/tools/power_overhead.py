#!/usr/bin/env python
"""What the channel-power set costs (DESIGN 3.11), on the GPU.

bench.py's cfg2 configuration (uint8 IQ, mode fast, pipelined batches, 512 frames per
step, EMA 0.3) timed with the power set off and on (3 bands: the main channel and its two
neighbours), legs alternated in one process over the same K steps, with CUDA events on the
engine's stream.  A third leg has the trace set on instead: one small launch per group on
the same finishing stream, the yardstick for what any one-launch row set costs there.  The
rows of the last step of every leg must be the same bit for bit in all three legs.  The
power kernel's own device time per cfg2 step comes from the engine's profile (class 18,
plain path, set off and on).  Then the measurement's own device time at cfg3's width (crop=None,
W = 65536, one whole-row band, 16 frames per step), from the engine's profile (class 18
with the set off and on), and the host-to-host latency of power_log for 4096 rows x 3
bands.  The card's name, power limit and maximum SM clock are read in the same run.

    python tests/tools/power_overhead.py [--steps 40] [--reps 5] [--out profiles/power_overhead.jsonl]
"""
from __future__ import annotations

import argparse
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "power_overhead.jsonl"))
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
    chans = [(-6000.0, -2000.0), (-2000.0, 2000.0), (2000.0, 6000.0)]     # 12.5 kHz wide rows

    def step():
        eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())

    def leg(on):
        eng.traces_enable(on == "traces")
        if on is True:
            eng.power_enable(chans, log_rows=4096)
        else:
            eng.power_disable()
        eng.reset_ema()
        for _ in range(args.warmup):
            step()
        eng.join()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(K):
            step()
        eng.join()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) / K, d_rows.cpu().numpy(), eng.power_count

    rec = {"what": "cfg2 fast pipelined, ms per step, power set off vs on (3 bands)", "card": info, "frames": F,
           "steps": K, "reps": args.reps, "bands_hz": chans}
    ms = {False: [], True: [], "traces": []}
    rows, count = {}, 0
    for _rep in range(args.reps):
        for on in (False, True, "traces"):
            t, r, c = leg(on)
            ms[on].append(t)
            if on in rows:
                assert np.array_equal(rows[on], r, equal_nan=True)
            rows[on] = r
            count = c if on is True else count
    assert np.array_equal(rows[False], rows[True], equal_nan=True), "the power set changed the rows"
    assert np.array_equal(rows[False], rows["traces"], equal_nan=True)
    eng.traces_enable(False)
    off, on = float(np.median(ms[False])), float(np.median(ms[True]))
    rec["cfg2"] = {"ms_off": ms[False], "ms_on": ms[True], "median_off": off, "median_on": on,
                   "overhead_pct": 100.0 * (on - off) / off,
                   "input_gsps_off": F * w.frame_len / (off * 1e-3) / 1e9,
                   "input_gsps_on": F * w.frame_len / (on * 1e-3) / 1e9,
                   "rows_measured_last_leg": count, "rows_bit_identical": True,
                   "ms_traces": ms["traces"], "median_traces": float(np.median(ms["traces"])),
                   "traces_overhead_pct": 100.0 * (float(np.median(ms["traces"])) - off) / off}

    # the power kernel's own device time per cfg2 step (plain path: the profile's events sit on one stream)
    def configure():
        eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                      f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode="fast")

    eng.set_option("pipeline", 0)
    configure()
    eng.set_profiling(True)
    for on in (False, True):
        if on:
            eng.power_enable(chans, log_rows=4096)
        for _ in range(3):
            step()
        eng.synchronize()
        eng.profile()
        k0 = eng.counters()["kernels"]
        for _ in range(10):
            step()
        eng.synchronize()
        p = eng.profile().get("finalize", (0.0, 0))
        key = "on" if on else "off"
        rec["cfg2_finalize_ms_per_step_%s" % key] = p[0] / 10
        rec["cfg2_launches_per_step_%s" % key] = (eng.counters()["kernels"] - k0) / 10
    eng.set_profiling(False)
    eng.set_option("pipeline", 1)
    configure()
    rec["cfg2_power_ms_per_step"] = rec["cfg2_finalize_ms_per_step_on"] - rec["cfg2_finalize_ms_per_step_off"]
    assert count == (K + args.warmup) * F

    # latency, host to host: the whole log of 4096 rows x 3 bands (the set is on, its log full)
    eng.power_enable(chans, log_rows=4096)
    for _ in range(-(-4096 // F)):
        step()
    eng.join()
    assert eng.power_count >= 4096

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

    first = eng.power_count - 4096
    assert len(eng.power_log(first, 4096)) == 4096
    rec["latency"] = {"power_log 4096 x 3": latency(lambda: eng.power_log(first, 4096)),
                      "power_summary 3": latency(eng.power_summary)}
    eng.power_disable()

    # cfg3's rows: crop=None, W = 65536, one whole-row band, 16 frames of 2^20 samples per step
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
    for on in (False, True):
        if on:
            e3.power_enable([(0, e3.row_width)], units="cols")
        k0 = e3.counters()["kernels"]
        for _ in range(n3):
            step3()
        e3.synchronize()
        p = e3.profile().get("finalize", (0.0, 0))
        key = "on" if on else "off"
        rec["cfg3_W65536_16frames_finalize_ms_per_step_%s" % key] = p[0] / n3
        rec["cfg3_W65536_16frames_launches_per_step_%s" % key] = (e3.counters()["kernels"] - k0) / n3
    e3.set_profiling(False)
    rec["cfg3_W65536_16frames_power_ms_per_step"] = (rec["cfg3_W65536_16frames_finalize_ms_per_step_on"]
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
