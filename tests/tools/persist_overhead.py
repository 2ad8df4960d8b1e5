#!/usr/bin/env python
"""What the decaying persistence spectrum costs (DESIGN 3.9), on the GPU.

bench.py's cfg2 configuration (uint8 IQ, mode fast, pipelined batches, 512 frames per
step, EMA 0.3) timed with the set off and on, legs alternated in one process over the
same K steps, with CUDA events on the engine's stream; the rows of the last step of
every leg must be the same bit for bit.  Then the update's own device time at cfg2's
width (W = 256) and at cfg3's (crop=None, W = 65536), from the engine's profile (class
18, finalisation, with the set off and on), and the latency of one U8 persistence image,
host to host, at 256 x 256 and 256 x 65536.  The card's name, power limit and maximum SM
clock are read in the same run.

    python tests/tools/persist_overhead.py [--steps 40] [--reps 5] [--out profiles/persist_overhead.jsonl]
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

LEVELS = (-240.0, -40.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "persist_overhead.jsonl"))
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
        eng.persistence_enable(on, levels=LEVELS, decay=0.99)
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
            assert eng.persistence_count == (args.warmup + K) * F
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
    assert np.array_equal(rows[False], rows[True]), "the persistence set changed the rows"
    off, on = float(np.median(ms[False])), float(np.median(ms[True]))
    rec = {"what": "cfg2 fast pipelined, ms per step, persistence off vs on (decay 0.99)", "card": info,
           "frames": F, "steps": K, "reps": args.reps, "ms_off": ms[False], "ms_on": ms[True],
           "median_off": off, "median_on": on, "overhead_pct": 100.0 * (on - off) / off,
           "cell_updates_per_step": 256 * W * F,
           "input_gsps_off": F * w.frame_len / (off * 1e-3) / 1e9, "input_gsps_on": F * w.frame_len / (on * 1e-3) / 1e9}

    def finalize_ms(e, run, label, n=10):
        """device time of class 18 per step with the set off and on: the difference is the update"""
        e.set_profiling(True)
        e.profile()
        for on_ in (False, True):
            e.persistence_enable(on_, levels=LEVELS, decay=0.99)
            for _ in range(n):
                run()
            e.synchronize()
            p = e.profile().get("finalize", (0.0, 0))
            rec["%s_finalize_ms_per_step_%s" % (label, "on" if on_ else "off")] = p[0] / n
            rec["%s_finalize_launches_per_step_%s" % (label, "on" if on_ else "off")] = p[1] / n
        e.set_profiling(False)
        rec["%s_update_ms_per_step" % label] = (rec["%s_finalize_ms_per_step_on" % label]
                                               - rec["%s_finalize_ms_per_step_off" % label])

    def step2():
        eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
        eng.join()

    finalize_ms(eng, step2, "cfg2_W256_512frames")

    def image_latency(e, n_calls=100):
        for _ in range(10):
            e.persistence_image("u8", levels=(0.0, 50.0))
        ts = []
        for _ in range(n_calls):
            t0 = time.perf_counter()
            e.persistence_image("u8", levels=(0.0, 50.0))
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        return {"median_us": float(np.median(ts)), "p90_us": float(np.percentile(ts, 90))}

    eng.persistence_enable(True, levels=LEVELS, decay=0.99)
    step2()
    lat = {"u8 256 x %d" % W: image_latency(eng)}
    eng.persistence_enable(False)

    # cfg3's rows: crop=None, W = 65536, 16 frames of 2^20 samples per step
    w3 = synth.CFG3
    e3 = ZoomPSD(0)
    e3.configure(w3.fs, w3.fft_size, w3.fft_ratio, w3.frame_len, w3.window, crop=w3.crop, mode="exact")
    assert e3.row_width == 65536
    F3 = 16
    d_in3 = torch.from_numpy(synth.make_frames(w3, F3, distinct=4)).cuda()
    d_rows3 = torch.empty((F3, e3.row_width), dtype=torch.float32, device="cuda")
    e3.set_stream(stream.cuda_stream)

    def step3():
        e3.process_device(d_in3.data_ptr(), F3, d_rows3.data_ptr())

    for _ in range(3):
        step3()
    finalize_ms(e3, step3, "cfg3_W65536_16frames")
    rec["cfg3_cell_updates_per_step"] = 256 * 65536 * F3
    e3.persistence_enable(True, levels=LEVELS, decay=0.99)
    step3()
    lat["u8 256 x 65536"] = image_latency(e3)
    rec["image_latency"] = lat
    e3.close()
    eng.close()
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
