"""A/B measurement of engine tuning options (zfb_set_option) in ONE process, so
that a variant costs seconds of GPU time instead of a box:

    python -m tests.tools.ab --workload cfg2 --set strips_async=1,0 --set late_mix=1,0
    python -m tests.tools.ab --workload cfg1 --mode exact --set decim_threads=0,128,256

Every combination of the listed values is configured on the same engine and
timed on the device (CUDA events on the engine's stream, inputs larger than
L2, `--warmup` untimed steps), the combinations interleaved over `--rounds`
so that clock drift hits all alike.  Per combination one JSON line: ms per
step, Gsamples/s, per-kernel-class ms per launch from the engine's profile,
and whether its rows are bit-identical to the first combination's.  The last
line holds the best round of each.  Measurement tool (tests/), not product.
"""
from __future__ import annotations

import argparse
import itertools
import json

import numpy as np


def parse_sets(items):
    names, values = [], []
    for it in items or []:
        name, _, vals = it.partition("=")
        if not name or not vals:
            raise SystemExit("--set wants name=v1,v2,...: %r" % it)
        names.append(name)
        values.append([int(v) for v in vals.split(",")])
    return names, [dict(zip(names, combo)) for combo in itertools.product(*values)] or [{}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--mode", default="fast", choices=["fast", "exact"])
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--set", action="append", dest="sets", metavar="OPTION=V1,V2")
    args = ap.parse_args()
    names, combos = parse_sets(args.sets)

    import torch
    from pypanadapter_b200 import synth
    from pypanadapter_b200.engine import ZoomPSD

    w = synth.WORKLOADS[args.workload]
    F = args.frames or {"cfg3": 64, "cfg4": 8}.get(w.name, 512)      # bench.py's defaults
    host = synth.make_frames(w, F, distinct=min(F, 8))
    d_in = torch.from_numpy(host.view(np.uint8).reshape(F, -1)).cuda()
    eng = ZoomPSD(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)

    first_rows = None
    best = [None] * len(combos)
    for rnd in range(args.rounds):
        for ci, combo in enumerate(combos):
            for k, v in combo.items():
                eng.set_option(k, v)
            eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                          f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode=args.mode)
            d_rows = torch.empty((F, eng.row_width), dtype=torch.float32, device="cuda")
            for _ in range(args.warmup):
                eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
            torch.cuda.synchronize()
            eng.profile()
            eng.set_profiling(True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
            e1.record(stream)
            torch.cuda.synchronize()
            eng.set_profiling(False)
            prof = eng.profile()
            ms = e0.elapsed_time(e1) / args.steps
            eng.reset_ema()
            eng.process_device(d_in.data_ptr(), F, d_rows.data_ptr())
            torch.cuda.synchronize()
            rows = d_rows.cpu().numpy()
            if first_rows is None:
                first_rows = rows
            rec = dict(combo)
            rec.update(round=rnd, ms_per_step=ms, gsamples_per_s=F * w.frame_len / ms / 1e6,
                       fast_active=eng.fast_active,
                       ms_per_launch={k: round(t / max(n, 1), 5) for k, (t, n) in prof.items()},
                       rows_equal_to_first=bool(np.array_equal(rows, first_rows)),
                       max_abs_diff_to_first=float(np.nanmax(np.abs(np.where(np.isfinite(rows) & np.isfinite(first_rows),
                                                                              rows - first_rows, 0.0)))))
            if best[ci] is None or ms < best[ci]["ms_per_step"]:
                best[ci] = rec
            print(json.dumps(rec), flush=True)
    print(json.dumps({"workload": args.workload, "mode": args.mode, "frames": F, "best": best}), flush=True)


if __name__ == "__main__":
    main()
