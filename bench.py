#!/usr/bin/env python
"""bench.py -- input Msamples/s through the zoom-FFT PSD path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload cfg2|cfg1|cfg3|cfg4] [--frames F] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of F synthetic frames of
the workload (default: BASELINE.json configs[1], the RTL-SDR uint8 replay).
``value`` is measured over exactly K steps with the batch already resident in
HBM and no profiling events between the kernels; ``e2e`` goes
through the public host API (pinned host buffers, H2D + D2H inside the timed
region).  For N > 1 launch with torch.distributed.run: one rank per GPU, every
rank processes its own F frames (weak scaling, no data-path collective) and
the finished rows are gathered to rank 0 over NCCL inside the timed region.

``--dump-outputs DIR`` writes the rows the last timed step returned (gathered
on rank 0 for N > 1) to DIR/rows.npy as float32.  The frames are generated
from fixed seeds, so two builds run with the same arguments can be compared
row for row.

``--impl reference`` times the reference's own CPU arithmetic (the oracle
port: the same scipy.signal.decimate / welch calls, oracle/zoompsd_oracle.py)
on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pypanadapter_b200 import synth  # noqa: E402  (pure numpy)

METRIC = "input Msamples/s through zoom-FFT PSD"
UNIT = "Msamples/s"
HBM_FALLBACK_GBS = 6650.0


# --------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (fork pool, before any CUDA use)
# --------------------------------------------------------------------------
_cpu_frames = None
_cpu_w = None


def _cpu_one(i):
    from oracle import zoompsd_oracle as zo
    w = _cpu_w
    f = _cpu_frames[i % len(_cpu_frames)]
    row = zo.zoom_psd(f, w.fs, w.fft_size, w.fft_ratio, w.window, f_demod=w.f_demod,
                      crop=w.crop, flip=w.flip)
    return float(row[0])


def cpu_throughput(w, nframes_total, workers):
    """Msamples/s of the oracle port over ``nframes_total`` independent frames
    spread over ``workers`` forked processes (wall clock)."""
    import multiprocessing as mp
    global _cpu_frames, _cpu_w
    _cpu_w = w
    _cpu_frames = [synth.make_frame(w, i) for i in range(4)]
    _cpu_one(0)                                     # import + warm caches in the parent
    if workers <= 1:
        t0 = time.perf_counter()
        for i in range(nframes_total):
            _cpu_one(i)
        dt = time.perf_counter() - t0
    else:
        ctx = mp.get_context("fork")
        with ctx.Pool(workers) as pool:
            pool.map(_cpu_one, range(workers))      # start-up outside the timed region
            t0 = time.perf_counter()
            pool.map(_cpu_one, range(nframes_total), chunksize=max(1, nframes_total // (workers * 4)))
            dt = time.perf_counter() - t0
    return nframes_total * w.frame_len / dt / 1e6, dt


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def workload_config(w, frames):
    return {
        "workload": "%s: %s" % (w.name, w.description),
        "fs": w.fs, "fft_size": w.fft_size, "fft_ratio": w.fft_ratio, "frame_len": w.frame_len,
        "window": w.window if isinstance(w.window, str) else list(w.window),
        "sample_dtype": w.dtype, "flip": w.flip, "ema_alpha": w.ema_alpha,
        "row_width": w.row_width, "frames_per_step_per_gpu": frames,
    }


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_cores()
    # per step: a bounded sample of the workload sized for ~2-4 s of wall time
    per_core = max(1, int(round(2.5 / 0.1)) // 4)
    frames = cores * per_core
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt = cpu_throughput(w, frames, cores)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    sample = "%d frames of %d samples per step (%d per core), %d processes" % (
        frames, w.frame_len, per_core, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(w, frames),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock + clock-event reasons of one GPU while the timed regions run, sampled by
    `nvidia-smi -lms` in its OWN process (B200_PROFILING.md's clocks line): an NVML thread
    inside this process gets one sample per region -- its queries queue behind the kernel
    launches on the driver's locks."""
    REASONS = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown",
    }

    def __init__(self, uuid, index, period_ms=50):
        import subprocess
        self.samples = []        # (unix time, sm_mhz, reasons_mask, power_w)
        self.max_mhz = None
        self.proc = None
        self.err = None
        self._lines = []
        sel = uuid if (isinstance(uuid, str) and len(uuid) > 8) else str(index)
        cmd = ["nvidia-smi", "-i", sel,
               "--query-gpu=timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.active,power.draw",
               "--format=csv,noheader,nounits", "-lms", str(int(period_ms))]
        try:
            self.proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception as exc:          # pragma: no cover
            self.err = repr(exc)
        self._thread = threading.Thread(target=self._pump, daemon=True)

    def start(self):
        if self.proc is not None:
            self._thread.start()

    def _pump(self):
        import datetime
        for ln in self.proc.stdout:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 5:
                continue
            try:
                t = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                mask = int(f[3], 16) if f[3].lower().startswith("0x") else 0
                self.samples.append((t, float(f[1]), mask, float(f[4]) if f[4][:1].isdigit() else 0.0))
                self.max_mhz = float(f[2])
            except ValueError:
                continue

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        """t0, t1: time.time() bounds of the region"""
        inside = [x for x in list(self.samples) if t0 <= x[0] <= t1]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": self.err or "no nvidia-smi sample fell inside the region"}
        mask = 0
        for x in inside:
            mask |= x[2]
        reasons = [name for bit, name in self.REASONS.items() if mask & bit]
        return {"sm_mhz": float(np.median([x[1] for x in inside])), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside),
                "power_w_max": max(x[3] for x in inside)}


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def algorithmic_flops(w, eng, nch=1):
    """Algorithmic fp32 FLOP per INPUT sample of the chain as planned (SURVEY 8d):
    conversion, LO mix, the decimator structure actually run (FIR taps as designed, the
    zero-phase IIR in the form the kernels evaluate), Welch (FFT 10*log2(N)/R at 50 %
    overlap, detrend + window + |.|^2 + accumulate 24/R).  A real coefficient times a
    complex sample is 2 multiply-adds = 4 FLOP.  Returned per part; with ``nch`` virtual
    receivers everything but the conversion is per channel."""
    R = max(1, int(w.fft_ratio))
    k = int(np.log2(R))
    parts = {"convert_u8": 2.0 if w.dtype == "u8" else 0.0}
    parts["lo_mix"] = 0.0 if k == 0 else 8.0
    dec = {}
    if k > 0 and eng.fast_active:
        plan = eng.fast_plan
        for s_, taps in enumerate(plan["stages"]):
            ntaps = 2 * (len(taps) - 1) + 1
            dec["fir_stage%d(%d taps)" % (s_, ntaps)] = 4.0 * ntaps / 2 ** (s_ + 1)
        ne = len(plan["stages"])
        dec["compensator(%d taps)" % (2 * (len(plan["comp"]) - 1) + 1)] = 4.0 * (2 * (len(plan["comp"]) - 1) + 1) / 2 ** ne
        # causal + anti-causal order-8 recursion (2 x 8 packed FMAs) + 9-tap numerators at the kept samples
        dec["iir_last_stage"] = 4.0 * 25.0 / 2 ** ne
        parts["lo_mix"] = 8.0 / 2 ** ne if getattr(eng, "late_mix_active", True) and abs(w.f_demod) * R / w.fs <= 1e-3 else 8.0
    elif k > 0:
        for s_ in range(k):                       # all-pole sweeps twice (hand-off) + binomial numerators
            dec["iir_stage%d" % s_] = 4.0 * 44.5 / 2 ** s_
    parts.update(dec)
    parts["welch_fft"] = 10.0 * np.log2(w.fft_size) / R
    parts["welch_other"] = 24.0 / R
    per_channel = sum(v for n_, v in parts.items() if n_ != "convert_u8")
    total = parts["convert_u8"] + nch * per_channel
    return total, parts


def ncu_traffic(workload, kernel, frames_per_launch):
    """Per-launch DRAM bytes (read + write) of the dominant kernel, from the
    committed ncu --set full capture (profiles/roofline_traffic.json holds it
    per frame; a launch processes ``frames_per_launch`` frames), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            rec = json.load(f).get(workload, {}).get(kernel)
        return None if rec is None else rec["dram_bytes_per_frame"] * frames_per_launch
    except Exception:
        return None


DUMP_MAX_BYTES = 60 * 10**6          # rows.npy stays under 64 MB, header included


def dump_rows(path, rows):
    """``path``/rows.npy: float32 rows, or -- past DUMP_MAX_BYTES -- a fixed, seeded sample of
    whole rows kept in their order (the same rows for the same arguments)."""
    if rows.nbytes > DUMP_MAX_BYTES:
        keep = DUMP_MAX_BYTES // rows[0].nbytes
        rows = rows[np.sort(np.random.default_rng(0).choice(len(rows), keep, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "rows.npy"), np.ascontiguousarray(rows, dtype=np.float32))


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------
def run_b200(args, w):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    F = args.frames

    # CPU baseline first: it forks, which must happen before CUDA is touched
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        per_core = 32                   # ~20 s of CPU work in all (16 cores x 1.4 s; 12 per core was 8.7 core-seconds)
        v, dt = cpu_throughput(w, cores * per_core, cores)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "%d frames of %d samples (%d per core) through the oracle port "
                                  "(scipy decimate/welch), %.1f s wall" % (cores * per_core, w.frame_len,
                                                                            per_core, dt)}

    import torch
    import torch.distributed as dist
    from pypanadapter_b200.engine import ZoomPSD

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    host_affinity = None
    if world > 1 and not args.no_numa_bind:
        # one process per GPU: sit on the CPUs (hence the memory) of this GPU's NUMA node before
        # any pinned staging buffer is allocated
        from pypanadapter_b200 import dist as zdist0
        pr = torch.cuda.get_device_properties(local_rank)
        try:
            bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            host_affinity = zdist0.bind_host_to_gpu(bus)
            host_affinity["gpu"] = bus
        except Exception as exc:                      # never let placement stop a run
            host_affinity = {"bound": False, "why": repr(exc)}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a mismatch between ranks must end the run in minutes, not hold the GPUs for the default 10
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=180))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.lib:        # tuning experiments: an alternative sm_100a build of the same sources
        from pypanadapter_b200 import _lib
        alt = _lib.load_library(args.lib)
        assert alt.zfb_build_kind() == b"sm_100a"
        eng = ZoomPSD(local_rank, lib=alt)
    else:
        eng = ZoomPSD(local_rank)
    if args.group:
        eng.set_group(args.group)
    if args.decim_threads:
        eng.set_option("decim_threads", args.decim_threads)
    if args.welch_splits:
        eng.set_option("welch_splits", args.welch_splits)
    if args.strips_async is not None:
        eng.set_option("strips_async", args.strips_async)
    if args.late_mix is not None:
        eng.set_option("late_mix", args.late_mix)
    if args.slabs is not None:
        eng.set_option("slabs", args.slabs)
    # pipelined batches: zfb_process_device returns without making `stream` wait for the rows; the
    # bench joins (zfb_join) where something consumes them -- the NCCL gather, the end of a timed leg
    # (auto: on for 1- and 2-byte wire formats; complex64 input loses -- cfg1 166.7 -> 147.9 Gs/s, the two
    # lanes' streams evict each other from L2 -- profiles/r02ac_*)
    # cfg4 (64 virtual receivers: 64x the compute per byte, launches that fill the GPU): no change, 205.1 vs
    # 204.7 G channel-samples/s (profiles/r02ae_*) -- left off
    pipelined = args.pipeline == 1 or (args.pipeline < 0 and w.dtype in ("u8", "cs16"))
    eng.set_option("pipeline", 1 if pipelined else 0)
    for it in args.sets or []:
        name, _, val = it.partition("=")
        eng.set_option(name, int(val))
    eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                  f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode=args.mode)
    # a real (non-default) stream: the engine launches on it, NCCL enqueues on
    # it and the timing events are recorded on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)
    W = eng.row_width

    # BASELINE configs[3]: 64 virtual receivers over one stream, channels sharded across ranks
    centres = None
    if w.name == "cfg4":
        from pypanadapter_b200 import dist as zdist
        mine = zdist.channels_for_rank(64, rank, world)
        centres = synth.cfg4_centres()[mine.start:mine.stop]
    nch = 1 if centres is None else len(centres)
    host = synth.make_frames(w, F, distinct=min(F, 8))
    h_in = torch.from_numpy(host.view(np.uint8).reshape(F, -1)).pin_memory()
    h_rows = torch.empty((nch * F, W), dtype=torch.float32).pin_memory()
    d_in = h_in.cuda()
    # rows are double-buffered so that the NCCL gather of step k (side stream)
    # overlaps the kernels of step k+1
    d_rows2 = [torch.empty((nch * F, W), dtype=torch.float32, device="cuda") for _ in range(2)]
    d_rows = d_rows2[0]
    gather_list = [torch.empty_like(d_rows) for _ in range(world)] if (world > 1 and rank == 0) else None
    comm_stream = torch.cuda.Stream() if world > 1 else None
    rows_ready = [torch.cuda.Event() for _ in range(2)]
    gathered = [torch.cuda.Event() for _ in range(2)]
    step_no = [0]
    in_bytes = int(h_in.numel())
    frame_wire = host.reshape(F, -1)

    def gather_async(buf_idx):
        """rows of this step -> rank 0, on the side stream"""
        if pipelined and joinable[0]:
            eng.join(comm_stream.cuda_stream)        # the side stream waits for the rows, `stream` does not
        else:
            rows_ready[buf_idx].record(stream)
            comm_stream.wait_event(rows_ready[buf_idx])
        with torch.cuda.stream(comm_stream):
            dist.gather(d_rows2[buf_idx], gather_list, dst=0)
            gathered[buf_idx].record(comm_stream)

    joinable = [False]                               # the last engine call was a (pipelined) device batch

    def step_device():
        b = step_no[0] & 1
        step_no[0] += 1
        if world > 1:
            stream.wait_event(gathered[b])          # the gather that last read this buffer
        if centres is None:
            eng.process_device(d_in.data_ptr(), F, d_rows2[b].data_ptr())
        else:
            eng.process_channels_device(d_in.data_ptr(), F, centres, d_rows2[b].data_ptr())
        joinable[0] = True
        if world > 1:
            gather_async(b)

    def join_device():
        """`stream` waits for every batch handed to the engine (no-op unless pipelined)"""
        if pipelined:
            eng.join()

    h_in_np = h_in.numpy().view(frame_wire.dtype).reshape(frame_wire.shape)
    h_rows_np = h_rows.numpy()

    # cfg4 on several GPUs: every rank needs the SAME stream.  It crosses PCIe once (rank 0) and
    # reaches the other GPUs over NVLink (ncclBroadcast); only the rows come back per rank.
    # "allgather" (default): every rank H2Ds 1/N of the stream over its own PCIe link and the parts
    # are all-gathered over NVLink -- N links feed instead of one; "broadcast": rank 0 H2Ds all of it
    feed = args.cfg4_feed if (centres is not None and world > 1) else "replicate"
    if feed == "allgather" and F % world != 0:
        feed = "broadcast"
    bcast_feed = feed in ("broadcast", "allgather")       # the stream crosses PCIe once in all
    gather_feed = feed == "allgather"
    d_feed = torch.empty_like(d_in) if bcast_feed else None
    d_rows_e2e = torch.empty((nch * F, W), dtype=torch.float32, device="cuda") if bcast_feed else None
    Fs = F // world if gather_feed else F                  # frames this rank uploads

    def step_e2e():
        if gather_feed:
            d_feed[rank * Fs:(rank + 1) * Fs].copy_(h_in[rank * Fs:(rank + 1) * Fs], non_blocking=True)
            dist.all_gather_into_tensor(d_feed, d_feed[rank * Fs:(rank + 1) * Fs])     # in place, on `stream`
        elif bcast_feed:
            if rank == 0:
                d_feed.copy_(h_in, non_blocking=True)
            dist.broadcast(d_feed, src=0)            # on `stream` (the current stream)
            eng.process_channels_device(d_feed.data_ptr(), F, centres, d_rows_e2e.data_ptr())
            join_device()
            h_rows.copy_(d_rows_e2e, non_blocking=True)
            stream.synchronize()                     # rows are on the host, like eng.process()
        elif centres is None:                        # H2D + kernels + D2H, returns when rows are on the host
            eng.process(h_in_np, out=h_rows_np)
        else:
            eng.process_channels(h_in_np, centres, out=h_rows_np.reshape(nch, F, W))
        if world > 1:
            b = step_no[0] & 1
            step_no[0] += 1
            stream.wait_event(gathered[b])
            d_rows2[b].copy_(h_rows, non_blocking=True)
            joinable[0] = False
            gather_async(b)

    props = torch.cuda.get_device_properties(local_rank)
    uuid = "GPU-" + str(getattr(props, "uuid", ""))
    sampler = ClockSampler(uuid, local_rank)
    sampler.start()

    # ---------------- device-resident throughput: the K timed steps ----------------
    for _ in range(args.warmup):
        step_device()
    join_device()
    barrier()
    k0 = eng.counters()["kernels"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    join_device()                                   # the rows of every step belong to the timed region
    if world > 1:                                   # ... and so does the last gather
        stream.wait_event(gathered[(step_no[0] - 1) & 1])
    ev1.record(stream)
    barrier()
    t1 = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = eng.counters()["kernels"] - k0
    clocks = sampler.summary(t0 - 0.06, t1 + 0.06)     # K steps take milliseconds: the samples around them
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = (d_rows2[(step_no[0] - 1) & 1] if world == 1 else torch.cat(gather_list)).cpu().numpy()

    # ---------------- per-kernel times: K more steps with events around every kernel ----------------
    # (a pass of its own: the events are recorded between the kernels, so they stay out of the timed steps)
    eng.profile()
    eng.set_profiling(True)
    for _ in range(args.steps):
        step_device()
    join_device()
    barrier()
    eng.set_profiling(False)
    prof = eng.profile()

    # ---------------- end to end (host buffers) ----------------
    for _ in range(max(1, min(args.warmup, 3))):
        step_e2e()
    barrier()
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record(stream)
    for _ in range(e2e_steps):
        step_e2e()
    if world > 1:
        stream.wait_event(gathered[(step_no[0] - 1) & 1])
    ev3.record(stream)
    barrier()
    ms_e2e = ev2.elapsed_time(ev3)

    # ---------------- copy-only ceiling of the end-to-end leg ----------------
    # the same pinned buffers over the same PCIe link, no kernels: what e2e could reach at best
    copy_feeds = (rank == 0) if (bcast_feed and not gather_feed) else True
    d_copy = torch.empty_like(d_in)
    d_rows_c = d_rows2[0]

    def copy_step():
        if gather_feed:
            d_copy[rank * Fs:(rank + 1) * Fs].copy_(h_in[rank * Fs:(rank + 1) * Fs], non_blocking=True)
            dist.all_gather_into_tensor(d_copy, d_copy[rank * Fs:(rank + 1) * Fs])
        else:
            if copy_feeds:
                d_copy.copy_(h_in, non_blocking=True)
            if bcast_feed:
                dist.broadcast(d_copy, src=0)
        h_rows.copy_(d_rows_c, non_blocking=True)

    for _ in range(2):
        copy_step()
    barrier()
    ev4, ev5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev4.record(stream)
    for _ in range(e2e_steps):
        copy_step()
    ev5.record(stream)
    barrier()
    ms_copy = ev4.elapsed_time(ev5)
    del d_copy

    # ---------------- sustained leg: >= args.sustain_s seconds of back-to-back steps ----------------
    sustained = None
    if args.sustain_s > 0:
        n_sus = max(args.steps, int(np.ceil(args.sustain_s * 1e3 / max(ms / args.steps, 1e-3))))
        if world > 1:
            # every rank must issue the same number of gathers: take rank 0's count
            nt = torch.tensor([n_sus], dtype=torch.int64, device="cuda")
            dist.broadcast(nt, src=0)
            n_sus = int(nt.item())
        barrier()
        ev6, ev7 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts0 = time.time()
        ev6.record(stream)
        for i in range(n_sus):
            step_device()
            if (i & 63) == 63:
                join_device()
                stream.synchronize()                 # bound the launch queue; negligible against 64 steps
        join_device()
        if world > 1:
            stream.wait_event(gathered[(step_no[0] - 1) & 1])
        ev7.record(stream)
        barrier()
        ts1 = time.time()
        sustained = {"ms": ev6.elapsed_time(ev7), "steps": n_sus, "clocks": sampler.summary(ts0, ts1)}
    sampler.stop()

    # ---------------- per-kernel times with nothing overlapped (strips on the main stream, one lane) ----------
    lanes = eng.slab_lanes                   # lanes the timed batches ran through (2: slab pipelining)
    serial_prof = serial_step = None
    if world == 1 and eng.fast_active:
        eng.set_option("strips_async", 0)
        eng.set_option("slabs", 1)
        eng.set_option("pipeline", 0)
        eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                      f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode=args.mode)
        for _ in range(2):
            step_device()
        barrier()
        eng.profile()
        eng.set_profiling(True)
        for _ in range(5):
            step_device()
        barrier()
        eng.set_profiling(False)
        serial_raw = eng.profile()
        serial_prof = {k: v[0] / max(1, v[1]) for k, v in serial_raw.items()}
        serial_step = {k: v[0] / 5.0 for k, v in serial_raw.items()}      # ms per step, all launches of the class
        eng.set_option("strips_async", 1 if args.strips_async is None else args.strips_async)
        eng.set_option("slabs", 1 if args.slabs is None else args.slabs)
        eng.set_option("pipeline", 1 if pipelined else 0)

    # ---------------- N > 1: the gathered rows ARE the single-GPU rows, bit for bit ----------------
    # frames are independent (LO phase, filter state and Welch mean restart per chunk: S:2092, 2098,
    # 2111): rank r computes frames [r*Fv, (r+1)*Fv) of one list, rank 0 also computes all of them
    verify = None
    if world > 1 and centres is None:
        Fv = min(F, 48)
        allf = synth.make_frames(w, world * Fv, distinct=world * Fv)
        eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                      f_demod=w.f_demod, crop=w.crop, ema_alpha=None, mode=args.mode)
        mine = torch.from_numpy(allf[rank * Fv:(rank + 1) * Fv].view(np.uint8).reshape(Fv, -1)).cuda()
        rows_mine = torch.empty((Fv, W), dtype=torch.float32, device="cuda")
        eng.process_device(mine.data_ptr(), Fv, rows_mine.data_ptr())
        eng.join()
        glist = [torch.empty_like(rows_mine) for _ in range(world)] if rank == 0 else None
        dist.gather(rows_mine, glist, dst=0)
        stream.synchronize()
        if rank == 0:
            everything = torch.from_numpy(allf.view(np.uint8).reshape(world * Fv, -1)).cuda()
            rows_all = torch.empty((world * Fv, W), dtype=torch.float32, device="cuda")
            eng.set_option("pipeline", 0)            # the plain path on one GPU is the yardstick
            eng.process_device(everything.data_ptr(), world * Fv, rows_all.data_ptr())
            stream.synchronize()
            got = torch.cat(glist, 0).cpu().numpy()
            want = rows_all.cpu().numpy()
            verify = {"frames": world * Fv, "rows_equal_single_gpu": bool(np.array_equal(got, want)),
                      "max_abs_diff": float(np.max(np.abs(got - want)))}

    ms_sus = sustained["ms"] if sustained else 0.0
    t = torch.tensor([ms, ms_e2e, float(launches), ms_copy, ms_sus], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, ms_e2e, launches, ms_copy, ms_sus = (float(tmax[0]), float(tmax[1]), int(tsum[2]), float(tmax[3]),
                                                 float(tmax[4]))
    samples_step = world * F * w.frame_len * nch      # cfg4: channel-samples (every channel consumes the stream)
    value = samples_step * args.steps / (ms * 1e-3) / 1e6
    e2e_value = samples_step * e2e_steps / (ms_e2e * 1e-3) / 1e6
    copy_value = samples_step * e2e_steps / (ms_copy * 1e-3) / 1e6
    if sustained:
        sus_value = samples_step * sustained["steps"] / (ms_sus * 1e-3) / 1e6
        sustained.update(value=sus_value, unit=UNIT, seconds=ms_sus * 1e-3, ratio_to_value=sus_value / value)

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        # Dominant kernel: largest share of device time in the timed region.  The edge strips of
        # mode fast run on a side stream beside the other kernels, so their event interval is not
        # exclusive; they are ranked by their time in the serialised pass below (kernel_ms_serial).
        names = {"decimate_stage15": "edge_strips"}
        exclusive = {k: v for k, v in prof.items() if k != "decimate_stage15"} or prof
        if serial_prof:
            top = max(serial_prof, key=lambda k: serial_prof[k] if k in exclusive else -1.0)
        else:
            # N > 1: the same kernel as at N = 1 (the FIR chain / stage 0 / the R = 1 Welch), whose
            # interval holds no wait on another stream
            top = "decimate_stage0" if "decimate_stage0" in exclusive else max(exclusive, key=lambda k: exclusive[k][0])
        top_ms, top_n = prof[top]
        # algorithmic bytes (SURVEY 8d): every input sample read ONCE -- not once per virtual receiver,
        # not per overlap re-read, not per stage; rows 4*W (x3 with EMA: read-modify-write of the state)
        row_bytes = 4 * W * (3 if w.ema_alpha is not None else 1)
        frame_bytes = w.frame_len * w.bytes_per_sample + nch * row_bytes
        if top.startswith("decimate_stage") and top not in ("decimate_stage0",):
            s_ = int(top[len("decimate_stage"):])
            algo_launch = F * nch * (w.frame_len >> s_) * 8 / max(1, top_n // args.steps)
        else:
            algo_launch = F * w.frame_len * w.bytes_per_sample / max(1, top_n // args.steps)
        avg_launch_ms = top_ms / max(1, top_n)
        achieved = algo_launch / (avg_launch_ms * 1e-3) / 1e9
        step_ms = ms / args.steps
        roofline = {
            "bound": "hbm", "kernel": names.get(top, top), "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak,
            "traffic": ncu_traffic(w.name, top, F / max(1, top_n // args.steps)), "peak_source": peak_src,
            "launches": top_n, "avg_launch_ms": avg_launch_ms,
            "algorithmic_bytes_per_launch": algo_launch,
            "kernel_share_of_step": top_ms / ms,
            "kernel_ms": {names.get(k, k) + ("(concurrent)" if k == "decimate_stage15" else ""): round(v[0], 4)
                          for k, v in prof.items()},
            "kernel_ms_serial_per_launch": None if serial_prof is None else
                {names.get(k, k): round(v, 5) for k, v in serial_prof.items()},
            "lanes": lanes,
            "step_algorithmic_bytes": F * frame_bytes,
            "step_achieved_gbs": world * F * frame_bytes / (step_ms * 1e-3) / 1e9,
            "step_frac": F * frame_bytes / (step_ms * 1e-3) / 1e9 / peak,
        }
        if serial_step and top in serial_step and serial_step[top] > 0:
            # the same kernel with the GPU to itself (one lane, strips on the main stream, 5 steps after
            # the timed legs): with two slab lanes its interval in the timed region above is shared with
            # the other lane's last stage / strips / Welch, so `achieved` there is a lower bound
            ex_ms = serial_step[top]
            step_bytes_top = algo_launch * max(1, top_n // args.steps)
            roofline["exclusive"] = {"ms_per_step": ex_ms, "achieved": step_bytes_top / (ex_ms * 1e-3) / 1e9,
                                     "frac": step_bytes_top / (ex_ms * 1e-3) / 1e9 / peak,
                                     "what": "all launches of this kernel for one step, nothing else running"}
            if lanes == 2:
                # pipelined batches: the kernel's event interval in the timed region is shared with the
                # other lane's kernels and says nothing about the kernel; the figure with the GPU to
                # itself is the roofline entry, the shared one is kept beside it
                roofline["timed_region_overlapped"] = {"achieved": roofline["achieved"], "frac": roofline["frac"],
                                                       "avg_launch_ms": roofline["avg_launch_ms"]}
                roofline["achieved"] = roofline["exclusive"]["achieved"]
                roofline["frac"] = roofline["exclusive"]["frac"]
                roofline["avg_launch_ms"] = ex_ms / max(1.0, serial_raw[top][1] / 5.0)
                roofline["avg_launch_ms_source"] = ("CUDA events around the kernel, 5 steps with nothing "
                                                    "overlapped, after the timed legs of this run")
        # the binding roofline: fp32 FMA pipe (SURVEY 8d "report both")
        flops_sample, flop_parts = algorithmic_flops(w, eng, nch)
        if clocks["sm_mhz"]:
            sm_mhz, mhz_src = clocks["sm_mhz"], "SM clock sampled around the timed steps"
        else:
            sm_mhz = clocks.get("sm_max_mhz") or 1965.0
            mhz_src = "maximum SM clock: no clock sample fell around the timed steps"
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        peak_tf = sms * 128 * 2 * sm_mhz * 1e6 / 1e12
        ach_tf = flops_sample * (F * w.frame_len) / (step_ms * 1e-3) / 1e12
        roofline_fp32 = {
            "bound": "fp32", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
            "peak_source": "%d SMs x 128 lanes x 2 FLOP x %.0f MHz (%s)" % (sms, sm_mhz, mhz_src),
            "algorithmic_flop_per_input_sample": flops_sample,
            "flop_parts_per_input_sample%s" % ("_per_channel" if nch > 1 else ""): {k: round(v, 3) for k, v in flop_parts.items()},
            "scope": "whole step, one GPU",
        }
        cfg = workload_config(w, F)
        cfg["l2"] = "inputs larger than L2: %.0f MB per step per GPU" % (in_bytes / 1e6)
        cfg["parallelism"] = "frames sharded, %d rank(s), rows gathered to rank 0 over NCCL" % world
        cfg["group_frames"] = args.group or "auto"
        cfg["decim_threads"] = args.decim_threads or "auto"
        if centres is not None:
            cfg["stream_feed"] = {"allgather": "every rank H2Ds 1/N of the stream, NCCL all-gather over NVLink",
                                  "broadcast": "rank 0 H2D + NCCL broadcast over NVLink",
                                  "replicate": "H2D on every rank"}[feed]
            cfg["channels_per_gpu"] = nch
            cfg["value_counts"] = "channel-samples: every virtual receiver consumes the whole stream"
        cfg["decimator_mode"] = "fast" if eng.fast_active else "exact"
        cfg["slab_lanes"] = lanes
        cfg["pipelined_batches"] = pipelined
        if host_affinity is not None:
            cfg["host_affinity_rank0"] = host_affinity
        h2d_step = in_bytes if bcast_feed else world * in_bytes
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "rows_per_s": world * nch * F * args.steps / (ms * 1e-3),
            "sustained": sustained,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_step,
                    "d2h_bytes_per_step": world * nch * F * W * 4, "steps": e2e_steps,
                    "ms_per_step": ms_e2e / e2e_steps,
                    "copy_only": {"value": copy_value, "unit": UNIT, "ms_per_step": ms_copy / e2e_steps,
                                  "h2d_gbs": h2d_step / (ms_copy / e2e_steps * 1e-3) / 1e9,
                                  "what": "the same pinned buffers over PCIe%s, no kernels"
                                          % (" + the NCCL all-gather" if gather_feed else
                                             " + the NCCL broadcast" if bcast_feed else "")},
                    "e2e_over_copy_only": e2e_value / copy_value},
            "gpu_launches": launches,
            "roofline": roofline,
            "roofline_fp32": roofline_fp32,
            "reference_arm_note": "bench.py --impl reference runs the scipy port without the EMA (one "
                                  "multiply-add per row bin: negligible)",
        }
        if verify is not None:
            line["multi_gpu_check"] = verify
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if dumped is not None:
            dump_rows(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--frames", type=int, default=None,
                    help="frames per step per GPU (default: 512 for cfg1/cfg2, 64 for cfg3, 8 for cfg4)")
    ap.add_argument("--group", type=int, default=0, help="frames per launch group (0 = auto)")
    ap.add_argument("--decim-threads", type=int, default=0, help="tuning: 0 auto, 128 or 256")
    ap.add_argument("--mode", default="fast", choices=["exact", "fast"],
                    help="decimator: exact zero-phase IIR everywhere, or polyphase-FIR interior + exact edges")
    ap.add_argument("--welch-splits", type=int, default=0, help="tuning: CTAs per frame in the Welch kernel")
    ap.add_argument("--strips-async", type=int, default=None, help="tuning: 0 = edge strips on the main stream")
    ap.add_argument("--late-mix", type=int, default=None, help="tuning: 0 = always mix before the FIR chain")
    ap.add_argument("--slabs", type=int, default=None,
                    help="tuning: 2 = cut every batch into slabs across two lane engines (default 1: one lane)")
    ap.add_argument("--pipeline", type=int, default=-1,
                    help="1: batches alternate between the engine's two lanes, rows joined where they are "
                         "consumed (zfb_join); 0: every batch ordered on the bench stream at once; "
                         "-1 (default): 1 for uint8 / int16 IQ, 0 for complex64")
    ap.add_argument("--set", action="append", dest="sets", metavar="OPTION=VALUE", help="tuning: zfb_set_option")
    ap.add_argument("--lib", default=None, help="tuning: path of an alternative sm_100a build")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--sustain-s", type=float, default=0.0,
                    help="seconds of back-to-back steps for a sustained leg reported beside the value "
                         "(default 0: none)")
    ap.add_argument("--cfg4-feed", default="allgather", choices=["allgather", "broadcast", "replicate"],
                    help="cfg4, N > 1: H2D on rank 0 + NCCL broadcast over NVLink, or H2D on every rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="N > 1: do not bind each rank to the CPUs of its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows of the last timed step to DIR/rows.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.warmup < 3:
        args.warmup = 3
    w = synth.WORKLOADS[args.workload]
    if args.frames is None:
        args.frames = {"cfg3": 64, "cfg4": 8}.get(w.name, 512)
    if args.impl == "reference":
        return run_reference(args, w)
    return run_b200(args, w)


if __name__ == "__main__":
    sys.exit(main())
