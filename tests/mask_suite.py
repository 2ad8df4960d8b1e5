"""Frequency-mask trigger (DESIGN 3.10), shared by tests/test_mask.py on the CPU emulation
build and, marked gpu, on the B200.  Every function takes a ``ZoomPSD`` and, where device
pointers are needed, a device helper of tests/engine_suite.py (``HostAsDevice`` /
``TorchDevice``).  The oracle restates the mask's rules in numpy on the rows the engine
returned (float32 subtraction for the excess) and the engine's log must equal it field for
field, value and excess bit for bit."""
from __future__ import annotations

import ctypes as C
import types

import numpy as np
import pytest

from pypanadapter_b200 import _lib, synth
from pypanadapter_b200.buffers import PSD, Data
from pypanadapter_b200.engine import MASK_EVENT_DTYPE, ZoomFFTError, ZoomPSD
from tests import traces_suite as ts

N7 = ts.N7                          # cfg2's geometry with 7 Welch segments: the fp32 path, mode fast active
FIELDS = MASK_EVENT_DTYPE.names
DTYPE_CODES = {"c64": _lib.ZFB_DTYPE_C64, "u8": _lib.ZFB_DTYPE_U8, "cs16": _lib.ZFB_DTYPE_CS16}


# ---- the oracle ----------------------------------------------------------------------------------
def oracle_events(rows, upper=None, lower=None, min_cols=1, row0=0, k0=0, capture_slots=0,
                  capture_samples=0, frame_len=0, dtype=0):
    """The events of `rows` (float32 [n][W]) in frame order, event numbers from k0, rows from row0"""
    rows = np.asarray(rows, dtype=np.float32)
    W = rows.shape[1]
    nan = np.full(W, np.nan, dtype=np.float32)
    up = nan if upper is None else np.broadcast_to(np.asarray(upper, dtype=np.float32), (W,))
    lo = nan if lower is None else np.broadcast_to(np.asarray(lower, dtype=np.float32), (W,))
    out = []
    k = k0
    with np.errstate(all="ignore"):
        for i, v in enumerate(rows):
            a, b = v > up, v < lo
            viol = a | b
            if viol.sum() < min_cols:
                continue
            ea = np.where(a, v - up, np.float32(0)).astype(np.float32)
            eb = np.where(b, lo - v, np.float32(0)).astype(np.float32)
            above = a & ~(eb > ea)
            ex = np.where(viol, np.where(above, ea, eb), np.float32(-1))
            worst = int(np.argmax(ex))                     # first maximum: ties to the lower column
            cols = np.flatnonzero(viol)
            slot = k if k < capture_slots else -1
            out.append((row0 + i, len(cols), cols[0], cols[-1], worst, v[worst], ex[worst], int(above[worst]),
                        slot, min(frame_len, capture_samples) if slot >= 0 else 0, dtype))
            k += 1
    return np.array(out, dtype=MASK_EVENT_DTYPE)


def assert_events_equal(got, want, what=""):
    assert len(got) == len(want), (what, len(got), len(want))
    for name in FIELDS:
        g, w = np.asarray(got[name]), np.asarray(want[name])
        if g.dtype == np.float32:
            g, w = g.view(np.uint32), w.view(np.uint32)        # bit for bit, inf and all
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, (what, name, bad[:5], got[bad[:3]], want[bad[:3]])


def check_log(engine, rows, what="", **mask):
    """counts and the whole log against the oracle on `rows` (everything the log has seen)"""
    mask.setdefault("dtype", DTYPE_CODES[engine.dtype])
    want = oracle_events(rows, **mask)
    assert engine.mask_counts == (len(rows), len(want)), (what, engine.mask_counts, len(want))
    got = engine.mask_events()
    assert_events_equal(got, want, what)
    assert np.array_equal(got["freq_hz"], engine.row_frequencies()[want["worst_col"]]), what
    return want


def _errcode(fn, *a, **kw):
    with pytest.raises(ZoomFFTError) as ei:
        fn(*a, **kw)
    return ei.value.code


def _cfg2(engine, n=N7, mode="fast", ema=0.3, **kw):
    w = synth.CFG2
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n or w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", ema_alpha=ema, mode=mode, **kw)


def shapes(rows):
    """Mask shapes from the rows they will be checked against: (name, upper, lower, min_cols)"""
    r = np.where(np.isfinite(rows), rows, np.nan).astype(np.float32)
    srt = np.sort(np.where(np.isnan(r), -np.inf, r), axis=0)
    W = rows.shape[1]
    hi, lo = srt[-2].copy(), srt[1].copy()                   # one row above / below per column at most
    hi_nan, lo_nan = hi.copy(), lo.copy()
    hi_nan[::3] = np.nan
    lo_nan[::5] = np.nan
    lo_nan[1::7] = -np.inf
    hi_nan[2::11] = np.inf
    med = np.nanmedian(r, axis=0).astype(np.float32)
    return [("upper", hi, None, 1),
            ("lower", None, lo, 1),
            ("both, NaN and inf columns", hi_nan, lo_nan, 1),
            ("min_cols", med, None, max(2, W // 2))]


def _mask_kw(upper, lower, min_cols):
    return dict(upper=upper, lower=lower, min_cols=min_cols)


# ---- scenarios -----------------------------------------------------------------------------------
def off_changes_nothing(engine, nframes=5):
    """Off (the default, or enabled and then disabled): rows, ring and launch count as an engine
    that never heard of the mask, and every read is ESTATE.  On: the same rows bit for bit, at
    most 2 launches more per group, 3 with capture slots."""
    frames = synth.make_frames(synth.CFG2, nframes)

    def run(e, mode):
        _cfg2(e, n=None)
        if mode == "on-off":
            e.mask_enable(upper=-100.0, capture=2)
            e.mask_disable()
        elif mode == "on":
            e.mask_enable(upper=-150.0)
        elif mode == "on, capture":
            e.mask_enable(upper=-150.0, capture=2)
        e.reset_ema()
        k0 = e.counters()["kernels"]
        rows = np.concatenate([e.process(frames[:2]), e.process(frames[2:])])
        return rows, e.read_rows(nframes), e.counters()["kernels"] - k0

    with ZoomPSD(0, lib=engine._lib) as plain:
        want = run(plain, "never")
        for fn in (lambda: plain.mask_counts, plain.mask_events, lambda: plain.mask_capture(0), plain.mask_reset):
            assert _errcode(fn) == _lib.ZFB_ESTATE
    got = run(engine, "on-off")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]
    for fn in (lambda: engine.mask_counts, engine.mask_events, lambda: engine.mask_capture(0), engine.mask_reset):
        assert _errcode(fn) == _lib.ZFB_ESTATE
    lib, h = engine._lib, engine._h
    out2, n = (C.c_int64 * 2)(), C.c_int(0)
    buf = np.zeros(64, dtype=np.uint8)
    assert lib.zfb_mask_counts(h, out2) == _lib.ZFB_ESTATE
    assert lib.zfb_mask_events(h, 0, 1, C.c_void_p(buf.ctypes.data), C.byref(n)) == _lib.ZFB_ESTATE
    assert lib.zfb_mask_capture(h, 0, C.c_void_p(buf.ctypes.data), 0) == _lib.ZFB_ESTATE
    for mode, per_group in (("on", 2), ("on, capture", 3)):
        on = run(engine, mode)
        assert np.array_equal(on[0], want[0]) and np.array_equal(on[1], want[1]), mode
        extra = on[2] - want[2]
        assert extra > 0 and extra % per_group == 0 and extra <= per_group * nframes, (mode, extra)
        check_log(engine, on[0], mode, upper=-150.0, capture_slots=2 if "capture" in mode else 0,
                  capture_samples=engine.frame_len, frame_len=engine.frame_len, dtype=_lib.ZFB_DTYPE_U8)
    engine.mask_disable()
    assert _errcode(lambda: engine.mask_counts) == _lib.ZFB_ESTATE


def _samples_rows(engine, mask, nrows=4):
    """rows of zfb_samples_process, fed through buffers.Data / PSD.update"""
    w = synth.CFG1
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    rows = []
    for i in range(nrows):
        x = synth.make_frame(w, i, n=w.fft_size * 24)
        if i == 2:
            x = x * 3                                          # this row stands out
        for j in range(0, len(x), d.chunk_size):
            d.add(x[j:j + d.chunk_size])
        psd.update()
        if i == 0:
            engine.mask_enable(**mask(psd.psd.astype(np.float32)))   # after the configure of update()
        else:
            rows.append(psd.psd.astype(np.float32))
    return np.array(rows)


def exact_against_oracle(engine, dev):
    """The log, field for field, against the oracle on the rows the engine returned, on every
    path a row can take, for the mask shapes of `shapes`."""
    w1, w2 = synth.CFG1, synth.CFG2
    rng = np.random.default_rng(7)
    real = rng.standard_normal((3, 1024 * 6)).astype(np.complex64)     # one-sided: real samples at R = 1
    wide = rng.standard_normal((3, 65536)) + 1j * rng.standard_normal((3, 65536))
    wide[:, :] += np.exp(2j * np.pi * 0.123 * np.arange(65536))
    const = np.full((3, 1024 * 6), 0.25 + 0.5j, dtype=np.complex64)   # R = 1: the detrend leaves 0 power
    const[1] = real[0]
    const[2] = real[1]
    cases = [
        ("cfg2 fast ema", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 fast ema pipelined", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 exact", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="exact"), synth.make_frames(w2, 3, n=N7), dict(dtype="u8", flip=True)),
        ("cfg2 fp64 ema", dict(fs=w2.fs, N=4096, R=16, n=4096 * 16 + 1234, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=4096 * 16 + 1234), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("one-sided", dict(fs=48e3, N=1024, R=1, n=1024 * 6, window="hann", mode="exact"), real, dict(onesided=True, crop=512)),
        ("crop None 65536", dict(fs=2.4e6, N=65536, R=1, n=65536, window="hann", mode="exact"), wide.astype(np.complex64), dict(crop=None)),
        ("cfg1 fast linear", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="fast"), synth.make_frames(w1, 3, n=2048 * 24), dict(linear=True)),
    ]

    def run(what, frames):
        engine.reset_ema()
        if "pipelined" not in what:
            return np.concatenate([engine.process(frames[:1]), engine.process(frames[1:])])
        p_in, keep = dev.put(frames)
        p_rows, rows = dev.empty((len(frames), engine.row_width))
        engine.process_device(p_in, 1, p_rows)
        engine.process_device(p_in + frames[0].nbytes, len(frames) - 1, p_rows + engine.row_width * 4)
        engine.join()
        engine.synchronize()
        assert engine.slab_lanes == 2, what
        return np.array(dev.get(rows))

    try:
        for what, g, frames, kw in cases:
            kw = dict(kw)
            crop = kw.pop("crop", "thread")
            engine.set_option("pipeline", 1 if "pipelined" in what else 0)
            engine.configure(g["fs"], g["N"], g["R"], g["n"], g["window"], crop=crop, mode=g["mode"], **kw)
            ref = run(what, frames)                            # the mask is off: rows to shape it from
            total = 0
            for name, up, lo, mc in shapes(ref):
                engine.mask_enable(up, lo, min_cols=mc)
                rows = run(what, frames)
                assert np.array_equal(rows, ref, equal_nan=True), (what, name)
                total += len(check_log(engine, rows, (what, name), **_mask_kw(up, lo, mc)))
            assert total > 0, what
    finally:
        engine.set_option("pipeline", 0)
    # a DC-only frame: its -inf columns pass a finite lower line, excess +inf
    engine.configure(2.4e6, 1024, 1, 1024 * 6, "hann", crop="thread", mode="exact")
    ref = engine.process(const)
    assert np.isneginf(ref[0]).any() and np.isfinite(ref[1:]).all()
    lower = np.float32(np.min(ref[1:]) - 1.0)
    engine.mask_enable(lower=lower)
    rows = engine.process(const)
    want = check_log(engine, rows, "DC-only frame", lower=lower)
    assert len(want) == 1 and want[0]["row"] == 0 and np.isposinf(want[0]["excess"]) and want[0]["above"] == 0
    assert want[0]["worst_col"] == np.flatnonzero(np.isneginf(rows[0]))[0]
    # zfb_samples_process through PSD.update
    mask = {}

    def arm(first_row):
        mask.update(upper=first_row + np.float32(3.0), min_cols=3)
        return mask

    rows = _samples_rows(engine, arm)
    want = check_log(engine, rows, "samples_process", **mask)
    assert len(want) >= 1
    engine.mask_disable()


def batch_independence(engine, dev, nframes=37):
    """The same 37 frames cut into calls, groups (8, 3, 1), one by one, through the host path and
    pipelined batches, with traces and persistence on as well: the log, both counters and the
    capture bytes identical."""
    w = synth.CFG2
    frames = synth.make_frames(w, nframes, n=N7)
    p_in, keep = dev.put(frames)
    fbytes = frames[0].nbytes
    _cfg2(engine)
    engine.reset_ema()
    ref = engine.process(frames)
    upper = np.sort(ref, axis=0)[-5]                            # about 4 rows above per column
    mc = max(1, int(np.sort((ref > upper).sum(axis=1))[2 * nframes // 3]))     # about a third of the rows
    want = oracle_events(ref, upper=upper, min_cols=mc)
    assert 4 <= len(want) <= nframes - 4, len(want)
    slots, max_events = 6, len(want) - 2                       # slots run out and the log overflows
    results = {}

    def device_calls(calls, rows_too=True):
        p_rows, rows = dev.empty((nframes, engine.row_width))
        f0 = 0
        for cnt in calls:
            engine.process_device(p_in + f0 * fbytes, cnt, (p_rows + f0 * engine.row_width * 4) if rows_too else None)
            f0 += cnt
        engine.join()
        engine.synchronize()

    def run(name, body, group=0, **opts):
        for k, v in opts.items():
            engine.set_option(k, v)
        engine.set_group(group)
        _cfg2(engine)
        engine.traces_enable(True)
        engine.persistence_enable(True, levels=(-240.0, -40.0), decay=0.9)
        engine.mask_enable(upper, min_cols=mc, max_events=max_events, capture=slots)
        engine.reset_ema()
        body()
        counts = engine.mask_counts
        ev = engine.mask_events()
        results[name] = dict(counts=np.array(counts), log=ev.view(np.uint8),
                             caps=np.concatenate([engine.mask_capture(s).view(np.uint8) for s in range(slots)]),
                             persist=engine.persistence_image("f32"), avg=engine.read_trace("avg"))
        for k in opts:
            engine.set_option(k, 0)

    try:
        run("one batch", lambda: device_calls([nframes]))
        run("5 + 32", lambda: device_calls([5, 32]))
        run("no row buffer", lambda: device_calls([nframes], rows_too=False))
        run("groups of 8", lambda: device_calls([nframes]), group=8)
        run("groups of 3", lambda: device_calls([20, 17]), group=3)
        run("groups of 1", lambda: device_calls([nframes], rows_too=False), group=1)
        run("one by one", lambda: [engine.process(frames[i]) for i in range(nframes)])
        run("host path", lambda: engine.process(frames))
        run("pipelined", lambda: device_calls([5, 32]), pipeline=1)
        run("pipelined, no rows", lambda: device_calls([20, 17], rows_too=False), pipeline=1)
    finally:
        engine.set_group(0)
        engine.traces_enable(False)
        engine.persistence_enable(False)
        engine.mask_disable()
    first = results["one batch"]
    assert list(first["counts"]) == [nframes, len(want)]
    for name, got in results.items():
        for k in first:
            assert np.array_equal(got[k], first[k], equal_nan=True), (name, k)
    # and the log is the oracle's, the captures the triggering frames
    _cfg2(engine)
    engine.mask_enable(upper, min_cols=mc, max_events=max_events, capture=slots)
    engine.reset_ema()
    rows = engine.process(frames)
    assert np.array_equal(rows, ref)
    want = oracle_events(rows, upper=upper, min_cols=mc, capture_slots=slots, capture_samples=N7, frame_len=N7,
                         dtype=_lib.ZFB_DTYPE_U8)
    assert engine.mask_counts == (nframes, len(want))
    got = engine.mask_events()
    assert_events_equal(got, want[:max_events], "37 frames")
    for s in range(slots):
        assert np.array_equal(engine.mask_capture(s), frames[want[s]["row"]]), s
    engine.mask_disable()


def capture(engine, dev):
    """Capture bytes are the caller's input frames: uint8 with flip at an odd frame_len (frames
    2 mod 4 bytes apart), complex64, int16 IQ on the fused-loader path; truncation; slots that
    run out; a log that overflows; the device output."""
    w2 = synth.CFG2
    odd = N7 + 1
    u8 = synth.make_frames(w2, 5, n=odd)
    c64 = synth.make_frames(synth.CFG1, 3, n=2048 * 24)
    cs16 = synth.make_frames(synth.WORKLOADS["cfg2cs16"], 4, n=N7)
    W2 = 2 * int(.5 * 4096 / 16)
    everything = np.float32(-np.inf)                           # every finite value is above: every row triggers

    # uint8 + flip, odd frame_len: every frame captured whole
    _cfg2(engine, n=odd, ema=None)
    engine.mask_enable(everything, capture=5)
    engine.process(u8)
    ev = engine.mask_events()
    assert list(ev["capture"]) == [0, 1, 2, 3, 4] and (ev["capture_samples"] == odd).all()
    assert (ev["dtype"] == _lib.ZFB_DTYPE_U8).all() and (ev["ncols"] == W2).all()
    for s in range(5):
        got = engine.mask_capture(s)
        assert got.dtype == np.uint8 and np.array_equal(got, u8[s]), s
    # truncation to an odd sample count, slots that run out, a log that overflows
    engine.mask_enable(everything, max_events=3, capture=2, capture_samples=1001)
    engine.process(u8)
    assert engine.mask_counts == (5, 5)
    ev = engine.mask_events()
    assert list(ev["row"]) == [0, 1, 2] and list(ev["capture"]) == [0, 1, -1]
    assert list(ev["capture_samples"]) == [1001, 1001, 0]
    for s in range(2):
        assert np.array_equal(engine.mask_capture(s), u8[s][:2002]), s
    assert len(engine.mask_events(3)) == 0 and len(engine.mask_events(1, 1)) == 1
    # the device output: the same bytes, wherever the destination starts
    for off in (0, 1, 2, 3):
        p_out, buf = dev.empty((1024,))
        engine.mask_capture_device(1, p_out + off)
        engine.synchronize()
        raw = np.ascontiguousarray(dev.get(buf)).view(np.uint8)
        assert np.array_equal(raw[off:off + 2002], u8[1][:2002]), off
        assert not raw[:off].any() and not raw[off + 2002:].any(), off
    # complex64
    engine.configure(synth.CFG1.fs, 2048, 8, 2048 * 24, "hamming", crop="thread")
    engine.mask_enable(everything, capture=3)
    engine.process(c64[:1])
    engine.process(c64[1:])
    for s in range(3):
        got = engine.mask_capture(s)
        assert got.dtype == np.complex64 and np.array_equal(got, c64[s]), s
    # int16 IQ, fused into the FIR chain's loads: the slot holds the caller's int16, not the widened copy
    engine.configure(w2.fs, 4096, 16, N7, "hamming", dtype="cs16", crop="thread", mode="fast")
    assert engine.fast_active
    engine.mask_enable(everything, capture=4, capture_samples=N7 - 3)
    engine.process(cs16)
    for s in range(4):
        got = engine.mask_capture(s)
        assert got.dtype == np.int16 and np.array_equal(got, cs16[s][:2 * (N7 - 3)]), s
    # the slot stays in its dtype after a configure that keeps the mask armed
    engine.configure(w2.fs, 4096, 16, N7, "hamming", dtype="u8", flip=True, crop="thread", mode="fast")
    assert engine.mask_counts == (4, 4)
    assert np.array_equal(engine.mask_capture(0), cs16[0][:2 * (N7 - 3)])
    engine.mask_disable()


def reset_rules(engine, dev):
    """ESTATE before configure; every EINVAL; channels refused; a key-changing configure turns the
    mask off, a frame_len change keeps it armed and counting; rows kept out of the ring are
    checked, rows pushed into it are not; mask_reset keeps the lines."""
    with ZoomPSD(0, lib=engine._lib) as fresh:
        assert _errcode(fresh.mask_enable, -100.0) == _lib.ZFB_ESTATE
    w = synth.CFG1
    n = 2048 * 24
    frames = synth.make_frames(w, 6, n=n + 512)
    base = dict(fs=w.fs, N=2048, R=8, window="hamming", crop=256, f_demod=1.0)

    def conf(nn=n, **kw):
        g = dict(base, **kw)
        extra = {k: v for k, v in g.items() if k not in ("fs", "N", "R", "window")}
        engine.configure(g["fs"], g["N"], g["R"], nn, g["window"], **extra)

    conf()
    ref = engine.process(frames[:3, :n])
    W = engine.row_width
    upper = np.sort(ref, axis=0)[-2]
    lower = upper - np.float32(30.0)
    lib, h = engine._lib, engine._h

    def enable(up, lo, mc=1, me=16, cs=2, ns=100):
        pu = None if up is None else C.c_void_p(np.ascontiguousarray(up, dtype=np.float32).ctypes.data)
        pl = None if lo is None else C.c_void_p(np.ascontiguousarray(lo, dtype=np.float32).ctypes.data)
        return lib.zfb_mask_enable(h, 1, pu, pl, mc, me, cs, ns)

    keep = [np.ascontiguousarray(upper), np.ascontiguousarray(lower)]
    bad_lo = lower.copy()
    bad_lo[7] = upper[7] + 1
    nan_ok = bad_lo.copy()
    nan_ok[7] = np.nan                                     # NaN: that side off, not an inversion
    inf_ok = upper.copy()
    inf_ok[3] = -np.inf                                    # lower > upper only counts where both are finite
    for args in ((None, None), (upper, bad_lo), (upper, lower, 0), (upper, lower, W + 1), (upper, lower, 1, 0),
                 (upper, lower, 1, (1 << 20) + 1), (upper, lower, 1, 4, 5), (upper, lower, 1, 4, -1),
                 (upper, lower, 1, 4, 2, 0)):
        assert enable(*args) == _lib.ZFB_EINVAL, args
        assert _errcode(lambda: engine.mask_counts) == _lib.ZFB_ESTATE, args
    assert enable(upper, nan_ok) == 0 and enable(inf_ok, lower) == 0
    assert enable(upper, lower, W, 1 << 20, 0, 0) == 0
    del keep
    engine.mask_enable(upper, lower, max_events=16, capture=2)
    out = np.zeros(4 * n, dtype=np.uint8)
    o = C.c_void_p(out.ctypes.data)
    for slot in (-1, 2, 100):
        assert lib.zfb_mask_capture(h, slot, o, 0) == _lib.ZFB_EINVAL, slot
    assert lib.zfb_mask_capture(h, 0, None, 0) == _lib.ZFB_EINVAL
    assert lib.zfb_mask_capture(h, 0, o, 0) == _lib.ZFB_ESTATE             # not filled yet
    cnt = C.c_int(0)
    assert lib.zfb_mask_events(h, -1, 1, o, C.byref(cnt)) == _lib.ZFB_EINVAL
    assert lib.zfb_mask_events(h, 0, -1, o, C.byref(cnt)) == _lib.ZFB_EINVAL
    assert _errcode(engine.mask_capture, 2) == _lib.ZFB_EINVAL
    assert _errcode(engine.mask_capture, 0) == _lib.ZFB_ESTATE
    # virtual receivers: one mask per engine
    assert _errcode(engine.process_channels, frames[:1, :n], [1.0, 5000.0]) == _lib.ZFB_EINVAL
    p_in, keep_in = dev.put(frames[:1, :n])
    p_rows, rows = dev.empty((2, 1, W))
    assert _errcode(engine.process_channels_device, p_in, 1, [1.0, 5000.0], p_rows) == _lib.ZFB_EINVAL
    mask = dict(upper=upper, lower=lower)
    engine.mask_enable(upper, lower)
    r1 = engine.process(frames[:3, :n])
    check_log(engine, r1, "armed", **mask)
    # frame_len, window, EMA, wire format, flip, mode: the mask stays armed and counting
    r2 = []
    for kw in (dict(nn=n + 512), dict(window="hann"), dict(ema_alpha=0.5), dict(flip=True), dict(mode="exact")):
        conf(**kw)
        assert engine.mask_counts[0] == 3 + len(r2), kw
        r2.append(engine.process(frames[3:4, :kw.get("nn", n)]))
    conf(dtype="u8")
    assert engine.mask_counts[0] == 8
    conf()
    rows = np.concatenate([r1] + r2)
    check_log(engine, rows, "kept counting", **mask)
    # rows pushed into the ring are not checked; rows kept out of the ring are
    engine.push_rows(r1 + 50)
    assert engine.mask_counts[0] == 8
    engine.set_option("ring_append", 0)
    conf()
    written = engine.rows_written
    r3 = engine.process(frames[5, :n] * 4)
    assert engine.rows_written == written
    rows = np.concatenate([rows, r3])
    check_log(engine, rows, "ring_append 0", **mask)
    engine.set_option("ring_append", 1)
    conf()
    # mask_reset: log and counters empty, lines kept
    engine.mask_reset()
    assert engine.mask_counts == (0, 0) and len(engine.mask_events()) == 0
    r4 = engine.process(frames[:3, :n])
    check_log(engine, r4, "after reset", **mask)
    # fs, fft_size, fft_ratio, row_width, f_demod, flags: the lines mean other columns, the mask is off
    for kw in (dict(fs=w.fs * 1.5), dict(N=4096), dict(R=4), dict(crop=128), dict(f_demod=5000.0),
               dict(linear=True), dict(no_lo=True)):
        conf()
        engine.mask_enable(upper, lower)
        engine.process(frames[:1, :n])
        conf(**kw)
        assert _errcode(lambda: engine.mask_counts) == _lib.ZFB_ESTATE, kw
        assert _errcode(engine.mask_events) == _lib.ZFB_ESTATE, kw
        engine.process(frames[:1, :n])                         # and nothing is checked
    conf()
    assert engine.process_channels(frames[:1, :n], [1.0, 5000.0]).shape == (2, 1, W)


def burst_end_to_end(engine, nframes=37, bursts=(5, 17, 30)):
    """What the trigger is for: cfg1 frames, EMA off, a short tone burst about 30 dB above the
    floor in three frames.  Armed at the average of 8 clean frames + 10 dB with capture on, the
    log holds exactly those rows, worst_col within one bin of the tone, and each captured frame
    processed alone gives a row whose value at worst_col is the logged value bit for bit."""
    w = synth.CFG1
    n = w.frame_len
    f_burst = 9000.0
    frames = []
    for i in range(nframes + 8):
        x = synth.make_frame_complex(w, i, n)
        if i - 8 in bursts:
            k = np.arange(n // 8, dtype=np.float64)
            x[n // 2:n // 2 + n // 8] += 0.02 * np.exp(2j * np.pi * (f_burst / w.fs) * k)
        frames.append(x.astype(np.complex64))
    frames = np.array(frames)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop=w.crop, f_demod=w.f_demod)
    engine.traces_enable(True)
    engine.process(frames[:8])
    avg = engine.read_trace("avg")
    engine.traces_enable(False)
    engine.mask_enable(avg + np.float32(10.0), capture=4)
    rows = engine.process(frames[8:])
    freqs = engine.row_frequencies()
    c = int(np.argmin(np.abs(freqs - f_burst)))
    assert rows[bursts[0], c] - np.median(avg) > 25.0, (rows[bursts[0], c], np.median(avg))
    ev = check_log(engine, rows, "bursts", upper=avg + np.float32(10.0), capture_slots=4, capture_samples=n,
                   frame_len=n, dtype=_lib.ZFB_DTYPE_C64)
    assert list(ev["row"]) == list(bursts)
    got = engine.mask_events()
    bin_hz = w.fs / (w.fft_ratio * w.fft_size)
    assert (np.abs(got["freq_hz"] - f_burst) <= bin_hz).all(), got["freq_hz"]
    engine.mask_disable()
    engine.mask_enable(avg + np.float32(10.0), capture=4)
    engine.process(frames[8:])
    for s, e in enumerate(engine.mask_events()):
        x = engine.mask_capture(s)
        assert np.array_equal(x, frames[8 + e["row"]])
        row = engine.process(x)[0]
        assert row[e["worst_col"]].view(np.uint32) == np.float32(e["value"]).view(np.uint32), s
    engine.mask_disable()


def abi_layout():
    """struct zfb_mask_event: 48 bytes, offsets as in the header"""
    E = _lib.ZfbMaskEvent
    assert C.sizeof(E) == 48
    want = dict(row=0, ncols=8, first_col=12, last_col=16, worst_col=20, value=24, excess=28, above=32,
                capture=36, capture_samples=40, dtype=44)
    assert {k: getattr(E, k).offset for k in want} == want
    assert MASK_EVENT_DTYPE.itemsize == 48
    assert {k: MASK_EVENT_DTYPE.fields[k][1] for k in want} == want
