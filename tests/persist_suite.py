"""Decaying persistence spectrum (DESIGN 3.9), shared by tests/test_persist.py on the CPU
emulation build and, marked gpu, on the B200.  Every function takes a ``ZoomPSD`` and,
where device pointers are needed, a device helper of tests/engine_suite.py
(``HostAsDevice`` / ``TorchDevice``).  The oracle bins the rows the engine returned with
``oracle.waterfall_indices`` and runs the recurrence in numpy float32, frame by frame."""
from __future__ import annotations

import ctypes as C
import types

import numpy as np
import pytest

from oracle import zoompsd_oracle as zo
from pypanadapter_b200 import _lib, synth
from pypanadapter_b200.buffers import PSD, Data
from pypanadapter_b200.engine import ZoomFFTError, ZoomPSD
from tests import traces_suite as ts

N7 = ts.N7                          # cfg2's geometry with 7 Welch segments: the fp32 path, mode fast active
LEVELS = 256
DB = (-240.0, -40.0)                # the dB20 rows of these workloads lie within -232 .. -67


# ---- the oracle ----------------------------------------------------------------------------------
def oracle_persist(rows, levels, decay, P=None) -> np.ndarray:
    """P[k][c] after the rows, in frame order: P = P * decay + (k == bin), float32 throughout"""
    rows = np.asarray(rows, dtype=np.float32)
    bins = zo.waterfall_indices(rows, levels[0], levels[1])
    if P is None:
        P = np.zeros((LEVELS, rows.shape[1]), dtype=np.float32)
    d = np.float32(decay)
    k = np.arange(LEVELS)[:, None]
    for b in bins:
        P = P * d + (k == b[None, :]).astype(np.float32)
    return P


def check_persist(engine, rows, levels, decay, what=""):
    want = oracle_persist(rows, levels, decay)
    assert engine.persistence_count == len(rows), what
    got = engine.persistence_image("f32")
    assert got.shape == (LEVELS, engine.row_width), what
    assert np.array_equal(got, want[::-1]), (what, np.argwhere(got != want[::-1])[:5])
    return want


def _errcode(fn, *a, **kw):
    with pytest.raises(ZoomFFTError) as ei:
        fn(*a, **kw)
    return ei.value.code


def _cfg2(engine, n=None, mode="fast", ema=0.3, **kw):
    w = synth.CFG2
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n or w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", ema_alpha=ema, mode=mode, **kw)


# ---- scenarios -----------------------------------------------------------------------------------
def off_changes_nothing(engine, nframes=5):
    """Off (the default, or enabled and then disabled): rows, ring and launch count as an engine
    that never heard of the set.  On: the same rows bit for bit, at most one launch more per group."""
    frames = synth.make_frames(synth.CFG2, nframes)

    def run(e, mode):
        _cfg2(e)
        if mode == "on-off":
            e.persistence_enable(True)
            e.persistence_enable(False)
        elif mode == "on":
            e.persistence_enable(True, levels=DB, decay=0.9)
        e.reset_ema()
        k0 = e.counters()["kernels"]
        rows = np.concatenate([e.process(frames[:2]), e.process(frames[2:])])
        return rows, e.read_rows(nframes), e.counters()["kernels"] - k0

    with ZoomPSD(0, lib=engine._lib) as plain:
        want = run(plain, "never")
    got = run(engine, "on-off")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]
    assert engine.persistence_count == 0
    assert _errcode(engine.persistence_image, "f32") == _lib.ZFB_ESTATE
    _cfg2(engine)
    engine.persistence_enable(True, levels=DB)
    assert _errcode(engine.persistence_image, "f32") == _lib.ZFB_ESTATE      # on, but empty
    on = run(engine, "on")
    assert np.array_equal(on[0], want[0]) and np.array_equal(on[1], want[1])
    assert 1 <= on[2] - want[2] <= nframes                                    # at most one per group
    check_persist(engine, on[0], DB, 0.9, "cfg2 on")
    engine.persistence_enable(False)
    assert _errcode(engine.persistence_image, "f32") == _lib.ZFB_ESTATE


def _samples_rows(engine, levels, decay, nrows=3):
    """rows of zfb_samples_process, fed through buffers.Data / PSD.update"""
    w = synth.CFG1
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    rows = []
    for i in range(nrows):
        x = synth.make_frame(w, i, n=w.fft_size * 24)
        for j in range(0, len(x), d.chunk_size):
            d.add(x[j:j + d.chunk_size])
        psd.update()
        if i == 0:
            engine.persistence_enable(True, levels=levels, decay=decay)   # after the configure of update()
        else:
            rows.append(psd.psd.astype(np.float32))
    return np.array(rows)


def exact_against_oracle(engine, decays=(1.0, 0.9)):
    """The state, bit for bit, against the numpy recurrence on the rows the engine returned, with
    decay 1 and 0.9, on every path a row can take."""
    w1, w2 = synth.CFG1, synth.CFG2
    rng = np.random.default_rng(7)
    real = rng.standard_normal((3, 1024 * 6)).astype(np.complex64)     # one-sided: real samples at R = 1
    wide = rng.standard_normal((3, 65536)) + 1j * rng.standard_normal((3, 65536))
    wide[:, :] += np.exp(2j * np.pi * 0.123 * np.arange(65536))
    const = np.full((2, 1024 * 6), 0.25 + 0.5j, dtype=np.complex64)   # R = 1: the detrend leaves 0 power
    const[1] = real[0]
    db, lin = DB, (0.0, 5e-9)
    cases = [
        ("cfg2 fast ema", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3), db),
        ("cfg2 exact", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="exact"), synth.make_frames(w2, 3, n=N7), dict(dtype="u8", flip=True), db),
        ("cfg2 fp64 ema", dict(fs=w2.fs, N=4096, R=16, n=4096 * 16 + 1234, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=4096 * 16 + 1234), dict(dtype="u8", flip=True, ema_alpha=0.3), db),
        ("one-sided", dict(fs=48e3, N=1024, R=1, n=1024 * 6, window="hann", mode="exact"), real, dict(onesided=True, crop=512), db),
        ("crop None 65536", dict(fs=2.4e6, N=65536, R=1, n=65536, window="hann", mode="exact"), wide.astype(np.complex64), dict(crop=None), db),
        ("cfg1 fast linear", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="fast"), synth.make_frames(w1, 3, n=2048 * 24), dict(linear=True), lin),
        ("cfg1 narrow levels", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="exact"), synth.make_frames(w1, 3, n=2048 * 24), {}, (-210.0, -190.0)),
        ("constant frame", dict(fs=2.4e6, N=1024, R=1, n=1024 * 6, window="hann", mode="exact"), const, {}, db),
    ]
    for decay in decays:
        for what, g, frames, kw, levels in cases:
            kw = dict(kw)
            crop = kw.pop("crop", "thread")
            engine.configure(g["fs"], g["N"], g["R"], g["n"], g["window"], crop=crop, mode=g["mode"], **kw)
            engine.persistence_enable(True, levels=levels, decay=decay)
            engine.reset_ema()
            rows = np.concatenate([engine.process(frames[:1]), engine.process(frames[1:])])
            check_persist(engine, rows, levels, decay, (what, decay))
            bins = zo.waterfall_indices(rows, *levels)
            if what == "cfg1 narrow levels":                         # both clamps are hit
                assert (bins == 0).any() and (bins == 255).any()
            if what == "constant frame":                             # a DC-only frame: -inf columns, bin 0
                assert np.isneginf(rows[0]).any() and (bins[0][np.isneginf(rows[0])] == 0).all()
        rows = _samples_rows(engine, db, decay)
        check_persist(engine, rows, db, decay, ("samples_process", decay))
    engine.persistence_enable(False)


def batch_independence(engine, dev, nframes=37):
    """The same 37 frames cut into calls, groups (8, 3, 1), one by one, through the host path and
    pipelined batches: the persistence state and the traces (both on) bit-identical."""
    w = synth.CFG2
    frames = synth.make_frames(w, nframes, n=N7)
    p_in, keep = dev.put(frames)
    fbytes = frames[0].nbytes
    levels = DB
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
        _cfg2(engine, N7)
        engine.traces_enable(True)
        engine.persistence_enable(True, levels=levels, decay=0.9)
        engine.reset_ema()
        body()
        assert engine.persistence_count == nframes and engine.trace_count == nframes, name
        results[name] = {k: engine.read_trace(k) for k in ("last", "max", "min", "avg")}
        results[name]["persist"] = engine.persistence_image("f32")
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
    want = results["one batch"]
    for name, got in results.items():
        for k in want:
            assert np.array_equal(got[k], want[k], equal_nan=True), (name, k)
    # and the state agrees with the oracle on these rows
    _cfg2(engine, N7)
    engine.persistence_enable(True, levels=levels, decay=0.9)
    engine.reset_ema()
    rows = engine.process(frames)
    check_persist(engine, rows, levels, 0.9, "37 frames")
    assert np.array_equal(engine.persistence_image("f32"), want["persist"])
    engine.persistence_enable(False)


def reset_rules(engine, dev):
    """Every key of the reset rule starts the set empty, the others keep it counting; enabling
    again with new levels starts it empty; the arguments the C ABI refuses; channels."""
    w = synth.CFG1
    n = 2048 * 24
    frames = synth.make_frames(w, 6, n=n + 512)
    levels = DB
    base = dict(fs=w.fs, N=2048, R=8, window="hamming", crop=256, f_demod=1.0)

    def conf(nn=n, **kw):
        g = dict(base, **kw)
        extra = {k: v for k, v in g.items() if k not in ("fs", "N", "R", "window")}
        engine.configure(g["fs"], g["N"], g["R"], nn, g["window"], **extra)

    conf()
    assert engine.persistence_count == 0
    engine.persistence_enable(True, levels=levels)
    assert _errcode(engine.persistence_image, "f32") == _lib.ZFB_ESTATE       # nothing counted yet
    r1 = engine.process(frames[:3, :n])
    assert engine.persistence_count == 3
    held = engine.persistence_image("f32")
    # frame_len, window, EMA, wire format, flip, mode: the set keeps counting
    for kw in (dict(nn=n + 512), dict(window="hann"), dict(ema_alpha=0.5), dict(dtype="u8"), dict(flip=True),
               dict(mode="exact")):
        conf(**kw)
        assert engine.persistence_count == 3, kw
        assert np.array_equal(engine.persistence_image("f32"), held), kw
    conf(nn=n + 512, window="hann", mode="exact", ema_alpha=0.5)
    r2 = engine.process(frames[3:5])
    assert engine.persistence_count == 5
    check_persist(engine, np.concatenate([r1, r2]), levels, 1.0, "kept counting")
    # rows pushed into the ring do not enter the set; rows kept out of the ring do
    engine.push_rows(r2 + 50)
    assert engine.persistence_count == 5
    engine.set_option("ring_append", 0)
    conf()
    written = engine.rows_written
    r3 = engine.process(frames[5, :n] * 4)
    assert engine.rows_written == written and engine.persistence_count == 6
    check_persist(engine, np.concatenate([r1, r2, r3]), levels, 1.0, "ring_append 0")
    engine.set_option("ring_append", 1)
    # fs, fft_size, fft_ratio, row_width, f_demod, flags: a column means something else
    for kw in (dict(fs=w.fs * 1.5), dict(N=4096), dict(R=4), dict(crop=128), dict(f_demod=5000.0),
               dict(linear=True), dict(no_lo=True)):
        conf()
        engine.process(frames[:1, :n])
        assert engine.persistence_count >= 1, kw
        conf(**kw)
        assert engine.persistence_count == 0, kw
        assert _errcode(engine.persistence_image, "f32") == _lib.ZFB_ESTATE, kw
    conf()
    engine.process(frames[:2, :n])
    assert engine.persistence_count == 2
    engine.persistence_reset()
    assert engine.persistence_count == 0
    r4 = engine.process(frames[2:3, :n])
    check_persist(engine, r4, levels, 1.0, "after reset")
    # enabling again with new levels starts the set empty
    engine.persistence_enable(True, levels=(-140.0, -40.0), decay=0.5)
    assert engine.persistence_count == 0
    r5 = engine.process(frames[3:5, :n])
    check_persist(engine, r5, (-140.0, -40.0), 0.5, "new levels")
    assert np.array_equal(engine.persistence_levels(), -140.0 + np.arange(256) * (100.0 / 256))
    # bad arguments: EINVAL, and the set stays as it was
    for lv, dc in (((-20.0, -150.0), 1.0), ((-20.0, -20.0), 1.0), ((np.nan, 0.0), 1.0), ((-np.inf, 0.0), 1.0),
                   ((0.0, np.inf), 1.0), ((0.0, 1.0), 0.0), ((0.0, 1.0), -0.1), ((0.0, 1.0), 1.5),
                   ((0.0, 1.0), np.nan)):
        assert _errcode(engine.persistence_enable, True, levels=lv, decay=dc) == _lib.ZFB_EINVAL, (lv, dc)
    assert engine.persistence_count == 2
    lib, h = engine._lib, engine._h
    out = np.empty((256, engine.row_width, 4), dtype=np.uint8)
    lut = np.zeros((256, 4), dtype=np.uint8)
    o, t = C.c_void_p(out.ctypes.data), C.c_void_p(lut.ctypes.data)
    for args in ((3, 0.0, 1.0, t, o), (-1, 0.0, 1.0, t, o), (_lib.ZFB_IMAGE_U8, 1.0, 1.0, None, o),
                 (_lib.ZFB_IMAGE_U8, 2.0, 1.0, None, o), (_lib.ZFB_IMAGE_U8, np.nan, 1.0, None, o),
                 (_lib.ZFB_IMAGE_RGBA, 1.0, 0.0, t, o), (_lib.ZFB_IMAGE_RGBA, 0.0, 1.0, None, o),
                 (_lib.ZFB_IMAGE_F32, 0.0, 1.0, None, None)):
        assert lib.zfb_persist_image(h, *args, 0) == _lib.ZFB_EINVAL, args
    with pytest.raises(ValueError):
        engine.persistence_image("u8")                             # levels needed
    with pytest.raises(ValueError):
        engine.persistence_image("rgb", levels=(0, 1))
    # virtual receivers: one set per engine
    assert _errcode(engine.process_channels, frames[:1, :n], [1.0, 5000.0]) == _lib.ZFB_EINVAL
    p_in, keep = dev.put(frames[:1, :n])
    p_rows, rows = dev.empty((2, 1, engine.row_width))
    assert _errcode(engine.process_channels_device, p_in, 1, [1.0, 5000.0], p_rows) == _lib.ZFB_EINVAL
    engine.persistence_enable(False)
    assert engine.persistence_count == 0
    assert engine.process_channels(frames[:1, :n], [1.0, 5000.0]).shape == (2, 1, engine.row_width)


def image(engine, dev):
    """F32 = the oracle state upside down, U8 = its colour indices, RGBA = lut[U8]; the device
    variant equals the host output; degenerate intensity pairs (the wide guess) too."""
    w = synth.CFG1
    frames = synth.make_frames(w, 6, n=2048 * 24)
    levels = DB
    engine.configure(w.fs, 2048, 8, 2048 * 24, "hamming", crop="thread")
    engine.persistence_enable(True, levels=levels, decay=0.8)
    rows = engine.process(frames)
    P = check_persist(engine, rows, levels, 0.8, "image")
    img = P[::-1]
    W = engine.row_width
    lut = np.random.default_rng(3).integers(0, 256, (256, 4), dtype=np.uint8)
    for imin, imax in ((0.0, 4.0), (0.5, 1.5), (-1.0, 0.3), (1e7, 1e7 + 1.0), (-1e-30, 1e-30), (0.0, 5e-39)):
        want = zo.waterfall_indices(img, imin, imax)
        u8 = engine.persistence_image("u8", levels=(imin, imax))
        assert u8.shape == (256, W) and np.array_equal(u8, want), (imin, imax)
        rgba = engine.persistence_image("rgba", levels=(imin, imax), lut=lut)
        assert rgba.shape == (256, W, 4) and np.array_equal(rgba, zo.waterfall_rgba(want, lut)), (imin, imax)
    u8 = engine.persistence_image("u8", levels=(0.0, 4.0))
    assert len(np.unique(u8)) > 2                                   # the pair above spreads the state
    for kind, want, shape in (("u8", u8, (256, W)), ("rgba", zo.waterfall_rgba(u8, lut), (256, W * 4)),
                              ("f32", img, (256, W))):
        p_out, buf = dev.empty(shape)
        engine.persistence_image_device(p_out, kind, levels=(0.0, 4.0), lut=lut)
        engine.synchronize()
        got = np.ascontiguousarray(dev.get(buf)).view(np.uint8).reshape(-1)
        nb = want.nbytes
        assert np.array_equal(got[:nb], np.ascontiguousarray(want).view(np.uint8).reshape(-1)), kind
    engine.persistence_enable(False)


def intermittent_tone(engine, nframes=16):
    """What the display is for: cfg1 with its continuous tone and a weaker tone present in every
    fourth frame only.  At the weak tone's column the decay-1 state holds exactly n/4 hits within
    one bin of the burst's level and 3n/4 in bins at least 20 dB below it; the MAX trace there
    shows only the burst level and the AVG trace a mix of the two."""
    w = synth.CFG1
    f_burst = w.tones[1][0]
    n = w.frame_len
    frames = []
    for i in range(nframes):
        x = synth.make_frame_complex(w, i, n)
        if i % 4:
            k = np.arange(n, dtype=np.float64) + float(i) * n
            x -= w.tones[1][1] * np.exp(2j * np.pi * (f_burst / w.fs) * k)
        frames.append(x.astype(np.complex64))
    frames = np.array(frames)
    levels = DB                                                # 0.78 dB20 per bin
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop=w.crop, f_demod=w.f_demod)
    engine.traces_enable(True)
    engine.persistence_enable(True, levels=levels)
    rows = engine.process(frames)
    c = int(np.argmin(np.abs(engine.row_frequencies() - f_burst)))
    P = engine.persistence_image("f32")[::-1]                  # P[k] = bin k
    col = P[:, c]
    assert col.sum() == nframes
    burst_rows = rows[0::4, c]
    burst_bins = zo.waterfall_indices(burst_rows, *levels).astype(int)
    lo, hi = burst_bins.min() - 1, burst_bins.max() + 1
    assert hi - lo <= 3
    assert col[lo:hi + 1].sum() == nframes // 4
    below = int(np.ceil(20.0 / ((levels[1] - levels[0]) / 256)))
    assert col[:lo - below + 1].sum() == nframes - nframes // 4
    mx = engine.read_trace("max")[c]
    assert zo.waterfall_indices(np.float32([mx]), *levels)[0] in burst_bins
    avg = float(engine.read_trace("avg")[c])
    quiet = rows[1::4, c].max()
    assert quiet + 3.0 < avg < burst_rows.min() - 3.0, (quiet, avg, burst_rows)
    engine.traces_enable(False)
    engine.persistence_enable(False)
