"""Max-hold / min-hold / average traces and peak markers (DESIGN 3.8), shared by
tests/test_traces.py on the CPU emulation build and, marked gpu, on the B200.
Every function takes a ``ZoomPSD`` and, where device pointers are needed, a
device helper of tests/engine_suite.py (``HostAsDevice`` / ``TorchDevice``)."""
from __future__ import annotations

import numpy as np
import pytest

from pypanadapter_b200 import _lib, synth
from pypanadapter_b200.engine import ZoomFFTError, ZoomPSD

N7 = 4096 * 16 * 4 + 1234          # cfg2's geometry with 7 Welch segments: the fp32 path, mode fast active


# ---- the oracle: numpy restatements of the issue's table and of find_peaks ------------------------
def oracle_traces(rows: np.ndarray, linear: bool) -> dict:
    rows = np.asarray(rows, dtype=np.float32)
    lin = rows.astype(np.float64) if linear else 10.0 ** (rows.astype(np.float64) / 20.0)
    m = np.cumsum(lin, axis=0)[-1] / len(rows)
    return {"last": rows[-1], "max": np.fmax.reduce(rows, axis=0), "min": np.fmin.reduce(rows, axis=0),
            "avg": (m if linear else 20.0 * np.log10(m)).astype(np.float32)}


def check_traces(engine, rows, linear, what=""):
    want = oracle_traces(rows, linear)
    assert engine.trace_count == len(rows), what
    for kind in ("last", "max", "min"):
        got = engine.read_trace(kind)
        assert np.array_equal(got, want[kind], equal_nan=True), (what, kind)
    got = engine.read_trace("avg")
    if linear:
        assert np.array_equal(got, want["avg"], equal_nan=True), what
    else:
        ok = np.isfinite(want["avg"])
        assert np.array_equal(np.isfinite(got), ok), what
        assert np.abs(got[ok].astype(np.float64) - want["avg"][ok]).max() <= 1e-5, what


def candidates(x: np.ndarray, height=None) -> np.ndarray:
    """scipy's _local_maxima_1d: a rise, a plateau of equal values (not past n-2), a fall;
    the plateau's midpoint.  NaN compares false everywhere."""
    x = np.asarray(x, dtype=np.float32)
    n = len(x)
    if n < 3:
        return np.zeros(0, dtype=np.int64)
    with np.errstate(invalid="ignore"):
        brk = np.nonzero(~(x[1:] == x[:-1]))[0]               # j: x[j+1] is not x[j]
        end = np.full(n, n - 1, dtype=np.int64)               # last index of the equal run from i
        nxt = np.searchsorted(brk, np.arange(n))
        has = nxt < len(brk)
        end[has] = brk[nxt[has]]
        i = np.arange(1, n - 1)
        rise = x[i - 1] < x[i]
        a = np.minimum(end[i] + 1, n - 1)
        peak = rise & (x[a] < x[i])
        if height is not None:
            peak &= x[i].astype(np.float64) >= height
    i, a = i[peak], a[peak]
    return (i + a - 1) // 2


def oracle_peaks(x: np.ndarray, k: int, distance: int, height=None):
    """k rounds of argmax among surviving candidates (ties to the lower column), then every
    candidate closer than ``distance`` leaves; parabolic offsets in fp64."""
    x = np.asarray(x, dtype=np.float32)
    cand = candidates(x, height)
    alive = np.ones(len(cand), dtype=bool)
    cols = []
    for _ in range(k):
        if not alive.any():
            break
        idx = np.nonzero(alive)[0]
        v = x[cand[idx]]
        best = idx[np.flatnonzero(v == v.max())[0]]          # cand is ascending: first = lowest column
        p = cand[best]
        cols.append(p)
        alive &= ~(np.abs(cand - p) < distance)
    cols = np.array(cols, dtype=np.int64)
    offs = np.zeros(len(cols))
    for r, j in enumerate(cols):
        a, b, c = float(x[j - 1]), float(x[j]), float(x[j + 1])
        if a != b and c != b and np.isfinite([a, b, c]).all():
            offs[r] = 0.5 * (a - c) / (a - 2.0 * b + c)
    return cols, x[cols] if len(cols) else np.zeros(0, np.float32), offs


def random_vector(rng, n):
    x = rng.standard_normal(n).astype(np.float32)
    if rng.random() < 0.5:
        x = np.round(x * 4).astype(np.float32)                # coarse values: many plateaus and ties
    for _ in range(rng.integers(0, 6)):                        # plateaus, some of them long
        a = int(rng.integers(0, n))
        ln = int(rng.integers(2, max(3, min(n, 1 + n // int(rng.choice([4, 50, 1000]))))))
        x[a:a + ln] = x[a]
    for val in (np.nan, np.inf, -np.inf):
        for _ in range(rng.integers(0, 4)):
            x[int(rng.integers(0, n))] = val
    for _ in range(rng.integers(0, 4)):                        # exact ties between distant values
        x[int(rng.integers(0, n))] = x[int(rng.integers(0, n))]
    return x


def _put_floats(dev, x):
    """a float32 vector in device memory (host memory on the emulation build)"""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if type(dev).__name__ == "HostAsDevice":
        return x.ctypes.data, x
    import torch
    t = torch.from_numpy(x).cuda()
    return t.data_ptr(), t


# ---- scenarios ---------------------------------------------------------------------------------
def _cfg2(engine, n=None, mode="fast", ema=0.3, **kw):
    w = synth.CFG2
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n or w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", ema_alpha=ema, mode=mode, **kw)


def off_changes_nothing(engine, nframes=5):
    """Off (the default, or enabled and then disabled): rows, ring and launch count as an engine
    that never heard of traces.  On: the same rows bit for bit, at most one launch more per group."""
    frames = synth.make_frames(synth.CFG2, nframes)

    def run(e, mode):
        _cfg2(e)
        if mode == "on-off":
            e.traces_enable(True)
            e.traces_enable(False)
        elif mode == "on":
            e.traces_enable(True)
        e.reset_ema()
        k0 = e.counters()["kernels"]
        rows = np.concatenate([e.process(frames[:2]), e.process(frames[2:])])
        return rows, e.read_rows(nframes), e.counters()["kernels"] - k0

    with ZoomPSD(0, lib=engine._lib) as plain:
        want = run(plain, "never")
    got = run(engine, "on-off")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]
    assert engine.trace_count == 0
    with pytest.raises(ZoomFFTError) as ei:
        engine.read_trace("max")
    assert ei.value.code == _lib.ZFB_ESTATE
    on = run(engine, "on")
    assert np.array_equal(on[0], want[0]) and np.array_equal(on[1], want[1])
    assert 1 <= on[2] - want[2] <= nframes
    check_traces(engine, on[0], False, "cfg2 on")
    engine.traces_enable(False)


def exact_against_numpy(engine):
    """LAST / MAX / MIN bit-equal to numpy on the rows the engine returned; AVG bit-equal in
    linear mode and within 1e-5 dB20 in dB mode -- on the paths a row can take."""
    w1, w2 = synth.CFG1, synth.CFG2
    rng = np.random.default_rng(7)
    real = rng.standard_normal((3, 1024 * 6)).astype(np.complex64)     # one-sided: real samples at R = 1
    wide = rng.standard_normal((3, 65536)) + 1j * rng.standard_normal((3, 65536))
    wide[:, :] += np.exp(2j * np.pi * 0.123 * np.arange(65536))
    cases = [
        ("cfg1 exact", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="exact"), synth.make_frames(w1, 4, n=2048 * 24), {}),
        ("cfg1 fast linear", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="fast"), synth.make_frames(w1, 4, n=2048 * 24), dict(linear=True)),
        ("cfg2 fast ema", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 exact", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="exact"), synth.make_frames(w2, 3, n=N7), dict(dtype="u8", flip=True)),
        ("cfg2 fp64 ema", dict(fs=w2.fs, N=4096, R=16, n=4096 * 16 + 1234, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=4096 * 16 + 1234), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 fp64 linear", dict(fs=w2.fs, N=4096, R=16, n=4096 * 16 + 1234, window="hamming", mode="exact"), synth.make_frames(w2, 3, n=4096 * 16 + 1234), dict(dtype="u8", flip=True, linear=True)),
        ("one-sided", dict(fs=48e3, N=1024, R=1, n=1024 * 6, window="hann", mode="exact"), real, dict(onesided=True, crop=512)),
        ("crop None 65536", dict(fs=2.4e6, N=65536, R=1, n=65536, window="hann", mode="exact"), wide.astype(np.complex64), dict(crop=None)),
    ]
    for what, g, frames, kw in cases:
        kw = dict(kw)
        crop = kw.pop("crop", "thread")
        engine.configure(g["fs"], g["N"], g["R"], g["n"], g["window"], crop=crop, mode=g["mode"], **kw)
        engine.traces_enable(True)
        engine.reset_ema()
        rows = np.concatenate([engine.process(frames[:1]), engine.process(frames[1:])])
        check_traces(engine, rows, kw.get("linear", False), what)
    engine.traces_enable(False)


def batch_independence(engine, dev, nframes=37):
    """The same 37 frames in one batch, 5 + 32, one by one, through the host path and pipelined
    batches: all four traces bit-identical, 37 rows counted each time."""
    w = synth.CFG2
    frames = synth.make_frames(w, nframes, n=N7)
    p_in, keep = dev.put(frames)
    fbytes = frames[0].nbytes
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
        engine.reset_ema()
        body()
        assert engine.trace_count == nframes, name
        results[name] = {k: engine.read_trace(k) for k in ("last", "max", "min", "avg")}
        for k in opts:
            engine.set_option(k, 0)

    try:
        run("one batch", lambda: device_calls([nframes]))
        run("5 + 32", lambda: device_calls([5, 32]))
        run("no row buffer", lambda: device_calls([nframes], rows_too=False))
        run("groups of 8", lambda: device_calls([nframes]), group=8)
        run("one by one", lambda: [engine.process(frames[i]) for i in range(nframes)])
        run("host path", lambda: engine.process(frames))
        run("pipelined", lambda: device_calls([5, 32]), pipeline=1)
        run("pipelined, no rows", lambda: device_calls([20, 17], rows_too=False), pipeline=1)
    finally:
        engine.set_group(0)
        engine.traces_enable(False)
    want = results["one batch"]
    for name, got in results.items():
        for k in want:
            assert np.array_equal(got[k], want[k], equal_nan=True), (name, k)
    # and the fp32 path agrees with the numpy table on these rows
    _cfg2(engine, N7)
    engine.traces_enable(True)
    engine.reset_ema()
    check_traces(engine, engine.process(frames), False, "37 frames")
    engine.traces_enable(False)


def reset_rules(engine, dev):
    w = synth.CFG1
    n = 2048 * 24
    frames = synth.make_frames(w, 6, n=n + 512)

    def conf(nn=n, R=8, **kw):
        engine.configure(w.fs, 2048, R, nn, "hamming", crop="thread", **kw)

    conf()
    engine.traces_enable(True)
    with pytest.raises(ZoomFFTError) as ei:
        engine.read_trace("max")                                   # nothing counted yet
    assert ei.value.code == _lib.ZFB_ESTATE
    with pytest.raises(ZoomFFTError) as ei:
        engine.trace_peaks("max")
    assert ei.value.code == _lib.ZFB_ESTATE
    r1 = engine.process(frames[:3, :n])
    assert engine.trace_count == 3
    held = engine.read_trace("max")
    # frame_len, window, EMA, mode change: the traces keep counting
    engine.configure(w.fs, 2048, 8, n + 512, "hann", crop="thread", mode="exact", ema_alpha=0.5)
    assert engine.trace_count == 3 and np.array_equal(engine.read_trace("max"), held)
    r2 = engine.process(frames[3:5])
    assert engine.trace_count == 5
    assert np.array_equal(engine.read_trace("max"), np.fmax.reduce(np.concatenate([r1, r2]), axis=0))
    # rows pushed into the ring do not enter the traces
    engine.push_rows(r2 + 50)
    assert engine.trace_count == 5
    # rows kept out of the ring still enter them
    engine.set_option("ring_append", 0)
    conf()
    written = engine.rows_written
    r3 = engine.process(frames[5, :n] * 4)
    assert engine.rows_written == written and engine.trace_count == 6
    assert np.array_equal(engine.read_trace("max"), np.fmax.reduce(np.concatenate([r1, r2, r3]), axis=0))
    engine.set_option("ring_append", 1)
    # fft_ratio, flags: a column means something else -- start afresh
    conf(R=4)
    assert engine.trace_count == 0
    with pytest.raises(ZoomFFTError) as ei:
        engine.read_trace("last")
    assert ei.value.code == _lib.ZFB_ESTATE
    conf()
    engine.process(frames[:1, :n])
    assert engine.trace_count == 1
    conf(linear=True)
    assert engine.trace_count == 0
    conf()
    engine.process(frames[:2, :n])
    engine.traces_reset()
    assert engine.trace_count == 0
    # virtual receivers: one trace set per engine
    with pytest.raises(ZoomFFTError) as ei:
        engine.process_channels(frames[:1, :n], [1.0, 5000.0])
    assert ei.value.code == _lib.ZFB_EINVAL
    p_in, keep = dev.put(frames[:1, :n])
    p_rows, rows = dev.empty((2, 1, engine.row_width))
    with pytest.raises(ZoomFFTError) as ei:
        engine.process_channels_device(p_in, 1, [1.0, 5000.0], p_rows)
    assert ei.value.code == _lib.ZFB_EINVAL
    engine.traces_enable(False)
    assert engine.process_channels(frames[:1, :n], [1.0, 5000.0]).shape == (2, 1, engine.row_width)
    # bad arguments
    engine.traces_enable(True)
    engine.process(frames[:1, :n])
    for bad in (dict(k=0), dict(k=65), dict(distance=0)):
        with pytest.raises(ZoomFFTError) as ei:
            engine.trace_peaks("max", **bad)
        assert ei.value.code == _lib.ZFB_EINVAL
    with pytest.raises(ValueError):
        engine.read_trace("peak")
    engine.traces_enable(False)


def peaks_random(engine, dev, nvec=200, seed=11):
    """find_peaks_device == the numpy restatement (columns, values, offsets exactly), and on
    tie-free inputs == scipy.signal.find_peaks(x, height, distance) sorted by value, first k."""
    import scipy.signal
    rng = np.random.default_rng(seed)
    lens = np.unique(np.concatenate([[3, 4, 5, 1 << 18], np.round(np.exp(rng.uniform(np.log(3), np.log(1 << 18), nvec)))]))
    lens = rng.permutation(np.resize(lens.astype(np.int64), nvec))
    for vi, n in enumerate(lens):
        n = int(n)
        x = random_vector(rng, n)
        k = int(rng.choice([1, 8, 64]))
        d = int(rng.choice([1, 3, 50]))
        height = None
        if rng.random() < 0.5 and np.isfinite(x).any():
            height = float(np.quantile(x[np.isfinite(x)], rng.uniform(0.2, 0.9)))
        p, keep = _put_floats(dev, x)
        got = engine.find_peaks_device(p, n, k=k, distance=d, height=height)
        cols, vals, offs = oracle_peaks(x, k, d, height)
        what = (vi, n, k, d, height)
        assert np.array_equal(got["column"], cols), what
        assert np.array_equal(got["value"], vals, equal_nan=True), what
        assert np.array_equal(got["offset"], offs), what
        cand = candidates(x, height)
        if len(np.unique(x[cand])) == len(cand):                  # no ties: scipy's order is defined
            sp, _ = scipy.signal.find_peaks(x, height=height, distance=d)
            sp = sp[np.argsort(-x[sp].astype(np.float64), kind="stable")][:k]
            assert np.array_equal(sp, cols), what


def peaks_edges(engine, dev):
    """Hand-made edge cases: plateaus (midpoint, not at the ends), NaN breaks a run, +inf peaks,
    the ends are never peaks, height before distance, ties to the lower column."""
    cases = [
        ([0, 1, 1, 1, 0], [2], [0.0]),
        ([0, 1, 1, 0], [1], [0.0]),
        ([1, 0, 0, 1], [], []),
        ([0, 2, 1, 3, 1, 3, 0], [3, 5, 1], None),
        ([0, 1, np.nan, 1, 0], [], []),
        ([0, 1, 0, np.inf, 0], [3, 1], None),
        ([5, 1, 5], [], []),
        ([0, 1, 2, 2], [], []),
    ]
    for x, want, offs in cases:
        x = np.array(x, dtype=np.float32)
        p, keep = _put_floats(dev, x)
        got = engine.find_peaks_device(p, len(x), k=8, distance=1)
        assert list(got["column"]) == want, x
        if offs is not None:
            assert list(got["offset"]) == offs
        assert (got["offset"][np.isinf(got["value"])] == 0).all()
    # distance: the higher peak removes its lower neighbour; height is applied first
    x = np.array([0, 5, 0, 6, 0, 0, 0, 4, 0], dtype=np.float32)
    p, keep = _put_floats(dev, x)
    assert list(engine.find_peaks_device(p, 9, k=8, distance=3)["column"]) == [3, 7]
    assert list(engine.find_peaks_device(p, 9, k=8, distance=3, height=5.5)["column"]) == [3]
    assert list(engine.find_peaks_device(p, 9, k=1, distance=1)["column"]) == [3]
    # equal values: lower column first
    x = np.array([0, 3, 0, 3, 0, 3, 0], dtype=np.float32)
    p, keep = _put_floats(dev, x)
    assert list(engine.find_peaks_device(p, 7, k=8, distance=1)["column"]) == [1, 3, 5]
    assert list(engine.find_peaks_device(p, 7, k=8, distance=3)["column"]) == [1, 5]
    with pytest.raises(ZoomFFTError):
        engine.find_peaks_device(p, 0, k=1)
    with pytest.raises(ZoomFFTError):
        engine.find_peaks_device(p, (1 << 18) + 1, k=1)


def two_tones_end_to_end(engine, dev):
    """cfg1's two tones come out of trace_peaks("max", k=2) strongest first, at their frequencies
    within a quarter bin; find_peaks_device on a device row agrees with the LAST trace's markers."""
    w = synth.CFG1
    frames = synth.make_frames(w, 3)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, crop=w.crop, f_demod=w.f_demod)
    engine.traces_enable(True)
    engine.process(frames)
    pk = engine.trace_peaks("max", k=2)
    assert len(pk) == 2
    bin_hz = w.fs / (w.fft_ratio * w.fft_size)
    for got, (f, _a) in zip(pk, w.tones):
        assert abs(got["freq_hz"] - f) <= 0.25 * bin_hz, (got, f)
    fr = engine.row_frequencies()
    assert len(fr) == engine.row_width and np.allclose(np.diff(fr), bin_hz)
    # a row from the device path
    p_in, keep = dev.put(frames[-1:])
    p_rows, rows = dev.empty((1, engine.row_width))
    engine.process_device(p_in, 1, p_rows)
    engine.synchronize()
    row = dev.get(rows)[0]
    assert np.array_equal(engine.read_trace("last"), row)
    a = engine.find_peaks_device(p_rows, engine.row_width, k=8, distance=3)
    b = engine.trace_peaks("last", k=8, distance=3)
    assert np.array_equal(a, b)
    cols, _v, offs = oracle_peaks(row, 8, 3)
    assert np.array_equal(a["column"], cols) and np.array_equal(a["offset"], offs)
    # one-sided rows: bins k fs/N in fftshift order, no LO at R = 1
    engine.configure(48e3, 1024, 1, 1024 * 4, "hann", crop=512, onesided=True)
    f1 = engine.row_frequencies()
    assert f1.shape == (257,) and np.array_equal(f1, np.arange(257) * (48e3 / 1024))
    engine.traces_enable(False)
