"""Channel power and occupied bandwidth (DESIGN 3.11), shared by tests/test_power.py on the CPU
emulation build and, marked gpu, on the B200.  Every function takes a ``ZoomPSD`` and, where device
pointers are needed, a device helper of tests/engine_suite.py (``HostAsDevice`` /
``TorchDevice``).  The restatement computes each band's power and OBW edges in numpy (fp64,
``cumsum``, ``searchsorted`` and the interpolation of the header) on the rows the engine returned;
two further checks do not rest on it: Parseval over the frame's Welch segments, and the oracle's
own rows."""
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
RTOL = 1e-10                        # power, summary
ETOL = 1e-6                         # OBW edges, columns


# ---- the restatement -----------------------------------------------------------------------------
def linear_power(rows, linear):
    r = np.asarray(rows, dtype=np.float32).astype(np.float64)
    return r if linear else 10.0 ** (r / 20.0)


def restate(rows, bands, fs, N, linear, q=0.99):
    """(power, obw_lo, obw_hi), each [nrows][nbands], of `rows` (float32 [n][W])"""
    p = linear_power(rows, linear)
    n, nb = len(p), len(bands)
    out = np.full((3, n, nb), np.nan)
    for b, (a, e) in enumerate(bands):
        x = p[:, a:e]
        for i in range(n):
            cs = np.cumsum(x[i])
            T = cs[-1]
            out[0, i, b] = T * (fs / N)
            if not T > 0:
                continue
            for k, t in ((1, (1 - q) / 2 * T), (2, (1 + q) / 2 * T)):
                j = int(np.searchsorted(cs, t, side="left"))
                c = cs[j - 1] if j > 0 else 0.0
                out[k, i, b] = a + j + (t - c) / x[i, j]
    return out


def check_power(engine, rows, bands, linear, what="", q=0.99):
    """count, the whole log (every row of `rows`, which must all still be in it) and the summary
    against the restatement on `rows` (everything the set has seen)"""
    fs, N = engine._axis[0], engine._axis[1]
    want = restate(rows, bands, fs, N, linear, q)
    assert engine.power_count == len(rows), (what, engine.power_count, len(rows))
    log = engine.power_log(0, len(rows))
    assert np.array_equal(log["row"], np.arange(len(rows))), what
    got = np.array([log["power"], log["obw_lo"], log["obw_hi"]])
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, np.argwhere(np.isnan(got) != np.isnan(want))[:5])
    ok = ~np.isnan(want)
    scale = np.where(want[0] > 0, want[0], 1.0)
    assert np.all(np.abs(got[0] - want[0]) <= RTOL * scale), (what, np.max(np.abs(got[0] / scale - want[0] / scale)))
    assert np.all(np.abs(got[1:][ok[1:]] - want[1:][ok[1:]]) <= ETOL), (what, np.max(np.abs(got[1:][ok[1:]] - want[1:][ok[1:]])))
    level = want[0] if linear else 20 * np.log10(np.where(want[0] > 0, want[0], np.nan))
    lv = np.where(want[0] > 0, log["level"], np.nan)
    assert np.allclose(lv, level, rtol=0, atol=1e-8, equal_nan=True), what
    summ = engine.power_summary()
    for k, ref in (("max", want[0].max(axis=0)), ("min", want[0].min(axis=0)), ("mean", want[0].mean(axis=0))):
        s = np.where(ref > 0, ref, 1.0)
        assert np.all(np.abs(summ[k] - ref) <= RTOL * s), (what, k, summ[k], ref)
    return want


def band_set(W):
    """whole row, a wide band, a narrow (1-column) band, an overlapping band, and both edges"""
    return [(0, W), (W // 4, W // 2), (W // 3, W // 3 + 1), (W // 2 - 5, 3 * W // 4), (0, 3), (W - 3, W)]


def _errcode(fn, *a, **kw):
    with pytest.raises(ZoomFFTError) as ei:
        fn(*a, **kw)
    return ei.value.code


def _cfg2(engine, n=N7, mode="fast", ema=0.3, **kw):
    w = synth.CFG2
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n or w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", ema_alpha=ema, mode=mode, **kw)


# ---- scenarios -----------------------------------------------------------------------------------
def off_changes_nothing(engine, nframes=5):
    """Off (the default, or enabled and then disabled): rows, ring and launch count as an engine
    that never heard of the power set, and every read is ESTATE.  On: the same rows bit for bit,
    one launch more per group."""
    frames = synth.make_frames(synth.CFG2, nframes)

    def run(e, mode):
        _cfg2(e, n=None)
        if mode == "on-off":
            e.power_enable([(0, 10)], units="cols")
            e.power_disable()
        elif mode == "on":
            e.power_enable([(0, e.row_width), (3, 40), (100, 101)], units="cols")
        e.reset_ema()
        k0 = e.counters()["kernels"]
        rows = np.concatenate([e.process(frames[:2]), e.process(frames[2:])])
        return rows, e.read_rows(nframes), e.counters()["kernels"] - k0

    def all_estate(e):
        lib, h = e._lib, e._h
        out = np.zeros(64 * 3)
        p = C.c_void_p(out.ctypes.data)
        assert lib.zfb_power_count(h) == 0
        assert lib.zfb_power_read(h, 0, 0, p, p, p) == _lib.ZFB_ESTATE
        assert lib.zfb_power_read(h, 0, 1, p, p, p) == _lib.ZFB_ESTATE
        assert lib.zfb_power_summary(h, p) == _lib.ZFB_ESTATE
        assert lib.zfb_power_reset(h) == _lib.ZFB_ESTATE
        assert e.power_count == 0
        for fn in (e.power_log, e.power_summary, e.power_reset):
            assert _errcode(fn) == _lib.ZFB_ESTATE

    with ZoomPSD(0, lib=engine._lib) as plain:
        want = run(plain, "never")
        all_estate(plain)
    got = run(engine, "on-off")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]
    all_estate(engine)
    on = run(engine, "on")
    assert np.array_equal(on[0], want[0]) and np.array_equal(on[1], want[1])
    extra = on[2] - want[2]
    assert 1 <= extra <= nframes, extra
    check_power(engine, on[0], [(0, engine.row_width), (3, 40), (100, 101)], False, "on")
    engine.power_disable()
    all_estate(engine)


def _samples_rows(engine, bands, nrows=4):
    """rows of zfb_samples_process, fed through buffers.Data / PSD.update (the set enabled after
    the first row, whose update configured the engine)"""
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
            engine.power_enable(bands, units="cols")
        else:
            rows.append(psd.psd.astype(np.float32))
    return np.array(rows)


def exact_against_restatement(engine, dev):
    """The log and summary against the restatement on the rows the engine returned, on every path
    a row can take, for whole-row, wide, 1-column, overlapping and edge bands; a DC-only frame."""
    w1, w2 = synth.CFG1, synth.CFG2
    rng = np.random.default_rng(7)
    real = rng.standard_normal((3, 1024 * 6)).astype(np.complex64)     # one-sided: real samples at R = 1
    wide = rng.standard_normal((3, 65536)) + 1j * rng.standard_normal((3, 65536))
    wide[:, :] += np.exp(2j * np.pi * 0.123 * np.arange(65536))
    cases = [
        ("cfg2 fast ema", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 fast ema device", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 fast ema pipelined", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=N7), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("cfg2 exact", dict(fs=w2.fs, N=4096, R=16, n=N7, window="hamming", mode="exact"), synth.make_frames(w2, 3, n=N7), dict(dtype="u8", flip=True)),
        ("cfg2 fp64 ema", dict(fs=w2.fs, N=4096, R=16, n=4096 * 16 + 1234, window="hamming", mode="fast"), synth.make_frames(w2, 4, n=4096 * 16 + 1234), dict(dtype="u8", flip=True, ema_alpha=0.3)),
        ("one-sided", dict(fs=48e3, N=1024, R=1, n=1024 * 6, window="hann", mode="exact"), real, dict(onesided=True, crop=512)),
        ("crop None 65536", dict(fs=2.4e6, N=65536, R=1, n=65536, window="hann", mode="exact"), wide.astype(np.complex64), dict(crop=None)),
        ("cfg1 fast linear", dict(fs=w1.fs, N=2048, R=8, n=2048 * 24, window="hamming", mode="fast"), synth.make_frames(w1, 3, n=2048 * 24), dict(linear=True)),
    ]

    def run(what, frames):
        engine.reset_ema()
        if "device" not in what and "pipelined" not in what:
            return np.concatenate([engine.process(frames[:1]), engine.process(frames[1:])])
        p_in, keep = dev.put(frames)
        p_rows, rows = dev.empty((len(frames), engine.row_width))
        engine.process_device(p_in, 1, p_rows)
        engine.process_device(p_in + frames[0].nbytes, len(frames) - 1, p_rows + engine.row_width * 4)
        engine.join()
        engine.synchronize()
        if "pipelined" in what:
            assert engine.slab_lanes == 2, what
        return np.array(dev.get(rows))

    try:
        for what, g, frames, kw in cases:
            kw = dict(kw)
            crop = kw.pop("crop", "thread")
            engine.set_option("pipeline", 1 if "pipelined" in what else 0)
            engine.configure(g["fs"], g["N"], g["R"], g["n"], g["window"], crop=crop, mode=g["mode"], **kw)
            W = engine.row_width
            if what == "one-sided":
                # bands given in Hz, OBW fraction 0.9
                f = engine.row_frequencies()
                engine.power_enable([(f[0], f[99]), (f[100], f[W - 1]), (f[50], f[50])], obw=0.9)
                bands = [(0, 100), (100, W), (50, 51)]
                q = 0.9
            elif what == "crop None 65536":
                # whole row and a 6000-column band (one CTA per row each), a narrow band (one warp)
                bands, q = [(0, W), (100, 130), (W // 2 - 3000, W // 2 + 3000)], 0.99
                engine.power_enable(bands, units="cols")
            else:
                bands, q = band_set(W), 0.99
                engine.power_enable(bands, units="cols")
            rows = run(what, frames)
            check_power(engine, rows, bands, kw.get("linear", False), what, q)
            engine.power_disable()
    finally:
        engine.set_option("pipeline", 0)
    # a DC-only frame: its band of -inf columns has power 0 and NaN edges, the other rows do not
    const = np.full((3, 1024 * 6), 0.25 + 0.5j, dtype=np.complex64)   # R = 1: the detrend leaves 0 power
    const[1:] = real[:2]
    engine.configure(2.4e6, 1024, 1, 1024 * 6, "hann", crop="thread", mode="exact")
    ref = engine.process(const)
    dead = np.flatnonzero(np.isneginf(ref[0]))
    assert dead.size > 0 and np.isfinite(ref[1:]).all()
    d0 = int(dead[0])
    d1 = d0 + int(np.argmax(~np.isneginf(ref[0, d0:]))) if np.isfinite(ref[0, d0:]).any() else engine.row_width
    bands = [(d0, d1), (0, engine.row_width)]
    engine.power_enable(bands, units="cols")
    rows = engine.process(const)
    want = check_power(engine, rows, bands, False, "DC-only frame")
    assert want[0, 0, 0] == 0.0 and np.isnan(want[1:, 0, 0]).all() and want[0, 1:, 0].min() > 0
    log = engine.power_log()
    assert log["power"][0, 0] == 0.0 and np.isnan(log["obw_lo"][0, 0]) and np.isnan(log["obw_hi_hz"][0, 0])
    assert np.isneginf(log["level"][0, 0])
    # zfb_samples_process through PSD.update
    bands = band_set(synth.CFG1.row_width)
    rows = _samples_rows(engine, bands)
    check_power(engine, rows, bands, False, "samples_process")
    engine.power_disable()


def hz_mapping(engine):
    """Bands given in Hz are the columns whose row_frequencies() lie in [f_lo, f_hi]; the edges in
    Hz are f(floor(x)) + (x - floor(x) - 0.5) spacing; a band of no column or of two runs of
    columns is a ValueError."""
    w = synth.CFG1
    engine.configure(w.fs, w.fft_size, w.fft_ratio, 2048 * 24, w.window, crop=w.crop, f_demod=w.f_demod)
    f = engine.row_frequencies()
    spacing = w.fs / (w.fft_ratio * w.fft_size)
    engine.power_enable([(-3000.0, 3000.0), (f[10], f[10]), (f[0] - 1e6, f[-1] + 1e6)])
    want = [(int(np.flatnonzero(f >= -3000.0)[0]), int(np.flatnonzero(f <= 3000.0)[-1]) + 1), (10, 11),
            (0, engine.row_width)]
    assert [tuple(b) for b in engine._power[0]] == want
    frames = synth.make_frames(w, 3, n=2048 * 24)
    rows = engine.process(frames)
    check_power(engine, rows, want, False, "Hz bands")
    log = engine.power_log()
    for k in ("lo", "hi"):
        x = log["obw_" + k]
        fl = np.clip(np.floor(x), [a for a, _ in want], [e - 1 for _, e in want]).astype(int)
        assert np.allclose(log["obw_%s_hz" % k], f[fl] + (x - fl - 0.5) * spacing, rtol=0, atol=1e-6)
    assert np.allclose(log["obw_hz"], log["obw_hi_hz"] - log["obw_lo_hz"])
    # cfg1's tones at -11.1 kHz (1 % of the power) and 5.3 kHz: the whole row's 99 % OBW runs from
    # inside the first to the upper skirt of the second
    assert np.all(np.abs(log["obw_lo_hz"][:, 2] + 11100.0) < 10 * spacing), log["obw_lo_hz"][:, 2]
    assert np.all(np.abs(log["obw_hi_hz"][:, 2] - 5300.0) < 10 * spacing), log["obw_hi_hz"][:, 2]
    for bad in ([(f[-1] + 10.0, f[-1] + 20.0)], [(f[3] + 0.1 * spacing, f[3] + 0.2 * spacing)]):
        with pytest.raises(ValueError):
            engine.power_enable(bad)
    with pytest.raises(ValueError):
        engine.power_enable([(0, 10)], units="bins")
    # uncropped one-sided rows wrap in frequency in the middle of the row: a band across the wrap is
    # two runs of columns; bands on either side of it are one run each
    engine.configure(48e3, 1024, 1, 1024 * 6, "hann", crop=None, mode="exact", onesided=True)
    f = engine.row_frequencies()
    cut = int(np.argmin(f))
    assert 0 < cut < engine.row_width - 1 and f[cut - 1] > f[cut + 1]
    with pytest.raises(ValueError):
        engine.power_enable([(f[cut + 5], f[cut - 5])])
    engine.power_enable([(f[cut], f[cut + 20]), (f[cut - 30], f[cut - 1])])
    assert [tuple(b) for b in engine._power[0]] == [(cut, cut + 21), (cut - 30, cut)]
    engine.power_disable()


def parseval(engine):
    """Independent of the implementation: at R = 1, crop=None, the power of a band over the whole
    row is mean_s sum |w (x_s - m_s)|^2 / sum w^2 over the frame's Welch segments."""
    N, n, fs = 4096, 4096 * 5 + 1000, 1.0e6
    rng = np.random.default_rng(3)
    k = np.arange(n)
    x = (0.3 * np.exp(2j * np.pi * 0.0123 * k) + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
         + (0.4 - 0.2j)).astype(np.complex64)
    engine.configure(fs, N, 1, n, "hann", crop=None, mode="exact")
    engine.power_enable([(0, engine.row_width)], units="cols")
    engine.process(x[None])
    got = engine.power_log()["power"][0, 0]
    nperseg, hop, nseg = zo.welch_plan(n, N)
    w = zo.scipy.signal.get_window("hann", nperseg)
    xs = x.astype(np.complex128)
    want = np.mean([np.sum(np.abs(w * (xs[s * hop:s * hop + nperseg] - xs[s * hop:s * hop + nperseg].mean())) ** 2)
                    for s in range(nseg)]) / np.sum(w * w)
    assert abs(got / want - 1) < 1e-4, (got, want)
    engine.power_disable()


def acpr_scenario(nframes=3):
    """cfg1 frames: band-limited noise filling |f| < 2.5 kHz of the main channel and a spur 40 dB
    below its power at +6.5 kHz, in the adjacent channel above"""
    w = synth.CFG1
    n = w.frame_len
    rng = np.random.default_rng(11)
    frames = []
    f = np.fft.fftfreq(n, 1 / w.fs)
    for i in range(nframes):
        z = rng.standard_normal(n) + 1j * rng.standard_normal(n)
        z = np.fft.ifft(np.fft.fft(z) * (np.abs(f) < 2500.0))
        z *= 0.1 / np.sqrt(np.mean(np.abs(z) ** 2))                  # power 0.01
        k = np.arange(n) + i * n
        z += np.sqrt(0.01 * 1e-4) * np.exp(2j * np.pi * 6500.0 / w.fs * k)
        z += 1e-4 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
        frames.append(z.astype(np.complex64))
    chans = [(-16000.0, -10000.0), (-9500.0, -3500.0), (-3000.0, 3000.0), (3500.0, 9500.0), (10000.0, 16000.0)]
    return w, np.array(frames), chans


def against_oracle_rows(engine):
    """On the ACPR scenario, band powers within 0.01 dB20 of sum p fs/N over the oracle's linear
    rows, ACPR within 0.01 dB, and the 99 % OBW edges within one column."""
    w, frames, chans = acpr_scenario()
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, crop=w.crop, f_demod=w.f_demod)
    engine.power_enable(chans)
    engine.process(frames)
    log = engine.power_log()
    bands = [tuple(b) for b in engine._power[0]]
    orows = np.array([zo.zoom_psd_power(x, w.fs, w.fft_size, w.fft_ratio, w.window, f_demod=w.f_demod, crop=w.crop)
                      for x in frames])
    ref = restate(orows, bands, w.fs, w.fft_size, True)
    assert np.all(np.abs(20 * np.log10(log["power"] / ref[0])) <= 0.01), 20 * np.log10(log["power"] / ref[0])
    acpr = 10 * np.log10(log["power"] / log["power"][:, 2:3])
    acpr_ref = 10 * np.log10(ref[0] / ref[0][:, 2:3])
    assert np.all(np.abs(acpr - acpr_ref) <= 0.01), (acpr, acpr_ref)
    # the spur, about -40 dBc (plus the main channel's skirt and the chain's droop over the channel)
    assert np.all(np.abs(acpr[:, 3] + 40.0) < 2.0), acpr[:, 3]
    assert np.all(np.abs(log["obw_lo"][:, 2] - ref[1][:, 2]) <= 1.0)
    assert np.all(np.abs(log["obw_hi"][:, 2] - ref[2][:, 2]) <= 1.0)
    assert np.all(np.abs(log["obw_hz"][:, 2] - 5000.0) < 400.0), log["obw_hz"][:, 2]  # 99 % of |f| < 2.5 kHz
    engine.power_disable()


def batch_independence(engine, dev, nframes=37):
    """The same 37 frames cut ten ways (calls, groups of 8 / 3 / 1, one by one, host path,
    pipelined batches), with traces, persistence and the mask on as well: the log, summary and
    count bit-identical; and a log of 3 rows fed by groups of 8 holds the newest 3 rows."""
    w = synth.CFG2
    frames = synth.make_frames(w, nframes, n=N7)
    p_in, keep = dev.put(frames)
    fbytes = frames[0].nbytes
    _cfg2(engine)
    W = engine.row_width
    bands = band_set(W)
    results = {}

    def device_calls(calls, rows_too=True):
        p_rows, rows = dev.empty((nframes, W))
        f0 = 0
        for cnt in calls:
            engine.process_device(p_in + f0 * fbytes, cnt, (p_rows + f0 * W * 4) if rows_too else None)
            f0 += cnt
        engine.join()
        engine.synchronize()

    def run(name, body, group=0, log_rows=64, **opts):
        for k, v in opts.items():
            engine.set_option(k, v)
        engine.set_group(group)
        _cfg2(engine)
        engine.traces_enable(True)
        engine.persistence_enable(True, levels=(-240.0, -40.0), decay=0.9)
        engine.mask_enable(upper=-150.0, max_events=8)
        engine.power_enable(bands, units="cols", log_rows=log_rows)
        engine.reset_ema()
        body()
        log = engine.power_log()
        results[name] = dict(count=engine.power_count, log=np.ascontiguousarray(log).view(np.uint8),
                             summary=engine.power_summary().view(np.uint8))
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
        run("log of 3, groups of 8", lambda: device_calls([nframes]), group=8, log_rows=3)
        assert list(engine.power_log()["row"]) == [nframes - 3, nframes - 2, nframes - 1]
        for first in (0, nframes - 4, nframes - 1):
            n = 2 if first == nframes - 1 else 1
            assert _errcode(engine.power_log, first, n) == _lib.ZFB_EINVAL, first
    finally:
        engine.set_group(0)
        engine.traces_enable(False)
        engine.persistence_enable(False)
        engine.mask_disable()
        engine.power_disable()
    first = results["one batch"]
    assert first["count"] == nframes
    short = results.pop("log of 3, groups of 8")
    assert short["count"] == nframes and np.array_equal(short["summary"], first["summary"])
    rec = first["log"].size // nframes
    assert np.array_equal(short["log"], first["log"][-3 * rec:])
    for name, got in results.items():
        for k in first:
            assert np.array_equal(got[k], first[k]), (name, k)
    # and they are the restatement's on these rows
    _cfg2(engine)
    engine.power_enable(bands, units="cols")
    engine.reset_ema()
    rows = engine.process(frames)
    check_power(engine, rows, bands, False, "37 frames")
    got = engine.power_log()
    assert np.ascontiguousarray(got).view(np.uint8).tobytes() == first["log"].tobytes()
    engine.power_disable()


def reset_rules(engine, dev):
    """ESTATE before configure; every EINVAL; channels refused; a key-changing configure turns the
    set off, a change of frame_len, window, EMA, wire format, flip or mode keeps it counting; rows
    kept out of the ring are measured, rows pushed into it are not; power_reset keeps the bands;
    a failed enable leaves the set as it was."""
    with ZoomPSD(0, lib=engine._lib) as fresh:
        assert _errcode(fresh.power_enable, [(0, 1)], units="cols") == _lib.ZFB_ESTATE
    w = synth.CFG1
    n = 2048 * 24
    frames = synth.make_frames(w, 6, n=n + 512)
    base = dict(fs=w.fs, N=2048, R=8, window="hamming", crop=256, f_demod=1.0)

    def conf(nn=n, **kw):
        g = dict(base, **kw)
        extra = {k: v for k, v in g.items() if k not in ("fs", "N", "R", "window")}
        engine.configure(g["fs"], g["N"], g["R"], nn, g["window"], **extra)

    conf()
    W = engine.row_width
    lib, h = engine._lib, engine._h

    def enable(bands, nb=None, q=0.99, log_rows=16):
        arr = np.ascontiguousarray(np.array(bands, dtype=np.int32).reshape(-1, 2))
        ptr = C.c_void_p(arr.ctypes.data) if len(arr) else None
        return lib.zfb_power_enable(h, 1, ptr, len(arr) if nb is None else nb, q, log_rows)

    many = [(i, i + 1) for i in range(65)]
    for args in (([], 1), ([(0, 1)], 0), (many, None), ([(-1, 4)],), ([(5, 5)],), ([(6, 5)],), ([(0, W + 1)],),
                 ([(0, 1)], None, 0.0), ([(0, 1)], None, 1.0), ([(0, 1)], None, float("nan")), ([(0, 1)], None, -0.5),
                 ([(0, 1)], None, 0.99, 0), ([(0, 1)], None, 0.99, -3), ([(0, 1), (1, 2)], None, 0.99, (1 << 25) + 1),
                 ([(0, 1)], None, 0.99, (1 << 26) + 1)):
        assert enable(*args) == _lib.ZFB_EINVAL, args
        assert engine.power_count == 0 and lib.zfb_power_reset(h) == _lib.ZFB_ESTATE, args
    # the limits themselves are accepted (checked small: a log of 2^26 entries would hold 1.6 GB)
    assert enable(many[:64]) == 0 and enable([(0, W)], q=1e-9, log_rows=1) == 0
    engine.power_disable()
    bands = [(0, W), (100, 140)]
    engine.power_enable(bands, units="cols", log_rows=16)
    # a failed enable leaves the set as it was
    r0 = engine.process(frames[:1, :n])
    assert enable([(0, W + 1)]) == _lib.ZFB_EINVAL and engine.power_count == 1
    engine.power_reset()
    out = np.zeros(64)
    o = C.c_void_p(out.ctypes.data)
    assert lib.zfb_power_summary(h, None) == _lib.ZFB_EINVAL
    assert lib.zfb_power_summary(h, o) == 0 and np.isnan(out[:6]).all()          # no row yet
    assert np.isnan(engine.power_summary()["max"]).all()
    assert lib.zfb_power_read(h, 0, 0, o, o, o) == 0
    for first, cnt in ((0, 1), (-1, 0), (0, -1)):
        assert lib.zfb_power_read(h, first, cnt, o, o, o) == _lib.ZFB_EINVAL, (first, cnt)
    # virtual receivers: one power set per engine
    assert _errcode(engine.process_channels, frames[:1, :n], [1.0, 5000.0]) == _lib.ZFB_EINVAL
    p_in, keep_in = dev.put(frames[:1, :n])
    p_rows, rows = dev.empty((2, 1, W))
    assert _errcode(engine.process_channels_device, p_in, 1, [1.0, 5000.0], p_rows) == _lib.ZFB_EINVAL
    r1 = engine.process(frames[:3, :n])
    check_power(engine, r1, bands, False, "on")
    # frame_len, window, EMA, wire format, flip, mode: the set keeps counting
    r2 = []
    for kw in (dict(nn=n + 512), dict(window="hann"), dict(ema_alpha=0.5), dict(flip=True), dict(mode="exact")):
        conf(**kw)
        assert engine.power_count == 3 + len(r2), kw
        r2.append(engine.process(frames[3:4, :kw.get("nn", n)]))
    conf(dtype="u8")
    assert engine.power_count == 8
    conf()
    rows = np.concatenate([r1] + r2)
    check_power(engine, rows, bands, False, "kept counting")
    # rows pushed into the ring are not measured; rows kept out of the ring are
    engine.push_rows(r1 + 50)
    assert engine.power_count == 8
    engine.set_option("ring_append", 0)
    conf()
    written = engine.rows_written
    r3 = engine.process(frames[5, :n] * 4)
    assert engine.rows_written == written
    rows = np.concatenate([rows, r3])
    check_power(engine, rows, bands, False, "ring_append 0")
    engine.set_option("ring_append", 1)
    conf()
    # the log holds the newest 16 rows: older ones and rows not measured yet are EINVAL
    more = engine.process(frames[:, :n].repeat(2, axis=0))
    assert engine.power_count == 21
    assert len(engine.power_log()) == 16 and engine.power_log()["row"][0] == 5
    for first, cnt in ((4, 1), (20, 2), (21, 1)):
        assert lib.zfb_power_read(h, first, cnt, o, None, None) == _lib.ZFB_EINVAL, (first, cnt)
    assert lib.zfb_power_read(h, 5, 16, None, None, None) == 0
    got = engine.power_log(17, 4)
    want = restate(more[-4:], bands, w.fs, 2048, False)
    assert np.allclose(got["power"], want[0], rtol=RTOL, atol=0)
    # power_reset: log, summary and count empty, bands kept
    engine.power_reset()
    assert engine.power_count == 0 and len(engine.power_log()) == 0
    r4 = engine.process(frames[:3, :n])
    check_power(engine, r4, bands, False, "after reset")
    # fs, fft_size, fft_ratio, row_width, f_demod, flags: the columns mean other frequencies, the set is off
    for kw in (dict(fs=w.fs * 1.5), dict(N=4096), dict(R=4), dict(crop=128), dict(f_demod=5000.0),
               dict(linear=True), dict(no_lo=True)):
        conf()
        engine.power_enable(bands, units="cols")
        engine.process(frames[:1, :n])
        conf(**kw)
        assert engine.power_count == 0, kw
        assert _errcode(engine.power_log) == _lib.ZFB_ESTATE, kw
        assert _errcode(engine.power_summary) == _lib.ZFB_ESTATE, kw
        engine.process(frames[:1, :n])                         # and nothing is measured
    conf()
    assert engine.process_channels(frames[:1, :n], [1.0, 5000.0]).shape == (2, 1, W)
    del r0


def burst_end_to_end(engine, nframes=37, bursts=(5, 17, 30)):
    """What the log is for: cfg1 frames, EMA off, a tone burst in frames 5, 17 and 30.  In the
    burst's channel exactly those rows stand at least 20 dB20 above all the others, and the
    summary's max is the largest of them bit for bit."""
    w = synth.CFG1
    n = w.frame_len
    f_burst = 9000.0
    frames = []
    for i in range(nframes):
        x = synth.make_frame_complex(w, i, n)
        if i in bursts:
            k = np.arange(n // 8, dtype=np.float64)
            x[n // 2:n // 2 + n // 8] += 0.02 * np.exp(2j * np.pi * (f_burst / w.fs) * k)
        frames.append(x.astype(np.complex64))
    frames = np.array(frames)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop=w.crop, f_demod=w.f_demod)
    engine.power_enable([(f_burst - 1000.0, f_burst + 1000.0), (-3000.0, 3000.0)], log_rows=64)
    engine.process(frames[:20])
    engine.process(frames[20:])
    log = engine.power_log()
    lv = log["level"][:, 0]
    quiet = np.delete(lv, bursts)
    assert np.all(lv[list(bursts)] >= quiet.max() + 20.0), (lv[list(bursts)], quiet.max())
    assert list(np.flatnonzero(lv >= quiet.max() + 20.0)) == list(bursts)
    s = engine.power_summary()
    assert s["max"][0] == log["power"][list(bursts), 0].max()
    assert s["min"][0] == log["power"][:, 0].min()
    engine.power_disable()
