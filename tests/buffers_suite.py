"""Checks of the buffer mirrors (pypanadapter_b200.buffers), shared by the CPU
emulation tests and the GPU tests."""
from __future__ import annotations

import os
import types

import numpy as np
import pytest

from oracle import golden_cases as gc
from oracle import make_golden as mg
from oracle import zoompsd_oracle as zo
from pypanadapter_b200 import synth
from pypanadapter_b200.buffers import PSD, Data, Waterfall
from tests import parity


def data_foldback(engine):
    """Data.add / get_data_* reproduce the reference's fold-back trace
    (golden data_trace.npz, recorded from T:1400-1483) and contents."""
    g = np.load(os.path.join(parity.GOLDEN_DIR, "data_trace.npz"))
    d = Data(engine=engine).new_complex()
    assert d.max_size == int(g["max_size"]) and d.maxsize == d.max_size
    assert d.data.dtype == np.complex64 and len(d.data) == d.max_size
    trace = []
    for chunk in mg.data_trace_chunks():
        d.add(chunk)
        trace.append((d.size, d.real_size, d.total_size))
    assert np.array_equal(np.array(trace), g["trace"])
    d.get_data_start()
    tail = d.data[:d.real_size].copy()
    d.get_data_end()
    assert (d.size, d.real_size, d.total_size) == (0, 0, 0)
    assert np.array_equal(tail, g["tail"].astype(np.complex64))


def data_random_sequences(engine, seeds=range(8)):
    """Random chunk-length sequences (incl. lengths that force the fold-back,
    takes in between, and raw uint8 storage): counters and contents of
    buffers.Data equal the oracle's restatement of T:1433-1468 at every step."""
    for seed in seeds:
        rng = np.random.default_rng(500 + seed)
        cs = int(rng.choice([512, 1000, 4096]))
        u8 = bool(seed % 2)
        d = Data(cs, engine=engine)
        d = d.new_u8() if u8 else d.new_complex()
        o = zo.DataOracle(cs).new_complex()
        assert d.max_size == o.max_size
        for step in range(60):
            if rng.random() < 0.15:
                d.get_data_start()
                got = np.array(d.data[:(2 if u8 else 1) * d.real_size], copy=True)
                d.get_data_end()
                want = o.take()
                if u8:
                    assert np.array_equal(got.astype(np.float64).view(np.complex128), want)
                else:
                    assert np.array_equal(got, want.astype(np.complex64))
                assert (d.size, d.real_size, d.total_size) == (0, 0, 0)
                continue
            n = int(rng.integers(1, 3 * cs))
            if u8:
                b = rng.integers(0, 256, 2 * n, dtype=np.uint8)
                d.add(b)
                o.add(b.astype(np.float64).view(np.complex128))       # the bytes as (I, Q) pairs
            else:
                c = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
                d.add(c)
                o.add(c)
            assert (d.size, d.real_size, d.total_size) == (o.size, o.real_size, o.total_size), (seed, step)


def psd_update_matches_reference(engine):
    """PSD.update on Data fed chunk by chunk == the golden row the reference's
    own PSD.update produced for the same samples (cfg1_T)."""
    case = gc.case_by_name("cfg1_T")
    x = gc.make_input(case)
    state = types.SimpleNamespace(fft_size=case["N"], fft_ratio=case["R"], fft_tapering=case["window"],
                                  panadapter=types.SimpleNamespace(SampleRate=case["fs"]))
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    assert psd.psd.shape == (case["N"],) and not psd.psd.any()
    for i in range(0, len(x), d.chunk_size):
        d.add(x[i:i + d.chunk_size])
    assert d.real_size == len(x)
    psd.update()
    psd.lock.lock()
    row = psd.psd
    psd.lock.unlock()
    floor = parity.floor_db20(case["fs"], case["window"], case["N"], True)
    parity.assert_row_parity(row, parity.golden_rows()["cfg1_T"], floor, "PSD.update")
    assert (d.size, d.real_size, d.total_size) == (0, 0, 0)
    # too little data: psd stays as it is (T:1522)
    d.add(x[:1000])
    before = psd.psd
    psd.update()
    assert psd.psd is before
    # a second, different frame goes through the other device mirror
    x2 = synth.make_frame(synth.CFG1, 1)
    for i in range(0, len(x2), d.chunk_size):
        d.add(x2[i:i + d.chunk_size])
    psd.update()
    want = zo.zoom_psd(x2, case["fs"], case["N"], case["R"], case["window"])
    parity.assert_row_parity(psd.psd, want, floor, "PSD.update frame 2")


def psd_update_u8(engine):
    """uint8 wire format through Data.new_u8 (conversion on the device)."""
    w = synth.CFG2
    raw = synth.make_frame(w, 0, n=4096 * 32)
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    d = Data(engine=engine).new_u8()
    psd = PSD(d, state, flip=True)
    step = 2 * d.chunk_size
    for i in range(0, len(raw), step):
        d.add(raw[i:i + step])
    psd.update()
    want = zo.zoom_psd(raw, w.fs, w.fft_size, w.fft_ratio, w.window, flip=True)
    parity.assert_row_parity(psd.psd, want, parity.floor_db20(w.fs, w.window, w.fft_size, True), "u8 PSD.update")


def psd_update_cs16(engine):
    """SoapySDR CS16 through Data.new_cs16 (pinned int16 ring, widened on the
    device), fold-back included: the row equals the oracle's on the samples the
    ring holds."""
    fs, N, R = 2.4e6, 1024, 8
    n = N * R * 5
    k = np.arange(n)
    rng = np.random.default_rng(5)
    x = 0.4 * np.exp(2j * np.pi * 1700.0 / fs * k) + 3e-3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    raw = synth.quantise_cs16(x)
    state = types.SimpleNamespace(fft_size=N, fft_ratio=R, fft_tapering="hamming",
                                  panadapter=types.SimpleNamespace(SampleRate=fs))
    d = Data(chunk_size=4096, engine=engine).new_cs16()
    assert d.data.dtype == np.int16 and d.data.shape == (2 * d.max_size,)
    psd = PSD(d, state)
    step = 2 * 4096
    for i in range(0, len(raw), step):
        d.add(raw[i:i + step])
    assert d.real_size == n
    psd.update()
    want = zo.zoom_psd(raw, fs, N, R, "hamming")
    parity.assert_row_parity(psd.psd, want, parity.floor_db20(fs, "hamming", N, True), "cs16 PSD.update")
    with pytest.raises(TypeError):
        d.add(np.zeros(64, dtype=np.uint8))


def psd_update_real(engine):
    """Data.new_real (T:1413-1417) + PSD.update without zoom: welch of real
    samples is one-sided and the reference fftshifts / crops those N/2+1 bins
    (golden audio_R1_Treal, recorded from the reference's own methods)."""
    case = gc.case_by_name("audio_R1_Treal")
    x = gc.make_input(case)
    state = types.SimpleNamespace(fft_size=case["N"], fft_ratio=case["R"], fft_tapering=case["window"],
                                  panadapter=types.SimpleNamespace(SampleRate=case["fs"]))
    d = Data(engine=engine).new_real()
    psd = PSD(d, state)
    for i in range(0, len(x), 4096):
        d.add(x[i:i + 4096])
    psd.update()
    want = parity.golden_rows()["audio_R1_Treal"]
    assert psd.psd.shape == want.shape == (case["N"] // 2 + 1,)
    parity.assert_row_parity(psd.psd, want, parity.floor_db20(case["fs"], case["window"], case["N"], False),
                             "real PSD.update")
    # zoomed: the mix makes the chunk complex, rows are two-sided again (T:1525-1536)
    state.fft_ratio = 4
    for i in range(0, len(x), 4096):
        d.add(x[i:i + 4096])
    psd.update()
    want = zo.zoom_psd(x, case["fs"], case["N"], 4, case["window"])
    parity.assert_row_parity(psd.psd, want, parity.floor_db20(case["fs"], case["window"], case["N"], True),
                             "real PSD.update R=4")


def waterfall_image(engine):
    """Waterfall.img_array assembled from the device ring == the reference's
    img_array after the same image_update calls (golden waterfall.npz)."""
    g = np.load(os.path.join(parity.GOLDEN_DIR, "waterfall.npz"))
    rows = [np.full(256, -100.0 - i) + np.arange(256) * 0.01 for i in range(70)]
    engine.configure(2.4e6, 2048, 8, 2048 * 10, "hamming", crop="thread")      # row_width 256
    for scroll, key in ((1, "img_pos"), (-1, "img_neg")):
        wf = Waterfall(engine, scroll=scroll)
        img = None
        for n, r in enumerate(rows, 1):
            r = r.copy()
            wf.image_update(r)
            assert r[0] == 0 and r[128] == 0 and r[255] == 0       # mutated in place like the reference
            if n in (1, 2, 5, 6, 7, 20, 63, 64, 65, 70):
                ref = None
                for rr in rows[:n]:
                    ref = zo.waterfall_update(ref, rr.copy(), scroll)
                got = wf.img_array
                # device rows are float32
                assert got.shape == ref.shape
                assert np.abs(got - ref).max() < 1e-4, (scroll, n)
        assert np.abs(wf.img_array - g[key]).max() < 1e-4


def waterfall_display(engine):
    """Device-side display path (SURVEY 8f.1): colour indices / RGBA of the
    image and the autolevel percentiles, against the oracle's restatement of
    pyqtgraph's level mapping and the reference's own autolevel (golden)."""
    g = np.load(os.path.join(parity.GOLDEN_DIR, "waterfall.npz"))
    engine.configure(2.4e6, 2048, 8, 2048 * 10, "hamming", crop="thread")      # row_width 256
    lut = zo.colormap_lut([0., 0.5, 1.], [[0, 0, 0, 255], [0, 255, 0, 255], [255, 0, 0, 255]])   # 'Red Green' S:1583
    for name, rows in (("noise", gc.waterfall_rows_noise()), ("ramp", gc.waterfall_rows_ramp())):
        for scroll, tag in ((1, "pos"), (-1, "neg")):
            wf = Waterfall(engine, scroll=scroll)
            ref = None
            for n, r in enumerate(rows, 1):
                wf.image_update(r.copy())
                ref = zo.waterfall_update(ref, r.copy(), scroll)
                if n not in (1, 3, 7, len(rows)):
                    continue
                img = wf.img_array                                   # float32 rows on the device
                assert np.abs(img - ref).max() < 1e-4
                # bit-exact against the oracle on the pixels the device holds
                for levels in ((-220, -120), (-180.5, -99.25), (-150.001, -149.999), (-1e6, 1e6)):
                    idx = wf.image_indices(levels)
                    assert idx.dtype == np.uint8 and idx.shape == img.shape
                    assert np.array_equal(idx, zo.waterfall_indices(img, *levels)), (name, tag, n, levels)
                rgba = wf.image_rgba(lut)
                assert np.array_equal(rgba, zo.waterfall_rgba(zo.waterfall_indices(img), lut))
                wf.autolevel()
                want = zo.waterfall_autolevel(img)
                assert (wf.minlevel, wf.maxlevel) == want, (name, tag, n, wf.minlevel, wf.maxlevel, want)
            ret = wf.autolevel()
            assert ret == (-220, -120)                               # S:1676-1677: levels in use are untouched
            gold = g["auto_%s_%s" % (name, tag)]
            if name == "noise":                                      # float32-representable rows: exact
                assert (wf.minlevel, wf.maxlevel) == (gold[0], gold[1])
            else:
                assert abs(wf.minlevel - gold[0]) < 1e-4 and abs(wf.maxlevel - gold[1]) < 1e-4
            assert wf.autolevel(fix=True) == (wf.minlevel, wf.maxlevel)
    # quantile edge cases: nothing below zero yet / every requested rank
    wf = Waterfall(engine)
    wf.fftwidth = 256
    wf.init_image()
    q, n = engine.ring_quantiles(64, 1, 0, [0.0, 0.5, 1.0])
    assert n == 64 * 254 and list(q) == [-500.0, -500.0, -500.0]
    row = np.linspace(-90.0, -10.0, 256).astype(np.float32)
    wf.image_update(row.astype(np.float64))
    img = wf.img_array
    qs = [0.0, 0.001, 0.25, 0.5, 0.75, 0.98, 0.9999, 1.0]
    got, n = engine.ring_quantiles(64, 1, 1, qs)
    sel = img[img < 0]
    assert n == sel.size
    assert np.array_equal(got, np.quantile(sel, qs))


def waterfall_random_shapes(engine, seeds=range(6)):
    """Image / indices / percentiles against the oracle for random row widths
    (incl. widths that are not a multiple of 4: the scalar pixel path), scroll
    directions, row counts around the wrap and level pairs."""
    for seed in seeds:
        rng = np.random.default_rng(1000 + seed)
        w = int(rng.choice([60, 62, 100, 130, 250, 256, 510, 1000]))
        h = w // 4
        scroll = int(rng.choice([1, -1]))
        nrows = int(rng.choice([1, 4, 6, 7, h - 1, h, h + 1, h + 9]))
        # any configuration with that row width: no zoom, crop = w
        engine.configure(1e6, 1024, 1, 4096, "hann", crop=w)
        assert engine.row_width == w
        wf = Waterfall(engine, scroll=scroll)
        ref = None
        for i in range(nrows):
            r = (-160.0 + 25.0 * rng.standard_normal(w)).astype(np.float32).astype(np.float64)
            if i % 3 == 0:
                r[rng.integers(0, w, 3)] = [np.float32(3.5), -np.inf, 0.0]      # above zero, -inf, zero
            wf.image_update(r.copy())
            ref = zo.waterfall_update(ref, r.copy(), scroll)
        img = wf.img_array
        assert img.shape == (h, w) and np.array_equal(img, ref), (seed, w, scroll, nrows)
        lo = float(rng.uniform(-300, -100))
        levels = (lo, lo + float(rng.uniform(0.5, 200)))
        assert np.array_equal(wf.image_indices(levels), zo.waterfall_indices(ref, *levels)), (seed, w, levels)
        qs = np.sort(rng.uniform(0, 1, 3))
        got, n = engine.ring_quantiles(h, scroll, wf.rows_seen, qs)
        sel = ref[ref < 0]
        assert n == sel.size and np.array_equal(got, np.quantile(sel, qs)), (seed, w, qs)


def level_mapping_edges(engine):
    """Colour index at, just below and just above every one of the 255 index
    steps, for several level pairs: the device's fp32 guess + threshold
    compares must land on the double-precision formula's index everywhere."""
    w = 768
    engine.configure(1e6, 1024, 1, 4096, "hann", crop=w)
    pairs = [(-220.0, -120.0), (-180.5, -99.25), (-300.0, 0.0), (-100.0, 100.0), (-153.7, -151.2),
             (-1e4, 1e4), (-130.0, -129.0), (3.0, 40.0)]
    for lo, hi in pairs:
        scale = 256.0 / (hi - lo)
        # float32 values around the exact step positions lo + k / scale
        steps = (lo + np.arange(1, 256) / scale).astype(np.float32)
        vals = np.concatenate([steps, np.nextafter(steps, np.float32(-np.inf)), np.nextafter(steps, np.float32(np.inf))])
        assert vals.size == 765
        row = np.concatenate([vals, np.float32([lo, hi, -np.inf])]).astype(np.float32)
        wf = Waterfall(engine)
        wf.image_update(row.astype(np.float64))
        img = wf.img_array
        idx = wf.image_indices((lo, hi))
        assert np.array_equal(idx, zo.waterfall_indices(img, lo, hi)), (lo, hi)
        # and the steps really are exercised: the three rows of values straddle index changes
        got = idx[idx.shape[0] - 2, 1:255]
        assert len(np.unique(got)) > 200


def waterfall_from_engine_rows(engine):
    """Rows the engine produced itself are not pushed twice."""
    w = synth.CFG1
    n = 2048 * 10
    frames = synth.make_frames(w, 3, n=n)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop="thread")
    wf = Waterfall(engine)
    wf.fftwidth = 256
    wf.init_image()
    for f in frames:
        row = engine.process(f)[0].astype(np.float64)
        wf.note_engine_rows(1)
        wf.image_update(row)
    assert engine.rows_written == 3
    img = wf.img_array
    h = img.shape[0]
    last = engine.read_rows(1)[0].astype(np.float64)
    last[[0, 128, 255]] = 0
    assert np.array_equal(img[h - 2], last)


def scipy_shaped_calls(engine):
    """pypanadapter_b200.signal.decimate / welch against scipy's own."""
    import scipy.signal
    from pypanadapter_b200 import signal as zsig
    rng = np.random.default_rng(17)
    x = (rng.standard_normal(6000) + 1j * rng.standard_normal(6000)) * 0.3
    x += 0.5 * np.exp(2j * np.pi * 0.0123 * np.arange(6000))
    y = zsig.decimate(x, 2, engine=engine)
    ref = scipy.signal.decimate(x, 2)
    assert y.dtype == np.complex128 and y.shape == ref.shape
    assert np.abs(y - ref).max() < 2e-6 * np.abs(ref).max() + 1e-7
    y4 = zsig.decimate(x.astype(np.complex64), 4, engine=engine)
    ref4 = scipy.signal.decimate(scipy.signal.decimate(x, 2), 2)
    assert y4.dtype == np.complex64 and np.abs(y4 - ref4).max() < 5e-6
    f, p = zsig.welch(x, 48e3, window="hamming", nperseg=512, nfft=512, engine=engine)
    fr, pr = scipy.signal.welch(x, 48e3, window="hamming", nperseg=512, nfft=512)
    assert np.array_equal(f, fr) and p.dtype == np.float64
    assert np.abs(10 * np.log10(p / pr)).max() < 0.005
    import pytest
    with pytest.raises(NotImplementedError):
        zsig.decimate(x, 3, engine=engine)
    # real input: one-sided density, natural order (scipy:_spectral_py.py:915-916)
    xr = np.ascontiguousarray(x.real)
    f1, p1 = zsig.welch(xr, 48e3, window="hann", nperseg=512, nfft=512, engine=engine)
    f1r, p1r = scipy.signal.welch(xr, 48e3, window="hann", nperseg=512, nfft=512)
    assert np.array_equal(f1, f1r) and p1.shape == (257,) and p1.dtype == np.float64
    assert np.abs(10 * np.log10(p1 / p1r)).max() < 0.005
    p32 = zsig.welch(xr.astype(np.float32), 48e3, nperseg=256, nfft=256, engine=engine)[1]
    assert p32.dtype == np.float32 and p32.shape == (129,)
    with pytest.raises(NotImplementedError):
        zsig.welch(xr, 48e3, nperseg=512, return_onesided=False, engine=engine)
    with pytest.raises(ValueError):
        zsig.decimate(x[:27], 2, engine=engine)          # scipy: padlen


def dropin_on_standin_modules(engine):
    """dropin.install on stand-in modules with the reference's class / method
    names and EMPTY hot-path bodies (tests/standin_pan.py) -- runs wherever the
    library runs, the GPU box included: every row below comes out of the engine
    and is held to the reference-recorded goldens."""
    from pypanadapter_b200 import dropin
    from tests import standin_pan as sp
    # ---- spectrum variant: ApplicationDisplay.update(chunk), zoomfft, Waterfall ----
    mod = sp.make("spectrum")
    saved = dropin.install(mod, engine=engine)
    try:
        for name in ("cfg1_S1024", "cfg1_S256", "defaults_S"):
            case = gc.case_by_name(name)
            x = gc.make_input(case)
            sp.set_state(mod, case["fs"], case["N"], case["R"], len(x) // case["N"], case["window"])
            app = mod.ApplicationDisplay(case["n_win"])
            got = {}
            app.waterfall = types.SimpleNamespace(image_update=lambda psd: got.__setitem__("psd", psd.copy()))
            app.update(x)
            floor = parity.floor_db20(case["fs"], case["window"], case["N"], case["R"] > 1)
            parity.assert_row_parity(got["psd"], parity.golden_rows()[name], floor, "stand-in dropin " + name)
            assert "N_FFT: %d" % case["N"] in app.win.calls["setWindowTitle"][0][0]          # S:2105-2106
            assert app.spectrum_plot.calls["setData"][0][0].shape == (case["n_win"],)        # S:2128-2130
        case = gc.ZOOMFFT_CASES[0]
        x = gc.make_input(case)
        sp.set_state(mod, case["fs"], case["N"], case["R"], len(x) // case["N"], "hamming")
        z = mod.ApplicationDisplay(256).zoomfft(x, case["R"])
        ref = np.load(os.path.join(parity.GOLDEN_DIR, "zoomfft.npz"))[case["name"]]
        assert np.abs(z - ref).max() < 2e-5 * np.abs(ref).max()
        # raw RTL bytes (rtl_tcp byte callback): converted and flipped on the device == the
        # reference's update on what RTLSDRstream.read_callback would have emitted (S:459-460)
        case = gc.case_by_name("cfg1_S256")
        raw = synth.quantise_u8(0.8 * gc.make_input(case))
        sp.set_state(mod, case["fs"], case["N"], case["R"], len(raw) // 2 // case["N"], case["window"])
        app = mod.ApplicationDisplay(case["n_win"])
        got = {}
        app.waterfall = types.SimpleNamespace(image_update=lambda psd: got.__setitem__("psd", psd.copy()))
        app.update(raw)
        want = zo.zoom_psd(raw, case["fs"], case["N"], case["R"], case["window"], crop=case["n_win"], flip=True)
        parity.assert_row_parity(got["psd"], want, parity.floor_db20(case["fs"], case["window"], case["N"], True),
                                 "stand-in dropin raw u8")
        # ---- Waterfall in both scroll directions: its methods on the device ring ----
        g = np.load(os.path.join(parity.GOLDEN_DIR, "waterfall.npz"))
        engine.configure(2.4e6, 2048, 8, 2048 * 10, "hamming", crop="thread")      # row_width 256
        for scroll, tag in ((1, "pos"), (-1, "neg")):
            mod.AppState.scroll = scroll
            wf = mod.Waterfall()
            ref = None
            for r in gc.waterfall_rows_noise():
                psd = r.copy()
                wf.image_update(psd)
                assert psd[0] == 0 and psd[128] == 0 and psd[255] == 0             # S:1647-1648
                ref = zo.waterfall_update(ref, r.copy(), scroll)
            assert wf.shown["kw"]["levels"] == [0, 256] and wf.shown["kw"]["autoLevels"] is False
            assert np.array_equal(wf.shown["img"], zo.waterfall_indices(ref, -220, -120).T)
            assert np.abs(wf.img_array - ref).max() < 1e-4
            assert wf.autolevel() == (-220, -120)
            gold = g["auto_noise_" + tag]
            assert (wf.minlevel, wf.maxlevel) == (gold[0], gold[1])                # the reference's own autolevel
            assert wf.newlevel(-180.0, -100.0) == (-180.0, -100.0)
            wf.image_update(gc.waterfall_rows_noise()[-1].copy())
            ref = zo.waterfall_update(ref, gc.waterfall_rows_noise()[-1].copy(), scroll)
            assert np.array_equal(wf.shown["img"], zo.waterfall_indices(ref, -180.0, -100.0).T)
        mod.AppState.scroll = 1
        # update(chunk) -> Waterfall.image_update: the image the reference would hold, each row
        # entering the ring once, in order
        case = gc.case_by_name("cfg1_S256")
        app = mod.ApplicationDisplay(256)
        ref_img = None
        rows = []
        for i in range(4):
            x = synth.make_frame(synth.CFG1, i)
            sp.set_state(mod, case["fs"], case["N"], case["R"], len(x) // case["N"], case["window"])
            app.update(x)
            rows.append(engine.read_rows(1)[0].astype(np.float64))
            ref_img = zo.waterfall_update(ref_img, rows[-1].copy(), 1)
        assert np.array_equal(app.waterfall.img_array, ref_img)
        assert np.array_equal(app.waterfall.shown["img"], zo.waterfall_indices(ref_img, -220, -120).T)
        for j, r in enumerate(reversed(rows)):
            r = r.copy()
            r[[0, 128, 255]] = 0
            assert np.array_equal(app.waterfall.img_array[64 - 2 - j], r), j
        # ---- the taper dialog's ShowCurve (S:1354-1379) ----
        import scipy.signal
        for tname, p0, p1, spec in (("hamming", 0, 0, "hamming"), ("kaiser", 9.5, 0, ("kaiser", 9.5)),
                                    ("general gaussian", 1.5, 7.0, ("general gaussian", 1.5, 7.0))):
            dlg = mod.FFTTaperingControl(tname, p0, p1)
            dlg.ShowCurve()
            assert mod.AppState.fft_tapering == spec
            ref_t = scipy.signal.get_window(spec, 51)
            assert np.abs(dlg.taperplot.calls["setData"][0][0] - ref_t).max() < 1e-12
            fft = np.fft.fft(ref_t, 2048) / (len(ref_t) / 2.0)
            ref_f = 20 * np.log10(np.abs(fft / np.max(np.abs(fft))))
            shown = dlg.fftplot.calls["setData"][0][0]
            vis = ref_f > -140.0
            assert np.abs(shown[vis] - ref_f[vis]).max() < 2e-3
            dlg.P0val.v = p0 + 1
            dlg.ShowCurve()                                   # second call: existing curves are updated
            assert len(dlg.plot0.items) == 1 and len(dlg.plot1.items) == 1
    finally:
        dropin.uninstall(mod, saved)
    assert mod.ApplicationDisplay.update is saved["ApplicationDisplay.update"]
    assert mod.Waterfall.__dict__["image_update"] is saved["Waterfall.image_update"]
    assert "img_array" not in mod.Waterfall.__dict__                    # added by install: removed again
    # ---- thread variant: Data, PSD.update, and the GUI timer (T:2140-2157) ----
    mod = sp.make("thread")
    saved = dropin.install(mod, engine=engine)
    try:
        case = gc.case_by_name("cfg1_T")
        x = gc.make_input(case)
        st = sp.set_state(mod, case["fs"], case["N"], case["R"], 1, case["window"])
        d = mod.Data()
        assert isinstance(d, buffers_Data())
        d.new_complex()
        psd = mod.PSD(d)
        app = mod.ApplicationDisplay(psd)
        # the timer fires before any row exists: the blank np.zeros(fft_size) row (T:1490) is shown
        app.update()
        assert app.waterfall.fftwidth == case["N"] and app.waterfall.shown["img"].shape == (case["N"], case["N"] // 4)
        blank = zo.waterfall_update(None, np.zeros(case["N"]), 1)
        assert np.array_equal(app.waterfall.img_array, blank)

        def feed():
            for i in range(0, len(x), d.chunk_size):
                d.add(x[i:i + d.chunk_size])
        feed()
        psd.update()
        floor = parity.floor_db20(case["fs"], case["window"], case["N"], True)
        parity.assert_row_parity(psd.psd, parity.golden_rows()["cfg1_T"], floor, "stand-in PSD.update")
        app.update()                                          # new width: the image starts over (S:1641-1643)
        W = 2 * int(.5 * case["N"] / case["R"])
        assert app.waterfall.fftwidth == W and app.waterfall.shown["img"].shape == (W, W // 4)
        assert engine.rows_written == 1
        img = zo.waterfall_update(None, np.array(psd.psd, dtype=np.float32).astype(np.float64), 1)
        assert np.array_equal(app.waterfall.img_array, img)
        # a row PSD.update computes but the timer never shows stays out of the ring (T:2140-2148)
        feed()
        psd.update()
        assert engine.rows_written == 1
        # a zoom click (S:2079-2086 makes fft_ratio a float): PSD.update has re-planned for the new
        # width while the timer still shows the row of the old one -- then the new row arrives
        st.fft_ratio = case["R"] * 2.0
        feed()
        stale = np.array(psd.psd, copy=True)
        engine.configure(case["fs"], case["N"], st.fft_ratio, len(x), case["window"], crop="thread")
        app.update()                                          # stale 256-wide row, engine now at 128
        img = zo.waterfall_update(img, np.array(stale, dtype=np.float32).astype(np.float64), 1)
        assert np.array_equal(app.waterfall.img_array, img)
        psd.update()
        assert psd.psd.shape == (W // 2,)
        app.update()
        assert app.waterfall.fftwidth == W // 2
        assert np.array_equal(app.waterfall.img_array,
                              zo.waterfall_update(None, np.array(psd.psd, dtype=np.float32).astype(np.float64), 1))
        # a second Data on the same engine takes the pinned ring over; the first one goes on
        # working on private memory (late add() of an old reader thread)
        d2 = mod.Data()
        d2.new_complex()
        assert d._detached and not d2._detached
        d.add(x[:d.chunk_size])
        for i in range(0, len(x), d2.chunk_size):
            d2.add(x[i:i + d2.chunk_size])
        st.fft_ratio = case["R"]
        psd2 = mod.PSD(d2)
        psd2.update()
        parity.assert_row_parity(psd2.psd, parity.golden_rows()["cfg1_T"], floor, "stand-in PSD.update (2nd Data)")
        d2.target = 100000
        assert d2.target == 100000
        d2.target = 10                                        # below fft_size: ignored (T:1476)
        assert d2.target == 100000
    finally:
        dropin.uninstall(mod, saved)
    assert mod.Data is saved["Data"] and mod.PSD.update is saved["PSD.update"]
    engine.configure(2.4e6, 2048, 16, 2048 * 10, "hamming", crop="thread")
    assert engine.row_width == engine.ring_width == W // 2    # the ring keeps rows of its own width only
    n0 = engine.rows_written
    engine.process(synth.make_frame(synth.CFG1, 0, 2048 * 10))
    assert engine.rows_written == n0 + 1                      # uninstall restored ring_append


def fast_mode_state_survives_frame_len(engine):
    """A live stream hands PSD.update a different number of samples every take
    (T:1516-1520).  In mode fast that must neither restart the EMA nor empty the
    waterfall ring (zfb_configure keeps both unless W, N, R change)."""
    fs, N, R = 2.4e6, 1024, 8
    rows = []
    engine.ring_configure(16)
    for i, n in enumerate((N * 24, N * 24 + 512, N * 25, N * 24)):
        x = gc.tone_noise(n, fs, [(3000.0 + 500 * i, 0.4)], 3e-3, 40 + i, np.complex64)
        engine.configure(fs, N, R, n, "hamming", crop="thread", ema_alpha=0.3, mode="fast")
        assert engine.fast_active
        rows.append(engine.process(x)[0].astype(np.float64))
    assert engine.rows_written == 4
    assert np.array_equal(engine.read_rows(4).astype(np.float64), np.array(rows))
    # the oracle's EMA over the same four frames
    lin = []
    for i, n in enumerate((N * 24, N * 24 + 512, N * 25, N * 24)):
        x = gc.tone_noise(n, fs, [(3000.0 + 500 * i, 0.4)], 3e-3, 40 + i, np.complex64)
        lin.append(zo.zoom_psd_power(x, fs, N, R, "hamming", crop="thread"))
    want = zo.ema_rows_db20(np.array(lin), 0.3)
    floor = parity.floor_db20(fs, "hamming", N, True)
    for r, w in zip(rows, want):
        parity.assert_row_parity(r, w, floor, "EMA across frame_len changes")
    engine.ring_configure(256)


def ring_wrap_within_one_launch(engine):
    """More frames in one launch than the ring has rows: the ring ends up with
    the NEWEST rows, each row whole (no per-column mix of frames sharing a slot)."""
    fs, N = 2.4e6, 256
    n = N * 4
    frames = np.stack([gc.tone_noise(n, fs, [(1.0e5 * (1 + i % 7), 0.3)], 3e-3, 100 + i, np.complex64)
                       for i in range(40)])
    engine.ring_configure(8)
    engine.configure(fs, N, 1, n, "hann", crop=None)
    rows = engine.process(frames)
    assert engine.rows_written == 40
    assert np.array_equal(engine.read_rows(8), rows[-8:])
    engine.ring_configure(256)


def event_driven_run(engine):
    """PSD.run(event_driven=True): rows appear when enough samples have arrived,
    not on a timer (SURVEY 8f.2): a producer delivering one frame's worth every
    ~100 ms yields ~one row per delivery, and nothing while it is silent."""
    import threading
    import time
    w = synth.CFG1
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    psd.FRAME_TIME = 0.05
    frame = synth.make_frame(w, 0)
    need = 4 * d.chunk_size                                   # 65568 samples per row
    count = [0]
    orig = psd.update

    def counted():
        orig()
        count[0] += 1
    psd.update = counted
    t = threading.Thread(target=psd.run, kwargs=dict(event_driven=True, frame_samples=need))
    t.start()
    try:
        time.sleep(0.15)
        assert count[0] == 0                                   # silent source: no rows
        for _ in range(5):
            for k in range(4):
                d.add(frame[k * d.chunk_size:(k + 1) * d.chunk_size])
            time.sleep(0.1)
        deadline = time.time() + 5
        while count[0] < 5 and time.time() < deadline:
            time.sleep(0.01)
        assert 3 <= count[0] <= 6, count[0]              # (a slow consumer may merge deliveries)
        assert psd.psd.shape == (2 * int(.5 * w.fft_size / w.fft_ratio),) and np.all(np.isfinite(psd.psd))
    finally:
        psd.loop = False
        t.join(timeout=10)
    assert not t.is_alive()


def rtl_tcp_source(engine):
    """RtlTcpPan against a fake rtl_tcp server on localhost: greeting parsed,
    commands framed as rtl_tcp expects, raw bytes streamed into Data.new_u8()
    and PSD.update's row equals the oracle's for the same bytes (cfg2 shape)."""
    import socket
    import threading
    import time
    from pypanadapter_b200.replay import RtlTcpPan
    w = synth.CFG2
    raw = synth.make_frame(w, 0)                               # uint8 IQ, 2*frame_len bytes
    assert raw.dtype == np.uint8
    srv = socket.socket()
    srv.bind(("127.0.0.1", 0))
    srv.listen(1)
    port = srv.getsockname()[1]
    got_cmds = []

    def serve():
        conn, _ = srv.accept()
        conn.sendall(b"RTL0" + (5).to_bytes(4, "big") + (29).to_bytes(4, "big"))
        conn.settimeout(0.5)
        try:
            for _ in range(3):                                   # sample rate, direct sampling, frequency
                got_cmds.append(conn.recv(5, socket.MSG_WAITALL))
        except OSError:
            pass
        try:
            conn.sendall(raw.tobytes())
            time.sleep(0.5)
        finally:
            conn.close()
    th = threading.Thread(target=serve, daemon=True)
    th.start()
    pan = RtlTcpPan("127.0.0.1", port, sample_rate=w.fs)
    assert (pan.tuner_type, pan.gain_count, pan.Mode) == (5, 29, "Stream")
    pan.SetFrequency(8.8315e6)                                   # TS-180S IF (S:106): direct sampling
    d = Data(engine=engine).new_u8()
    chunk = 16384
    nchunks = 15                                                 # 245760 samples: below Data's fold-back (T:1440)
    seen = []
    done = threading.Event()

    def on_chunk(b):
        if len(seen) >= nchunks:                                 # the pump keeps reading until Close()
            return
        d.add(b)
        seen.append(len(b))
        if len(seen) == nchunks:
            done.set()
    pan.Stream(on_chunk, chunk)
    assert done.wait(10), "stream stalled after %d chunks" % len(seen)
    pan.Close()
    th.join(timeout=5)
    srv.close()
    assert got_cmds[0] == bytes([0x02]) + int(w.fs).to_bytes(4, "big")
    assert got_cmds[1] == bytes([0x09]) + (2).to_bytes(4, "big")
    assert got_cmds[2] == bytes([0x01]) + int(8.8315e6).to_bytes(4, "big")
    assert all(n == 2 * chunk for n in seen[:nchunks])
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    psd = PSD(d, state, flip=True)
    psd.update()
    n = nchunks * chunk
    want = zo.zoom_psd(raw[:2 * n], w.fs, w.fft_size, w.fft_ratio, w.window, flip=True)
    parity.assert_row_parity(psd.psd, want, parity.floor_db20(w.fs, w.window, w.fft_size, True), "rtl_tcp row")


def buffers_Data():
    from pypanadapter_b200.buffers import Data as D
    return D


def producer_consumer_threads(engine):
    """DataReader-style producer thread (T:2187-2195) and PSD.run-style consumer
    thread (T:1498-1511) hammering one Data/PSD pair: no deadlock, no torn
    state, every published row is a finite full-width row."""
    import threading
    import time
    w = synth.CFG1
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    frame = synth.make_frame(w, 0)
    stop = threading.Event()
    errors = []

    def producer():
        i = 0
        try:
            while not stop.is_set():
                a = (i * d.chunk_size) % (len(frame) - d.chunk_size)
                d.add(frame[a:a + d.chunk_size])
                i += 1
        except Exception as exc:                      # pragma: no cover
            errors.append(exc)

    rows = []

    def consumer():
        try:
            while not stop.is_set():
                psd.update()
                psd.lock.lock()
                r = psd.psd
                psd.lock.unlock()
                if len(r) == 2 * int(.5 * w.fft_size / w.fft_ratio):
                    rows.append(np.array(r, copy=True))
                time.sleep(0.002)
        except Exception as exc:                      # pragma: no cover
            errors.append(exc)

    ts = [threading.Thread(target=producer), threading.Thread(target=consumer)]
    for t in ts:
        t.start()
    time.sleep(1.0)
    stop.set()
    for t in ts:
        t.join(timeout=20)
        assert not t.is_alive(), "thread did not finish (deadlock?)"
    assert not errors, errors
    assert len(rows) >= 3
    for r in rows:
        assert r.shape == (256,) and np.all(np.isfinite(r)) and r.max() > -120.0
    assert 0 <= d.size <= d.max_size and d.real_size <= d.max_size


def replay_source_through_plugin_api(engine):
    """cfg2 through the reference's own plug-in surface: ReplayPan.Read ->
    Data.add -> PSD.update (complex path, flipped per chunk like RTLSDR.Read),
    and ReplayPan.ReadRaw -> Data.new_u8 (wire format, device conversion)."""
    from pypanadapter_b200.replay import ReplayPan
    w = synth.CFG2
    n = w.fft_size * 40
    raw = synth.make_frame(w, 0, n=n)
    state = types.SimpleNamespace(fft_size=w.fft_size, fft_ratio=w.fft_ratio, fft_tapering=w.window,
                                  panadapter=types.SimpleNamespace(SampleRate=w.fs))
    floor = parity.floor_db20(w.fs, w.window, w.fft_size, True)
    # complex path: DataReader.run's loop (T:2187-2191)
    pan = ReplayPan(raw, w.fs)
    assert pan.Mode == "Block" and pan.SampleRate == w.fs and pan.driver
    d = Data(engine=engine).new_complex()
    psd = PSD(d, state)
    chunks = []
    for _ in range(n // d.chunk_size):
        c = pan.Read(d.chunk_size)
        chunks.append(c)
        d.add(c)
    psd.update()
    want = zo.zoom_psd(np.concatenate(chunks), w.fs, w.fft_size, w.fft_ratio, w.window)
    parity.assert_row_parity(psd.psd, want, floor, "replay complex path")
    # wire-format path
    pan = ReplayPan(raw, w.fs)
    d = Data(engine=engine).new_u8()
    psd = PSD(d, state, flip=True)
    got_raw = []
    for _ in range(n // d.chunk_size):
        c = pan.ReadRaw(d.chunk_size)
        got_raw.append(c)
        d.add(c)
    psd.update()
    want = zo.zoom_psd(np.concatenate(got_raw), w.fs, w.fft_size, w.fft_ratio, w.window, flip=True)
    parity.assert_row_parity(psd.psd, want, floor, "replay u8 path")
    # looping and EOF
    small = ReplayPan(raw[:20], w.fs, loop=True)
    assert len(small.ReadRaw(25)) == 50
    import pytest
    with pytest.raises(EOFError):
        ReplayPan(raw[:20], w.fs, loop=False).ReadRaw(25)


def taper_design_and_preview(engine):
    """SURVEY 8f.4: the taper dialog's two curves (S:1354-1379) from the device, against the
    scipy / numpy calls the reference makes, for every entry of its taper_list (S:1222-1243)."""
    import warnings
    import scipy.signal
    from pypanadapter_b200 import taper
    dialog = {                                            # FFTTaperingControl.taper_list with its defaults
        "barthann": (), "bartlett": (), "blackmanharris": (), "blackman": (), "bohman": (), "boxcar": (),
        "flattop": (), "hamming": (), "hann": (), "parzen": (), "nuttall": (), "triang": (),
        "kaiser": (14,), "gaussian": (7,), "general gaussian": (1.5, 7), "dpss": (3,), "chebwin": (100,),
        "exponential": (3,), "tukey": (.3,),
    }
    ndev = 0
    for name, par in dialog.items():
        spec = name if not par else (name,) + par
        for n in (51, 52, 2048, 1):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                want = scipy.signal.get_window(spec, n)
            got = taper.get_window(spec, n, engine=engine)
            assert got.shape == want.shape
            assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (name, n)
        ndev += taper.on_device(spec)
        taperdata, taperfft = taper.show_curve(spec, engine=engine)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref_t = scipy.signal.get_window(spec, 51)
            fft = np.fft.fft(ref_t, 2048) / (len(ref_t) / 2.0)
            ref_f = 20 * np.log10(np.abs(fft / np.max(np.abs(fft))))
        assert np.abs(taperdata - ref_t).max() < 1e-12
        # the dialog's plot spans 0 .. -140 dB (S:1278): compare there, nulls are bottomless
        vis = ref_f > -140.0
        assert np.abs(taperfft[vis] - ref_f[vis]).max() < 2e-3, name
    assert ndev == 17
    # symmetric designs and other parameters
    for spec in (("kaiser", 8.6), ("tukey", 0.0), ("tukey", 1.0), ("tukey", 0.5), ("gaussian", 300.0),
                 ("general gaussian", 0.7, 12.0), "hann", "triang", "parzen", "bohman"):
        for n in (8, 9, 64):
            want = scipy.signal.get_window(spec, n, fftbins=False)
            got = taper.get_window(spec, n, fftbins=False, engine=engine)
            assert np.abs(got - want).max() <= 1e-12, (spec, n)
    with pytest.raises(ValueError):
        taper.get_window("kaiser", 51, engine=engine)
