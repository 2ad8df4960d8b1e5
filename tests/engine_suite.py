"""Engine-level checks shared by tests/test_emu_engine.py (CPU emulation of
the same sources -- logic only) and tests/test_gpu_parity.py (the product, on
a B200, through the C ABI).  Every function takes a configured-or-not
``ZoomPSD`` and asserts."""
from __future__ import annotations

import numpy as np
import pytest

from oracle import golden_cases as gc
from oracle import zoompsd_oracle as zo
from pypanadapter_b200 import synth
from pypanadapter_b200.engine import ZoomFFTError
from tests import parity


def golden_case(engine, name):
    return parity.check_case(engine, name)


def ema_rows(engine, nframes=4):
    """cfg2: uint8 + flip + EMA 0.3 across rows (EMA = builder-defined
    extension, oracle ema_rows_db20).  Frames pushed in two calls to check
    that the state carries across calls and groups."""
    w = synth.CFG2
    frames = synth.make_frames(w, nframes)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8",
                     flip=True, crop="thread", ema_alpha=w.ema_alpha)
    engine.reset_ema()
    got = np.concatenate([engine.process(frames[:1]), engine.process(frames[1:])])
    pw = np.stack([zo.zoom_psd_power(f, w.fs, w.fft_size, w.fft_ratio, w.window, flip=True)
                   for f in frames])
    want = zo.ema_rows_db20(pw, w.ema_alpha)
    floor = parity.floor_db20(w.fs, w.window, w.fft_size, True)
    for i in range(nframes):
        parity.assert_row_parity(got[i], want[i], floor, "ema row %d" % i)
    # and without EMA each row equals the golden reference row
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8",
                     flip=True, crop="thread", ema_alpha=None)
    plain = engine.process(frames)
    for i in range(nframes):
        parity.assert_row_parity(plain[i], parity.golden_rows()["cfg2_T_f%d" % i], floor,
                                 "cfg2 frame %d" % i)


def batch_equals_single(engine, lib):
    """Frames are independent (S:2092, S:2098, S:2111 restart per chunk): a
    batch must give bit-identical rows to one-at-a-time calls, in any group
    size."""
    w = synth.CFG1
    n = 2048 * 24
    frames = synth.make_frames(w, 5, n=n)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop=1024)
    single = np.stack([engine.process(frames[i])[0] for i in range(5)])
    batch = engine.process(frames)
    assert np.array_equal(single, batch)
    engine.set_group(2)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop=1024)
    assert np.array_equal(engine.process(frames), batch)
    engine.set_group(0)


class HostAsDevice:
    """Device buffers of the CPU emulation build are host memory."""

    def put(self, a):
        a = np.ascontiguousarray(a)
        return a.ctypes.data, a

    def empty(self, shape):
        a = np.zeros(shape, dtype=np.float32)
        return a.ctypes.data, a

    def get(self, obj):
        return np.array(obj)


class TorchDevice:
    def put(self, a):
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)).cuda()
        return t.data_ptr(), t

    def empty(self, shape):
        import torch
        t = torch.zeros(shape, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        return t.data_ptr(), t

    def get(self, obj):
        return obj.cpu().numpy()


def ema_batch_independent(engine):
    """EMA rows do not depend on where a launch group or a call ends -- on the fp64 path of
    few-segment rows too (its state between launches is fp32 like the fp32 path's)."""
    w = synth.CFG2
    for n in (4096 * 16 + 1234, 4096 * 16 * 4 + 1234):          # 1 segment (fp64 path), 7 segments
        frames = synth.make_frames(w, 7, n=n)
        rows = []
        for group, calls in ((0, [7]), (2, [7]), (3, [4, 3]), (0, [1] * 7)):
            engine.set_group(group)
            engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, dtype="u8", flip=True, crop="thread",
                             ema_alpha=0.3)
            engine.reset_ema()
            f0, got = 0, []
            for cnt in calls:
                got.append(engine.process(frames[f0:f0 + cnt]))
                f0 += cnt
            rows.append(np.concatenate(got))
        engine.set_group(0)
        for r in rows[1:]:
            assert np.array_equal(r, rows[0])


def pipeline_equals_one_lane(engine, dev, nframes=9, w=None, n=None):
    """``pipeline`` = 1: whole batches alternate between the lane engines, rows are finished on a
    stream of the engine's own and the caller's stream joins later (zfb_join).  Rows, EMA across
    batches, ring, counters: bit-identical to the plain path; other calls join implicitly.  An
    option changed between batches reaches the lanes, and the decimated chunk is read from the
    lane that ran the last batch."""
    w = w or synth.CFG2
    n = n or 4096 * 16 * 4 + 1234           # 7 Welch segments: the fp32 path
    frames = synth.make_frames(w, nframes, n=n)
    p_in, keep = dev.put(frames)
    fbytes = frames[0].nbytes

    def run(pipeline, group, calls, host_tail=0):
        engine.set_option("pipeline", pipeline)
        engine.set_group(group)
        engine.ring_configure(4)
        engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, dtype=w.dtype, flip=w.flip, crop="thread",
                         ema_alpha=0.3)
        assert engine.fast_active
        engine.reset_ema()
        k0 = engine.counters()
        p_rows, rows = dev.empty((nframes, engine.row_width))
        f0 = 0
        for cnt in calls:
            engine.process_device(p_in + f0 * fbytes, cnt, p_rows + f0 * engine.row_width * 4)
            assert engine.slab_lanes == (2 if pipeline else 1)
            f0 += cnt
        tail = None
        if host_tail:                        # a host-path call right behind pipelined batches: implicit join
            tail = engine.process(frames[:host_tail])
        else:
            engine.join()
        engine.synchronize()
        k1 = engine.counters()
        return dev.get(rows)[:f0], engine.read_rows(4), tail, {k: k1[k] - k0[k] for k in ("frames", "samples")}, \
            engine.read_decimated().shape

    try:
        for host_tail in (0, 2):
            want = run(0, 0, [nframes - host_tail], host_tail)
            for group, calls in ((0, [nframes - host_tail]), (0, [3, 1, nframes - host_tail - 4]),
                                 (2, [5, nframes - host_tail - 5]), (0, [1] * (nframes - host_tail))):
                got = run(1, group, calls, host_tail)
                assert np.array_equal(got[0], want[0]), (group, calls)
                assert np.array_equal(got[1], want[1]), (group, calls)
                assert (got[2] is None and want[2] is None) or np.array_equal(got[2], want[2])
                assert got[3] == want[3] and got[4] == want[4]
        # one engine option changed between batches reaches the lanes (want: the last host_tail's)
        engine.set_option("strips_async", 0)
        got = run(1, 0, [3, nframes - host_tail - 3], host_tail)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        assert (got[2] is None and want[2] is None) or np.array_equal(got[2], want[2])
        assert got[3] == want[3] and got[4] == want[4]
    finally:
        engine.set_option("strips_async", 1)
        engine.set_option("pipeline", 0)
        engine.set_group(0)
        engine.ring_configure(256)


def ring_behaviour(engine):
    w = synth.CFG1
    n = 2048 * 10
    frames = synth.make_frames(w, 7, n=n)
    engine.ring_configure(4)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, n, w.window, crop="thread")
    assert engine.rows_written == 0
    rows = engine.process(frames)
    assert engine.rows_written == 7
    assert np.array_equal(engine.read_rows(1)[0], rows[6])
    assert np.array_equal(engine.read_rows(4), rows[3:7])          # wraps the 4-row ring
    assert np.array_equal(engine.read_rows(2, age=1), rows[4:6])
    with pytest.raises(ZoomFFTError):
        engine.read_rows(5)
    engine.ring_configure(256)


def decimated_chunk(engine):
    """zoomfft output (S:2100) against the golden mixed+decimated chunk."""
    import os
    z = np.load(os.path.join(parity.GOLDEN_DIR, "zoomfft.npz"))
    for case in gc.ZOOMFFT_CASES:
        x = gc.make_input(case)
        engine.configure(case["fs"], case["N"], case["R"], len(x), "hamming", crop=None)
        engine.process(x)
        y = engine.read_decimated()
        ref = z[case["name"]]
        assert y.shape == ref.shape
        err = np.abs(y - ref).max() / np.abs(ref).max()
        assert err < 2e-5, "%s: relative error %.2e" % (case["name"], err)


def plain_decimate_and_linear(engine):
    """no_lo + linear: the chain is scipy.signal.decimate x log2(R) + welch's
    Pxx itself (the two scipy calls the reference makes, S:2098 / S:2111)."""
    import scipy.signal
    rng = np.random.default_rng(5)
    x = (rng.standard_normal(4096 * 3) + 1j * rng.standard_normal(4096 * 3)).astype(np.complex64)
    engine.configure(1e6, 512, 4, len(x), "hann", crop=None, no_lo=True, linear=True)
    p = engine.process(x)[0].astype(np.float64)
    y = scipy.signal.decimate(scipy.signal.decimate(x.astype(np.complex128), 2), 2)
    _f, want = scipy.signal.welch(y, 1e6, window="hann", nperseg=512, nfft=512)
    want = np.fft.fftshift(want)
    dec = engine.read_decimated()
    assert np.abs(dec - y).max() < 2e-5 * np.abs(y).max()
    rel = np.abs(p - want) / want
    assert rel[want > want.max() * 1e-6].max() < 1e-3


def error_paths(engine):
    with pytest.raises(ValueError):                      # scipy: padlen 27
        engine.configure(2.4e6, 32, 2, 27, "hamming")
    with pytest.raises(ZoomFFTError):
        engine.configure(2.4e6, 1000, 2, 4096, "hamming")        # not a power of two
    with pytest.raises(ZoomFFTError):
        engine.configure(2.4e6, 16, 2, 4096, "hamming")          # too small
    engine.configure(2.4e6, 64, 2, 256, "hamming")
    with pytest.raises(ValueError):
        engine.process(np.zeros(255, dtype=np.complex64))          # wrong frame length
    with pytest.raises(TypeError):
        engine.process(np.zeros(512, dtype=np.uint8))              # wrong wire dtype
    row = engine.process(np.zeros(256, dtype=np.complex64))[0]
    assert np.all(np.isneginf(row))                                # zero power -> -inf like numpy
    # display path arguments
    with pytest.raises(ZoomFFTError):
        engine.ring_image(16, 1, 1, "u8", levels=(-120.0, -120.0))   # empty level range
    with pytest.raises(ValueError):
        engine.ring_image(16, 1, 1, "u8")                            # levels missing
    with pytest.raises(ValueError):
        engine.ring_image(16, 1, 1, "rgba", levels=(-220, -120), lut=np.zeros((255, 4), np.uint8))
    with pytest.raises(ZoomFFTError):
        engine.ring_image(0, 1, 1, "f32")                            # height
    with pytest.raises(ZoomFFTError):
        engine.ring_quantiles(16, 1, 1, [1.5])                       # quantile outside [0, 1]
    with pytest.raises(ZoomFFTError):
        engine.set_option("no_such_knob", 1)
    for name, bad in (("slabs", 3), ("slab_min", 1), ("big_cluster", 3), ("welch_splits", 17), ("slabs", 2),
                      ("strips_async", 2), ("iir_depth", 0), ("strips_priority", 0), ("fir_smem_pad", 0),
                      ("fir_threads", 128)):
        with pytest.raises(ZoomFFTError):
            engine.set_option(name, bad)
    # pipelined batches fall back to the plain path where there are no lanes (mode exact, fft_ratio 2):
    # the batch is ordered on the engine's stream at once and zfb_join has nothing to wait for
    engine.set_option("pipeline", 1)
    try:
        engine.configure(2.4e6, 64, 2, 256, "hamming")
        x = np.ones((3, 256), dtype=np.complex64)
        rows = np.zeros((3, engine.row_width), dtype=np.float32)
        if engine._lib.zfb_build_kind() == b"emulated":              # host memory is device memory there
            engine.process_device(x.ctypes.data, 3, rows.ctypes.data)
            assert engine.slab_lanes == 1
        engine.join()
        engine.join()
        engine.synchronize()
    finally:
        engine.set_option("pipeline", 0)
    # unknown wire format / decimator mode: rejected before anything is planned
    with pytest.raises(ValueError):
        engine.configure(2.4e6, 64, 2, 256, "hamming", dtype="cf64")
    with pytest.raises(ValueError):
        engine.configure(2.4e6, 64, 4, 4096, "hamming", mode="turbo")
    with pytest.raises(ValueError):
        engine.ring_image_device(0, 16, 1, 1, "rgba", lut=np.zeros((16, 4), np.uint8))
    # one-sided rows are the real-input, no-zoom case only
    with pytest.raises(ValueError):
        engine.configure(48e3, 64, 2, 256, "hamming", onesided=True)
    with pytest.raises(ValueError):
        engine.configure(48e3, 64, 1, 256, "hamming", dtype="u8", onesided=True)
    with pytest.raises(ZoomFFTError):
        engine.configure(48e3, 16384, 1, 65536, "hamming", onesided=True)   # beyond the one-CTA FFT
    engine.configure(48e3, 64, 1, 256, "hamming", crop=32, onesided=True)
    assert engine.row_width == 17 and engine.process(np.ones(256, np.float32)).shape == (1, 17)


def f_demod_extension(engine):
    """General software LO (the reference hard-wires 1 Hz, S:2090): tone at
    f_demod + delta must land where the oracle puts it."""
    fs, N, R = 20e6, 1024, 16
    n = N * R * 6
    fc = -7.3e6
    k = np.arange(n)
    x = (0.3 * np.exp(2j * np.pi * ((fc + 2100.0) / fs) * k)).astype(np.complex64)
    rng = np.random.default_rng(3)
    x += (1e-3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
    engine.configure(fs, N, R, n, "hamming", f_demod=fc, crop="thread")
    row = engine.process(x)[0].astype(np.float64)
    want = zo.zoom_psd(x, fs, N, R, "hamming", f_demod=fc, crop="thread")
    parity.assert_row_parity(row, want, parity.floor_db20(fs, "hamming", N, True), "f_demod")


def tile_geometries(engine, names=("cfg1_T", "cfg2_T_f0", "ragged_T", "zoom_R64")):
    """Both decimator region sizes (zfb_set_option decim_threads) meet parity;
    multi-tile frames exercise interior warm-up tiles, true-edge tiles and the
    odd extension in both."""
    try:
        for nt in (256, 128):
            engine.set_option("decim_threads", nt)
            for name in names:
                parity.check_case(engine, name)
    finally:
        engine.set_option("decim_threads", 0)
    with pytest.raises(ZoomFFTError):
        engine.set_option("decim_threads", 64)
    with pytest.raises(ZoomFFTError):
        engine.set_option("no_such_option", 1)


# ---- ZFB_MODE_FAST: polyphase-FIR interior + exact last stage + exact edge strips ----
FAST_CASES = [c["name"] for c in gc.CASES if c["R"] >= 4]


def fast_golden_case(engine, name):
    """Same golden rows, same tolerance, through mode='fast'."""
    err = parity.check_case(engine, name, mode="fast")
    return err, engine.fast_active


def fast_activation(engine):
    """FAST engages for long chunks with R >= 4 and silently stays EXACT otherwise."""
    engine.configure(2.4e6, 2048, 8, 239616, "hamming", mode="fast")
    assert engine.fast_active
    engine.configure(2.4e6, 2048, 2, 65536, "hamming", mode="fast")        # one stage: nothing to replace
    assert not engine.fast_active
    engine.configure(2.4e6, 512, 8, 4096, "hamming", mode="fast")          # strips would cover the chunk
    assert not engine.fast_active
    engine.configure(2.4e6, 2048, 8, 239616, "hamming", mode="exact")
    assert not engine.fast_active


def fast_matches_exact_chunk(engine):
    """The decimated chunk (zoomfft output, S:2100) of FAST agrees with EXACT
    to fp32 resolution over the whole chunk, edges included; odd lengths and
    uint8 + flip covered."""
    rng = np.random.default_rng(99)
    for n, R, dtype, flip in ((100003, 8, "c64", False), (319488, 16, "u8", True), (77777, 4, "c64", True),
                              (262144 + 10, 32, "c64", False)):
        k = np.arange(n)
        x = 0.4 * np.exp(2j * np.pi * 0.0031 / R * k) + 0.2 * np.exp(-2j * np.pi * 0.37 * k)
        x += 0.01 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
        wire = synth.quantise_u8(x) if dtype == "u8" else x.astype(np.complex64)
        out = {}
        for mode in ("exact", "fast"):
            engine.configure(1e6, 256, R, n, "hann", dtype=dtype, flip=flip, crop=None, mode=mode)
            engine.process(wire)
            out[mode] = engine.read_decimated().astype(np.complex128)
            assert engine.fast_active == (mode == "fast")
        err = np.abs(out["fast"] - out["exact"]).max() / np.abs(out["exact"]).max()
        assert err < 1e-5, (n, R, dtype, flip, err)


def fast_batch_and_ema(engine):
    """FAST over a batch == FAST frame by frame (bit-exact), EMA state carried."""
    w = synth.CFG2
    frames = synth.make_frames(w, 3)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", mode="fast")
    assert engine.fast_active
    batch = engine.process(frames)
    single = np.stack([engine.process(frames[i])[0] for i in range(3)])
    assert np.array_equal(batch, single)
    floor = parity.floor_db20(w.fs, w.window, w.fft_size, True)
    for i in range(3):
        parity.assert_row_parity(batch[i], parity.golden_rows()["cfg2_T_f%d" % i], floor, "fast cfg2 %d" % i)
    engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8", flip=True,
                     crop="thread", ema_alpha=0.3, mode="fast")
    engine.reset_ema()
    got = engine.process(frames)
    pw = np.stack([zo.zoom_psd_power(f, w.fs, w.fft_size, w.fft_ratio, w.window, flip=True) for f in frames])
    want = zo.ema_rows_db20(pw, 0.3)
    for i in range(3):
        parity.assert_row_parity(got[i], want[i], floor, "fast ema %d" % i)


def fast_strong_out_of_band(engine):
    """Full-scale interferers outside the returned band (adjacent stations):
    alias rejection and transition-band fidelity of the FIR interior."""
    fs, N, R = 2.4e6, 2048, 16
    n = N * R * 6
    k = np.arange(n)
    rng = np.random.default_rng(7)
    x = 1e-3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for f, a in ((0.23 * fs, 0.25), (-0.49 * fs, 0.25), (fs / R * 0.31, 0.2), (-fs / R * 0.22, 0.2),
                 (1700.0, 0.02)):
        x = x + a * np.exp(2j * np.pi * f / fs * k)
    x = x.astype(np.complex64)
    want = zo.zoom_psd(x, fs, N, R, "hamming", crop=None)
    engine.configure(fs, N, R, n, "hamming", crop=None, mode="fast")
    assert engine.fast_active
    row = engine.process(x)[0].astype(np.float64)
    parity.assert_row_parity(row, want, parity.floor_db20(fs, "hamming", N, True), "fast interferers")


def fast_generic_fir_kernel(engine):
    """The general shared-memory FIR kernel (fallback for tap sets the
    register-blocked kernel is not built for) meets the same parity."""
    try:
        engine.set_option("fir_generic", 1)
        engine._key = None
        for name in ("cfg1_T", "cfg2_T_f0", "zoom_R4", "zoom_R64"):
            parity.check_case(engine, name, mode="fast")
            assert engine.fast_active
    finally:
        engine.set_option("fir_generic", 0)
        engine._key = None


def cs16_wire_format(engine):
    """SoapySDR CS16 (interleaved int16 I,Q, SURVEY 8f.3): (I + jQ) / 32768 on the device.
    Every int16 is exact in fp32, so with the widening pass (option cs16_fused = 0, and wherever
    the fused loader does not apply: mode exact, no zoom, virtual receivers) rows are
    BIT-IDENTICAL to those of the same samples handed over as complex64 -- both decimator
    modes, no zoom, flip, batches, odd lengths, virtual receivers.  By default mode fast
    converts inside the FIR interior's loads (the first stage works on the integer values,
    its taps carry the 1/32768): rows then agree with the complex64 rows to rounding
    (<= 2e-3 dB20) and everything meets parity against the oracle's own conversion."""
    rng = np.random.default_rng(1616)
    cases = ((2.4e6, 2048, 8, 2048 * 8 * 6, "hamming", False, 3), (3.2e6, 1024, 16, 100003, "hann", True, 2),
             (1e6, 512, 1, 512 * 9 + 5, "hamming", False, 2), (2.4e6, 256, 4, 77777, "blackman", True, 1))
    for fs, N, R, n, win, flip, nframes in cases:
        k = np.arange(n)
        x = 0.45 * np.exp(2j * np.pi * 0.011 / R * k) + 0.05 * np.exp(-2j * np.pi * 0.023 / R * k)
        x = x[None, :] + 3e-3 * (rng.standard_normal((nframes, n)) + 1j * rng.standard_normal((nframes, n)))
        wire = np.stack([synth.quantise_cs16(f) for f in x])
        as_c64 = np.stack([zo.cs16_to_iq(f).astype(np.complex64) for f in wire])
        assert np.array_equal(as_c64.astype(np.complex128), np.stack([zo.cs16_to_iq(f) for f in wire]))
        for mode, fused in (("fast", 0), ("fast", 1), ("exact", 1)):
            engine.set_option("cs16_fused", fused)
            engine.configure(fs, N, R, n, win, dtype="cs16", flip=flip, crop="thread", mode=mode)
            converts_on_load = bool(fused) and mode == "fast" and engine.fast_active
            rows = engine.process(wire)
            dec = engine.read_decimated().copy() if R > 1 else None
            single = np.stack([engine.process(wire[i])[0] for i in range(nframes)])
            assert np.array_equal(rows, single), (fs, N, R, mode)
            engine.configure(fs, N, R, n, win, dtype="c64", flip=flip, crop="thread", mode=mode)
            ref_rows = engine.process(as_c64)
            floor = parity.floor_db20(fs, win, engine.geometry["nperseg"], R > 1)
            if not converts_on_load:
                assert np.array_equal(rows, ref_rows), (fs, N, R, mode)
                if R > 1:
                    assert np.array_equal(dec, engine.read_decimated())
            else:
                m = ref_rows > floor
                assert np.abs(rows - ref_rows)[m].max() <= 2e-3, (fs, N, R, mode)
                ref_dec = engine.read_decimated()
                assert np.abs(dec - ref_dec).max() <= 1e-5 * np.abs(ref_dec).max()
            for i in range(nframes):
                want = zo.zoom_psd(wire[i], fs, N, R, win, crop="thread", flip=flip)
                parity.assert_row_parity(rows[i].astype(np.float64), want, floor, "cs16 %s R=%d" % (mode, R))
        engine.set_option("cs16_fused", 1)
    # the fused frame call infers the format from the dtype; virtual receivers over int16 frames
    fs, N, R, n = 2.4e6, 1024, 8, 1024 * 8 * 4
    x = 0.3 * np.exp(2j * np.pi * (250e3 + 900.0) / fs * np.arange(n))
    wire = synth.quantise_cs16(x)
    from pypanadapter_b200.engine import zoom_psd
    got = zoom_psd(wire, fs, N, R, "hamming", f_demod=250e3, engine=engine)
    want = zo.zoom_psd(wire, fs, N, R, "hamming", f_demod=250e3)
    parity.assert_row_parity(got, want, parity.floor_db20(fs, "hamming", N, True), "cs16 zoom_psd")
    centres = np.array([250e3, -1.0e6, 1.0])
    engine.configure(fs, N, R, n, "hamming", dtype="cs16", crop="thread")
    rows = engine.process_channels(np.stack([wire, wire]), centres)
    engine.configure(fs, N, R, n, "hamming", dtype="c64", crop="thread")
    ref = engine.process_channels(np.stack([zo.cs16_to_iq(wire).astype(np.complex64)] * 2), centres)
    assert np.array_equal(rows, ref)
    with pytest.raises(TypeError):
        engine.configure(fs, N, R, n, "hamming", dtype="cs16")
        engine.process(np.zeros(2 * n, dtype=np.uint8))
    with pytest.raises(ValueError):
        zoom_psd(np.zeros(2 * n + 1, dtype=np.int16), fs, N, R, "hamming", engine=engine)


def multi_channel(engine):
    """BASELINE configs[3] in small: virtual receivers with distinct zoom centres
    over the same frames (process_channels) == one configure+process per centre,
    bit for bit, and each meets parity against the oracle."""
    fs, N, R = 20e6, 1024, 16
    n = N * R * 6
    centres = np.array([-9.5e6, -3.1e6, 1.0, 4.44e6, 9.5e6])
    k = np.arange(n)
    rng = np.random.default_rng(21)
    x = 1e-3 * (rng.standard_normal((2, n)) + 1j * rng.standard_normal((2, n)))
    for fc in centres:
        x = x + 0.1 * np.exp(2j * np.pi * ((fc + 7000.0) / fs) * k)
    x = x.astype(np.complex64)
    for mode in ("fast", "exact"):
        engine.configure(fs, N, R, n, "hamming", crop="thread", mode=mode)
        rows = engine.process_channels(x, centres)
        assert rows.shape == (len(centres), 2, engine.row_width)
        floor = parity.floor_db20(fs, "hamming", N, True)
        for c, fc in enumerate(centres):
            engine.configure(fs, N, R, n, "hamming", f_demod=float(fc), crop="thread", mode=mode)
            one = engine.process(x)
            assert np.array_equal(one, rows[c]), (mode, c)
            want = zo.zoom_psd(x[1], fs, N, R, "hamming", f_demod=float(fc), crop="thread")
            parity.assert_row_parity(rows[c, 1], want, floor, "channel %d %s" % (c, mode))
            engine.configure(fs, N, R, n, "hamming", crop="thread", mode=mode)
    engine.configure(fs, N, R, n, "hamming", crop="thread", ema_alpha=0.3)
    with pytest.raises(ZoomFFTError):
        engine.process_channels(x, centres)


def pipeline_channels_equal_plain(engine, dev):
    """Virtual receivers through pipelined batches (each batch, finalisation included, on the next
    lane's stream; zfb_join orders the consumer) == the plain device path, bit for bit; plain
    pipelined batches in between keep their own order."""
    fs, N, R = 20e6, 1024, 16
    n = N * R * 8
    centres = np.array([-9.5e6, -3.1e6, 1.0, 4.44e6, 9.5e6])
    k = np.arange(n)
    rng = np.random.default_rng(22)
    nf = 6
    x = 1e-3 * (rng.standard_normal((nf, n)) + 1j * rng.standard_normal((nf, n)))
    for fc in centres:
        x = x + 0.1 * np.exp(2j * np.pi * ((fc + 7000.0) / fs) * k)
    x = np.ascontiguousarray(x.astype(np.complex64))
    p_in, keep = dev.put(x)
    fbytes = x[0].nbytes

    def run(pipeline):
        engine.set_option("pipeline", pipeline)
        engine.configure(fs, N, R, n, "hamming", crop="thread", mode="fast")
        W = engine.row_width
        outs = []
        for f0, cnt in ((0, 2), (2, 1), (3, 3)):
            p_rows, rows = dev.empty((len(centres), cnt, W))
            engine.process_channels_device(p_in + f0 * fbytes, cnt, centres, p_rows)
            outs.append(rows)
            if f0 == 2:                      # a plain batch between two channel batches
                p_one, one = dev.empty((cnt, W))
                engine.process_device(p_in + f0 * fbytes, cnt, p_one)
                outs.append(one)
        assert engine.slab_lanes == (2 if pipeline else 1)
        engine.join()
        engine.synchronize()
        return [dev.get(o) for o in outs]

    try:
        want = run(0)
        got = run(1)
        for a, b in zip(want, got):
            assert np.array_equal(a, b)
        assert np.isfinite(got[0]).all() and got[0].max() > np.median(got[0]) + 20.0      # the tones stand out
    finally:
        engine.set_option("pipeline", 0)


def pipeline_random_ops(engine, dev, seed=0, nops=40):
    """A seeded random sequence of calls -- device batches (pipelined or not), host batches, virtual
    receivers, ring reads, EMA resets, group and frame-length changes -- gives the same outputs, in the
    same order, with ``pipeline`` = 1 as with 0: every call that is not a pipelined batch joins first."""
    w = synth.CFG2
    lens = (4096 * 16 * 4 + 1234, 4096 * 16 * 5)
    nf = 6
    frames = {n: synth.make_frames(w, nf, n=n) for n in lens}
    dptr = {n: dev.put(frames[n]) for n in lens}
    centres = np.array([-3.1e5, 1.0, 4.44e5])

    def run(pipeline):
        rng = np.random.default_rng(seed)
        engine.set_option("pipeline", pipeline)
        engine.set_group(0)
        state = {"n": lens[0], "ema": 0.3}

        def conf():
            engine.configure(w.fs, w.fft_size, w.fft_ratio, state["n"], w.window, dtype="u8", flip=True,
                             crop="thread", ema_alpha=state["ema"])
        conf()
        engine.ring_configure(4)
        engine.ring_configure(8)                         # a ring of another size starts empty
        assert engine.rows_written == 0
        engine.reset_ema()
        outs, pending = [], []
        for _ in range(nops):
            op = int(rng.integers(0, 9))
            n = state["n"]
            a = int(rng.integers(0, nf - 1))
            cnt = int(rng.integers(1, nf - a + 1))
            if op <= 3:                                  # device batch
                p_rows, rows = dev.empty((cnt, engine.row_width))
                engine.process_device(dptr[n][0] + a * frames[n][0].nbytes, cnt, p_rows)
                pending.append(rows)
            elif op == 4:                                # host batch (joins)
                outs.append(engine.process(frames[n][a:a + cnt]))
            elif op == 5 and engine.rows_written >= 2:   # ring read (joins)
                outs.append(engine.read_rows(2))
            elif op == 6:
                engine.reset_ema()
            elif op == 7:                                # group / frame length / EMA on-off
                engine.set_group(int(rng.choice([0, 2, 3])))
                state["n"] = lens[int(rng.integers(0, 2))]
                state["ema"] = None if rng.random() < 0.4 else 0.3
                conf()
            elif op == 8 and state["ema"] is None:       # virtual receivers on the device
                p_rows, rows = dev.empty((len(centres), cnt, engine.row_width))
                engine.process_channels_device(dptr[n][0] + a * frames[n][0].nbytes, cnt, centres, p_rows)
                pending.append(rows)
        engine.join()
        engine.synchronize()
        outs.extend(dev.get(r) for r in pending)
        outs.append(engine.read_rows(min(8, engine.rows_written)) if engine.rows_written else np.zeros(1))
        return outs

    try:
        want = run(0)
        got = run(1)
        assert len(want) == len(got)
        for i, (a, b) in enumerate(zip(want, got)):
            assert a.shape == b.shape and np.array_equal(a, b), i
    finally:
        engine.set_option("pipeline", 0)
        engine.set_group(0)
        engine.ring_configure(256)


def big_r16_parity(engine, nframes=3):
    """N = 65536 on the radix-16 path (front pass into the scratch buffer, then the one-CTA FFT of
    every block of N/16) against the oracle: a DC offset, sparse (hann) and dense (kaiser)
    FFT(window) tables, complex64; uint8 + flip gives finite rows."""
    fs, N = 2.4e6, 65536
    for window, dtype, nsegs in (("hann", "c64", 7), (("kaiser", 8.6), "c64", 3), ("hamming", "u8", 4)):
        n = N * (nsegs + 1) // 2 + 321
        xs = []
        for i in range(nframes):
            x = gc.tone_noise(n, fs, [(0.11 * fs, 0.3), (-0.23 * fs, 0.02)], 2e-3, 4300 + i, np.complex64)
            xs.append((x + np.complex64(0.2 - 0.1j)).astype(np.complex64) * np.complex64(0.6))
        x = np.stack(xs)
        wire = np.stack([synth.quantise_u8(f) for f in x]) if dtype == "u8" else x
        try:
            engine.set_option("precise", 0)                  # keep few-segment rows on the fp32 path
            engine.configure(fs, N, 1, n, window, dtype=dtype, flip=(dtype == "u8"), crop=None)
            rows = engine.process(wire)
        finally:
            engine.set_option("precise", -1)
        assert rows.shape[0] == nframes and np.all(np.isfinite(rows)), (window, dtype)
        if dtype == "c64":
            want = zo.zoom_psd(x[0], fs, N, 1, window, crop=None)
            parity.assert_row_parity(rows[0].astype(np.float64), want, parity.floor_db20(fs, window, N, False) + 30.0,
                                     "radix-16 %s" % (window,))


def random_configs(engine, seed, count):
    """Seeded sweep over frame length (ragged/odd), N, R, window, wire dtype, flip,
    crop, f_demod and decimator mode against the oracle."""
    rng = np.random.default_rng(seed)
    windows = ["hamming", "hann", "boxcar", "blackmanharris", ("kaiser", 8.6), ("tukey", 0.5), "flattop"]
    for it in range(count):
        N = int(2 ** rng.integers(5, 12))
        R = int(2 ** rng.integers(0, 6))
        segs = int(rng.integers(2, 9))
        n = int(N * R * (segs + 1) // 2 + rng.integers(0, 2 * R + 3))
        if R > 1:
            n = max(n, 28 * R + 5)
        dtype = "u8" if rng.random() < 0.3 else "c64"
        flip = bool(rng.random() < 0.4)
        window = windows[int(rng.integers(len(windows)))]
        crop = [None, "thread", int(2 * rng.integers(1, N // 2 + 1))][int(rng.integers(3))]
        if crop == "thread" and N < 2 * R:
            crop = None                     # the reference's slice would be empty (W = 0): rejected here
        f_demod = 1.0 if rng.random() < 0.5 else float(rng.uniform(-0.5, 0.5) * 1e6)
        mode = "fast" if rng.random() < 0.6 else "exact"
        fs = 1e6
        k = np.arange(n)
        ftone = f_demod + rng.uniform(-0.3, 0.3) * fs / R / max(1, R if crop == "thread" else 1)
        x = 0.45 * np.exp(2j * np.pi * ftone / fs * k) + 0.2 * np.exp(2j * np.pi * rng.uniform(-0.5, 0.5) * k)
        x = x + 5e-3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
        wire = synth.quantise_u8(x * 0.9) if dtype == "u8" else x.astype(np.complex64)
        what = "case %d: N=%d R=%d n=%d %s flip=%s win=%s crop=%s f=%g %s" % (
            it, N, R, n, dtype, flip, window, crop, f_demod, mode)
        engine.configure(fs, N, R, n, window, dtype=dtype, flip=flip, f_demod=f_demod, crop=crop, mode=mode)
        row = engine.process(wire)[0].astype(np.float64)
        want = zo.zoom_psd(wire, fs, N, R, window, f_demod=f_demod, crop=crop, flip=flip)
        floor = parity.floor_db20(fs, window, engine.geometry["nperseg"], R > 1)
        # strict floor: rows of few segments take the engine's fp64 path (zfb_precise.cuh)
        parity.assert_row_parity(row, want, floor, what)


def reconfigure_stress(engine, rounds=4):
    """The reference lets N, R, window and frame length change between any two
    frames (S:1753-1757, S:2079-2086): cycling through very different plans on
    ONE engine must reproduce each plan's first-run rows bit for bit (no stale
    workspace, LO table, FIR plan or EMA state leaks between configurations)."""
    rng = np.random.default_rng(5)
    plans = [
        dict(fs=2.4e6, N=2048, R=8, n=2048 * 20, window="hamming", dtype="c64", mode="fast", crop="thread"),
        dict(fs=3.2e6, N=4096, R=16, n=4096 * 20, window="hann", dtype="u8", flip=True, mode="fast", crop="thread"),
        dict(fs=1e6, N=256, R=1, n=256 * 9 + 17, window=("kaiser", 9.0), dtype="c64", mode="exact", crop=None),
        dict(fs=2.4e6, N=1024, R=4, n=1024 * 12 + 1, window="hamming", dtype="c64", mode="exact", crop=512),
        dict(fs=2.4e6, N=16384, R=2, n=16384 * 6, window="hann", dtype="c64", mode="fast", crop="thread"),
        dict(fs=20e6, N=512, R=32, n=512 * 32 * 12, window="blackmanharris", dtype="c64", mode="fast",
             crop="thread", f_demod=-3.3e6),
        dict(fs=2.4e6, N=2048, R=8, n=2048 * 20, window="hamming", dtype="c64", mode="fast", crop="thread",
             ema_alpha=0.5),
    ]
    data, first = [], []
    for p in plans:
        n = p["n"]
        x = 0.3 * np.exp(2j * np.pi * rng.uniform(-0.02, 0.02) * np.arange(n)) \
            + 1e-2 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
        data.append(synth.quantise_u8(x) if p["dtype"] == "u8" else x.astype(np.complex64))

    def run(i):
        p = plans[i]
        engine.configure(p["fs"], p["N"], p["R"], p["n"], p["window"], dtype=p["dtype"],
                         flip=p.get("flip", False), f_demod=p.get("f_demod", 1.0), crop=p["crop"],
                         ema_alpha=p.get("ema_alpha"), mode=p["mode"])
        if p.get("ema_alpha") is not None:
            engine.reset_ema()
        return engine.process(np.stack([data[i], data[i]]))

    for i in range(len(plans)):
        first.append(run(i))
        assert np.all(np.isfinite(first[i]))
    order = list(range(len(plans)))
    for _ in range(rounds):
        rng.shuffle(order)
        for i in order:
            assert np.array_equal(run(i), first[i]), "plan %d changed after reconfiguration" % i
