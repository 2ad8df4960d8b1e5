"""The large-FFT Welch paths against the oracle, shared by tests/test_bigfft.py on the CPU
emulation build and, marked gpu, on the B200:

* four-step path, N = 16384, 32768 and 262144 (zfb_bigfft.cuh: big_dc_kernel, bigfft_col_kernel,
  bigfft_mean_kernel, bigfft_row_kernel);
* radix-16 path, N = 65536 and 131072 (big_dc_kernel, big_r16_kernel, big_mean16_kernel, welch_kernel
  with prepared = 1, big_gather_kernel).

Both apply scipy's detrend='constant' after the FFT, X -= (m - dc) FFT(w), with a per-frame DC
estimate dc removed before the window.  That cancellation only matters when the segment mean is
large, so most scenarios here carry a DC offset, up to near full scale.  Every frame of a batch is
held to the oracle at the strict floor (parity.floor_db20, no margin) with an exact argmax.

complex64 samples reach the oracle widened to complex128 (the same values): scipy.signal.welch
computes in its input's precision, and in complex64 its own rounding at the DC column of such a
chunk reaches the 0.01 dB20 bar.  uint8 and CS16 samples the oracle converts in float64 itself."""
from __future__ import annotations

import numpy as np

from oracle import golden_cases as gc
from oracle import zoompsd_oracle as zo
from pypanadapter_b200 import synth
from tests import parity

FS = 2.4e6
FOUR_STEP = (16384, 32768, 262144)
RADIX16 = (65536, 131072)
LARGE = FOUR_STEP + RADIX16
WIRES = ("c64", "u8", "u8flip", "cs16")
WINDOWS = ("hann", "hamming", ("kaiser", 8.6), "bartlett")   # kaiser, bartlett: dense FFT(window) tables
DCS = (0.0, 0.4, 0.9 - 0.7j)        # added before the 0.6 scale: 0, 0.24 and 0.54-0.42j on the wire


def frame_len(N, R, nseg):
    """a chunk of nseg Welch segments with a short ragged tail"""
    return N * R * (nseg + 1) // 2 + 3 * R + 5


def make_frame(N, R, n, dc, seed=0, f_demod=1.0, span=1.0):
    """tone + noise, plus a DC offset, all times 0.6 (complex64).  Seed 0 gives the chunk of the
    pinned cases; the tones sit at 0.11 and -0.23 of the row's span (FS / R times the kept fraction
    of the spectrum) from the zoom centre."""
    f0 = f_demod if R > 1 else 0.0
    band = FS / R * span
    x = gc.tone_noise(n, FS, [(f0 + 0.11 * band, 0.3), (f0 - 0.23 * band, 0.02)], 2e-3, 4242 + N + 7919 * seed,
                      np.complex64)
    return (x + np.complex64(dc)).astype(np.complex64) * np.complex64(0.6)


def to_wire(x, wire):
    if wire == "c64":
        return x
    return synth.quantise_cs16(x) if wire == "cs16" else synth.quantise_u8(x)


def oracle_row(wire_frame, N, R, window, crop, flip, f_demod=1.0):
    x = wire_frame.astype(np.complex128) if np.iscomplexobj(wire_frame) else wire_frame
    return zo.zoom_psd(x, FS, N, R, window, f_demod=f_demod, crop=crop, flip=flip)


def run(engine, frames, N, R, window, wire, crop=None, f_demod=1.0, precise=-1):
    """rows of a batch of wire-format frames; ``precise`` = 0 keeps rows of few segments off the
    fp64 path (zfb_precise.cuh), which is not what these tests are about"""
    try:
        engine.set_option("precise", precise)
        engine.configure(FS, N, R, frames.shape[1] // (1 if wire == "c64" else 2), window,
                         dtype={"u8flip": "u8"}.get(wire, wire), flip=(wire == "u8flip"), crop=crop,
                         f_demod=f_demod)
        return engine.process(frames).astype(np.float64)
    finally:
        engine.set_option("precise", -1)


def check_rows(engine, rows, frames, N, R, window, wire, crop=None, f_demod=1.0, what=""):
    """every row against the oracle; returns the largest |diff| in dB20"""
    floor = parity.floor_db20(FS, window, engine.geometry["nperseg"], R > 1)
    err = 0.0
    assert rows.shape[0] == len(frames), what
    for i, f in enumerate(frames):
        want = oracle_row(f, N, R, window, crop, wire == "u8flip", f_demod)
        err = max(err, parity.assert_row_parity(rows[i], want, floor, "%s frame %d" % (what, i)))
    return err


def check(engine, N, R, n, window, wire, dcs, crop=None, f_demod=1.0, precise=-1, seed0=0, span=1.0, what=""):
    """one batch, one frame per DC offset in ``dcs``, through the engine and the oracle"""
    frames = np.stack([to_wire(make_frame(N, R, n, dc, seed0 + i, f_demod, span), wire) for i, dc in enumerate(dcs)])
    rows = run(engine, frames, N, R, window, wire, crop, f_demod, precise)
    what = what or "N=%d R=%d n=%d %s %s crop=%s" % (N, R, n, wire, window, crop)
    return check_rows(engine, rows, frames, N, R, window, wire, crop, f_demod, what), rows, frames


# ---- the rows of the DC-offset table: 7 segments (the fp32 path), R = 1, all N bins ---------------
PINNED = {
    "n32768_u8_dc_hamming": (32768, "u8", 0.9 - 0.7j, "hamming", 0),
    "n32768_u8flip_dc_hann": (32768, "u8flip", 0.9 - 0.7j, "hann", 0),
    "n32768_c64_dc_hamming": (32768, "c64", 0.9 - 0.7j, "hamming", 0),
    "n32768_c64_dc04_hamming": (32768, "c64", 0.4, "hamming", 0),
    "n16384_u8_dc_hamming": (16384, "u8", 0.9 - 0.7j, "hamming", 0),
    "n262144_u8_dc_hamming": (262144, "u8", 0.9 - 0.7j, "hamming", 0),
    "n65536_u8_dc_hamming": (65536, "u8", 0.9 - 0.7j, "hamming", 0),
    "n131072_u8_dc_hamming": (131072, "u8", 0.9 - 0.7j, "hamming", 0),
    "n32768_u8_dc_hamming_fp64": (32768, "u8", 0.9 - 0.7j, "hamming", 1),
}


def pinned_case(engine, name):
    N, wire, dc, window, precise = PINNED[name]
    return check(engine, N, 1, frame_len(N, 1, 7), window, wire, [dc], precise=precise, what=name)[0]


# ---- scenarios ------------------------------------------------------------------------------------
def dc_offsets(engine, N):
    """wire format x DC offset, the windows taken in turn so that each meets every offset;
    two frames of distinct noise per batch"""
    n = frame_len(N, 1, 7)
    worst = 0.0
    for i, wire in enumerate(WIRES):
        for j, dc in enumerate(DCS):
            window = WINDOWS[(i + j) % len(WINDOWS)]
            worst = max(worst, check(engine, N, 1, n, window, wire, [dc, dc], seed0=10 * j)[0])
    return worst


PER_FRAME_DC = (0.9 - 0.7j, 0.0, -0.5 + 0.3j, 0.4, 0.15j)


def per_frame_dc(engine, N):
    """a different DC offset in every frame of a batch (per-frame indexing of dc, means and partial),
    in one launch group and across groups of two; each frame meets parity and the batched rows are
    the single-frame rows bit for bit"""
    n = frame_len(N, 1, 7)
    for wire, window in (("c64", ("kaiser", 8.6)), ("u8flip", "hamming")):
        _, rows, frames = check(engine, N, 1, n, window, wire, PER_FRAME_DC, seed0=3)
        single = np.concatenate([run(engine, frames[i:i + 1], N, 1, window, wire) for i in range(len(frames))])
        assert np.array_equal(rows, single), (N, wire)
        try:
            engine.set_group(2)
            grouped = run(engine, frames, N, 1, window, wire)
        finally:
            engine.set_group(0)
        assert np.array_equal(rows, grouped), (N, wire)


def crop_and_zoom(engine, N, ratios=(2, 4, 8)):
    """R > 1 with crop='thread' and an integer crop (W < N: big_gather_kernel's crop on the radix-16
    path, the row pass's on the four-step path), then an odd frame length whose decimated tail is a
    hop short of one more segment, with flip (the last segment must not read past the chunk)"""
    nseg = 3
    for R in ratios:
        n = frame_len(N, R, nseg)
        for k, crop in enumerate(("thread", N // 3 + 1)):
            W = zo.crop_width(N, R, crop)
            wire = ("c64", "u8", "cs16")[(R + k) % 3]
            check(engine, N, R, n, "hann" if k else "hamming", wire, [0.9 - 0.7j, 0.4], crop=crop, precise=0,
                  span=W / N)
    hop = N // 2
    for R, wire in ((1, "u8flip"), (2, "u8flip"), (2, "c64")):
        n = R * ((nseg + 2) * hop - 1) - R + 1
        assert n % 2 == 1 and engine.configure(FS, N, R, n, "hamming").geometry["nseg"] == nseg
        check(engine, N, R, n, ("kaiser", 8.6), wire, [0.9 - 0.7j, -0.3 + 0.2j, 0.0], crop=N // 2 - 6, precise=0,
              span=0.5)


def fp64_fp32_boundary(engine, N):
    """6 segments take the fp64 path (zfb_precise.cuh) by default, 7 the fp32 path; both hold parity,
    and each equals its path forced by the option ``precise``"""
    for nseg, forced in ((6, 1), (7, 0)):
        n = frame_len(N, 1, nseg)
        for wire, window in (("u8", "hamming"), ("c64", "bartlett")):
            _, rows, frames = check(engine, N, 1, n, window, wire, [0.9 - 0.7j, 0.4])
            assert engine.geometry["nseg"] == nseg
            assert np.array_equal(rows, run(engine, frames, N, 1, window, wire, precise=forced)), (N, nseg, wire)


def keep_crop(N, cls):
    """an integer crop whose row keeps ``cls`` = 1, 2, 4 or 16 (all) bins per spectrum end of each
    welch_kernel thread (welch_keep: 16 points per thread from N = 2048, N/16 threads)"""
    nt = N // 16
    lo, hi = {1: (1, nt), 2: (nt + 1, 2 * nt), 4: (2 * nt + 1, 4 * nt), 16: (4 * nt + 1, N // 2)}[cls]
    return 2 * int((lo + hi) // 2)


def random_large(engine, seed, count):
    """seeded sweep for N >= 4096: N, R, segments, crop, window, wire format, DC offset and f_demod.
    Rows of N = 4096 and 8192 with R > 1 take the integer crops that reach every welch_keep variant
    in turn."""
    rng = np.random.default_rng(seed)
    windows = ["hamming", "hann", "boxcar", "blackmanharris", ("kaiser", 8.6), ("tukey", 0.5), "bartlett"]
    keeps = [1, 2, 4, 16]
    for it in range(count):
        N = int(2 ** rng.integers(12, 19))
        R = int(2 ** rng.integers(0, 5))
        segs = int(rng.integers(1, 13))
        if N <= 8192 and R > 1:
            segs = max(segs, 7)                                      # welch_kernel, not the fp64 path
        while segs > 1 and N * R * (segs + 1) // 2 > (3 << 20):      # bounded chunk: the oracle's time
            segs -= 1
        n = N * R * (segs + 1) // 2 + int(rng.integers(0, 2 * R + 3))
        if N <= 8192 and R > 1:
            crop = keep_crop(N, keeps[(seed + it) % 4])
        else:
            crop = [None, "thread", 2 * int(rng.integers(1, N // 2 + 1))][int(rng.integers(3))]
        W = zo.crop_width(N, R, crop)
        wire = WIRES[int(rng.integers(len(WIRES)))]
        window = windows[int(rng.integers(len(windows)))]
        dc = [0.0, 0.4, 0.9 - 0.7j, complex(*rng.uniform(-0.7, 0.7, 2))][int(rng.integers(4))]
        f_demod = 1.0 if rng.random() < 0.5 else float(rng.uniform(-0.4, 0.4) * FS)
        what = "case %d: N=%d R=%d segs=%d n=%d %s %s crop=%s dc=%s f=%g" % (
            it, N, R, segs, n, wire, window, crop, dc, f_demod)
        check(engine, N, R, n, window, wire, [dc], crop=crop, f_demod=f_demod, seed0=100 * seed + it,
              span=W / N, what=what)
