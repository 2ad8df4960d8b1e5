"""The oracle against (i) the golden vectors recorded from the reference's own
methods, (ii) its own explicit restatement and (iii) closed forms."""
import json
import os

import numpy as np
import pytest
import scipy

from oracle import golden_cases as gc
from oracle import make_golden as mg
from oracle import zoompsd_oracle as zo
from tests import parity

GOLD = parity.GOLDEN_DIR
ALL = [c["name"] for c in gc.CASES]
FAST = [n for n in ALL if n not in ("n65536_R1_T",)]


def _manifest():
    with open(os.path.join(GOLD, "MANIFEST.json")) as f:
        return json.load(f)


def test_manifest_lists_every_case():
    m = _manifest()
    assert m["cases"] == [c["name"] for c in gc.CASES + gc.ZOOMFFT_CASES]
    assert set(parity.golden_rows()) == set(ALL)


def _tight(a, b):
    """fp64 agreement in dB20: exact for the same library versions, loose
    enough to survive a different BLAS/pocketfft build."""
    m = np.isfinite(a) & np.isfinite(b)
    assert np.array_equal(np.isneginf(a), np.isneginf(b))
    # bins near the fp64 noise floor (< -550 dB20) are rounding noise
    big = m & (b > -550)
    return float(np.abs(a[big] - b[big]).max()) if big.any() else 0.0


@pytest.mark.parametrize("name", ALL)
def test_oracle_matches_reference_golden(name):
    """The rows the reference's own methods computed (oracle/make_golden.py's reference_row)."""
    same_versions = (_manifest()["numpy"] == np.__version__
                     and _manifest()["scipy"] == scipy.__version__)
    row = parity.oracle_row(gc.case_by_name(name))
    ref = parity.golden_rows()[name]
    assert row.shape == ref.shape
    assert _tight(row, ref) <= (1e-10 if same_versions else 1e-6)


@pytest.mark.parametrize("name", ["cfg1_T", "zoom_R16", "ragged_odd_T", "short_T", "win_kaiser",
                                  "r1_hann_T", "cfg2_T_f0", "n32_T"])
def test_explicit_restatement_matches(name):
    case = gc.case_by_name(name)
    x = gc.make_input(case)
    crop, _ = parity.case_config(case)
    a = zo.zoom_psd(x, case["fs"], case["N"], case["R"], case["window"], crop=crop,
                    flip=bool(case.get("flip")), explicit=True)
    assert _tight(a, parity.golden_rows()[name]) <= 1e-7


def test_zoomfft_golden():
    z = np.load(os.path.join(GOLD, "zoomfft.npz"))
    for case in gc.ZOOMFFT_CASES:
        x = gc.make_input(case)
        for explicit in (False, True):
            y = zo.zoom_mix_decimate(x, case["fs"], case["R"], explicit=explicit)
            ref = z[case["name"]]
            assert y.shape == ref.shape
            assert np.abs(y - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())


def test_decimate_rejects_short_input():
    with pytest.raises(ValueError):
        zo.decimate2_explicit(np.ones(27, dtype=complex))
    with pytest.raises(ValueError):
        zo.decimate2_ref(np.ones(27, dtype=complex))
    assert len(zo.decimate2_explicit(np.ones(28, dtype=complex))) == 14


def test_sos_zi_matches_scipy():
    sos = zo.decim_sos()
    assert np.allclose(zo.sos_zi(sos), scipy.signal.sosfilt_zi(sos), rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("zoomed,R", [(False, 1), (True, 4)])
def test_bin_centred_tone_closed_form(zoomed, R):
    fs, N, A = 2.4e6, 1024, 0.37
    n = N * 8 * R
    kbin = 37
    f = kbin * fs / R / N + (1.0 if zoomed else 0.0)      # the LO shifts by f_demod = 1 Hz
    x = A * np.exp(2j * np.pi * f / fs * np.arange(n))
    row = zo.zoom_psd(x, fs, N, R, "hamming", crop=None)
    want = zo.tone_peak_db20(A, fs, "hamming", N, zoomed)
    assert int(np.argmax(row)) == N // 2 + kbin
    # zoomed: each zero-phase stage adds up to 2 x 0.05 dB passband ripple = 0.2 dB20
    assert abs(row.max() - want) < (0.2 * np.log2(R) + 1e-3 if zoomed else 1e-9)


def test_u8_conversion_and_flip():
    raw = np.array([0, 255, 127, 128, 1, 2], dtype=np.uint8)
    iq = zo.rtlsdr_bytes_to_iq(raw)
    assert np.allclose(iq, [(-1 + 1j), (127 / 127.5 - 1) + (128 / 127.5 - 1) * 1j,
                            (1 / 127.5 - 1) + (2 / 127.5 - 1) * 1j])
    assert np.array_equal(zo.flip_chunk(iq), iq[::-1])
    with pytest.raises(ValueError):
        zo.rtlsdr_bytes_to_iq(raw[:5])


def test_cs16_conversion():
    """SoapySDR CS16 -> complex: (I + jQ) / 32768, exact in fp32 (the device path
    relies on that for bit-identical rows)."""
    raw = np.array([-32768, 32767, 0, 16384, -1, 1], dtype=np.int16)
    iq = zo.cs16_to_iq(raw)
    assert np.array_equal(iq, [-1 + (32767 / 32768) * 1j, 0.5j, (-1 + 1j) / 32768])
    assert np.array_equal(iq.astype(np.complex64).astype(np.complex128), iq)
    every = np.arange(-32768, 32768, dtype=np.int64).astype(np.int16)
    assert np.array_equal((every.astype(np.float32) * np.float32(1 / 32768)).astype(np.float64), every / 32768.0)
    with pytest.raises(ValueError):
        zo.cs16_to_iq(raw[:5])
    from pypanadapter_b200 import synth
    x = np.array([0.5 - 0.25j, 1.0 + 1.0j, -1.0 - 1.0j])
    assert np.array_equal(synth.quantise_cs16(x), [16384, -8192, 32767, 32767, -32768, -32768])


def test_ema_definition():
    p = np.array([[1.0, 4.0], [3.0, 0.0], [1.0, 1.0]])
    out = zo.ema_rows_db20(p, 0.3)
    a1 = 0.3 * p[1] + 0.7 * p[0]
    a2 = 0.3 * p[2] + 0.7 * a1
    assert np.allclose(out[0], 20 * np.log10(p[0]))
    assert np.allclose(out[1], 20 * np.log10(a1))
    assert np.allclose(out[2], 20 * np.log10(a2))


def test_data_foldback_golden():
    g = np.load(os.path.join(GOLD, "data_trace.npz"))
    d = zo.DataOracle().new_complex()
    assert d.max_size == int(g["max_size"])
    trace = []
    for chunk in mg.data_trace_chunks():
        if len(chunk) > d.max_size:
            with pytest.raises(ValueError):
                d.add(chunk)
            trace.append((d.size, d.real_size, d.total_size))
            continue
        d.add(chunk)
        trace.append((d.size, d.real_size, d.total_size))
    assert np.array_equal(np.array(trace), g["trace"])
    assert np.array_equal(d.take(), g["tail"])


def test_waterfall_golden():
    g = np.load(os.path.join(GOLD, "waterfall.npz"))
    rows = [np.full(256, -100.0 - i) + np.arange(256) * 0.01 for i in range(70)]
    for scroll, key in ((1, "img_pos"), (-1, "img_neg")):
        img = None
        for r in rows:
            img = zo.waterfall_update(img, r.copy(), scroll)
        assert np.array_equal(img, g[key])


def test_waterfall_autolevel_golden():
    """oracle autolevel == the reference's own Waterfall.autolevel (recorded by
    make_golden under Qt stubs), which also pins its minlevel/minlev slip."""
    g = np.load(os.path.join(GOLD, "waterfall.npz"))
    for name, rows in (("ramp", gc.waterfall_rows_ramp()), ("noise", gc.waterfall_rows_noise())):
        for scroll, tag in ((1, "pos"), (-1, "neg")):
            img = None
            for r in rows:
                img = zo.waterfall_update(img, r.copy(), scroll)
            lo, hi = zo.waterfall_autolevel(img)
            want = g["auto_%s_%s" % (name, tag)]
            assert lo == want[0] and hi == want[1], (name, tag, lo, hi, want)
            assert list(g["autoret_%s_%s" % (name, tag)]) == [-220.0, -120.0]
    img = None
    for r in gc.waterfall_rows_noise():
        img = zo.waterfall_update(img, r.copy(), 1)
    assert np.array_equal(img, g["img_noise_pos"])


def test_waterfall_indices_properties():
    """level mapping restatement: monotone, clipped, -500 fill and -inf -> 0,
    grid zeros -> 255, bin edges at minlev + k (max - min)/256."""
    v = np.array([-np.inf, -500.0, -220.0, -219.7, -170.0, -120.4, -120.0, 0.0])
    idx = zo.waterfall_indices(v, -220, -120)
    assert list(idx) == [0, 0, 0, 0, 128, 254, 255, 255]
    lut = zo.colormap_lut([0., 1.], [[0, 0, 0, 255], [0, 255, 0, 255]])      # 'Matrix' (S:1582)
    assert lut.shape == (256, 4) and list(lut[0]) == [0, 0, 0, 255] and list(lut[255]) == [0, 255, 0, 255]
    assert np.all(np.diff(lut[:, 1].astype(int)) >= 0)

