"""Run the reference's OWN hot-path lines -- TEST INFRASTRUCTURE ONLY.

The reference is a PyQt5 GUI program; PyQt5, pyqtgraph, rtlsdr, SoapySDR and
pyaudio are not installed and there is no network, so it cannot run as a
program.  Its hot path, however, is plain numpy/scipy inside Qt class methods.
This module puts stub ``PyQt5`` / ``pyqtgraph`` modules into ``sys.modules``,
exec-loads the UNMODIFIED ``/root/reference/pypanadapter_spectrum.py`` and
``pypanadapter_thread.py`` and calls those methods on light fake ``self``
objects:

* ``ApplicationDisplay.update`` / ``.zoomfft``   (S:2088-2130)
* ``PSD.update``                                  (T:1513-1549)
* ``Data.new_complex/add/get_data_start/get_data_end`` (T:1400-1483)
* ``Waterfall.init_image/image_update``           (S:1625-1664)

It only works where the reference's source tree is present
(``PYPAN_REFERENCE_DIR``); ``oracle/make_golden.py`` uses it to record
``tests/golden/*.npz``, which the tests compare against.
No reference source is copied: the files are read where they lie.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import numpy as np

REFERENCE_DIR = os.environ.get("PYPAN_REFERENCE_DIR", "/root/reference")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "pypanadapter_thread.py"))


# ------------------------------------------------------------------ stubs
class _Anything:
    """Subclassable, callable, attribute-tolerant stand-in for any Qt class."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()


class _Signal:
    def __init__(self, *a, **k):
        self._slots = []

    def connect(self, fn):
        self._slots.append(fn)

    def emit(self, *a):
        for fn in self._slots:
            fn(*a)


class _Mutex:
    def lock(self):
        pass

    def unlock(self):
        pass


def _identity_decorator(*_a, **_k):
    def deco(fn):
        return fn
    return deco


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        cls = type(name, (_Anything,), {})
        setattr(self, name, cls)
        return cls


def _install_stubs():
    if "PyQt5" in sys.modules and not isinstance(sys.modules["PyQt5"], _StubModule):
        return                                       # a real PyQt5: leave it
    qt = _StubModule("PyQt5")
    qt.__path__ = []
    for sub in ("QtCore", "QtWidgets", "QtGui", "QtDBus"):
        m = _StubModule("PyQt5." + sub)
        setattr(qt, sub, m)
        sys.modules["PyQt5." + sub] = m
    qt.QtCore.pyqtSignal = _Signal
    qt.QtCore.Signal = _Signal
    qt.QtCore.pyqtSlot = _identity_decorator
    qt.QtCore.Slot = _identity_decorator
    qt.QtCore.QMutex = _Mutex
    sys.modules["PyQt5"] = qt
    pg = _StubModule("pyqtgraph")
    sys.modules.setdefault("pyqtgraph", pg)


_loaded = {}


def load(which: str):
    """which = 'spectrum' | 'thread' -> the exec-loaded reference module."""
    if which in _loaded:
        return _loaded[which]
    if not available():
        raise RuntimeError("reference tree not present at " + REFERENCE_DIR)
    _install_stubs()
    if REFERENCE_DIR not in sys.path:
        sys.path.insert(0, REFERENCE_DIR)            # for `import newtrap`
    path = os.path.join(REFERENCE_DIR, "pypanadapter_%s.py" % which)
    spec = importlib.util.spec_from_file_location("_ref_pypan_" + which, path)
    mod = importlib.util.module_from_spec(spec)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):  # "Could not find ..." prints
        spec.loader.exec_module(mod)
    _loaded[which] = mod
    return mod


class _FakePan:
    def __init__(self, fs):
        self.SampleRate = fs
        self.driver = object()


def _set_state(mod, fs, fft_size, fft_ratio, fft_avg, window):
    st = mod.AppState
    st._panadapter = _FakePan(fs)
    st.fft_size = fft_size
    st.fft_ratio = fft_ratio
    st.fft_avg = fft_avg
    st.fft_tapering = window
    return st


# ------------------------------------------------------ S: update / zoomfft
def spectrum_update(chunk, fs, fft_size, fft_ratio, window, n_win):
    """ApplicationDisplay.update(fake_self, chunk) (S:2102-2130) -> the psd
    row handed to Waterfall.image_update (before its in-place grid zeros)."""
    mod = load("spectrum")
    n = len(chunk)
    if n % fft_size:
        raise ValueError("S: path reads avg*N samples (S:1764)")
    _set_state(mod, fs, fft_size, fft_ratio, n // fft_size, window)
    got = {}

    class _WF:
        def image_update(self, psd):
            got["psd"] = np.array(psd, copy=True)

    fake = types.SimpleNamespace()
    fake.N_WIN = n_win
    fake.win = _Anything()
    fake.waterfall = _WF()
    fake.spectrum_plot = _Anything()
    fake.zoomfft = types.MethodType(mod.ApplicationDisplay.zoomfft, fake)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mod.ApplicationDisplay.update(fake, chunk)
    return got["psd"]


def spectrum_zoomfft(chunk, fs, fft_size, fft_ratio):
    """ApplicationDisplay.zoomfft (S:2088-2100): mixed + decimated chunk."""
    mod = load("spectrum")
    n = len(chunk)
    _set_state(mod, fs, fft_size, fft_ratio, n // fft_size, "hamming")
    fake = types.SimpleNamespace()
    return mod.ApplicationDisplay.zoomfft(fake, chunk, fft_ratio)


# ------------------------------------------------------------ T: PSD.update
def _quiet_data(mod, chunk_size=None):
    d = mod.Data() if chunk_size is None else mod.Data(chunk_size)
    d.NR = types.SimpleNamespace(next=lambda y: 0.0, target=0)
    return d


def thread_update(chunk, fs, fft_size, fft_ratio, window, real=False):
    """Data.add(chunk) + PSD.update() (T:1433-1468, T:1513-1549) -> psd row.
    The chunk must fit the fold-back buffer (max_size = 16*chunk_size).
    ``real``: allocate with Data.new_real (T:1413-1417) instead of the
    new_complex the reference's own set-up calls (T:1807)."""
    import contextlib
    import io
    import warnings
    mod = load("thread")
    _set_state(mod, fs, fft_size, fft_ratio, 1, window)
    d = _quiet_data(mod, max(8196 * 2, -(-len(chunk) // 16)))
    if real:
        d.new_real()
    else:
        d.new_complex()
    d.delay_time = 0.
    d.add(chunk)
    d.delay_time = 0.
    psd = types.SimpleNamespace()
    psd.dataclass = d
    psd.lock = _Mutex()
    psd.psd = None
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mod.PSD.update(psd)
    return psd.psd


def thread_data_trace(chunks, chunk_size=8196 * 2):
    """Feed chunks through the reference's Data.add; return the list of
    (size, real_size, total_size) after each add and the final data[:real_size]."""
    mod = load("thread")
    d = _quiet_data(mod, chunk_size)
    d.new_complex()
    trace = []
    for c in chunks:
        d.delay_time = 0.
        d.add(c)
        trace.append((d.size, d.real_size, d.total_size))
    return np.array(trace), np.array(d.data[:d.real_size], copy=True), d.max_size


# --------------------------------------------------------------- Waterfall
def waterfall_rows(rows, scroll=1):
    """Waterfall.image_update for each row (S:1638-1664); returns img_array."""
    mod = load("spectrum")
    mod.AppState.scroll = scroll
    _set_state(mod, 2.4e6, 2048, 8, 1, "hamming")
    wf = mod.Waterfall.__new__(mod.Waterfall)
    wf.fftwidth = 0
    wf.scale = lambda *a, **k: None
    wf.setImage = lambda *a, **k: None
    for r in rows:
        wf.image_update(np.array(r, dtype=np.float64, copy=True))
    return np.array(wf.img_array, copy=True)


def waterfall_autolevel(rows, scroll=1):
    """The reference's own Waterfall.autolevel (S:1668-1680) after image_update
    for each row: returns (minlevel, maxlevel) -- the attributes its
    np.percentile(img_array[img_array<0], [2, 98]) lands in (S:1676) -- and the
    (minlev, maxlev) pair it returns (unchanged defaults: the attribute-name
    slip at S:1676-1677)."""
    mod = load("spectrum")
    mod.AppState.scroll = scroll
    _set_state(mod, 2.4e6, 2048, 8, 1, "hamming")
    wf = mod.Waterfall.__new__(mod.Waterfall)
    wf.fftwidth = 0
    wf.minlev = -220                      # S:1592-1593 (set in __init__, which needs Qt)
    wf.maxlev = -120
    wf.scale = lambda *a, **k: None
    wf.setImage = lambda *a, **k: None
    wf.setLevels = lambda *a, **k: None
    for r in rows:
        wf.image_update(np.array(r, dtype=np.float64, copy=True))
    ret = wf.autolevel()
    return np.array([wf.minlevel, wf.maxlevel]), np.array(ret, dtype=np.float64)

