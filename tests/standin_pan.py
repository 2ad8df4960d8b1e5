"""TEST INFRASTRUCTURE: minimal stand-ins for the two reference programs.

The reference programs are not part of this repository, so `dropin.install` is
exercised on stand-ins.  `make("spectrum")` / `make("thread")` build
modules with the SAME class, method and attribute names the drop-in touches --
`AppState`, `ApplicationDisplay.zoomfft/update`, `PSD`, `Data`, `Waterfall`
(pypanadapter_spectrum.py:1577-1686, 2088-2130; pypanadapter_thread.py:1400-1549,
2140-2157) -- whose hot-path bodies are deliberately EMPTY (they raise): every
row a test sees after `install` was computed by the product library.  The few
methods the drop-in leaves alone (the threaded GUI timer's `update`, `PSD.__init__`)
carry the reference's call sequence in a few lines of our own.
"""
from __future__ import annotations

import types

import numpy as np


class _Recorder:
    """Qt widget stand-in: swallows any call, remembers the last one per name."""

    def __init__(self):
        self.calls = {}

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def fn(*a, **k):
            self.calls[name] = (a, k)
        return fn


class _Lock:
    def lock(self):
        pass

    def unlock(self):
        pass


def _not_replaced(*_a, **_k):
    raise NotImplementedError("hot-path body of the stand-in: dropin.install must replace it")


def make(which: str) -> types.ModuleType:
    mod = types.ModuleType("standin_pypanadapter_" + which)
    st = types.SimpleNamespace(fft_size=2048, fft_ratio=2, fft_avg=128, fft_tapering="hamming", scroll=1,
                               panadapter=types.SimpleNamespace(SampleRate=2.56e6, driver=object()))
    mod.AppState = st

    class Waterfall:
        """Image item (S:1579-1686): the drop-in supplies init_image / image_update /
        autolevel / newlevel / img_array; scale and setImage are pyqtgraph's."""

        def __init__(self):
            self.fftwidth = 0
            self.minlev, self.maxlev = -220, -120              # S:1592-1593
            self.shown = {}

        def scale(self, *a, **k):
            pass

        def setImage(self, img, **k):
            self.shown = dict(img=np.array(img), kw=k)

        init_image = image_update = autolevel = newlevel = _not_replaced

    mod.Waterfall = Waterfall

    class _Spin:
        def __init__(self, v=0.0):
            self.v = v

        def value(self):
            return self.v

    class _Plot:
        def __init__(self):
            self.items = []

        def plot(self, data, pen=None):
            item = _Recorder()
            item.calls["setData"] = ((np.array(data),), {})
            self.items.append(item)
            return item

    class FFTTaperingControl:
        """The taper dialog (S:1220-1379) reduced to what ShowCurve touches."""
        taper_list = {"hamming": [], "kaiser": [("beta", 14)], "general gaussian": [("power", 1.5), ("stndrd dev", 7)]}
        taper_size = 51
        fft_size = 2048

        def __init__(self, taper, p0=0.0, p1=0.0):
            self.taper = taper
            self.P0val, self.P1val = _Spin(p0), _Spin(p1)
            self.plot0, self.plot1 = _Plot(), _Plot()
            self.taperplot = self.fftplot = None

        ShowCurve = _not_replaced

    mod.FFTTaperingControl = FFTTaperingControl

    if which == "spectrum":
        class ApplicationDisplay:
            """S:1687-2139: read() hands a chunk of fft_size*fft_avg samples to update()."""

            def __init__(self, n_win):
                self.N_WIN = n_win                              # S:1712
                self.win = _Recorder()
                self.spectrum_plot = _Recorder()
                self.waterfall = Waterfall()

            zoomfft = update = _not_replaced

        mod.ApplicationDisplay = ApplicationDisplay
        return mod

    if which != "thread":
        raise ValueError(which)

    class Data:
        """T:1400-1483; replaced wholesale by the drop-in's pinned-ring Data."""

        def __init__(self, chunk_size=8196 * 2):
            self.chunk_size = chunk_size
            self.max_size = 16 * chunk_size
            self.NR = None

        new_complex = new_real = add = get_data_start = get_data_end = _not_replaced

    class PSD:
        def __init__(self, dataclass):
            self.psd = np.zeros(st.fft_size)                    # T:1490: blank row until the first update
            self.dataclass = dataclass
            self.lock = _Lock()
            self.loop = True

        update = _not_replaced                                  # T:1513-1549

    class ApplicationDisplay:
        """T:2140-2157: the GUI timer shows whatever row PSD holds right now."""

        def __init__(self, psd):
            self.psd = psd
            self.waterfall = Waterfall()
            self.spectrum_plot = _Recorder()

        def update(self):
            self.psd.lock.lock()
            row = self.psd.psd
            self.psd.lock.unlock()
            self.waterfall.image_update(row)
            hz = st.panadapter.SampleRate / 4
            self.spectrum_plot.setData(np.linspace(-hz, hz, row.shape[0]), row, pen="g")

    mod.Data, mod.PSD, mod.ApplicationDisplay = Data, PSD, ApplicationDisplay
    return mod


def set_state(mod, fs, fft_size, fft_ratio, fft_avg, window):
    st = mod.AppState
    st.panadapter.SampleRate = fs
    st.fft_size, st.fft_ratio, st.fft_avg, st.fft_tapering = fft_size, fft_ratio, fft_avg, window
    return st
