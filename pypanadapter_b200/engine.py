"""Python face of the zoom-FFT PSD engine (thin layer over the C ABI).

``ZoomPSD`` wraps one ``zfb_engine`` (one CUDA device).  ``zoom_psd`` is the
fused frame call that replaces the bodies of the reference's
``ApplicationDisplay.zoomfft`` + ``update`` (pypanadapter_spectrum.py:2088-2119)
and ``PSD.update`` (pypanadapter_thread.py:1513-1549):

    chunk -> [uint8 -> complex, np.flip] -> x * sqrt(2) exp(-2j pi f_demod t)
          -> scipy.signal.decimate(., 2) x log2(R) -> scipy.signal.welch
          -> fftshift + centre crop -> 20*log10(abs(.)) [-> EMA]

All arithmetic happens in the sm_100a kernels; this file only validates
arguments, builds the window table (host, ``scipy.signal.get_window`` -- the
same call the reference's welch makes, scipy:_spectral_py.py:901) and moves
pointers.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib

_ERRNAMES = {
    _lib.ZFB_EINVAL: "EINVAL", _lib.ZFB_ENOMEM: "ENOMEM", _lib.ZFB_ENODEV: "ENODEV",
    _lib.ZFB_ECUDA: "ECUDA", _lib.ZFB_ESTATE: "ESTATE", _lib.ZFB_ETOOSHORT: "ETOOSHORT",
}


class ZoomFFTError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("%s (%s)" % (message, _ERRNAMES.get(code, code)))
        self.code = code


# wire formats: name -> (ZFB_DTYPE_*, numpy dtype of the interleaved stream or None for complex64,
#                        stream elements per sample)
_DTYPES = {
    "c64": (_lib.ZFB_DTYPE_C64, None, 1),
    "u8": (_lib.ZFB_DTYPE_U8, np.uint8, 2),        # RTL-SDR offset binary
    "cs16": (_lib.ZFB_DTYPE_CS16, np.int16, 2),    # SoapySDR CS16
}

_window_cache: dict = {}
_window_lock = threading.Lock()


def window_table(window, nperseg: int) -> np.ndarray:
    """Periodic window of ``nperseg`` taps exactly as ``scipy.signal.welch``
    builds it (``get_window(window, nperseg)``, fftbins=True); accepts the
    taper dialog's ``str`` or ``(name, p0[, p1])`` forms (S:1354-1363) or an
    explicit array (scipy's array_like window)."""
    if isinstance(window, (str, tuple)):
        key = (window if isinstance(window, str) else tuple(window), int(nperseg))
        with _window_lock:
            w = _window_cache.get(key)
        if w is None:
            from scipy.signal import get_window
            w = np.ascontiguousarray(get_window(window, int(nperseg)), dtype=np.float64)
            w.setflags(write=False)
            with _window_lock:
                _window_cache[key] = w
        return w
    w = np.ascontiguousarray(window, dtype=np.float64)
    if w.ndim != 1 or w.shape[0] != nperseg:
        raise ValueError("window must have length nperseg")   # scipy:_spectral_py.py _triage_segments
    return w


def crop_width(fft_size: int, fft_ratio, crop) -> int:
    """Row width W: ``'thread'`` -> ``2*int(.5*N/R)`` (T:1542); int -> the
    ``N_WIN`` of S:2114 (rounded down to even, as the slice does); None -> N."""
    if crop is None:
        return int(fft_size)
    if isinstance(crop, str):
        if crop != "thread":
            raise ValueError("crop must be 'thread', an int or None")
        return 2 * int(.5 * fft_size / fft_ratio)
    return 2 * (int(crop) // 2)


def plan_geometry(frame_len: int, fft_size: int, fft_ratio: int, lib=None) -> dict:
    """Lengths the reference's scipy calls produce for this frame shape."""
    lib = lib or _lib.product_library()
    out = (C.c_int * 5)()
    rc = lib.zfb_plan_geometry(int(frame_len), int(fft_size), int(fft_ratio), out)
    if rc == _lib.ZFB_ETOOSHORT:
        # scipy raises ValueError from sosfiltfilt's _validate_pad
        raise ValueError("The length of the input vector x must be greater than padlen, which is 27.")
    if rc != 0:
        raise ZoomFFTError(rc, "bad frame geometry (frame_len=%r, fft_size=%r, fft_ratio=%r)"
                           % (frame_len, fft_size, fft_ratio))
    return dict(ndec=out[0], nperseg=out[1], hop=out[2], nseg=out[3], nstages=out[4])


class ZoomPSD:
    """One engine on one CUDA device.  Thread-safe (the C side serialises)."""

    def __init__(self, device: int = 0, *, lib=None):
        self._lib = lib or _lib.product_library()
        self._h = C.c_void_p()
        rc = self._lib.zfb_create(int(device), C.byref(self._h))
        if rc != 0:
            msg = self._lib.zfb_last_error(None)
            raise ZoomFFTError(rc, "zfb_create(device=%d): %s" % (device, msg.decode() if msg else "?"))
        self.device = int(device)
        self._key = None
        self.row_width = 0
        self.frame_len = 0
        self.dtype = None
        self.geometry = None

    # -- life cycle ------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.zfb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc, what):
        if rc < 0:
            msg = self._lib.zfb_last_error(self._h)
            raise ZoomFFTError(rc, "%s: %s" % (what, msg.decode() if msg else "?"))
        return rc

    # -- configuration ---------------------------------------------------
    def configure(self, fs, fft_size, fft_ratio, frame_len, window="hamming", *,
                  dtype="c64", flip=False, f_demod=1.0, crop="thread",
                  ema_alpha=None, no_lo=False, linear=False, mode="fast", onesided=False):
        """Plan for a frame shape (cheap if nothing changed).  Mirrors the
        AppState the reference reads per frame (S:1492-1497).

        ``mode``: ``"exact"`` -- every decimate call by the zero-phase IIR
        kernels; ``"fast"`` -- polyphase-FIR interior + exact last stage +
        exact chunk edges (same parity bar; falls back to exact for
        fft_ratio < 4 or short chunks, see ``fast_active``).

        ``onesided``: the samples are REAL (AudioPan S:712-714; stored as
        complex64 with zero imaginary part) and ``fft_ratio`` is 1: rows are what
        the reference gets from welch's one-sided spectrum (N/2+1 bins) after
        its fftshift and crop (T:1538-1543), ``crop_width/2 + 1`` bins wide."""
        fft_ratio_i = int(fft_ratio)
        if dtype not in _DTYPES:
            raise ValueError("dtype must be one of %s, got %r" % (", ".join(map(repr, _DTYPES)), dtype))
        if mode not in ("exact", "fast"):
            raise ValueError("mode must be 'exact' or 'fast'")
        if onesided and (fft_ratio_i != 1 or dtype != "c64"):
            raise ValueError("onesided rows are the real-input, fft_ratio == 1 case")
        wkey = window if isinstance(window, (str, tuple)) else ("array", np.asarray(window).tobytes())
        key = (float(fs), int(fft_size), float(fft_ratio), int(frame_len), wkey, dtype, bool(flip),
               float(f_demod), crop, ema_alpha, bool(no_lo), bool(linear), mode, bool(onesided))
        if key == self._key:
            return self
        geo = plan_geometry(frame_len, fft_size, fft_ratio_i, self._lib)
        W = crop_width(fft_size, fft_ratio, crop)
        w = window_table(window, geo["nperseg"])
        cfg = _lib.ZfbConfig()
        cfg.fs = float(fs)
        cfg.fft_size = int(fft_size)
        cfg.fft_ratio = fft_ratio_i
        cfg.frame_len = int(frame_len)
        cfg.row_width = int(W)
        cfg.nperseg = geo["nperseg"]
        cfg.dtype = _DTYPES[dtype][0]
        cfg.flip = 1 if flip else 0
        cfg.mode = _lib.ZFB_MODE_EXACT
        if mode == "fast" and geo["nstages"] >= 2:
            self._set_fast_plan(1 << geo["nstages"])
            cfg.mode = _lib.ZFB_MODE_FAST
        cfg.flags = (_lib.ZFB_FLAG_NO_LO if no_lo else 0) | (_lib.ZFB_FLAG_LINEAR if linear else 0) | \
                    (_lib.ZFB_FLAG_ONESIDED if onesided else 0)
        cfg.f_demod = float(f_demod)
        cfg.ema_alpha = -1.0 if ema_alpha is None else float(ema_alpha)
        cfg.window = w.ctypes.data_as(C.POINTER(C.c_double))
        self._key = None               # a failed zfb_configure leaves the engine unconfigured
        self._check(self._lib.zfb_configure(self._h, C.byref(cfg)), "zfb_configure")
        self._key = key
        self._axis = (float(fs), int(fft_size), fft_ratio_i, int(W), bool(onesided),
                      float(f_demod) if fft_ratio_i > 1 and not no_lo else 0.0)
        self.row_width = int(W) // 2 + 1 if onesided else int(W)
        self.frame_len = int(frame_len)
        self.dtype = dtype
        self.geometry = geo
        return self

    def _set_fast_plan(self, ratio: int):
        # one plan per zoom ratio: a change of frame_len alone (PSD.update hands over whatever
        # the ring holds, T:1516-1520) must not touch the engine's plan, ring or EMA state
        if getattr(self, "_fast_ratio", None) == ratio:
            return
        from . import fastdesign
        plan = fastdesign.design(ratio, decim_sos(self._lib))
        fp = _lib.ZfbFastPlan()
        fp.nstages = len(plan["stages"])
        keep = []
        for i, a in enumerate(plan["stages"]):
            fp.half[i] = len(a) - 1
            fp.taps[i] = a.ctypes.data_as(C.POINTER(C.c_double))
            keep.append(a)
        fp.comp_half = len(plan["comp"]) - 1
        fp.comp_taps = plan["comp"].ctypes.data_as(C.POINTER(C.c_double))
        fp.strip = plan["strip"]
        self._check(self._lib.zfb_set_fast_plan(self._h, C.byref(fp)), "zfb_set_fast_plan")
        self.fast_plan = plan
        self._fast_ratio = ratio

    @property
    def fast_active(self) -> bool:
        return bool(self._lib.zfb_fast_active(self._h))

    @property
    def slab_lanes(self) -> int:
        """lanes the last ``process_device`` batch ran through (2: pipelined, else 1)"""
        return int(self._lib.zfb_slab_lanes(self._h))

    def join(self, cuda_stream_ptr: int | None = None):
        """Pipelined batches (``set_option("pipeline", 1)``): make a stream -- default: the engine's --
        wait for every ``process_device`` batch handed over so far."""
        self._check(self._lib.zfb_join(self._h, C.c_void_p(cuda_stream_ptr or 0)), "zfb_join")

    def set_group(self, frames_per_group: int):
        self._check(self._lib.zfb_set_group(self._h, int(frames_per_group)), "zfb_set_group")
        self._key = None

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.zfb_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)), "zfb_set_stream")

    def set_option(self, name: str, value: int):
        """Tuning knobs (zfb_set_option); the next configure() replans."""
        self._check(self._lib.zfb_set_option(self._h, name.encode(), int(value)), "zfb_set_option")
        self._key = None

    def reset_ema(self):
        self._check(self._lib.zfb_reset_ema(self._h), "zfb_reset_ema")

    def ring_configure(self, rows: int, width: int | None = None):
        """``width=None``: the ring follows the configured row width.  With a
        ``width`` the ring is the waterfall's own (S:1638-1643: any row width is
        taken, a new width re-initialises the image) and works before the
        first ``configure``."""
        if width is None:
            self._check(self._lib.zfb_ring_configure(self._h, int(rows)), "zfb_ring_configure")
        else:
            self._check(self._lib.zfb_ring_configure_width(self._h, int(rows), int(width)),
                        "zfb_ring_configure_width")

    @property
    def ring_width(self) -> int:
        return int(self._lib.zfb_ring_width(self._h))

    # -- hot path --------------------------------------------------------
    def _as_wire(self, frames):
        """(nframes, frame_len) in the configured wire dtype, C-contiguous.
        complex128 (what pyrtlsdr / the reference's Data hand over) is cast to
        complex64 here -- the device computes in fp32."""
        a = np.asarray(frames)
        _code, raw, per_sample = _DTYPES[self.dtype]
        if raw is not None:
            if a.dtype != raw:
                raise TypeError("engine is configured for %s IQ, got %s" % (np.dtype(raw).name, a.dtype))
            per = per_sample * self.frame_len
        else:
            if a.dtype != np.complex64:
                if a.dtype in (np.uint8, np.int16):
                    raise TypeError("engine is configured for complex samples, got raw %s IQ" % a.dtype)
                if not np.issubdtype(a.dtype, np.number):
                    raise TypeError("unsupported sample dtype %s" % a.dtype)
                a = a.astype(np.complex64)
            per = self.frame_len
        if a.ndim == 1:
            a = a.reshape(1, -1)
        if a.ndim != 2 or a.shape[1] != per:
            raise ValueError("frames must have shape (nframes, %d), got %r" % (per, a.shape))
        return np.ascontiguousarray(a)

    def process(self, frames, out=None) -> np.ndarray:
        """HOST buffers in, HOST rows out (float32 (nframes, W)); H2D / D2H are
        overlapped with compute on the engine's copy stream."""
        if self._key is None:
            raise ZoomFFTError(_lib.ZFB_ESTATE, "process: engine is not configured")
        a = self._as_wire(frames)
        n = a.shape[0]
        if out is None:
            out = np.empty((n, self.row_width), dtype=np.float32)
        elif out.dtype != np.float32 or out.shape != (n, self.row_width) or not out.flags.c_contiguous:
            raise ValueError("out must be C-contiguous float32 of shape (%d, %d)" % (n, self.row_width))
        self._check(self._lib.zfb_process_host(self._h, C.c_void_p(a.ctypes.data), n,
                                               C.c_void_p(out.ctypes.data)), "zfb_process_host")
        return out

    def process_channels(self, frames, f_demod, out=None) -> np.ndarray:
        """Several virtual receivers (zoom centres ``f_demod[c]`` Hz) over the
        same frames, uploaded once: rows (nch, nframes, W) float32."""
        if self._key is None:
            raise ZoomFFTError(_lib.ZFB_ESTATE, "process: engine is not configured")
        a = self._as_wire(frames)
        f = np.ascontiguousarray(f_demod, dtype=np.float64).ravel()
        n = a.shape[0]
        shape = (len(f), n, self.row_width)
        if out is None:
            out = np.empty(shape, dtype=np.float32)
        elif out.dtype != np.float32 or out.shape != shape or not out.flags.c_contiguous:
            raise ValueError("out must be C-contiguous float32 of shape %r" % (shape,))
        self._check(self._lib.zfb_process_channels_host(
            self._h, C.c_void_p(a.ctypes.data), n, f.ctypes.data_as(C.POINTER(C.c_double)), len(f),
            C.c_void_p(out.ctypes.data)), "zfb_process_channels_host")
        return out

    def process_channels_device(self, d_in_ptr: int, nframes: int, f_demod, d_rows_ptr: int):
        f = np.ascontiguousarray(f_demod, dtype=np.float64).ravel()
        self._check(self._lib.zfb_process_channels_device(
            self._h, C.c_void_p(d_in_ptr), int(nframes), f.ctypes.data_as(C.POINTER(C.c_double)), len(f),
            C.c_void_p(d_rows_ptr)), "zfb_process_channels_device")

    def process_device(self, d_in_ptr: int, nframes: int, d_rows_ptr: int | None = None):
        """DEVICE pointers in/out (asynchronous; rows also land in the ring)."""
        self._check(self._lib.zfb_process_device(self._h, C.c_void_p(d_in_ptr), int(nframes),
                                                 C.c_void_p(d_rows_ptr or 0)), "zfb_process_device")

    def synchronize(self):
        self._check(self._lib.zfb_synchronize(self._h), "zfb_synchronize")

    def read_decimated(self) -> np.ndarray:
        """Mixed + decimated chunk of the last group's first frame (what the
        reference's zoomfft returns, S:2100), complex64."""
        n = self.geometry["ndec"]
        out = np.empty(n, dtype=np.complex64)
        got = self._check(self._lib.zfb_debug_read_decimated(self._h, C.c_void_p(out.ctypes.data), n),
                          "zfb_debug_read_decimated")
        return out[:got]

    # -- device-resident waterfall ring ------------------------------------
    @property
    def rows_written(self) -> int:
        return int(self._lib.zfb_ring_rows_written(self._h))

    def read_rows(self, nrows: int = 1, age: int = 0) -> np.ndarray:
        out = np.empty((int(nrows), self.ring_width or self.row_width), dtype=np.float32)
        self._check(self._lib.zfb_read_rows(self._h, int(age), int(nrows), C.c_void_p(out.ctypes.data)),
                    "zfb_read_rows")
        return out

    # -- max-hold / min-hold / average traces and peak markers (DESIGN 3.8) --------
    def traces_enable(self, on: bool = True):
        """Keep the LAST / MAX / MIN / AVG traces on the device over every row the engine
        computes from now on (starts them empty); ``False`` drops them."""
        self._check(self._lib.zfb_traces_enable(self._h, 1 if on else 0), "zfb_traces_enable")

    def traces_reset(self):
        self._check(self._lib.zfb_traces_reset(self._h), "zfb_traces_reset")

    @property
    def trace_count(self) -> int:
        """rows in the traces since they last started empty"""
        return int(self._lib.zfb_traces_count(self._h))

    def read_trace(self, kind: str) -> np.ndarray:
        """Trace ``"last" | "max" | "min" | "avg"`` in the rows' units, float32 (row_width,)."""
        out = np.empty(self.row_width, dtype=np.float32)
        self._check(self._lib.zfb_trace_read(self._h, _trace_kind(kind), out.ctypes.data_as(C.POINTER(C.c_float))),
                    "zfb_trace_read")
        return out

    def trace_peaks(self, kind: str, k: int = 8, distance: int = 1, height=None) -> np.ndarray:
        """The ``k`` highest markers of ``scipy.signal.find_peaks(trace, height=height,
        distance=distance)`` on trace ``kind``, highest first: a structured array of
        ``column``, ``value``, ``offset`` (parabolic, in columns) and ``freq_hz``."""
        kind_i = _trace_kind(kind)
        return self._peaks(lambda *a: self._lib.zfb_trace_peaks(self._h, kind_i, *a), "zfb_trace_peaks",
                           k, distance, height, self.row_width)

    def find_peaks_device(self, ptr: int, n: int, k: int = 8, distance: int = 1, height=None) -> np.ndarray:
        """The same markers for ``n`` float32 at device address ``ptr`` (e.g. a row of
        ``process_device``); ``freq_hz`` is filled when ``n`` is the row width."""
        return self._peaks(lambda *a: self._lib.zfb_find_peaks_device(self._h, C.c_void_p(ptr), int(n), *a),
                           "zfb_find_peaks_device", k, distance, height, int(n))

    def _peaks(self, call, what, k, distance, height, n):
        k = int(k)
        cols = np.zeros(max(k, 1), dtype=np.int32)
        vals = np.zeros(max(k, 1), dtype=np.float32)
        offs = np.zeros(max(k, 1), dtype=np.float64)
        got = C.c_int(0)
        self._check(call(k, int(distance), float("nan") if height is None else float(height),
                         cols.ctypes.data_as(C.POINTER(C.c_int32)), vals.ctypes.data_as(C.POINTER(C.c_float)),
                         offs.ctypes.data_as(C.POINTER(C.c_double)), C.byref(got)), what)
        m = got.value
        out = np.zeros(m, dtype=PEAK_DTYPE)
        out["column"], out["value"], out["offset"] = cols[:m], vals[:m], offs[:m]
        if self._key is not None and n == self.row_width:
            out["freq_hz"] = self.row_frequencies()[cols[:m]] + offs[:m] * self._bin_hz()
        else:
            out["freq_hz"] = np.nan
        return out

    def _bin_hz(self) -> float:
        fs, N, R, _W, _os, _f = self._axis
        return fs / (R * N)

    def row_frequencies(self) -> np.ndarray:
        """Frequency of each row column in Hz (float64), by the column -> bin map of the
        finalisation: (j - N/2) fs/(R N) for fftshifted bin j = column + N/2 - W/2, or
        k fs/N for one-sided rows; plus f_demod where the chain mixes (R > 1, not no_lo)."""
        if self._key is None:
            raise ZoomFFTError(_lib.ZFB_ESTATE, "row_frequencies: engine is not configured")
        fs, N, R, W, onesided, f_lo = self._axis
        c = np.arange(self.row_width, dtype=np.int64)
        os_lo = N // 2 - W // 2
        if onesided:
            M = N // 2 + 1
            k = (c + os_lo + (M + 1) // 2) % M
            return k * (fs / N)
        return (c + os_lo - N // 2) * (fs / (R * N)) + f_lo

    def set_profiling(self, on: bool):
        self._check(self._lib.zfb_set_profiling(self._h, 1 if on else 0), "zfb_set_profiling")

    def profile(self) -> dict:
        """{kernel class: (total device ms, launches)} since the last call."""
        ms = (C.c_double * _lib.PROF_CLASSES)()
        n = (C.c_uint64 * _lib.PROF_CLASSES)()
        self._check(self._lib.zfb_get_profile(self._h, ms, n), "zfb_get_profile")
        return {_prof_name(c): (float(ms[c]), int(n[c])) for c in range(_lib.PROF_CLASSES) if n[c]}

    def push_rows(self, rows):
        """Append host rows to the device ring (rows computed elsewhere)."""
        r = np.ascontiguousarray(rows, dtype=np.float32)
        if r.ndim == 1:
            r = r.reshape(1, -1)
        if r.shape[1] != (self.ring_width or self.row_width):
            raise ValueError("rows must be %d wide" % (self.ring_width or self.row_width))
        self._check(self._lib.zfb_ring_push_rows(self._h, C.c_void_p(r.ctypes.data), r.shape[0]),
                    "zfb_ring_push_rows")

    # -- waterfall image / autolevel on the device (S:1625-1676) ---------------
    def ring_image(self, height: int, scroll: int, rows_seen: int, kind: str = "f32", *,
                   levels=None, lut=None) -> np.ndarray:
        """The (height, row_width) image the reference's Waterfall would hold
        after ``rows_seen`` image_update calls, assembled on the device from the
        ring: ``kind`` 'f32' = img_array, 'u8' = colour indices for ``levels``
        (minlev, maxlev), 'rgba' = ``lut[index]`` (lut: (256, 4) uint8)."""
        code = {"f32": _lib.ZFB_IMAGE_F32, "u8": _lib.ZFB_IMAGE_U8, "rgba": _lib.ZFB_IMAGE_RGBA}[kind]
        h, w = int(height), (self.ring_width or self.row_width)
        lo, hi = (0.0, 1.0) if levels is None else (float(levels[0]), float(levels[1]))
        if kind != "f32" and levels is None:
            raise ValueError("kind %r needs levels=(minlev, maxlev)" % kind)
        lut_p = None
        if kind == "rgba":
            lut = np.ascontiguousarray(lut, dtype=np.uint8)
            if lut.shape != (256, 4):
                raise ValueError("lut must be (256, 4) uint8")
            lut_p = C.c_void_p(lut.ctypes.data)
        out = np.empty((h, w) if kind != "rgba" else (h, w, 4), dtype=np.float32 if kind == "f32" else np.uint8)
        self._check(self._lib.zfb_ring_image(self._h, h, int(scroll), int(rows_seen), code, lo, hi, lut_p,
                                             C.c_void_p(out.ctypes.data), 0), "zfb_ring_image")
        return out

    def ring_image_device(self, d_out_ptr: int, height: int, scroll: int, rows_seen: int, kind: str = "u8", *,
                          levels=(-220.0, -120.0), lut=None):
        """Same, into a caller-owned device buffer (asynchronous)."""
        code = {"f32": _lib.ZFB_IMAGE_F32, "u8": _lib.ZFB_IMAGE_U8, "rgba": _lib.ZFB_IMAGE_RGBA}[kind]
        lut_p = None
        if kind == "rgba":
            lut = np.ascontiguousarray(lut, dtype=np.uint8)
            if lut.shape != (256, 4):
                raise ValueError("lut must be (256, 4) uint8")
            lut_p = C.c_void_p(lut.ctypes.data)
        self._check(self._lib.zfb_ring_image(self._h, int(height), int(scroll), int(rows_seen), code,
                                             float(levels[0]), float(levels[1]), lut_p, C.c_void_p(d_out_ptr), 1),
                    "zfb_ring_image")

    def ring_quantiles(self, height: int, scroll: int, rows_seen: int, q) -> tuple[np.ndarray, int]:
        """np.quantile(img[img < 0], q) of that image (exact order statistics,
        numpy's linear interpolation) and the number of pixels below zero."""
        qq = np.ascontiguousarray(q, dtype=np.float64).ravel()
        out = np.empty(qq.size, dtype=np.float64)
        n = C.c_int64(0)
        self._check(self._lib.zfb_ring_quantiles(self._h, int(height), int(scroll), int(rows_seen),
                                                 qq.ctypes.data_as(C.POINTER(C.c_double)), qq.size,
                                                 out.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n)),
                    "zfb_ring_quantiles")
        return out, int(n.value)

    # -- pinned sample ring (storage of buffers.Data) ------------------------
    def samples_create(self, capacity: int, dtype: str = "c64") -> np.ndarray:
        """Allocate the pinned sample ring + device mirrors; returns a numpy
        view of the pinned host storage (complex64[capacity], uint8[2*capacity]
        or int16[2*capacity])."""
        code, raw_dtype, per = _DTYPES[dtype]
        self._check(self._lib.zfb_samples_create(self._h, int(capacity), code), "zfb_samples_create")
        ptr = self._lib.zfb_samples_host_ptr(self._h)
        view = np.dtype(np.complex64 if raw_dtype is None else raw_dtype)
        nbytes = int(capacity) * per * view.itemsize
        raw = (C.c_ubyte * nbytes).from_address(ptr)
        return np.frombuffer(raw, dtype=np.uint8).view(view)

    def samples_begin_write(self, offset: int, n: int):
        self._check(self._lib.zfb_samples_begin_write(self._h, int(offset), int(n)), "zfb_samples_begin_write")

    def samples_commit(self, offset: int, n: int):
        self._check(self._lib.zfb_samples_commit(self._h, int(offset), int(n)), "zfb_samples_commit")

    def samples_process(self) -> np.ndarray:
        out = np.empty(self.row_width, dtype=np.float32)
        self._check(self._lib.zfb_samples_process(self._h, C.c_void_p(out.ctypes.data)), "zfb_samples_process")
        return out

    def counters(self) -> dict:
        c = (C.c_uint64 * 5)()
        self._check(self._lib.zfb_get_counters(self._h, c), "zfb_get_counters")
        return dict(frames=int(c[0]), samples=int(c[1]), kernels=int(c[2]),
                    h2d_bytes=int(c[3]), d2h_bytes=int(c[4]))


PEAK_DTYPE = np.dtype([("column", np.int32), ("value", np.float32), ("offset", np.float64),
                       ("freq_hz", np.float64)])

_TRACE_KINDS = {"last": _lib.ZFB_TRACE_LAST, "max": _lib.ZFB_TRACE_MAX, "min": _lib.ZFB_TRACE_MIN,
                "avg": _lib.ZFB_TRACE_AVG}


def _trace_kind(kind: str) -> int:
    if kind not in _TRACE_KINDS:
        raise ValueError("trace kind must be one of %s, got %r" % (", ".join(map(repr, _TRACE_KINDS)), kind))
    return _TRACE_KINDS[kind]


def _prof_name(c: int) -> str:
    if c < 16:
        return "decimate_stage%d" % c
    return {16: "welch", 17: "welch_rowpass", 18: "finalize", 19: "waterfall_image", 20: "autolevel_select"}[c]


def decim_sos(lib=None) -> np.ndarray:
    """The cheby1(8, 0.05, 0.4) SOS the device decimator realises."""
    lib = lib or _lib.product_library()
    out = (C.c_double * 24)()
    lib.zfb_decim_sos(out)
    return np.array(out[:], dtype=np.float64).reshape(4, 6)


# ---------------------------------------------------------------------------
# module-level convenience: one cached engine per device
# ---------------------------------------------------------------------------
_engines: dict = {}
_engines_lock = threading.Lock()


def default_engine(device: int = 0) -> ZoomPSD:
    with _engines_lock:
        e = _engines.get(device)
        if e is None:
            e = _engines[device] = ZoomPSD(device)
        return e


def zoom_psd(chunk, fs, fft_size, fft_ratio, window, *, f_demod=1.0, crop="thread",
             flip=False, ema_alpha=None, mode="fast", engine: ZoomPSD | None = None) -> np.ndarray:
    """One dB20 waterfall row of one chunk (float64 ndarray[W]).

    ``chunk``: 1-D complex64/complex128, interleaved uint8 I,Q (RTL-SDR),
    interleaved int16 I,Q (SoapySDR CS16), or
    real floats (AudioPan, S:712-714; without zoom the row is then the
    reference's fftshifted one-sided spectrum, T:1538-1543).
    ``crop``: ``'thread'`` reproduces PSD.update (T:1542-1543); an int N_WIN
    reproduces ApplicationDisplay.update (S:2114); None keeps all N bins.
    """
    chunk = np.asarray(chunk)
    if chunk.ndim != 1:
        raise ValueError("chunk must be 1-D")
    eng = engine or default_engine()
    if chunk.dtype == np.uint8 or chunk.dtype == np.int16:
        if chunk.size % 2:
            raise ValueError("interleaved IQ stream must hold an even number of values")
        dtype, n = ("u8" if chunk.dtype == np.uint8 else "cs16"), chunk.size // 2
    else:
        dtype, n = "c64", chunk.size
    onesided = dtype == "c64" and np.isrealobj(chunk) and not fft_ratio > 1
    eng.configure(fs, fft_size, fft_ratio, n, window, dtype=dtype, flip=flip,
                  f_demod=f_demod, crop=crop, ema_alpha=ema_alpha, mode=mode, onesided=onesided)
    return eng.process(chunk)[0].astype(np.float64)
