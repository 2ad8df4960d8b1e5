/*
 * zoomfft_b200.h -- C ABI of the B200-native zoom-FFT PSD engine.
 *
 * This is the drop-in boundary for the one hot path of alfille/pypanadapter:
 * sample chunk -> LO mix -> cascade of decimate-by-2 -> Welch PSD ->
 * fftshift/crop -> 20*log10 -> (EMA) -> waterfall row.  The reference has no
 * FFI for this path (it is inline numpy/scipy in Qt methods); every entry
 * point below cites the reference lines whose work it replaces.
 *   S: = pypanadapter_spectrum.py   T: = pypanadapter_thread.py
 *
 * Conventions: plain C, no torch/CUDA types in signatures (streams and device
 * pointers travel as void*), every call returns 0 or a negative errno-style
 * code and never throws/aborts; zfb_last_error() gives the message.  Caller
 * owns every host/device buffer it passes; the engine owns its workspaces.
 * One engine = one CUDA device; calls on one engine must be serialised by the
 * caller (the Python shim holds a lock), different engines are independent.
 * There is no CPU fallback: without a CUDA device zfb_create fails.
 */
#ifndef ZOOMFFT_B200_H
#define ZOOMFFT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZFB_ABI_VERSION 3

/* status codes */
#define ZFB_OK            0
#define ZFB_EINVAL      (-22)  /* bad argument / unsupported configuration   */
#define ZFB_ENOMEM      (-12)  /* host or device allocation failed           */
#define ZFB_ENODEV      (-19)  /* no usable CUDA device                      */
#define ZFB_ECUDA       (-5)   /* CUDA runtime error (see zfb_last_error)    */
#define ZFB_ESTATE      (-1)   /* call out of order (e.g. not configured)    */
#define ZFB_ETOOSHORT   (-34)  /* chunk shorter than the reference accepts   */

/* sample wire formats (zfb_config.dtype) */
#define ZFB_DTYPE_C64   0      /* interleaved float32 I,Q  (SoapySDR CF32, S:602) */
#define ZFB_DTYPE_U8    1      /* interleaved uint8 offset-binary I,Q (RTL-SDR;
                                  converted as pyrtlsdr does: u/127.5 - 1, S:543) */
#define ZFB_DTYPE_CS16  2      /* interleaved int16 I,Q (SoapySDR CS16 -- the native format of
                                  most Soapy devices; the reference asks for CF32, S:602, and
                                  lets SoapySDR convert on the host): (I + jQ) / 32768, by one
                                  streaming pass on the device in front of the complex64 path
                                  (SURVEY 8f.3; no reference code to match: unpinned) */

/* decimator implementations (zfb_config.mode) */
#define ZFB_MODE_EXACT  0      /* per-chunk zero-phase cheby1 IIR, scipy semantics */

#define ZFB_MODE_FAST   1      /* interior: fused NCO mix + multistage polyphase FIR
                                  decimator + compensator for all but the last
                                  decimate call, last call and both chunk edges by
                                  the exact kernels (needs zfb_set_fast_plan; falls
                                  back to EXACT for fft_ratio < 4 or short chunks) */

/* zfb_config.flags */
#define ZFB_FLAG_NO_LO   1     /* skip the LO mix (amplitude 1, f = 0): the chain is
                                  then exactly scipy.signal.decimate(x, 2) x log2(R)
                                  -- the call S:2098 / T:1534 makes -- plus welch   */
#define ZFB_FLAG_LINEAR  2     /* rows hold the linear PSD (welch's Pxx, S:2111)
                                  instead of 20*log10(abs(.)) (S:2117-2119)         */
#define ZFB_FLAG_ONESIDED 4    /* the chunk is REAL (imaginary parts zero: AudioPan,
                                 S:712-714, Data.new_real T:1413-1417) and fft_ratio is 1:
                                 scipy.signal.welch then returns the one-sided density
                                 (N/2+1 bins, doubled except DC and Nyquist) and the
                                 reference fftshifts and crops THAT array (T:1538-1543,
                                 S:2111-2114).  Rows are row_width/2 + 1 bins wide:
                                 shifted[N/2 - row_width/2 : N/2 + 1].  N <= 8192.      */

typedef struct zfb_engine zfb_engine;

/*
 * One frame configuration == the AppState the reference reads each frame
 * (S:1492-1497: fft_size, fft_ratio, fft_avg, fft_tapering; SampleRate).
 */
typedef struct zfb_config {
    double  fs;          /* AppState.panadapter.SampleRate (S:2091,2111)       */
    int32_t fft_size;    /* AppState.fft_size N, power of two 32..262144       */
    int32_t fft_ratio;   /* AppState.fft_ratio R, power of two 1..512 (S:2079) */
    int32_t frame_len;   /* samples per chunk (avg*N in S:1764; any in T:1516) */
    int32_t row_width;   /* W bins kept around DC (S:2114 N_WIN; T:1542)       */
    int32_t nperseg;     /* window length = min(N, decimated length)           */
    int32_t dtype;       /* ZFB_DTYPE_*                                        */
    int32_t flip;        /* 1 = np.flip the chunk first (S:460,543; T:460)     */
    int32_t mode;        /* ZFB_MODE_*                                         */
    int32_t flags;       /* ZFB_FLAG_* bits                                    */
    double  f_demod;     /* software LO in Hz; reference hard-wires 1.0 (S:2090) */
    double  ema_alpha;   /* <0: off.  a=alpha*p+(1-alpha)*a on linear power    */
    const double *window;/* nperseg taps = scipy.signal.get_window(taper,nperseg) */
} zfb_config;

/* ---- life cycle ------------------------------------------------------- */
int  zfb_abi_version(void);
/* "sm_100a" for the product library. */
const char *zfb_build_kind(void);
/* sha256 of the sources and compiler flags this library was built from
 * (pypanadapter_b200/build.py compares it with the tree before reusing a build). */
const char *zfb_source_hash(void);
/* create an engine on CUDA device `device`; fails with ZFB_ENODEV when there
 * is no GPU (no CPU fallback exists). */
int  zfb_create(int device, zfb_engine **out);
void zfb_destroy(zfb_engine *e);
/* message of the last failure on `e` (or of the last failed zfb_create when
 * e == NULL).  Valid until the next call on the same engine/thread. */
const char *zfb_last_error(const zfb_engine *e);

/* FIR plan of ZFB_MODE_FAST for one fft_ratio: nstages = log2(R) - 1 symmetric
 * decimate-by-2 FIRs (stage s at rate fs/2^s, 2*half[s]+1 taps, centre tap
 * first) that replace the first log2(R)-1 scipy.signal.decimate calls of
 * S:2097-2098 in the chunk interior, one symmetric compensator at rate
 * 2fs/R, and the number of decimated samples at either chunk end that the
 * exact path recomputes.  Designed by pypanadapter_b200/fastdesign.py. */
#define ZFB_FAST_MAX_STAGES 12
typedef struct zfb_fast_plan {
    int32_t nstages;
    int32_t half[ZFB_FAST_MAX_STAGES];
    const double *taps[ZFB_FAST_MAX_STAGES];   /* half[s] + 1 values each */
    int32_t comp_half;
    const double *comp_taps;                   /* comp_half + 1 values */
    int32_t strip;                             /* even, >= 64 */
} zfb_fast_plan;

/* ---- configuration ---------------------------------------------------- */
/* (Re)plan for a frame shape.  Cheap when only frame_len changes; the
 * reference lets N, R, window, avg change between any two frames (S:1753,
 * S:2079-2086).  Resets the EMA state when the row geometry changes. */
int  zfb_configure(zfb_engine *e, const zfb_config *cfg);
/* Hand over (a copy of) the FIR plan the next zfb_configure with
 * mode == ZFB_MODE_FAST uses; plan->nstages must be log2(fft_ratio) - 1. */
int  zfb_set_fast_plan(zfb_engine *e, const zfb_fast_plan *plan);
/* 1 if the current configuration runs the FAST interior, 0 if it runs EXACT. */
int  zfb_fast_active(const zfb_engine *e);
/* Use the caller's CUDA stream (cudaStream_t as void*) for all kernels;
 * NULL restores the engine's own stream. */
int  zfb_set_stream(zfb_engine *e, void *cuda_stream);
/* Frames processed per launch group (intermediates of one group are sized to
 * stay L2-resident).  0 = automatic. */
int  zfb_set_group(zfb_engine *e, int frames_per_group);
int  zfb_reset_ema(zfb_engine *e);
/* tuning knobs: "decim_threads" = 0 (auto) | 128 | 256
 * threads per decimator CTA (8192- / 16384-sample shared-memory region);
 * "welch_splits" = CTAs per frame in the Welch kernel, 0 = auto.
 * "late_mix" = 1 (default): mode FAST may apply the software LO at the output
 * of the first FIR chain instead of its input when |f_demod| * fft_ratio / fs
 * <= 1e-3 (the reference's LO sits at 1 Hz, S:2090; the chain's gain then moves
 * by < 1e-3 dB); 0: always mix first.
 * "ring_append" = 1 (default): every processed row also enters the waterfall
 * ring; 0: only zfb_ring_push_rows does (display loops that show a subset of
 * the rows, like the threaded variant's GUI timer, T:2140-2148).
 * "precise" = -1 (default: rows of <= 6 Welch segments take the fp64 path),
 * 0 never, 1 always.
 * Measurement knobs of mode FAST (defaults are the measured best; rows do not
 * depend on them beyond 1e-3 dB): "strips_async" 0 | 1 (edge strips on the
 * main stream | side stream, submitted before the FIR chain), "strip_split",
 * "strip_decay", "strip_decay_early", "fir_generic", "iir_stream" 0 | 1
 * (streaming last stage), "iir_stream_len", "iir_stream_warm", "iir_l2_keep",
 * "welch_prune" 0 | 1 | 2.
 * "slabs" = 0 | 1: accepted for existing callers and changes nothing (a batch
 * always runs through one lane unless it is pipelined).
 * "pipeline": see zfb_join.
 * "host_taper" = 1 (default): zfb_process_host cuts a batch into sub-groups
 * that halve towards its end (copies overlap compute; only the last, smallest
 * sub-group's kernels are left after the last copy); 0: four equal sub-groups.
 * Unknown names: ZFB_EINVAL. */
int  zfb_set_option(zfb_engine *e, const char *name, long long value);
/* Lanes the last zfb_process_device batch ran through: 2 (pipeline) or 1. */
int  zfb_slab_lanes(const zfb_engine *e);
/* Pipelined batches, zfb_set_option("pipeline", 1) (default 0; mode FAST, rows
 * on the fp32 path): zfb_process_device hands whole batches to the two lane
 * engines in turn and finishes their rows (EMA in frame order, ring) on a
 * stream of its own WITHOUT making the engine's stream wait: the FIR interior
 * of batch k + 1 runs beside the last stage / strips / Welch of batch k.  The
 * caller orders the rows (and the reuse of d_in) with zfb_join: the given
 * stream -- NULL or the engine's own: that one -- waits for every batch handed
 * over so far.  zfb_synchronize and every other call on the engine join
 * implicitly.  Rows are bit-identical to "pipeline" = 0. */
int  zfb_join(zfb_engine *e, void *cuda_stream);

/* ---- the hot path ----------------------------------------------------- */
/*
 * Replaces the bodies of ApplicationDisplay.zoomfft+update (S:2088-2119) and
 * PSD.update (T:1525-1548) for `nframes` independent chunks laid out
 * back to back ([nframes][frame_len] samples of cfg.dtype).
 *   d_in   : device pointer to the chunks
 *   d_rows : device pointer, [nframes][row_width] float32 dB20 rows, or NULL
 * Rows are also appended to the engine's device-resident waterfall ring.
 * Asynchronous: kernels are enqueued on the engine's stream and the call
 * returns; use zfb_synchronize / zfb_read_rows to wait.
 */
int  zfb_process_device(zfb_engine *e, const void *d_in, int nframes,
                        float *d_rows);
/*
 * Same, for HOST buffers: h_in is copied to the device in groups with async
 * H2D copies on a dedicated copy stream (directly if h_in is pinned, through
 * the engine's pinned staging ring otherwise), overlapped with compute; the
 * rows are copied back to h_rows.  Blocks until h_rows is complete.
 */
int  zfb_process_host(zfb_engine *e, const void *h_in, int nframes,
                      float *h_rows);
/*
 * Several virtual receivers over the SAME chunks (BASELINE configs[3]: distinct
 * zoom centres over one wide stream): channel c runs the configured chain with
 * the software LO (S:2090) at f_demod[c] Hz instead of cfg.f_demod.  The input
 * is uploaded / read once per group, rows come back as [nch][nframes][row_width].
 * Needs fft_ratio >= 2 and ema_alpha < 0 (the EMA state is per engine).
 */
int  zfb_process_channels_device(zfb_engine *e, const void *d_in, int nframes,
                                 const double *f_demod, int nch, float *d_rows);
int  zfb_process_channels_host(zfb_engine *e, const void *h_in, int nframes,
                               const double *f_demod, int nch, float *h_rows);
int  zfb_synchronize(zfb_engine *e);

/* mixed + decimated chunk of the last processed frame group's FIRST frame
 * (what zoomfft returns, S:2100), for parity tests of the decimator alone:
 * copies up to `max_samples` complex64 samples to h_out, returns the count
 * (>=0) or a negative status. */
int  zfb_debug_read_decimated(zfb_engine *e, float *h_out_iq, int max_samples);

/* ---- device-resident waterfall ring (replaces Waterfall.img_array,
 *      S:1631,1651-1652: rows stay on the device until displayed) -------- */
int  zfb_ring_configure(zfb_engine *e, int rows);      /* default 256 rows; the ring's width
                                                         * follows the configured row_width */
/* A ring with a width of its own, independent of what is configured (usable before
 * the first zfb_configure): the reference's Waterfall takes rows of ANY width and
 * re-initialises its image when the width changes (S:1638-1643) -- e.g. the blank
 * np.zeros(fft_size) row PSD publishes before the first real one (T:1490, T:2140-2148),
 * or the stale-width row right after a zoom click.  The ring starts empty.  Rows the
 * engine computes enter such a ring only while row_width == width; zfb_ring_push_rows,
 * zfb_read_rows, zfb_ring_image and zfb_ring_quantiles work on `width` columns. */
int  zfb_ring_configure_width(zfb_engine *e, int rows, int width);
int  zfb_ring_width(const zfb_engine *e);              /* columns of the ring, 0: none yet */
int64_t zfb_ring_rows_written(const zfb_engine *e);    /* monotone counter  */
/* copy `nrows` rows ending `age` rows before the newest one to host
 * (age 0 = newest); blocks only until those rows are complete. */
int  zfb_read_rows(zfb_engine *e, int age, int nrows, float *h_out);

/* append `nrows` host rows (float32 [nrows][row_width]) to the device ring, as
 * if the engine had produced them (Waterfall.image_update(psd) with a row
 * that was computed elsewhere, S:1638-1652). */
int  zfb_ring_push_rows(zfb_engine *e, const float *h_rows, int nrows);

/* ---- max-hold, min-hold and average traces, peak markers (DESIGN 3.8) -----
 * The reference plots each row as it arrives (spectrum_plot.setData(psd),
 * S:2130) and keeps nothing across rows.  A trace set extends that plot with the
 * standard traces of a spectrum analyser, kept on the device over EVERY row the
 * engine computes -- also rows that never reach the ring (ring_append = 0, the
 * threaded GUI's skipped rows, T:2140-2148) -- in the rows' own units (dB20, or
 * linear power with ZFB_FLAG_LINEAR):
 *   ZFB_TRACE_LAST  the newest row
 *   ZFB_TRACE_MAX   running maximum per column (NaN ignored, fmaxf)
 *   ZFB_TRACE_MIN   running minimum per column (fminf)
 *   ZFB_TRACE_AVG   mean linear power (the row, or 10^(v/20) of a dB20 row), summed
 *                   in fp64 in frame order; read out as sum/count, in dB20 as
 *                   20 log10(sum/count), rounded to float
 * Rows of zfb_process_device, zfb_process_host and zfb_samples_process feed it on
 * every path (slabs, pipelined batches, fp64 rows), with EMA applied as the
 * caller gets them; rows of zfb_ring_push_rows do not.  LAST, MAX, MIN and the
 * fp64 sum are bit-identical however the same frames are split into calls,
 * groups, slabs or batches.  The set is off by default: then nothing is
 * allocated or launched and rows, ring and counters are as without it.  It
 * starts empty on zfb_traces_enable, zfb_traces_reset and a zfb_configure that
 * changes fs, fft_size, fft_ratio, row_width, f_demod or flags; it keeps
 * counting over a change of frame_len (PSD.update hands over chunks of varying
 * length, T:1516-1520), window, ema_alpha, dtype, flip or mode.  While it is on,
 * zfb_process_channels_* return ZFB_EINVAL (one trace set per engine). */
#define ZFB_TRACE_LAST 0
#define ZFB_TRACE_MAX  1
#define ZFB_TRACE_MIN  2
#define ZFB_TRACE_AVG  3
int  zfb_traces_enable(zfb_engine *e, int on);
int  zfb_traces_reset(zfb_engine *e);
/* rows in the traces since they last started empty (0 while off) */
int64_t zfb_traces_count(const zfb_engine *e);
/* row_width floats of trace `kind` to h_out; joins pending work, blocks.
 * ZFB_ESTATE when the traces are off or hold no row. */
int  zfb_trace_read(zfb_engine *e, int kind, float *h_out);
/* Peak markers of trace `kind`: scipy.signal.find_peaks(trace, height=height,
 * distance=distance) -- local maxima, a plateau's midpoint, never the first or
 * last column, NaN never a peak; height filter first, then scipy's greedy
 * distance selection -- and of those the k highest in descending order (ties to
 * the lower column).  Per marker: its column, the trace value there and the
 * parabolic offset 0.5(a-c)/(a-2b+c) in fp64 from the three values around it
 * (0 on a plateau or next to a non-finite value).  1 <= k <= 64, distance >= 1,
 * height NaN = none.  *npeaks = markers written.  Only the markers are copied
 * back.  Errors as zfb_trace_read. */
int  zfb_trace_peaks(zfb_engine *e, int kind, int k, int distance, double height, int32_t *cols, float *values,
                     double *offsets, int *npeaks);
/* the same on any device vector of n float32 (1 <= n <= 262144), e.g. a row of
 * zfb_process_device; ordered on the engine's stream, blocks. */
int  zfb_find_peaks_device(zfb_engine *e, const float *d_x, int n, int k, int distance, double height,
                           int32_t *cols, float *values, double *offsets, int *npeaks);

/* ---- waterfall image and autolevel on the device (SURVEY 8f.1) -----------
 * Replaces Waterfall.init_image / image_update's img_array bookkeeping
 * (S:1625-1662: -500 fill, grid columns, np.roll of the whole image per row,
 * tick marks) and the level -> colour-table mapping pyqtgraph applies to it
 * (S:1592-1594 setLevels, S:1612-1623 lookuptable, S:1664 setImage): the
 * [height][row_width] image the reference would hold after `rows_seen`
 * image_update calls with AppState.scroll = `scroll` is produced from the ring
 * by one kernel when it is displayed.
 *   kind ZFB_IMAGE_F32 : float32 img_array itself
 *   kind ZFB_IMAGE_U8  : colour indices clip(trunc((v-minlev)*256/(maxlev-minlev)),0,255)
 *   kind ZFB_IMAGE_RGBA: lut_rgba[index] (256 x 4 bytes, R G B A in memory order)
 * `out` is a host buffer (blocks until it is filled) or, with out_on_device
 * != 0, a device buffer (asynchronous on the engine's stream). */
#define ZFB_IMAGE_F32  0
#define ZFB_IMAGE_U8   1
#define ZFB_IMAGE_RGBA 2
int  zfb_ring_image(zfb_engine *e, int height, int scroll, int64_t rows_seen,
                    int kind, double minlev, double maxlev,
                    const uint8_t *lut_rgba, void *out, int out_on_device);
/* Replaces Waterfall.autolevel's np.percentile(img_array[img_array < 0],
 * [2, 98]) (S:1676): out_values[i] = the q[i]-quantile (0..1, numpy's default
 * linear interpolation between exact order statistics) of the image pixels
 * below zero; *out_count = how many there are (0: values are NaN). */
int  zfb_ring_quantiles(zfb_engine *e, int height, int scroll, int64_t rows_seen,
                        const double *q, int nq, double *out_values,
                        int64_t *out_count);

/* ---- taper design and preview on the device (SURVEY 8f.4) ----------------
 * The taper dialog's live preview (FFTTaperingControl.ShowCurve, S:1354-1379):
 * zfb_taper_design replaces scipy.signal.get_window(AppState.fft_tapering, 51)
 * (S:1366) for the closed-form families of its taper_list (S:1222-1243), in
 * fp64 on the device; `periodic` = get_window's fftbins=True.  kind:
 *   0 boxcar 1 triang 2 bartlett 3 hann 4 hamming 5 blackman 6 nuttall
 *   7 blackmanharris 8 flattop 9 bohman 10 barthann 11 parzen 12 kaiser(p0=beta)
 *   13 gaussian(p0=std) 14 general gaussian(p0=power, p1=std)
 *   15 exponential(p0=center, p1=tau) 16 tukey(p0=taper fraction)
 * (chebwin / dpss / slepian need a polynomial design or an eigenproblem: host.)
 * zfb_taper_preview replaces S:1374-1376: h_db_out[k] = 20*log10(|FFT(taper
 * zero-padded to nfft)[k]| / max_k |.|), nfft float32 values. */
int  zfb_taper_design(zfb_engine *e, int kind, double p0, double p1, int n,
                      int periodic, double *h_out);
int  zfb_taper_preview(zfb_engine *e, const double *taper, int ntaps, int nfft,
                       float *h_db_out);

/* ---- pinned sample ring with double-buffered device mirror -------------
 * Replaces Data.data (T:1415-1421) and the copy-in of Data.add (T:1447): the
 * producer thread writes chunks into pinned host memory and each chunk is sent
 * to the device at once by an async H2D copy on the engine's copy stream, so
 * the samples are already resident when PSD.update (T:1513) asks for a row.
 * Fold-back bookkeeping (size / real_size / total_size) stays with the caller. */
int  zfb_samples_create(zfb_engine *e, int64_t capacity_samples, int dtype);
/* pinned host storage of the ring (capacity * sample size bytes) or NULL */
void *zfb_samples_host_ptr(zfb_engine *e);
/* call before writing host samples [offset, offset+n): waits until no earlier
 * H2D copy still reads that memory */
int  zfb_samples_begin_write(zfb_engine *e, int64_t offset, int64_t n);
/* samples [offset, offset+n) are written: enqueue their H2D copy */
int  zfb_samples_commit(zfb_engine *e, int64_t offset, int64_t n);
/* run the configured chain on samples [0, cfg.frame_len) of the device mirror
 * (one frame), copy the row to h_row (row_width floats) and switch the
 * producer to the other device mirror.  Blocks until h_row is complete. */
int  zfb_samples_process(zfb_engine *e, float *h_row);

/* ---- pinned host memory for the sample ring (replaces Data.data,
 *      T:1415,1421) ------------------------------------------------------ */
int  zfb_alloc_pinned(size_t bytes, void **out);
int  zfb_free_pinned(void *p);

/* ---- introspection (host only; usable without a GPU) ------------------- */
/* the 4x6 SOS of scipy.signal.cheby1(8, 0.05, 0.4) the decimator realises
 * (scipy:_signaltools.py:5317-5319), row-major [b0 b1 b2 a0 a1 a2]. */
int  zfb_decim_sos(double out24[24]);
/* geometry of a configuration without touching the device: fills
 * out[0]=decimated length, out[1]=nperseg, out[2]=hop, out[3]=nseg,
 * out[4]=number of decimation stages. */
int  zfb_plan_geometry(int frame_len, int fft_size, int fft_ratio, int out5[5]);
/* counters since create: [0] frames, [1] input samples, [2] kernels launched,
 * [3] H2D bytes, [4] D2H bytes. */
int  zfb_get_counters(const zfb_engine *e, uint64_t out5[5]);


/* ---- per-kernel device timing (bench.py's roofline leg) ------------------ */
/* kernel classes: 0..15 = decimate-by-2 stage s (replaces scipy.signal.
 * decimate call s of the loop at S:2097-2098), 16 = Welch kernel / four-step
 * column pass, 17 = four-step row pass (both: scipy.signal.welch, S:2111),
 * 18 = row finalisation (S:2114-2119 + EMA, trace update), 19 = waterfall image
 * (S:1625-1664), 20 = autolevel selection sweep (S:1676). */
#define ZFB_PROF_CLASSES 21
/* on != 0: bracket every kernel launch with CUDA events on the engine's
 * stream (no host synchronisation is added). */
int  zfb_set_profiling(zfb_engine *e, int on);
/* synchronise, add up the recorded intervals per class and clear them:
 * ms_out[c] = total device milliseconds, launches_out[c] = launches timed. */
int  zfb_get_profile(zfb_engine *e, double ms_out[ZFB_PROF_CLASSES],
                     uint64_t launches_out[ZFB_PROF_CLASSES]);

#ifdef __cplusplus
}
#endif
#endif /* ZOOMFFT_B200_H */
