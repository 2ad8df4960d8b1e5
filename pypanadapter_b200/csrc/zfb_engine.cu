// zfb_engine.cu -- host side of the B200 zoom-FFT PSD engine and its C ABI
// (include/zoomfft_b200.h).  Plans a frame shape, owns the device workspaces,
// the pinned staging buffers, the copy stream and the device-resident
// waterfall ring, and enqueues the kernels of zfb_decim.cuh / zfb_welch.cuh.
//
// Reference lines replaced (S: = pypanadapter_spectrum.py, T: = _thread.py):
//   zoomfft + update bodies S:2088-2119, PSD.update T:1513-1549,
//   Data.data storage T:1415-1421, Waterfall.img_array S:1631,1651-1652.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <limits.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "zoomfft_b200.h"
#include "zfb_decim.cuh"
#include "zfb_welch.cuh"
#include "zfb_bigfft.cuh"
#include "zfb_firchain.cuh"
#include "zfb_iirstream.cuh"
#include "zfb_image.cuh"
#include "zfb_taper.cuh"
#include "zfb_precise.cuh"
#include "zfb_trace.cuh"

using namespace zfb;

namespace {

constexpr int kMaxStages = 16;
constexpr int kMinLog2N = 5;          // 32
constexpr int kMaxLog2Small = 13;     // 8192: one CTA per segment
constexpr int kMaxLog2N = 18;         // 262144: four-step path
constexpr int kMinLog2R16 = 16;       // 65536 and 131072: radix-16 front pass + one-CTA FFT of N/16
constexpr int kMaxLog2R16 = 17;       // (measured: 16384 is faster on the generic four-step kernels)
constexpr double kPi = 3.14159265358979323846264338327950288;

thread_local std::string g_create_error;

struct DevBuf {
    void  *p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct zfb_engine {
    int device = 0;
    int sm_count = 148;
    // Pipelined batches (zfb_set_option("pipeline") = 1): whole zfb_process_device batches alternate
    // between two LANE engines (same plan and options, own workspaces, own streams).  A lane runs a
    // batch up to the Welch power sums; this engine turns the sums into rows on fin_stream, in call
    // order (EMA strictly in frame order, dB20, ring) with the one-lane path's kernel on the same
    // operands: rows are bit-identical (virtual receivers: the lane finishes its rows itself).
    // e->stream is NOT made to wait for them until zfb_join / zfb_synchronize (or any other call on
    // the engine): the FIR interior of batch k + 1 runs beside the last stage / strips / Welch of batch k.
    bool is_lane = false, lanes_ready = false, lanes_stale = true;
    std::vector<double> window_host;             // the configured window (the caller's table may go away)
    zfb_engine *lane[2] = {nullptr, nullptr};
    int pipeline = 0;
    int next_lane = 0;
    cudaStream_t fin_stream = nullptr;
    cudaEvent_t ev_done = nullptr;               // everything issued so far is finished (on fin_stream)
    bool join_pending = false;
    int last_lanes = 1;                          // zfb_slab_lanes: 2 after a pipelined batch, else 1
    zfb_engine *last_front = nullptr;            // whose mid[] holds the last decimated chunks (debug read)
    cudaEvent_t ev_batch_in = nullptr;           // the batch's input is ready (recorded on `stream`)
    cudaEvent_t ev_lane[2] = {nullptr, nullptr}; // a lane's power sums are ready
    cudaEvent_t ev_fin[2] = {nullptr, nullptr};  // ... and consumed: the lane may overwrite them
    bool ev_fin_used[2] = {false, false};
    mutable std::mutex mu;
    std::string err;

    cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;           // edge strips of mode fast run beside the FIR interior
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int strips_async = 1;                        // zfb_set_option("strips_async"): 0 = strips on the main stream
    int strip_split = 1;                         // zfb_set_option("strip_split"): narrower regions for the late strip stages
    int strip_decay = 192;                       // zfb_set_option("strip_decay"): samples between the last stage's cut and its outputs
    int strip_decay_early = 64;                  // zfb_set_option("strip_decay_early"): the same for the stages before it
    int ring_append = 1;                         // zfb_set_option("ring_append"): processed rows enter the ring
    int late_mix = 1;                            // zfb_set_option("late_mix"): FIR chain may mix at its output
    int iir_stream = 1;                          // zfb_set_option("iir_stream"): streaming last stage of mode fast
    int iir_S = 640, iir_Wm = 256;               // zfb_set_option("iir_stream_len" (target) / "iir_stream_warm")
    int iir_l2_keep = 70;                        // zfb_set_option("iir_l2_keep"): % of a stream's blocks kept in L2
    // plan of the streaming last stage (zfb_iirstream.cuh), valid while iis.active
    struct IirStreamPlan {
        bool active = false;
        IirStreamParams q{};
        long long in_stride = 0, out_stride = 0;     // frame strides of its input / output buffers (samples)
        int tail = 0;                                // samples [L, nspf*S) of every input frame kept at zero
        TensorMap tm_in, tm_out;
    } iis;
    // fp64 path for rows of few segments (zfb_precise.cuh)
    int precise = -1;                            // zfb_set_option("precise"): -1 auto, 0 never, 1 always
    bool precise_active = false;
    int px_group = 1;
    long long px_stride = 0;
    DevBuf px_a, px_b, px_work, px_pow, px_win, px_tw;
    DevBuf taper_buf;                            // window design / preview scratch (zfb_taper.cuh)
    DevBuf strip_out;                            // [group][2][K] edge samples of the strips, patched in afterwards
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    bool slot_busy[2] = {false, false};

    bool configured = false;
    zfb_config cfg{};
    // plan
    int nstages = 0;
    int len[kMaxStages + 1] = {0};     // len[s] = input length of stage s; len[nstages] = Welch input
    int tiles[kMaxStages][2] = {{0}}, T[kMaxStages][2] = {{0}};   // [stage][0: NT=256, 1: NT=128]
    int decim_threads = 0;             // 0 = automatic per launch
    int welch_splits = 0;              // 0 = automatic
    int cs16_fused = 1;                // zfb_set_option("cs16_fused"): 0 = always widen int16 IQ by a pass of its own
    int wf_sparse_n = 0;               // non-zero bins of FFT(window) when there are few (cosine-sum windows), else 0
    int wf_sparse_bin[WF_SPARSE_MAX] = {0};
    float2 wf_sparse_val[WF_SPARSE_MAX] = {};
    int welch_prune = 2;               // 0: all bins accumulated; 1: only keepable ones; 2: + 3 CTAs/SM where it fits
    int host_taper = 1;                // zfb_set_option("host_taper"): host batches end in ever smaller sub-groups
    int fir_generic = 0;               // 1: never use the register-blocked FIR kernel (tests)
    int nperseg = 0, hop = 0, nseg = 0, W = 0, log2N = 0;
    int Wp = 0;                        // width of a pow row: W, or N for one-sided rows
    bool onesided = false;             // ZFB_FLAG_ONESIDED
    double sum_w2 = 0.0;
    int group = 1, group_user = 0;
    int nsplit_cap = 1;
    StageParams sp0[3]{};              // LO tables of stage 0 for NT = 256 / 128 / 64 (strips)

    DevBuf cvt;                        // complex64 copy of an int16 IQ launch group (ZFB_DTYPE_CS16)
    DevBuf window, winfft, winfft16, wf_sparse, twiddle, twiddle_sub, pow16, mid[2], pow, rows_tmp, ema, ring, stage_in[2], big, img_out, img_lut, img_thr, sel_hist;
    void  *h_stage[2] = {nullptr, nullptr};
    size_t h_stage_cap[2] = {0, 0};
    float *h_rows = nullptr;
    size_t h_rows_cap = 0;
    int ring_rows = 256, ring_rows_req = 256, ring_W = 0;
    int ring_user_W = 0;               // zfb_ring_configure_width: the ring keeps this width whatever is configured
    // geometry of the last successful configure (ring / EMA validity): W, N, R, onesided
    bool geom_valid = false;
    int geom[4] = {0, 0, 0, 0};
    int64_t ring_written = 0;
    int last_group_frames = 0;
    bool thr_valid = false;            // img_thr holds the level thresholds of thr_levels
    double thr_levels[2] = {0.0, 0.0};
    bool ema_have = false;             // the EMA state holds a row (host side; launch order = stream order)
    // trace set (zfb_traces_enable; zfb_trace.cuh): nothing is allocated or launched while it is off
    bool traces_on = false;
    int64_t trace_count = 0;           // rows in the traces (host side; launch order = stream order)
    double trace_key[6] = {0, 0, 0, 0, 0, 0};   // fs, N, R, row_width, f_demod, flags of the last configure
    DevBuf trace;                      // [W] fp64 sums, then LAST, MAX, MIN, AVG read-out [4][W] float
    DevBuf trace_rows;                 // [group][W] rows of a launch group the caller did not ask for
    DevBuf peaks;                      // PeakOut, then one flag byte per element

    // ZFB_MODE_FAST
    struct FastPlan {
        bool set = false;
        int ne = 0;                                   // FIR stages
        int M[ZFB_FAST_MAX_STAGES] = {0};
        float h[ZFB_FAST_MAX_STAGES][FIR_MAX_HALF + 1] = {{0}};
        int Mc = -1;
        float hc[FIR_COMP_MAX_HALF + 1] = {0};
        int K = 128;
    } fplan;
    bool fast_active = false;
    int nchains = 0;
    FirChainParams chain[4]{};
    int chain_level_out[4] = {0};      // decimation level (stage count) after chain j
    size_t chain_smem[4] = {0};
    int chain_run[4] = {0};            // 0: generic kernel; 1..3: fir_run_kernel with NS = that
    FirRunParams runp[4]{};
    int strip_len[kMaxStages] = {0};   // i_s: samples per strip at the input of stage s
    int strip_q[kMaxStages] = {0};     // Q_s: absolute position of the right strip's first sample
    int strip_cap = 0;
    DevBuf sbuf[2];
    int final_buf = 0;                 // mid[] index holding the decimated chunk of the last group
    // channel-batched launch in flight (zfb_process_channels_*): 0 = off
    int cur_nch = 0, cur_chan_frames = 0;
    long long cur_row_stride = 0;
    DevBuf chan_dev;
    std::vector<ChannelLo> chan_host;

    // pinned sample ring + double-buffered device mirror
    void   *sr_host = nullptr;
    DevBuf  sr_dev[2];
    int64_t sr_cap = 0;
    int     sr_dtype = 0;
    int     sr_active = 0;               // mirror the producer currently fills
    cudaEvent_t sr_copied = nullptr;     // last H2D enqueued on the copy stream
    cudaEvent_t sr_free[2] = {nullptr, nullptr};   // compute finished reading mirror i
    bool    sr_free_pending[2] = {false, false};
    bool    sr_copy_pending = false;

    uint64_t counters[5] = {0, 0, 0, 0, 0};

    // optional per-kernel timing
    struct ProfRec { cudaEvent_t a, b; int cls; };
    bool profiling = false;
    std::vector<ProfRec> prof_used, prof_free;
};

namespace {

}  // namespace

namespace zfb {
#ifdef ZFB_EMULATE
int make_tensor_map(const TensorMapSpec &spec, TensorMap *out) {
    out->base = (unsigned char *)spec.base;
    for (int i = 0; i < 4; ++i) {
        out->dim[i] = spec.dim[i];
        out->stride[i] = spec.stride[i];
        out->box[i] = spec.box[i];
    }
    out->stride[0] = 8;
    out->swizzle = spec.swizzle;
    return 0;
}
#else
int make_tensor_map(const TensorMapSpec &spec, TensorMap *out) {
    typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                 const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                 CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess || !fn) {
            cudaGetLastError();
            return -1;
        }
        encode = (EncodeFn)fn;
    }
    cuuint64_t dim[4], stride[3];
    cuuint32_t box[4], estr[4] = {1, 1, 1, 1};
    for (int i = 0; i < 4; ++i) {
        dim[i] = spec.dim[i];
        box[i] = spec.box[i];
    }
    for (int i = 0; i < 3; ++i) stride[i] = spec.stride[i + 1];
    const CUtensorMapSwizzle sw = spec.swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : spec.swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
    const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, spec.base, dim, stride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -1;
}
#endif
}  // namespace zfb

namespace {

int fail(zfb_engine *e, int code, const char *fmt, ...) __attribute__((format(printf, 3, 4)));
int fail(zfb_engine *e, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->err = buf; else g_create_error = buf;
    return code;
}

#define CK(e, call)                                                                     \
    do {                                                                                \
        cudaError_t _st = (call);                                                       \
        if (_st != cudaSuccess)                                                         \
            return fail(e, ZFB_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), \
                        __FILE__, __LINE__);                                            \
    } while (0)

int ensure(zfb_engine *e, DevBuf &b, size_t need) {
    if (need <= b.cap && b.p) return ZFB_OK;
    if (b.p) {
        CK(e, cudaStreamSynchronize(e->stream));
        CK(e, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t cap = need < 256 ? 256 : need;
    cudaError_t st = cudaMalloc(&b.p, cap);
    if (st != cudaSuccess) {
        b.p = nullptr;
        return fail(e, ZFB_ENOMEM, "cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(st));
    }
    b.cap = cap;
    return ZFB_OK;
}

void release(DevBuf &b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

// ---- the reference's decimation filter --------------------------------------
// scipy.signal.cheby1(8, 0.05, 0.8/2, output='sos') (scipy:_signaltools.py:
// 5317-5319), designed here from the closed form: analog Chebyshev-I
// prototype, pre-warped low-pass transform, bilinear transform; conjugate pole
// pairs become sections ordered by pole radius (sharpest last) and the whole
// gain sits in the first section, as scipy's zpk2sos does for this filter.
void design_cheby1_sos(double sos[NSEC][6]) {
    const int n = 2 * NSEC;
    const double rp = 0.05, wn = 0.4;
    const double eps = sqrt(pow(10.0, 0.1 * rp) - 1.0);
    const double mu = asinh(1.0 / eps) / n;
    const double fs2 = 4.0;                              // 2*fs with fs = 2
    const double warped = fs2 * tan(kPi * wn / 2.0);
    double pre[NSEC], pim[NSEC];                         // upper-half-plane analog poles
    double kre = 1.0, kim = 0.0;                         // prod(-p) over all poles
    for (int k = 0; k < NSEC; ++k) {
        const double theta = kPi * (2.0 * (k + 1) - 1.0) / (2.0 * n);
        pre[k] = -sinh(mu) * sin(theta) * warped;
        pim[k] = cosh(mu) * cos(theta) * warped;
        const double m2 = pre[k] * pre[k] + pim[k] * pim[k];   // (-p)(-conj p)
        kre *= m2;
    }
    (void)kim;
    double gain = kre / sqrt(1.0 + eps * eps);           // even order: ripple at DC
    // bilinear: z = (fs2 + s)/(fs2 - s); gain *= real(prod(fs2 - z_analog)/prod(fs2 - p))
    // (no finite analog zeros: numerator product is 1; n zeros land at z = -1)
    double zr[NSEC], zi_[NSEC], rad[NSEC];
    for (int k = 0; k < NSEC; ++k) {
        const double dr = fs2 - pre[k], di = -pim[k];
        const double d2 = dr * dr + di * di;
        gain /= d2;                                      // (fs2-p)(fs2-conj p) = |fs2-p|^2
        const double nr = fs2 + pre[k], ni = pim[k];
        zr[k] = (nr * dr + ni * di) / d2;
        zi_[k] = (ni * dr - nr * di) / d2;
        rad[k] = sqrt(zr[k] * zr[k] + zi_[k] * zi_[k]);
    }
    int order[NSEC];
    for (int k = 0; k < NSEC; ++k) order[k] = k;
    for (int a = 0; a < NSEC; ++a)
        for (int b = a + 1; b < NSEC; ++b)
            if (rad[order[b]] < rad[order[a]]) { int t = order[a]; order[a] = order[b]; order[b] = t; }
    for (int s = 0; s < NSEC; ++s) {
        const int k = order[s];
        const double b0 = (s == 0) ? gain : 1.0;
        sos[s][0] = b0;
        sos[s][1] = 2.0 * b0;
        sos[s][2] = b0;
        sos[s][3] = 1.0;
        sos[s][4] = -2.0 * zr[k];
        sos[s][5] = rad[k] * rad[k];
    }
}

void mat_mul(const double a[NSTATE][NSTATE], const double b[NSTATE][NSTATE], double out[NSTATE][NSTATE]) {
    double t[NSTATE][NSTATE];
    for (int i = 0; i < NSTATE; ++i)
        for (int j = 0; j < NSTATE; ++j) {
            double s = 0.0;
            for (int k = 0; k < NSTATE; ++k) s += a[i][k] * b[k][j];
            t[i][j] = s;
        }
    memcpy(out, t, sizeof t);
}

// constants of the block-parallel IIR (zfb_decim.cuh): -a1, -a2, the squared
// gain (forward and backward pass folded into one input scale), the steady
// state of the all-pole cascade per unit (scaled) input, and powers of its
// zero-input state transition over one BLK-sample run.
static void compute_decim_const(DecimConst &dc) {
    double sos[NSEC][6];
    design_cheby1_sos(sos);
    double a1[NSEC], a2[NSEC];
    for (int k = 0; k < NSEC; ++k) {
        a1[k] = sos[k][4];
        a2[k] = sos[k][5];
        dc.na1[k] = (float)(-a1[k]);
        dc.na2[k] = (float)(-a2[k]);
    }
    dc.g = (float)(sos[0][0] * sos[0][0]);
    double c = 1.0;
    for (int k = 0; k < NSEC; ++k) {
        c /= (1.0 + a1[k] + a2[k]);       // all-pole section: constant in -> constant out
        dc.zi[k] = (float)c;
    }
    // one-sample zero-input transition A of the DF2 cascade, state order
    // (w1_0, w2_0, w1_1, w2_1, ...): column j = response to unit state j
    double A[NSTATE][NSTATE];
    for (int j = 0; j < NSTATE; ++j) {
        double w1[NSEC], w2[NSEC];
        for (int k = 0; k < NSEC; ++k) {
            w1[k] = (j == 2 * k) ? 1.0 : 0.0;
            w2[k] = (j == 2 * k + 1) ? 1.0 : 0.0;
        }
        double v = 0.0;
        for (int k = 0; k < NSEC; ++k) {
            const double w = v - a1[k] * w1[k] - a2[k] * w2[k];
            v = w;                              // all-pole cascade (zfb_decim.cuh)
            w2[k] = w1[k];
            w1[k] = w;
        }
        for (int k = 0; k < NSEC; ++k) {
            A[2 * k][j] = w1[k];
            A[2 * k + 1][j] = w2[k];
        }
    }
    for (int variant = 0; variant < 2; ++variant) {
        const int run = variant == 0 ? BLK : 32;
        const int terms = variant == 0 ? JTERMS : JTERMS32;
        double M[NSTATE][NSTATE];
        memcpy(M, A, sizeof M);
        for (int i = 1; i < run; i <<= 1) mat_mul(M, M, M);   // run lengths are powers of two
        double P[NSTATE][NSTATE];
        for (int i = 0; i < NSTATE; ++i)
            for (int j = 0; j < NSTATE; ++j) P[i][j] = (i == j) ? 1.0 : 0.0;
        for (int j = 0; j < terms; ++j) {
            for (int r = 0; r < NSTATE; ++r)
                for (int cc = 0; cc < NSTATE; ++cc)
                    (variant == 0 ? dc.Mp[j][r][cc] : dc.Mp32[j][r][cc]) = (float)P[r][cc];
            mat_mul(M, P, P);
        }
    }
    // Partial fractions of the zero-phase response (zfb_iirstream.cuh):
    // H(z)H(1/z) = G(z) + G(1/z), G(z) = Bc(z) / prod A_k(z).  G's impulse response is the
    // autocorrelation of H's (halved at lag 0); multiplying by the denominator leaves Bc.
    {
        const int n = 8192;                               // 0.935^8192: far below double precision
        std::vector<double> h((size_t)n, 0.0);
        {
            double w1[NSEC] = {0}, w2[NSEC] = {0};
            for (int i = 0; i < n; ++i) {
                double v = (i == 0) ? 1.0 : 0.0;
                for (int k = 0; k < NSEC; ++k) {          // direct form II section of the sos
                    const double w = v - sos[k][4] * w1[k] - sos[k][5] * w2[k];
                    v = sos[k][0] * w + sos[k][1] * w1[k] + sos[k][2] * w2[k];
                    w2[k] = w1[k];
                    w1[k] = w;
                }
                h[(size_t)i] = v;
            }
        }
        double gimp[9];
        for (int lag = 0; lag < 9; ++lag) {
            double acc = 0.0;
            for (int i = 0; i + lag < n; ++i) acc += h[(size_t)i] * h[(size_t)(i + lag)];
            gimp[lag] = acc;
        }
        gimp[0] *= 0.5;
        double A[2 * NSEC + 1] = {1.0};
        int deg = 0;
        for (int k = 0; k < NSEC; ++k) {
            double nxt[2 * NSEC + 1] = {0};
            for (int i = 0; i <= deg; ++i) {
                nxt[i] += A[i];
                nxt[i + 1] += A[i] * a1[k];
                nxt[i + 2] += A[i] * a2[k];
            }
            deg += 2;
            memcpy(A, nxt, sizeof A);
        }
        for (int i = 0; i < 9; ++i) {
            double acc = 0.0;
            for (int k = 0; k <= i; ++k) acc += gimp[k] * A[i - k];
            dc.bc[i] = (float)acc;
        }
    }
}

// The constants depend on nothing but the filter: computed once per process (the partial-fraction
// part runs an 8192-sample impulse response -- per-call it cost a virtual-receiver step of 8
// channels 1.4 ms of host time against 0.74 ms of kernels, profiles/r02w_bench_cfg4_8gpu.json)
void build_decim_const(DecimConst &dc) {
    static const DecimConst cached = [] {
        DecimConst d;
        compute_decim_const(d);
        return d;
    }();
    dc = cached;
}

// in-place radix-2 FFT in double (host; window spectra only)
void host_fft(std::vector<double> &re, std::vector<double> &im) {
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const size_t half = len >> 1;
        for (size_t k = 0; k < half; ++k) {
            const double a = -2.0 * kPi * (double)k / (double)len;
            const double wr = cos(a), wi = sin(a);
            for (size_t i = k; i < n; i += len) {
                const size_t j2 = i + half;
                const double xr = re[j2] * wr - im[j2] * wi, xi = re[j2] * wi + im[j2] * wr;
                re[j2] = re[i] - xr; im[j2] = im[i] - xi;
                re[i] += xr; im[i] += xi;
            }
        }
    }
}

// engine-owned intermediates: frames start on 32-byte boundaries (bulk copies need 16)
long long stride4(long long n) { return (n + 3) & ~3LL; }

int ilog2_floor(long long v) {
    int l = -1;
    while (v > 0) { v >>= 1; ++l; }
    return l;
}

struct Geometry {
    int nstages, ndec, nperseg, hop, nseg;
    int len[kMaxStages + 1];
};

// lengths the reference produces: decimate keeps y[::2] (ceil), needs len > 27
// (scipy:_signaltools.py:4944-4947); welch: nperseg = min(N, n), noverlap =
// nperseg//2, nseg = (n - noverlap)//hop (scipy:_spectral_py.py:897-912,932-937)
int geometry(int frame_len, int fft_size, int fft_ratio, Geometry &g) {
    if (frame_len < 1 || fft_size < 1 || fft_ratio < 1) return ZFB_EINVAL;
    g.nstages = ilog2_floor(fft_ratio);                  // int(np.log2(ratio)), S:2096
    if (g.nstages > kMaxStages) return ZFB_EINVAL;
    int L = frame_len;
    for (int s = 0; s < g.nstages; ++s) {
        g.len[s] = L;
        if (L <= PADLEN) return ZFB_ETOOSHORT;
        L = (L + 1) / 2;
    }
    g.len[g.nstages] = L;
    g.ndec = L;
    g.nperseg = fft_size < L ? fft_size : L;
    const int noverlap = g.nperseg / 2;
    g.hop = g.nperseg - noverlap;
    g.nseg = (L - noverlap) / g.hop;
    return ZFB_OK;
}

// exp(-2 pi i * frac(r * m)) in double, with the product reduced exactly
void lo_entry(double r, long long m, double amp, float2 &out) {
    // r in [0,1); r*m may be large: split m to keep the fractional part accurate
    long double ph = (long double)r * (long double)m;
    ph -= floorl(ph);
    const double a = -2.0 * kPi * (double)ph;
    out.x = (float)(amp * cos(a));
    out.y = (float)(amp * sin(a));
}

// ---- kernel tables ------------------------------------------------------------
typedef void (*WelchFn)(const WelchParams);
struct WelchEntry { WelchFn fn; int threads; size_t smem; };

// prune: 0 = every bin accumulated; 1 = only the bins of the thread that can fall inside the kept
// W columns (KEEP per spectrum end, welch_kernel); 2 = the same at 3 CTAs/SM where that fits
template <int LOG2N, int KIND>
WelchEntry welch_entry(int keep, int prune) {
#ifndef ZFB_WELCH_PPT16_FROM
#define ZFB_WELCH_PPT16_FROM 11
#endif
    // 16 points per thread from N = 2048 up: half the threads per barrier, twice the ILP
    constexpr int PPT = (LOG2N >= ZFB_WELCH_PPT16_FROM) ? 16 : 8;
    using S = WelchShape<LOG2N, PPT>;
    if constexpr (PPT == 16 && KIND == KIND_C64_MID) {
        if (prune >= 1) {
            if constexpr (S::NTHREADS <= 256) {
                if (prune >= 2 && keep <= 1) return WelchEntry{welch_kernel<LOG2N, PPT, KIND, 1, true>, S::NTHREADS, S::SMEM};
                if (prune >= 2 && keep <= 2) return WelchEntry{welch_kernel<LOG2N, PPT, KIND, 2, true>, S::NTHREADS, S::SMEM};
            }
            if (keep <= 1) return WelchEntry{welch_kernel<LOG2N, PPT, KIND, 1>, S::NTHREADS, S::SMEM};
            if (keep <= 2) return WelchEntry{welch_kernel<LOG2N, PPT, KIND, 2>, S::NTHREADS, S::SMEM};
            if (keep <= 4) return WelchEntry{welch_kernel<LOG2N, PPT, KIND, 4>, S::NTHREADS, S::SMEM};
        }
    }
    return WelchEntry{welch_kernel<LOG2N, PPT, KIND>, S::NTHREADS, S::SMEM};
}

template <int KIND>
WelchEntry welch_lookup_kind(int log2n, int keep, int prune) {
    switch (log2n) {
        case 5: return welch_entry<5, KIND>(keep, prune);
        case 6: return welch_entry<6, KIND>(keep, prune);
        case 7: return welch_entry<7, KIND>(keep, prune);
        case 8: return welch_entry<8, KIND>(keep, prune);
        case 9: return welch_entry<9, KIND>(keep, prune);
        case 10: return welch_entry<10, KIND>(keep, prune);
        case 11: return welch_entry<11, KIND>(keep, prune);
        case 12: return welch_entry<12, KIND>(keep, prune);
        case 13: return welch_entry<13, KIND>(keep, prune);
        default: return WelchEntry{nullptr, 0, 0};
    }
}

// keep: bins per spectrum end and thread that can be kept (16 = all); see welch_keep()
WelchEntry welch_lookup(int log2n, int kind, int keep = 16, int prune = 0) {
    switch (kind) {
        case KIND_C64_RAW: return welch_lookup_kind<KIND_C64_RAW>(log2n, keep, prune);
        case KIND_U8_RAW: return welch_lookup_kind<KIND_U8_RAW>(log2n, keep, prune);
        default: return welch_lookup_kind<KIND_C64_MID>(log2n, keep, prune);
    }
}

// bins k = tid + m*NT of a thread that can fall inside the kept columns [0, W/2) u [N - W/2, N):
// m < keep or m >= PPT - keep
int welch_keep(int log2n, int W) {
    const int ppt = (log2n >= ZFB_WELCH_PPT16_FROM) ? 16 : 8;
    const int nt = (1 << log2n) / ppt;
    const int k = ((W + 1) / 2 + nt - 1) / nt;
    return k < 1 ? 1 : k;
}

typedef void (*DecimFn)(const StageParams);
template <int NT>
DecimFn decim_lookup_nt(int kind) {
    switch (kind) {
        case KIND_C64_RAW: return decim2_exact_kernel<KIND_C64_RAW, NT>;
        case KIND_U8_RAW: return decim2_exact_kernel<KIND_U8_RAW, NT>;
        default: return decim2_exact_kernel<KIND_C64_MID, NT>;
    }
}
DecimFn decim_lookup(int kind, int nt) {
    return nt == NTHR_BIG ? decim_lookup_nt<NTHR_BIG>(kind) : decim_lookup_nt<NTHR_SMALL>(kind);
}

constexpr size_t decim_smem(int nt) { return (size_t)(nt * BLK_PAD + NSTATE * nt) * sizeof(float2); }

typedef void (*ChainFn0)(const FirChainParams);
ChainFn0 chain_lookup_fn(int kind) {
    switch (kind) {
        case KIND_C64_RAW: return fir_chain_kernel<KIND_C64_RAW>;
        case KIND_U8_RAW: return fir_chain_kernel<KIND_U8_RAW>;
        default: return fir_chain_kernel<KIND_C64_MID>;
    }
}

template <int KIND> int fir_run_setup_kind(zfb_engine *e);
int fir_run_setup_cs16(zfb_engine *e);
constexpr int kIirNS = 3, kIirNO = 3;      // x pieces / output rows in flight per lane (zfb_iirstream.cuh)

int setup_device_once(zfb_engine *e) {
    DecimConst dc;
    build_decim_const(dc);
    CK(e, cudaMemcpyToSymbol(c_dec, &dc, sizeof dc));
    {   // fp64 path: scipy's sos and sosfilt_zi (steady DF2T state per unit input, cascaded gains)
        PreciseConst pc;
        design_cheby1_sos(pc.sos);
        for (int k = 0; k < NSEC; ++k) {          // per unit input of the section; the kernel cascades the gains
            const double *b = pc.sos[k], *a = pc.sos[k] + 3;
            const double G = (b[0] + b[1] + b[2]) / (a[0] + a[1] + a[2]);
            const double z2 = b[2] - a[2] * G;
            pc.zi[k][0] = b[1] - a[1] * G + z2;
            pc.zi[k][1] = z2;
        }
        CK(e, cudaMemcpyToSymbol(c_px, &pc, sizeof pc));
    }
    for (int kind = 0; kind < 3; ++kind)
        for (int nt : {NTHR_BIG, NTHR_SMALL})
            CK(e, cudaFuncSetAttribute(decim_lookup(kind, nt), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)decim_smem(nt)));
    for (int kind = 0; kind < 3; ++kind)
        for (int l = kMinLog2N; l <= kMaxLog2Small; ++l) {
            for (int variant = 0; variant < 12; ++variant) {      // every (keep, prune) the lookup can return
                WelchEntry w = welch_lookup(l, kind, 1 << (variant & 3), variant >> 2);
                if (w.smem > 48 * 1024)
                    CK(e, cudaFuncSetAttribute(w.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.smem));
                if (l >= 11)   // N >= 2048: room for several CTAs' exchange buffers; small N keeps its L1
                    CK(e, cudaFuncSetAttribute(w.fn, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            }
        }
    CK(e, cudaFuncSetAttribute(strip_cascade_kernel<KIND_U8_RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem()));
    CK(e, cudaFuncSetAttribute(strip_cascade_kernel<KIND_C64_RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem()));
    CK(e, cudaFuncSetAttribute(strip_cascade_kernel<KIND_C64_MID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem()));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_C64_MID, false, 64>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(64)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_U8_RAW, false, 64>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(64)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_C64_RAW, false, 64>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(64)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_U8_RAW, true, 64>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(64)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_C64_RAW, true, 64>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(64)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_C64_MID, false, 32>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem(32)));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_U8_RAW, true>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem()));
    CK(e, cudaFuncSetAttribute((strip_cascade_kernel<KIND_C64_RAW, true>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)strip_smem()));
    for (int kind = 0; kind < 3; ++kind)
        CK(e, cudaFuncSetAttribute(chain_lookup_fn(kind), cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    CK(e, cudaFuncSetAttribute((iir_stream_kernel<kIirNS, kIirNO>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)IirStreamShape<kIirNS, kIirNO>::SMEM));
    int rc = fir_run_setup_kind<KIND_C64_RAW>(e);
    if (rc == ZFB_OK) rc = fir_run_setup_kind<KIND_U8_RAW>(e);
    if (rc == ZFB_OK) rc = fir_run_setup_kind<KIND_C64_MID>(e);
    if (rc == ZFB_OK) rc = fir_run_setup_cs16(e);
    return rc;
}

// kind of the samples the kernels see (int16 IQ has been widened to complex64 by then)
int raw_kind(const zfb_config &c) { return c.dtype == ZFB_DTYPE_U8 ? KIND_U8_RAW : KIND_C64_RAW; }
size_t dtype_bytes(int dtype) { return dtype == ZFB_DTYPE_U8 ? 2 : dtype == ZFB_DTYPE_CS16 ? 4 : 8; }
// bytes per sample on the wire (caller's buffers, staging, sample ring)
size_t sample_bytes(const zfb_config &c) { return dtype_bytes(c.dtype); }

// SoapySDR CS16 -> complex64, (I + jQ) / 32768: one coalesced streaming pass (4 B in, 8 B out
// per sample) in front of the complex64 path
__global__ void __launch_bounds__(256) cs16_to_c64_kernel(const unsigned int *in, float2 *out, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned int w = in[i];                       // little endian: I in the low half
        const float fi = (float)(short)(w & 0xffffu), fq = (float)(short)(w >> 16);
        out[i] = make_float2(fi * (1.0f / 32768.0f), fq * (1.0f / 32768.0f));
    }
}

// the same for the first and last `ends` samples of every frame only (the exact edge strips of mode
// fast read nothing else when the FIR interior converts its own input)
__global__ void __launch_bounds__(256) cs16_ends_to_c64_kernel(const unsigned int *in, float2 *out, int frame_len, int ends,
                                                               long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long f = i / (2 * ends);
    const int j = (int)(i % (2 * ends));
    const long long at = f * frame_len + (j < ends ? j : frame_len - 2 * ends + j);
    const unsigned int w = in[at];
    out[at] = make_float2((float)(short)(w & 0xffffu) * (1.0f / 32768.0f), (float)(short)(w >> 16) * (1.0f / 32768.0f));
}

// FAST engages when the plan fits and the chunk is long enough for the strips
bool fast_wanted(const zfb_engine *e, int *strip_len, int *strip_q) {
    const zfb_config &c = e->cfg;
    const int k = e->nstages;
    if (c.mode != ZFB_MODE_FAST || k < 2 || !e->fplan.set || e->fplan.ne != k - 1) return false;
    // strips: i_{k-1} = 2K + D, i_s = 2 i_{s+1} + D, right strip starts at an even position
    const int K = e->fplan.K;
    // decay distance of a strip's artificial inner edge: 0.935^D of that edge's transient is left
    // where the strip's outputs are used (320: 5e-10, 256: 3e-8, 192: 2.5e-6 = 2e-5 dB)
    // The transient of stage s's cut reaches the K outputs only through the decay zones of ALL the
    // later stages (it sits at the inner end of stage s+1's strip, D_(s+1) samples from what that
    // stage must get right, and so on): what counts is the sum of the distances from s on.  The
    // last stage carries the full distance, the earlier ones a short one.
    const int D = e->strip_decay, De = e->strip_decay_early < D ? e->strip_decay_early : D;
    int need = 2 * K + D;
    for (int s = k - 1; s >= 0; --s) {
        int i = need;
        if ((e->len[s] - i) & 1) i += 1;
        strip_len[s] = i;
        strip_q[s] = e->len[s] - i;
        need = 2 * i + De;
    }
    return e->len[0] >= 4 * strip_len[0] && e->len[k] >= 4 * K;
}

// chains of FAST: sizes from the back (the last chain takes up to 3 stages)
int fast_chain_sizes(int ne, int sizes[4]) {
    int n = 0, done = 0;
    while (done < ne && n < 4) {
        int ns = (ne - done) % FIR_MAX_STAGES;
        if (ns == 0) ns = FIR_MAX_STAGES;
        sizes[n++] = ns;
        done += ns;
    }
    return done == ne ? n : -1;
}

// frame strides of mode fast's intermediates: the streaming last stage reads whole streams
// (its input frames span nspf*S >= L samples) and stores whole streams of results
long long fast_level_stride(const zfb_engine *e, int lvl) {
    if (e->iis.active && lvl == e->nstages - 1) return e->iis.in_stride;
    return stride4(e->len[lvl]);
}
long long final_stride(const zfb_engine *e) {
    if (e->fast_active && e->iis.active) return e->iis.out_stride;
    return stride4(e->len[e->nstages]);
}

// capacity (samples per frame) the two ping-pong buffers need in the active mode
void mid_lengths(const zfb_engine *e, bool fast, long long need[2]) {
    need[0] = need[1] = 0;
    int b = 0;
    auto put = [&](long long len) { len = stride4(len); if (len > need[b]) need[b] = len; b ^= 1; };
    const int k = e->nstages;
    if (fast) {
        int sizes[4];
        const int n = fast_chain_sizes(k - 1, sizes);
        int lvl = 0;
        for (int j = 0; j < n; ++j) { lvl += sizes[j]; put(fast_level_stride(e, lvl)); }
        put(final_stride(e));
    } else {
        for (int s = 0; s < k; ++s) put(e->len[s + 1]);
    }
}

int choose_group(const zfb_engine *e, bool fast) {
    if (e->group_user > 0) return e->group_user;
    // enough frames per launch that the late, small stages still fill the GPU
    // (the chain is fp32-bound, not bandwidth-bound: L2 residency of the
    // intermediates is worth less than full waves); bounded to 512 MB of workspace
    long long need[2];
    mid_lengths(e, fast, need);
    size_t per_frame = (size_t)(need[0] + need[1]) * 8;
    size_t budget = 512ull << 20;       // (256 MB cut cfg1's 512 frames into 352 + 160: 155 -> 161 Gs/s with one group, r02s)
    if (e->log2N > kMaxLog2Small) {
        per_frame += (size_t)e->nseg * ((size_t)8 << e->log2N);       // four-step scratch
        budget = (e->log2N >= kMinLog2R16 && e->log2N <= kMaxLog2R16) ? (1100ull << 20) : (512ull << 20);
    }
    if (per_frame == 0) return 2048;
    long long g = (long long)budget / (long long)per_frame;
    if (g < 1) g = 1;
    if (g > 1024) g = 1024;
    if (g > 32) g -= g % 32;              // typical batches (powers of two) split into equal groups
    return (int)g;
}

// tile geometry per stage for both region sizes; run_group picks per launch
void plan_tiles(zfb_engine *e) {
    for (int s = 0; s < e->nstages; ++s)
        for (int v = 0; v < 2; ++v) {
            const int L = e->len[s];
            const int tmax = tmax_of(v == 0 ? NTHR_BIG : NTHR_SMALL);
            const int tiles = (L + tmax - 1) / tmax;
            int T = (L + tiles - 1) / tiles;
            T = (T + 15) / 16 * 16;
            e->tiles[s][v] = (L + T - 1) / T;
            e->T[s][v] = T;
        }
}

constexpr size_t kMaxProfRecs = 1 << 16;

// returns the index of the open record, or -1 when profiling is off
int prof_begin(zfb_engine *e, int cls, cudaStream_t on = nullptr) {
    if (!e->profiling || e->prof_used.size() >= kMaxProfRecs) return -1;
    zfb_engine::ProfRec r;
    if (!e->prof_free.empty()) {
        r = e->prof_free.back();
        e->prof_free.pop_back();
    } else {
        if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return -1;
    }
    r.cls = cls;
    cudaEventRecord(r.a, on ? on : e->stream);
    e->prof_used.push_back(r);
    return (int)e->prof_used.size() - 1;
}

void prof_end(zfb_engine *e, int idx, cudaStream_t on = nullptr) {
    if (idx >= 0) cudaEventRecord(e->prof_used[(size_t)idx].b, on ? on : e->stream);
}

// the tap sets fastdesign.py produces for the last chain of R = 4 / 8 / >= 16
// ... and, without compensator (D = -1), for the light first chains of deeper
// zooms (every stage there has <= 7 taps; shorter ones are zero-padded)
#define ZFB_RUN_COMBOS(X, KIND) \
    X(1, KIND, 1, 13, 0, 0, 15)  \
    X(2, KIND, 2, 5, 13, 0, 16)  \
    X(3, KIND, 3, 4, 5, 13, 16)  \
    X(4, KIND, 1, 3, 0, 0, -1)   \
    X(5, KIND, 2, 3, 3, 0, -1)   \
    X(6, KIND, 3, 3, 3, 3, -1)

// 128-thread CTAs: 256 were slower (0.292 against 0.273 ms per 512 cfg2 frames, DESIGN §3.0)
template <int KIND>
void launch_fir_run_kind(int variant, const FirRunParams &rp, int L_out, int gf, cudaStream_t st) {
#define ZFB_X(ID, K, NS, A, B, C, D)                                                              \
    if (variant == ID) {                                                                          \
        using SH = FirRunShape<NS, A, B, C, D, 128>;                                              \
        const int per_tile = SH::SPAN >> NS;                                                      \
        const unsigned tiles = (unsigned)((L_out + per_tile - 1) / per_tile);                     \
        if (K != KIND_C64_MID && rp.chan) {                                                       \
            ZFB_LAUNCH((fir_run_kernel<K, NS, A, B, C, D, (K != KIND_C64_MID), 128>), dim3(tiles, (unsigned)gf), \
                       dim3(128), SH::SMEM, st, rp);                                              \
        } else {                                                                                  \
            ZFB_LAUNCH((fir_run_kernel<K, NS, A, B, C, D, false, 128>), dim3(tiles, (unsigned)gf), dim3(128), SH::SMEM, st, rp); \
        }                                                                                         \
        return;                                                                                   \
    }
    ZFB_RUN_COMBOS(ZFB_X, KIND)
#undef ZFB_X
}

// int16 IQ read by the kernel itself: 128-thread CTAs, no channel batch (fir_cs16_fused() decides)
void launch_fir_run_cs16(int variant, const FirRunParams &rp, int L_out, int gf, cudaStream_t st) {
#define ZFB_X(ID, K, NS, A, B, C, D)                                                              \
    if (variant == ID) {                                                                          \
        using SH = FirRunShape<NS, A, B, C, D, 128>;                                              \
        const int per_tile = SH::SPAN >> NS;                                                      \
        const unsigned tiles = (unsigned)((L_out + per_tile - 1) / per_tile);                     \
        ZFB_LAUNCH((fir_run_kernel<KIND_CS16_RAW, NS, A, B, C, D, false, 128>), dim3(tiles, (unsigned)gf), dim3(128), \
                   SH::SMEM, st, rp);                                                             \
        return;                                                                                   \
    }
    ZFB_RUN_COMBOS(ZFB_X, KIND_CS16_RAW)
#undef ZFB_X
}

void launch_fir_run(int variant, int kind, const FirRunParams &rp, int L_out, int gf, cudaStream_t st) {
    if (kind == KIND_CS16_RAW) launch_fir_run_cs16(variant, rp, L_out, gf, st);
    else if (kind == KIND_U8_RAW) launch_fir_run_kind<KIND_U8_RAW>(variant, rp, L_out, gf, st);
    else if (kind == KIND_C64_RAW) launch_fir_run_kind<KIND_C64_RAW>(variant, rp, L_out, gf, st);
    else launch_fir_run_kind<KIND_C64_MID>(variant, rp, L_out, gf, st);
}

// which specialised variant (0 = none) handles this chain
int fir_run_variant(const FirChainParams &p) {
    // exact tap sets with a compensator; "<=" (zero-padded taps) for the chains without
#define ZFB_X(ID, K, NS, A, B, C, D)                                                             \
    if (D >= 0 && p.ns == NS && p.Mc == D && p.M[0] == A && (NS < 2 || p.M[1] == B) && (NS < 3 || p.M[2] == C)) \
        return ID;                                                                               \
    if (D < 0 && p.ns == NS && p.Mc < 0 && p.M[0] <= A && (NS < 2 || p.M[1] <= B) && (NS < 3 || p.M[2] <= C)) \
        return ID;
    ZFB_RUN_COMBOS(ZFB_X, 0)
#undef ZFB_X
    return 0;
}

template <int KIND>
int fir_run_setup_kind(zfb_engine *e) {
#define ZFB_X(ID, K, NS, A, B, C, D)                                                              \
    CK(e, cudaFuncSetAttribute((fir_run_kernel<K, NS, A, B, C, D, false, 128>), cudaFuncAttributeMaxDynamicSharedMemorySize, \
                               (int)FirRunShape<NS, A, B, C, D, 128>::SMEM));                     \
    if (K != KIND_C64_MID) {                                                                      \
        CK(e, cudaFuncSetAttribute((fir_run_kernel<K, NS, A, B, C, D, (K != KIND_C64_MID), 128>), \
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FirRunShape<NS, A, B, C, D, 128>::SMEM)); \
    }
    ZFB_RUN_COMBOS(ZFB_X, KIND)
#undef ZFB_X
    return ZFB_OK;
}

int fir_run_setup_cs16(zfb_engine *e) {
#define ZFB_X(ID, K, NS, A, B, C, D)                                                              \
    CK(e, cudaFuncSetAttribute((fir_run_kernel<KIND_CS16_RAW, NS, A, B, C, D, false, 128>),        \
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FirRunShape<NS, A, B, C, D, 128>::SMEM));
    ZFB_RUN_COMBOS(ZFB_X, KIND_CS16_RAW)
#undef ZFB_X
    return ZFB_OK;
}

typedef void (*ChainFn)(const FirChainParams);
ChainFn chain_lookup(int kind) {
    switch (kind) {
        case KIND_C64_RAW: return fir_chain_kernel<KIND_C64_RAW>;
        case KIND_U8_RAW: return fir_chain_kernel<KIND_U8_RAW>;
        default: return fir_chain_kernel<KIND_C64_MID>;
    }
}

// streaming IIR stage: one warp per CTA, 32 streams per warp
void launch_iir_stream(zfb_engine *e, int gf, cudaStream_t st) {
    const zfb_engine::IirStreamPlan &pl = e->iis;
    const unsigned ctas = (unsigned)(gf * pl.q.groups);
    ZFB_LAUNCH((iir_stream_kernel<kIirNS, kIirNO>), dim3(ctas), dim3(32), (IirStreamShape<kIirNS, kIirNO>::SMEM), st,
               pl.tm_in, pl.tm_out, pl.q);
}

// the K samples at either end of every decimated chunk, computed by the exact edge strips into
// strip_out[frame][side][K], overwrite what the streaming last stage left there
__global__ void __launch_bounds__(256) strip_patch_kernel(const float2 *strip_out, float2 *out, long long out_stride,
                                                          int ndec, int K, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int j = (int)(i % (2 * K));
    const long long f = i / (2 * K);
    const int m = j < K ? j : ndec - 2 * K + j;
    out[f * out_stride + m] = strip_out[i];
}

void launch_stage(zfb_engine *e, int kind, int v, const StageParams &p, unsigned tiles, unsigned ny, int cls) {
    const int nt = v == 0 ? NTHR_BIG : NTHR_SMALL;
    const int pr = prof_begin(e, cls);
    ZFB_LAUNCH(decim_lookup(kind, nt), dim3(tiles, ny), dim3((unsigned)nt), decim_smem(nt), e->stream, p);
    prof_end(e, pr);
    e->counters[2] += 1;
}

// ZFB_MODE_FAST: FIR chains + exact last stage over the whole frames, then the
// exact cascade on the two end strips of every frame; leaves the decimated
// chunks in mid[*out_buf]
// the fused tail (up to 4 stages) of the exact edge strips, one CTA per strip,
// writing the first / last K samples of the decimated chunks in `final_out`
template <int NT>
void launch_strip_mid(const StripParams &sp, dim3 grid, cudaStream_t st) {
    ZFB_LAUNCH((strip_cascade_kernel<KIND_C64_MID, false, NT>), grid, dim3(NT), strip_smem(NT), st, sp);
}

void launch_fused_strips(zfb_engine *e, const void *d_in, int gf, float2 *final_out, cudaStream_t st) {
    const zfb_config &c = e->cfg;
    const int k = e->nstages;
    const int kf = k < 4 ? k : 4;
    const int s0 = k - kf;
    const long long cap = e->strip_cap;
    const dim3 grid(2, (unsigned)gf);
    const int pr = prof_begin(e, 15, st);
    // the strips halve from stage to stage: consecutive stages that fit the same region size
    // share a launch, a narrower region starts a new one (strip_cascade_kernel)
    bool from_fused = false;            // the input was left by a fused launch (exactly the samples needed)
    for (int a = s0; a < k;) {
        // raw input (stage 0): LO tables exist for 128 and 64 threads; channel-batched launches keep 128
        int nt = !e->strip_split ? STRIP_NT : strip_threads_for(e->strip_len[a]);
        if (a == 0 && nt < 64) nt = 64;
        int b = a + 1;
        while (b < k && (!e->strip_split || strip_threads_for(e->strip_len[b]) == nt)) ++b;
        StripParams sp{};
        sp.st = e->sp0[nt == 64 ? 2 : 1];               // LO tables for this many threads per CTA
        sp.st.L = e->strip_len[a];
        sp.st.T = 0;
        sp.st.strips = 1;
        int skind;
        if (a == 0) {
            skind = raw_kind(c);
            sp.st.in = d_in;
            sp.st.in_stride = c.frame_len;
            sp.st.side_in_off = 0;
            sp.st.flip = c.flip;
            sp.st.pos_off = e->strip_q[0];
            sp.st.Lfull = c.frame_len;
        } else {
            skind = KIND_C64_MID;
            sp.st.in = e->sbuf[(a - 1) & 1].p;
            sp.st.in_stride = 2 * cap;
            sp.st.side_in_off = from_fused ? cap : cap + (e->strip_q[a] - e->strip_q[a - 1] / 2);
            sp.st.flip = 0;
            sp.st.pos_off = 0;
            sp.st.Lfull = sp.st.L;
        }
        sp.nstages = b - a;
        for (int s = a; s < b; ++s) sp.len[s - a] = e->strip_len[s];
        sp.last = (b == k) ? 1 : 0;
        sp.keep = e->fplan.K;
        if (e->iis.active) {
            // compact [frame][side][K]: patched into the chunks once the streaming last stage is done
            sp.out = (float2 *)e->strip_out.p;
            sp.out_stride = 2 * e->fplan.K;
            sp.ndec = 2 * e->fplan.K;
        } else {
            sp.out = final_out;
            sp.out_stride = final_stride(e);
            sp.ndec = e->len[k];
        }
        if (!sp.last) {
            sp.mid_out = (float2 *)e->sbuf[(b - 1) & 1].p;
            sp.mid_cap = cap;
            sp.next_len = e->strip_len[b];
        }
        if (e->cur_nch > 0 && a == 0) {
            sp.st.chan = (const ChannelLo *)e->chan_dev.p;
            sp.st.chan_frames = e->cur_chan_frames;
            if (skind == KIND_U8_RAW) {
                if (nt == 64) ZFB_LAUNCH((strip_cascade_kernel<KIND_U8_RAW, true, 64>), grid, dim3(64), strip_smem(64), st, sp);
                else ZFB_LAUNCH((strip_cascade_kernel<KIND_U8_RAW, true>), grid, dim3(STRIP_NT), strip_smem(), st, sp);
            } else {
                if (nt == 64) ZFB_LAUNCH((strip_cascade_kernel<KIND_C64_RAW, true, 64>), grid, dim3(64), strip_smem(64), st, sp);
                else ZFB_LAUNCH((strip_cascade_kernel<KIND_C64_RAW, true>), grid, dim3(STRIP_NT), strip_smem(), st, sp);
            }
        } else if (skind == KIND_U8_RAW) {
            if (nt == 64) ZFB_LAUNCH((strip_cascade_kernel<KIND_U8_RAW, false, 64>), grid, dim3(64), strip_smem(64), st, sp);
            else ZFB_LAUNCH(strip_cascade_kernel<KIND_U8_RAW>, grid, dim3(STRIP_NT), strip_smem(), st, sp);
        } else if (skind == KIND_C64_RAW) {
            if (nt == 64) ZFB_LAUNCH((strip_cascade_kernel<KIND_C64_RAW, false, 64>), grid, dim3(64), strip_smem(64), st, sp);
            else ZFB_LAUNCH(strip_cascade_kernel<KIND_C64_RAW>, grid, dim3(STRIP_NT), strip_smem(), st, sp);
        } else if (nt == 32) {
            launch_strip_mid<32>(sp, grid, st);
        } else if (nt == 64) {
            launch_strip_mid<64>(sp, grid, st);
        } else {
            launch_strip_mid<128>(sp, grid, st);
        }
        e->counters[2] += 1;
        from_fused = true;
        a = b;
    }
    prof_end(e, pr, st);
}

// ZFB_MODE_FAST: FIR chains + exact last stage over the whole frames, and the
// exact cascade on the two end strips of every frame; leaves the decimated
// chunks in mid[*out_buf].  Returns a CUDA status.
// d_in_cs16: the caller's int16 IQ when the first FIR chain reads it itself (fir_cs16_fused), else null;
// d_in is then a complex64 buffer that holds only the chunk ends the strips read
cudaError_t run_decimation_fast(zfb_engine *e, const void *d_in, int gf, int *out_buf, const void *d_in_cs16 = nullptr) {
    const zfb_config &c = e->cfg;
    cudaStream_t st = e->stream;
    const int k = e->nstages;
    const int kf = k < 4 ? k : 4;
    const int s0 = k - kf;
    const int b_final = e->nchains & 1;             // every chain flips the ping-pong buffer once
    float2 *final_out = (float2 *)e->mid[b_final].p;
    const int K = e->fplan.K;
    // Strips read only the raw input and own the first / last K decimated samples; the
    // interior owns the rest, so the two need no order between them: with k <= 4 the
    // strips go to a side stream and fill the SMs beside the FIR interior.  They are submitted
    // before the FIR chain, so their CTAs are dispatched first.
    const bool async_strips = e->strips_async && s0 == 0;
    cudaError_t err = cudaSuccess;
    if (async_strips) {
        if ((err = cudaEventRecord(e->ev_fork, st)) != cudaSuccess) return err;      // input ready, buffers free
        if ((err = cudaStreamWaitEvent(e->aux_stream, e->ev_fork, 0)) != cudaSuccess) return err;
        launch_fused_strips(e, d_in, gf, final_out, e->aux_stream);
        if ((err = cudaEventRecord(e->ev_join, e->aux_stream)) != cudaSuccess) return err;
    }
    const void *src = d_in_cs16 ? d_in_cs16 : d_in;
    long long src_stride = c.frame_len;
    int kind = d_in_cs16 ? KIND_CS16_RAW : raw_kind(c);
    int b = 0;
    for (int j = 0; j < e->nchains; ++j) {
        FirChainParams p = e->chain[j];
        const int lvl = e->chain_level_out[j];
        p.in = src;
        p.in_stride = src_stride;
        p.out = (float2 *)e->mid[b].p;
        p.out_stride = fast_level_stride(e, lvl);
        const int pr = prof_begin(e, j == 0 ? 0 : 1);
        if (e->chain_run[j]) {
            FirRunParams rp = e->runp[j];
            rp.in = p.in;
            rp.in_stride = p.in_stride;
            rp.out = p.out;
            rp.out_stride = p.out_stride;
            if (j == 0 && e->cur_nch > 0) {
                rp.chan = (const ChannelLo *)e->chan_dev.p;
                rp.chan_frames = e->cur_chan_frames;
            }
            launch_fir_run(e->chain_run[j], kind, rp, e->len[lvl], gf, st);
        } else {
            const unsigned tiles = (unsigned)((e->len[lvl] + p.TO - 1) / p.TO);
            ZFB_LAUNCH(chain_lookup(kind), dim3(tiles, (unsigned)gf), dim3(FIR_NT), e->chain_smem[j], st, p);
        }
        prof_end(e, pr);
        e->counters[2] += 1;
        src = p.out;
        src_stride = p.out_stride;
        kind = KIND_C64_MID;
        b ^= 1;
    }
    const int v = (e->decim_threads == NTHR_BIG) ? 0 : 1;
    {   // the last decimate call, exact, over the whole (FIR-filtered) chunk; it leaves the
        // K samples at either end to the strips
        const int s = k - 1;
        StageParams p = e->sp0[v];
        p.in = src;
        p.in_stride = src_stride;
        p.out = final_out;
        p.out_stride = final_stride(e);
        p.L = e->len[s];
        p.T = e->T[s][v];
        p.flip = 0;
        p.strips = 0;
        p.Lfull = p.L;
        p.w_lo[0] = p.w_lo[1] = K;
        p.w_hi[0] = p.w_hi[1] = e->len[k] - K;
        if (e->iis.active) {
            // streaming form (zfb_iirstream.cuh): LTI interior; the K outputs at either end, the
            // only ones the chunk-edge rules of this stage reach, are patched in from the strips.
            // The copy engine reads whole streams: keep [L, nspf*S) of every frame at zero.
            if (e->iis.tail > 0) {
                cudaError_t me = cudaMemset2DAsync((float2 *)const_cast<void *>(src) + p.L, (size_t)src_stride * sizeof(float2),
                                                   0, (size_t)e->iis.tail * sizeof(float2), (size_t)gf, st);
                if (me != cudaSuccess) return me;
            }
            const int pr = prof_begin(e, k - 1);
            launch_iir_stream(e, gf, st);
            prof_end(e, pr);
            e->counters[2] += 1;
        } else {
            launch_stage(e, KIND_C64_MID, v, p, (unsigned)e->tiles[s][v], (unsigned)gf, k - 1);
        }
    }
    *out_buf = b_final;
    auto patch = [&]() {
        if (!e->iis.active) return;
        const long long total = (long long)gf * 2 * K;
        ZFB_LAUNCH(strip_patch_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st,
                   (const float2 *)e->strip_out.p, final_out, final_stride(e), e->len[k], K, total);
        e->counters[2] += 1;
    };
    if (async_strips) {
        err = cudaStreamWaitEvent(st, e->ev_join, 0);
        patch();
        return err;
    }

    // deeper zooms: the first stages' strips are longer than one region and go through the
    // tiled kernel (on the main stream), then the fused tail
    const int tmax = tmax_of(v == 0 ? NTHR_BIG : NTHR_SMALL);
    const long long cap = e->strip_cap;
    for (int s = 0; s < s0; ++s) {
        StageParams p = e->sp0[v];
        const int L = e->strip_len[s];
        p.strips = 1;
        p.L = L;
        const int tiles = (L + tmax - 1) / tmax;
        int T = (L + tiles - 1) / tiles;
        T = (T + 15) / 16 * 16;
        p.T = T;
        if (s == 0) {
            p.in = d_in;
            p.in_stride = c.frame_len;
            p.side_in_off = 0;
            p.pos_off = e->strip_q[0];
            p.Lfull = c.frame_len;
            p.flip = c.flip;
        } else {
            p.in = e->sbuf[(s - 1) & 1].p;
            p.in_stride = 2 * cap;
            p.side_in_off = cap + (e->strip_q[s] - e->strip_q[s - 1] / 2);
            p.pos_off = 0;
            p.Lfull = L;
            p.flip = 0;
        }
        p.out = (float2 *)e->sbuf[s & 1].p;
        p.out_stride = 2 * cap;
        p.side_out_off = cap;
        p.w_lo[0] = p.w_lo[1] = 0;
        p.w_hi[0] = p.w_hi[1] = INT_MAX;
        launch_stage(e, s == 0 ? raw_kind(c) : KIND_C64_MID, v, p, (unsigned)((L + T - 1) / T),
                     (unsigned)(2 * gf), 15);
    }
    launch_fused_strips(e, d_in, gf, final_out, st);
    patch();
    return cudaSuccess;
}

// traces on: the rows of a launch group go to the caller's buffer or, without one, to this scratch
float *trace_rows_or(zfb_engine *e, float *d_rows) {
    return (d_rows || !e->traces_on || e->cur_nch > 0) ? d_rows : (float *)e->trace_rows.p;
}

// fold `nf` finished rows into the trace set, on the stream that finished them (after them)
int trace_update(zfb_engine *e, const float *rows, int nf, cudaStream_t st) {
    if (!e->traces_on || e->cur_nch > 0 || nf < 1) return ZFB_OK;
    const int W = e->W;
    TraceParams tp{};
    tp.rows = rows;
    tp.nframes = nf;
    tp.W = W;
    tp.linear = (e->cfg.flags & ZFB_FLAG_LINEAR) ? 1 : 0;
    tp.have = e->trace_count > 0 ? 1 : 0;
    tp.sum = (double *)e->trace.p;
    tp.last = (float *)(tp.sum + W);
    tp.mx = tp.last + W;
    tp.mn = tp.mx + W;
    const int pr = prof_begin(e, 18, st);
    ZFB_LAUNCH(trace_update_kernel, dim3((unsigned)((W + TR_COLS - 1) / TR_COLS)), dim3(TR_NT), 0, st, tp);
    prof_end(e, pr, st);
    e->counters[2] += 1;
    e->trace_count += nf;
    CK(e, cudaGetLastError());
    return ZFB_OK;
}

// fp64 path (zfb_precise.cuh): rows of few Welch segments, `gf` frames resident on the device
int run_group_precise(zfb_engine *e, const void *d_in, int gf, float *d_rows) {
    const zfb_config &c = e->cfg;
    cudaStream_t st = e->stream;
    const int k = e->nstages;
    const int N = 1 << e->log2N;
    const bool no_lo = (c.flags & ZFB_FLAG_NO_LO) != 0;
    const int kind = raw_kind(c);
    const size_t fbytes = (size_t)c.frame_len * (kind == KIND_U8_RAW ? 2 : 8);
    for (int g0 = 0; g0 < gf; g0 += e->px_group) {
        const int nf = (gf - g0 < e->px_group) ? gf - g0 : e->px_group;
        const char *in = (const char *)d_in + (size_t)g0 * fbytes;
        double2 *A = (double2 *)e->px_a.p, *B = (double2 *)e->px_b.p;
        if (k > 0) {
            PxLoadParams lp{};
            lp.in = in;
            lp.in_stride = c.frame_len;
            lp.n = c.frame_len;
            lp.kind = kind;
            lp.flip = c.flip;
            lp.mix = no_lo ? 0 : 1;
            lp.phase_inc = e->sp0[0].phase_inc;
            lp.amp = sqrt(2.0);
            lp.out = A;
            lp.out_stride = e->px_stride;
            lp.frames = nf;
            long long blocks = ((long long)nf * c.frame_len + 255) / 256;
            if (blocks > (long long)e->sm_count * 32) blocks = (long long)e->sm_count * 32;
            const int pr = prof_begin(e, 0);
            ZFB_LAUNCH(px_load_kernel, dim3((unsigned)blocks), dim3(256), 0, st, lp);
            e->counters[2] += 1;
            for (int s = 0; s < k; ++s) {
                PxIirParams ip{};
                ip.L = e->len[s];
                ip.nstreams = (ip.L + 2 * PADLEN + PX_STREAM - 1) / PX_STREAM;
                ip.frames = nf;
                ip.x_stride = ip.y_stride = e->px_stride;
                const unsigned blocks_i = (unsigned)((nf * ip.nstreams + 127) / 128);
                ip.x = A; ip.y = B; ip.backward = 0;
                ZFB_LAUNCH(px_iir_kernel, dim3(blocks_i), dim3(128), 0, st, ip);
                ip.x = B; ip.y = A; ip.backward = 1;
                ZFB_LAUNCH(px_iir_kernel, dim3(blocks_i), dim3(128), 0, st, ip);
                e->counters[2] += 2;
            }
            prof_end(e, pr);
            if (g0 + nf == gf) {             // zfb_debug_read_decimated: first frame of the last sub-group
                const int nd = e->len[k];
                ZFB_LAUNCH(px_to_c64_kernel, dim3((unsigned)((nd + 255) / 256)), dim3(256), 0, st,
                           (const double2 *)A, (float2 *)e->mid[0].p, nd);
                e->counters[2] += 1;
                e->final_buf = 0;
            }
        }
        PxWelchParams wp{};
        wp.from_wire = (k == 0) ? 1 : 0;
        wp.x = (k == 0) ? (const void *)in : (const void *)A;
        wp.x_stride = (k == 0) ? c.frame_len : e->px_stride;
        wp.kind = kind;
        wp.flip = (k == 0) ? c.flip : 0;
        wp.len = e->len[k];
        wp.nperseg = e->nperseg;
        wp.hop = e->hop;
        wp.nseg = e->nseg;
        wp.log2N = e->log2N;
        wp.window = (const double *)e->px_win.p;
        wp.twiddle = (const double2 *)e->px_tw.p;
        wp.work = (double2 *)e->px_work.p;
        wp.pow = (double *)e->px_pow.p;
        const int prw = prof_begin(e, 16);
        ZFB_LAUNCH(px_welch_kernel, dim3((unsigned)e->nseg, (unsigned)nf), dim3(PX_WELCH_NT), 0, st, wp);
        prof_end(e, prw);
        PxRowsParams rp{};
        rp.pow = (const double *)e->px_pow.p;
        rp.frames = nf;
        rp.nseg = e->nseg;
        rp.log2N = e->log2N;
        rp.W = e->W;
        rp.onesided = e->onesided ? 1 : 0;
        rp.os_lo = N / 2 - c.row_width / 2;
        rp.scale = 1.0 / (c.fs * e->sum_w2) / (double)e->nseg;
        rp.alpha = (c.ema_alpha >= 0.0) ? c.ema_alpha : -1.0;
        rp.linear = (c.flags & ZFB_FLAG_LINEAR) ? 1 : 0;
        rp.ema_state = (float *)e->ema.p;
        rp.ema_have = e->ema_have ? 1 : 0;
        rp.rows = trace_rows_or(e, d_rows ? d_rows + (size_t)g0 * e->W : nullptr);
        const bool to_ring = e->ring_append && e->ring.p && e->ring_W == e->W && e->cur_nch == 0;
        rp.ring = to_ring ? (float *)e->ring.p : nullptr;
        rp.ring_pos = (long long)(e->ring_written % e->ring_rows);
        rp.ring_rows = e->ring_rows;
        const int prf = prof_begin(e, 18);
        // EMA: the recurrence runs along the frames (one row of blocks); else frames in parallel
        const unsigned rows_y = rp.alpha >= 0.0 ? 1u : (unsigned)(nf < 64 ? nf : 64);
        ZFB_LAUNCH(px_rows_kernel, dim3((unsigned)((e->W + 255) / 256), rows_y), dim3(256), 0, st, rp);
        prof_end(e, prf);
        e->counters[2] += 2;
        if (rp.alpha >= 0.0) e->ema_have = true;
        if (to_ring) e->ring_written += nf;
        const int rc = trace_update(e, rp.rows, nf, st);
        if (rc) return rc;
    }
    CK(e, cudaGetLastError());
    e->last_group_frames = gf;
    e->last_front = e;
    e->counters[0] += (uint64_t)gf;
    e->counters[1] += (uint64_t)gf * (uint64_t)c.frame_len;
    return ZFB_OK;
}

// int16 IQ converted by the first FIR chain's own loads (no widening pass over the chunk)?
bool fir_cs16_fused(const zfb_engine *e) {
    return e->cs16_fused && e->fast_active && !e->precise_active && e->nchains >= 1 && e->chain_run[0] != 0 &&
           e->cur_nch == 0;
}

// one group of frames, all resident on the device, through the whole chain
int finish_rows(zfb_engine *e, zfb_engine *from, int gf, int nsplit, float *d_rows, cudaStream_t st);

// a launch group up to the Welch power sums (e->pow, nsplit partial sums per row); finish_rows makes
// rows of them.  *done: the fp64 path (run_group_precise) has written the rows itself
int run_group_front(zfb_engine *e, const void *d_in, int gf, float *d_rows, int *nsplit_out, bool *done) {
    const zfb_config &c = e->cfg;
    cudaStream_t st = e->stream;
    *done = false;
    const void *d_in_cs16 = nullptr;
    if (c.dtype == ZFB_DTYPE_CS16 && fir_cs16_fused(e)) {
        // the FIR interior converts on load (zfb_firchain.cuh, KIND_CS16_RAW); only the chunk ends the
        // exact strips read are widened, at their own positions of the complex64 buffer
        const long long n = (long long)gf * (long long)c.frame_len;
        int rc = ensure(e, e->cvt, (size_t)n * sizeof(float2));
        if (rc) return rc;
        int ends = e->strip_len[0] + 512;
        if (2 * ends > c.frame_len) ends = (c.frame_len + 1) / 2;
        const long long total = (long long)gf * 2 * ends;
        long long blocks = (total + 255) / 256;
        ZFB_LAUNCH(cs16_ends_to_c64_kernel, dim3((unsigned)blocks), dim3(256), 0, st, (const unsigned int *)d_in,
                   (float2 *)e->cvt.p, c.frame_len, ends, total);
        e->counters[2] += 1;
        d_in_cs16 = d_in;
        d_in = e->cvt.p;
    } else if (c.dtype == ZFB_DTYPE_CS16) {
        // channel-batched launches read cur_chan_frames input frames for gf = frames * channels rows
        const long long in_frames = e->cur_nch > 0 ? e->cur_chan_frames : gf;
        const long long n = in_frames * (long long)c.frame_len;
        int rc = ensure(e, e->cvt, (size_t)n * sizeof(float2));
        if (rc) return rc;
        if (n > 0) {
            long long blocks = (n + 255) / 256;
            const long long cap = (long long)e->sm_count * 16;
            if (blocks > cap) blocks = cap;
            ZFB_LAUNCH(cs16_to_c64_kernel, dim3((unsigned)blocks), dim3(256), 0, st, (const unsigned int *)d_in,
                       (float2 *)e->cvt.p, n);
            e->counters[2] += 1;
        }
        d_in = e->cvt.p;
    }
    if (e->precise_active) {
        *done = true;
        return run_group_precise(e, d_in, gf, d_rows);
    }
    const void *src = d_in;
    long long src_stride = c.frame_len;
    int kind = raw_kind(c);

    if (e->fast_active) {
        int ob = 0;
        CK(e, run_decimation_fast(e, d_in, gf, &ob, d_in_cs16));
        e->final_buf = ob;
        src = e->mid[ob].p;
        src_stride = final_stride(e);
        kind = KIND_C64_MID;
    } else
    for (int s = 0; s < e->nstages; ++s) {
        // 8192-sample region (3 CTAs/SM: one CTA's load overlaps another's sweeps)
        // unless zfb_set_option asked for the 16384-sample one (1 CTA/SM, half the halo)
        // (fixed per engine, never per launch: a frame's row must not depend on
        // how many frames share its launch)
        const int v = (e->decim_threads == NTHR_BIG) ? 0 : 1;
        const int nt = v == 0 ? NTHR_BIG : NTHR_SMALL;
        StageParams p = e->sp0[v];        // LO tables only matter for stage 0
        float2 *out = (float2 *)e->mid[s & 1].p;
        const long long out_stride = stride4(e->len[s + 1]);
        p.in = src;
        p.out = out;
        p.in_stride = src_stride;
        p.out_stride = out_stride;
        p.L = e->len[s];
        p.T = e->T[s][v];
        p.flip = (s == 0) ? c.flip : 0;
        p.strips = 0;
        p.Lfull = p.L;
        p.w_lo[0] = p.w_lo[1] = 0;
        p.w_hi[0] = p.w_hi[1] = INT_MAX;
        dim3 grid((unsigned)e->tiles[s][v], (unsigned)gf);
        const int pr = prof_begin(e, s);
        ZFB_LAUNCH(decim_lookup(kind, nt), grid, dim3((unsigned)nt), decim_smem(nt), st, p);
        prof_end(e, pr);
        e->counters[2] += 1;
        src = out;
        src_stride = out_stride;
        kind = KIND_C64_MID;
        e->final_buf = s & 1;
    }

    // Welch
    int nsplit = 1;
    if (e->log2N <= kMaxLog2Small) {
        // CTAs per frame: fixed per configuration (not per launch) so that the
        // summation order, hence every bit of a row, is independent of batching
        // auto: 4, or 8 from 24 segments per frame (cfg1, 28 segments: 60.5 -> 56.3 us per launch, r02o)
        int want = e->welch_splits > 0 ? e->welch_splits : (e->nseg >= 24 ? 8 : 4);
        if (want > e->nseg) want = e->nseg;
        if (want > e->nsplit_cap) want = e->nsplit_cap;
        if (want < 1) want = 1;
        const int per = (e->nseg + want - 1) / want;
        nsplit = (e->nseg + per - 1) / per;
        WelchParams w{};
        w.in = src;
        w.in_stride = src_stride;
        w.len = e->len[e->nstages];
        w.flip = (e->nstages == 0) ? c.flip : 0;
        w.nperseg = e->nperseg;
        w.hop = e->hop;
        w.nseg = e->nseg;
        w.seg_per_split = per;
        w.nsplit = nsplit;
        w.reuse = (e->nperseg == (1 << e->log2N) && e->hop * 2 == e->nperseg) ? 1 : 0;
        w.window = (const float *)e->window.p;
        w.twiddle = (const float2 *)e->twiddle.p;
        w.W = e->Wp;
        w.pow_out = (float *)e->pow.p;
        WelchEntry we = welch_lookup(e->log2N, kind, welch_keep(e->log2N, e->Wp), e->welch_prune);
        const int pr = prof_begin(e, 16);
        ZFB_LAUNCH(we.fn, dim3((unsigned)nsplit, (unsigned)gf), dim3((unsigned)we.threads), we.smem, st, w);
        prof_end(e, pr);
        e->counters[2] += 1;
    } else if (e->log2N >= kMinLog2R16 && e->log2N <= kMaxLog2R16) {
        // radix-16 decimation in frequency, then the one-CTA FFT on every block of N/16
        const int lS = e->log2N - 4, S = 1 << lS;
        int want = e->welch_splits > 0 ? e->welch_splits : 4;
        if (want > 4) want = 4;                          // pow16 is sized for 4 splits
        if (want > e->nseg) want = e->nseg;
        if (want < 1) want = 1;
        const int per = (e->nseg + want - 1) / want;
        const int ns16 = (e->nseg + per - 1) / per;
        BigR16Params r{};
        r.in = src;
        r.in_stride = src_stride;
        r.len = e->len[e->nstages];
        r.flip = (e->nstages == 0) ? c.flip : 0;
        r.log2N = e->log2N;
        r.hop = e->hop;
        r.nseg = e->nseg;
        r.window = (const float *)e->window.p;
        r.twiddle = (const float2 *)e->twiddle.p;
        r.scratch = (float2 *)e->big.p;
        // behind the scratch: per-CTA raw sums [group][nseg][S/256], then the means [group][nseg]
        r.partial = r.scratch + ((size_t)e->group * (size_t)e->nseg << e->log2N);
        r.means = r.partial + (size_t)e->group * (size_t)e->nseg * (size_t)(S / 256);
        r.dc = r.means + (size_t)e->group * (size_t)e->nseg;
        const int pr = prof_begin(e, 16);
        const dim3 gr((unsigned)(S / 256), (unsigned)e->nseg, (unsigned)gf);
        if (kind == KIND_C64_RAW) {
            ZFB_LAUNCH((big_dc_kernel<KIND_C64_RAW, BigR16Params>), dim3((unsigned)gf), dim3(1024), 0, st, r);
            ZFB_LAUNCH(big_r16_kernel<KIND_C64_RAW>, gr, dim3(256), 0, st, r);
        } else if (kind == KIND_U8_RAW) {
            ZFB_LAUNCH((big_dc_kernel<KIND_U8_RAW, BigR16Params>), dim3((unsigned)gf), dim3(1024), 0, st, r);
            ZFB_LAUNCH(big_r16_kernel<KIND_U8_RAW>, gr, dim3(256), 0, st, r);
        } else {
            ZFB_LAUNCH((big_dc_kernel<KIND_C64_MID, BigR16Params>), dim3((unsigned)gf), dim3(1024), 0, st, r);
            ZFB_LAUNCH(big_r16_kernel<KIND_C64_MID>, gr, dim3(256), 0, st, r);
        }
        const int nsegs_total = gf * e->nseg;
        ZFB_LAUNCH(big_mean16_kernel, dim3((unsigned)((nsegs_total + 127) / 128)), dim3(128), 0, st, r, nsegs_total);
        prof_end(e, pr);
        WelchParams w{};
        w.in = r.scratch;
        w.in_stride = (long long)e->nseg * S;
        w.len = e->nseg * S;
        w.flip = 0;
        w.nperseg = S;
        w.hop = S;
        w.nseg = e->nseg;
        w.seg_per_split = per;
        w.nsplit = ns16;
        w.reuse = 0;
        w.prepared = 1;
        w.window = nullptr;
        w.twiddle = (const float2 *)e->twiddle_sub.p;
        w.W = S;
        w.pow_out = (float *)e->pow16.p;
        w.seg_mean = r.means;
        w.wf16 = (const float2 *)e->winfft16.p;
        w.wf_n = e->wf_sparse_n;
        w.wf_bin = (const int *)e->wf_sparse.p;
        w.wf_val = (const float2 *)((const char *)e->wf_sparse.p + WF_SPARSE_MAX * sizeof(int));
        WelchEntry we = welch_lookup(lS, KIND_C64_MID);
        const int pr2 = prof_begin(e, 17);
        ZFB_LAUNCH(we.fn, dim3((unsigned)ns16, (unsigned)(gf * 16)), dim3((unsigned)we.threads), we.smem, st, w);
        BigGatherParams g{};
        g.pow16 = (const float *)e->pow16.p;
        g.pow_out = (float *)e->pow.p;
        g.log2N = e->log2N;
        g.nsplit = ns16;
        g.W = e->W;
        g.frames = gf;
        const long long cellsg = (long long)gf * e->W;
        ZFB_LAUNCH(big_gather_kernel, dim3((unsigned)((cellsg + 255) / 256)), dim3(256), 0, st, g);
        prof_end(e, pr2);
        e->counters[2] += 5;
        nsplit = 1;
    } else {
        int want = e->welch_splits > 0 ? e->welch_splits : 4;
        if (want > e->nseg) want = e->nseg;
        if (want > e->nsplit_cap) want = e->nsplit_cap;
        if (want < 1) want = 1;
        const int per = (e->nseg + want - 1) / want;
        nsplit = (e->nseg + per - 1) / per;
        BigParams b{};
        b.in = src;
        b.in_stride = src_stride;
        b.len = e->len[e->nstages];
        b.flip = (e->nstages == 0) ? c.flip : 0;
        b.log2N = e->log2N;
        b.hop = e->hop;
        b.nseg = e->nseg;
        b.seg_per_split = per;
        b.nsplit = nsplit;
        b.ntiles_col = big_ntiles_col(e->log2N);
        b.window = (const float *)e->window.p;
        b.twiddle = (const float2 *)e->twiddle.p;
        b.winfft = (const float2 *)e->winfft.p;
        b.scratch = (float2 *)e->big.p;
        b.partial = b.scratch + ((size_t)e->group * (size_t)e->nseg << e->log2N);
        b.means = b.partial + (size_t)e->group * (size_t)e->nseg * (size_t)b.ntiles_col;
        b.dc = b.means + (size_t)e->group * (size_t)e->nseg;
        b.W = e->W;
        b.pow_out = (float *)e->pow.p;
        const int pr = prof_begin(e, 16);
        big_run_col(b, kind, gf, st);
        prof_end(e, pr);
        const int pr2 = prof_begin(e, 17);
        big_run_row(b, gf, st);
        prof_end(e, pr2);
        e->counters[2] += 4;
    }

    CK(e, cudaGetLastError());
    *nsplit_out = nsplit;
    return ZFB_OK;
}

// rows of one launch group from the power sums in from->pow (this engine's, or a lane's): scale,
// EMA in frame order, dB20, ring -- on stream st (e->stream, or fin_stream for pipelined batches)
int finish_rows(zfb_engine *e, zfb_engine *from, int gf, int nsplit, float *d_rows, cudaStream_t st) {
    const zfb_config &c = e->cfg;
    FinalizeParams f{};
    f.pow_io = (float *)from->pow.p;
    f.nframes = gf;
    f.nsplit = nsplit;
    f.W = e->W;
    f.Wp = e->Wp;
    f.onesided = e->onesided ? 1 : 0;
    f.os_lo = (1 << e->log2N) / 2 - c.row_width / 2;
    f.os_N = 1 << e->log2N;
    f.scale = (float)(1.0 / (c.fs * e->sum_w2) / (double)e->nseg);
    f.alpha = (c.ema_alpha >= 0.0) ? (float)c.ema_alpha : -1.f;
    f.linear = (c.flags & ZFB_FLAG_LINEAR) ? 1 : 0;
    f.ema_state = (float *)e->ema.p;
    f.ema_have = e->ema_have ? 1 : 0;
    f.rows = trace_rows_or(e, d_rows);
    // rows enter the ring when it has their width; channel-batched launches (rows of different
    // receivers) never do
    const bool to_ring = e->ring_append && e->ring.p && e->ring_W == e->W && e->cur_nch == 0;
    f.ring = to_ring ? (float *)e->ring.p : nullptr;
    f.ring_pos = (long long)(e->ring_written % e->ring_rows);
    f.ring_rows = e->ring_rows;
    f.chan_frames = e->cur_nch > 0 ? e->cur_chan_frames : 0;
    f.chan_row_stride = e->cur_row_stride;
    const int prf = prof_begin(e, 18, st);
    const long long cells = (long long)gf * e->W;
    if (f.alpha >= 0.f) {
        ZFB_LAUNCH(ema_rows_kernel, dim3((unsigned)((e->W + EMA_COLS - 1) / EMA_COLS)), dim3(EMA_NT), 0, st, f);
        e->ema_have = true;
    } else {
        ZFB_LAUNCH(reduce_rows_kernel, dim3((unsigned)((cells + 255) / 256)), dim3(256), 0, st, f);
    }
    e->counters[2] += 1;
    prof_end(e, prf, st);
    CK(e, cudaGetLastError());
    const int rc = trace_update(e, f.rows, gf, st);
    if (rc) return rc;
    if (to_ring) e->ring_written += gf;
    e->last_group_frames = gf;
    e->last_front = from;
    e->counters[0] += (uint64_t)gf;
    e->counters[1] += (uint64_t)gf * (uint64_t)c.frame_len;
    return ZFB_OK;
}

int run_group(zfb_engine *e, const void *d_in, int gf, float *d_rows) {
    int nsplit = 1;
    bool done = false;
    const int rc = run_group_front(e, d_in, gf, d_rows, &nsplit, &done);
    if (rc != ZFB_OK || done) return rc;
    return finish_rows(e, e, gf, nsplit, d_rows, e->stream);
}

// late mix of the first register-blocked chain (zfb_firchain.cuh): allowed when the LO
// offset r (cycles per input sample, folded to [0,1)) times the zoom ratio is <= 1e-3
void set_late_mix(zfb_engine *e, FirRunParams &rp, double r, double amp, int ns) {
    const double off = r < 0.5 ? r : 1.0 - r;
    const bool no_lo = (e->cfg.flags & ZFB_FLAG_NO_LO) != 0;
    rp.late = (e->late_mix && !no_lo && off * (double)e->cfg.fft_ratio <= 1.0e-3) ? 1 : 0;
    for (int j = 0; j < (RUN0 >> ns); ++j) lo_entry(r, (long long)j << ns, amp, rp.lo_out[j]);
}

// ZFB_MODE_FAST planning: strip geometry, FIR chains (<= 3 stages per launch),
// tile sizes; decides whether the frame is long enough for the FAST interior
int plan_fast(zfb_engine *e) {
    const zfb_config &c = e->cfg;
    e->nchains = 0;
    if (!e->fast_active) return ZFB_OK;
    const int k = e->nstages;
    e->strip_cap = (e->strip_len[0] + 1) / 2 + 8;
    for (int i = 0; i < 2; ++i) {               // the strips' hand-off between launches
        int rc = ensure(e, e->sbuf[i], (size_t)e->group * 2 * (size_t)e->strip_cap * sizeof(float2));
        if (rc) return rc;
    }
    // chains
    const int ne = k - 1;
    const bool no_lo = (c.flags & ZFB_FLAG_NO_LO) != 0;
    double r = no_lo ? 0.0 : c.f_demod / c.fs;
    r -= floor(r);
    if (r >= 1.0) r = 0.0;
    int done = 0;
    while (done < ne) {
        if (e->nchains >= 4) return fail(e, ZFB_EINVAL, "fft_ratio too deep for mode FAST");
        FirChainParams &p = e->chain[e->nchains];
        memset(&p, 0, sizeof p);
        // the LAST chain takes up to 3 stages (it has the specialised kernel);
        // what is left over goes to the first chain (fast_chain_sizes)
        int ns = (ne - done) % FIR_MAX_STAGES;
        if (ns == 0) ns = FIR_MAX_STAGES;
        p.ns = ns;
        for (int s = 0; s < ns; ++s) {
            p.M[s] = e->fplan.M[done + s];
            memcpy(p.h[s], e->fplan.h[done + s], sizeof p.h[s]);
        }
        const bool lastc = (done + ns == ne);
        p.Mc = lastc ? e->fplan.Mc : -1;
        if (lastc) memcpy(p.hc, e->fplan.hc, sizeof p.hc);
        p.L = e->len[done];
        p.flip = (done == 0) ? c.flip : 0;
        if (done == 0) {
            const double scaled = ldexp(r, 64);
            p.phase_inc = (scaled >= 18446744073709551615.0) ? 0ull : (unsigned long long)scaled;
            const int vec = (c.dtype == ZFB_DTYPE_U8) ? 8 : 2;
            const double amp = no_lo ? 1.0 : sqrt(2.0);
            for (int i = 0; i < 8; ++i) lo_entry(r, i, amp, p.lo_small[i]);
            for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * FIR_NT * vec, 1.0, p.lo_big[it]);
        }
        // tile: as many outputs as keep level 0 near 4096 samples (about 50 KB of smem)
        const int vec0 = (done == 0 && c.dtype == ZFB_DTYPE_U8) ? 8 : 2;
        int best = 0;
        for (int to = 16; to <= 4096; to += 16) {
            p.TO = to;
            FirTile t;
            fir_tile_geometry(p, 0, t);
            if (t.n[0] > 4352 || t.n[0] / vec0 > 32 * FIR_NT) break;
            best = to;
        }
        if (best == 0) return fail(e, ZFB_EINVAL, "FIR plan too long for one tile");
        p.TO = best;
        FirTile t;
        fir_tile_geometry(p, 0, t);
        for (int l = 0; l <= ns; ++l) p.n[l] = t.n[l];
        e->chain_smem[e->nchains] = fir_chain_smem(p);
        // register-blocked kernel when the tap set is one it is built for
        e->chain_run[e->nchains] = e->fir_generic ? 0 : fir_run_variant(p);
        if (e->chain_run[e->nchains]) {
            FirRunParams &rp = e->runp[e->nchains];
            memset(&rp, 0, sizeof rp);
            rp.L = p.L;
            rp.flip = p.flip;
            rp.phase_inc = p.phase_inc;
            if (done == 0) {
                const double amp = no_lo ? 1.0 : sqrt(2.0);
                for (int i = 0; i < RUN0; ++i) lo_entry(r, i, amp, rp.lo_run[i]);
                set_late_mix(e, rp, r, amp, ns);
            }
            memcpy(rp.h0, p.h[0], sizeof rp.h0);
            {   // first stage on raw uint8 / int16 values (zfb_firchain.cuh: FirRunParams::h0s)
                const bool s16 = c.dtype == ZFB_DTYPE_CS16;
                double sum = 0.0;
                for (int j = 0; j <= FIR_MAX_HALF; ++j) {
                    rp.h0s[j] = (float)((double)p.h[0][j] / (s16 ? 32768.0 : 127.5));
                    sum += (j == 0 ? 1.0 : 2.0) * (double)rp.h0s[j];
                }
                rp.bias0 = s16 ? 0.f : (float)(127.5 * sum);      // uint8 is offset binary, int16 is not
            }
            memcpy(rp.h1, p.h[1], sizeof rp.h1);
            memcpy(rp.h2, p.h[2], sizeof rp.h2);
            memcpy(rp.hc, p.hc, sizeof rp.hc);
        }
        done += ns;
        e->chain_level_out[e->nchains] = done;
        e->nchains += 1;
    }
    return ZFB_OK;
}

// Streaming last stage of mode fast (zfb_iirstream.cuh): every frame's stage input is cut into
// nspf streams of S samples, 32 consecutive streams per warp.  S and nspf depend on the stage
// length only -- never on how many frames share a launch -- so a frame's row stays
// bit-identical whatever batch it is in.
void plan_iir_stream(zfb_engine *e) {
    zfb_engine::IirStreamPlan &pl = e->iis;
    pl.active = false;
    if (!e->fast_active || !e->iir_stream) return;
    const int k = e->nstages;
    const int L = e->len[k - 1];
    const int Wb = e->iir_Wm / IS_BLK;
    // whole warps: nspf a multiple of 32 whose streams come closest to the target length
    int g = (int)((double)L / (32.0 * (double)e->iir_S) + 0.5);
    if (g < 1) g = 1;
    int nspf = 32 * g;
    int S16 = (L + nspf * IS_BLK - 1) / (nspf * IS_BLK);
    // the warm-up (and the lag block) must fit into the neighbouring stream
    if (S16 < Wb + 1) return;                 // short frames keep the shared-memory kernel
    const int S = S16 * IS_BLK;
    nspf = (L + S - 1) / S;                   // streams actually holding samples
    pl.q.S16 = S16;
    pl.q.Wb = Wb;
    pl.q.nspf = nspf;
    pl.q.groups = (nspf + 31) / 32;
    pl.q.keep_from = S16 - (int)((long long)S16 * e->iir_l2_keep / 100);
    pl.in_stride = stride4((long long)nspf * S);
    pl.out_stride = stride4((long long)nspf * (S / 2));
    pl.tail = nspf * S - L;
    pl.active = true;
}

// tensor maps over the (now allocated) intermediates, and the strips' patch buffer
int finish_iir_stream(zfb_engine *e) {
    zfb_engine::IirStreamPlan &pl = e->iis;
    const int k = e->nstages;
    const int b_final = e->nchains & 1;
    void *in = e->mid[b_final ^ 1].p, *out = e->mid[b_final].p;
    const unsigned long long S = (unsigned long long)pl.q.S16 * IS_BLK;
    TensorMapSpec si{};
    si.base = in;
    si.dim[0] = IS_BLK; si.dim[1] = (unsigned long long)pl.q.S16; si.dim[2] = (unsigned long long)pl.q.nspf;
    si.dim[3] = (unsigned long long)e->group;
    si.stride[0] = 8; si.stride[1] = IS_BLK * 8; si.stride[2] = S * 8; si.stride[3] = (unsigned long long)pl.in_stride * 8;
    si.box[0] = IS_BLK; si.box[1] = 1; si.box[2] = 32; si.box[3] = 1;
    si.swizzle = 128;
    TensorMapSpec so{};
    so.base = out;
    so.dim[0] = IS_BLK / 2; so.dim[1] = (unsigned long long)pl.q.S16; so.dim[2] = (unsigned long long)pl.q.nspf;
    so.dim[3] = (unsigned long long)e->group;
    so.stride[0] = 8; so.stride[1] = IS_BLK * 4; so.stride[2] = S * 4; so.stride[3] = (unsigned long long)pl.out_stride * 8;
    so.box[0] = IS_BLK / 2; so.box[1] = 1; so.box[2] = 32; so.box[3] = 1;
    so.swizzle = 64;
    if (make_tensor_map(si, &pl.tm_in) != 0 || make_tensor_map(so, &pl.tm_out) != 0)
        return fail(e, ZFB_ECUDA, "cuTensorMapEncodeTiled failed for the streaming last stage (stage length %d)",
                    e->len[k - 1]);
    return ensure(e, e->strip_out, (size_t)e->group * 2 * (size_t)e->fplan.K * sizeof(float2));
}

// point every LO table of the current plan at software-LO frequency f_demod
// (zfb_process_channels_*: one configuration, many zoom centres)
void apply_lo(zfb_engine *e, double f_demod) {
    const zfb_config &c = e->cfg;
    const bool no_lo = (c.flags & ZFB_FLAG_NO_LO) != 0;
    double r = no_lo ? 0.0 : f_demod / c.fs;
    r -= floor(r);
    if (r >= 1.0) r = 0.0;
    const double scaled = ldexp(r, 64);
    const unsigned long long inc = (scaled >= 18446744073709551615.0) ? 0ull : (unsigned long long)scaled;
    const int vec = (c.dtype == ZFB_DTYPE_U8) ? 8 : 2;
    DecimConst dc;
    build_decim_const(dc);
    const double amp0 = no_lo ? 1.0 : sqrt(2.0);
    for (int v = 0; v < 3; ++v) {
        const int nt = v == 0 ? NTHR_BIG : (v == 1 ? NTHR_SMALL : 64);
        StageParams &p = e->sp0[v];
        p.phase_inc = inc;
        for (int i = 0; i < 8; ++i) lo_entry(r, i, amp0 * (double)dc.g, p.lo_small[i]);
        for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * nt * vec, 1.0, p.lo_big[it]);
    }
    if (e->fast_active && e->nchains > 0) {
        FirChainParams &p = e->chain[0];
        p.phase_inc = inc;
        for (int i = 0; i < 8; ++i) lo_entry(r, i, amp0, p.lo_small[i]);
        for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * FIR_NT * vec, 1.0, p.lo_big[it]);
        if (e->chain_run[0]) {
            FirRunParams &rp = e->runp[0];
            rp.phase_inc = inc;
            for (int i = 0; i < RUN0; ++i) lo_entry(r, i, amp0, rp.lo_run[i]);
            set_late_mix(e, rp, r, amp0, e->chain[0].ns);
        }
    }
}

bool is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace

// =============================================================================
extern "C" {

// pipelined batches: e->stream catches up with everything the lanes and fin_stream still hold
static void join_pending_work(zfb_engine *e) {
    if (!e->join_pending) return;
    cudaSetDevice(e->device);
    cudaStreamWaitEvent(e->stream, e->ev_done, 0);
    e->join_pending = false;
}

int zfb_abi_version(void) { return ZFB_ABI_VERSION; }

const char *zfb_build_kind(void) { return ZFB_BUILD_KIND; }

#ifndef ZFB_SOURCE_HASH
#define ZFB_SOURCE_HASH "unknown"
#endif
const char *zfb_source_hash(void) { return ZFB_SOURCE_HASH; }

const char *zfb_last_error(const zfb_engine *e) {
    return e ? e->err.c_str() : g_create_error.c_str();
}

int zfb_create(int device, zfb_engine **out) {
    if (!out) return fail(nullptr, ZFB_EINVAL, "zfb_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return fail(nullptr, ZFB_ENODEV,
                    "no CUDA device (%s); this engine has no CPU fallback",
                    st != cudaSuccess ? cudaGetErrorString(st) : "device count is 0");
    }
    if (device < 0 || device >= ndev)
        return fail(nullptr, ZFB_ENODEV, "device %d out of range (%d present)", device, ndev);
    zfb_engine *e = new (std::nothrow) zfb_engine();
    if (!e) return fail(nullptr, ZFB_ENOMEM, "out of host memory");
    e->device = device;
    int rc = ZFB_OK;
    do {
        if (cudaSetDevice(device) != cudaSuccess) { rc = fail(nullptr, ZFB_ENODEV, "cudaSetDevice(%d) failed", device); break; }
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) e->sm_count = prop.multiProcessorCount;
        if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&e->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) {
            rc = fail(nullptr, ZFB_ECUDA, "stream creation failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        e->stream = e->own_stream;
        for (int i = 0; i < 2; ++i) {
            if (cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&e->ev_free[i], cudaEventDisableTiming) != cudaSuccess) {
                rc = fail(nullptr, ZFB_ECUDA, "event creation failed");
                break;
            }
        }
        if (rc != ZFB_OK) break;
        rc = setup_device_once(e);
        if (rc != ZFB_OK) { g_create_error = e->err; break; }
    } while (0);
    if (rc != ZFB_OK) {
        zfb_destroy(e);
        return rc;
    }
    *out = e;
    return ZFB_OK;
}

void zfb_destroy(zfb_engine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->fin_stream) cudaStreamSynchronize(e->fin_stream);     // rows of pipelined batches read the lanes' sums
    for (int i = 0; i < 2; ++i) {
        if (e->lane[i]) zfb_destroy(e->lane[i]);
        e->lane[i] = nullptr;
        if (e->ev_lane[i]) cudaEventDestroy(e->ev_lane[i]);
        if (e->ev_fin[i]) cudaEventDestroy(e->ev_fin[i]);
    }
    if (e->ev_batch_in) cudaEventDestroy(e->ev_batch_in);
    if (e->fin_stream) {
        cudaStreamSynchronize(e->fin_stream);
        cudaStreamDestroy(e->fin_stream);
    }
    if (e->ev_done) cudaEventDestroy(e->ev_done);
    if (e->own_stream) cudaStreamSynchronize(e->own_stream);
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    if (e->aux_stream) cudaStreamSynchronize(e->aux_stream);
    DevBuf *bufs[] = {&e->window, &e->winfft, &e->winfft16, &e->wf_sparse, &e->twiddle, &e->twiddle_sub, &e->pow16, &e->mid[0], &e->mid[1], &e->pow, &e->rows_tmp, &e->ema,
                      &e->img_out, &e->img_lut, &e->img_thr, &e->sel_hist, &e->ring, &e->stage_in[0], &e->stage_in[1], &e->big,
                      &e->trace, &e->trace_rows, &e->peaks};
    for (DevBuf *b : bufs) release(*b);
    for (int i = 0; i < 2; ++i) {
        if (e->h_stage[i]) cudaFreeHost(e->h_stage[i]);
        if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]);
        if (e->ev_free[i]) cudaEventDestroy(e->ev_free[i]);
    }
    for (auto *v : {&e->prof_used, &e->prof_free})
        for (auto &r : *v) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    if (e->sr_host) cudaFreeHost(e->sr_host);
    release(e->sr_dev[0]);
    release(e->sr_dev[1]);
    release(e->sbuf[0]);
    release(e->sbuf[1]);
    release(e->chan_dev);
    release(e->cvt);
    release(e->strip_out);
    release(e->taper_buf);
    for (DevBuf *b : {&e->px_a, &e->px_b, &e->px_work, &e->px_pow, &e->px_win, &e->px_tw}) release(*b);
    if (e->sr_copied) cudaEventDestroy(e->sr_copied);
    for (int i = 0; i < 2; ++i) if (e->sr_free[i]) cudaEventDestroy(e->sr_free[i]);
    if (e->h_rows) cudaFreeHost(e->h_rows);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->aux_stream) cudaStreamDestroy(e->aux_stream);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    delete e;
}

int zfb_decim_sos(double out24[24]) {
    if (!out24) return ZFB_EINVAL;
    double sos[NSEC][6];
    design_cheby1_sos(sos);
    memcpy(out24, sos, sizeof sos);
    return ZFB_OK;
}

int zfb_plan_geometry(int frame_len, int fft_size, int fft_ratio, int out5[5]) {
    if (!out5) return ZFB_EINVAL;
    Geometry g;
    int rc = geometry(frame_len, fft_size, fft_ratio, g);
    if (rc != ZFB_OK) return rc;
    out5[0] = g.ndec;
    out5[1] = g.nperseg;
    out5[2] = g.hop;
    out5[3] = g.nseg;
    out5[4] = g.nstages;
    return ZFB_OK;
}

static int configure_impl(zfb_engine *e, const zfb_config *cfg);
static void setup_lanes(zfb_engine *e);

// trace state and the scratch for rows of launch groups without a caller's row buffer
static int trace_buffers(zfb_engine *e) {
    const size_t W = (size_t)e->W;
    int rc = ensure(e, e->trace, W * (sizeof(double) + 4 * sizeof(float)));
    if (rc) return rc;
    return ensure(e, e->trace_rows, (size_t)e->group * W * sizeof(float));     // fp64 passes: px_group <= group
}

int zfb_configure(zfb_engine *e, const zfb_config *cfg) {
    if (!e) return ZFB_EINVAL;
    const int rc = configure_impl(e, cfg);
    std::lock_guard<std::mutex> lk(e->mu);
    // the lanes are planned lazily, by the first batch large enough to be cut in two (a live
    // front-end that hands over one chunk per call never pays for them)
    e->lanes_ready = false;
    e->lanes_stale = true;
    e->window_host.clear();
    if (rc == ZFB_OK && cfg && cfg->window && e->nperseg > 0) e->window_host.assign(cfg->window, cfg->window + e->nperseg);
    return rc;
}

static int configure_impl(zfb_engine *e, const zfb_config *cfg) {
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!cfg) return fail(e, ZFB_EINVAL, "configure: cfg is NULL");
    CK(e, cudaSetDevice(e->device));
    const int N = cfg->fft_size;
    const int l2 = ilog2_floor(N);
    if (N < (1 << kMinLog2N) || N > (1 << kMaxLog2N) || (1 << l2) != N)
        return fail(e, ZFB_EINVAL, "fft_size %d: must be a power of two in [%d, %d]", N, 1 << kMinLog2N,
                    1 << kMaxLog2N);
    if (!(cfg->fs > 0.0)) return fail(e, ZFB_EINVAL, "fs must be positive");
    if (cfg->fft_ratio < 1) return fail(e, ZFB_EINVAL, "fft_ratio %d: must be >= 1", cfg->fft_ratio);
    if (cfg->dtype != ZFB_DTYPE_C64 && cfg->dtype != ZFB_DTYPE_U8 && cfg->dtype != ZFB_DTYPE_CS16)
        return fail(e, ZFB_EINVAL, "unknown dtype %d", cfg->dtype);
    if (cfg->mode != ZFB_MODE_EXACT && cfg->mode != ZFB_MODE_FAST)
        return fail(e, ZFB_EINVAL, "unknown mode %d", cfg->mode);
    if (cfg->row_width < 2 || cfg->row_width > N || (cfg->row_width & 1))
        return fail(e, ZFB_EINVAL, "row_width %d: must be even and in [2, fft_size]", cfg->row_width);
    const bool onesided = (cfg->flags & ZFB_FLAG_ONESIDED) != 0;
    if (onesided && (cfg->fft_ratio != 1 || cfg->dtype != ZFB_DTYPE_C64 || l2 > kMaxLog2Small))
        return fail(e, ZFB_EINVAL, "one-sided rows need fft_ratio 1, complex64 storage of the real samples and "
                    "fft_size <= %d", 1 << kMaxLog2Small);
    const int row_w = onesided ? cfg->row_width / 2 + 1 : cfg->row_width;
    if (!cfg->window) return fail(e, ZFB_EINVAL, "window is NULL");
    Geometry g;
    int rc = geometry(cfg->frame_len, N, cfg->fft_ratio, g);
    if (rc == ZFB_ETOOSHORT)
        return fail(e, rc, "frame_len %d too short: every decimate-by-2 stage needs more than %d samples "
                    "(scipy padlen)", cfg->frame_len, PADLEN);
    if (rc != ZFB_OK) return fail(e, rc, "bad geometry (frame_len %d, fft_size %d, fft_ratio %d)",
                                  cfg->frame_len, N, cfg->fft_ratio);
    if (cfg->nperseg != g.nperseg)
        return fail(e, ZFB_EINVAL, "nperseg %d does not match the plan (%d): call zfb_plan_geometry first",
                    cfg->nperseg, g.nperseg);
    if (l2 > kMaxLog2Small && g.nperseg != N)
        return fail(e, ZFB_EINVAL, "fft_size %d needs a decimated chunk of at least fft_size samples (got %d)",
                    N, g.ndec);

    // (re-planning after zfb_set_fast_plan / zfb_set_group / an option does not change the
    // geometry: the ring and the EMA state survive a change of frame_len alone)
    const int geom_now[4] = {row_w, N, cfg->fft_ratio, onesided ? 1 : 0};
    const bool geom_changed = !e->geom_valid || memcmp(geom_now, e->geom, sizeof geom_now) != 0;
    // everything below may replace buffers still in use
    CK(e, cudaStreamSynchronize(e->stream));
    // the live plan is taken apart from here on: a failure must not leave it half updated
    e->configured = false;

    // window -> float, sum w^2 in double (scale = 1/(fs*sum w^2), scipy:_spectral_py.py 'density')
    std::vector<float> wf((size_t)g.nperseg);
    double s2 = 0.0;
    for (int i = 0; i < g.nperseg; ++i) {
        const double w = cfg->window[i];
        if (!(w == w) || fabs(w) > 1e30) return fail(e, ZFB_EINVAL, "window[%d] is not finite", i);
        s2 += w * w;
        wf[(size_t)i] = (float)w;
    }
    if (!(s2 > 0.0)) return fail(e, ZFB_EINVAL, "window has zero energy");
    rc = ensure(e, e->window, wf.size() * sizeof(float));
    if (rc) return rc;
    CK(e, cudaMemcpyAsync(e->window.p, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    if (l2 > kMaxLog2Small) {
        // FFT(window) in fp64 for the post-FFT mean removal of the four-step path
        std::vector<double> re((size_t)N), im((size_t)N, 0.0);
        for (int i = 0; i < N; ++i) re[(size_t)i] = cfg->window[i];
        host_fft(re, im);
        std::vector<float2> wff((size_t)N);
        for (int i = 0; i < N; ++i) wff[(size_t)i] = make_float2((float)re[(size_t)i], (float)im[(size_t)i]);
        rc = ensure(e, e->winfft, wff.size() * sizeof(float2));
        if (rc) return rc;
        CK(e, cudaMemcpyAsync(e->winfft.p, wff.data(), wff.size() * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        if (l2 >= kMinLog2R16 && l2 <= kMaxLog2R16) {
            // cosine-sum windows: FFT(w) is a few bins around DC (fp64 FFT noise ~1e-16 N elsewhere)
            double peak = 0.0;
            for (int i = 0; i < N; ++i) peak = std::max(peak, hypot(re[(size_t)i], im[(size_t)i]));
            int nnz = 0;
            e->wf_sparse_n = 0;
            for (int i = 0; i < N && nnz <= WF_SPARSE_MAX; ++i)
                if (hypot(re[(size_t)i], im[(size_t)i]) > 1e-11 * peak) {
                    if (nnz < WF_SPARSE_MAX) {
                        e->wf_sparse_bin[nnz] = i;
                        e->wf_sparse_val[nnz] = wff[(size_t)i];
                    }
                    ++nnz;
                }
            if (nnz >= 1 && nnz <= WF_SPARSE_MAX) e->wf_sparse_n = nnz;
            for (int a = 0; a < e->wf_sparse_n; ++a)       // one listed bin per residue, or the dense table
                for (int b2 = a + 1; b2 < e->wf_sparse_n; ++b2)
                    if ((e->wf_sparse_bin[a] & 15) == (e->wf_sparse_bin[b2] & 15)) nnz = WF_SPARSE_MAX + 1;
            if (nnz > WF_SPARSE_MAX) e->wf_sparse_n = 0;
            {   // [WF_SPARSE_MAX] bins, then [WF_SPARSE_MAX] values
                unsigned char blob[WF_SPARSE_MAX * (sizeof(int) + sizeof(float2))] = {0};
                memcpy(blob, e->wf_sparse_bin, sizeof e->wf_sparse_bin);
                memcpy(blob + WF_SPARSE_MAX * sizeof(int), e->wf_sparse_val, sizeof e->wf_sparse_val);
                rc = ensure(e, e->wf_sparse, sizeof blob);
                if (rc) return rc;
                CK(e, cudaMemcpyAsync(e->wf_sparse.p, blob, sizeof blob, cudaMemcpyHostToDevice, e->stream));
                CK(e, cudaStreamSynchronize(e->stream));
            }
            // the same per residue of the radix-16 front pass: winfft16[r][k] = FFT(w)[16 k + r]
            std::vector<float2> w16((size_t)N);
            const int S16 = N >> 4;
            for (int r = 0; r < 16; ++r)
                for (int k = 0; k < S16; ++k) w16[(size_t)r * S16 + k] = wff[(size_t)16 * k + r];
            rc = ensure(e, e->winfft16, w16.size() * sizeof(float2));
            if (rc) return rc;
            CK(e, cudaMemcpyAsync(e->winfft16.p, w16.data(), w16.size() * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
            CK(e, cudaStreamSynchronize(e->stream));
        }
    }

    if (!e->configured || e->cfg.fft_size != N) {
        std::vector<float2> tw((size_t)N);
        for (int k = 0; k < N; ++k) {
            const double a = -2.0 * kPi * (double)k / (double)N;
            tw[(size_t)k] = make_float2((float)cos(a), (float)sin(a));
        }
        rc = ensure(e, e->twiddle, tw.size() * sizeof(float2));
        if (rc) return rc;
        CK(e, cudaMemcpyAsync(e->twiddle.p, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
    }
    CK(e, cudaStreamSynchronize(e->stream));       // wf goes out of scope

    // plan
    e->cfg = *cfg;
    e->cfg.window = nullptr;
    e->nstages = g.nstages;
    memcpy(e->len, g.len, sizeof g.len);
    e->nperseg = g.nperseg;
    e->hop = g.hop;
    e->nseg = g.nseg;
    e->W = row_w;
    e->Wp = onesided ? N : row_w;
    e->onesided = onesided;
    e->log2N = l2;
    e->sum_w2 = s2;
    // stage-0 LO tables (one per tile geometry)
    for (int v = 0; v < 3; ++v) {
        const int nt = v == 0 ? NTHR_BIG : (v == 1 ? NTHR_SMALL : 64);
        StageParams &p = e->sp0[v];
        memset(&p, 0, sizeof p);
        const bool no_lo = (cfg->flags & ZFB_FLAG_NO_LO) != 0;
        double r = no_lo ? 0.0 : cfg->f_demod / cfg->fs;
        r -= floor(r);
        if (r >= 1.0) r = 0.0;
        const double scaled = ldexp(r, 64);
        p.phase_inc = (scaled >= 18446744073709551615.0) ? 0ull : (unsigned long long)scaled;
        DecimConst dc;
        build_decim_const(dc);
        const double amp = (no_lo ? 1.0 : sqrt(2.0)) * (double)dc.g;
        const int vec = (cfg->dtype == ZFB_DTYPE_U8) ? 8 : 2;
        for (int i = 0; i < 8; ++i) lo_entry(r, i, amp, p.lo_small[i]);
        for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * nt * vec, 1.0, p.lo_big[it]);
    }
    if (cfg->mode == ZFB_MODE_FAST && g.nstages >= 2 && (!e->fplan.set || e->fplan.ne != g.nstages - 1))
        return fail(e, ZFB_ESTATE, "mode FAST needs zfb_set_fast_plan with %d stages (got %d)", g.nstages - 1,
                    e->fplan.set ? e->fplan.ne : -1);
    e->fast_active = fast_wanted(e, e->strip_len, e->strip_q);
    plan_iir_stream(e);                          // (frame strides of the intermediates depend on it)
    e->group = choose_group(e, e->fast_active);
    plan_tiles(e);
    e->nsplit_cap = 16;
    rc = plan_fast(e);
    if (rc) return rc;

    // workspaces
    {
        long long need[2];
        mid_lengths(e, e->fast_active, need);
        for (int i = 0; i < 2; ++i)
            if (need[i] > 0) {
                rc = ensure(e, e->mid[i], (size_t)e->group * (size_t)need[i] * sizeof(float2));
                if (rc) return rc;
            }
    }
    if (e->iis.active) {
        rc = finish_iir_stream(e);
        if (rc) return rc;
    }
    rc = ensure(e, e->pow, (size_t)e->group * (size_t)e->nsplit_cap * (size_t)e->Wp * sizeof(float));
    if (rc) return rc;
    if (l2 > kMaxLog2Small) {
        rc = ensure(e, e->big, big_scratch_bytes(l2, g.nseg, e->group));
        if (rc) return rc;
    }
    if (l2 >= kMinLog2R16 && l2 <= kMaxLog2R16) {
        const int S = N >> 4;
        std::vector<float2> tws((size_t)S);
        for (int k = 0; k < S; ++k) {
            const double a = -2.0 * kPi * (double)k / (double)S;
            tws[(size_t)k] = make_float2((float)cos(a), (float)sin(a));
        }
        rc = ensure(e, e->twiddle_sub, tws.size() * sizeof(float2));
        if (rc) return rc;
        CK(e, cudaMemcpyAsync(e->twiddle_sub.p, tws.data(), tws.size() * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        rc = ensure(e, e->pow16, (size_t)e->group * 4 * (size_t)N * sizeof(float));   // <= 4 splits
        if (rc) return rc;
    }
    rc = ensure(e, e->ema, (size_t)e->W * sizeof(float));
    if (rc) return rc;
    if (geom_changed) e->ema_have = false;
    if (e->ring_user_W == 0 &&
        (geom_changed || e->ring_W != e->W || e->ring_rows != e->ring_rows_req || !e->ring.p)) {
        // the ring follows the configured row width (Waterfall.init_image on a new width, S:1641-1643)
        e->ring_W = 0;
        e->ring_rows = e->ring_rows_req;
        rc = ensure(e, e->ring, (size_t)e->ring_rows * (size_t)e->W * sizeof(float));
        if (rc) return rc;
        e->ring_W = e->W;
        e->ring_written = 0;
    }
    // fp64 path for rows of few segments (zfb_precise.cuh): small jobs by construction
    e->precise_active = e->precise == 1 ||
                        (e->precise < 0 && g.nseg <= 6 && (long long)g.nseg * N <= (1 << 21) && cfg->frame_len <= (1 << 23));
    if (e->precise_active) {
        const size_t stride = (size_t)stride4((long long)cfg->frame_len + 2 * PADLEN + 8);
        size_t per_frame = 2 * stride * sizeof(double2) + (size_t)g.nseg * (size_t)N * (2 * sizeof(double2) + sizeof(double));
        // frames per pass: these rows are small jobs, but a batch of them (BASELINE configs[4] sweeps)
        // should still fill the GPU: up to 1024 frames / 2 GB of fp64 workspace per pass
        long long pg = (long long)((2048ull << 20) / per_frame);
        e->px_group = (int)(pg < 1 ? 1 : (pg > 1024 ? 1024 : pg));
        if (e->px_group > e->group) e->px_group = e->group > 0 ? e->group : 1;
        e->px_stride = (long long)stride;
        if (g.nstages > 0) {
            rc = ensure(e, e->px_a, (size_t)e->px_group * stride * sizeof(double2));
            if (rc) return rc;
            rc = ensure(e, e->px_b, (size_t)e->px_group * stride * sizeof(double2));
            if (rc) return rc;
            rc = ensure(e, e->mid[0], (size_t)(g.ndec + 8) * sizeof(float2));
            if (rc) return rc;
        }
        rc = ensure(e, e->px_work, (size_t)e->px_group * g.nseg * 2 * (size_t)N * sizeof(double2));
        if (rc) return rc;
        rc = ensure(e, e->px_pow, (size_t)e->px_group * g.nseg * (size_t)N * sizeof(double));
        if (rc) return rc;
        rc = ensure(e, e->px_win, (size_t)g.nperseg * sizeof(double));
        if (rc) return rc;
        {   // twiddles of the radix-2 passes, fp64 on the host
            std::vector<double2> tw((size_t)(N / 2 > 0 ? N / 2 : 1));
            for (int m = 0; m < N / 2; ++m) {
                const double a = -kPi * (double)m / (double)(N / 2);
                tw[(size_t)m] = make_double2(cos(a), sin(a));
            }
            rc = ensure(e, e->px_tw, tw.size() * sizeof(double2));
            if (rc) return rc;
            CK(e, cudaMemcpyAsync(e->px_tw.p, tw.data(), tw.size() * sizeof(double2), cudaMemcpyHostToDevice, e->stream));
            CK(e, cudaStreamSynchronize(e->stream));
        }
        CK(e, cudaMemcpyAsync(e->px_win.p, cfg->window, (size_t)g.nperseg * sizeof(double), cudaMemcpyHostToDevice, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));       // the caller's window table may go away
    }
    // the traces keep counting over a change of frame_len, window, EMA, wire format, flip or mode;
    // anything that changes what a column means or its units starts them afresh
    const double key[6] = {cfg->fs, (double)N, (double)cfg->fft_ratio, (double)cfg->row_width, cfg->f_demod,
                           (double)cfg->flags};
    if (memcmp(key, e->trace_key, sizeof key) != 0) e->trace_count = 0;
    memcpy(e->trace_key, key, sizeof key);
    if (e->traces_on) {
        rc = trace_buffers(e);
        if (rc) return rc;
    }
    memcpy(e->geom, geom_now, sizeof geom_now);
    e->geom_valid = true;
    e->configured = true;
    return ZFB_OK;
}

// lanes of the pipelined batches: two engines on the same device with this engine's plan and options
// (best effort: any failure leaves the one-lane path in charge)
static void setup_lanes(zfb_engine *e) {          // e->mu is held by the caller
    e->lanes_ready = false;
    e->lanes_stale = false;
    if (e->is_lane || !e->pipeline || !e->configured || !e->fast_active || e->precise_active ||
        e->window_host.empty())
        return;
    // re-planning a lane may free workspaces that rows of earlier batches are still read from
    if (e->fin_stream) cudaStreamSynchronize(e->fin_stream);
    if (!e->fin_stream && cudaStreamCreateWithFlags(&e->fin_stream, cudaStreamNonBlocking) != cudaSuccess) return;
    if (!e->ev_done && cudaEventCreateWithFlags(&e->ev_done, cudaEventDisableTiming) != cudaSuccess) return;
    zfb_config c2 = e->cfg;
    c2.window = e->window_host.data();
    c2.ema_alpha = -1.0;                          // rows are finished by this engine: no EMA state in a lane
    if (!e->ev_batch_in && cudaEventCreateWithFlags(&e->ev_batch_in, cudaEventDisableTiming) != cudaSuccess) return;
    for (int i = 0; i < 2; ++i) {
        if (!e->lane[i]) {
            if (zfb_create(e->device, &e->lane[i]) != ZFB_OK) { e->lane[i] = nullptr; return; }
            e->lane[i]->is_lane = true;
        }
        zfb_engine *l = e->lane[i];
        {
            std::lock_guard<std::mutex> lk2(l->mu);
            l->strips_async = e->strips_async; l->strip_split = e->strip_split;
            l->strip_decay = e->strip_decay; l->strip_decay_early = e->strip_decay_early; l->ring_append = 0;
            l->late_mix = e->late_mix; l->iir_stream = e->iir_stream; l->iir_S = e->iir_S; l->iir_Wm = e->iir_Wm;
            l->iir_l2_keep = e->iir_l2_keep; l->precise = e->precise;
            l->decim_threads = e->decim_threads; l->welch_splits = e->welch_splits; l->cs16_fused = e->cs16_fused;
            l->welch_prune = e->welch_prune; l->fir_generic = e->fir_generic; l->group_user = e->group_user;
            l->fplan = e->fplan;
            l->configured = false;
        }
        if (configure_impl(l, &c2) != ZFB_OK || !l->fast_active || l->precise_active || l->group != e->group ||
            l->W != e->W || l->Wp != e->Wp)
            return;
        for (cudaEvent_t *ev : {&e->ev_lane[i], &e->ev_fin[i]})
            if (!*ev && cudaEventCreateWithFlags(ev, cudaEventDisableTiming) != cudaSuccess) return;
        // ev_fin_used[i] stays: rows of an earlier batch may still be read from this lane's sums
    }
    cudaGetLastError();
    e->lanes_ready = true;
}

// a whole batch on the next lane, its rows finished on fin_stream; e->stream joins later (zfb_join)
static int process_pipelined(zfb_engine *e, const void *d_in, int nframes, float *d_rows) {
    const size_t fbytes = (size_t)e->cfg.frame_len * sample_bytes(e->cfg);
    const int i = e->next_lane;
    e->next_lane ^= 1;
    zfb_engine *l = e->lane[i];
    // the input, and whatever the caller's stream did to the EMA state / ring before this call
    CK(e, cudaEventRecord(e->ev_batch_in, e->stream));
    CK(e, cudaStreamWaitEvent(l->stream, e->ev_batch_in, 0));
    CK(e, cudaStreamWaitEvent(e->fin_stream, e->ev_batch_in, 0));
    l->profiling = e->profiling;
    int rc = ZFB_OK;
    for (int g0 = 0; g0 < nframes && rc == ZFB_OK; g0 += e->group) {
        const int gf = (nframes - g0 < e->group) ? nframes - g0 : e->group;
        if (e->ev_fin_used[i]) CK(e, cudaStreamWaitEvent(l->stream, e->ev_fin[i], 0));
        int nsplit = 1;
        bool done = false;
        const uint64_t launches0 = l->counters[2];
        rc = run_group_front(l, (const char *)d_in + (size_t)g0 * fbytes, gf, nullptr, &nsplit, &done);
        e->counters[2] += l->counters[2] - launches0;
        if (rc != ZFB_OK) {
            e->err = l->err;
            break;
        }
        CK(e, cudaEventRecord(e->ev_lane[i], l->stream));
        CK(e, cudaStreamWaitEvent(e->fin_stream, e->ev_lane[i], 0));
        rc = finish_rows(e, l, gf, nsplit, d_rows ? d_rows + (size_t)g0 * e->W : nullptr, e->fin_stream);
        if (rc != ZFB_OK) break;
        CK(e, cudaEventRecord(e->ev_fin[i], e->fin_stream));
        e->ev_fin_used[i] = true;
    }
    if (rc != ZFB_OK) {
        for (int k = 0; k < 2; ++k) cudaStreamSynchronize(e->lane[k]->stream);
        cudaStreamSynchronize(e->fin_stream);
        cudaGetLastError();
        return rc;
    }
    CK(e, cudaEventRecord(e->ev_done, e->fin_stream));
    e->join_pending = true;
    return ZFB_OK;
}

int zfb_set_fast_plan(zfb_engine *e, const zfb_fast_plan *plan) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (!plan) return fail(e, ZFB_EINVAL, "fast plan is NULL");
    if (plan->nstages < 1 || plan->nstages > ZFB_FAST_MAX_STAGES)
        return fail(e, ZFB_EINVAL, "fast plan: nstages %d out of range", plan->nstages);
    if (plan->strip < 64 || (plan->strip & 1)) return fail(e, ZFB_EINVAL, "fast plan: strip must be even and >= 64");
    if (plan->comp_half < 0 || plan->comp_half > FIR_COMP_MAX_HALF || !plan->comp_taps)
        return fail(e, ZFB_EINVAL, "fast plan: compensator half length %d out of range", plan->comp_half);
    zfb_engine::FastPlan f;
    f.ne = plan->nstages;
    for (int s = 0; s < f.ne; ++s) {
        if (plan->half[s] < 1 || plan->half[s] > FIR_MAX_HALF || !plan->taps[s])
            return fail(e, ZFB_EINVAL, "fast plan: stage %d half length %d out of range", s, plan->half[s]);
        f.M[s] = plan->half[s];
        double dc = plan->taps[s][0];
        for (int j = 0; j <= f.M[s]; ++j) {
            if (!(plan->taps[s][j] == plan->taps[s][j])) return fail(e, ZFB_EINVAL, "fast plan: NaN tap");
            f.h[s][j] = (float)plan->taps[s][j];
            if (j) dc += 2.0 * plan->taps[s][j];
        }
        if (fabs(dc - 1.0) > 1e-6) return fail(e, ZFB_EINVAL, "fast plan: stage %d DC gain %.9f != 1", s, dc);
    }
    f.Mc = plan->comp_half;
    for (int j = 0; j <= f.Mc; ++j) f.hc[j] = (float)plan->comp_taps[j];
    f.K = plan->strip;
    f.set = true;
    {
        const zfb_engine::FastPlan &o = e->fplan;
        if (o.set && o.ne == f.ne && o.Mc == f.Mc && o.K == f.K && memcmp(o.M, f.M, sizeof f.M) == 0 &&
            memcmp(o.h, f.h, sizeof f.h) == 0 && memcmp(o.hc, f.hc, sizeof f.hc) == 0)
            return ZFB_OK;                                    // same plan again: nothing to re-plan
    }
    e->fplan = f;
    e->lanes_stale = true;
    e->configured = false;       // re-plan on the next configure (ring and EMA state are kept)
    return ZFB_OK;
}

int zfb_fast_active(const zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return (e->configured && e->fast_active) ? 1 : 0;
}

int zfb_join(zfb_engine *e, void *cuda_stream) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->join_pending) return ZFB_OK;
    CK(e, cudaSetDevice(e->device));
    if (cuda_stream && (cudaStream_t)cuda_stream != e->stream) {
        CK(e, cudaStreamWaitEvent((cudaStream_t)cuda_stream, e->ev_done, 0));
        return ZFB_OK;                            // e->stream itself still has to join
    }
    join_pending_work(e);
    return ZFB_OK;
}

int zfb_slab_lanes(const zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return e->last_lanes;
}

int zfb_set_stream(zfb_engine *e, void *cuda_stream) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return ZFB_OK;
}

int zfb_set_group(zfb_engine *e, int frames_per_group) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (frames_per_group < 0) return fail(e, ZFB_EINVAL, "frames_per_group must be >= 0");
    e->group_user = frames_per_group;
    e->lanes_stale = true;
    e->configured = false;      // workspaces are sized per group: re-plan on next configure
    return ZFB_OK;
}

int zfb_set_option(zfb_engine *e, const char *name, long long value) {
    if (!e || !name) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    e->lanes_stale = true;                       // the lanes take this engine's options when next used
    if (strcmp(name, "slabs") == 0) {            // kept for callers that set it: 0 and 1 both mean one lane per batch
        if (value < 0 || value > 1) return fail(e, ZFB_EINVAL, "slabs must be 0 or 1 (one lane)");
        return ZFB_OK;
    }
    if (strcmp(name, "pipeline") == 0) {
        join_pending_work(e);
        e->pipeline = value ? 1 : 0;
        return ZFB_OK;
    }
    if (strcmp(name, "decim_threads") == 0) {
        if (value != 0 && value != NTHR_BIG && value != NTHR_SMALL)
            return fail(e, ZFB_EINVAL, "decim_threads must be 0 (auto), %d or %d", NTHR_SMALL, NTHR_BIG);
        e->decim_threads = (int)value;
        return ZFB_OK;
    }
    if (strcmp(name, "welch_splits") == 0) {
        if (value < 0 || value > 16) return fail(e, ZFB_EINVAL, "welch_splits must be in [0, 16]");
        e->welch_splits = (int)value;
        return ZFB_OK;
    }
    if (strcmp(name, "cs16_fused") == 0) {
        e->cs16_fused = value ? 1 : 0;
        return ZFB_OK;
    }
    if (strcmp(name, "welch_prune") == 0) {
        if (value < 0 || value > 2) return fail(e, ZFB_EINVAL, "welch_prune must be 0, 1 or 2");
        e->welch_prune = (int)value;
        return ZFB_OK;
    }
    if (strcmp(name, "strips_async") == 0) {
        if (value < 0 || value > 1) return fail(e, ZFB_EINVAL, "strips_async must be 0 (main stream) or 1 (side stream)");
        e->strips_async = (int)value;
        return ZFB_OK;
    }
    if (strcmp(name, "strip_decay") == 0) {
        if (value < 64 || value > 1024 || (value & 1)) return fail(e, ZFB_EINVAL, "strip_decay must be even and in [64, 1024]");
        e->strip_decay = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "strip_decay_early") == 0) {
        if (value < 32 || value > 1024 || (value & 1)) return fail(e, ZFB_EINVAL, "strip_decay_early must be even and in [32, 1024]");
        e->strip_decay_early = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "strip_split") == 0) {
        e->strip_split = value ? 1 : 0;
        return ZFB_OK;
    }
    if (strcmp(name, "late_mix") == 0) {
        e->late_mix = value ? 1 : 0;
        e->configured = false;                   // replanned by the next zfb_configure
        return ZFB_OK;
    }
    if (strcmp(name, "iir_stream") == 0) {
        e->iir_stream = value ? 1 : 0;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "iir_stream_len") == 0) {
        if (value < 256 || value > (1 << 20))
            return fail(e, ZFB_EINVAL, "iir_stream_len (target samples per stream) must be in [256, 2^20]");
        e->iir_S = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "precise") == 0) {
        if (value < -1 || value > 1) return fail(e, ZFB_EINVAL, "precise must be -1 (auto), 0 or 1");
        e->precise = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "iir_l2_keep") == 0) {
        if (value < 0 || value > 100) return fail(e, ZFB_EINVAL, "iir_l2_keep is a percentage");
        e->iir_l2_keep = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "iir_stream_warm") == 0) {
        if (value < 2 * IS_BLK || value > 4096 || value % IS_BLK)
            return fail(e, ZFB_EINVAL, "iir_stream_warm must be a multiple of %d in [%d, 4096]", IS_BLK, 2 * IS_BLK);
        e->iir_Wm = (int)value;
        e->configured = false;
        return ZFB_OK;
    }
    if (strcmp(name, "ring_append") == 0) {
        e->ring_append = value ? 1 : 0;
        return ZFB_OK;
    }
    if (strcmp(name, "host_taper") == 0) {
        e->host_taper = value ? 1 : 0;
        return ZFB_OK;
    }
    if (strcmp(name, "fir_generic") == 0) {
        e->fir_generic = value ? 1 : 0;
        e->configured = false;
        return ZFB_OK;
    }
    return fail(e, ZFB_EINVAL, "unknown option '%s'", name);
}

int zfb_reset_ema(zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    e->ema_have = false;     // launch order is stream order: the next EMA group starts afresh
    return ZFB_OK;
}

// ---- max-hold / min-hold / average traces and peak markers (zfb_trace.cuh) ----------------------
int zfb_traces_enable(zfb_engine *e, int on) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    e->trace_count = 0;
    if (!on) {
        // rows still being folded in read these buffers
        CK(e, cudaStreamSynchronize(e->stream));
        e->traces_on = false;
        for (DevBuf *b : {&e->trace, &e->trace_rows, &e->peaks}) release(*b);
        return ZFB_OK;
    }
    e->traces_on = true;
    if (e->configured) {
        const int rc = trace_buffers(e);
        if (rc) {
            e->traces_on = false;
            return rc;
        }
    }
    return ZFB_OK;
}

int zfb_traces_reset(zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    e->trace_count = 0;      // launch order is stream order: the next update starts afresh
    return ZFB_OK;
}

int64_t zfb_traces_count(const zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return e->traces_on ? e->trace_count : 0;
}

// device address of a trace in row units (AVG: read out into its slot first, on e->stream)
static int trace_vector(zfb_engine *e, int kind, const float **out) {
    if (kind < ZFB_TRACE_LAST || kind > ZFB_TRACE_AVG) return fail(e, ZFB_EINVAL, "trace kind %d: must be 0..3", kind);
    if (!e->traces_on) return fail(e, ZFB_ESTATE, "traces are off (zfb_traces_enable)");
    if (!e->configured || e->trace_count < 1) return fail(e, ZFB_ESTATE, "the traces hold no row yet");
    const int W = e->W;
    const double *sum = (const double *)e->trace.p;
    float *f = (float *)(sum + W);             // LAST, MAX, MIN, AVG
    if (kind == ZFB_TRACE_AVG) {
        ZFB_LAUNCH(trace_avg_kernel, dim3((unsigned)((W + 255) / 256)), dim3(256), 0, e->stream, sum,
                   (long long)e->trace_count, W, (e->cfg.flags & ZFB_FLAG_LINEAR) ? 1 : 0, f + 3 * (size_t)W);
        CK(e, cudaGetLastError());
        e->counters[2] += 1;
    }
    *out = f + (size_t)kind * W;
    return ZFB_OK;
}

int zfb_trace_read(zfb_engine *e, int kind, float *h_out) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!h_out) return fail(e, ZFB_EINVAL, "trace_read: h_out is NULL");
    CK(e, cudaSetDevice(e->device));
    const float *src = nullptr;
    const int rc = trace_vector(e, kind, &src);
    if (rc) return rc;
    const size_t bytes = (size_t)e->W * sizeof(float);
    CK(e, cudaMemcpyAsync(h_out, src, bytes, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->counters[4] += bytes;
    return ZFB_OK;
}

// one peak query on e->stream over n floats at d_x; copies back the <= k markers only
static int find_peaks(zfb_engine *e, const float *d_x, int n, int k, int distance, double height, int32_t *cols,
                      float *values, double *offsets, int *npeaks) {
    if (!d_x || !cols || !values || !offsets || !npeaks) return fail(e, ZFB_EINVAL, "find_peaks: NULL argument");
    if (n < 1 || n > PK_MAX_N) return fail(e, ZFB_EINVAL, "find_peaks: n = %d must be in [1, %d]", n, PK_MAX_N);
    if (k < 1 || k > PK_MAX) return fail(e, ZFB_EINVAL, "find_peaks: k = %d must be in [1, %d]", k, PK_MAX);
    if (distance < 1) return fail(e, ZFB_EINVAL, "find_peaks: distance = %d must be >= 1", distance);
    int rc = ensure(e, e->peaks, sizeof(PeakOut) + (size_t)n);
    if (rc) return rc;
    PeakParams pp{};
    pp.x = d_x;
    pp.n = n;
    pp.k = k;
    pp.distance = distance;
    pp.use_height = height == height ? 1 : 0;
    // x >= height on float values == x >= the smallest float not below height
    float h = (float)height;
    if (pp.use_height && (double)h < height) h = nextafterf(h, INFINITY);
    pp.height = h;
    pp.out = (PeakOut *)e->peaks.p;
    pp.flag = (unsigned char *)e->peaks.p + sizeof(PeakOut);
    ZFB_LAUNCH(trace_peaks_kernel, dim3(1), dim3(PK_NT), 0, e->stream, pp);
    CK(e, cudaGetLastError());
    e->counters[2] += 1;
    PeakOut out;
    CK(e, cudaMemcpyAsync(&out, e->peaks.p, sizeof out, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->counters[4] += sizeof out;
    *npeaks = out.count;
    for (int i = 0; i < out.count; ++i) {
        cols[i] = out.column[i];
        values[i] = out.value[i];
        offsets[i] = out.offset[i];
    }
    return ZFB_OK;
}

int zfb_trace_peaks(zfb_engine *e, int kind, int k, int distance, double height, int32_t *cols, float *values,
                    double *offsets, int *npeaks) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    const float *src = nullptr;
    const int rc = trace_vector(e, kind, &src);
    if (rc) return rc;
    return find_peaks(e, src, e->W, k, distance, height, cols, values, offsets, npeaks);
}

int zfb_find_peaks_device(zfb_engine *e, const float *d_x, int n, int k, int distance, double height, int32_t *cols,
                          float *values, double *offsets, int *npeaks) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    return find_peaks(e, d_x, n, k, distance, height, cols, values, offsets, npeaks);
}

// channel-batched launches exist for the FAST path with one register-blocked
// chain and fused strips (fft_ratio 4, 8, 16 on raw input); everything else
// loops over the channels
static bool channels_batchable(const zfb_engine *e) {
    return !e->precise_active && e->fast_active && e->nchains == 1 && e->chain_run[0] != 0 && e->nstages <= 4;
}

static int upload_channels(zfb_engine *e, const double *f_demod, int nch) {
    const zfb_config &c = e->cfg;
    const bool no_lo = (c.flags & ZFB_FLAG_NO_LO) != 0;
    const int vec = (c.dtype == ZFB_DTYPE_U8) ? 8 : 2;
    DecimConst dc;
    build_decim_const(dc);
    const double amp0 = no_lo ? 1.0 : sqrt(2.0);
    e->chan_host.resize((size_t)nch);
    for (int ch = 0; ch < nch; ++ch) {
        ChannelLo &t = e->chan_host[(size_t)ch];
        double r = no_lo ? 0.0 : f_demod[ch] / c.fs;
        r -= floor(r);
        if (r >= 1.0) r = 0.0;
        const double scaled = ldexp(r, 64);
        t.phase_inc = (scaled >= 18446744073709551615.0) ? 0ull : (unsigned long long)scaled;
        for (int i = 0; i < 32; ++i) lo_entry(r, i, amp0, t.run[i]);
        for (int i = 0; i < 8; ++i) lo_entry(r, i, amp0 * (double)dc.g, t.dec_small[i]);
        for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * STRIP_NT * vec, 1.0, t.dec_big[it]);
        for (int it = 0; it < 32; ++it) lo_entry(r, (long long)it * 64 * vec, 1.0, t.dec_big64[it]);
        // same late-mix decision and table as a single-channel configuration at this f_demod
        // (batched == per-channel, bit for bit)
        t.late = 0;
        t.pad_ = 0;
        for (int j = 0; j < 16; ++j) t.out[j] = make_float2(0.f, 0.f);
        if (e->fast_active && e->nchains > 0 && e->chain_run[0]) {
            FirRunParams tmp{};
            set_late_mix(e, tmp, r, amp0, e->chain[0].ns);
            t.late = tmp.late;
            for (int j = 0; j < RUN0 / 2; ++j) t.out[j] = tmp.lo_out[j];
        }
    }
    int rc = ensure(e, e->chan_dev, (size_t)nch * sizeof(ChannelLo));
    if (rc) return rc;
    // pageable source: the runtime stages it before returning, chan_host may be reused afterwards
    CK(e, cudaMemcpyAsync(e->chan_dev.p, e->chan_host.data(), (size_t)nch * sizeof(ChannelLo),
                          cudaMemcpyHostToDevice, e->stream));
    return ZFB_OK;
}

// `gf` frames starting at d_in for all `nch` channels; rows at d_rows[ch*nframes*W + f*W]
static int run_channels(zfb_engine *e, const void *d_in, int gf, const double *f_demod, int nch, int nframes,
                        float *d_rows, bool batched) {
    const size_t fbytes = (size_t)e->cfg.frame_len * sample_bytes(e->cfg);
    int rc = ZFB_OK;
    if (batched) {
        int per = e->group / nch;
        if (per < 1) per = 1;
        for (int q0 = 0; q0 < gf && rc == ZFB_OK; q0 += per) {
            const int qf = (gf - q0 < per) ? gf - q0 : per;
            // more channels than the workspace holds at once: slices of channels
            const int chmax = e->group < nch ? e->group : nch;
            for (int c0 = 0; c0 < nch && rc == ZFB_OK; c0 += chmax) {
                const int cn = (nch - c0 < chmax) ? nch - c0 : chmax;
                e->cur_nch = cn;
                e->cur_chan_frames = qf;
                e->cur_row_stride = (long long)nframes * e->W;
                const ChannelLo *base = (const ChannelLo *)e->chan_dev.p;
                void *saved = e->chan_dev.p;
                e->chan_dev.p = (void *)(base + c0);
                rc = run_group(e, (const char *)d_in + (size_t)q0 * fbytes, qf * cn,
                               d_rows ? d_rows + ((size_t)c0 * nframes + q0) * e->W : nullptr);
                e->chan_dev.p = saved;
            }
        }
        e->cur_nch = 0;
        e->cur_chan_frames = 0;
    } else {
        for (int q0 = 0; q0 < gf && rc == ZFB_OK; q0 += e->group) {
            const int qf = (gf - q0 < e->group) ? gf - q0 : e->group;
            for (int ch = 0; ch < nch && rc == ZFB_OK; ++ch) {      // channels innermost: input stays in L2
                apply_lo(e, f_demod[ch]);
                rc = run_group(e, (const char *)d_in + (size_t)q0 * fbytes, qf,
                               d_rows ? d_rows + ((size_t)ch * nframes + q0) * e->W : nullptr);
            }
        }
        apply_lo(e, e->cfg.f_demod);
    }
    return rc;
}

static int check_channels(zfb_engine *e, const double *f_demod, int nch) {
    if (nch < 0 || (nch > 0 && !f_demod)) return fail(e, ZFB_EINVAL, "channels: bad arguments");
    if (nch > 0 && e->cfg.ema_alpha >= 0.0)
        return fail(e, ZFB_EINVAL, "channels: EMA state is per engine; configure with ema_alpha < 0");
    if (nch > 0 && e->traces_on)
        return fail(e, ZFB_EINVAL, "channels: the trace set is per engine; zfb_traces_enable(e, 0) first");
    if (nch > 0 && e->nstages == 0)
        return fail(e, ZFB_EINVAL, "channels: fft_ratio 1 has no software LO");
    return ZFB_OK;
}

static int process_pipelined_channels(zfb_engine *e, const void *d_in, int nframes, const double *f_demod, int nch,
                                      float *d_rows);

// nch == 0: the configured f_demod; rows [nframes][W].  nch > 0: rows [nch][nframes][W]
static int process_device_impl(zfb_engine *e, const void *d_in, int nframes, const double *f_demod, int nch,
                               float *d_rows) {
    if (!e->configured) return fail(e, ZFB_ESTATE, "process: engine is not configured");
    if (!d_in || nframes < 0) return fail(e, ZFB_EINVAL, "process: bad arguments");
    int rc = check_channels(e, f_demod, nch);
    if (rc) return rc;
    CK(e, cudaSetDevice(e->device));
    const size_t fbytes = (size_t)e->cfg.frame_len * sample_bytes(e->cfg);
    if (nch > 0) {
        const bool batched = channels_batchable(e);
        if (!e->is_lane && e->pipeline && batched && nframes >= 1) {
            if (e->lanes_stale) setup_lanes(e);
            if (e->lanes_ready) {
                e->last_lanes = 2;
                return process_pipelined_channels(e, d_in, nframes, f_demod, nch, d_rows);
            }
        }
        join_pending_work(e);
        if (batched) {
            rc = upload_channels(e, f_demod, nch);
            if (rc) return rc;
        }
        // the counters count frames per channel pass; rows [nch][nframes][W]
        return run_channels(e, d_in, nframes, f_demod, nch, nframes, d_rows, batched);
    }
    if (!e->is_lane && e->pipeline && nframes >= 1 && e->fast_active && !e->precise_active) {
        if (e->lanes_stale) setup_lanes(e);
        if (e->lanes_ready) {
            e->last_lanes = 2;
            return process_pipelined(e, d_in, nframes, d_rows);
        }
    }
    join_pending_work(e);
    e->last_lanes = 1;
    for (int g0 = 0; g0 < nframes; g0 += e->group) {
        const int gf = (nframes - g0 < e->group) ? nframes - g0 : e->group;
        rc = run_group(e, (const char *)d_in + (size_t)g0 * fbytes, gf,
                       d_rows ? d_rows + (size_t)g0 * e->W : nullptr);
        if (rc) break;
    }
    return rc;
}

// virtual receivers (channel-batched launches; no EMA, nothing appended to the ring, so the rows need
// no ordering among batches): the whole batch, finalisation included, on the next lane's stream
static int process_pipelined_channels(zfb_engine *e, const void *d_in, int nframes, const double *f_demod, int nch,
                                      float *d_rows) {
    const int i = e->next_lane;
    e->next_lane ^= 1;
    zfb_engine *l = e->lane[i];
    CK(e, cudaEventRecord(e->ev_batch_in, e->stream));
    CK(e, cudaStreamWaitEvent(l->stream, e->ev_batch_in, 0));
    l->profiling = e->profiling;
    uint64_t c0[5];
    memcpy(c0, l->counters, sizeof c0);
    const int rc = process_device_impl(l, d_in, nframes, f_demod, nch, d_rows);
    for (int k = 0; k < 5; ++k) e->counters[k] += l->counters[k] - c0[k];
    e->last_front = l;
    e->last_group_frames = l->last_group_frames;
    if (rc != ZFB_OK) {
        e->err = l->err;
        cudaStreamSynchronize(l->stream);
        cudaGetLastError();
        return rc;
    }
    // fin_stream collects the lanes' completions in the order of the calls: ev_done covers all of them
    CK(e, cudaEventRecord(e->ev_lane[i], l->stream));
    CK(e, cudaStreamWaitEvent(e->fin_stream, e->ev_lane[i], 0));
    CK(e, cudaEventRecord(e->ev_done, e->fin_stream));
    e->join_pending = true;
    return ZFB_OK;
}

int zfb_process_device(zfb_engine *e, const void *d_in, int nframes, float *d_rows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return process_device_impl(e, d_in, nframes, nullptr, 0, d_rows);
}

int zfb_process_channels_device(zfb_engine *e, const void *d_in, int nframes, const double *f_demod, int nch,
                                float *d_rows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (nch < 1) return fail(e, ZFB_EINVAL, "channels: nch must be >= 1");
    return process_device_impl(e, d_in, nframes, f_demod, nch, d_rows);
}

static int process_host_impl(zfb_engine *e, const void *h_in, int nframes, const double *f_demod, int nch,
                             float *h_rows) {
    if (!e->configured) return fail(e, ZFB_ESTATE, "process: engine is not configured");
    if (!h_in || !h_rows || nframes < 0) return fail(e, ZFB_EINVAL, "process: bad arguments");
    int rc = check_channels(e, f_demod, nch);
    if (rc) return rc;
    if (nframes == 0) return ZFB_OK;
    CK(e, cudaSetDevice(e->device));
    const int loops = nch > 0 ? nch : 1;
    const size_t fbytes = (size_t)e->cfg.frame_len * sample_bytes(e->cfg);
    const bool batched = nch > 0 && channels_batchable(e);
    if (batched) {
        rc = upload_channels(e, f_demod, nch);
        if (rc) return rc;
    }
    // host path pipelines in sub-groups so that copies overlap compute
    int hg = e->group;
    if (nframes > 1 && hg > (nframes + 3) / 4) hg = (nframes + 3) / 4;
    if (hg < 1) hg = 1;
    const bool pinned_src = is_pinned(h_in);
    for (int i = 0; i < 2; ++i) {
        rc = ensure(e, e->stage_in[i], (size_t)hg * fbytes);
        if (rc) return rc;
        if (!pinned_src && e->h_stage_cap[i] < (size_t)hg * fbytes) {
            if (e->h_stage[i]) CK(e, cudaFreeHost(e->h_stage[i]));
            e->h_stage[i] = nullptr;
            e->h_stage_cap[i] = 0;
            CK(e, cudaMallocHost(&e->h_stage[i], (size_t)hg * fbytes));
            e->h_stage_cap[i] = (size_t)hg * fbytes;
        }
    }
    const size_t rows_bytes = (size_t)loops * nframes * e->W * sizeof(float);
    rc = ensure(e, e->rows_tmp, rows_bytes);
    if (rc) return rc;
    const bool pinned_dst = is_pinned(h_rows);
    if (!pinned_dst && e->h_rows_cap < rows_bytes) {
        if (e->h_rows) CK(e, cudaFreeHost(e->h_rows));
        e->h_rows = nullptr;
        e->h_rows_cap = 0;
        CK(e, cudaMallocHost(&e->h_rows, rows_bytes));
        e->h_rows_cap = rows_bytes;
    }

    int it = 0;
    // The copies run back to back; what the call still pays after the last of them is the compute of
    // the last sub-group -- so the sub-groups taper towards the end (half of what is left, down to 8
    // frames): 128 128 128 64 32 16 8 8 for 512 frames.  Rows do not depend on the cut.
    int gf = 0;
    for (int g0 = 0; g0 < nframes && rc == ZFB_OK; g0 += gf, ++it) {
        const int left = nframes - g0;
        gf = left < hg ? left : hg;
        if (e->host_taper && left <= 2 * hg && left > 8) {
            gf = (left + 1) / 2;
            if (gf > hg) gf = hg;
        }
        const int slot = it & 1;
        const char *src = (const char *)h_in + (size_t)g0 * fbytes;
        const size_t bytes = (size_t)gf * fbytes;
        if (e->slot_busy[slot]) {
            // the device staging slot (and its pinned mirror) is free once the
            // compute that read it has finished
            if (!pinned_src) CK(e, cudaEventSynchronize(e->ev_free[slot]));
            CK(e, cudaStreamWaitEvent(e->copy_stream, e->ev_free[slot], 0));
        }
        if (!pinned_src) {
            memcpy(e->h_stage[slot], src, bytes);
            src = (const char *)e->h_stage[slot];
        }
        CK(e, cudaMemcpyAsync(e->stage_in[slot].p, src, bytes, cudaMemcpyHostToDevice, e->copy_stream));
        CK(e, cudaEventRecord(e->ev_h2d[slot], e->copy_stream));
        CK(e, cudaStreamWaitEvent(e->stream, e->ev_h2d[slot], 0));
        e->counters[3] += bytes;
        if (nch > 0) {
            rc = run_channels(e, e->stage_in[slot].p, gf, f_demod, nch, nframes,
                              (float *)e->rows_tmp.p + (size_t)g0 * e->W, batched);
        } else {
            for (int q0 = 0; q0 < gf && rc == ZFB_OK; q0 += e->group) {
                const int qf = (gf - q0 < e->group) ? gf - q0 : e->group;
                rc = run_group(e, (const char *)e->stage_in[slot].p + (size_t)q0 * fbytes, qf,
                               (float *)e->rows_tmp.p + (size_t)(g0 + q0) * e->W);
            }
        }
        CK(e, cudaEventRecord(e->ev_free[slot], e->stream));
        e->slot_busy[slot] = true;
    }
    if (rc) return rc;
    float *dst = pinned_dst ? h_rows : e->h_rows;
    CK(e, cudaMemcpyAsync(dst, e->rows_tmp.p, rows_bytes, cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    if (!pinned_dst) memcpy(h_rows, e->h_rows, rows_bytes);
    e->counters[4] += rows_bytes;
    e->slot_busy[0] = e->slot_busy[1] = false;
    return ZFB_OK;
}

int zfb_process_host(zfb_engine *e, const void *h_in, int nframes, float *h_rows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    return process_host_impl(e, h_in, nframes, nullptr, 0, h_rows);
}

int zfb_process_channels_host(zfb_engine *e, const void *h_in, int nframes, const double *f_demod, int nch,
                              float *h_rows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (nch < 1) return fail(e, ZFB_EINVAL, "channels: nch must be >= 1");
    return process_host_impl(e, h_in, nframes, f_demod, nch, h_rows);
}

int zfb_synchronize(zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    return ZFB_OK;
}

int zfb_debug_read_decimated(zfb_engine *e, float *h_out_iq, int max_samples) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!e->configured) return fail(e, ZFB_ESTATE, "engine is not configured");
    if (e->nstages < 1 || e->last_group_frames < 1)
        return fail(e, ZFB_ESTATE, "no decimated chunk available (fft_ratio < 2 or nothing processed)");
    if (!h_out_iq || max_samples < 0) return fail(e, ZFB_EINVAL, "bad arguments");
    CK(e, cudaSetDevice(e->device));
    int n = e->len[e->nstages];
    if (n > max_samples) n = max_samples;
    CK(e, cudaStreamSynchronize(e->stream));
    const zfb_engine *src = e->last_front ? e->last_front : e;     // a lane, after a pipelined batch
    CK(e, cudaMemcpy(h_out_iq, src->mid[src->final_buf].p, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
    e->counters[4] += (size_t)n * sizeof(float2);
    return n;
}

static int ring_realloc(zfb_engine *e, int rows, int width) {
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    e->ring_W = 0;                                  // no valid ring while it is replaced
    int rc = ensure(e, e->ring, (size_t)rows * (size_t)width * sizeof(float));
    if (rc) return rc;
    e->ring_rows = rows;
    e->ring_W = width;
    e->ring_written = 0;
    return ZFB_OK;
}

int zfb_ring_configure(zfb_engine *e, int rows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (rows < 1) return fail(e, ZFB_EINVAL, "ring rows must be >= 1");
    e->ring_rows_req = rows;
    e->ring_user_W = 0;                             // back to following the configured row width
    if (e->configured && (rows != e->ring_rows || e->ring_W != e->W)) return ring_realloc(e, rows, e->W);
    return ZFB_OK;
}

int zfb_ring_configure_width(zfb_engine *e, int rows, int width) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (rows < 1) return fail(e, ZFB_EINVAL, "ring rows must be >= 1");
    if (width < 1 || width > (1 << 24)) return fail(e, ZFB_EINVAL, "ring width %d out of range", width);
    e->ring_rows_req = rows;
    e->ring_user_W = width;
    return ring_realloc(e, rows, width);            // a (re)configured ring starts empty (S:1625-1635)
}

int zfb_ring_width(const zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return e->ring.p ? e->ring_W : 0;
}

int64_t zfb_ring_rows_written(const zfb_engine *e) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    return e->ring_written;
}

int zfb_read_rows(zfb_engine *e, int age, int nrows, float *h_out) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!e->ring.p || e->ring_W < 1) return fail(e, ZFB_ESTATE, "no ring (configure the engine or the ring first)");
    if (age < 0 || nrows < 1 || !h_out) return fail(e, ZFB_EINVAL, "read_rows: bad arguments");
    const int64_t have = e->ring_written < e->ring_rows ? e->ring_written : e->ring_rows;
    if ((int64_t)age + nrows > have)
        return fail(e, ZFB_EINVAL, "read_rows: asked for rows %d..%d back but the ring holds %lld", age,
                    age + nrows - 1, (long long)have);
    CK(e, cudaSetDevice(e->device));
    const int64_t first = e->ring_written - age - nrows;          // chronological index
    const size_t rb = (size_t)e->ring_W * sizeof(float);
    int done = 0;
    while (done < nrows) {
        const int64_t slot = (first + done) % e->ring_rows;
        int run = nrows - done;
        if (slot + run > e->ring_rows) run = (int)(e->ring_rows - slot);
        CK(e, cudaMemcpyAsync((char *)h_out + (size_t)done * rb, (const char *)e->ring.p + (size_t)slot * rb,
                              (size_t)run * rb, cudaMemcpyDeviceToHost, e->stream));
        done += run;
    }
    CK(e, cudaStreamSynchronize(e->stream));
    e->counters[4] += (size_t)nrows * rb;
    return ZFB_OK;
}

int zfb_ring_push_rows(zfb_engine *e, const float *h_rows, int nrows) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!e->ring.p || e->ring_W < 1) return fail(e, ZFB_ESTATE, "no ring (configure the engine or the ring first)");
    if (!h_rows || nrows < 0) return fail(e, ZFB_EINVAL, "push_rows: bad arguments");
    CK(e, cudaSetDevice(e->device));
    const size_t rb = (size_t)e->ring_W * sizeof(float);
    for (int i = 0; i < nrows; ++i) {
        const int64_t slot = e->ring_written % e->ring_rows;
        CK(e, cudaMemcpyAsync((char *)e->ring.p + (size_t)slot * rb, (const char *)h_rows + (size_t)i * rb, rb,
                              cudaMemcpyHostToDevice, e->stream));
        e->ring_written += 1;
    }
    CK(e, cudaStreamSynchronize(e->stream));      // caller's buffer may be pageable / reused
    e->counters[3] += (size_t)nrows * rb;
    return ZFB_OK;
}

// ---- waterfall image and autolevel on the device (zfb_image.cuh) -----------
static int image_params(zfb_engine *e, int height, int scroll, int64_t rows_seen, ImageParams &p) {
    if (!e->ring.p || e->ring_W < 1) return fail(e, ZFB_ESTATE, "no ring (configure the engine or the ring first)");
    if (height < 1 || rows_seen < 0) return fail(e, ZFB_EINVAL, "waterfall image: bad height / rows_seen");
    int64_t have = rows_seen;
    if (have > height) have = height;
    if (have > e->ring_written) have = e->ring_written;
    if (have > e->ring_rows) have = e->ring_rows;
    p.ring = (const float *)e->ring.p;
    p.ring_rows = e->ring_rows;
    p.written = e->ring_written;
    p.W = e->ring_W;
    p.H = height;
    p.have = (int)have;
    p.nseen = (int)(rows_seen > (1 << 20) ? (1 << 20) : rows_seen);
    p.scroll = scroll;
    p.tick_step = e->ring_W / 10;
    p.newest_slot = (int)((e->ring_written + (int64_t)e->ring_rows - 1) % e->ring_rows);
    p.thr = nullptr;
    p.fscale = 1.f;
    p.foff = 0.f;
    p.wide_guess = 0;
    p.lut = nullptr;
    p.out = nullptr;
    return ZFB_OK;
}

// pyqtgraph's level mapping in its own double arithmetic, and the float
// thresholds at which its result steps (zfb_image.cuh: wf_level)
static int level_index(double v, double minlev, double scale) {
    double d = (v - minlev) * scale;
    if (!(d > 0.0)) d = 0.0;
    if (d > 255.0) d = 255.0;
    return (int)d;
}
static uint32_t float_ord(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
static float ord_float(uint32_t o) {
    const uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
    float f;
    memcpy(&f, &u, 4);
    return f;
}
static void level_thresholds(double minlev, double maxlev, float thr[257]) {
    const double scale = 256.0 / (maxlev - minlev);
    thr[0] = -INFINITY;
    thr[256] = INFINITY;
    uint32_t lo = float_ord(-INFINITY);                   // index(lo) = 0 < k
    for (int k = 1; k <= 255; ++k) {
        uint32_t a = lo, b = float_ord(INFINITY);         // index(a) < k <= index(b)
        while (b - a > 1) {
            const uint32_t m = a + (b - a) / 2;
            if (level_index((double)ord_float(m), minlev, scale) >= k) b = m; else a = m;
        }
        thr[k] = ord_float(b);
        lo = a;
    }
}

int zfb_ring_image(zfb_engine *e, int height, int scroll, int64_t rows_seen, int kind, double minlev, double maxlev,
                   const uint8_t *lut_rgba, void *out, int out_on_device) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    ImageParams p{};
    int rc = image_params(e, height, scroll, rows_seen, p);
    if (rc) return rc;
    if (!out) return fail(e, ZFB_EINVAL, "waterfall image: out is NULL");
    if (kind != ZFB_IMAGE_F32 && kind != ZFB_IMAGE_U8 && kind != ZFB_IMAGE_RGBA)
        return fail(e, ZFB_EINVAL, "waterfall image: unknown kind %d", kind);
    if (kind != ZFB_IMAGE_F32 && !(maxlev > minlev)) return fail(e, ZFB_EINVAL, "waterfall image: maxlev must exceed minlev");
    if (kind == ZFB_IMAGE_RGBA && !lut_rgba) return fail(e, ZFB_EINVAL, "waterfall image: RGBA needs a 256-entry table");
    CK(e, cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    const size_t px = (size_t)height * (size_t)e->ring_W;
    const size_t bytes = px * (kind == ZFB_IMAGE_U8 ? 1 : 4);
    if (kind != ZFB_IMAGE_F32) {
        if (!e->thr_valid || e->thr_levels[0] != minlev || e->thr_levels[1] != maxlev) {
            float thr[257];
            level_thresholds(minlev, maxlev, thr);
            rc = ensure(e, e->img_thr, sizeof thr);
            if (rc) return rc;
            CK(e, cudaMemcpyAsync(e->img_thr.p, thr, sizeof thr, cudaMemcpyHostToDevice, st));
            CK(e, cudaStreamSynchronize(st));             // thr lives on this stack frame
            e->counters[3] += sizeof thr;
            e->thr_levels[0] = minlev;
            e->thr_levels[1] = maxlev;
            e->thr_valid = true;
        }
        p.thr = (const float *)e->img_thr.p;
        const double scale = 256.0 / (maxlev - minlev);
        p.fscale = (float)scale;
        p.foff = (float)(-minlev * scale);
        // fp32 guess error <= (256 + 2|foff|) * 2^-23: stays below 1/4 for |foff| < 1e6
        p.wide_guess = (fabs(minlev * scale) < 1.0e6 && scale < 1.0e30) ? 0 : 1;
    }
    if (kind == ZFB_IMAGE_RGBA) {
        rc = ensure(e, e->img_lut, 256 * sizeof(unsigned int));
        if (rc) return rc;
        CK(e, cudaMemcpyAsync(e->img_lut.p, lut_rgba, 256 * sizeof(unsigned int), cudaMemcpyHostToDevice, st));
        e->counters[3] += 256 * sizeof(unsigned int);
        p.lut = (const unsigned int *)e->img_lut.p;
    }
    if (out_on_device) {
        p.out = out;
    } else {
        if (e->img_out.cap < bytes) CK(e, cudaStreamSynchronize(st));
        rc = ensure(e, e->img_out, bytes);
        if (rc) return rc;
        p.out = e->img_out.p;
    }
    const int per_cta = IMG_NT * IMG_U * 4;
    const dim3 grid((unsigned)((e->ring_W + per_cta - 1) / per_cta), (unsigned)height);
    const int pr = prof_begin(e, 19);
    if (kind == ZFB_IMAGE_F32) ZFB_LAUNCH(wf_image_kernel<IMG_F32>, grid, dim3(256), 0, st, p);
    else if (kind == ZFB_IMAGE_U8) ZFB_LAUNCH(wf_image_kernel<IMG_U8>, grid, dim3(256), 0, st, p);
    else ZFB_LAUNCH(wf_image_kernel<IMG_RGBA>, grid, dim3(256), 0, st, p);
    prof_end(e, pr);
    CK(e, cudaGetLastError());
    e->counters[2] += 1;
    if (!out_on_device) {
        CK(e, cudaMemcpyAsync(out, p.out, bytes, cudaMemcpyDeviceToHost, st));
        CK(e, cudaStreamSynchronize(st));
        e->counters[4] += bytes;
    }
    return ZFB_OK;
}

// numpy's _lerp (numpy/lib/_function_base_impl.py), as np.percentile's default
// 'linear' method applies it between the two neighbouring order statistics
static double np_lerp(double a, double b, double t) {
    const double d = b - a;
    double r = a + d * t;
    if (t >= 0.5) r = b - d * (1.0 - t);
    if (d == 0.0) r = a;
    return r;
}

int zfb_ring_quantiles(zfb_engine *e, int height, int scroll, int64_t rows_seen, const double *q, int nq,
                       double *out_values, int64_t *out_count) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    SelectParams s{};
    int rc = image_params(e, height, scroll, rows_seen, s.img);
    if (rc) return rc;
    if (!q || !out_values || nq < 1 || nq > 64) return fail(e, ZFB_EINVAL, "quantiles: bad arguments");
    for (int i = 0; i < nq; ++i)
        if (!(q[i] >= 0.0 && q[i] <= 1.0)) return fail(e, ZFB_EINVAL, "quantiles: q[%d] outside [0, 1]", i);
    CK(e, cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    const size_t hbytes = (size_t)SEL_TARGETS * SEL_BINS * sizeof(unsigned int);
    rc = ensure(e, e->sel_hist, hbytes);
    if (rc) return rc;
    s.hist = (unsigned int *)e->sel_hist.p;
    // enough CTAs to fill the GPU, whole rows per CTA
    int ctas = e->sm_count * 8;
    if (ctas > height) ctas = height;
    s.rows_per_cta = (height + ctas - 1) / ctas;
    ctas = (height + s.rows_per_cta - 1) / s.rows_per_cta;
    std::vector<unsigned int> hist((size_t)SEL_TARGETS * SEL_BINS);
    auto sweep = [&](int pass, int nt) -> int {
        s.pass = pass;
        s.ntargets = nt;
        CK(e, cudaMemsetAsync(s.hist, 0, hbytes, st));
        const int pr = prof_begin(e, 20);
        const size_t hb = (size_t)(pass == 0 ? 1 : nt) * SEL_BINS * sizeof(unsigned int);
        if (pass == 0) ZFB_LAUNCH(wf_select_kernel<0>, dim3((unsigned)ctas), dim3(256), hb, st, s);
        else if (pass == 1) ZFB_LAUNCH(wf_select_kernel<1>, dim3((unsigned)ctas), dim3(256), hb, st, s);
        else ZFB_LAUNCH(wf_select_kernel<2>, dim3((unsigned)ctas), dim3(256), hb, st, s);
        prof_end(e, pr);
        CK(e, cudaGetLastError());
        e->counters[2] += 1;
        CK(e, cudaMemcpyAsync(hist.data(), s.hist, hbytes, cudaMemcpyDeviceToHost, st));
        CK(e, cudaStreamSynchronize(st));
        e->counters[4] += hbytes;
        return ZFB_OK;
    };
    // pass 0 is shared by every rank: key bits 30..20 (bit 31 is clear for every value below zero)
    rc = sweep(0, 1);
    if (rc) return rc;
    std::vector<unsigned long long> cum0(SEL_BINS + 1, 0);
    for (int b = 0; b < SEL_BINS; ++b) cum0[b + 1] = cum0[b] + hist[b];
    const long long n = (long long)cum0[SEL_BINS];
    if (out_count) *out_count = n;
    if (n == 0) {
        for (int i = 0; i < nq; ++i) out_values[i] = NAN;     // np.percentile of an empty selection
        return ZFB_OK;
    }
    // ranks np.percentile(method='linear') needs: floor and floor+1 of (n-1)*q
    std::vector<long long> ranks;
    std::vector<double> gamma(nq);
    std::vector<int> lo_at(nq), hi_at(nq);
    auto rank_slot = [&](long long r) {
        for (size_t i = 0; i < ranks.size(); ++i) if (ranks[i] == r) return (int)i;
        ranks.push_back(r);
        return (int)ranks.size() - 1;
    };
    for (int i = 0; i < nq; ++i) {
        const double virt = (double)(n - 1) * q[i];
        long long k = (long long)floor(virt);
        if (k > n - 1) k = n - 1;
        if (k < 0) k = 0;
        gamma[i] = virt - (double)k;
        lo_at[i] = rank_slot(k);
        hi_at[i] = rank_slot(k + 1 < n ? k + 1 : n - 1);
    }
    std::vector<float> value(ranks.size());
    for (size_t base = 0; base < ranks.size(); base += SEL_TARGETS) {
        const int nt = (int)std::min<size_t>(SEL_TARGETS, ranks.size() - base);
        long long resid[SEL_TARGETS];
        unsigned int key[SEL_TARGETS];
        for (int t = 0; t < nt; ++t) {
            const long long r = ranks[base + t];
            int b = 0;
            while (cum0[b + 1] <= (unsigned long long)r) ++b;
            key[t] = (unsigned int)b;
            resid[t] = r - (long long)cum0[b];
        }
        for (int pass = 1; pass <= 2; ++pass) {
            // neighbouring ranks usually share a prefix: one histogram per distinct prefix
            int slot_of[SEL_TARGETS], nu = 0;
            for (int t = 0; t < nt; ++t) {
                int u = 0;
                while (u < nu && s.prefix[u] != key[t]) ++u;
                if (u == nu) s.prefix[nu++] = key[t];
                slot_of[t] = u;
            }
            rc = sweep(pass, nu);
            if (rc) return rc;
            const int bins = pass == 1 ? 2048 : 512;
            for (int t = 0; t < nt; ++t) {
                const unsigned int *ht = hist.data() + (size_t)slot_of[t] * SEL_BINS;
                long long acc = 0;
                int b = 0;
                while (b < bins - 1 && acc + ht[b] <= resid[t]) acc += ht[b++];
                resid[t] -= acc;
                key[t] = (key[t] << (pass == 1 ? 11 : 9)) | (unsigned int)b;
            }
        }
        for (int t = 0; t < nt; ++t) value[base + t] = wf_unkey(key[t]);
    }
    for (int i = 0; i < nq; ++i)
        out_values[i] = np_lerp((double)value[(size_t)lo_at[i]], (double)value[(size_t)hi_at[i]], gamma[i]);
    return ZFB_OK;
}

int zfb_samples_create(zfb_engine *e, int64_t capacity_samples, int dtype) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (capacity_samples < 1 || capacity_samples > (1ll << 31))
        return fail(e, ZFB_EINVAL, "sample ring capacity out of range");
    if (dtype != ZFB_DTYPE_C64 && dtype != ZFB_DTYPE_U8 && dtype != ZFB_DTYPE_CS16)
        return fail(e, ZFB_EINVAL, "unknown dtype %d", dtype);
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    CK(e, cudaStreamSynchronize(e->copy_stream));
    const size_t bytes = (size_t)capacity_samples * dtype_bytes(dtype);
    if (e->sr_host) { CK(e, cudaFreeHost(e->sr_host)); e->sr_host = nullptr; }
    CK(e, cudaMallocHost(&e->sr_host, bytes));
    memset(e->sr_host, 0, bytes);
    for (int i = 0; i < 2; ++i) {
        int rc = ensure(e, e->sr_dev[i], bytes);
        if (rc) return rc;
        CK(e, cudaMemsetAsync(e->sr_dev[i].p, 0, bytes, e->stream));
        if (!e->sr_free[i]) CK(e, cudaEventCreateWithFlags(&e->sr_free[i], cudaEventDisableTiming));
        e->sr_free_pending[i] = false;
    }
    if (!e->sr_copied) CK(e, cudaEventCreateWithFlags(&e->sr_copied, cudaEventDisableTiming));
    CK(e, cudaStreamSynchronize(e->stream));
    e->sr_cap = capacity_samples;
    e->sr_dtype = dtype;
    e->sr_active = 0;
    e->sr_copy_pending = false;
    return ZFB_OK;
}

void *zfb_samples_host_ptr(zfb_engine *e) { return e ? e->sr_host : nullptr; }

int zfb_samples_begin_write(zfb_engine *e, int64_t offset, int64_t n) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->sr_host) return fail(e, ZFB_ESTATE, "no sample ring (zfb_samples_create)");
    if (offset < 0 || n < 0 || offset + n > e->sr_cap) return fail(e, ZFB_EINVAL, "sample span out of range");
    // copies are enqueued in order on one stream: once the newest has finished, none reads host memory
    if (e->sr_copy_pending) {
        CK(e, cudaSetDevice(e->device));
        CK(e, cudaEventSynchronize(e->sr_copied));
        e->sr_copy_pending = false;
    }
    return ZFB_OK;
}

int zfb_samples_commit(zfb_engine *e, int64_t offset, int64_t n) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->sr_host) return fail(e, ZFB_ESTATE, "no sample ring (zfb_samples_create)");
    if (offset < 0 || n < 0 || offset + n > e->sr_cap) return fail(e, ZFB_EINVAL, "sample span out of range");
    if (n == 0) return ZFB_OK;
    CK(e, cudaSetDevice(e->device));
    const size_t esz = dtype_bytes(e->sr_dtype);
    const int m = e->sr_active;
    if (e->sr_free_pending[m]) {       // a kernel may still be reading this mirror
        CK(e, cudaStreamWaitEvent(e->copy_stream, e->sr_free[m], 0));
        e->sr_free_pending[m] = false;
    }
    CK(e, cudaMemcpyAsync((char *)e->sr_dev[m].p + (size_t)offset * esz, (const char *)e->sr_host + (size_t)offset * esz,
                          (size_t)n * esz, cudaMemcpyHostToDevice, e->copy_stream));
    CK(e, cudaEventRecord(e->sr_copied, e->copy_stream));
    e->sr_copy_pending = true;
    e->counters[3] += (size_t)n * esz;
    return ZFB_OK;
}

int zfb_samples_process(zfb_engine *e, float *h_row) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!e->configured) return fail(e, ZFB_ESTATE, "process: engine is not configured");
    if (!e->sr_host) return fail(e, ZFB_ESTATE, "no sample ring (zfb_samples_create)");
    if (!h_row) return fail(e, ZFB_EINVAL, "process: h_row is NULL");
    if (e->cfg.dtype != e->sr_dtype) return fail(e, ZFB_EINVAL, "configured dtype differs from the sample ring's");
    if ((int64_t)e->cfg.frame_len > e->sr_cap) return fail(e, ZFB_EINVAL, "frame_len exceeds the sample ring");
    CK(e, cudaSetDevice(e->device));
    const int m = e->sr_active;
    if (e->sr_copy_pending) CK(e, cudaStreamWaitEvent(e->stream, e->sr_copied, 0));
    int rc = ensure(e, e->rows_tmp, (size_t)e->W * sizeof(float));
    if (rc) return rc;
    rc = run_group(e, e->sr_dev[m].p, 1, (float *)e->rows_tmp.p);
    if (rc) return rc;
    CK(e, cudaEventRecord(e->sr_free[m], e->stream));
    e->sr_free_pending[m] = true;
    e->sr_active = m ^ 1;                          // the producer moves to the other mirror
    if (e->h_rows_cap < (size_t)e->W * sizeof(float)) {
        if (e->h_rows) CK(e, cudaFreeHost(e->h_rows));
        e->h_rows = nullptr;
        CK(e, cudaMallocHost(&e->h_rows, (size_t)e->W * sizeof(float)));
        e->h_rows_cap = (size_t)e->W * sizeof(float);
    }
    CK(e, cudaMemcpyAsync(e->h_rows, e->rows_tmp.p, (size_t)e->W * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    memcpy(h_row, e->h_rows, (size_t)e->W * sizeof(float));
    e->counters[4] += (size_t)e->W * sizeof(float);
    return ZFB_OK;
}

// ---- taper design and preview on the device (SURVEY 8f.4; zfb_taper.cuh) -------------------
int zfb_taper_design(zfb_engine *e, int kind, double p0, double p1, int n, int periodic, double *h_out) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (kind < 0 || kind >= TAPER_COUNT) return fail(e, ZFB_EINVAL, "taper kind %d is not designed on the device", kind);
    if (n < 1 || n > (1 << 24) || !h_out) return fail(e, ZFB_EINVAL, "taper design: bad arguments");
    if ((kind == TAPER_GAUSSIAN && !(p0 > 0.0)) || (kind == TAPER_GENERAL_GAUSSIAN && !(p1 > 0.0)) ||
        (kind == TAPER_EXPONENTIAL && !(p1 > 0.0)) || (kind == TAPER_KAISER && !(p0 == p0)))
        return fail(e, ZFB_EINVAL, "taper design: bad shape parameter");
    CK(e, cudaSetDevice(e->device));
    int rc = ensure(e, e->taper_buf, (size_t)n * sizeof(double));
    if (rc) return rc;
    TaperParams tp{};
    tp.kind = kind;
    tp.n = n;
    tp.M = periodic ? n + 1 : n;
    tp.p0 = p0;
    tp.p1 = p1;
    tp.out = (double *)e->taper_buf.p;
    ZFB_LAUNCH(taper_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, e->stream, tp);
    CK(e, cudaGetLastError());
    e->counters[2] += 1;
    CK(e, cudaMemcpyAsync(h_out, e->taper_buf.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->counters[4] += (size_t)n * sizeof(double);
    return ZFB_OK;
}

int zfb_taper_preview(zfb_engine *e, const double *taper, int ntaps, int nfft, float *h_db_out) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    if (!taper || !h_db_out || ntaps < 1 || ntaps > 65536 || nfft < ntaps || nfft > (1 << 20))
        return fail(e, ZFB_EINVAL, "taper preview: bad arguments");
    CK(e, cudaSetDevice(e->device));
    const size_t need = (size_t)ntaps * sizeof(double) + (size_t)nfft * sizeof(double) + (size_t)nfft * sizeof(float);
    int rc = ensure(e, e->taper_buf, need);
    if (rc) return rc;
    double *d_taper = (double *)e->taper_buf.p;
    double *d_mag = d_taper + ntaps;
    float *d_db = (float *)(d_mag + nfft);
    CK(e, cudaMemcpyAsync(d_taper, taper, (size_t)ntaps * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));          // the caller's table may be pageable / short-lived
    ZFB_LAUNCH(taper_spectrum_kernel, dim3((unsigned)((nfft + 255) / 256)), dim3(256), 0, e->stream,
               (const double *)d_taper, ntaps, nfft, d_mag);
    ZFB_LAUNCH(taper_db_kernel, dim3(1), dim3(256), 0, e->stream, (const double *)d_mag, nfft, d_db);
    CK(e, cudaGetLastError());
    e->counters[2] += 2;
    e->counters[3] += (size_t)ntaps * sizeof(double);
    CK(e, cudaMemcpyAsync(h_db_out, d_db, (size_t)nfft * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->counters[4] += (size_t)nfft * sizeof(float);
    return ZFB_OK;
}

int zfb_alloc_pinned(size_t bytes, void **out) {
    if (!out) return ZFB_EINVAL;
    *out = nullptr;
    cudaError_t st = cudaMallocHost(out, bytes ? bytes : 1);
    if (st != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, ZFB_ENOMEM, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(st));
    }
    return ZFB_OK;
}

int zfb_free_pinned(void *p) {
    if (!p) return ZFB_OK;
    return cudaFreeHost(p) == cudaSuccess ? ZFB_OK : ZFB_ECUDA;
}

int zfb_set_profiling(zfb_engine *e, int on) {
    if (!e) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    e->profiling = on != 0;
    return ZFB_OK;
}

int zfb_get_profile(zfb_engine *e, double ms_out[ZFB_PROF_CLASSES], uint64_t launches_out[ZFB_PROF_CLASSES]) {
    if (!e || !ms_out || !launches_out) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    join_pending_work(e);
    CK(e, cudaSetDevice(e->device));
    CK(e, cudaStreamSynchronize(e->stream));
    for (int c = 0; c < ZFB_PROF_CLASSES; ++c) { ms_out[c] = 0.0; launches_out[c] = 0; }
    // the lanes' kernels belong to this engine's profile (e->stream has waited for all of them)
    for (zfb_engine *x : {e, e->lane[0], e->lane[1]}) {
        if (!x) continue;
        if (x != e) cudaStreamSynchronize(x->stream);
        for (auto &r : x->prof_used) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess && r.cls >= 0 && r.cls < ZFB_PROF_CLASSES) {
                ms_out[r.cls] += (double)ms;
                launches_out[r.cls] += 1;
            }
            x->prof_free.push_back(r);
        }
        x->prof_used.clear();
    }
    cudaGetLastError();
    return ZFB_OK;
}

int zfb_get_counters(const zfb_engine *e, uint64_t out5[5]) {
    if (!e || !out5) return ZFB_EINVAL;
    std::lock_guard<std::mutex> lk(e->mu);
    memcpy(out5, e->counters, sizeof e->counters);
    return ZFB_OK;
}

}  // extern "C"
