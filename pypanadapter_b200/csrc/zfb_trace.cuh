// Max-hold, min-hold and power-average traces over the engine's rows, and peak
// markers on any row-shaped vector (DESIGN 3.8).
//
// The reference draws each row as it comes (spectrum_plot.setData, S:2130) and
// keeps nothing across rows; a spectrum analyser's hold and average traces and
// its peak markers would be numpy on the host over rows read back one by one.
// Here the traces are a per-column state on the device, updated right behind
// the finalisation of every launch group, and a peak query copies back only
// the markers.
//
//   trace_update_kernel  LAST / MAX (fmaxf) / MIN (fminf) / fp64 sum of linear power,
//                        strictly in frame order per column: batch independent
//   trace_avg_kernel     the AVG trace in row units (sum / count, dB20 unless linear)
//   trace_peaks_kernel   scipy.signal.find_peaks(x, height, distance) and the k highest
//                        peaks, with a parabolic offset per peak
#pragma once
#include "zfb_common.cuh"

namespace zfb {

// state of a trace set: [W] doubles, then [4][W] floats (LAST, MAX, MIN, AVG read-out)
struct TraceParams {
    const float *rows;        // [nframes][W] finished rows
    int    nframes, W;
    int    linear;            // 1: rows are linear power; 0: dB20 (20 log10 P)
    int    have;              // the state holds at least one row (host-side knowledge, launch order)
    double *sum;              // [W]
    float  *last, *mx, *mn;   // [W] each
};

// one CTA owns TR_COLS columns, as ema_rows_kernel does: all threads load a tile of
// rows into shared memory (and convert dB20 to linear power in parallel), the first
// TR_COLS threads walk it in frame order, the state goes back to memory once
constexpr int TR_COLS = 4;
constexpr int TR_NT = 512;
constexpr int TR_CH = 4;
constexpr int TR_FPP = TR_NT / TR_COLS;       // frames per pass of the CTA
constexpr int TR_FR = TR_FPP * TR_CH;         // frames per tile

__global__ void __launch_bounds__(TR_NT) trace_update_kernel(const TraceParams p) {
    __shared__ float tv[TR_FR * TR_COLS];
    __shared__ double tl[TR_FR * TR_COLS];
    const int c = threadIdx.x % TR_COLS, fs = threadIdx.x / TR_COLS;
    const int col = blockIdx.x * TR_COLS + c;
    const bool ok = col < p.W;
    const bool walker = threadIdx.x < TR_COLS;
    // an empty state is NaN for MAX / MIN: fmaxf / fminf then take the first row as it is
    float last = 0.f, mx = NAN, mn = NAN;
    double sum = 0.0;
    if (walker && ok && p.have) {
        last = p.last[col];
        mx = p.mx[col];
        mn = p.mn[col];
        sum = p.sum[col];
    }
    for (int f0 = 0; f0 < p.nframes; f0 += TR_FR) {
        const int n = min(TR_FR, p.nframes - f0);
#pragma unroll
        for (int k = 0; k < TR_CH; ++k) {
            const int i = fs + k * TR_FPP;
            if (ok && i < n) {
                const float v = p.rows[(size_t)(f0 + i) * p.W + col];
                tv[i * TR_COLS + c] = v;
                tl[i * TR_COLS + c] = p.linear ? (double)v : exp10((double)v / 20.0);
            }
        }
        __syncthreads();
        if (walker && ok) {
#pragma unroll 8
            for (int i = 0; i < n; ++i) {
                const float v = tv[i * TR_COLS + c];
                mx = fmaxf(mx, v);
                mn = fminf(mn, v);
                sum += tl[i * TR_COLS + c];
            }
            last = tv[(n - 1) * TR_COLS + c];
        }
        __syncthreads();
    }
    if (walker && ok && p.nframes > 0) {
        p.last[col] = last;
        p.mx[col] = mx;
        p.mn[col] = mn;
        p.sum[col] = sum;
    }
}

__global__ void __launch_bounds__(256) trace_avg_kernel(const double *sum, long long count, int W, int linear,
                                                        float *out) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= W) return;
    const double m = sum[col] / (double)count;
    out[col] = linear ? (float)m : (float)(20.0 * log10(m));
}

// ---- peak markers -----------------------------------------------------------
constexpr int PK_MAX = 64;                    // most peaks one query returns
constexpr int PK_NT = 1024;
constexpr int PK_MAX_N = 1 << 18;             // the widest row (crop=None at N = 262144)

// results: offsets first (8-byte aligned), then values, columns and the count; the
// candidate flags (one byte per element) follow in the same scratch
struct PeakOut {
    double offset[PK_MAX];
    float  value[PK_MAX];
    int    column[PK_MAX];
    int    count;
};

struct PeakParams {
    const float *x;
    int    n, k, distance;
    int    use_height;
    float  height;            // x[peak] >= height (scipy compares the float row values)
    PeakOut *out;
    unsigned char *flag;      // [n] scratch: 1 = surviving candidate
};

// a is a better marker than b: higher value, ties to the lower column; col < 0 = none
__device__ __forceinline__ bool pk_better(float va, int ca, float vb, int cb) {
    if (ca < 0) return false;
    if (cb < 0) return true;
    return va > vb || (va == vb && ca < cb);
}

// One CTA.  Thread t owns the contiguous segment [t*S, (t+1)*S) of the vector.
//   1. candidates: scipy's _local_maxima_1d -- a rise x[i-1] < x[i], the plateau of
//      values == x[i] after it (not past the second-to-last element), then a fall; the
//      marker is the plateau's midpoint.  A plateau is found by the thread that owns its
//      rising edge, which flags the midpoint (every flag has one writer).  NaN compares
//      false and so never rises, continues a plateau or falls.  Height filter here.
//   2. each thread keeps the best surviving candidate of its segment
//   3. k rounds: block argmax, then every candidate closer than `distance` to the
//      winner is removed; a thread rescans its segment only if its best was removed
//   4. parabolic offsets of the winners in fp64
__global__ void __launch_bounds__(PK_NT) trace_peaks_kernel(const PeakParams p) {
    __shared__ float wv[PK_NT / 32];
    __shared__ int wc[PK_NT / 32];
    __shared__ int win_c;
    __shared__ float win_v;
    __shared__ int taken[PK_MAX];
    const int t = threadIdx.x;
    const int n = p.n;
    const int S = (n + PK_NT - 1) / PK_NT;
    const int lo = min(n, t * S), hi = min(n, lo + S);
    const float *x = p.x;
    for (int j = lo; j < hi; ++j) p.flag[j] = 0;
    __syncthreads();
    for (int i = max(lo, 1); i < hi && i < n - 1; ++i) {
        const float v = x[i];
        if (!(x[i - 1] < v)) continue;
        int a = i + 1;
        while (a < n - 1 && x[a] == v) ++a;
        if (x[a] < v && (!p.use_height || v >= p.height)) p.flag[(i + a - 1) / 2] = 1;
    }
    __syncthreads();
    float bv = 0.f;
    int bc = -1;
    for (int j = lo; j < hi; ++j)
        if (p.flag[j] && pk_better(x[j], j, bv, bc)) { bv = x[j]; bc = j; }
    int found = 0;
    for (int r = 0; r < p.k; ++r) {
        float v = bv;
        int c = bc;
        for (int m = 16; m >= 1; m >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, m);
            const int oc = __shfl_xor_sync(0xffffffffu, c, m);
            if (pk_better(ov, oc, v, c)) { v = ov; c = oc; }
        }
        if ((t & 31) == 0) { wv[t >> 5] = v; wc[t >> 5] = c; }
        __syncthreads();
        if (t < 32) {
            v = wv[t];
            c = wc[t];
            for (int m = 16; m >= 1; m >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, v, m);
                const int oc = __shfl_xor_sync(0xffffffffu, c, m);
                if (pk_better(ov, oc, v, c)) { v = ov; c = oc; }
            }
            if (t == 0) { win_v = v; win_c = c; }
        }
        __syncthreads();
        const int pc = win_c;
        if (pc < 0) break;
        if (t == 0) taken[r] = pc;
        found = r + 1;
        // neighbours closer than `distance` (the winner itself included) leave the race
        const long long d = p.distance;
        const int a = (int)max((long long)lo, (long long)pc - d + 1);
        const int b = (int)min((long long)hi, (long long)pc + d);
        if (a < b) {
            for (int j = a; j < b; ++j) p.flag[j] = 0;
            if (bc >= a && bc < b) {
                bc = -1;
                for (int j = lo; j < hi; ++j)
                    if (p.flag[j] && pk_better(x[j], j, bv, bc)) { bv = x[j]; bc = j; }
            }
        }
        __syncthreads();
    }
    if (t < found) {
        const int j = taken[t];
        const double a = x[j - 1], b = x[j], c = x[j + 1];
        double off = 0.0;
        if (a != b && c != b && isfinite(a) && isfinite(b) && isfinite(c))
            off = 0.5 * (a - c) / (a - 2.0 * b + c);
        p.out->column[t] = j;
        p.out->value[t] = x[j];
        p.out->offset[t] = off;
    }
    if (t == 0) p.out->count = found;
}

}  // namespace zfb
