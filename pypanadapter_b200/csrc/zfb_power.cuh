// Channel power and occupied bandwidth of column bands of the engine's rows (DESIGN 3.11).
//
// A spectrum analyser's measurement menu -- channel power, adjacent-channel leakage, 99 %
// occupied bandwidth, and how each of them moves over time -- over every row the engine
// finishes, without reading rows back.  One launch per group, right behind the other row
// updates on the stream that finished the rows:
//
//   power_measure_kernel  p[c] = row value (linear rows) or 10^(v/20) in fp64.  A band of at most
//                         PW_NARROW columns is measured by one warp per (row, band), PW_NW of them
//                         per CTA; a wider band by one whole CTA per (row, band).  Each thread sums
//                         its contiguous segment of the band serially; a butterfly scan per warp
//                         (and, in a CTA, a serial pass over the warp totals) gives every
//                         segment's prefix and the band total; the thread whose segment holds an
//                         OBW target rescans it for the crossing.  The band's power is fs/N times
//                         the total; both targets are fractions of the same total.  Results go to
//                         the group's scratch and to the log ring (only the newest log_rows rows
//                         of the group, so no slot is written twice).  The last CTA to finish (an
//                         integer completion counter, reset by that CTA) folds the group's powers
//                         into the per-band max / min / fp64 sum, strictly in frame order.
//
// The shape (warp or CTA) and the segment length (ceil(width / 32) or ceil(width / PW_NT)) depend
// on the band's width and compile-time constants only, never on the group, grid or position in
// the stream, and no floating-point atomics are used.  So every value is bit-identical however
// the frames are cut into calls, groups, host or device paths or pipelined batches.
#pragma once
#include "zfb_common.cuh"

namespace zfb {

constexpr int PW_NT = 512;
constexpr int PW_NW = PW_NT / 32;
constexpr int PW_MAX_BANDS = 64;
constexpr int PW_NARROW = 2048;                     // widest band measured by one warp
constexpr int PW_TILE = 2048;                       // powers per tile of the fold (doubles)

struct PowerParams {
    const float *rows;        // [nframes][W] finished rows
    const int *bands;         // [nbands][2]: first, end column
    const int *narrow;        // [nnarrow] indices of the bands of <= PW_NARROW columns
    const int *wide;          // [nwide] indices of the others
    int nframes, W, nbands, nnarrow, nwide, linear;
    double delta;             // fs / N: the density's bin width in Hz
    double q_lo, q_hi;        // (1 - q) / 2 and (1 + q) / 2 of the OBW fraction q
    double *meas;             // [nframes][nbands][3]: power, obw_lo, obw_hi of this group
    double *log;              // [log_rows][nbands][3], row k at slot k mod log_rows
    int log_rows;             // <= 2^26
    int slot0;                // slot of the group's first row: its index since the set started empty, mod log_rows
    double *summary;          // [nbands][3]: max, min, sum of power
    int have;                 // the summary holds at least one row (host-side knowledge, launch order)
    unsigned *done;           // CTAs of this launch that have finished; 0 between launches
};

// 10^(v/20) as exp10(v * 0.05): within 1e-14 of exp10(v / 20.0), whose division's slow-path call
// would make the kernel spill around it.  -inf (a DC-only frame): 0
__device__ __forceinline__ double pw_lin(float v, int linear) {
    return linear ? (double)v : exp10((double)v * 0.05);
}

// Column of the crossing of `target` in the segment [lo, hi) whose prefix is P: the first
// positive column j with P + (its partial sum through j) >= target, at j + (target - C(j)) / p[j].
// The partial sums repeat the segment's own serial sum bit for bit (both add with __dadd_rn,
// which is never fused), so a segment with P + s >= target always crosses.  Without a crossing
// (the fall-back segment, when rounding put the target past every prefix) the end of its last
// positive column.
__device__ __forceinline__ double pw_edge(const float *x, int lo, int hi, int linear, double P, double target) {
    double acc = 0.0;
    int jlast = lo - 1;
    for (int j = lo; j < hi; ++j) {
        const double v = pw_lin(x[j], linear);
        const double next = __dadd_rn(acc, v);
        if (v > 0.0) {
            if (P + next >= target) return (double)j + fmax(0.0, (target - (P + acc)) / v);
            jlast = j;
        }
        acc = next;
    }
    return (double)(jlast + 1);
}

__device__ __forceinline__ double pw_segment_sum(const float *x, int lo, int hi, int linear) {
    double s = 0.0;
    for (int j = lo; j < hi; ++j) s = __dadd_rn(s, pw_lin(x[j], linear));     // never fused into exp10's last step
    return s;
}

// exclusive prefix of s within the warp and the warp total: a butterfly with a fixed pairing
// (a + b == b + a, so both partners hold the same pair total, and every lane the same total)
__device__ __forceinline__ void pw_warp_scan(double s, int lane, double &ex, double &tot) {
    tot = s;
    ex = 0.0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane & o) ex += y;
        tot += y;
    }
}

__device__ __forceinline__ int pw_warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// one measurement of row f, band b to the group's scratch and, for the newest log_rows rows, the log
__device__ __forceinline__ void pw_store(const PowerParams &p, int f, int b, int k, double v) {
    p.meas[((size_t)f * p.nbands + b) * 3 + k] = v;
    if (f >= p.nframes - p.log_rows)
        p.log[((size_t)((p.slot0 + f) % p.log_rows) * p.nbands + b) * 3 + k] = v;
}

// NaN-propagating max / min, as numpy's
__device__ __forceinline__ double pw_max(double a, double v) { return (v > a || v != v) ? v : a; }
__device__ __forceinline__ double pw_min(double a, double v) { return (v < a || v != v) ? v : a; }

// grid: nframes * nwide CTAs (one per row and wide band), then ceil(nframes * nnarrow / PW_NW)
// CTAs of PW_NW (row, narrow band) warps
__global__ void __launch_bounds__(PW_NT) power_measure_kernel(const PowerParams p) {
    __shared__ double wsum[PW_NW];
    __shared__ int wsel[3][PW_NW];
    __shared__ int is_last;
    __shared__ double tile[PW_TILE];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int wide_ctas = p.nframes * p.nwide;
    // this thread's part of one (row f, band b): segment [lo, hi) of the band's columns x, its sum
    // s and prefix P, the band total; win0 / win1: it holds the lower / upper OBW target; lead:
    // it writes the power
    int f = -1, b = 0, first = 0, lo = 0, hi = 0;
    const float *x = p.rows;
    double P = 0.0, total = 0.0;
    bool win0 = false, win1 = false, lead = false;
    if ((int)blockIdx.x < wide_ctas) {
        // one band of more than PW_NARROW columns: the whole CTA, segments of ceil(width / PW_NT)
        f = blockIdx.x / p.nwide;
        b = p.wide[blockIdx.x % p.nwide];
        first = p.bands[2 * b];
        const int n = p.bands[2 * b + 1] - first;
        const int S = (n + PW_NT - 1) / PW_NT;
        lo = min(n, t * S);
        hi = min(n, lo + S);
        x = p.rows + (size_t)f * p.W + first;
        const double s = pw_segment_sum(x, lo, hi, p.linear);
        double ex, tot;
        pw_warp_scan(s, lane, ex, tot);
        if (lane == 0) wsum[warp] = tot;
        __syncthreads();
        double base = 0.0;
        for (int w = 0; w < PW_NW; ++w) {
            if (w < warp) base += wsum[w];
            total += wsum[w];
        }
        P = base + ex;
        const bool ok = total > 0.0;                           // false for 0 (and NaN)
        // the first segment that reaches each target; the last positive segment as the fall-back
        int c0 = pw_warp_min((ok && s > 0.0 && P + s >= p.q_lo * total) ? t : PW_NT);
        int c1 = pw_warp_min((ok && s > 0.0 && P + s >= p.q_hi * total) ? t : PW_NT);
        int c2 = pw_warp_min((ok && s > 0.0) ? PW_NT - 1 - t : PW_NT);   // min of this: the highest such t
        if (lane == 0) {
            wsel[0][warp] = c0;
            wsel[1][warp] = c1;
            wsel[2][warp] = c2;
        }
        __syncthreads();
        c0 = c1 = c2 = PW_NT;
        for (int w = 0; w < PW_NW; ++w) {
            c0 = min(c0, wsel[0][w]);
            c1 = min(c1, wsel[1][w]);
            c2 = min(c2, wsel[2][w]);
        }
        const int fall = PW_NT - 1 - c2;                       // -1 when no segment is positive
        win0 = t == (c0 == PW_NT ? fall : c0);
        win1 = t == (c1 == PW_NT ? fall : c1);
        lead = t == 0;
    } else {
        // one band of at most PW_NARROW columns per warp, segments of ceil(width / 32)
        const int k = ((int)blockIdx.x - wide_ctas) * PW_NW + warp;
        if (k < p.nframes * p.nnarrow) {                       // warp-uniform
            f = k / p.nnarrow;
            b = p.narrow[k % p.nnarrow];
            first = p.bands[2 * b];
            const int n = p.bands[2 * b + 1] - first;
            const int S = (n + 31) / 32;
            lo = min(n, lane * S);
            hi = min(n, lo + S);
            x = p.rows + (size_t)f * p.W + first;
            const double s = pw_segment_sum(x, lo, hi, p.linear);
            pw_warp_scan(s, lane, P, total);
            const bool ok = total > 0.0;
            const int c0 = pw_warp_min((ok && s > 0.0 && P + s >= p.q_lo * total) ? lane : 32);
            const int c1 = pw_warp_min((ok && s > 0.0 && P + s >= p.q_hi * total) ? lane : 32);
            const int fall = 31 - pw_warp_min((ok && s > 0.0) ? 31 - lane : 32);
            win0 = lane == (c0 == 32 ? fall : c0);
            win1 = lane == (c1 == 32 ? fall : c1);
            lead = lane == 0;
        }
    }
    const bool ok = total > 0.0;
    if (f >= 0) {
#pragma unroll 1
        for (int e = 1; e <= 2; ++e)                           // one rescan site: one division
            if (ok && (e == 1 ? win0 : win1))
                pw_store(p, f, b, e, (double)first + pw_edge(x, lo, hi, p.linear, P, (e == 1 ? p.q_lo : p.q_hi) * total));
        if (lead) {
            pw_store(p, f, b, 0, p.delta * total);
            if (!ok) {
                pw_store(p, f, b, 1, NAN);
                pw_store(p, f, b, 2, NAN);
            }
        }
    }
    const bool wrote = f >= 0 && (lead || (ok && (win0 || win1)));
    if (wrote) __threadfence();
    __syncthreads();
    if (t == 0) is_last = atomicAdd(p.done, 1u) == gridDim.x - 1u;
    __syncthreads();
    if (!is_last) return;
    // every CTA's results are visible: the summary, in frame order.  The group's powers come in
    // through shared memory a tile at a time, all threads loading at once, so the nbands serial
    // walkers wait on one L2 round trip per tile, not one per row
    __threadfence();
    const int rows_per_tile = PW_TILE / p.nbands;
    double mx = -INFINITY, mn = INFINITY, sum = 0.0;
    if (t < p.nbands && p.have) {
        mx = p.summary[3 * t];
        mn = p.summary[3 * t + 1];
        sum = p.summary[3 * t + 2];
    }
    for (int g0 = 0; g0 < p.nframes; g0 += rows_per_tile) {
        const int nv = min(rows_per_tile, p.nframes - g0) * p.nbands;
        for (int i = t; i < nv; i += PW_NT) tile[i] = __ldcg(p.meas + ((size_t)g0 * p.nbands + i) * 3);
        __syncthreads();
        if (t < p.nbands)
#pragma unroll 8
            for (int i = t; i < nv; i += p.nbands) {
                const double v = tile[i];
                mx = pw_max(mx, v);
                mn = pw_min(mn, v);
                sum += v;
            }
        __syncthreads();
    }
    if (t < p.nbands) {
        p.summary[3 * t] = mx;
        p.summary[3 * t + 1] = mn;
        p.summary[3 * t + 2] = sum;
    }
    if (t == 0) *p.done = 0u;
}

}  // namespace zfb
