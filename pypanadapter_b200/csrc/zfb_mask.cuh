// Frequency-mask trigger over the engine's rows (DESIGN 3.10).
//
// A real-time spectrum analyser's frequency-mask trigger: every row the engine finishes is
// checked against an upper and a lower limit line; a row with at least min_cols violating
// columns is an event.  Events are logged in frame order on the device (the host never
// waits to learn how many rows triggered) and the first capture_slots of them keep the
// triggering frame's wire-format samples.  Three launches per group, right behind the
// other row updates on the stream that finished the rows:
//
//   mask_check_kernel    per (row, 2048-column chunk): violating columns, first, last and
//                        the worst column (largest excess, ties to the lower column)
//   mask_log_kernel      one CTA: merges the chunks of each row in column order, ranks the
//                        triggering rows by a block scan in frame order, appends their
//                        records at counter + rank, assigns capture slots, advances the
//                        counter.  No atomics decide any order: the log is batch independent.
//   mask_capture_kernel  (capture_slots > 0 only) copies the frames that got a slot, by
//                        byte tiles, correct for any alignment of source and destination
#pragma once
#include "zoomfft_b200.h"
#include "zfb_common.cuh"

namespace zfb {

constexpr int MK_NT = 256;
constexpr int MK_PER = 8;                           // columns per thread
constexpr int MK_CHUNK = MK_NT * MK_PER;            // columns per CTA
constexpr unsigned MK_COLKEY = 0xFFFFFu;            // > 2^18, the widest row

// A violating column's rank: excess bits (a positive float orders as its bit pattern) above
// the inverted column (ties to the lower column) and the side, so one 64-bit max reduces all
// three.  0: no violating column.
__device__ __forceinline__ unsigned long long mask_key(float excess, int col, int above) {
    return ((unsigned long long)__float_as_uint(excess) << 32) |
           (unsigned long long)(((MK_COLKEY - (unsigned)col) << 1) | (unsigned)above);
}

struct MaskPart {                 // one row's summary over one chunk of columns
    int ncols, first, last, pad_;
    unsigned long long key;
};

struct MaskCheckParams {
    const float *rows;            // [nframes][W] finished rows
    const float *lines;           // [2][W]: upper, then lower; NaN = that side off at that column
    int nframes, W, nchunks;
    MaskPart *part;               // [nframes][nchunks]
};

__device__ __forceinline__ void mask_merge(MaskPart &a, int n, int f, int l, unsigned long long k) {
    a.ncols += n;
    a.first = min(a.first, f);
    a.last = max(a.last, l);
    if (k > a.key) a.key = k;
}

// grid (nchunks, <= nframes): a CTA keeps its columns' limits in registers (read once) and
// walks rows blockIdx.y, blockIdx.y + gridDim.y, ...
__global__ void __launch_bounds__(MK_NT) mask_check_kernel(const MaskCheckParams p) {
    __shared__ MaskPart wsum[MK_NT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.x * MK_CHUNK + (int)threadIdx.x;
    float up[MK_PER], lo[MK_PER];
#pragma unroll
    for (int j = 0; j < MK_PER; ++j) {
        const int c = c0 + j * MK_NT;
        up[j] = c < p.W ? p.lines[c] : __uint_as_float(0x7fc00000u);
        lo[j] = c < p.W ? p.lines[p.W + c] : __uint_as_float(0x7fc00000u);
    }
    for (int f = blockIdx.y; f < p.nframes; f += gridDim.y) {
        const float *row = p.rows + (size_t)f * p.W;
        MaskPart s{0, 0x7fffffff, -1, 0, 0ull};
#pragma unroll
        for (int j = 0; j < MK_PER; ++j) {
            const int c = c0 + j * MK_NT;
            if (c >= p.W) break;
            const float v = row[c];
            const bool a = v > up[j], b = v < lo[j];          // NaN row value or limit: false
            if (a || b) {
                const float ea = a ? v - up[j] : 0.f, eb = b ? lo[j] - v : 0.f;
                const int above = (a && !(eb > ea)) ? 1 : 0;  // both sides (infinite lines): the larger, upper on a tie
                mask_merge(s, 1, c, c, mask_key(above ? ea : eb, c, above));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int n = __shfl_xor_sync(0xffffffffu, s.ncols, o);
            const int fi = __shfl_xor_sync(0xffffffffu, s.first, o);
            const int la = __shfl_xor_sync(0xffffffffu, s.last, o);
            const unsigned long long k = __shfl_xor_sync(0xffffffffu, s.key, o);
            mask_merge(s, n, fi, la, k);
        }
        if (lane == 0) wsum[warp] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            MaskPart t = wsum[0];
            for (int w = 1; w < MK_NT / 32; ++w) mask_merge(t, wsum[w].ncols, wsum[w].first, wsum[w].last, wsum[w].key);
            p.part[(size_t)f * p.nchunks + blockIdx.x] = t;
        }
        __syncthreads();                                      // wsum is rewritten for the next row
    }
}

constexpr int ML_NT = 512;

struct MaskCap { int frame, slot; };

struct MaskLogParams {
    const MaskPart *part;         // [nframes][nchunks] of mask_check_kernel
    const float *rows;            // [nframes][W]
    int nframes, nchunks, W;
    long long row0;               // index of the group's first row among the rows checked
    int min_cols, max_events, capture_slots, capture_samples, frame_len, dtype;
    unsigned long long *counter;  // events detected so far (stored or not)
    zfb_mask_event *events;       // [max_events]
    MaskCap *cap_list;            // [nframes]: (frame, slot) of the group's captures, in slot order
    int *ncap;                    // how many entries of cap_list are valid
};

// one CTA: ranks follow frame order, whatever the group's size or position in the stream
__global__ void __launch_bounds__(ML_NT) mask_log_kernel(const MaskLogParams p) {
    __shared__ int wtot[ML_NT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long base0 = *p.counter;
    unsigned long long base = base0;
    for (int t0 = 0; t0 < p.nframes; t0 += ML_NT) {
        const int f = t0 + (int)threadIdx.x;
        MaskPart s{0, 0x7fffffff, -1, 0, 0ull};
        if (f < p.nframes)
            for (int ch = 0; ch < p.nchunks; ++ch) {
                const MaskPart &q = p.part[(size_t)f * p.nchunks + ch];
                mask_merge(s, q.ncols, q.first, q.last, q.key);
            }
        const bool trig = f < p.nframes && s.ncols >= p.min_cols;
        unsigned m = trig ? (1u << lane) : 0u;                // the warp's trigger flags
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
        if (lane == 0) wtot[warp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < ML_NT / 32; ++w) {
            before += w < warp ? wtot[w] : 0;
            total += wtot[w];
        }
        if (trig) {
            const unsigned long long k = base + (unsigned long long)(before + __popc(m & ((1u << lane) - 1u)));
            const int slot = k < (unsigned long long)p.capture_slots ? (int)k : -1;
            if (k < (unsigned long long)p.max_events) {
                const unsigned lowk = (unsigned)s.key;
                const int worst = (int)(MK_COLKEY - (lowk >> 1));
                zfb_mask_event ev;
                ev.row = p.row0 + f;
                ev.ncols = s.ncols;
                ev.first_col = s.first;
                ev.last_col = s.last;
                ev.worst_col = worst;
                ev.value = p.rows[(size_t)f * p.W + worst];
                ev.excess = __uint_as_float((unsigned)(s.key >> 32));
                ev.above = (int)(lowk & 1u);
                ev.capture = slot;
                ev.capture_samples = slot >= 0 ? min(p.frame_len, p.capture_samples) : 0;
                ev.dtype = p.dtype;
                p.events[k] = ev;
            }
            if (slot >= 0) p.cap_list[k - base0] = MaskCap{f, slot};
        }
        base += (unsigned long long)total;
        __syncthreads();                                      // wtot is rewritten for the next tile
    }
    if (threadIdx.x == 0) {
        *p.counter = base;
        const unsigned long long cs = (unsigned long long)p.capture_slots;
        *p.ncap = base0 >= cs ? 0 : (int)((base < cs ? base : cs) - base0);
    }
}

constexpr int MC_NT = 256;
constexpr int MC_U = 16;                                      // 4-byte words per thread and tile
constexpr int MC_TILE = MC_NT * MC_U * 4;                     // bytes per tile

struct MaskCopyParams {
    const unsigned char *src;     // entry e reads src + frame * src_stride
    size_t src_stride;
    unsigned char *dst;           // ... and writes dst + slot * dst_stride
    size_t dst_stride;
    long long nbytes;             // bytes per entry
    const MaskCap *list;          // (frame, slot) per entry; NULL: entry e = (e, e)
    const int *nlist;             // entries of list (device); NULL: gridDim.y
};

// grid (tiles, entries): a CTA whose entry got no frame exits at once.  The destination is
// written in aligned 4-byte words; a word's four source bytes come from the two aligned words
// that hold them (__byte_perm), so neither side needs any alignment.  Only words that hold a
// byte of the copy are read; the at most two partial words at the ends go byte by byte.
__global__ void __launch_bounds__(MC_NT) mask_capture_kernel(const MaskCopyParams p) {
    int f = blockIdx.y, slot = blockIdx.y;
    if (p.list) {
        if ((int)blockIdx.y >= *p.nlist) return;
        f = p.list[blockIdx.y].frame;
        slot = p.list[blockIdx.y].slot;
    }
    const unsigned char *S = p.src + (size_t)f * p.src_stride;
    unsigned char *D = p.dst + (size_t)slot * p.dst_stride;
    const long long lead = (long long)((size_t)D & 3u);
    const long long n = p.nbytes, nwords = (lead + n + 3) / 4;
    for (long long w0 = (long long)blockIdx.x * (MC_TILE / 4); w0 < nwords; w0 += (long long)gridDim.x * (MC_TILE / 4)) {
        unsigned v[MC_U];
#pragma unroll
        for (int j = 0; j < MC_U; ++j) {
            const long long o = (w0 + threadIdx.x + j * MC_NT) * 4 - lead;   // copy offset of the word's first byte
            v[j] = 0u;
            if (o >= 0 && o + 4 <= n) {
                const size_t s = (size_t)(S + o);
                const unsigned sh = (unsigned)(s & 3u);
                const unsigned *a = (const unsigned *)(s - sh);
                const unsigned lo = a[0], hi = sh ? a[1] : 0u;
                v[j] = __byte_perm(lo, hi, 0x3210u + 0x1111u * sh);
            }
        }
#pragma unroll
        for (int j = 0; j < MC_U; ++j) {
            const long long o = (w0 + threadIdx.x + j * MC_NT) * 4 - lead;
            if (o >= 0 && o + 4 <= n) {
                *(unsigned *)(D + o) = v[j];
            } else if (o + 4 > 0 && o < n) {
                for (int b = 0; b < 4; ++b)
                    if (o + b >= 0 && o + b < n) D[o + b] = S[o + b];
            }
        }
    }
}

}  // namespace zfb
