// Welch PSD for FFT sizes that do not fit one CTA (N = 2^14 .. 2^18): a
// four-step FFT, N = N1 * N2, as two kernels per group of frames.
//
// Same reference lines as zfb_welch.cuh (scipy.signal.welch called from
// pypanadapter_spectrum.py:2111 / pypanadapter_thread.py:1536,1538); this is
// the path BASELINE.json's offline-waterfall config (65536-pt, Hann, 50 %
// overlap) and the N sweep up to 262144 take.
//
//   n = n1*N2 + n2,  k = k1 + N1*k2
//   col pass : for every n2, window, N1-point FFT over n1, times W_N^(n2*k1)
//              -> Y[seg][k1][n2] (scratch, sized to stay L2 resident)
//   row pass : for every k1, N2-point FFT over n2 -> X[k1 + N1*k2]; |X|^2 is
//              accumulated over the segments in registers.
// Each CTA owns a 4096-point tile = B sub-FFTs of length M (M*B = 4096), 512
// threads x 8 points, radix-8/4 Stockham passes through padded shared memory.
//
// detrend='constant' needs the segment mean before windowing, but a column
// tile only sees 1/16..1/64 of a segment.  FFT(w*(x-m)) = FFT(w*x) - m*FFT(w),
// so the col pass also emits per-tile sums of the raw samples and the row pass
// subtracts m * Wf[k] (Wf = FFT of the window, fp64 on the host) per segment.
#pragma once
#include "zfb_welch.cuh"

namespace zfb {

struct BigParams {
    const void   *in;          // [frames][in_stride]
    long long     in_stride;
    int           len;
    int           flip;
    int           log2N;
    int           hop;
    int           nseg;
    int           seg_per_split;
    int           nsplit;
    int           ntiles_col;  // col-pass tiles per segment
    const float  *window;      // N taps
    const float2 *twiddle;     // N entries exp(-2 pi i k / N)
    const float2 *winfft;      // N entries FFT(window)
    float2       *scratch;     // [frames][nseg][N]  (k1-major)
    float2       *partial;     // [frames][nseg][ntiles_col] raw sums
    float2       *means;       // [frames][nseg] segment means
    int           W;
    float        *pow_out;     // [frames][nsplit][W]
};

constexpr int BIG_TILE = 4096;
constexpr int BIG_THREADS = BIG_TILE / 8;

__host__ __device__ constexpr int big_stride(int M) { return (M + (M >> 4)) | 1; }
constexpr size_t big_smem(int M) { return (size_t)(BIG_TILE / M) * big_stride(M) * sizeof(float2); }

// M-point forward FFT of the 8 values v[q] = a[j + q*M/8] of one sub-FFT that
// lives at `sub` in shared memory; twiddles from the N-entry table.
template <int LM>
__device__ __forceinline__ void sub_fft(float2 (&v)[8], int j, float2 *sub, const float2 *tw, int log2N) {
    constexpr int M = 1 << LM;
    constexpr int NT = M / 8;
    static_assert(LM >= 7 && LM <= 9, "sub-FFT length");
    fft_pass<8, 8>(v, j, NT, log2N, 0, tw, sub, false, true);
    if (LM == 7) {
        fft_pass<4, 8>(v, j, NT, log2N, 3, tw, sub, false, true);
        fft_pass<4, 8>(v, j, NT, log2N, 5, tw, sub, true, true);
    } else if (LM == 8) {
        fft_pass<8, 8>(v, j, NT, log2N, 3, tw, sub, false, true);
        fft_pass<4, 8>(v, j, NT, log2N, 6, tw, sub, true, true);
    } else {
        fft_pass<8, 8>(v, j, NT, log2N, 3, tw, sub, false, true);
        fft_pass<8, 8>(v, j, NT, log2N, 6, tw, sub, true, true);
    }
}

template <int LM, int KIND>
__global__ void __launch_bounds__(BIG_THREADS) bigfft_col_kernel(const BigParams p) {
    constexpr int M = 1 << LM;            // N1
    constexpr int C = BIG_TILE / M;       // columns per tile
    constexpr int S = big_stride(M);
    ZFB_DYN_SMEM(smem_raw);
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    __shared__ float2 red[33];

    const int t = threadIdx.x;
    const int c = t % C, j = t / C;
    const int tile = blockIdx.x, s = blockIdx.y, frame = blockIdx.z;
    const int N = 1 << p.log2N;
    const int log2N2 = p.log2N - LM;
    const int n2 = tile * C + c;
    const size_t esz = (KIND == KIND_U8_RAW) ? 2 : 8;
    const char *frame_in = (const char *)p.in + (size_t)frame * (size_t)p.in_stride * esz;
    const int base = s * p.hop;

    float2 v[8];
    float2 sum = make_float2(0.f, 0.f);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int idx = ((j + q * (M / 8)) << log2N2) + n2;
        const float2 x = welch_fetch<KIND>(frame_in, base + idx, p.len, p.flip);
        const float w = __ldg(p.window + idx);
        sum = cadd(sum, x);
        v[q] = make_float2(x.x * w, x.y * w);
    }
    sum = block_sum<BIG_THREADS>(sum, t, red);
    const size_t seg = (size_t)frame * p.nseg + s;
    if (t == 0) p.partial[seg * p.ntiles_col + tile] = sum;

    sub_fft<LM>(v, j, sm + c * S, p.twiddle, p.log2N);

    float2 *y = p.scratch + (seg << p.log2N);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int k1 = j + q * (M / 8);
        const float2 tw = __ldg(p.twiddle + ((n2 * k1) & (N - 1)));
        y[((size_t)k1 << log2N2) + n2] = cmul(v[q], tw);
    }
}

// segment means from the column pass's per-tile raw sums (fixed summation order)
__global__ void bigfft_mean_kernel(const BigParams p, int nsegs_total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsegs_total) return;
    const float2 *src = p.partial + (size_t)i * p.ntiles_col;
    float2 s = make_float2(0.f, 0.f);
    for (int t = 0; t < p.ntiles_col; ++t) s = cadd(s, src[t]);
    const float inv_n = 1.0f / (float)(1 << p.log2N);
    p.means[i] = make_float2(s.x * inv_n, s.y * inv_n);
}

template <int LM>
__global__ void __launch_bounds__(BIG_THREADS, 2) bigfft_row_kernel(const BigParams p) {
    constexpr int M = 1 << LM;            // N2
    constexpr int RR = BIG_TILE / M;      // rows (k1 values) per tile
    constexpr int S = big_stride(M);
    ZFB_DYN_SMEM(smem_raw);
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    const int t = threadIdx.x;
    const int r = t / (M / 8), j = t % (M / 8);
    const int tile = blockIdx.x, split = blockIdx.y, frame = blockIdx.z;
    const int N = 1 << p.log2N;
    const int log2N1 = p.log2N - LM;
    const int k1 = tile * RR + r;

    float2 wf[8];
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        wf[q] = __ldg(p.winfft + k1 + ((j + q * (M / 8)) << log2N1));
        acc[q] = 0.f;
    }
    const int s_begin = split * p.seg_per_split;
    const int s_end = min(p.nseg, s_begin + p.seg_per_split);
    for (int s = s_begin; s < s_end; ++s) {
        const size_t seg = (size_t)frame * p.nseg + s;
        const float2 *y = p.scratch + (seg << p.log2N) + ((size_t)k1 << LM);
        float2 v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = y[j + q * (M / 8)];
        const float2 mean = __ldg(p.means + seg);
        sub_fft<LM>(v, j, sm + r * S, p.twiddle, p.log2N);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float2 d = cmul(mean, wf[q]);
            const float re = v[q].x - d.x, im = v[q].y - d.y;
            acc[q] = fmaf(re, re, fmaf(im, im, acc[q]));
        }
    }

    // transpose through shared memory so that the global write runs along k
    __syncthreads();
    float *smf = reinterpret_cast<float *>(smem_raw);
#pragma unroll
    for (int q = 0; q < 8; ++q) smf[(j + q * (M / 8)) * (RR + 1) + r] = acc[q];
    __syncthreads();
    const int c0 = N / 2 - p.W / 2;
    float *row = p.pow_out + ((size_t)frame * p.nsplit + split) * p.W;
    for (int i = t; i < BIG_TILE; i += BIG_THREADS) {
        const int k2 = i / RR, rr = i % RR;
        const int k = tile * RR + rr + (k2 << log2N1);
        const int col = ((k + N / 2) & (N - 1)) - c0;
        if (col >= 0 && col < p.W) row[col] = smf[k2 * (RR + 1) + rr];
    }
}

// ===========================================================================
// N = 2^14 .. 2^17: decimation in frequency by 16 in front of the one-CTA FFT.
//   X[16k + r] = FFT_S( Z_r )[k],  S = N/16,
//   Z_r[n] = W_N^(r n) * sum_q x[n + S q] W_16^(q r),   x = window * (segment - mean)
// big_r16_kernel     : window + 16-point DFT across the 16 blocks + twiddle, coalesced in and
//                      out -> scratch [frame][r][segment][S]; also the raw sum of the CTA's 4096
//                      samples -> partial [frame][segment][S/256],
// big_mean16_kernel  : segment means from those partial sums (fixed order),
// then welch_kernel (prepared = 1) runs its shared-memory FFT on every S-point block, removes
// the mean there -- detrend='constant' is linear: FFT(w (x - m)) = FFT(w x) - m FFT(w), with
// FFT(w) from the host in fp64, stored per residue (winfft16 [r][k] = FFT(w)[16k + r]) -- and
// accumulates |X|^2 over the segments; big_gather_kernel puts bin 16k + r of residue r back in
// place (fftshift + crop).  ~Half the instructions of the generic four-step kernels above.
// (Round 1 removed the mean before the window, which took a pass of its own over the input --
// big_halfsum_kernel, 85 us of a 950 us cfg3 step at 78 % of the DRAM peak, ncu r02o.)
// ===========================================================================
struct BigR16Params {
    const void   *in;
    long long     in_stride;
    int           len, flip, log2N, hop, nseg;
    const float  *window;      // N taps
    const float2 *twiddle;     // N entries exp(-2 pi i k / N)
    float2       *partial;     // [frames][nseg][S/256] sums of the CTAs' samples (less the frame's DC estimate)
    float2       *means;       // [frames][nseg] segment mean less the frame's DC estimate
    float2       *dc;          // [frames] DC estimate of the frame (big_dc_kernel)
    float2       *scratch;     // [frames][16][nseg][S]
};

// A frame's DC estimate from 8192 samples spread over it (32 KB of an 8 MB row).  It is removed
// BEFORE the window, the rest of each segment's mean after the FFT: exact in exact arithmetic
// whatever the estimate is, and in fp32 the post-FFT correction then cancels a term proportional
// to |segment mean - estimate| instead of |segment mean| (a chunk with a DC offset of 0.4 and
// noise at 2e-3 read 0.015 dB20 off next to the DC bin with the plain post-FFT removal).
constexpr int BIG_DC_SAMPLES = 8192;
template <int KIND>
__global__ void __launch_bounds__(1024) big_dc_kernel(const BigR16Params p) {
    __shared__ float2 red[33];
    const int frame = blockIdx.x, t = threadIdx.x;
    const size_t esz = (KIND == KIND_U8_RAW) ? 2 : 8;
    const char *frame_in = (const char *)p.in + (size_t)frame * (size_t)p.in_stride * esz;
    const int used = (p.nseg + 1) * p.hop;                   // samples the segments cover
    const int stride = used / BIG_DC_SAMPLES > 0 ? used / BIG_DC_SAMPLES : 1;
    // 8 independent loads per thread (a serial loop of 32 took 20 us per launch: 32 DRAM round trips)
    float2 x[BIG_DC_SAMPLES / 1024];
#pragma unroll
    for (int j = 0; j < BIG_DC_SAMPLES / 1024; ++j) {
        const long long idx = (long long)(t + 1024 * j) * stride;
        x[j] = idx < used ? welch_fetch<KIND>(frame_in, (int)idx, p.len, p.flip) : make_float2(0.f, 0.f);
    }
    float2 sum = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < BIG_DC_SAMPLES / 1024; ++j) sum = cadd(sum, x[j]);
    sum = block_sum<1024>(sum, t, red);
    const int cnt = (used + stride - 1) / stride < BIG_DC_SAMPLES ? (used + stride - 1) / stride : BIG_DC_SAMPLES;
    if (t == 0) p.dc[frame] = make_float2(sum.x / (float)cnt, sum.y / (float)cnt);
}

// segment means (less the DC estimate) from the front pass's per-CTA sums (fixed summation order)
__global__ void big_mean16_kernel(const BigR16Params p, int nsegs_total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsegs_total) return;
    const int nblk = (1 << p.log2N) >> 12;                 // S / 256
    const float2 *src = p.partial + (size_t)i * nblk;
    float2 s = make_float2(0.f, 0.f);
    for (int t = 0; t < nblk; ++t) s = cadd(s, src[t]);
    const float inv_n = 1.0f / (float)(1 << p.log2N);
    p.means[i] = make_float2(s.x * inv_n, s.y * inv_n);
}

template <int KIND>
__global__ void __launch_bounds__(256) big_r16_kernel(const BigR16Params p) {
    const int N = 1 << p.log2N, S = N >> 4;
    const int n = blockIdx.x * 256 + threadIdx.x;          // < S
    const int s = blockIdx.y, frame = blockIdx.z;
    const size_t esz = (KIND == KIND_U8_RAW) ? 2 : 8;
    const char *frame_in = (const char *)p.in + (size_t)frame * (size_t)p.in_stride * esz;
    const int base = s * p.hop;
    __shared__ float2 red[33];
    float2 v[16];
    float2 raw_sum = make_float2(0.f, 0.f);
    const float2 dc = __ldg(p.dc + frame);
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int idx = n + S * q;
        float2 x = welch_fetch<KIND>(frame_in, base + idx, p.len, p.flip);
        const float w = __ldg(p.window + idx);
        x = make_float2(x.x - dc.x, x.y - dc.y);
        raw_sum = cadd(raw_sum, x);
        v[q] = make_float2(x.x * w, x.y * w);
    }
    raw_sum = block_sum<256>(raw_sum, threadIdx.x, red);
    if (threadIdx.x == 0) p.partial[((size_t)frame * p.nseg + s) * (S >> 8) + blockIdx.x] = raw_sum;
    dft16(v);
    float2 *out = p.scratch + (((size_t)frame * 16) * p.nseg + s) * (size_t)S + n;
    const size_t rstride = (size_t)p.nseg * S;
    // W_N^(r n), r = 1..15, from four table lookups (n, 2n, 4n, 8n) and products
    float2 w[16];
    w[1] = __ldg(p.twiddle + n);
    w[2] = __ldg(p.twiddle + ((2 * n) & (N - 1)));
    w[4] = __ldg(p.twiddle + ((4 * n) & (N - 1)));
    w[8] = __ldg(p.twiddle + ((8 * n) & (N - 1)));
    w[3] = cmul(w[1], w[2]);
    w[5] = cmul(w[1], w[4]);
    w[6] = cmul(w[2], w[4]);
    w[7] = cmul(w[3], w[4]);
#pragma unroll
    for (int r = 9; r < 16; ++r) w[r] = cmul(w[r - 8], w[8]);
    out[0] = v[0];
#pragma unroll
    for (int r = 1; r < 16; ++r) out[r * rstride] = cmul(v[r], w[r]);
}

// pow16 [frames*16][nsplit][S] (fftshifted sub-spectra) -> pow [frames][1][W]
struct BigGatherParams {
    const float *pow16;
    float       *pow_out;
    int          log2N, nsplit, W, frames;
};

__global__ void big_gather_kernel(const BigGatherParams p) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)p.frames * p.W) return;
    const int f = (int)(i / p.W), col = (int)(i % p.W);
    const int N = 1 << p.log2N, S = N >> 4;
    const int bin = (col - p.W / 2 + N) & (N - 1);          // undo fftshift + centre crop
    const int r = bin & 15, k = bin >> 4;
    const int sub = (k + S / 2) & (S - 1);                  // welch_kernel stored its block fftshifted
    const float *src = p.pow16 + ((size_t)(f * 16 + r) * p.nsplit) * S + sub;
    float acc = 0.f;
    for (int sp = 0; sp < p.nsplit; ++sp) acc += src[(size_t)sp * S];
    p.pow_out[(size_t)f * p.W + col] = acc;
}

// N = N1*N2 split used for a given log2N
inline void big_split(int log2N, int &lm1, int &lm2) {
    lm1 = (log2N + 1) / 2;
    lm2 = log2N - lm1;
}

inline int big_ntiles_col(int log2N) {
    int lm1, lm2;
    big_split(log2N, lm1, lm2);
    return (1 << lm2) / (BIG_TILE >> lm1);
}

inline size_t big_scratch_bytes(int log2N, int nseg, int frames) {
    return (size_t)frames * (size_t)nseg * (((size_t)1 << log2N) + (size_t)big_ntiles_col(log2N) + 2) * sizeof(float2);
}

template <int LM1>
inline void big_launch_col(const BigParams &p, int kind, dim3 grid, cudaStream_t st) {
    const size_t smem = big_smem(1 << LM1);
    if (kind == KIND_C64_RAW) {
        ZFB_LAUNCH((bigfft_col_kernel<LM1, KIND_C64_RAW>), grid, dim3(BIG_THREADS), smem, st, p);
    } else if (kind == KIND_U8_RAW) {
        ZFB_LAUNCH((bigfft_col_kernel<LM1, KIND_U8_RAW>), grid, dim3(BIG_THREADS), smem, st, p);
    } else {
        ZFB_LAUNCH((bigfft_col_kernel<LM1, KIND_C64_MID>), grid, dim3(BIG_THREADS), smem, st, p);
    }
}

// enqueue the column pass for `frames` frames
inline void big_run_col(const BigParams &p, int kind, int frames, cudaStream_t st) {
    int lm1, lm2;
    big_split(p.log2N, lm1, lm2);
    dim3 gcol((unsigned)p.ntiles_col, (unsigned)p.nseg, (unsigned)frames);
    switch (lm1) {
        case 7: big_launch_col<7>(p, kind, gcol, st); break;
        case 8: big_launch_col<8>(p, kind, gcol, st); break;
        default: big_launch_col<9>(p, kind, gcol, st); break;
    }
}

// enqueue the row pass
inline void big_run_row(const BigParams &p, int frames, cudaStream_t st) {
    int lm1, lm2;
    big_split(p.log2N, lm1, lm2);
    const int nsegs_total = frames * p.nseg;
    ZFB_LAUNCH(bigfft_mean_kernel, dim3((unsigned)((nsegs_total + 127) / 128)), dim3(128), 0, st, p, nsegs_total);
    const int rr = BIG_TILE >> lm2;
    dim3 grow((unsigned)((1 << lm1) / rr), (unsigned)p.nsplit, (unsigned)frames);
    switch (lm2) {
        case 7: ZFB_LAUNCH(bigfft_row_kernel<7>, grow, dim3(BIG_THREADS), big_smem(1 << 7), st, p); break;
        case 8: ZFB_LAUNCH(bigfft_row_kernel<8>, grow, dim3(BIG_THREADS), big_smem(1 << 8), st, p); break;
        default: ZFB_LAUNCH(bigfft_row_kernel<9>, grow, dim3(BIG_THREADS), big_smem(1 << 9), st, p); break;
    }
}

}  // namespace zfb
