// Waterfall image on the device (SURVEY 8f.1).  The reference keeps a float64
// img_array of (w//4, w) on the host, rolls the WHOLE image by one row per
// update (np.roll, pypanadapter_spectrum.py:1651-1652), redraws grid and tick
// marks (S:1647-1648, S:1655-1662) and hands it to pyqtgraph, which maps
// [minlev, maxlev] onto a 256-entry colour table (S:1592-1594, S:1612-1623;
// pyqtgraph ImageItem: index = clip(trunc((v - min) * 256 / (max - min)), 0,
// 255), reproduced bit for bit in fp32 by wf_level).
// Here the rows stay in the device ring.  A pixel of the image the reference
// would hold after the same sequence of updates is a pure function of (y, x),
// the ring and three counters (wf_row, wf_tick_row, wf_fix), so the image --
// as float32 img_array, as 8-bit colour indices or as RGBA through the table
// -- is produced by one streaming pass only when it is displayed, and only
// the 8-bit image crosses PCIe.  Waterfall.autolevel's np.percentile(
// img_array[img_array < 0], [2, 98]) (S:1676) is an exact order-statistic
// selection by three 11/11/9-bit radix histograms over the same pixel function.
#pragma once
#include "zfb_common.cuh"

namespace zfb {

constexpr int IMG_F32 = 0, IMG_U8 = 1, IMG_RGBA = 2;

// level mapping: index = clip(trunc((double(v) - minlev) * 256 / (maxlev - minlev)), 0, 255).
// thr[k], k = 1..255 = the smallest float whose index is >= k (found on the host with
// exactly that double arithmetic): the device makes an fp32 guess v * fscale + foff
// (within 1 of the index for any sane level pair) and settles it by comparing with the
// neighbouring thresholds, bit-exact with the double formula, no FP64 or F2I instructions.
struct LevelMap {
    const float *thr;         // [257]
    float  fscale, foff;
    int    wide_guess;        // the fp32 guess may be off by more than 1 (degenerate level pair)
    const unsigned int *lut;  // 256 packed RGBA entries (IMG_RGBA)
};

struct ImageParams {
    const float *ring;        // [ring_rows][W] finished rows
    int    ring_rows;
    long long written;        // rows written to the ring so far (monotone)
    int    W, H;              // image is [H][W], H = W//4 in the reference
    int    have;              // rows of the image that come from the ring
    int    nseen;             // image_update calls since init_image, saturated at 1<<20
    int    scroll;            // AppState.scroll: > 0 newest row near the bottom, else at the top
    int    tick_step;         // W // 10
    int    newest_slot;       // ring slot of the newest row: (written - 1) mod ring_rows
    LevelMap lv;              // (minlev, maxlev) -> colour index, and the RGBA table
    void  *out;
};

// tick marks are redrawn on every update and scroll with the image: every row
// that has passed through the marked band keeps them (S:1655-1662)
__device__ __forceinline__ bool wf_tick_row(const ImageParams &p, int y) {
    if (p.nseen <= 0) return false;
    if (p.scroll > 0) {
        if (y >= 5 && y < 15) return true;
        if (y < 5) return p.nseen > 5 - y;          // moved up out of the band
        if (y == p.H - 1) return p.nseen > 6;       // wrapped around from row 0
        return false;
    }
    if (y >= p.H - 10 && y < p.H - 2) return true;
    if (y >= p.H - 2 && y < p.H) return p.nseen > y - (p.H - 3);
    return false;
}

__device__ __forceinline__ bool wf_tick_col(const ImageParams &p, int x) {
    if (x >= p.W - 1 || p.tick_step <= 0) return false;
    const int i = x / p.tick_step;
    return (x - i * p.tick_step == 0) && i != 5 && i != 10;
}

// ring row shown at image row y, or -1 for the -500 fill (S:1631)
__device__ __forceinline__ const float *wf_row(const ImageParams &p, int y) {
    int j;                                           // age of the row, 0 = newest
    if (p.scroll > 0) {
        j = p.H - 2 - y;
        if (j < 0) j += p.H;
    } else {
        j = y;
    }
    if (j >= p.have) return nullptr;
    int slot = p.newest_slot - j;                    // j < have <= ring_rows
    if (slot < 0) slot += p.ring_rows;
    return p.ring + (size_t)slot * p.W;
}

__device__ __forceinline__ float wf_fix(const ImageParams &p, bool from_ring, bool tick_row, int x, float v) {
    const bool edge = (x == 0) || (x == p.W - 1);
    if (from_ring) {
        if (edge || x == p.W / 2) v = 0.f;           // grid bins zeroed on the row (S:1647-1648)
    } else {
        v = edge ? 0.f : -500.f;                     // init_image (S:1631-1635)
    }
    if (tick_row && wf_tick_col(p, x)) v = 0.f;
    return v;
}

// four consecutive pixels starting at x0 (x0 % 4 == 0): only the quads that
// hold a grid column, and the few tick rows, take the per-pixel path
__device__ __forceinline__ void wf_fix4(const ImageParams &p, bool from_ring, bool tick_row, int x0, float (&q)[4]) {
    const int mid = p.W >> 1;
    const bool special = tick_row || x0 == 0 || x0 + 4 >= p.W || (unsigned)(mid - x0) < 4u;
    if (special) {
#pragma unroll
        for (int e = 0; e < 4; ++e) q[e] = wf_fix(p, from_ring, tick_row, x0 + e, q[e]);
    } else if (!from_ring) {
#pragma unroll
        for (int e = 0; e < 4; ++e) q[e] = -500.f;
    }
}

// the shared-memory table wf_level reads: thr2[g] = (thr[g], thr[g + 1]) with
// thr[0] = -inf and thr[256] = NaN (never reached)
__device__ __forceinline__ void wf_load_levels(float2 *thr2, const float *thr) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        thr2[i] = make_float2(thr[i], i < 255 ? thr[i + 1] : __uint_as_float(0x7FC00000u));
}

__device__ __forceinline__ unsigned int wf_level(const float2 *thr2, float fscale, float foff, int wide_guess,
                                                 float v) {
    float x = fmaf(v, fscale, foff);
    x = fminf(fmaxf(x, 0.f), 255.f);                 // NaN -> 0
    int g = (int)(__float_as_uint(x + 8388608.0f) - 0x4B000000u);    // round to nearest, 0..255
    if (!wide_guess) {
        // |guess - index| <= 1 (the host checked the level pair): one LDS.64, two compares
        const float2 t = thr2[g];
        g += (v >= t.y) ? 1 : 0;
        g -= (v < t.x) ? 1 : 0;
    } else {
        while (g < 255 && v >= thr2[g].y) ++g;       // degenerate level pairs: walk to the index
        while (g > 0 && v < thr2[g].x) --g;
    }
    return (unsigned int)g;
}

constexpr int IMG_NT = 256;
constexpr int IMG_U = 4;                  // float4 loads in flight per thread

template <int KIND>
__global__ void __launch_bounds__(IMG_NT) wf_image_kernel(const ImageParams p) {
    __shared__ float2 thr[256];
    __shared__ unsigned int lut[256];
    if (KIND != IMG_F32) {
        wf_load_levels(thr, p.lv.thr);
        if (KIND == IMG_RGBA)
            for (int i = threadIdx.x; i < 256; i += IMG_NT) lut[i] = p.lv.lut[i];
        __syncthreads();
    }
    const LevelMap &m = p.lv;
    const int y = blockIdx.y;
    const float *row = wf_row(p, y);
    const bool tick_row = wf_tick_row(p, y);
    const int xb = (int)blockIdx.x * (IMG_NT * IMG_U * 4);
    if ((p.W & 3) == 0) {
        float4 v[IMG_U];
#pragma unroll
        for (int u = 0; u < IMG_U; ++u) {
            const int x0 = xb + (u * IMG_NT + (int)threadIdx.x) * 4;
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row && x0 < p.W) v[u] = __ldg((const float4 *)(row + x0));
        }
#pragma unroll
        for (int u = 0; u < IMG_U; ++u) {
            const int x0 = xb + (u * IMG_NT + (int)threadIdx.x) * 4;
            if (x0 >= p.W) break;
            float q[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            wf_fix4(p, row != nullptr, tick_row, x0, q);
            const size_t at = (size_t)y * p.W + x0;
            if (KIND == IMG_F32) {
                *(float4 *)((float *)p.out + at) = make_float4(q[0], q[1], q[2], q[3]);
            } else if (KIND == IMG_U8) {
                unsigned int pk = 0;
#pragma unroll
                for (int e = 0; e < 4; ++e) pk |= wf_level(thr, m.fscale, m.foff, m.wide_guess, q[e]) << (8 * e);
                *(unsigned int *)((unsigned char *)p.out + at) = pk;
            } else {
                uint4 c;
                c.x = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, q[0])];
                c.y = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, q[1])];
                c.z = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, q[2])];
                c.w = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, q[3])];
                *(uint4 *)((unsigned int *)p.out + at) = c;
            }
        }
    } else {
        const int xe = min(p.W, xb + IMG_NT * IMG_U * 4);
        for (int x = xb + (int)threadIdx.x; x < xe; x += IMG_NT) {
            const float v = wf_fix(p, row != nullptr, tick_row, x, row ? row[x] : 0.f);
            const size_t at = (size_t)y * p.W + x;
            if (KIND == IMG_F32) ((float *)p.out)[at] = v;
            else if (KIND == IMG_U8) ((unsigned char *)p.out)[at] = (unsigned char)wf_level(thr, m.fscale, m.foff, m.wide_guess, v);
            else ((unsigned int *)p.out)[at] = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, v)];
        }
    }
}

// ---- exact order statistics of {img[y][x] : img[y][x] < 0} ---------------
constexpr int SEL_TARGETS = 4;            // ranks resolved per sweep
constexpr int SEL_BINS = 2048;

struct SelectParams {
    ImageParams img;
    int pass;                             // 0: key bits 30..20, 1: bits 19..9, 2: bits 8..0
    int ntargets;
    unsigned int prefix[SEL_TARGETS];     // pass 1: key >> 20, pass 2: key >> 9 (distinct values)
    unsigned int *hist;                   // [SEL_TARGETS][SEL_BINS] (pass 0 uses histogram 0 only)
    int rows_per_cta;
};

// monotone map of the floats below zero onto unsigned keys (ascending)
__device__ __forceinline__ unsigned int wf_key(float v) { return ~__float_as_uint(v); }
__host__ inline float wf_unkey(unsigned int k) {
    const unsigned int u = ~k;
    float f;
    memcpy(&f, &u, 4);
    return f;
}

// one histogram slot per pixel (prefixes are distinct), warp-aggregated: the
// lanes that hit the same slot elect a leader which adds their count with ONE
// shared-memory atomic (dB rows crowd a handful of leading-bit bins: unaggregated,
// every warp would serialise 32 same-address atomics)
constexpr unsigned int SEL_NONE = 0xFFFFFFFFu;

template <int PASS>
__device__ __forceinline__ unsigned int wf_slot(const SelectParams &s, float v) {
    if (!(v < 0.f)) return SEL_NONE;
    const unsigned int k = wf_key(v);
    // keys of negative floats have bit 31 clear: digits are bits 30..20, 19..9, 8..0
    if (PASS == 0) return k >> 20;
    const unsigned int pre = (PASS == 1) ? (k >> 20) : (k >> 9);
    const unsigned int sub = (PASS == 1) ? ((k >> 9) & 0x7FFu) : (k & 0x1FFu);
    unsigned int at = SEL_NONE;
#pragma unroll
    for (int t = 0; t < SEL_TARGETS; ++t)
        if (t < s.ntargets && pre == s.prefix[t]) at = (unsigned int)t * SEL_BINS + sub;
    return at;
}

__device__ __forceinline__ void wf_count(unsigned int *h, unsigned int at, int lane) {
    const unsigned int peers = __match_any_sync(0xFFFFFFFFu, at);
    if (at != SEL_NONE && lane == __ffs((int)peers) - 1) atomicAdd(&h[at], (unsigned int)__popc(peers));
}

// (Measured and dropped, gpurun r02o: run-length merging a thread's four slots before the MATCH --
// one MATCH + three votes per four pixels -- made the sweeps SLOWER, 0.648 -> 0.711 ms on the
// 8192 x 32768 image: only the first sweep's digits repeat among neighbours; sweeps two and three
// spread the pixels of one prefix over 2048 / 512 bins, their cost is shared-memory atomics on
// colliding banks (ncu: 3.4 M conflicts in 5.8 M wavefronts, short scoreboard 15.9 per issue), not MATCH.)

template <int PASS>
__global__ void __launch_bounds__(256) wf_select_kernel(const SelectParams s) {
    ZFB_DYN_SMEM(smem_raw);                                  // nh * SEL_BINS counters
    unsigned int *h = reinterpret_cast<unsigned int *>(smem_raw);
    const ImageParams &p = s.img;
    const int nh = (PASS == 0) ? 1 : s.ntargets;
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < nh * SEL_BINS; i += blockDim.x) h[i] = 0u;
    __syncthreads();
    const int y0 = blockIdx.x * s.rows_per_cta;
    const int y1 = min(p.H, y0 + s.rows_per_cta);
    const bool vec = (p.W & 3) == 0;
    for (int y = y0; y < y1; ++y) {
        const float *row = wf_row(p, y);
        const bool tick_row = wf_tick_row(p, y);
        if (vec) {
            for (int xb = 0; xb < p.W; xb += 1024) {          // uniform trip count: warp collectives inside
                const int x0 = xb + (int)threadIdx.x * 4;
                const bool in = x0 < p.W;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (row && in) v = __ldg((const float4 *)(row + x0));
                float q[4] = {v.x, v.y, v.z, v.w};
                wf_fix4(p, row != nullptr, tick_row, x0, q);
#pragma unroll
                for (int e = 0; e < 4; ++e) wf_count(h, in ? wf_slot<PASS>(s, q[e]) : SEL_NONE, lane);
            }
        } else {
            for (int xb = 0; xb < p.W; xb += 256) {
                const int x = xb + (int)threadIdx.x;
                const bool in = x < p.W;
                const float v = wf_fix(p, row != nullptr, tick_row, x, (row && in) ? __ldg(row + x) : 0.f);
                wf_count(h, in ? wf_slot<PASS>(s, v) : SEL_NONE, lane);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nh * SEL_BINS; i += blockDim.x)
        if (h[i]) atomicAdd(&s.hist[i], h[i]);
}

}  // namespace zfb
