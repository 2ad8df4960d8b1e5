// Decaying persistence (level-density) spectrum over the engine's rows (DESIGN 3.9).
//
// The reference draws each row as it comes (spectrum_plot.setData, S:2130) and keeps
// nothing across rows.  A spectrum analyser's persistence display shows how the level
// at each frequency is distributed over time: per column, 256 level bins, each an
// intensity that every row decays and the row's own bin raises by one.  Here that state
// is on the device, updated right behind the finalisation of every launch group, like
// the trace set (zfb_trace.cuh), and only its image crosses PCIe.
//
//   persist_update_kernel  P[k][c] = fadd_rn(fmul_rn(P[k][c], decay), k == bin(row[c]))
//                          strictly in frame order per cell: batch independent
//   persist_image_kernel   [256][W] image, row 0 = level bin 255, as float32 intensities,
//                          colour indices of (imin, imax) or RGBA through the table
#pragma once
#include "zfb_image.cuh"

namespace zfb {

constexpr int PS_LEVELS = 256;

struct PersistParams {
    const float *rows;        // [nframes][W] finished rows
    int    nframes, W;
    int    have;              // the state holds at least one row (host-side knowledge, launch order)
    float  decay;             // 0 < decay <= 1
    float *state;             // [PS_LEVELS][W], level-major
    LevelMap lv;              // row value -> level bin: the waterfall's colour index for (minlev, maxlev)
};

// A CTA owns PS_COLS consecutive columns and PS_KG * PS_CELLS consecutive level bins of
// them (gridDim.y = PS_SLICES slices of the 256 bins, so that a narrow row still fills the
// GPU).  All threads turn a tile of PS_FR frames x PS_COLS columns into level bins in
// shared memory (row loads coalesced over columns, as in trace_update_kernel); then every
// thread walks its PS_CELLS cells of one column over the tile in frame order, the state in
// registers.  A warp holds one bin of 32 consecutive columns: the state is read and written
// once per launch, coalesced, level-major.
constexpr int PS_COLS = 32;
constexpr int PS_NT = 256;
constexpr int PS_KG = PS_NT / PS_COLS;               // level groups per CTA
constexpr int PS_CELLS = 2;                          // level bins per thread: 16 slices fill the GPU at W = 256
constexpr int PS_SLICES = PS_LEVELS / (PS_KG * PS_CELLS);
constexpr int PS_FR = 64;                            // frames per tile

__global__ void __launch_bounds__(PS_NT) persist_update_kernel(const PersistParams p) {
    __shared__ float2 thr[256];
    __shared__ unsigned char bins[PS_FR][PS_COLS];
    wf_load_levels(thr, p.lv.thr);
    const int c = threadIdx.x % PS_COLS, kg = threadIdx.x / PS_COLS;
    const int col = blockIdx.x * PS_COLS + c;
    const bool ok = col < p.W;
    const int k0 = (blockIdx.y * PS_KG + kg) * PS_CELLS;       // this thread's bins k0 .. k0 + PS_CELLS - 1
    float s[PS_CELLS];
#pragma unroll
    for (int j = 0; j < PS_CELLS; ++j) s[j] = (ok && p.have) ? p.state[(size_t)(k0 + j) * p.W + col] : 0.f;
    for (int f0 = 0; f0 < p.nframes; f0 += PS_FR) {
        const int n = min(PS_FR, p.nframes - f0);
        __syncthreads();                                          // table loaded / previous tile walked
        for (int i = kg; i < n; i += PS_KG)
            if (ok) bins[i][c] = (unsigned char)wf_level(thr, p.lv.fscale, p.lv.foff, p.lv.wide_guess,
                                                         p.rows[(size_t)(f0 + i) * p.W + col]);
        __syncthreads();
        if (ok) {
#pragma unroll 4
            for (int i = 0; i < n; ++i) {
                const int b = (int)bins[i][c] - k0;
                // separately rounded (no FMA): numpy's float32 P * decay + hit, bit for bit (adding
                // the 0 of a missed bin leaves the product as it is, so only the hit bin adds)
#pragma unroll
                for (int j = 0; j < PS_CELLS; ++j) {
                    s[j] = __fmul_rn(s[j], p.decay);
                    if (b == j) s[j] = __fadd_rn(s[j], 1.f);
                }
            }
        }
    }
    if (ok && p.nframes > 0) {
#pragma unroll
        for (int j = 0; j < PS_CELLS; ++j) p.state[(size_t)(k0 + j) * p.W + col] = s[j];
    }
}

struct PersistImageParams {
    const float *state;       // [PS_LEVELS][W]
    int    W;
    LevelMap lv;              // intensity -> colour index for (imin, imax), and the RGBA table
    void  *out;               // [PS_LEVELS][W] float, uint8 or packed RGBA
};

constexpr int PI_NT = 256;
constexpr int PI_U = 4;                   // pixels per thread

// one streaming pass: image row y is level bin 255 - y (high levels at the top)
template <int KIND>
__global__ void __launch_bounds__(PI_NT) persist_image_kernel(const PersistImageParams p) {
    __shared__ float2 thr[256];
    __shared__ unsigned int lut[256];
    if (KIND != IMG_F32) {
        wf_load_levels(thr, p.lv.thr);
        if (KIND == IMG_RGBA)
            for (int i = threadIdx.x; i < 256; i += PI_NT) lut[i] = p.lv.lut[i];
        __syncthreads();
    }
    const LevelMap &m = p.lv;
    const int y = blockIdx.y;
    const float *src = p.state + (size_t)(PS_LEVELS - 1 - y) * p.W;
    const int x0 = blockIdx.x * (PI_NT * PI_U);
    const int xe = min(p.W, x0 + PI_NT * PI_U);
    for (int x = x0 + (int)threadIdx.x; x < xe; x += PI_NT) {
        const float v = __ldg(src + x);
        const size_t at = (size_t)y * p.W + x;
        if (KIND == IMG_F32) ((float *)p.out)[at] = v;
        else if (KIND == IMG_U8) ((unsigned char *)p.out)[at] = (unsigned char)wf_level(thr, m.fscale, m.foff, m.wide_guess, v);
        else ((unsigned int *)p.out)[at] = lut[wf_level(thr, m.fscale, m.foff, m.wide_guess, v)];
    }
}

}  // namespace zfb
