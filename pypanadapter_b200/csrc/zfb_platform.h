// Build-mode glue.  The product is compiled by nvcc for sm_100a.  The only
// other mode, ZFB_EMULATE, exists for tests/emu (a CPU stand-in for the CUDA
// runtime used to exercise kernel logic in the GPU-less build container); it
// is never built into or loaded by the package.
#pragma once
#ifdef ZFB_EMULATE
#include "cuda_emu.h"
#define ZFB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    ::cuemu::launch(kernel, grid, block, smem, __VA_ARGS__)
#define ZFB_DYN_SMEM(name) unsigned char *name = ::cuemu::dyn_smem()
#define ZFB_BUILD_KIND "emulated"
// The device's separately rounded fp32 multiply and add (zfb_persist.cuh relies on them to
// match numpy's float32 P * decay + hit).  They must not be plain a * b and a + b: under
// g++ -O2 -mfma those contract into one vfmadd, so each result goes through a volatile
// (one vmulss, then one vaddss).
static inline float __fmul_rn(float a, float b) {
    volatile float p = a * b;
    return p;
}
static inline float __fadd_rn(float a, float b) {
    volatile float s = a + b;
    return s;
}
static inline double __dadd_rn(double a, double b) {
    volatile double s = a + b;
    return s;
}
// zfb_power.cuh's last-CTA hand-off: CTAs run on several OS threads, so the fence is a real one;
// an L2-only load is a plain load here
static inline void __threadfence() { std::atomic_thread_fence(std::memory_order_seq_cst); }
template <typename T>
static inline T __ldcg(const T *p) { return *p; }
#else
#include <cuda_runtime.h>
#define ZFB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#define ZFB_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define ZFB_BUILD_KIND "sm_100a"
#endif
