// cuda_emu.h -- TEST INFRASTRUCTURE ONLY.
//
// A tiny CPU stand-in for the slice of CUDA that pypanadapter_b200/csrc uses,
// so that the kernels' *logic* (indexing, hand-offs, edge cases) and the whole
// host side of the C-ABI can be exercised in the GPU-less build container.
// tests/emu/build_emu.py compiles csrc/zfb_engine.cu with g++ -DZFB_EMULATE
// into tests/emu/_build/libzoomfft_emu.so; ONLY tests/test_emu_*.py load it
// (by explicit path).  The product (pypanadapter_b200) never loads it, never
// falls back to it, and knows nothing about it.
//
// Execution model: every CTA runs as blockDim.x ucontext fibers on one OS
// thread, round-robin; __syncthreads() and warp shuffles are fiber yield
// points.  Independent CTAs are spread over a few OS threads.  Arithmetic is
// host fp32 (fmaf), close to -- not bit-identical with -- the device.
#pragma once
#include <ucontext.h>

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>

// ------------------------------------------------------------ qualifiers
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __launch_bounds__(...)
#define __restrict__ __restrict
#define __constant__
#define __shared__ static thread_local
#define __align__(n) alignas(n)

// ------------------------------------------------------------ vector types
struct alignas(8) float2 { float x, y; };
struct alignas(16) float4 { float x, y, z, w; };
struct alignas(16) uint4 { unsigned int x, y, z, w; };
struct alignas(8) uint2 { unsigned int x, y; };
struct dim3 {
    unsigned int x, y, z;
    dim3(unsigned int a = 1, unsigned int b = 1, unsigned int c = 1) : x(a), y(b), z(c) {}
};
struct alignas(16) double2 { double x, y; };
static inline double2 make_double2(double x, double y) { return double2{x, y}; }
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return uint4{a, b, c, d}; }
static inline uint2 make_uint2(unsigned a, unsigned b) { return uint2{a, b}; }

namespace cuemu {

constexpr size_t kStack = 96 * 1024;

struct Fiber {
    ucontext_t ctx;
    char *stack = nullptr;
    bool done = false;
    // wait descriptor: runnable when *counter >= target (counter == nullptr: runnable)
    const long *wait_counter = nullptr;
    long wait_target = 0;
};

struct Warp {
    long arrived = 0;                 // total shuffle arrivals
    long gen[32] = {0};               // per-lane shuffle generation
    uint64_t slot[2][32];
};

struct Cta {
    ucontext_t sched;
    std::vector<Fiber> fib;
    std::vector<Warp> warps;
    long bar_arrived = 0;
    std::vector<long> bar_gen;        // per-thread barrier generation
    int nthreads = 0;
    int live = 0;
    int cur = 0;
    unsigned char *smem = nullptr;
    const std::function<void()> *body = nullptr;
};

struct Idx { unsigned int x, y, z; };
extern thread_local Idx t_threadIdx, t_blockIdx, t_blockDim, t_gridDim;
extern thread_local Cta *t_cta;

void run_grid(const std::function<void()> &body, dim3 grid, dim3 block, size_t smem);
void yield_until(const long *counter, long target);

inline unsigned char *dyn_smem() { return t_cta->smem; }

template <typename... KArgs, typename... Args>
inline void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args) {
    std::function<void()> body = [=]() { kernel(args...); };
    run_grid(body, grid, block, smem);
}

}  // namespace cuemu

#define threadIdx (::cuemu::t_threadIdx)
#define blockIdx (::cuemu::t_blockIdx)
#define blockDim (::cuemu::t_blockDim)
#define gridDim (::cuemu::t_gridDim)

// ------------------------------------------------------------ device intrinsics
static inline void __syncthreads() {
    cuemu::Cta *c = cuemu::t_cta;
    const int t = c->cur;
    c->bar_arrived += 1;
    c->bar_gen[t] += 1;
    cuemu::yield_until(&c->bar_arrived, c->bar_gen[t] * (long)c->nthreads);
}
// warp barrier: a fiber yield point like the shuffles (all lanes of the warp must take part)
static inline void __syncwarp(unsigned = 0xffffffffu) {
    cuemu::Cta *c = cuemu::t_cta;
    const int t = c->cur, lane = t & 31;
    cuemu::Warp &w = c->warps[t >> 5];
    const int wsize = (c->nthreads - (t & ~31)) < 32 ? (c->nthreads - (t & ~31)) : 32;
    const long g = ++w.gen[lane];
    w.arrived += 1;
    cuemu::yield_until(&w.arrived, g * (long)wsize);
}

template <typename T>
static inline T __shfl_xor_sync(unsigned, T v, int lane_mask) {
    static_assert(sizeof(T) <= 8, "shuffle payload");
    cuemu::Cta *c = cuemu::t_cta;
    const int t = c->cur, lane = t & 31;
    cuemu::Warp &w = c->warps[t >> 5];
    const int wsize = (c->nthreads - (t & ~31)) < 32 ? (c->nthreads - (t & ~31)) : 32;
    const long g = ++w.gen[lane];
    uint64_t bits = 0;
    memcpy(&bits, &v, sizeof(T));
    w.slot[g & 1][lane] = bits;
    w.arrived += 1;
    cuemu::yield_until(&w.arrived, g * (long)wsize);
    const int src = lane ^ lane_mask;
    uint64_t r = w.slot[g & 1][src < wsize ? src : lane];
    T out;
    memcpy(&out, &r, sizeof(T));
    return out;
}

// every lane of the warp posts its value; the result is the mask of lanes that
// posted the same one (all lanes of the warp must take part, as with shuffles)
static inline unsigned int __match_any_sync(unsigned, unsigned int v) {
    cuemu::Cta *c = cuemu::t_cta;
    const int t = c->cur, lane = t & 31;
    cuemu::Warp &w = c->warps[t >> 5];
    const int wsize = (c->nthreads - (t & ~31)) < 32 ? (c->nthreads - (t & ~31)) : 32;
    const long g = ++w.gen[lane];
    w.slot[g & 1][lane] = v;
    w.arrived += 1;
    cuemu::yield_until(&w.arrived, g * (long)wsize);
    unsigned int m = 0;
    for (int l = 0; l < wsize; ++l)
        if ((unsigned int)w.slot[g & 1][l] == v) m |= 1u << l;
    return m;
}
// vote: true if any lane of the warp posted a non-zero predicate
static inline int __any_sync(unsigned, int pred) {
    cuemu::Cta *c = cuemu::t_cta;
    const int t = c->cur, lane = t & 31;
    cuemu::Warp &w = c->warps[t >> 5];
    const int wsize = (c->nthreads - (t & ~31)) < 32 ? (c->nthreads - (t & ~31)) : 32;
    const long g = ++w.gen[lane];
    w.slot[g & 1][lane] = pred ? 1u : 0u;
    w.arrived += 1;
    cuemu::yield_until(&w.arrived, g * (long)wsize);
    int any = 0;
    for (int l = 0; l < wsize; ++l) any |= (int)w.slot[g & 1][l];
    return any;
}
static inline int __popc(unsigned int x) { return __builtin_popcount(x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }

template <typename T>
static inline T __ldg(const T *p) { return *p; }

static inline float2 __ffma2_rn(float2 a, float2 b, float2 c) {
    return float2{fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)};
}
static inline float2 __fadd2_rn(float2 a, float2 b) { return float2{a.x + b.x, a.y + b.y}; }
static inline float2 __fmul2_rn(float2 a, float2 b) { return float2{a.x * b.x, a.y * b.y}; }
static inline void sincospif(float x, float *s, float *c) {
    const double a = 3.14159265358979323846 * (double)x;
    *s = (float)sin(a);
    *c = (float)cos(a);
}
static inline double cospi(double x) { return cos(3.14159265358979323846 * x); }
static inline double sinpi(double x) { return sin(3.14159265358979323846 * x); }
static inline void sincospi(double x, double *s, double *c) {
    *s = sin(3.14159265358979323846 * x);
    *c = cos(3.14159265358979323846 * x);
}
static inline double cyl_bessel_i0(double x) { return std::cyl_bessel_i(0.0, x); }
static inline unsigned int __byte_perm(unsigned int x, unsigned int y, unsigned int sel) {
    const uint64_t src = ((uint64_t)y << 32) | x;
    unsigned int r = 0;
    for (int i = 0; i < 4; ++i) {
        const unsigned int n = (sel >> (4 * i)) & 0x7u;
        r |= (unsigned int)((src >> (8 * n)) & 0xffu) << (8 * i);
    }
    return r;
}
static inline float __uint_as_float(unsigned int u) { float f; memcpy(&f, &u, 4); return f; }
static inline unsigned int __float_as_uint(float f) { unsigned int u; memcpy(&u, &f, 4); return u; }
// CTAs run on several OS threads: global atomics must be real ones (shared
// memory of a CTA is only touched by its own fibers, one OS thread)
static inline unsigned int atomicAdd(unsigned int *p, unsigned int v) {
    return __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
}
static inline int min(int a, int b) { return a < b ? a : b; }
static inline int max(int a, int b) { return a > b ? a : b; }

// ------------------------------------------------------------ runtime API
typedef int cudaError_t;
typedef void *cudaStream_t;
typedef void *cudaEvent_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorInvalidValue = 1 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice,
                      cudaMemcpyHostToHost, cudaMemcpyDefault };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaHostAllocDefault = 0 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaFuncAttributePreferredSharedMemoryCarveout = 9 };
struct cudaDeviceProp { int multiProcessorCount; size_t sharedMemPerBlockOptin; int major, minor; int l2CacheSize; };
struct cudaPointerAttributes { int type; };
enum { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2 };

static inline const char *cudaGetErrorString(cudaError_t e) { return e ? "emulated CUDA error" : "no error"; }
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline cudaError_t cudaPeekAtLastError() { return cudaSuccess; }
static inline cudaError_t cudaGetDeviceCount(int *n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int *d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp *p, int) {
    p->multiProcessorCount = 148; p->sharedMemPerBlockOptin = 227 * 1024; p->major = 10; p->minor = 0;
    p->l2CacheSize = 126 << 20;
    return cudaSuccess;
}
static inline cudaError_t cudaMalloc(void **p, size_t n) {
    *p = aligned_alloc(256, (n + 255) / 256 * 256);
    return *p ? cudaSuccess : cudaErrorMemoryAllocation;
}
template <typename T> static inline cudaError_t cudaMalloc(T **p, size_t n) { return cudaMalloc((void **)p, n); }
static inline cudaError_t cudaFree(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaMallocHost(void **p, size_t n) { return cudaMalloc(p, n); }
template <typename T> static inline cudaError_t cudaMallocHost(T **p, size_t n) { return cudaMalloc((void **)p, n); }
static inline cudaError_t cudaHostAlloc(void **p, size_t n, unsigned) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFreeHost(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void *d, const void *s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void *d, int v, size_t n, cudaStream_t = nullptr) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void *d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemset2DAsync(void *d, size_t pitch, int v, size_t width, size_t height, cudaStream_t = nullptr) {
    for (size_t r = 0; r < height; ++r) memset((char *)d + r * pitch, v, width);
    return cudaSuccess;
}
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned) { *s = (void *)1; return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned) { *e = (void *)1; return cudaSuccess; }
static inline cudaError_t cudaEventCreate(cudaEvent_t *e) { *e = (void *)1; return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = nullptr) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float *ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes *a, const void *) { a->type = cudaMemoryTypeUnregistered; return cudaSuccess; }
template <typename T> static inline cudaError_t cudaMemcpyToSymbol(T &sym, const void *src, size_t n) { memcpy((void *)&sym, src, n); return cudaSuccess; }
template <typename T> static inline cudaError_t cudaMemcpyToSymbolAsync(T &sym, const void *src, size_t n, size_t, cudaMemcpyKind, cudaStream_t) { memcpy((void *)&sym, src, n); return cudaSuccess; }
template <typename F> static inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return cudaSuccess; }
