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
#else
#include <cuda_runtime.h>
#define ZFB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#define ZFB_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define ZFB_BUILD_KIND "sm_100a"
#endif
