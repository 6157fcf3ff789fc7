// cuda_compat.cuh — the two spellings that differ between the nvcc build (the product) and the
// host-side SIMT emulator build of the same sources (tests/simt, test infrastructure only):
// the dynamic shared-memory declaration and the kernel launch.
#pragma once
#if defined(LT_SIMT_EMU)
#include "simt.h"        // tests/simt/ — on the include path of the emulator build only
#define LT_DEVICE_CODE 1
#else
#include <cuda_runtime.h>
#define LT_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define LT_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#if defined(__CUDACC__)
#define LT_DEVICE_CODE 1
#endif
#endif
