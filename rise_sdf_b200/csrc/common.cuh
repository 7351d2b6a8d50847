// Shared helpers for the sm_100a kernels of librsdf_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rsdf_b200.h"

#define RSDF_EBADARG (-1)
#define RSDF_ECAPACITY (-2)

#define RSDF_LAUNCH_CHECK()                         \
    do {                                            \
        cudaError_t e__ = cudaGetLastError();       \
        if (e__ != cudaSuccess) return (int)e__;    \
    } while (0)

static inline int rsdf_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// launch a kernel with `smem` bytes of dynamic shared memory (above the 48 KB default: the limit is raised first)
template <class... P, class... A>
static inline int rsdf_launch(void (*kernel)(P...), int grid, int block, size_t smem, void *stream, const A &...args) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kernel<<<grid, block, smem, (cudaStream_t)stream>>>(args...);
    RSDF_LAUNCH_CHECK();
    return 0;
}

// B200: 148 SMs.  Grid-stride kernels size their grids as a multiple of this.
#define RSDF_NUM_SMS 148

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
// full-precision sigmoid (parity-critical paths)
__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
