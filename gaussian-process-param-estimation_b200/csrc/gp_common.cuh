// Shared helpers for the gpgp CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>

#define GP_TILE 128  // every dense matrix is padded to a multiple of this (identity padding)

#define GP_CUDA_CHECK(expr)                                   \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return -(int)_e - 1000;        \
    } while (0)

#define GP_LAUNCH_CHECK()                                     \
    do {                                                      \
        cudaError_t _e = cudaGetLastError();                  \
        if (_e != cudaSuccess) return -(int)_e - 1000;        \
    } while (0)

namespace gp {

// number of kernels launched by this library in this process (bench.py reports it as gpu_launches)
extern std::atomic<unsigned long long> g_launch_count;
#define GP_COUNT(k) (gp::g_launch_count.fetch_add((unsigned long long)(k), std::memory_order_relaxed))

// FP64 tensor-core MMA, D(8x8) += A(8x4) * B(4x8); lowers to DMMA.8x8x4 on sm_100a.
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile(
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(d0), "+d"(d1)
        : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum; result valid in thread 0. `red` must hold >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    int nw = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nw) ? red[threadIdx.x] : 0.0;
    if (w == 0) v = warp_sum(v);
    return v;
}

}  // namespace gp
