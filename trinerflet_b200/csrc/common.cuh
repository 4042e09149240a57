// Shared helpers for the trinerflet_b200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/trinerflet_b200.h"

namespace tnl {

void set_error(const char* fmt, ...);

// Launch-status convention of the C ABI: 0 = ok, >0 = cudaError_t, <0 = argument error.
inline int finish_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}

#define TNL_ARG_CHECK(cond, msg)                      \
    do {                                              \
        if (!(cond)) {                                \
            tnl::set_error("%s: %s", __func__, msg);  \
            return TNL_ERR_INVALID_ARGUMENT;          \
        }                                             \
    } while (0)

template <typename T>
__host__ __device__ inline T ceil_div(T a, T b) { return (a + b - 1) / b; }

constexpr int kNumSM = 148;  // B200

// sum over the 32 lanes of a warp by a fixed xor tree: every lane gets the same bits, whatever the schedule
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace tnl
