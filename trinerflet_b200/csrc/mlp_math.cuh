// Scalar pieces shared by the two fused-MLP implementations (mlp.cu: mma.sync, mlp_tc.cu: tcgen05): fp16 packing with
// the autocast rounding, SH degree 4 (shencoder.cu:50-68 of the reference), sigmoid.
#pragma once
#include <cuda_fp16.h>
#include <stddef.h>
#include <stdint.h>

namespace tnl {

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ uint32_t relu_h2(uint32_t v) {
    __half2 h = *reinterpret_cast<__half2*>(&v);
    h = __hmax2(h, __float2half2_rn(0.f));
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t v) { return __half22float2(*reinterpret_cast<__half2*>(&v)); }

__device__ __forceinline__ void sh16(float x, float y, float z, float (&o)[16]) {
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    o[0] = 0.28209479177387814f;
    o[1] = -0.48860251190291987f * y;
    o[2] = 0.48860251190291987f * z;
    o[3] = -0.48860251190291987f * x;
    o[4] = 1.0925484305920792f * xy;
    o[5] = -1.0925484305920792f * yz;
    o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
    o[7] = -1.0925484305920792f * xz;
    o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
    o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2);
    o[10] = 2.8906114426405538f * xy * z;
    o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
    o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
    o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
    o[14] = 1.4453057213202769f * z * (x2 - y2);
    o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
}

// Jacobian of sh16: J[a][ch] = d o[ch] / d (x, y, z)[a] (the reference's dy_dx, shencoder.cu kernel_sh)
__device__ __forceinline__ void sh16_jacobian(float x, float y, float z, float (&jx)[16], float (&jy)[16], float (&jz)[16]) {
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    jx[0] = 0.f; jy[0] = 0.f; jz[0] = 0.f;
    jx[1] = 0.f; jy[1] = -0.48860251190291987f; jz[1] = 0.f;
    jx[2] = 0.f; jy[2] = 0.f; jz[2] = 0.48860251190291987f;
    jx[3] = -0.48860251190291987f; jy[3] = 0.f; jz[3] = 0.f;
    jx[4] = 1.0925484305920792f * y; jy[4] = 1.0925484305920792f * x; jz[4] = 0.f;
    jx[5] = 0.f; jy[5] = -1.0925484305920792f * z; jz[5] = -1.0925484305920792f * y;
    jx[6] = 0.f; jy[6] = 0.f; jz[6] = 1.89234939151512f * z;
    jx[7] = -1.0925484305920792f * z; jy[7] = 0.f; jz[7] = -1.0925484305920792f * x;
    jx[8] = 1.0925484305920792f * x; jy[8] = -1.0925484305920792f * y; jz[8] = 0.f;
    jx[9] = -3.540261539559861f * xy; jy[9] = 1.7701307697799304f * (-x2 + y2); jz[9] = 0.f;
    jx[10] = 2.8906114426405538f * yz; jy[10] = 2.8906114426405538f * xz; jz[10] = 2.8906114426405538f * xy;
    jx[11] = 0.f; jy[11] = 0.45704579946446572f - 2.2852289973223288f * z2; jz[11] = -4.5704579946446575f * yz;
    jx[12] = 0.f; jy[12] = 0.f; jz[12] = 5.597644988851731f * z2 - 1.1195289977703462f;
    jx[13] = 0.45704579946446572f - 2.2852289973223288f * z2; jy[13] = 0.f; jz[13] = -4.5704579946446575f * xz;
    jx[14] = 2.8906114426405538f * xz; jy[14] = -2.8906114426405538f * yz; jz[14] = 1.4453057213202769f * (x2 - y2);
    jx[15] = 1.7701307697799304f * (-x2 + y2); jy[15] = 3.540261539559861f * xy; jz[15] = 0.f;
}

// g_d[a] = sum_ch g[ch] J[a][ch] over the first NCH = degree^2 channels, accumulated in channel order as the reference's
// kernel_sh_backward does
template <int NCH>
__device__ __forceinline__ void sh_backward(float x, float y, float z, const float* g, float (&gd)[3]) {
    float jx[16], jy[16], jz[16];
    sh16_jacobian(x, y, z, jx, jy, jz);
    gd[0] = gd[1] = gd[2] = 0.f;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        gd[0] = fmaf(g[ch], jx[ch], gd[0]);
        gd[1] = fmaf(g[ch], jy[ch], gd[1]);
        gd[2] = fmaf(g[ch], jz[ch], gd[2]);
    }
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float r16(float v) { return __half2float(__float2half_rn(v)); }

// Weight-gradient flush of the backward kernels.  Default: one fp32 atomicAdd per element per CTA (the sum depends on the CTA
// order).  DET (tnl_mlp_backward_det): the CTA writes its partial sums to its own slot of a workspace instead, and
// k_wgrad_reduce adds the slots in index order.  A slot holds g_W1 | g_W2 | g_W3 | g_W4 | g_W5 (fp32, their shapes).
struct WgradSlot {
    size_t o2, o3, o4, o5, size;   // offsets of g_W2 .. g_W5 and the slot size, in floats
};
__host__ __device__ constexpr WgradSlot wgrad_slot(uint32_t K1, uint32_t H) {
    return WgradSlot{(size_t)H * K1, (size_t)H * K1 + 16 * H, (size_t)H * K1 + 16 * H + 31 * H, (size_t)H * K1 + 47 * H + (size_t)H * H,
                     (size_t)H * K1 + 50 * H + (size_t)H * H};
}
template <bool DET>
__device__ __forceinline__ void wgrad_add(float* p, float v) {
    if constexpr (DET) *p = v;
    else atomicAdd(p, v);
}

}  // namespace tnl
