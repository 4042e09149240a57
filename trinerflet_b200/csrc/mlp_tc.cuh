// Host-side entry points of the tcgen05 implementation of the fused MLP heads (mlp_tc.cu: 64-wide heads, mlp_tc128.cu:
// 128-wide heads); called by the C-ABI functions in mlp.cu when the feature stream is fp16.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include "../../include/trinerflet_b200.h"
#include <stdint.h>

namespace tnl {

bool mlp_tc_supported(uint32_t in_dim, uint32_t hidden, uint32_t hidden_c);
size_t mlp_tc_packed_bytes(uint32_t in_dim, uint32_t hidden);
void mlp_tc_pack(uint32_t in_dim, uint32_t hidden, const float* W1, const float* W2, const float* W3, const float* W4, const float* W5,
                 void* out, cudaStream_t s);
void mlp_tc_forward(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                    const int32_t* n_valid, float* sigma, float* rgb, float* geo, cudaStream_t s);
void mlp_tc_backward(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                     const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3,
                     float* gW4, float* gW5, cudaStream_t s);
// the same, also writing the direction gradient g_dirs [M,3] of the valid rows (tnl_mlp_backward_dirs)
void mlp_tc_backward_dirs(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                          const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2,
                          float* gW3, float* gW4, float* gW5, float* g_dirs, cudaStream_t s);
// the same with the weight gradients written per CTA into `slots` (layout wgrad_slot, one slot per CTA, mlp_tc_backward_blocks
// of them; tnl_mlp_backward_det reduces them); g_dirs may be nullptr
void mlp_tc_backward_det(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                         const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* slots, float* g_dirs,
                         cudaStream_t s);
// CTAs of the tcgen05 backward kernels for M points
uint32_t mlp_tc_backward_blocks(uint32_t hidden, uint32_t M);
// mlp.cu: where the tcgen05 tiles start inside the packed weight block, and whether the tcgen05 kernels serve these dims
// (fp16 feature stream, not forced off by TNL_MLP_LEGACY)
size_t mlp_tc_packed_offset(const tnl_mlp_dims* dims);
bool mlp_tc_selected(const tnl_mlp_dims* dims);
// mlp_tc128.cu
void mlp_tc128_forward(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                       float* sigma, float* rgb, float* geo, cudaStream_t s);
void mlp_tc128_backward(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                        const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3, float* gW4, float* gW5, float* g_dirs,
                        cudaStream_t s);
void mlp_tc128_backward_det(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                            const float* g_sigma, const float* g_rgb, void* g_feat, float* slots, float* g_dirs, cudaStream_t s);

}  // namespace tnl
