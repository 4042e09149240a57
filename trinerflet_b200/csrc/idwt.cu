// Inverse 2-D DWT level (zero mode; bior6.8, haar, bior2.2, bior2.6 or bior4.4) and its exact adjoint -- sm_100a,
// channels-last.  The wavelet is a template parameter of the kernels (idwt_core.cuh: its taps in the 18-tap frame).
//
// The reference spends ~7 full-size passes per level (2 F.pad, 6 conv_transpose2d, 3 adds, see
// triplane_encoder.py:391-394 + pytorch_wavelets sfb1d); here one kernel per level reads each
// coefficient once and writes each plane element once.
//
// Layout: x [3][n][n][C], yh [3][3][n][n][C], out [3][2n][2n][C] (C fastest).  A row of pixels is one
// contiguous run of n*C floats, so "thread <-> one float of the row" is fully coalesced for any C.
//
// Kernel structure (forward; the backward kernel mirrors it), per-thread code in idwt_core.cuh:
//   CTA = one column strip (32 fine columns) x one row chunk x CG channels, NT = 24*CG threads.
//   phase A  thread <-> input column (pixel column, channel): streams rows top to bottom with 9-deep
//            register windows per sub-band (static ring indices, no register moves), emits two
//            H-synthesised rows per input row into a double-buffered shared-memory ring.  Inputs are
//            staged global->shared one step ahead with cp.async (thread-private slots; src-size 0
//            zero-fill implements the zero padding of mode='zero').
//   phase B  thread <-> (mid row, strip of 8 output columns, channel): W-axis synthesis from the mid
//            rows with a register sliding window; lanes <-> channels => 128-byte coalesced stores.
//   One __syncthreads per step (3 coarse rows).  ~35 FMA per output element => FMA-pipe / HBM
//   co-limited (DESIGN.md, "IDWT roofline").
#include "common.cuh"
#include "idwt_core.cuh"
#include <stdlib.h>

#include <type_traits>

namespace tnl {

template <typename Cfg, int W>
__global__ void __launch_bounds__(Cfg::NT, (768 / Cfg::NT) > 0 ? (768 / Cfg::NT) : 1)
k_idwt_fwd(const float* __restrict__ x, const float* __restrict__ yh, float* __restrict__ out, int n, int C,
           int rows_per_cta, float* __restrict__ abs_sum, const int4* __restrict__ items, const int* __restrict__ n_items) {
    extern __shared__ __align__(16) float smem[];
    float* mid0 = smem;
    float* stage0 = smem + 2 * Cfg::MID_F;
    const int tid = threadIdx.x;
    IdwtGeom g;
    if (items != nullptr) {   // work-list mode: blockIdx.x = item * chunks + chunk
        const int chunks = C / Cfg::CG;
        const int idx = blockIdx.x / chunks;
        if (idx >= __ldg(n_items)) return;
        const int4 it = __ldg(items + idx);
        g = idwt_geom_item<Cfg>(tid, blockIdx.x % chunks, IdwtItem{it.x, it.y, it.z, it.w}, n, C);
    } else {
        g = idwt_geom<Cfg>(tid, IdwtBlock{(int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z}, n, C, rows_per_cta);
    }
    FwdState st;
    fwd_state_init<Cfg>(st, g, x, yh, tid);
    fwd_issue_stage<Cfg>(g, st, stage0, tid);
    fwd_issue_stage<Cfg>(g, st, stage0 + Cfg::STAGE, tid);
    for (int s = 0; s < g.nsteps; s += 3) {
#define TNL_STEP(PH)                                                                          \
    if (s + PH < g.nsteps) {                                                                  \
        const int ss = s + PH;                                                                \
        fwd_issue_stage<Cfg>(g, st, stage0 + ((PH + 2) % 3) * Cfg::STAGE, tid);               \
        cp_async_wait<2>();                                                                   \
        float* mid = mid0 + (ss & 1) * Cfg::MID_F;                                            \
        fwd_phase_a<Cfg, PH, W>(g, st, stage0 + PH * Cfg::STAGE, mid, tid, ss);               \
        __syncthreads();                                                                      \
        fwd_phase_b<Cfg, W>(g, st, mid, out, ss);                                             \
    }
        TNL_STEP(0) TNL_STEP(1) TNL_STEP(2)
#undef TNL_STEP
    }
    cp_async_wait<0>();
    if (abs_sum != nullptr) {  // block-reduce the |yh| partial sums, one atomic per CTA
        float v = st.abs_acc;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        __syncthreads();
        if ((tid & 31) == 0) smem[tid >> 5] = v;
        __syncthreads();
        if (tid < 32) {
            float w = tid < (Cfg::NT + 31) / 32 ? smem[tid] : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
            if (tid == 0) atomicAdd(abs_sum, w);
        }
    }
}

template <typename Cfg, int W>
__global__ void __launch_bounds__(Cfg::NT, (768 / Cfg::NT) > 0 ? (768 / Cfg::NT) : 1)
k_idwt_bwd(const float* __restrict__ gout, float* __restrict__ g_x, float* __restrict__ g_yh, int n, int C,
           int rows_per_cta, const float* __restrict__ yh, const float* __restrict__ reg_grad, float reg_coef, int plane0,
           const int4* __restrict__ items, const int* __restrict__ n_items) {
    extern __shared__ __align__(16) float smem[];
    float* mid0 = smem;
    float* stage0 = smem + 2 * Cfg::MID_B;
    const int tid = threadIdx.x;
    IdwtGeom g;
    if (items != nullptr) {
        const int chunks = C / Cfg::CG;
        const int idx = blockIdx.x / chunks;
        if (idx >= __ldg(n_items)) return;
        const int4 it = __ldg(items + idx);
        g = idwt_geom_item<Cfg>(tid, blockIdx.x % chunks, IdwtItem{it.x, it.y, it.z, it.w}, n, C);
    } else {
        g = idwt_geom<Cfg>(tid, IdwtBlock{(int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z + plane0}, n, C, rows_per_cta);
    }
    BwdState st;
    bwd_state_init<Cfg>(st, g, gout);
    const float reg = (yh != nullptr && reg_grad != nullptr) ? reg_coef * __ldg(reg_grad) : 0.f;
    const float* yh_reg = (yh != nullptr && reg_grad != nullptr) ? yh : nullptr;
    bwd_issue_stage<Cfg>(g, st, stage0, tid);
    bwd_issue_stage<Cfg>(g, st, stage0 + Cfg::STAGE, tid);
    for (int s = 0; s < g.nsteps; s += 3) {
#define TNL_STEP(PH)                                                                          \
    if (s + PH < g.nsteps) {                                                                  \
        const int ss = s + PH;                                                                \
        bwd_issue_stage<Cfg>(g, st, stage0 + ((PH + 2) % 3) * Cfg::STAGE, tid);               \
        cp_async_wait<2>();                                                                   \
        float* mid = mid0 + (ss & 1) * Cfg::MID_B;                                            \
        bwd_phase_a<Cfg, PH, W>(st, stage0 + PH * Cfg::STAGE, mid, tid);                      \
        __syncthreads();                                                                      \
        bwd_phase_b<Cfg, W>(g, mid, g_x, g_yh, tid, ss, yh_reg, reg);                         \
    }
        TNL_STEP(0) TNL_STEP(1) TNL_STEP(2)
#undef TNL_STEP
    }
    cp_async_wait<0>();
}

// ---- clean blocks of the work-list mode: nothing to reconstruct / no incoming gradient -------------------------------
// item = {plane, m0, row_lo, row_hi}: 16 coarse columns x rows; every (row, band) is one contiguous run of 16*C floats
__global__ void __launch_bounds__(256)
k_idwt_clean_fwd(const float* __restrict__ yh, int n, int C, const int4* __restrict__ items, const int* __restrict__ n_items,
                 float* __restrict__ abs_sum) {
    __shared__ float red[8];
    const int cnt = __ldg(n_items);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc = 0.f;
    const int run4 = 16 * C / 4;
    for (int idx = blockIdx.x; idx < cnt; idx += gridDim.x) {
        const int4 it = __ldg(items + idx);
        const int rows = min(it.w, n) - it.z;
        for (int rb = warp; rb < 3 * rows; rb += 8) {          // one warp per (band, row) run of 16*C contiguous floats
            const int b = rb / rows, r = rb - b * rows;
            const float4* src = reinterpret_cast<const float4*>(yh + (((size_t)(it.x * 3 + b) * n + it.z + r) * n + it.y) * C);
            for (int q = lane; q < run4; q += 32) {
                const float4 v = __ldg(src + q);
                acc += fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(v.w);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float w = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
        if (threadIdx.x == 0 && w != 0.f) atomicAdd(abs_sum, w);
    }
}

__global__ void __launch_bounds__(256)
k_idwt_clean_bwd(const float* __restrict__ yh, float* __restrict__ g_x, float* __restrict__ g_yh, int n, int C,
                 const int4* __restrict__ items, const int* __restrict__ n_items, const float* __restrict__ reg_grad, float reg_coef,
                 float* __restrict__ abs_sum) {
    __shared__ float red[8];
    const int cnt = __ldg(n_items);
    const bool use_reg = yh != nullptr && reg_grad != nullptr;
    const float reg = use_reg ? reg_coef * __ldg(reg_grad) : 0.f;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int run4 = 16 * C / 4;
    float acc = 0.f;   // sum |yh| over the clean blocks (the forward value of the regulariser, read here anyway)
    for (int idx = blockIdx.x; idx < cnt; idx += gridDim.x) {
        const int4 it = __ldg(items + idx);
        const int rows = min(it.w, n) - it.z;
        for (int rb = warp; rb < 4 * rows; rb += 8) {          // bands 0..2: coefficient gradients; 3: the low-pass gradient
            const int b = rb / rows, r = rb - b * rows;
            if (b == 3) {
                float4* dst = reinterpret_cast<float4*>(g_x + (((size_t)it.x * n + it.z + r) * n + it.y) * C);
                for (int q = lane; q < run4; q += 32) dst[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                const size_t off = (((size_t)(it.x * 3 + b) * n + it.z + r) * n + it.y) * C;
                float4* dst = reinterpret_cast<float4*>(g_yh + off);
                if (use_reg) {   // 0 + reg * sign(yh): the same fmaf the active blocks apply to their accumulated gradient
                    const float4* src = reinterpret_cast<const float4*>(yh + off);
                    for (int q = lane; q < run4; q += 32) {
                        const float4 v = __ldg(src + q);
                        acc += fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(v.w);
                        dst[q] = make_float4(fmaf(reg, signf_(v.x), 0.f), fmaf(reg, signf_(v.y), 0.f), fmaf(reg, signf_(v.z), 0.f),
                                             fmaf(reg, signf_(v.w), 0.f));
                    }
                } else {
                    for (int q = lane; q < run4; q += 32) dst[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    }
    if (abs_sum != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x < 32) {
            float w = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
            if (threadIdx.x == 0 && w != 0.f) atomicAdd(abs_sum, w);
        }
    }
}

template <typename Cfg, int W>
static int launch_fwd_sparse(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum, const int32_t* active,
                             const int32_t* clean, const int32_t* counts, uint32_t max_active, uint32_t max_clean, uint32_t parts,
                             cudaStream_t stream) {
    // (per device, cheap: no process-wide "already set" flag -- a process may drive several devices)
    cudaFuncSetAttribute(k_idwt_fwd<Cfg, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_F);
    if (max_active > 0 && (parts & 1u))
        k_idwt_fwd<Cfg, W><<<max_active * (C / Cfg::CG), Cfg::NT, Cfg::SMEM_F, stream>>>(x, yh, out, (int)n, (int)C, 0, abs_sum,
                                                                                     reinterpret_cast<const int4*>(active), counts);
    if (abs_sum != nullptr && max_clean > 0 && (parts & 2u))
        k_idwt_clean_fwd<<<min(max_clean, (uint32_t)kNumSM * 8u), 256, 0, stream>>>(yh, (int)n, (int)C, reinterpret_cast<const int4*>(clean),
                                                                                   counts + 1, abs_sum);
    return finish_launch("idwt_level_forward_sparse");
}

template <typename Cfg, int W>
static int launch_bwd_sparse(const float* g, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh, const float* reg_grad,
                             float reg_coef, const int32_t* active, const int32_t* clean, const int32_t* counts, uint32_t max_active,
                             uint32_t max_clean, uint32_t parts, float* abs_sum, cudaStream_t stream) {
    // (per device, cheap: no process-wide "already set" flag -- a process may drive several devices)
    cudaFuncSetAttribute(k_idwt_bwd<Cfg, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_B);
    if (max_active > 0 && (parts & 1u))
        k_idwt_bwd<Cfg, W><<<max_active * (C / Cfg::CG), Cfg::NT, Cfg::SMEM_B, stream>>>(g, g_x, g_yh, (int)n, (int)C, 0, yh, reg_grad, reg_coef,
                                                                                     0, reinterpret_cast<const int4*>(active), counts);
    if (max_clean > 0 && (parts & 2u))
        k_idwt_clean_bwd<<<min(max_clean, (uint32_t)kNumSM * 8u), 256, 0, stream>>>(yh, g_x, g_yh, (int)n, (int)C,
                                                                                   reinterpret_cast<const int4*>(clean), counts + 1, reg_grad,
                                                                                   reg_coef, abs_sum);
    return finish_launch("idwt_level_backward_sparse");
}

template <typename Cfg, int W>
static int launch_fwd(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                      cudaStream_t stream) {
    // (per device, cheap: no process-wide "already set" flag -- a process may drive several devices)
    cudaFuncSetAttribute(k_idwt_fwd<Cfg, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_F);
    unsigned gx, gy, gz, rows;
    idwt_grid<Cfg>(n, C, kNumSM, gx, gy, gz, rows);
    k_idwt_fwd<Cfg, W><<<dim3(gx, gy, gz), Cfg::NT, Cfg::SMEM_F, stream>>>(x, yh, out, (int)n, (int)C, (int)rows, abs_sum, nullptr, nullptr);
    return finish_launch("idwt_level_forward");
}

template <typename Cfg, int W>
static int launch_bwd(const float* g, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                      const float* reg_grad, float reg_coef, uint32_t plane0, uint32_t nplanes, cudaStream_t stream) {
    // (per device, cheap: no process-wide "already set" flag -- a process may drive several devices)
    cudaFuncSetAttribute(k_idwt_bwd<Cfg, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_B);
    unsigned gx, gy, gz, rows;
    idwt_grid<Cfg>(n, C, kNumSM, gx, gy, gz, rows);
    gz = nplanes;
    k_idwt_bwd<Cfg, W><<<dim3(gx, gy, gz), Cfg::NT, Cfg::SMEM_B, stream>>>(g, g_x, g_yh, (int)n, (int)C, (int)rows, yh, reg_grad,
                                                                        reg_coef, (int)plane0, nullptr, nullptr);
    return finish_launch("idwt_level_backward");
}

// runtime wavelet id -> the kernels' template argument
template <typename Fn>
static int with_wavelet(uint32_t wavelet, Fn&& fn) {
    switch (wavelet) {
        case TNL_WAVELET_BIOR6_8: return fn(std::integral_constant<int, TNL_WAVELET_BIOR6_8>());
        case TNL_WAVELET_HAAR: return fn(std::integral_constant<int, TNL_WAVELET_HAAR>());
        case TNL_WAVELET_BIOR2_2: return fn(std::integral_constant<int, TNL_WAVELET_BIOR2_2>());
        case TNL_WAVELET_BIOR2_6: return fn(std::integral_constant<int, TNL_WAVELET_BIOR2_6>());
        case TNL_WAVELET_BIOR4_4: return fn(std::integral_constant<int, TNL_WAVELET_BIOR4_4>());
        default: set_error("idwt: unknown wavelet id %u", wavelet); return TNL_ERR_INVALID_ARGUMENT;
    }
}

}  // namespace tnl

using namespace tnl;

extern "C" {

int tnl_idwt_level_forward_wavelet(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                   uint32_t wavelet, tnl_stream_t stream) {
    TNL_ARG_CHECK(x && yh && out, "null pointer");
    TNL_ARG_CHECK(n >= 8 && n % 8 == 0 && n <= 16384, "n must be a multiple of 8 in [8, 16384]");
    TNL_ARG_CHECK(C >= 8 && C % 8 == 0, "C must be a multiple of 8");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return with_wavelet(wavelet, [&](auto w) {
        constexpr int W = decltype(w)::value;
        if (C % 32 == 0 && getenv("TNL_IDWT_CG32")) return launch_fwd<IdwtCfg<32, 32>, W>(x, yh, out, n, C, abs_sum, s);
        if (C % 24 == 0) return launch_fwd<IdwtCfg<24, 32>, W>(x, yh, out, n, C, abs_sum, s);
        if (C % 16 == 0) return launch_fwd<IdwtCfg<16, 32>, W>(x, yh, out, n, C, abs_sum, s);
        return launch_fwd<IdwtCfg<8, 32>, W>(x, yh, out, n, C, abs_sum, s);
    });
}

int tnl_idwt_level_backward_wavelet(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                    const float* reg_grad, float reg_coef, uint32_t plane0, uint32_t nplanes, uint32_t wavelet,
                                    tnl_stream_t stream) {
    TNL_ARG_CHECK(nplanes >= 1 && plane0 + nplanes <= 3, "plane range must lie in [0, 3)");
    TNL_ARG_CHECK(g_out && g_x && g_yh, "null pointer");
    TNL_ARG_CHECK(n >= 8 && n % 8 == 0 && n <= 16384, "n must be a multiple of 8 in [8, 16384]");
    TNL_ARG_CHECK(C >= 8 && C % 8 == 0, "C must be a multiple of 8");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return with_wavelet(wavelet, [&](auto w) {
        constexpr int W = decltype(w)::value;
        if (C % 32 == 0 && getenv("TNL_IDWT_CG32"))
            return launch_bwd<IdwtCfg<32, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, plane0, nplanes, s);
        if (C % 24 == 0) return launch_bwd<IdwtCfg<24, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, plane0, nplanes, s);
        if (C % 16 == 0) return launch_bwd<IdwtCfg<16, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, plane0, nplanes, s);
        return launch_bwd<IdwtCfg<8, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, plane0, nplanes, s);
    });
}

int tnl_idwt_level_forward_sparse_wavelet(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                          const int32_t* active, const int32_t* clean, const int32_t* counts, uint32_t max_active,
                                          uint32_t max_clean, uint32_t parts, uint32_t wavelet, tnl_stream_t stream) {
    TNL_ARG_CHECK(x && yh && out && counts, "null pointer");
    TNL_ARG_CHECK(parts >= 1 && parts <= 3, "parts: bit 0 = active blocks, bit 1 = |yh| sum of the clean blocks");
    TNL_ARG_CHECK((max_active == 0 || active) && (max_clean == 0 || clean), "null work list");
    TNL_ARG_CHECK(n >= 16 && n % 16 == 0 && n <= 16384, "work-list mode: n must be a multiple of 16 in [16, 16384]");
    TNL_ARG_CHECK(C >= 8 && C % 8 == 0, "C must be a multiple of 8");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return with_wavelet(wavelet, [&](auto w) {
        constexpr int W = decltype(w)::value;
        if (C % 24 == 0)
            return launch_fwd_sparse<IdwtCfg<24, 32>, W>(x, yh, out, n, C, abs_sum, active, clean, counts, max_active, max_clean, parts, s);
        if (C % 16 == 0)
            return launch_fwd_sparse<IdwtCfg<16, 32>, W>(x, yh, out, n, C, abs_sum, active, clean, counts, max_active, max_clean, parts, s);
        return launch_fwd_sparse<IdwtCfg<8, 32>, W>(x, yh, out, n, C, abs_sum, active, clean, counts, max_active, max_clean, parts, s);
    });
}

int tnl_idwt_level_backward_sparse_wavelet(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                           const float* reg_grad, float reg_coef, const int32_t* active, const int32_t* clean,
                                           const int32_t* counts, uint32_t max_active, uint32_t max_clean, uint32_t parts,
                                           float* abs_sum, uint32_t wavelet, tnl_stream_t stream) {
    TNL_ARG_CHECK((g_out || !(parts & 1u)) && g_x && g_yh && counts, "null pointer");
    TNL_ARG_CHECK(parts >= 1 && parts <= 3, "parts: bit 0 = active blocks, bit 1 = clean blocks");
    TNL_ARG_CHECK((max_active == 0 || active) && (max_clean == 0 || clean), "null work list");
    TNL_ARG_CHECK(n >= 16 && n % 16 == 0 && n <= 16384, "work-list mode: n must be a multiple of 16 in [16, 16384]");
    TNL_ARG_CHECK(C >= 8 && C % 8 == 0, "C must be a multiple of 8");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return with_wavelet(wavelet, [&](auto w) {
        constexpr int W = decltype(w)::value;
        if (C % 24 == 0)
            return launch_bwd_sparse<IdwtCfg<24, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, active, clean, counts, max_active,
                                                         max_clean, parts, abs_sum, s);
        if (C % 16 == 0)
            return launch_bwd_sparse<IdwtCfg<16, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, active, clean, counts, max_active,
                                                         max_clean, parts, abs_sum, s);
        return launch_bwd_sparse<IdwtCfg<8, 32>, W>(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, active, clean, counts, max_active,
                                                    max_clean, parts, abs_sum, s);
    });
}

// the bior6.8 entry points of ABI version 1
int tnl_idwt_level_forward(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                           tnl_stream_t stream) {
    return tnl_idwt_level_forward_wavelet(x, yh, out, n, C, abs_sum, TNL_WAVELET_BIOR6_8, stream);
}

int tnl_idwt_level_backward(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                            const float* reg_grad, float reg_coef, uint32_t plane0, uint32_t nplanes, tnl_stream_t stream) {
    return tnl_idwt_level_backward_wavelet(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, plane0, nplanes, TNL_WAVELET_BIOR6_8,
                                           stream);
}

int tnl_idwt_level_forward_sparse(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                  const int32_t* active, const int32_t* clean, const int32_t* counts, uint32_t max_active,
                                  uint32_t max_clean, uint32_t parts, tnl_stream_t stream) {
    return tnl_idwt_level_forward_sparse_wavelet(x, yh, out, n, C, abs_sum, active, clean, counts, max_active, max_clean, parts,
                                                 TNL_WAVELET_BIOR6_8, stream);
}

int tnl_idwt_level_backward_sparse(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                   const float* reg_grad, float reg_coef, const int32_t* active, const int32_t* clean,
                                   const int32_t* counts, uint32_t max_active, uint32_t max_clean, uint32_t parts, float* abs_sum,
                                   tnl_stream_t stream) {
    return tnl_idwt_level_backward_sparse_wavelet(g_out, g_x, g_yh, n, C, yh, reg_grad, reg_coef, active, clean, counts, max_active,
                                                  max_clean, parts, abs_sum, TNL_WAVELET_BIOR6_8, stream);
}

}  // extern "C"
