// Sigma / color MLP heads on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM) -- sm_100a only.
//
// Same behavioural contract as mlp.cu (NeRFNetwork.forward under fp16 autocast,
// /root/reference/reconstruction/nerf/network.py:118-166): fp16 operands, fp32 accumulation, fp16-rounded layer
// outputs, ReLU on the fp16 value, sigma = exp(float(h2[0])), SH degree 4 in fp32 rounded to fp16, fp32 sigmoid of the
// fp16 logits rounded to fp16; backward = the autocast backward (fp16 activation gradients, fp32 weight gradients).
//
// Mapping.  CTA = 128 threads = one 128-point tile per iteration (persistent over tiles); thread t owns point t:
// it owns TMEM lane t, so after every product it reads its own accumulator row with tcgen05.ld, applies the
// activation / rounding, and writes the row of the next operand tile into shared memory.  All operand tiles use the
// un-swizzled canonical layout (umma.cuh) so that one copy of a tile serves every product it takes part in:
//   forward      h_l  [128 x N]  = act_{l-1} (K-major A) x W_l        (K-major B)      M = 128
//   input grad   dIn  [128 x K]  = dOut_l    (K-major A) x W_l        (MN-major B)     M = 128
//   weight grad  dW_l [64  x K] += dOut_l    (MN-major A, contraction over the 128 points) x In_l (MN-major B)   M = 64
// The five weight-gradient accumulators stay in TMEM for the whole kernel (fp32) and are flushed once per CTA.
// One elected thread issues the MMAs of a stage, tcgen05.commit arrives on an mbarrier, everybody waits on it.
#include "common.cuh"
#include "mlp_math.cuh"
#include "mlp_tc.cuh"
#include "mlp_tc_util.cuh"
#include "sample_coords.cuh"
#include "umma.cuh"
#include <stdlib.h>

namespace tnl {
using namespace umma;

// ------------------------------------------------------------------------------------------------
// packed weights: the five fp16 weight tiles, in the order / layout they have in shared memory
//   W1 tile(64, K1) | W2 tile(16, 64) rows = reference rows (0 = sigma logit, 1..15 = geo) | W3 tile(64, 32) columns
//   0..15 SH, 16..30 geo, 31 zero | W4 tile(64, 64) | W5 tile(16, 64) rows 0..2 real, 3..15 zero
// ------------------------------------------------------------------------------------------------
template <int K1>
struct TcW {
    static constexpr uint32_t W1 = 0;
    static constexpr uint32_t W2 = W1 + tile_bytes(64, K1);
    static constexpr uint32_t W3 = W2 + tile_bytes(16, 64);
    static constexpr uint32_t W4 = W3 + tile_bytes(64, 32);
    static constexpr uint32_t W5 = W4 + tile_bytes(64, 64);
    static constexpr uint32_t END = W5 + tile_bytes(16, 64);
};

__global__ void k_mlp_tc_pack(int K1, int H, const float* __restrict__ W1, const float* __restrict__ W2, const float* __restrict__ W3,
                              const float* __restrict__ W4, const float* __restrict__ W5, uint8_t* __restrict__ out) {
    // H = hidden = hidden_color (64: this file, 128: mlp_tc128.cu); tile shapes W1 (H, K1) | W2 (16, H) | W3 (H, 32) | W4 (H, H) | W5 (16, H)
    const uint32_t n1 = H * K1, n2 = 16 * H, n3 = H * 32, n4 = H * H, n5 = 16 * H;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t base = 0, R, Cc;
    float v;
    if (i < n1) { R = H; Cc = K1; v = W1[i]; }
    else if ((i -= n1, base += n1 * 2, i < n2)) { R = 16; Cc = H; v = W2[i]; }
    else if ((i -= n2, base += n2 * 2, i < n3)) { R = H; Cc = 32; const uint32_t r = i / 32, c = i % 32; v = c < 31 ? W3[r * 31 + c] : 0.f; }
    else if ((i -= n3, base += n3 * 2, i < n4)) { R = H; Cc = H; v = W4[i]; }
    else if ((i -= n4, base += n4 * 2, i < n5)) { R = 16; Cc = H; v = (i / H) < 3 ? W5[i] : 0.f; }
    else return;
    const uint32_t r = i / Cc, c = i % Cc;
    *reinterpret_cast<__half*>(out + base + tile_off(R, r, c)) = __float2half_rn(v);
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int K1>
struct TcFwdSmem {
    static constexpr uint32_t X = TcW<K1>::END;                      // feat tile(128, K1); reused for [SH | geo | 0] tile(128, 32)
    static constexpr uint32_t I3 = X;                                //   (the feature tile is dead once h1 has been computed)
    static constexpr uint32_t XB = tile_bytes(128, K1) > tile_bytes(128, 32) ? tile_bytes(128, K1) : tile_bytes(128, 32);
    static constexpr uint32_t ACT = X + XB;                          // h1 / h3 / h4 tile(128, 64)
    static constexpr uint32_t BAR = ACT + tile_bytes(128, 64);       // mbarrier (8 B) + TMEM base slot (4 B)
    static constexpr uint32_t TOTAL = BAR + 16;
};

template <int K1, bool COLOR>
__global__ void __launch_bounds__(128)
k_mlp_tc_fwd(const uint8_t* __restrict__ wpk, const __half* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
             const int32_t* __restrict__ n_valid_ptr, float* __restrict__ sigma, float* __restrict__ rgb, float* __restrict__ geo) {
    using W = TcW<K1>;
    using S = TcFwdSmem<K1>;
    constexpr uint32_t TM_A = 0, TM_B = 64, TM_COLS = 128;   // 64-wide and 16-wide accumulators
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + S::BAR + 8);
    for (uint32_t i = tid * 16; i < W::END; i += 128 * 16) *reinterpret_cast<uint4*>(smem + i) = __ldg(reinterpret_cast<const uint4*>(wpk + i));
    if (tid == 0) { mbar_init(bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(tslot, TM_COLS);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t trow = tmem + ((warp * 32u) << 16);
    const uint32_t sb4 = smem_u32(smem) >> 4;
    const uint32_t X4 = sb4 + (S::X >> 4), A4 = sb4 + (S::ACT >> 4);
    const uint32_t W14 = sb4 + (W::W1 >> 4), W24 = sb4 + (W::W2 >> 4), W34 = sb4 + (W::W3 >> 4), W44 = sb4 + (W::W4 >> 4), W54 = sb4 + (W::W5 >> 4);
    uint32_t phase = 0;
    const uint32_t nvalid = clamp_valid(n_valid_ptr, M);
    const uint32_t ntiles = ceil_div(nvalid, 128u);
#define TNL_STAGE(ISSUE)                   \
    fence_async_smem();                    \
    fence_before_sync();                   \
    __syncthreads();                       \
    if (warp == 0) {                       \
        fence_after_sync();                \
        ISSUE;                             \
        commit_elected(bar);               \
    }                                      \
    mbar_wait(bar, phase); phase ^= 1;     \
    fence_after_sync()
    uint4 x[K1 / 8];
    {
        const uint32_t p0 = blockIdx.x * 128 + tid;
        const uint4* src = reinterpret_cast<const uint4*>(feat + (size_t)p0 * K1);
#pragma unroll
        for (int kc = 0; kc < K1 / 8; ++kc) x[kc] = p0 < nvalid ? __ldg(src + kc) : make_uint4(0u, 0u, 0u, 0u);
    }
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint32_t p = tile * 128 + tid;
        const bool v = p < nvalid;
#pragma unroll
        for (int kc = 0; kc < K1 / 8; ++kc) *reinterpret_cast<uint4*>(smem + S::X + (kc * 128 + tid) * 16) = x[kc];
        float d[3] = {0.f, 0.f, 0.f};
        if (COLOR && v) { d[0] = __ldg(dirs + 3 * (size_t)p); d[1] = __ldg(dirs + 3 * (size_t)p + 1); d[2] = __ldg(dirs + 3 * (size_t)p + 2); }
        // h1 = feat W1^T
        TNL_STAGE(mma_group<K1 / 16>(tmem + TM_A, op_kmajor(X4, 128, 0, 0), op_kmajor(W14, 64, 0, 0), make_idesc(128, 64, false, false), false));
        {   // prefetch the next tile's feature row; consumed at the top of the next iteration
            const uint32_t pn = (tile + gridDim.x) * 128 + tid;
            const uint4* src = reinterpret_cast<const uint4*>(feat + (size_t)pn * K1);
            const bool vn = pn < nvalid;
#pragma unroll
            for (int kc = 0; kc < K1 / 8; ++kc) x[kc] = vn ? __ldg(src + kc) : make_uint4(0u, 0u, 0u, 0u);
        }
        {
            float a[64];
            tmem_load_row<64>(trow + TM_A, a);
#pragma unroll
            for (int kc = 0; kc < 8; ++kc) *reinterpret_cast<uint4*>(smem + S::ACT + (kc * 128 + tid) * 16) = pack8<true>(a + 8 * kc);
        }
        // h2 = relu(h1) W2^T
        TNL_STAGE(mma_group<4>(tmem + TM_B, op_kmajor(A4, 128, 0, 0), op_kmajor(W24, 16, 0, 0), make_idesc(128, 16, false, false), false));
        float h2[16];
        tmem_load_row<16>(trow + TM_B, h2);
#pragma unroll
        for (int j = 0; j < 16; ++j) h2[j] = r16(h2[j]);
        if (p < M) {
            sigma[p] = v ? expf(h2[0]) : 0.f;
            if (geo) {
#pragma unroll
                for (int j = 0; j < 15; ++j) geo[15 * (size_t)p + j] = v ? h2[1 + j] : 0.f;
            }
        }
        if (!COLOR) continue;
        {   // color_net input row: [fp16(SH16(d)) | geo | 0]
            float in3[32];
            {
                float sh[16];
                sh16(d[0], d[1], d[2], sh);
#pragma unroll
                for (int j = 0; j < 16; ++j) in3[j] = sh[j];
            }
#pragma unroll
            for (int j = 0; j < 15; ++j) in3[16 + j] = h2[1 + j];
            in3[31] = 0.f;
#pragma unroll
            for (int kc = 0; kc < 4; ++kc) *reinterpret_cast<uint4*>(smem + S::I3 + (kc * 128 + tid) * 16) = pack8<false>(in3 + 8 * kc);
        }
        // h3 = in3 W3^T
        TNL_STAGE(mma_group<2>(tmem + TM_A, op_kmajor(X4, 128, 0, 0), op_kmajor(W34, 64, 0, 0), make_idesc(128, 64, false, false), false));
        {
            float a[64];
            tmem_load_row<64>(trow + TM_A, a);
#pragma unroll
            for (int kc = 0; kc < 8; ++kc) *reinterpret_cast<uint4*>(smem + S::ACT + (kc * 128 + tid) * 16) = pack8<true>(a + 8 * kc);
        }
        // h4 = relu(h3) W4^T
        TNL_STAGE(mma_group<4>(tmem + TM_A, op_kmajor(A4, 128, 0, 0), op_kmajor(W44, 64, 0, 0), make_idesc(128, 64, false, false), false));
        {
            float a[64];
            tmem_load_row<64>(trow + TM_A, a);
#pragma unroll
            for (int kc = 0; kc < 8; ++kc) *reinterpret_cast<uint4*>(smem + S::ACT + (kc * 128 + tid) * 16) = pack8<true>(a + 8 * kc);
        }
        // o5 = relu(h4) W5^T
        TNL_STAGE(mma_group<4>(tmem + TM_B, op_kmajor(A4, 128, 0, 0), op_kmajor(W54, 16, 0, 0), make_idesc(128, 16, false, false), false));
        {
            float o[8];
            tmem_load_row<8>(trow + TM_B, o);
            if (p < M && rgb) {
#pragma unroll
                for (int j = 0; j < 3; ++j) rgb[3 * (size_t)p + j] = v ? r16(sigmoidf_(r16(o[j]))) : 0.f;
            }
        }
    }
#undef TNL_STAGE
    // rows past the last tile that holds valid points: defined zeros
    for (uint32_t p = ntiles * 128 + blockIdx.x * 128 + tid; p < M; p += gridDim.x * 128) {
        sigma[p] = 0.f;
        if (COLOR && rgb) { rgb[3 * (size_t)p] = 0.f; rgb[3 * (size_t)p + 1] = 0.f; rgb[3 * (size_t)p + 2] = 0.f; }
        if (geo) for (int j = 0; j < 15; ++j) geo[15 * (size_t)p + j] = 0.f;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, TM_COLS);
}

// ------------------------------------------------------------------------------------------------
// backward.  CTA = 17 warps: two 128-point sub-tiles in flight (own shared-memory tiles, own chain accumulator in TMEM), each
// served by TWO warpgroups that split the accumulator columns of every epilogue (thread (t, hf): point t <-> TMEM lane t,
// column half hf; warps w and w + 8 share a lane quarter), and one MMA-issuer warp.  The epilogues (tcgen05.ld -> convert ->
// st.shared) are latency-bound, so twice the threads per tile nearly halves them.  A sub-tile's 256 threads hand a stage to
// the issuer through an mbarrier (`ready`, 256 arrivals), the issuer's tcgen05.commit arrives on the sub-tile's `done`
// barrier.  The issuer serves the sub-tiles alternately, so the tensor core works on one while the other runs its epilogue;
// being the only issuer it also keeps the accumulation order of the shared weight-gradient accumulators defined.
// ------------------------------------------------------------------------------------------------
template <int K1>
struct TcBwdSmem {
    // one sub-tile
    static constexpr uint32_t X = 0;                              // feat            tile(128, K1)
    static constexpr uint32_t H1 = X + tile_bytes(128, K1);       // relu(h1) -> dh1 tile(128, 64)
    static constexpr uint32_t I3 = H1 + tile_bytes(128, 64);      // in3 tile(128, 32) -> dh2 tile(128, 16)
    static constexpr uint32_t H3 = I3 + tile_bytes(128, 32);      // relu(h3) -> dh3
    static constexpr uint32_t H4 = H3 + tile_bytes(128, 64);      // relu(h4) -> dh4
    static constexpr uint32_t D5 = H4 + tile_bytes(128, 64);      // d5 tile(128, 16)
    static constexpr uint32_t SUB = D5 + tile_bytes(128, 16);
    // whole CTA
    static constexpr uint32_t SUB0 = TcW<K1>::END;
    static constexpr uint32_t BAR = SUB0 + 2 * SUB;               // ready[2], done[2] (8 B each), TMEM base slot
    static constexpr uint32_t TOTAL = BAR + 48;
};

// lane of the TMEM accumulator that holds row i of an M = 64 product (cta_group::1): rows 16w .. 16w+15 live in
// lanes 32w .. 32w+15 (the lower half of every warp's lane quarter) -- pinned by tests/test_gpu_umma.py
__device__ __forceinline__ bool m64_row_of_lane(uint32_t warp, uint32_t lane, uint32_t& row) {
    row = warp * 16 + lane;
    return lane < 16;
}

constexpr int kBwdStages = 10;

// SCATTER variant: tile row i is point perm[i] (the cell order of tnl_cell_sort, rows >= *n_valid last), and the input
// gradient goes straight into the planes instead of into g_feat: the adjoint of the tri-plane gather (k_sample_bwd4 of
// sample.cu) applied to the fp16-rounded row, so the [M, K1] gradient stream never leaves the SM.
struct PlaneScatter {
    const int32_t* perm;
    const float* xyz;
    float* g_planes;      // [3][R][R][C] fp32, accumulated
    int R;
    float inv_bound;
    int fp16_coords;
};

__device__ __forceinline__ void red_add_v4(float* addr, float4 v, float w) {   // (same instruction as sample.cu's scatter)
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" ::"l"(addr), "f"(v.x * w), "f"(v.y * w), "f"(v.z * w),
                 "f"(v.w * w)
                 : "memory");
}

// DIRS variant: stage 7 takes d(in3) over all 32 columns, and the point's thread applies the SH Jacobian at its direction to the
// fp16-rounded SH columns (0..15) -> g_dirs [M,3] (valid rows only).
template <int K1, bool SCATTER, bool DIRS, bool DET = false>
__global__ void __launch_bounds__(544, 1)
k_mlp_tc_bwd(const uint8_t* __restrict__ wpk, const __half* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
             const int32_t* __restrict__ n_valid_ptr, const float* __restrict__ g_sigma, const float* __restrict__ g_rgb,
             __half* __restrict__ g_feat, float* __restrict__ gW1, float* __restrict__ gW2, float* __restrict__ gW3,
             float* __restrict__ gW4, float* __restrict__ gW5, unsigned long long* __restrict__ dbg, const PlaneScatter sc,
             float* __restrict__ g_dirs) {
    static_assert(!(SCATTER && DIRS), "the direction gradient is not on the training path");
    using W = TcW<K1>;
    using S = TcBwdSmem<K1>;
    // TMEM columns: chain accumulators of the two warpgroups | dW1 [64 x K1] | dW4 [64 x 64] | dW3 [64 x 32] | dW2^T, dW5^T [64 x 16]
    constexpr uint32_t CW = K1 < 64 ? 64 : K1;
    constexpr uint32_t TM_C = 0, TM_W1 = 2 * CW, TM_W4 = TM_W1 + K1, TM_W3 = TM_W4 + 64, TM_W2 = TM_W3 + 32, TM_W5 = TM_W2 + 16;
    constexpr uint32_t TM_COLS = 512;
    static_assert(TM_W5 + 16 <= TM_COLS, "TMEM column budget");
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* ready = reinterpret_cast<uint64_t*>(smem + S::BAR);
    uint64_t* done = reinterpret_cast<uint64_t*>(smem + S::BAR + 16);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + S::BAR + 32);
    for (uint32_t i = tid * 16; i < W::END; i += 544 * 16) *reinterpret_cast<uint4*>(smem + i) = __ldg(reinterpret_cast<const uint4*>(wpk + i));
    if (tid == 0) {
        mbar_init(&ready[0], 256); mbar_init(&ready[1], 256);
        mbar_init(&done[0], 1); mbar_init(&done[1], 1);
        mbar_init_fence();
    }
    if (warp == 16) tmem_alloc(tslot, TM_COLS);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t nvalid = clamp_valid(n_valid_ptr, M);
    const uint32_t ntiles = ceil_div(nvalid, 128u);
    const uint32_t npairs = ceil_div(ntiles, 2u);
    const uint32_t my_pairs = blockIdx.x < npairs ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;

    __shared__ unsigned long long sdbg[64];
    const bool profiling = dbg != nullptr && blockIdx.x == 0;
    if (profiling && tid < 64) sdbg[tid] = 0ull;
    if (profiling) __syncthreads();
    if (warp == 16) {
        // ============================== MMA issuer (whole warp, converged; one elected lane issues) ==============================
        const uint32_t sb4 = smem_u32(smem) >> 4;
        const uint32_t W14 = sb4 + (W::W1 >> 4), W24 = sb4 + (W::W2 >> 4), W34 = sb4 + (W::W3 >> 4), W44 = sb4 + (W::W4 >> 4),
                       W54 = sb4 + (W::W5 >> 4);
        uint32_t ph[2] = {0u, 0u};
        for (uint32_t it = 0; it < my_pairs; ++it) {
#pragma unroll
            for (int st = 0; st < kBwdStages; ++st) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    const uint32_t sub = sb4 + ((S::SUB0 + g * S::SUB) >> 4);
                    const uint32_t tc = tmem + TM_C + g * CW;
                    const bool accw = !(it == 0 && g == 0);   // weight-gradient accumulators: initialised by the very first product
                    const uint32_t X4 = sub + (S::X >> 4), H14 = sub + (S::H1 >> 4), I34 = sub + (S::I3 >> 4), H34 = sub + (S::H3 >> 4),
                                   H44 = sub + (S::H4 >> 4), D54 = sub + (S::D5 >> 4);
                    long long c0 = 0, c1 = 0;
                    if (profiling) c0 = clock64();
                    mbar_wait(&ready[g], ph[g]); ph[g] ^= 1;
                    fence_after_sync();
                    if (profiling) c1 = clock64();
                    if (st == 0) {          // h1 = feat W1^T
                        mma_group<K1 / 16>(tc, op_kmajor(X4, 128, 0, 0), op_kmajor(W14, 64, 0, 0), make_idesc(128, 64, false, false), false);
                    } else if (st == 1) {   // h2 = relu(h1) W2^T
                        mma_group<4>(tc, op_kmajor(H14, 128, 0, 0), op_kmajor(W24, 16, 0, 0), make_idesc(128, 16, false, false), false);
                    } else if (st == 2) {   // h3 = in3 W3^T
                        mma_group<2>(tc, op_kmajor(I34, 128, 0, 0), op_kmajor(W34, 64, 0, 0), make_idesc(128, 64, false, false), false);
                    } else if (st == 3) {   // h4 = relu(h3) W4^T
                        mma_group<4>(tc, op_kmajor(H34, 128, 0, 0), op_kmajor(W44, 64, 0, 0), make_idesc(128, 64, false, false), false);
                    } else if (st == 4) {   // o5 = relu(h4) W5^T
                        mma_group<4>(tc, op_kmajor(H44, 128, 0, 0), op_kmajor(W54, 16, 0, 0), make_idesc(128, 16, false, false), false);
                    } else if (st == 5) {   // dh4 = d5 W5 ;  dW5^T += h4^T d5
                        mma_group<1>(tc, op_kmajor(D54, 128, 0, 0), op_mnmajor(W54, 16, 0, 0), make_idesc(128, 64, false, true), false);
                        mma_group<8>(tmem + TM_W5, op_mnmajor(H44, 128, 0, 0), op_mnmajor(D54, 128, 0, 0), make_idesc(64, 16, true, true), accw);
                    } else if (st == 6) {   // dh3 = dh4 W4 ;  dW4 += dh4^T h3
                        mma_group<4>(tc, op_kmajor(H44, 128, 0, 0), op_mnmajor(W44, 64, 0, 0), make_idesc(128, 64, false, true), false);
                        mma_group<8>(tmem + TM_W4, op_mnmajor(H44, 128, 0, 0), op_mnmajor(H34, 128, 0, 0), make_idesc(64, 64, true, true), accw);
                    } else if (st == 7) {   // d(in3)[:, 16:32] = dh3 W3[:, 16:32] (DIRS: all of d(in3) = dh3 W3) ;  dW3 += dh3^T in3
                        if (DIRS) mma_group<4>(tc, op_kmajor(H34, 128, 0, 0), op_mnmajor(W34, 64, 0, 0), make_idesc(128, 32, false, true), false);
                        else mma_group<4>(tc, op_kmajor(H34, 128, 0, 0), op_mnmajor(W34, 64, 0, 16), make_idesc(128, 16, false, true), false);
                        mma_group<8>(tmem + TM_W3, op_mnmajor(H34, 128, 0, 0), op_mnmajor(I34, 128, 0, 0), make_idesc(64, 32, true, true), accw);
                    } else if (st == 8) {   // dh1 = dh2 W2 ;  dW2^T += h1^T dh2
                        mma_group<1>(tc, op_kmajor(I34, 128, 0, 0), op_mnmajor(W24, 16, 0, 0), make_idesc(128, 64, false, true), false);
                        mma_group<8>(tmem + TM_W2, op_mnmajor(H14, 128, 0, 0), op_mnmajor(I34, 128, 0, 0), make_idesc(64, 16, true, true), accw);
                    } else {                // g_feat = dh1 W1 ;  dW1 += dh1^T feat
                        mma_group<4>(tc, op_kmajor(H14, 128, 0, 0), op_mnmajor(W14, 64, 0, 0), make_idesc(128, K1, false, true), false);
                        mma_group<8>(tmem + TM_W1, op_mnmajor(H14, 128, 0, 0), op_mnmajor(X4, 128, 0, 0), make_idesc(64, K1, true, true), accw);
                    }
                    commit_elected(&done[g]);
                    if (profiling && lane == 0) {
                        sdbg[20 + st * 2 + g] += (unsigned long long)(c1 - c0);
                        sdbg[40 + st * 2 + g] += (unsigned long long)(clock64() - c1);
                    }
                }
            }
        }
    } else {
        // ============================== warpgroups ==============================
        const uint32_t g = (warp >> 2) & 1u, hf = warp >> 3, t = tid & 127;     // sub-tile, column half, point
        constexpr int XH = K1 / 16;                                             // feature-row chunks per half
        constexpr int KH = K1 / 2;                                              // g_feat columns per half
        uint8_t* sub = smem + S::SUB0 + g * S::SUB;
        const uint32_t trow = tmem + (((warp & 3u) * 32u) << 16) + TM_C + g * CW;
        uint32_t phase = 0;
        long long tprev = 0;
        int stg = 0;
        const bool prof = profiling && tid == 0;
        if (prof) tprev = clock64();
#define TNL_HANDOFF()                                \
    fence_async_smem();                              \
    fence_before_sync();                             \
    if (prof) { const long long c = clock64(); sdbg[10 + stg] += (unsigned long long)(c - tprev); tprev = c; } \
    mbar_arrive(&ready[g]);                          \
    mbar_wait(&done[g], phase); phase ^= 1;          \
    fence_after_sync();                              \
    if (prof) { const long long c = clock64(); sdbg[stg] += (unsigned long long)(c - tprev); tprev = c; stg = (stg + 1) % kBwdStages; }
        // this thread's 32 of the 64 accumulator columns -> fp16 row chunks of a tile(128, 64); in place masked by the ReLU output
#define TNL_EPI_RELU(TILE)                                                                                              \
    {                                                                                                                   \
        float a[32];                                                                                                    \
        tmem_load_row<32>(trow + hf * 32u, a);                                                                          \
        _Pragma("unroll") for (int kc = 0; kc < 4; ++kc)                                                                \
            *reinterpret_cast<uint4*>(sub + (TILE) + ((hf * 4u + kc) * 128u + t) * 16u) = pack8<true>(a + 8 * kc);     \
    }
#define TNL_EPI_MASK(TILE)                                                                                              \
    {                                                                                                                   \
        float a[32];                                                                                                    \
        tmem_load_row<32>(trow + hf * 32u, a);                                                                          \
        _Pragma("unroll") for (int kc = 0; kc < 4; ++kc) {                                                              \
            uint4* q = reinterpret_cast<uint4*>(sub + (TILE) + ((hf * 4u + kc) * 128u + t) * 16u);                      \
            *q = mask8(pack8<false>(a + 8 * kc), *q);                                                                   \
        }                                                                                                               \
    }
        // first tile's feature row; mx = the point it belongs to (row i of the tile sequence is point i, or perm[i])
        uint4 x[XH];
        uint32_t mx;
        {
            const uint32_t p0 = (2 * blockIdx.x + g) * 128 + t;
            const bool v0 = my_pairs > 0 && p0 < nvalid;
            mx = (SCATTER && v0) ? (uint32_t)__ldg(sc.perm + p0) : p0;
            const uint4* src = reinterpret_cast<const uint4*>(feat + (size_t)mx * K1) + hf * XH;
#pragma unroll
            for (int kc = 0; kc < XH; ++kc) x[kc] = v0 ? __ldg(src + kc) : make_uint4(0u, 0u, 0u, 0u);
        }
        for (uint32_t it = 0; it < my_pairs; ++it) {
            const uint32_t tile = 2 * (blockIdx.x + it * gridDim.x) + g;
            const uint32_t p = tile * 128 + t;
            const bool v = p < nvalid;
            const uint32_t m = mx;
#pragma unroll
            for (int kc = 0; kc < XH; ++kc) *reinterpret_cast<uint4*>(sub + S::X + ((hf * XH + kc) * 128 + t) * 16) = x[kc];
            float d[3] = {0.f, 0.f, 0.f}, gr[3] = {0.f, 0.f, 0.f}, gs = 0.f;
            if (v && hf == 0) {            // (the 16-column stages are half 0's)
#pragma unroll
                for (int j = 0; j < 3; ++j) { d[j] = __ldg(dirs + 3 * (size_t)m + j); gr[j] = __ldg(g_rgb + 3 * (size_t)m + j); }
                gs = __ldg(g_sigma + m);
            }
            TNL_HANDOFF();   // stage 0
            {   // prefetch the next tile's feature row; it is consumed at the top of the next iteration
                const uint32_t pn = (2 * (blockIdx.x + (it + 1) * gridDim.x) + g) * 128 + t;
                const bool vn = (it + 1 < my_pairs) && pn < nvalid;
                mx = (SCATTER && vn) ? (uint32_t)__ldg(sc.perm + pn) : pn;
                const uint4* src = reinterpret_cast<const uint4*>(feat + (size_t)mx * K1) + hf * XH;
#pragma unroll
                for (int kc = 0; kc < XH; ++kc) x[kc] = vn ? __ldg(src + kc) : make_uint4(0u, 0u, 0u, 0u);
            }
            TNL_EPI_RELU(S::H1);
            TNL_HANDOFF();   // stage 1
            float logit = 0.f;
            if (hf == 0) {
                float h2[16];
                tmem_load_row<16>(trow, h2);
#pragma unroll
                for (int j = 0; j < 16; ++j) h2[j] = r16(h2[j]);
                logit = h2[0];
                float in3[32];
                {
                    float sh[16];
                    sh16(d[0], d[1], d[2], sh);
#pragma unroll
                    for (int j = 0; j < 16; ++j) in3[j] = sh[j];
                }
#pragma unroll
                for (int j = 0; j < 15; ++j) in3[16 + j] = h2[1 + j];
                in3[31] = 0.f;
#pragma unroll
                for (int kc = 0; kc < 4; ++kc) *reinterpret_cast<uint4*>(sub + S::I3 + (kc * 128 + t) * 16) = pack8<false>(in3 + 8 * kc);
            }
            TNL_HANDOFF();   // stage 2
            TNL_EPI_RELU(S::H3);
            TNL_HANDOFF();   // stage 3
            TNL_EPI_RELU(S::H4);
            TNL_HANDOFF();   // stage 4
            if (hf == 0) {   // d5 = half(g_rgb) * s * (1 - s), rounded to fp16; columns 3..15 zero
                float o[8];
                tmem_load_row<8>(trow, o);
                float d5[8];
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const float sg = r16(sigmoidf_(r16(o[j])));
                    d5[j] = v ? r16(gr[j]) * sg * (1.f - sg) : 0.f;
                }
#pragma unroll
                for (int j = 3; j < 8; ++j) d5[j] = 0.f;
                *reinterpret_cast<uint4*>(sub + S::D5 + (0 * 128 + t) * 16) = pack8<false>(d5);
                *reinterpret_cast<uint4*>(sub + S::D5 + (1 * 128 + t) * 16) = make_uint4(0u, 0u, 0u, 0u);
            }
            TNL_HANDOFF();   // stage 5
            TNL_EPI_MASK(S::H4);
            TNL_HANDOFF();   // stage 6
            TNL_EPI_MASK(S::H3);
            TNL_HANDOFF();   // stage 7
            float pos[3] = {0.f, 0.f, 0.f};   // the point's position, for the scatter after stage 9 (loaded two stages ahead)
            if (SCATTER && v) {
#pragma unroll
                for (int j = 0; j < 3; ++j) pos[j] = __ldg(sc.xyz + 3 * (size_t)m + j);
            }
            if (hf == 0) {   // dh2: column 0 <- g_sigma * exp(clamp(logit, -15, 15)) (trunc_exp backward), columns 1..15 <- d(geo)
                float a[16];
                tmem_load_row<16>(trow + (DIRS ? 16u : 0u), a);
                float dh2[16];
                dh2[0] = gs * expf(fminf(fmaxf(logit, -15.f), 15.f));
#pragma unroll
                for (int j = 0; j < 15; ++j) dh2[1 + j] = a[j];
                *reinterpret_cast<uint4*>(sub + S::I3 + (0 * 128 + t) * 16) = pack8<false>(dh2);
                *reinterpret_cast<uint4*>(sub + S::I3 + (1 * 128 + t) * 16) = pack8<false>(dh2 + 8);
                if constexpr (DIRS) {   // the SH columns, rounded to fp16 as the autocast linear backward returns them
                    float gsh[16];
                    tmem_load_row<16>(trow, gsh);
#pragma unroll
                    for (int j = 0; j < 16; ++j) gsh[j] = r16(gsh[j]);
                    if (v) {
                        float gd[3];
                        sh_backward<16>(d[0], d[1], d[2], gsh, gd);
#pragma unroll
                        for (int j = 0; j < 3; ++j) g_dirs[3 * (size_t)m + j] = gd[j];
                    }
                }
            }
            TNL_HANDOFF();   // stage 8
            TNL_EPI_MASK(S::H1);
            TNL_HANDOFF();   // stage 9
            if constexpr (SCATTER) {
                // 1. the row's input gradient, rounded to fp16 as the g_feat store of the unfused path rounds it, and the point's
                //    projected coordinates go to a staging area in the H3 | H4 tiles: both are dead from here until the next tile's
                //    stage-2 epilogue, which no thread reaches before all 256 have handed off that tile's stage 0, i.e. finished below
                constexpr int C = K1 / 3, CH = KH % 16 == 0 ? 16 : 8, RS = 2 * K1 + 16;   // row stride padded: conflict-free stores
                static_assert(128 * RS + 128 * 12 <= 2 * tile_bytes(128, 64), "staging area exceeds the H3 | H4 tiles");
                uint8_t* stg = sub + S::H3;
                float* su = reinterpret_cast<float*>(stg + 128 * RS);
#pragma unroll
                for (int j = 0; j < KH / CH; ++j) {
                    float a[CH];
                    tmem_load_row<CH>(trow + hf * KH + j * CH, a);
#pragma unroll
                    for (int kc = 0; kc < CH / 8; ++kc)
                        *reinterpret_cast<uint4*>(stg + t * RS + (hf * KH + j * CH + 8 * kc) * 2) = pack8<false>(a + 8 * kc);
                }
                if (hf == 0) {
#pragma unroll
                    for (int j = 0; j < 3; ++j) su[3 * t + j] = project_coord(pos[j], sc.inv_bound, sc.fp16_coords);
                }
                asm volatile("bar.sync %0, 256;" ::"r"(1u + g) : "memory");   // the sub-tile's two warpgroups
                // 2. the adjoint of the gather with k_sample_bwd4's mapping: thread <-> (point, plane, 4-channel group), so that
                //    the C / 4 lanes of one (point, plane) add to one contiguous run of texel channels per corner
                const uint32_t r = hf * 128 + t;
                const uint32_t nvt = nvalid - tile * 128 < 128u ? nvalid - tile * 128 : 128u;   // valid rows of this tile
#pragma unroll 4
                for (int k = 0; k < K1 / 8; ++k) {       // 128 * K1 / 4 tasks over 256 threads
                    const uint32_t task = k * 256 + r;
                    const uint32_t q = task % (C / 4), pl = (task / (C / 4)) % 3, pt = task / (3 * C / 4);
                    if (pt >= nvt) break;
                    const float4 gq = unpack4h(*reinterpret_cast<const uint2*>(stg + pt * RS + (pl * C + 4 * q) * 2));
                    if (gq.x == 0.f && gq.y == 0.f && gq.z == 0.f && gq.w == 0.f) continue;   // adding zeros is a no-op
                    // plane 0 samples (u_x, u_z), plane 1 (u_x, u_y), plane 2 (u_y, u_z): plane_coords of sample_coords.cuh
                    const float* u = su + 3 * pt;
                    const Tap tp = make_tap(pl == 2 ? u[1] : u[0], pl == 1 ? u[1] : u[2], sc.R);
                    float* base = sc.g_planes + (((size_t)pl * sc.R + tp.y0) * sc.R + tp.x0) * C + 4 * q;
                    const size_t dx = (size_t)C, dy = (size_t)sc.R * C;
                    red_add_v4(base, gq, tp.nw);
                    if (tp.x1ok) red_add_v4(base + dx, gq, tp.ne);
                    if (tp.y1ok) red_add_v4(base + dy, gq, tp.sw);
                    if (tp.x1ok && tp.y1ok) red_add_v4(base + dy + dx, gq, tp.se);
                }
            } else {
                float a[KH];
                tmem_load_row<KH>(trow + hf * KH, a);
                if (g_feat && p < M) {
                    uint4* dst = reinterpret_cast<uint4*>(g_feat + (size_t)p * K1 + hf * KH);
#pragma unroll
                    for (int kc = 0; kc < KH / 8; ++kc) dst[kc] = v ? pack8<false>(a + 8 * kc) : make_uint4(0u, 0u, 0u, 0u);
                }
            }
            // the next sub-tile's stage-0 hand-off is ordered behind these loads, so the issuer cannot overwrite the accumulator early
        }
#undef TNL_HANDOFF
#undef TNL_EPI_RELU
#undef TNL_EPI_MASK
    }
    // every product has completed: each warpgroup waited on the commit that followed its last one
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    if (profiling && tid < 64) dbg[tid] += sdbg[tid];
    // ---------------- flush the weight gradients (fp32, one atomicAdd per element per CTA) ----------------
    if (warp < 4 && my_pairs > 0) {
        if constexpr (DET) {   // this CTA's slot of the workspace (wgrad_add)
            const size_t o = (size_t)blockIdx.x * wgrad_slot(K1, 64).size;
            gW1 += o; gW2 += o; gW3 += o; gW4 += o; gW5 += o;
        }
        const uint32_t tl = tmem + ((warp * 32u) << 16);
        uint32_t row;
        const bool have = m64_row_of_lane(warp, lane, row);
#pragma unroll 1
        for (int c0 = 0; c0 < K1; c0 += 16) {
            float a[16];
            tmem_load_row<16>(tl + TM_W1 + c0, a);
            if (have)
#pragma unroll
                for (int k = 0; k < 16; ++k) wgrad_add<DET>(gW1 + (size_t)row * K1 + c0 + k, a[k]);
        }
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += 16) {
            float a[16];
            tmem_load_row<16>(tl + TM_W4 + c0, a);
            if (have)
#pragma unroll
                for (int k = 0; k < 16; ++k) wgrad_add<DET>(gW4 + (size_t)row * 64 + c0 + k, a[k]);
        }
        {
            float a[32];
            tmem_load_row<32>(tl + TM_W3, a);
            if (have)
#pragma unroll
                for (int k = 0; k < 31; ++k) wgrad_add<DET>(gW3 + (size_t)row * 31 + k, a[k]);
        }
        {   // transposed accumulators: lane row = input feature k, column = output row n
            float a[16];
            tmem_load_row<16>(tl + TM_W2, a);
            if (have)
#pragma unroll
                for (int n = 0; n < 16; ++n) wgrad_add<DET>(gW2 + (size_t)n * 64 + row, a[n]);
            float b[16];
            tmem_load_row<16>(tl + TM_W5, b);
            if (have)
#pragma unroll
                for (int n = 0; n < 3; ++n) wgrad_add<DET>(gW5 + (size_t)n * 64 + row, b[n]);
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 16) tmem_free(tmem, TM_COLS);
}

// ------------------------------------------------------------------------------------------------
// probe: one product with operands given as plain row-major fp16 matrices, raw TMEM dump.  Used by
// profiles/probe_umma.py and tests/test_gpu_umma.py to pin the descriptor conventions on real hardware.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_umma_probe(const __half* __restrict__ A, int a_rows, int a_cols, const __half* __restrict__ B, int b_rows, int b_cols, int a_mn,
             int b_mn, int Mm, int Nn, int Kk, float* __restrict__ out, int ncols) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tslot;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const uint32_t a_bytes = tile_bytes(a_rows, a_cols);
    for (int i = tid; i < a_rows * a_cols; i += 128) *reinterpret_cast<__half*>(smem + tile_off(a_rows, i / a_cols, i % a_cols)) = A[i];
    for (int i = tid; i < b_rows * b_cols; i += 128) *reinterpret_cast<__half*>(smem + a_bytes + tile_off(b_rows, i / b_cols, i % b_cols)) = B[i];
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tslot, 256);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tslot;
    const uint32_t sb = smem_u32(smem);
    if (tid == 0) {
        const uint32_t idesc = make_idesc(Mm, Nn, a_mn != 0, b_mn != 0);
        for (int ks = 0; ks < Kk / 16; ++ks) {
            const uint64_t a = a_mn ? desc_mnmajor(sb, a_rows, 16 * ks, 0) : desc_kmajor(sb, a_rows, 0, 16 * ks);
            const uint64_t b = b_mn ? desc_mnmajor(sb + a_bytes, b_rows, 16 * ks, 0) : desc_kmajor(sb + a_bytes, b_rows, 0, 16 * ks);
            mma_f16(tmem, a, b, idesc, ks > 0 ? 1u : 0u);
        }
        commit(&bar);
    }
    mbar_wait(&bar, 0);
    fence_after_sync();
    for (int c = 0; c < ncols; c += 8) {
        uint32_t r[8];
        tmem_ld8(tmem + ((warp * 32u) << 16) + c, r);
        tmem_ld_wait();
        pin<8>(r);
        for (int j = 0; j < 8; ++j) out[(size_t)tid * ncols + c + j] = __uint_as_float(r[j]);
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 256);
}

// micro-benchmark: `reps` rounds of one product's K loop issued back to back by one thread; cycles from first issue to
// completion -> out[0] (tensor-pipe cost of one shape / operand layout, profiles/bench_umma.py)
__global__ void __launch_bounds__(128)
k_umma_bench(int a_rows, int b_rows, int a_mn, int b_mn, int Mm, int Nn, int Kk, int reps, long long* __restrict__ out) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tslot;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    for (uint32_t i = tid * 16; i < 160 * 1024; i += 128 * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tslot, 256);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tslot;
    const uint32_t sb4 = smem_u32(smem) >> 4;
    if (tid == 0) {
        const uint32_t idesc = make_idesc(Mm, Nn, a_mn != 0, b_mn != 0);
        const Operand a = a_mn ? op_mnmajor(sb4, a_rows, 0, 0) : op_kmajor(sb4, a_rows, 0, 0);
        const Operand b = b_mn ? op_mnmajor(sb4 + 4096, b_rows, 0, 0) : op_kmajor(sb4 + 4096, b_rows, 0, 0);
        const long long c0 = clock64();
        for (int r = 0; r < reps; ++r) mma_steps(tmem, a, b, idesc, Kk / 16, r > 0);
        const long long c1 = clock64();
        commit(&bar);
        mbar_wait(&bar, 0);
        const long long c2 = clock64();
        out[0] = c2 - c0;
        out[1] = c1 - c0;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 256);
}

// same with free descriptor fields (16-byte units) and layout type, to compare swizzle modes; operand contents are zero
__global__ void __launch_bounds__(128)
k_umma_bench2(uint32_t a_lbo, uint32_t a_sbo, uint32_t a_step, uint32_t a_type, uint32_t b_lbo, uint32_t b_sbo, uint32_t b_step,
              uint32_t b_type, int a_mn, int b_mn, int Mm, int Nn, int ksteps, int reps, long long* __restrict__ out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tslot;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    for (uint32_t i = tid * 16; i < 160 * 1024; i += 128 * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tslot, 256);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tslot;
    const uint32_t sb4 = smem_u32(smem) >> 4;
    if (warp == 0) {
        const uint32_t idesc = make_idesc(Mm, Nn, a_mn != 0, b_mn != 0);
        Operand a, b;
        a.lo = (sb4 & 0x3FFFu) | (a_lbo << 16); a.hi = a_sbo | (1u << 14) | (a_type << 29); a.step = a_step;
        b.lo = ((sb4 + 4096) & 0x3FFFu) | (b_lbo << 16); b.hi = b_sbo | (1u << 14) | (b_type << 29); b.step = b_step;
        const long long c0 = clock64();
        for (int r = 0; r < reps; ++r) {
            if (ksteps == 4) mma_group<4>(tmem, a, b, idesc, r > 0);
            else mma_group<8>(tmem, a, b, idesc, r > 0);
        }
        const long long c1 = clock64();
        commit_elected(&bar);
        mbar_wait(&bar, 0);
        const long long c2 = clock64();
        if (tid == 0) { out[0] = c2 - c0; out[1] = c1 - c0; }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
// host side (called from mlp.cu's C-ABI entry points)
// ------------------------------------------------------------------------------------------------
bool mlp_tc_supported(uint32_t in_dim, uint32_t hidden, uint32_t hidden_c) {
    if (hidden != hidden_c) return false;
    if (hidden == 64) return in_dim == 48 || in_dim == 96;                       // C = 16 / 32 (small / base configs): this file
    if (hidden == 128) return in_dim == 48 || in_dim == 96 || in_dim == 144;      // "large" heads: mlp_tc128.cu
    return false;
}

size_t mlp_tc_packed_bytes(uint32_t in_dim, uint32_t hidden) {
    return 2 * ((size_t)hidden * in_dim + 16 * hidden + 32 * hidden + (size_t)hidden * hidden + 16 * hidden);
}

void mlp_tc_pack(uint32_t in_dim, uint32_t hidden, const float* W1, const float* W2, const float* W3, const float* W4, const float* W5,
                 void* out, cudaStream_t s) {
    const uint32_t total = (uint32_t)(mlp_tc_packed_bytes(in_dim, hidden) / 2);
    k_mlp_tc_pack<<<ceil_div(total, 256u), 256, 0, s>>>((int)in_dim, (int)hidden, W1, W2, W3, W4, W5, static_cast<uint8_t*>(out));
}

template <int K1>
static void launch_fwd(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, float* sigma,
                       float* rgb, float* geo, cudaStream_t s) {
    using S = TcFwdSmem<K1>;
    // (the attribute is per device and setting it is cheap: no process-wide "already set" flag)
    cudaFuncSetAttribute(k_mlp_tc_fwd<K1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
    cudaFuncSetAttribute(k_mlp_tc_fwd<K1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
    const uint32_t per_sm = (227u * 1024u) / (S::TOTAL + 1024u);
    const uint32_t blocks = min(ceil_div(M, 128u), (uint32_t)kNumSM * (per_sm < 1 ? 1u : per_sm));
    if (dirs)
        k_mlp_tc_fwd<K1, true><<<blocks, 128, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M,
                                                              n_valid, sigma, rgb, geo);
    else
        k_mlp_tc_fwd<K1, false><<<blocks, 128, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M,
                                                               n_valid, sigma, rgb, geo);
}

void mlp_tc_forward(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                    const int32_t* n_valid, float* sigma, float* rgb, float* geo, cudaStream_t s) {
    if (hidden == 128) { mlp_tc128_forward(in_dim, wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s); return; }
    if (in_dim == 48) launch_fwd<48>(wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s);
    else launch_fwd<96>(wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s);
}

// optional device buffer of 64 cycle counters (tnl_mlp_tc_profile); nullptr in normal operation
static unsigned long long* g_tc_dbg = nullptr;

uint32_t mlp_tc_backward_blocks(uint32_t hidden, uint32_t M) {
    // one CTA per SM: it owns all 512 TMEM columns; a CTA of the 64-wide kernel takes two 128-point tiles at a time
    return min(ceil_div(M, hidden == 128 ? 128u : 256u), (uint32_t)kNumSM);
}

template <int K1, bool SCATTER, bool DIRS, bool DET = false>
static void launch_bwd(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, const float* g_sigma,
                       const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3, float* gW4, float* gW5, const PlaneScatter& sc,
                       float* g_dirs, cudaStream_t s) {
    using S = TcBwdSmem<K1>;
    cudaFuncSetAttribute(k_mlp_tc_bwd<K1, SCATTER, DIRS, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
    const uint32_t blocks = mlp_tc_backward_blocks(64, M);
    k_mlp_tc_bwd<K1, SCATTER, DIRS, DET><<<blocks, 544, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M,
                                                                  n_valid, g_sigma, g_rgb, static_cast<__half*>(g_feat), gW1, gW2, gW3, gW4,
                                                                  gW5, g_tc_dbg, sc, g_dirs);
}

void mlp_tc_backward(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                     const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3,
                     float* gW4, float* gW5, cudaStream_t s) {
    if (hidden == 128) {
        mlp_tc128_backward(in_dim, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, nullptr, s);
        return;
    }
    const PlaneScatter none{};
    if (in_dim == 48) launch_bwd<48, false, false>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, none, nullptr, s);
    else launch_bwd<96, false, false>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, none, nullptr, s);
}

void mlp_tc_backward_dirs(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                          const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2,
                          float* gW3, float* gW4, float* gW5, float* g_dirs, cudaStream_t s) {
    if (hidden == 128) {
        mlp_tc128_backward(in_dim, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, g_dirs, s);
        return;
    }
    const PlaneScatter none{};
    if (in_dim == 48) launch_bwd<48, false, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, none, g_dirs, s);
    else launch_bwd<96, false, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, none, g_dirs, s);
}

void mlp_tc_backward_det(uint32_t in_dim, uint32_t hidden, const void* wpk, const void* feat, const float* dirs, uint32_t M,
                         const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* slots, float* g_dirs,
                         cudaStream_t s) {
    if (hidden == 128) {
        mlp_tc128_backward_det(in_dim, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, slots, g_dirs, s);
        return;
    }
    const PlaneScatter none{};
    const WgradSlot L = wgrad_slot(in_dim, 64);
    float *w1 = slots, *w2 = slots + L.o2, *w3 = slots + L.o3, *w4 = slots + L.o4, *w5 = slots + L.o5;
    if (in_dim == 48) {
        if (g_dirs) launch_bwd<48, false, true, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, none, g_dirs, s);
        else launch_bwd<48, false, false, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, none, nullptr, s);
    } else {
        if (g_dirs) launch_bwd<96, false, true, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, none, g_dirs, s);
        else launch_bwd<96, false, false, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, none, nullptr, s);
    }
}

}  // namespace tnl

using namespace tnl;

extern "C" int tnl_mlp_tc_profile(unsigned long long* counters64) {
    g_tc_dbg = counters64;
    return 0;
}

extern "C" int tnl_mlp_backward_scatter(const tnl_mlp_dims* dims, const void* packed, const void* feat, const float* dirs, uint32_t M,
                                        const int32_t* n_valid, const int32_t* perm, const float* g_sigma, const float* g_rgb,
                                        const float* xyz, uint32_t R, uint32_t C, float inv_bound, int fp16_coords, float* g_planes,
                                        float* g_W1, float* g_W2, float* g_W3, float* g_W4, float* g_W5, tnl_stream_t stream) {
    if (M == 0) return 0;
    if (!dims || !mlp_tc_selected(dims) || dims->hidden != 64 || dims->in_dim != 3 * C) {
        set_error("mlp_backward_scatter: the 64-wide heads on the tcgen05 kernels (in_dim = 3C in {48, 96}, hidden = hidden_color = 64)");
        return TNL_ERR_UNSUPPORTED;
    }
    TNL_ARG_CHECK(packed && feat && dirs && perm && g_sigma && g_rgb && xyz && g_planes && g_W1 && g_W2 && g_W3 && g_W4 && g_W5,
                  "null pointer");
    TNL_ARG_CHECK(R >= 2, "R >= 2");
    TNL_ARG_CHECK(((uintptr_t)feat & 15) == 0 && ((uintptr_t)g_planes & 15) == 0, "feat/g_planes must be 16-byte aligned");
    const PlaneScatter sc{perm, xyz, g_planes, (int)R, inv_bound, fp16_coords};
    const uint8_t* wpk = static_cast<const uint8_t*>(packed) + mlp_tc_packed_offset(dims);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (C == 16) launch_bwd<48, true, false>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, nullptr, g_W1, g_W2, g_W3, g_W4, g_W5, sc, nullptr, s);
    else launch_bwd<96, true, false>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, nullptr, g_W1, g_W2, g_W3, g_W4, g_W5, sc, nullptr, s);
    return finish_launch("mlp_backward_scatter(tcgen05)");
}

extern "C" int tnl_umma_bench(int a_rows, int b_rows, int a_mn, int b_mn, int M, int N, int K, int reps, long long* out2,
                              tnl_stream_t stream) {
    TNL_ARG_CHECK(out2, "null pointer");
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(k_umma_bench, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        attr = true;
    }
    k_umma_bench<<<1, 128, 160 * 1024, reinterpret_cast<cudaStream_t>(stream)>>>(a_rows, b_rows, a_mn, b_mn, M, N, K, reps, out2);
    return finish_launch("umma_bench");
}

extern "C" int tnl_umma_bench2(uint32_t a_lbo, uint32_t a_sbo, uint32_t a_step, uint32_t a_type, uint32_t b_lbo, uint32_t b_sbo,
                               uint32_t b_step, uint32_t b_type, int a_mn, int b_mn, int M, int N, int ksteps, int reps, long long* out2,
                               tnl_stream_t stream) {
    TNL_ARG_CHECK(out2 && (ksteps == 4 || ksteps == 8), "bench2: ksteps must be 4 or 8");
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(k_umma_bench2, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        attr = true;
    }
    k_umma_bench2<<<1, 128, 160 * 1024, reinterpret_cast<cudaStream_t>(stream)>>>(a_lbo, a_sbo, a_step, a_type, b_lbo, b_sbo, b_step, b_type,
                                                                                  a_mn, b_mn, M, N, ksteps, reps, out2);
    return finish_launch("umma_bench2");
}

extern "C" int tnl_umma_probe(const void* A, int a_rows, int a_cols, const void* B, int b_rows, int b_cols, int a_mn, int b_mn, int M,
                              int N, int K, float* out, int ncols, tnl_stream_t stream) {
    TNL_ARG_CHECK(A && B && out, "null pointer");
    TNL_ARG_CHECK(a_rows % 8 == 0 && a_cols % 8 == 0 && b_rows % 8 == 0 && b_cols % 8 == 0 && K % 16 == 0 && ncols % 8 == 0 && ncols <= 256,
                  "probe: dimensions must be multiples of 8 (K of 16), at most 256 columns dumped");
    const size_t bytes = (size_t)a_rows * a_cols * 2 + (size_t)b_rows * b_cols * 2;
    TNL_ARG_CHECK(bytes <= 200 * 1024, "probe: operands exceed shared memory");
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(k_umma_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr = true;
    }
    k_umma_probe<<<1, 128, bytes, reinterpret_cast<cudaStream_t>(stream)>>>(static_cast<const __half*>(A), a_rows, a_cols,
                                                                            static_cast<const __half*>(B), b_rows, b_cols, a_mn, b_mn, M,
                                                                            N, K, out, ncols);
    return finish_launch("umma_probe");
}
