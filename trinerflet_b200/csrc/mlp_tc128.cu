// Sigma / color MLP heads, 128 wide ("large" config of the reference: --hidden_dim 128 --hidden_dim_color 128,
// /root/reference/README.md:55, reconstruction/nerf/network.py:37-74,118-147), on the 5th-generation tensor cores
// (tcgen05.mma, accumulators and weight gradients in TMEM) -- sm_100a only.  Same behavioural contract and the same
// operand-tile conventions as mlp_tc.cu (64-wide heads); what changes is the budget:
//
//   * the five fp16 weight tiles take 84 KB of shared memory (K1 = 144) and one 128-point tile's operand tiles 144 KB, so a
//     CTA holds ONE point tile (backward) and the feature tile X shares its 36 KB with relu(h4) + d5: X is consumed by the
//     first product, re-fetched (cp.async, L2-resident: the CTA read it microseconds earlier) while the input-gradient chain
//     runs, and is back in place for the last stage (g_feat = dh1 W1, dW1 += dh1^T X);
//   * every weight-gradient product is a full M = 128 product (rows = the 128 neurons of the layer), so all 128 TMEM lanes
//     carry accumulators: chain accumulator 144 columns + dW1 144 + dW4 128 + dW3 32 + dW2^T 16 + dW5^T 16 = 480 of 512;
//   * the forward kernel keeps two 128-point tiles in flight (two warpgroups + one MMA-issuer warp, as the 64-wide backward),
//     so the tensor pipe works on one tile while the other runs its epilogue.
#include "common.cuh"
#include "mlp_math.cuh"
#include "mlp_tc.cuh"
#include "mlp_tc_util.cuh"
#include "umma.cuh"

namespace tnl {
using namespace umma;

// packed weights (k_mlp_tc_pack with H = 128): W1 tile(128, K1) | W2 tile(16, 128) | W3 tile(128, 32) | W4 tile(128, 128) |
// W5 tile(16, 128)
template <int K1>
struct TcW128 {
    static constexpr uint32_t W1 = 0;
    static constexpr uint32_t W2 = W1 + tile_bytes(128, K1);
    static constexpr uint32_t W3 = W2 + tile_bytes(16, 128);
    static constexpr uint32_t W4 = W3 + tile_bytes(128, 32);
    static constexpr uint32_t W5 = W4 + tile_bytes(128, 128);
    static constexpr uint32_t END = W5 + tile_bytes(16, 128);
};

// thread t's feature row (K1 halves = K1/8 16-byte chunks) -> rows t of the X tile, asynchronously; rows past the valid
// range are zero-filled (src-size 0)
template <int K1>
__device__ __forceinline__ void load_x_async(uint8_t* xtile, uint32_t t, const __half* __restrict__ feat, uint32_t p, bool valid) {
    const __half* src = valid ? feat + (size_t)p * K1 : feat;
    const uint32_t dst = smem_u32(xtile) + t * 16u;
    const uint32_t nbytes = valid ? 16u : 0u;
#pragma unroll
    for (int kc = 0; kc < K1 / 8; ++kc)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + kc * 2048u), "l"(src + kc * 8), "r"(nbytes) : "memory");
}

// accumulator columns [0, NC) of this thread's TMEM lane -> fp16 row of a tile(128, NC), 64 columns at a time
template <int NC, bool RELU>
__device__ __forceinline__ void epi_store(uint32_t trow, uint8_t* tile, uint32_t t) {
#pragma unroll
    for (int c0 = 0; c0 < NC; c0 += 64) {
        float a[64];
        tmem_load_row<64>(trow + c0, a);
#pragma unroll
        for (int kc = 0; kc < 8; ++kc) *reinterpret_cast<uint4*>(tile + ((c0 / 8 + kc) * 128 + t) * 16) = pack8<RELU>(a + 8 * kc);
    }
}
// the same, masked by the ReLU output the tile holds (in place: relu(h) -> dh)
template <int NC>
__device__ __forceinline__ void epi_mask_store(uint32_t trow, uint8_t* tile, uint32_t t) {
#pragma unroll
    for (int c0 = 0; c0 < NC; c0 += 64) {
        float a[64];
        tmem_load_row<64>(trow + c0, a);
#pragma unroll
        for (int kc = 0; kc < 8; ++kc) {
            uint4* q = reinterpret_cast<uint4*>(tile + ((c0 / 8 + kc) * 128 + t) * 16);
            *q = mask8(pack8<false>(a + 8 * kc), *q);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// forward: CTA = two warpgroups (one 128-point tile each) + one MMA-issuer warp
// ------------------------------------------------------------------------------------------------
template <int K1>
struct TcFwd128Smem {
    static constexpr uint32_t X = 0;                                  // feat tile(128, K1); reused for [SH | geo | 0] tile(128, 32)
    static constexpr uint32_t XB = tile_bytes(128, K1) > tile_bytes(128, 32) ? tile_bytes(128, K1) : tile_bytes(128, 32);
    static constexpr uint32_t ACT = X + XB;                           // relu(h1) / relu(h3) / relu(h4) tile(128, 128)
    static constexpr uint32_t SUB = ACT + tile_bytes(128, 128);
    static constexpr uint32_t SUB0 = TcW128<K1>::END;
    static constexpr uint32_t BAR = SUB0 + 2 * SUB;                   // ready[2], done[2], TMEM base slot
    static constexpr uint32_t TOTAL = BAR + 48;
};

template <int K1, bool COLOR>
__global__ void __launch_bounds__(288, 1)
k_mlp_tc_fwd128(const uint8_t* __restrict__ wpk, const __half* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
                const int32_t* __restrict__ n_valid_ptr, float* __restrict__ sigma, float* __restrict__ rgb, float* __restrict__ geo) {
    using W = TcW128<K1>;
    using S = TcFwd128Smem<K1>;
    constexpr uint32_t TM_A = 0, TM_B = 128, TM_WG = 144, TM_COLS = 512;
    constexpr int NSTAGES = COLOR ? 5 : 2;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    uint64_t* ready = reinterpret_cast<uint64_t*>(smem + S::BAR);
    uint64_t* done = reinterpret_cast<uint64_t*>(smem + S::BAR + 16);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + S::BAR + 32);
    for (uint32_t i = tid * 16; i < W::END; i += 288 * 16) *reinterpret_cast<uint4*>(smem + i) = __ldg(reinterpret_cast<const uint4*>(wpk + i));
    if (tid == 0) {
        mbar_init(&ready[0], 128); mbar_init(&ready[1], 128);
        mbar_init(&done[0], 1); mbar_init(&done[1], 1);
        mbar_init_fence();
    }
    if (warp == 8) tmem_alloc(tslot, TM_COLS);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t nvalid = clamp_valid(n_valid_ptr, M);
    const uint32_t ntiles = ceil_div(nvalid, 128u);
    const uint32_t npairs = ceil_div(ntiles, 2u);
    const uint32_t my_pairs = blockIdx.x < npairs ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;
    if (warp == 8) {
        // ============================== MMA issuer ==============================
        const uint32_t sb4 = smem_u32(smem) >> 4;
        const uint32_t W14 = sb4 + (W::W1 >> 4), W24 = sb4 + (W::W2 >> 4), W34 = sb4 + (W::W3 >> 4), W44 = sb4 + (W::W4 >> 4),
                       W54 = sb4 + (W::W5 >> 4);
        uint32_t ph[2] = {0u, 0u};
        for (uint32_t it = 0; it < my_pairs; ++it) {
#pragma unroll
            for (int st = 0; st < NSTAGES; ++st) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    const uint32_t sub = sb4 + ((S::SUB0 + g * S::SUB) >> 4);
                    const uint32_t X4 = sub + (S::X >> 4), A4 = sub + (S::ACT >> 4);
                    const uint32_t ta = tmem + g * TM_WG + TM_A, tb = tmem + g * TM_WG + TM_B;
                    mbar_wait(&ready[g], ph[g]); ph[g] ^= 1;
                    fence_after_sync();
                    if (st == 0) {          // h1 = feat W1^T
                        mma_group<K1 / 16>(ta, op_kmajor(X4, 128, 0, 0), op_kmajor(W14, 128, 0, 0), make_idesc(128, 128, false, false), false);
                    } else if (st == 1) {   // h2 = relu(h1) W2^T
                        mma_group<8>(tb, op_kmajor(A4, 128, 0, 0), op_kmajor(W24, 16, 0, 0), make_idesc(128, 16, false, false), false);
                    } else if (st == 2) {   // h3 = in3 W3^T
                        mma_group<2>(ta, op_kmajor(X4, 128, 0, 0), op_kmajor(W34, 128, 0, 0), make_idesc(128, 128, false, false), false);
                    } else if (st == 3) {   // h4 = relu(h3) W4^T
                        mma_group<8>(ta, op_kmajor(A4, 128, 0, 0), op_kmajor(W44, 128, 0, 0), make_idesc(128, 128, false, false), false);
                    } else {                // o5 = relu(h4) W5^T
                        mma_group<8>(tb, op_kmajor(A4, 128, 0, 0), op_kmajor(W54, 16, 0, 0), make_idesc(128, 16, false, false), false);
                    }
                    commit_elected(&done[g]);
                }
            }
        }
    } else {
        // ============================== warpgroups ==============================
        const uint32_t g = warp >> 2, t = tid & 127;
        uint8_t* sub = smem + S::SUB0 + g * S::SUB;
        const uint32_t trow = tmem + (((warp & 3u) * 32u) << 16) + g * TM_WG;
        uint32_t phase = 0;
#define TNL_HANDOFF()                         \
    fence_async_smem();                       \
    fence_before_sync();                      \
    mbar_arrive(&ready[g]);                   \
    mbar_wait(&done[g], phase); phase ^= 1;   \
    fence_after_sync()
        if (my_pairs > 0) {
            const uint32_t p0 = (2 * blockIdx.x + g) * 128 + t;
            load_x_async<K1>(sub + S::X, t, feat, p0, p0 < nvalid);
        }
        for (uint32_t it = 0; it < my_pairs; ++it) {
            const uint32_t tile = 2 * (blockIdx.x + it * gridDim.x) + g;
            const uint32_t p = tile * 128 + t;
            const bool v = p < nvalid;
            const uint32_t pn = (2 * (blockIdx.x + (it + 1) * gridDim.x) + g) * 128 + t;
            const bool more = it + 1 < my_pairs;
            float d[3] = {0.f, 0.f, 0.f};
            if (COLOR && v) { d[0] = __ldg(dirs + 3 * (size_t)p); d[1] = __ldg(dirs + 3 * (size_t)p + 1); d[2] = __ldg(dirs + 3 * (size_t)p + 2); }
            cp_async_wait_all();
            TNL_HANDOFF();   // stage 0
            if (!COLOR && more) load_x_async<K1>(sub + S::X, t, feat, pn, pn < nvalid);   // (density only: X is not reused)
            epi_store<128, true>(trow + 0, sub + S::ACT, t);
            TNL_HANDOFF();   // stage 1
            float h2[16];
            tmem_load_row<16>(trow + 128, h2);
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
                for (int kc = 0; kc < 4; ++kc) *reinterpret_cast<uint4*>(sub + S::X + (kc * 128 + t) * 16) = pack8<false>(in3 + 8 * kc);
            }
            TNL_HANDOFF();   // stage 2
            if (more) load_x_async<K1>(sub + S::X, t, feat, pn, pn < nvalid);   // in3 has been consumed: fetch the next feature tile
            epi_store<128, true>(trow + 0, sub + S::ACT, t);
            TNL_HANDOFF();   // stage 3
            epi_store<128, true>(trow + 0, sub + S::ACT, t);
            TNL_HANDOFF();   // stage 4
            {
                float o[8];
                tmem_load_row<8>(trow + 128, o);
                if (p < M && rgb) {
#pragma unroll
                    for (int j = 0; j < 3; ++j) rgb[3 * (size_t)p + j] = v ? r16(sigmoidf_(r16(o[j]))) : 0.f;
                }
            }
        }
        cp_async_wait_all();
#undef TNL_HANDOFF
        // rows past the last tile pair that holds valid points: defined zeros
        for (uint32_t p = npairs * 256 + blockIdx.x * 256 + (tid & 255); p < M; p += gridDim.x * 256) {
            sigma[p] = 0.f;
            if (COLOR && rgb) { rgb[3 * (size_t)p] = 0.f; rgb[3 * (size_t)p + 1] = 0.f; rgb[3 * (size_t)p + 2] = 0.f; }
            if (geo) for (int j = 0; j < 15; ++j) geo[15 * (size_t)p + j] = 0.f;
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 8) tmem_free(tmem, TM_COLS);
}

// ------------------------------------------------------------------------------------------------
// backward: CTA = 256 threads = one 128-point tile per iteration.  Thread (t, hf): point t = tid & 127 (TMEM lane t; warps w and
// w + 4 share a lane quarter), column half hf = tid >> 7: after every product the two halves read / convert / store their own
// 64 of the 128 accumulator columns, which halves the (latency-bound) epilogue of the single tile a CTA can hold.  Warp 0
// issues the MMAs of a stage.
// ------------------------------------------------------------------------------------------------
template <int K1>
struct TcBwd128Smem {
    static constexpr uint32_t HD = tile_bytes(128, 128) + tile_bytes(128, 16);                       // relu(h4) -> dh4, then d5
    static constexpr uint32_t XRB = tile_bytes(128, K1) > HD ? tile_bytes(128, K1) : HD;
    static constexpr uint32_t XR = TcW128<K1>::END;          // feat tile(128, K1)  <->  H4 tile(128, 128) | D5 tile(128, 16)
    static constexpr uint32_t H4 = XR;
    static constexpr uint32_t D5 = XR + tile_bytes(128, 128);
    static constexpr uint32_t H1 = XR + XRB;                 // relu(h1) -> dh1
    static constexpr uint32_t I3 = H1 + tile_bytes(128, 128);   // in3 tile(128, 32) -> dh2 tile(128, 16)
    static constexpr uint32_t H3 = I3 + tile_bytes(128, 32);    // relu(h3) -> dh3
    static constexpr uint32_t BAR = H3 + tile_bytes(128, 128);
    static constexpr uint32_t TOTAL = BAR + 16;
};

// half of thread t's feature row (chunks [hf * K1/16, (hf + 1) * K1/16)) -> the X tile, asynchronously
template <int K1>
__device__ __forceinline__ void load_x_half_async(uint8_t* xtile, uint32_t t, uint32_t hf, const __half* __restrict__ feat, uint32_t p, bool valid) {
    constexpr int NCH = K1 / 16;
    const __half* src = (valid ? feat + (size_t)p * K1 : feat) + hf * NCH * 8;
    const uint32_t dst = smem_u32(xtile) + (hf * NCH * 128u + t) * 16u;
    const uint32_t nbytes = valid ? 16u : 0u;
#pragma unroll
    for (int kc = 0; kc < NCH; ++kc)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + kc * 2048u), "l"(src + kc * 8), "r"(nbytes) : "memory");
}

// DIRS: d(in3) over all 32 columns, and g_dirs [M,3] <- the SH Jacobian at the point's direction applied to the fp16-rounded
// SH columns 0..15 (valid rows only)
template <int K1, bool DIRS, bool DET = false>
__global__ void __launch_bounds__(256, 1)
k_mlp_tc_bwd128(const uint8_t* __restrict__ wpk, const __half* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
                const int32_t* __restrict__ n_valid_ptr, const float* __restrict__ g_sigma, const float* __restrict__ g_rgb,
                __half* __restrict__ g_feat, float* __restrict__ gW1, float* __restrict__ gW2, float* __restrict__ gW3,
                float* __restrict__ gW4, float* __restrict__ gW5, float* __restrict__ g_dirs) {
    using W = TcW128<K1>;
    using S = TcBwd128Smem<K1>;
    // TMEM columns: chain accumulator | dW1 [128 x K1] | dW4 [128 x 128] | dW3 [128 x 32] | dW2^T [128 x 16] | dW5^T [128 x 16]
    constexpr uint32_t CW = K1 < 128 ? 128 : K1;
    constexpr uint32_t TM_C = 0, TM_W1 = CW, TM_W4 = TM_W1 + K1, TM_W3 = TM_W4 + 128, TM_W2 = TM_W3 + 32, TM_W5 = TM_W2 + 16;
    constexpr uint32_t TM_COLS = 512;
    constexpr int KH = K1 / 2;             // g_feat / dW1 columns per half (72, 48, 24: multiples of 8)
    static_assert(TM_W5 + 16 <= TM_COLS, "TMEM column budget");
    static_assert(S::TOTAL <= 227 * 1024, "shared memory budget");
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = tid >> 5, t = tid & 127, hf = tid >> 7;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + S::BAR + 8);
    for (uint32_t i = tid * 16; i < W::END; i += 256 * 16) *reinterpret_cast<uint4*>(smem + i) = __ldg(reinterpret_cast<const uint4*>(wpk + i));
    if (tid == 0) { mbar_init(bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(tslot, TM_COLS);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t tlane = tmem + (((warp & 3u) * 32u) << 16);   // this warp's lane quarter
    const uint32_t trow = tlane + TM_C;
    const uint32_t tc = tmem + TM_C;
    const uint32_t sb4 = smem_u32(smem) >> 4;
    const uint32_t W14 = sb4 + (W::W1 >> 4), W24 = sb4 + (W::W2 >> 4), W34 = sb4 + (W::W3 >> 4), W44 = sb4 + (W::W4 >> 4), W54 = sb4 + (W::W5 >> 4);
    const uint32_t X4 = sb4 + (S::XR >> 4), H44 = sb4 + (S::H4 >> 4), D54 = sb4 + (S::D5 >> 4), H14 = sb4 + (S::H1 >> 4),
                   I34 = sb4 + (S::I3 >> 4), H34 = sb4 + (S::H3 >> 4);
    uint32_t phase = 0;
    const uint32_t nvalid = clamp_valid(n_valid_ptr, M);
    const uint32_t ntiles = ceil_div(nvalid, 128u);
    const uint32_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;
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
    // this thread's 64 of the 128 accumulator columns -> fp16 row chunks of a tile(128, 128)
#define TNL_EPI_RELU(TILE)                                                                                                   \
    {                                                                                                                        \
        float a[64];                                                                                                         \
        tmem_load_row<64>(trow + hf * 64u, a);                                                                               \
        _Pragma("unroll") for (int kc = 0; kc < 8; ++kc)                                                                     \
            *reinterpret_cast<uint4*>(smem + (TILE) + ((hf * 8u + kc) * 128u + t) * 16u) = pack8<true>(a + 8 * kc);         \
    }
#define TNL_EPI_MASK(TILE)                                                                                                   \
    {                                                                                                                        \
        float a[64];                                                                                                         \
        tmem_load_row<64>(trow + hf * 64u, a);                                                                               \
        _Pragma("unroll") for (int kc = 0; kc < 8; ++kc) {                                                                   \
            uint4* q = reinterpret_cast<uint4*>(smem + (TILE) + ((hf * 8u + kc) * 128u + t) * 16u);                          \
            *q = mask8(pack8<false>(a + 8 * kc), *q);                                                                        \
        }                                                                                                                    \
    }
    if (my_tiles > 0) {
        const uint32_t p0 = blockIdx.x * 128 + t;
        load_x_half_async<K1>(smem + S::XR, t, hf, feat, p0, p0 < nvalid);
    }
    for (uint32_t it = 0; it < my_tiles; ++it) {
        const uint32_t tile = blockIdx.x + it * gridDim.x;
        const uint32_t p = tile * 128 + t;
        const bool v = p < nvalid;
        const bool accw = it > 0;          // weight-gradient accumulators: initialised by the first tile's products
        float d[3] = {0.f, 0.f, 0.f}, gr[3] = {0.f, 0.f, 0.f}, gs = 0.f;
        if (v && hf == 0) {                // (the 16-column stages are half 0's)
#pragma unroll
            for (int j = 0; j < 3; ++j) { d[j] = __ldg(dirs + 3 * (size_t)p + j); gr[j] = __ldg(g_rgb + 3 * (size_t)p + j); }
            gs = __ldg(g_sigma + p);
        }
        cp_async_wait_all();
        // ---- recompute ----
        TNL_STAGE(mma_group<K1 / 16>(tc, op_kmajor(X4, 128, 0, 0), op_kmajor(W14, 128, 0, 0), make_idesc(128, 128, false, false), false));   // h1
        TNL_EPI_RELU(S::H1);
        TNL_STAGE(mma_group<8>(tc, op_kmajor(H14, 128, 0, 0), op_kmajor(W24, 16, 0, 0), make_idesc(128, 16, false, false), false));          // h2
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
            for (int kc = 0; kc < 4; ++kc) *reinterpret_cast<uint4*>(smem + S::I3 + (kc * 128 + t) * 16) = pack8<false>(in3 + 8 * kc);
        }
        TNL_STAGE(mma_group<2>(tc, op_kmajor(I34, 128, 0, 0), op_kmajor(W34, 128, 0, 0), make_idesc(128, 128, false, false), false));        // h3
        TNL_EPI_RELU(S::H3);
        TNL_STAGE(mma_group<8>(tc, op_kmajor(H34, 128, 0, 0), op_kmajor(W44, 128, 0, 0), make_idesc(128, 128, false, false), false));        // h4
        TNL_EPI_RELU(S::H4);               // (overwrites the feature tile: re-fetched below)
        TNL_STAGE(mma_group<8>(tc, op_kmajor(H44, 128, 0, 0), op_kmajor(W54, 16, 0, 0), make_idesc(128, 16, false, false), false));          // o5
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
            *reinterpret_cast<uint4*>(smem + S::D5 + (0 * 128 + t) * 16) = pack8<false>(d5);
            *reinterpret_cast<uint4*>(smem + S::D5 + (1 * 128 + t) * 16) = make_uint4(0u, 0u, 0u, 0u);
        }
        // ---- input-gradient chain + weight gradients ----
        TNL_STAGE((mma_group<1>(tc, op_kmajor(D54, 128, 0, 0), op_mnmajor(W54, 16, 0, 0), make_idesc(128, 128, false, true), false),         // dh4 = d5 W5
                   mma_group<8>(tmem + TM_W5, op_mnmajor(H44, 128, 0, 0), op_mnmajor(D54, 128, 0, 0), make_idesc(128, 16, true, true), accw)));   // dW5^T += h4^T d5
        TNL_EPI_MASK(S::H4);
        TNL_STAGE((mma_group<8>(tc, op_kmajor(H44, 128, 0, 0), op_mnmajor(W44, 128, 0, 0), make_idesc(128, 128, false, true), false),        // dh3 = dh4 W4
                   mma_group<8>(tmem + TM_W4, op_mnmajor(H44, 128, 0, 0), op_mnmajor(H34, 128, 0, 0), make_idesc(128, 128, true, true), accw)));  // dW4 += dh4^T h3
        load_x_half_async<K1>(smem + S::XR, t, hf, feat, p, v);   // relu(h4) / dh4 / d5 are dead: bring the feature tile back
        TNL_EPI_MASK(S::H3);
        TNL_STAGE((DIRS ? mma_group<8>(tc, op_kmajor(H34, 128, 0, 0), op_mnmajor(W34, 128, 0, 0), make_idesc(128, 32, false, true), false)   // d(in3)
                        : mma_group<8>(tc, op_kmajor(H34, 128, 0, 0), op_mnmajor(W34, 128, 0, 16), make_idesc(128, 16, false, true), false),  // d(in3)[:, 16:32]
                   mma_group<8>(tmem + TM_W3, op_mnmajor(H34, 128, 0, 0), op_mnmajor(I34, 128, 0, 0), make_idesc(128, 32, true, true), accw)));   // dW3 += dh3^T in3
        if (hf == 0) {   // dh2: column 0 <- g_sigma * exp(clamp(logit, -15, 15)) (trunc_exp backward), columns 1..15 <- d(geo)
            float a[16];
            tmem_load_row<16>(trow + (DIRS ? 16u : 0u), a);
            float dh2[16];
            dh2[0] = gs * expf(fminf(fmaxf(logit, -15.f), 15.f));
#pragma unroll
            for (int j = 0; j < 15; ++j) dh2[1 + j] = a[j];
            *reinterpret_cast<uint4*>(smem + S::I3 + (0 * 128 + t) * 16) = pack8<false>(dh2);
            *reinterpret_cast<uint4*>(smem + S::I3 + (1 * 128 + t) * 16) = pack8<false>(dh2 + 8);
            if constexpr (DIRS) {   // the SH columns, rounded to fp16 as the autocast linear backward returns them
                float gsh[16];
                tmem_load_row<16>(trow, gsh);
#pragma unroll
                for (int j = 0; j < 16; ++j) gsh[j] = r16(gsh[j]);
                if (v) {
                    float gd[3];
                    sh_backward<16>(d[0], d[1], d[2], gsh, gd);
#pragma unroll
                    for (int j = 0; j < 3; ++j) g_dirs[3 * (size_t)p + j] = gd[j];
                }
            }
        }
        TNL_STAGE((mma_group<1>(tc, op_kmajor(I34, 128, 0, 0), op_mnmajor(W24, 16, 0, 0), make_idesc(128, 128, false, true), false),         // dh1 = dh2 W2
                   mma_group<8>(tmem + TM_W2, op_mnmajor(H14, 128, 0, 0), op_mnmajor(I34, 128, 0, 0), make_idesc(128, 16, true, true), accw)));   // dW2^T += h1^T dh2
        TNL_EPI_MASK(S::H1);
        cp_async_wait_all();                                  // the feature tile is back
        TNL_STAGE((mma_group<8>(tc, op_kmajor(H14, 128, 0, 0), op_mnmajor(W14, 128, 0, 0), make_idesc(128, K1, false, true), false),         // g_feat = dh1 W1
                   mma_group<8>(tmem + TM_W1, op_mnmajor(H14, 128, 0, 0), op_mnmajor(X4, 128, 0, 0), make_idesc(128, K1, true, true), accw)));    // dW1 += dh1^T feat
        if (it + 1 < my_tiles) {                              // the feature tile has been consumed: prefetch the next one
            const uint32_t pn = (tile + gridDim.x) * 128 + t;
            load_x_half_async<K1>(smem + S::XR, t, hf, feat, pn, pn < nvalid);
        }
        {   // (tcgen05.ld is warp-collective: every lane executes it, the stores are predicated)
            float a[KH];
            tmem_load_row<KH>(trow + hf * KH, a);
            if (g_feat != nullptr && p < M) {
                uint4* dst = reinterpret_cast<uint4*>(g_feat + (size_t)p * K1 + hf * KH);
#pragma unroll
                for (int kc = 0; kc < KH / 8; ++kc) dst[kc] = v ? pack8<false>(a + 8 * kc) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
        // the next tile's first product is ordered behind these loads by the stage's __syncthreads
    }
#undef TNL_STAGE
#undef TNL_EPI_RELU
#undef TNL_EPI_MASK
    cp_async_wait_all();
    // rows of g_feat past the last processed tile: defined zeros
    if (g_feat) {
        for (uint32_t p = ntiles * 128 + blockIdx.x * 128 + t; p < M; p += gridDim.x * 128) {
            uint4* dst = reinterpret_cast<uint4*>(g_feat + (size_t)p * K1 + hf * KH);
#pragma unroll
            for (int kc = 0; kc < KH / 8; ++kc) dst[kc] = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    // ---------------- flush the weight gradients (fp32, one atomicAdd per element per CTA): TMEM lane = row ----------------
    if (my_tiles > 0) {
        if constexpr (DET) {   // this CTA's slot of the workspace (wgrad_add)
            const size_t o = (size_t)blockIdx.x * wgrad_slot(K1, 128).size;
            gW1 += o; gW2 += o; gW3 += o; gW4 += o; gW5 += o;
        }
        const uint32_t row = t;
        {
            float a[KH];
            tmem_load_row<KH>(tlane + TM_W1 + hf * KH, a);
#pragma unroll
            for (int k = 0; k < KH; ++k) wgrad_add<DET>(gW1 + (size_t)row * K1 + hf * KH + k, a[k]);
        }
        {
            float a[64];
            tmem_load_row<64>(tlane + TM_W4 + hf * 64u, a);
#pragma unroll
            for (int k = 0; k < 64; ++k) wgrad_add<DET>(gW4 + (size_t)row * 128 + hf * 64 + k, a[k]);
        }
        {
            float a[16];
            tmem_load_row<16>(tlane + TM_W3 + hf * 16u, a);
#pragma unroll
            for (int k = 0; k < 16; ++k)
                if (hf * 16 + k < 31) wgrad_add<DET>(gW3 + (size_t)row * 31 + hf * 16 + k, a[k]);
        }
        {   // transposed accumulators: lane row = input feature k, column = output row n; half 0 flushes dW2, half 1 dW5
            float a[16];
            tmem_load_row<16>(tlane + (hf == 0 ? TM_W2 : TM_W5), a);
            if (hf == 0) {
#pragma unroll
                for (int n = 0; n < 16; ++n) wgrad_add<DET>(gW2 + (size_t)n * 128 + row, a[n]);
            } else {
#pragma unroll
                for (int n = 0; n < 3; ++n) wgrad_add<DET>(gW5 + (size_t)n * 128 + row, a[n]);
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, TM_COLS);
}

// ------------------------------------------------------------------------------------------------
// host side (called from mlp_tc.cu's dispatchers)
// ------------------------------------------------------------------------------------------------
template <int K1>
static void launch_fwd128(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, float* sigma,
                          float* rgb, float* geo, cudaStream_t s) {
    using S = TcFwd128Smem<K1>;
    static_assert(S::TOTAL <= 227 * 1024, "shared memory budget");
    // (cudaFuncSetAttribute is per device and cheap: set on every launch so that a process driving several devices is correct)
    const uint32_t blocks = min(ceil_div(M, 256u), (uint32_t)kNumSM);
    if (dirs) {
        cudaFuncSetAttribute(k_mlp_tc_fwd128<K1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
        k_mlp_tc_fwd128<K1, true><<<blocks, 288, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M,
                                                               n_valid, sigma, rgb, geo);
    } else {
        cudaFuncSetAttribute(k_mlp_tc_fwd128<K1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
        k_mlp_tc_fwd128<K1, false><<<blocks, 288, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M,
                                                                n_valid, sigma, rgb, geo);
    }
}

void mlp_tc128_forward(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                       float* sigma, float* rgb, float* geo, cudaStream_t s) {
    if (in_dim == 48) launch_fwd128<48>(wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s);
    else if (in_dim == 96) launch_fwd128<96>(wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s);
    else launch_fwd128<144>(wpk, feat, dirs, M, n_valid, sigma, rgb, geo, s);
}

template <int K1, bool DIRS, bool DET = false>
static void launch_bwd128(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, const float* g_sigma,
                          const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3, float* gW4, float* gW5, float* g_dirs,
                          cudaStream_t s) {
    using S = TcBwd128Smem<K1>;
    cudaFuncSetAttribute(k_mlp_tc_bwd128<K1, DIRS, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL);
    const uint32_t blocks = mlp_tc_backward_blocks(128, M);
    k_mlp_tc_bwd128<K1, DIRS, DET><<<blocks, 256, S::TOTAL, s>>>(static_cast<const uint8_t*>(wpk), static_cast<const __half*>(feat), dirs, M, n_valid,
                                                            g_sigma, g_rgb, static_cast<__half*>(g_feat), gW1, gW2, gW3, gW4, gW5, g_dirs);
}

template <int K1>
static void launch_bwd128(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, const float* g_sigma,
                          const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3, float* gW4, float* gW5, float* g_dirs,
                          cudaStream_t s) {
    if (g_dirs) launch_bwd128<K1, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, g_dirs, s);
    else launch_bwd128<K1, false>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, nullptr, s);
}

void mlp_tc128_backward(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                        const float* g_sigma, const float* g_rgb, void* g_feat, float* gW1, float* gW2, float* gW3, float* gW4, float* gW5,
                        float* g_dirs, cudaStream_t s) {
    if (in_dim == 48) launch_bwd128<48>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, g_dirs, s);
    else if (in_dim == 96) launch_bwd128<96>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, g_dirs, s);
    else launch_bwd128<144>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, gW1, gW2, gW3, gW4, gW5, g_dirs, s);
}

template <int K1>
static void launch_bwd128_det(const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid, const float* g_sigma,
                              const float* g_rgb, void* g_feat, float* slots, float* g_dirs, cudaStream_t s) {
    const WgradSlot L = wgrad_slot(K1, 128);
    float *w1 = slots, *w2 = slots + L.o2, *w3 = slots + L.o3, *w4 = slots + L.o4, *w5 = slots + L.o5;
    if (g_dirs) launch_bwd128<K1, true, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, g_dirs, s);
    else launch_bwd128<K1, false, true>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, w1, w2, w3, w4, w5, nullptr, s);
}

void mlp_tc128_backward_det(uint32_t in_dim, const void* wpk, const void* feat, const float* dirs, uint32_t M, const int32_t* n_valid,
                            const float* g_sigma, const float* g_rgb, void* g_feat, float* slots, float* g_dirs, cudaStream_t s) {
    if (in_dim == 48) launch_bwd128_det<48>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, slots, g_dirs, s);
    else if (in_dim == 96) launch_bwd128_det<96>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, slots, g_dirs, s);
    else launch_bwd128_det<144>(wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, slots, g_dirs, s);
}

}  // namespace tnl
