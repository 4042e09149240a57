// Sigma / color MLP heads, forward and backward, fused per point tile -- sm_100a.
//
// Behavioural contract: NeRFNetwork.forward / .density
// (/root/reference/reconstruction/nerf/network.py:118-166) under the fp16 autocast the reference trains
// with (--fp16): every nn.Linear runs with fp16 operands, fp32 accumulation and an fp16-rounded output;
// ReLU on the fp16 value; sigma = exp(float(h[0])) (activation.py:5-17); SH degree 4 in fp32
// (shencoder.cu:50-68) rounded to fp16 when it enters color_net[0]; sigmoid in fp32 of the fp16 logits,
// rounded to fp16.  The reference issues ~25 cuBLAS/elementwise kernels that stream every activation
// through HBM; here one kernel keeps all activations of a 16-point tile in the registers of one warp
// (accumulator fragment of layer l == operand fragment of layer l+1) and only reads feat / writes
// sigma, rgb (forward) or reads feat, g_sigma, g_rgb / writes g_feat and the weight gradients (backward).
//
// Tensor-core path: mma.sync.m16n8k16 (f16 x f16 -> f32).  The contraction per point is tiny
// (K <= 144, N <= 128): the kernel is bound by the feature stream from HBM, not by the MMA pipe --
// see DESIGN.md "MLP roofline" and profiles/ for the ncu evidence.  Weights are re-packed once per
// optimizer step into per-lane fragment order (tnl_mlp_pack_weights) so a B operand is one coalesced
// 64-bit load that hits L1.
//
// Internal neuron order (applied by the packer, undone when gradients are written):
//   sigma_net[1] rows: internal j < 15 <-> reference row j+1 (geo_feat j), internal 15 <-> row 0 (sigma)
//   color_net[0] cols: internal k < 16 = SH k, 16..30 = geo_feat 0..14, 31 = zero padding
//   color_net[2] rows: 3 real rows padded with zero rows to 8 (forward) / 16 (backward)
#include "common.cuh"
#include "mlp_math.cuh"
#include "mlp_tc.cuh"
#include <stdlib.h>

namespace tnl {

// ------------------------------------------------------------------------------------------------
// packed-weight layout (units: uint32 = half2), shared by the packer and the kernels
// ------------------------------------------------------------------------------------------------
struct MlpLayout {
    int K1, H, HC;
    // forward fragments of layer l: index ((ks * NT + nt) * 32 + lane) * 2 + r
    int F1, F2, F3, F4, F5;
    // backward (dX) fragments of layer l: index ((ks' * NT' + nt') * 32 + lane) * 2 + r
    int B1, B2, B3, B4, B5;
    int total;
};

__host__ __device__ constexpr MlpLayout make_layout(int K1, int H, int HC) {
    MlpLayout L{};
    L.K1 = K1; L.H = H; L.HC = HC;
    L.F1 = 0;
    L.F2 = L.F1 + (K1 / 16) * (H / 8) * 64;
    L.F3 = L.F2 + (H / 16) * 2 * 64;
    L.F4 = L.F3 + 2 * (HC / 8) * 64;
    L.F5 = L.F4 + (HC / 16) * (HC / 8) * 64;
    L.B5 = L.F5 + (HC / 16) * 1 * 64;
    L.B4 = L.B5 + 1 * (HC / 8) * 64;
    L.B3 = L.B4 + (HC / 16) * (HC / 8) * 64;
    L.B2 = L.B3 + (HC / 16) * 4 * 64;
    L.B1 = L.B2 + 1 * (H / 8) * 64;
    L.total = L.B1 + (H / 16) * (K1 / 8) * 64;
    return L;
}

// internal (permuted / padded) weight element of layer l
__device__ __forceinline__ float w_internal(int layer, int n, int k, const MlpLayout& L, const float* W1, const float* W2,
                                            const float* W3, const float* W4, const float* W5) {
    switch (layer) {
        case 1: return W1[(size_t)n * L.K1 + k];
        case 2: return W2[(size_t)(n < 15 ? n + 1 : 0) * L.H + k];
        case 3: return k < 31 ? W3[(size_t)n * 31 + k] : 0.0f;
        case 4: return W4[(size_t)n * L.HC + k];
        default: return n < 3 ? W5[(size_t)n * L.HC + k] : 0.0f;
    }
}

// one thread per packed uint32
__global__ void k_mlp_pack(MlpLayout L, const float* __restrict__ W1, const float* __restrict__ W2,
                           const float* __restrict__ W3, const float* __restrict__ W4, const float* __restrict__ W5,
                           uint32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= L.total) return;
    // locate section
    int layer, base, NT;
    bool bwd;
    if (i < L.F2) { layer = 1; base = L.F1; NT = L.H / 8; bwd = false; }
    else if (i < L.F3) { layer = 2; base = L.F2; NT = 2; bwd = false; }
    else if (i < L.F4) { layer = 3; base = L.F3; NT = L.HC / 8; bwd = false; }
    else if (i < L.F5) { layer = 4; base = L.F4; NT = L.HC / 8; bwd = false; }
    else if (i < L.B5) { layer = 5; base = L.F5; NT = 1; bwd = false; }
    else if (i < L.B4) { layer = 5; base = L.B5; NT = L.HC / 8; bwd = true; }
    else if (i < L.B3) { layer = 4; base = L.B4; NT = L.HC / 8; bwd = true; }
    else if (i < L.B2) { layer = 3; base = L.B3; NT = 4; bwd = true; }
    else if (i < L.B1) { layer = 2; base = L.B2; NT = L.H / 8; bwd = true; }
    else { layer = 1; base = L.B1; NT = L.K1 / 8; bwd = true; }
    const int j = i - base;
    const int r = j & 1, lane = (j >> 1) & 31, tile = j >> 6;
    const int nt = tile % NT, ks = tile / NT;
    const int g = lane >> 2, t = lane & 3;
    float lo, hi;
    if (!bwd) {  // B[k][n] = W[n][k]:  b = {W[8nt+g][16ks+2t+8r], W[8nt+g][16ks+2t+8r+1]}
        const int n = 8 * nt + g, k = 16 * ks + 2 * t + 8 * r;
        lo = w_internal(layer, n, k, L, W1, W2, W3, W4, W5);
        hi = w_internal(layer, n, k + 1, L, W1, W2, W3, W4, W5);
    } else {     // dX: B[k=n_out][n'=k_in] = W[n_out][k_in]: b = {W[16ks+2t+8r][8nt+g], W[16ks+2t+8r+1][8nt+g]}
        const int n = 16 * ks + 2 * t + 8 * r, k = 8 * nt + g;
        lo = w_internal(layer, n, k, L, W1, W2, W3, W4, W5);
        hi = w_internal(layer, n + 1, k, L, W1, W2, W3, W4, W5);
    }
    out[i] = pack_h2(lo, hi);
}

// ------------------------------------------------------------------------------------------------
// warp-level building blocks
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint2 b) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}

__device__ __forceinline__ uint2 ldfrag(const uint32_t* __restrict__ wp, int off, int tile, int lane) {
    return __ldg(reinterpret_cast<const uint2*>(wp + off) + tile * 32 + lane);
}

// D[16 x 8*NT] (+)= A[16 x 16*KS] * W^T, A as packed fragments a[ks][4], result in acc[nt][4]
template <int KS, int NT>
__device__ __forceinline__ void layer_mma(float (&acc)[NT][4], const uint32_t (&a)[KS][4], const uint32_t* __restrict__ wp,
                                          int off, int lane) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) mma16816(acc[nt], a[ks], ldfrag(wp, off, ks * NT + nt, lane));
}

// accumulator fragments (fp32, 2 n-tiles per k-step) -> fp16-rounded operand fragments, optional ReLU
template <int NT, bool RELU>
__device__ __forceinline__ void acc_to_frag(const float (&acc)[NT][4], uint32_t (&a)[NT / 2][4]) {
#pragma unroll
    for (int ks = 0; ks < NT / 2; ++ks) {
        a[ks][0] = pack_h2(acc[2 * ks][0], acc[2 * ks][1]);
        a[ks][1] = pack_h2(acc[2 * ks][2], acc[2 * ks][3]);
        a[ks][2] = pack_h2(acc[2 * ks + 1][0], acc[2 * ks + 1][1]);
        a[ks][3] = pack_h2(acc[2 * ks + 1][2], acc[2 * ks + 1][3]);
        if (RELU) {
#pragma unroll
            for (int i = 0; i < 4; ++i) a[ks][i] = relu_h2(a[ks][i]);
        }
    }
}

// {o[2t+OFF], o[2t+OFF+1]} as packed fp16 without dynamic register indexing
template <int OFF>
__device__ __forceinline__ uint32_t sel_pair(const float (&o)[16], int t) {
    float lo = o[OFF], hi = o[OFF + 1];
    if (t == 1) { lo = o[OFF + 2]; hi = o[OFF + 3]; }
    if (t == 2) { lo = o[OFF + 4]; hi = o[OFF + 5]; }
    if (t == 3) { lo = o[OFF + 6]; hi = o[OFF + 7]; }
    return pack_h2(lo, hi);
}

// per-warp recomputable forward state for one 16-point tile
template <int K1, int H, int HC>
struct TileFwd {
    uint32_t a1[K1 / 16][4];  // feat (fp16 operand fragments)
    uint32_t a2[H / 16][4];   // relu(h1)
    uint32_t a3[2][4];        // [SH16 | geo15, 0]
    uint32_t a4[HC / 16][4];  // relu(h3)
    uint32_t a5[HC / 16][4];  // relu(h4)
    float logit0, logit1;     // sigma logits (valid in lanes t == 3) for rows g, g+8
    float geo[2][4];          // h2 tiles as floats: [tile][c0..c3] (col 15 = sigma logit in tile 1, t == 3)
    float rgb[4];             // sigmoid outputs of the 8-wide tile: c0,c1 (row g), c2,c3 (row g+8)
};

// fp16 feature rows (produced by k_sample_fwd<true>): the operand fragments are plain 32-bit loads
template <int K1>
__device__ __forceinline__ void load_feat_frags_h(uint32_t (&a1)[K1 / 16][4], const __half* __restrict__ feat, uint32_t r0,
                                                  uint32_t r1, bool v0, bool v1, int t) {
    const uint32_t* p0 = reinterpret_cast<const uint32_t*>(feat + (size_t)r0 * K1) + t;
    const uint32_t* p1 = reinterpret_cast<const uint32_t*>(feat + (size_t)r1 * K1) + t;
#pragma unroll
    for (int ks = 0; ks < K1 / 16; ++ks) {
        a1[ks][0] = v0 ? __ldg(p0 + 8 * ks) : 0u;
        a1[ks][1] = v1 ? __ldg(p1 + 8 * ks) : 0u;
        a1[ks][2] = v0 ? __ldg(p0 + 8 * ks + 4) : 0u;
        a1[ks][3] = v1 ? __ldg(p1 + 8 * ks + 4) : 0u;
    }
}

template <int K1>
__device__ __forceinline__ void load_feat_frags(uint32_t (&a1)[K1 / 16][4], const float* __restrict__ feat, uint32_t r0,
                                                uint32_t r1, bool v0, bool v1, int t) {
    const float2 z = make_float2(0.f, 0.f);
    const float2* p0 = reinterpret_cast<const float2*>(feat + (size_t)r0 * K1) + t;
    const float2* p1 = reinterpret_cast<const float2*>(feat + (size_t)r1 * K1) + t;
#pragma unroll
    for (int ks = 0; ks < K1 / 16; ++ks) {
        const float2 x0 = v0 ? __ldg(p0 + 8 * ks) : z, x2 = v0 ? __ldg(p0 + 8 * ks + 4) : z;
        const float2 x1 = v1 ? __ldg(p1 + 8 * ks) : z, x3 = v1 ? __ldg(p1 + 8 * ks + 4) : z;
        a1[ks][0] = pack_h2(x0.x, x0.y);
        a1[ks][1] = pack_h2(x1.x, x1.y);
        a1[ks][2] = pack_h2(x2.x, x2.y);
        a1[ks][3] = pack_h2(x3.x, x3.y);
    }
}

// forward through all layers for one tile; COLOR=false stops after the sigma head (density())
template <int K1, int H, int HC, bool COLOR>
__device__ __forceinline__ void tile_forward(TileFwd<K1, H, HC>& s, const MlpLayout& L, const uint32_t* __restrict__ wp,
                                             const float* __restrict__ dirs, uint32_t r0, uint32_t r1, bool v0, bool v1,
                                             int lane) {
    const int t = lane & 3;
    {
        float acc[H / 8][4];
        layer_mma<K1 / 16, H / 8>(acc, s.a1, wp, L.F1, lane);
        acc_to_frag<H / 8, true>(acc, s.a2);
    }
    {
        float acc[2][4];
        layer_mma<H / 16, 2>(acc, s.a2, wp, L.F2, lane);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s.geo[i][j] = r16(acc[i][j]);
        s.logit0 = s.geo[1][1];  // column 15 lives in lanes t == 3
        s.logit1 = s.geo[1][3];
    }
    if (!COLOR) return;
    {
        float d0[3] = {0.f, 0.f, 0.f}, d1[3] = {0.f, 0.f, 0.f};
        if (v0) { d0[0] = __ldg(dirs + 3 * (size_t)r0); d0[1] = __ldg(dirs + 3 * (size_t)r0 + 1); d0[2] = __ldg(dirs + 3 * (size_t)r0 + 2); }
        if (v1) { d1[0] = __ldg(dirs + 3 * (size_t)r1); d1[1] = __ldg(dirs + 3 * (size_t)r1 + 1); d1[2] = __ldg(dirs + 3 * (size_t)r1 + 2); }
        float sh0[16], sh1[16];
        sh16(d0[0], d0[1], d0[2], sh0);
        sh16(d1[0], d1[1], d1[2], sh1);
        s.a3[0][0] = sel_pair<0>(sh0, t);
        s.a3[0][1] = sel_pair<0>(sh1, t);
        s.a3[0][2] = sel_pair<8>(sh0, t);
        s.a3[0][3] = sel_pair<8>(sh1, t);
        const bool last = (t == 3);  // column 15 of the h2 tile pair is the sigma logit: not an input of color_net
        s.a3[1][0] = pack_h2(s.geo[0][0], s.geo[0][1]);
        s.a3[1][1] = pack_h2(s.geo[0][2], s.geo[0][3]);
        s.a3[1][2] = pack_h2(s.geo[1][0], last ? 0.f : s.geo[1][1]);
        s.a3[1][3] = pack_h2(s.geo[1][2], last ? 0.f : s.geo[1][3]);
    }
    {
        float acc[HC / 8][4];
        layer_mma<2, HC / 8>(acc, s.a3, wp, L.F3, lane);
        acc_to_frag<HC / 8, true>(acc, s.a4);
    }
    {
        float acc[HC / 8][4];
        layer_mma<HC / 16, HC / 8>(acc, s.a4, wp, L.F4, lane);
        acc_to_frag<HC / 8, true>(acc, s.a5);
    }
    {
        float acc[1][4];
        layer_mma<HC / 16, 1>(acc, s.a5, wp, L.F5, lane);
#pragma unroll
        for (int j = 0; j < 4; ++j) s.rgb[j] = r16(sigmoidf_(r16(acc[0][j])));
    }
}

// ------------------------------------------------------------------------------------------------
// forward kernel: one warp per 16-point tile, grid-stride over tiles
// ------------------------------------------------------------------------------------------------
template <int K1, int H, int HC, bool FH>
__global__ void __launch_bounds__(128)
k_mlp_fwd(const uint32_t* __restrict__ wp, const void* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
          const int32_t* __restrict__ n_valid_ptr, float* __restrict__ sigma, float* __restrict__ rgb,
          float* __restrict__ geo) {
    constexpr MlpLayout L = make_layout(K1, H, HC);
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    uint32_t nvalid = M;
    if (n_valid_ptr) {
        const int32_t nv = *n_valid_ptr;
        nvalid = nv < 0 ? 0u : ((uint32_t)nv < M ? (uint32_t)nv : M);
    }
    const uint32_t ntiles = ceil_div(M, 16u);
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; tile < ntiles; tile += warps) {
        const uint32_t base = tile * 16;
        const uint32_t r0 = base + g, r1 = r0 + 8;
        const bool v0 = r0 < nvalid, v1 = r1 < nvalid;
        if (base >= nvalid) {  // padding rows of the sample buffer: defined zeros, no work
            for (uint32_t r = base + lane; r < base + 16 && r < M; r += 32) {
                sigma[r] = 0.f;
                if (rgb) { rgb[3 * (size_t)r] = 0.f; rgb[3 * (size_t)r + 1] = 0.f; rgb[3 * (size_t)r + 2] = 0.f; }
                if (geo) for (int j = 0; j < 15; ++j) geo[15 * (size_t)r + j] = 0.f;
            }
            continue;
        }
        TileFwd<K1, H, HC> s;
        if (FH) load_feat_frags_h<K1>(s.a1, static_cast<const __half*>(feat), r0, r1, v0, v1, t);
        else load_feat_frags<K1>(s.a1, static_cast<const float*>(feat), r0, r1, v0, v1, t);
        if (dirs) tile_forward<K1, H, HC, true>(s, L, wp, dirs, r0, r1, v0, v1, lane);
        else tile_forward<K1, H, HC, false>(s, L, wp, dirs, r0, r1, v0, v1, lane);
        if (t == 3) {
            if (r0 < M) sigma[r0] = v0 ? expf(s.logit0) : 0.f;
            if (r1 < M) sigma[r1] = v1 ? expf(s.logit1) : 0.f;
        }
        if (geo) {
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int col = 8 * i + 2 * t + j;
                    if (col < 15) {
                        if (r0 < M) geo[15 * (size_t)r0 + col] = v0 ? s.geo[i][j] : 0.f;
                        if (r1 < M) geo[15 * (size_t)r1 + col] = v1 ? s.geo[i][2 + j] : 0.f;
                    }
                }
        }
        if (dirs && rgb) {
            if (t == 0) {
                if (r0 < M) { rgb[3 * (size_t)r0] = v0 ? s.rgb[0] : 0.f; rgb[3 * (size_t)r0 + 1] = v0 ? s.rgb[1] : 0.f; }
                if (r1 < M) { rgb[3 * (size_t)r1] = v1 ? s.rgb[2] : 0.f; rgb[3 * (size_t)r1 + 1] = v1 ? s.rgb[3] : 0.f; }
            } else if (t == 1) {
                if (r0 < M) rgb[3 * (size_t)r0 + 2] = v0 ? s.rgb[0] : 0.f;
                if (r1 < M) rgb[3 * (size_t)r1 + 2] = v1 ? s.rgb[2] : 0.f;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward kernel.  CTA = 8 warps = 128 points per iteration, persistent over tiles.
//   phase 1 (per warp, 16 points): recompute forward, run the dX chain in registers, write g_feat,
//            and leave (input, output-gradient) fp16 tiles of every layer in shared memory;
//   phase 2 (whole CTA): weight gradients dW_l += dOut_l^T * In_l with the point index as the MMA
//            reduction dimension; operands via ldmatrix.trans; each warp owns a fixed slice of every
//            dW and keeps it in fp32 accumulator registers for the whole kernel; one atomicAdd per
//            element per CTA at the end.
// ------------------------------------------------------------------------------------------------
template <int K1, int H, int HC, int NW>
struct BwdSmem {
    static constexpr int PTS = 16 * NW;
    static constexpr int P_F = K1 + 8, P_H = H + 8, P_I = 32 + 8, P_C = HC + 8, P_S = 16 + 8;  // pitches (halves)
    static constexpr int O_F = 0;                      // feat
    static constexpr int O_H1 = O_F + PTS * P_F;       // relu(h1)
    static constexpr int O_I2 = O_H1 + PTS * P_H;      // in2 = [SH | geo]
    static constexpr int O_H3 = O_I2 + PTS * P_I;      // relu(h3)
    static constexpr int O_H4 = O_H3 + PTS * P_C;      // relu(h4)
    static constexpr int O_D1 = O_H4 + PTS * P_C;      // dh1
    static constexpr int O_D2 = O_D1 + PTS * P_H;      // dh2
    static constexpr int O_D3 = O_D2 + PTS * P_S;      // dh3
    static constexpr int O_D4 = O_D3 + PTS * P_C;      // dh4
    static constexpr int O_D5 = O_D4 + PTS * P_C;      // d5 (padded to 16)
    static constexpr int TOTAL = O_D5 + PTS * P_S;     // halves
    static constexpr size_t BYTES = (size_t)TOTAL * 2;
};

// store an operand-fragment set (rows g / g+8 of the warp's 16 points) into a [pt][feature] tile
template <int KS>
__device__ __forceinline__ void store_frags(__half* tile, int pitch, int row0, const uint32_t (&a)[KS][4], int t) {
    uint32_t* p0 = reinterpret_cast<uint32_t*>(tile + (size_t)row0 * pitch) + t;
    uint32_t* p1 = reinterpret_cast<uint32_t*>(tile + (size_t)(row0 + 8) * pitch) + t;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        p0[8 * ks] = a[ks][0];
        p1[8 * ks] = a[ks][1];
        p0[8 * ks + 4] = a[ks][2];
        p1[8 * ks + 4] = a[ks][3];
    }
}

__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const __half* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t (&r)[2], const __half* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n" : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}

// dW block: rows [nb*16, nb*16+16) of dOut^T, k-in tiles [kt0, kt0+NTILES), one 16-point k-step at `pt0`
template <int NTILES>
__device__ __forceinline__ void dw_kstep(float (&acc)[NTILES][4], const __half* dOut, int pd, int nb, const __half* In,
                                         int pi, int kt0, int pt0, int lane) {
    uint32_t a[4];
    {   // A = dOut^T: matrices (pts 0-7,n 0-7), (pts 0-7,n 8-15), (pts 8-15,n 0-7), (pts 8-15,n 8-15)
        const int j = lane >> 3, i = lane & 7;
        ldsm_x4_t(a, dOut + (size_t)(pt0 + (j >> 1) * 8 + i) * pd + nb * 16 + (j & 1) * 8);
    }
#pragma unroll
    for (int q = 0; q + 1 < NTILES; q += 2) {  // two k-in tiles per ldmatrix.x4
        uint32_t b[4];
        const int j = lane >> 3, i = lane & 7;
        ldsm_x4_t(b, In + (size_t)(pt0 + (j & 1) * 8 + i) * pi + (kt0 + q + (j >> 1)) * 8);
        mma16816(acc[q], a, make_uint2(b[0], b[1]));
        mma16816(acc[q + 1], a, make_uint2(b[2], b[3]));
    }
    if (NTILES & 1) {
        uint32_t b[2];
        const int j = (lane >> 3) & 1, i = lane & 7;
        ldsm_x2_t(b, In + (size_t)(pt0 + j * 8 + i) * pi + (kt0 + NTILES - 1) * 8);
        mma16816(acc[NTILES - 1], a, make_uint2(b[0], b[1]));
    }
}

// reload an operand-fragment set written by store_frags (same warp; used for the ReLU masks so that the forward
// activations need not stay in registers across the backward chain)
template <int KS>
__device__ __forceinline__ void load_frags(const __half* tile, int pitch, int row0, uint32_t (&a)[KS][4], int t) {
    const uint32_t* p0 = reinterpret_cast<const uint32_t*>(tile + (size_t)row0 * pitch) + t;
    const uint32_t* p1 = reinterpret_cast<const uint32_t*>(tile + (size_t)(row0 + 8) * pitch) + t;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        a[ks][0] = p0[8 * ks];
        a[ks][1] = p1[8 * ks];
        a[ks][2] = p0[8 * ks + 4];
        a[ks][3] = p1[8 * ks + 4];
    }
}

template <int KS>
__device__ __forceinline__ void relu_mask(uint32_t (&d)[KS][4], const uint32_t (&h)[KS][4]) {
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // h > 0  <=>  fp16 magnitude bits non-zero (ReLU output is never negative)
            const uint32_t v = h[ks][i];
            const uint32_t m = (((v & 0x7fffu) != 0u) ? 0x0000ffffu : 0u) | (((v & 0x7fff0000u) != 0u) ? 0xffff0000u : 0u);
            d[ks][i] &= m;
        }
}

// DIRS: also g_dirs [M,3] <- the SH Jacobian applied to the fp16-rounded SH columns of d(in2) (valid rows only)
// DET: the weight gradients go to slot blockIdx.x of the workspace gW1 .. gW5 point into (wgrad_add)
template <int K1, int H, int HC, int NW, bool FH, bool DIRS, bool DET = false>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? 2 : 1)
k_mlp_bwd(const uint32_t* __restrict__ wp, const void* __restrict__ feat, const float* __restrict__ dirs, uint32_t M,
          const int32_t* __restrict__ n_valid_ptr, const float* __restrict__ g_sigma, const float* __restrict__ g_rgb,
          void* __restrict__ g_feat, float* __restrict__ gW1, float* __restrict__ gW2, float* __restrict__ gW3,
          float* __restrict__ gW4, float* __restrict__ gW5, float* __restrict__ g_dirs) {
    static_assert(H == 64 && HC == 64, "backward kernel: weight-gradient register tiling is laid out for 64-wide heads");
    static_assert(NW == 4 || NW == 8, "4 or 8 warps");
    constexpr MlpLayout L = make_layout(K1, H, HC);
    using SM = BwdSmem<K1, H, HC, NW>;
    constexpr int SPLIT = NW / 4;            // warps sharing one 16-row block of a weight gradient
    constexpr int T1 = (K1 / 8) / SPLIT;     // k-in tiles of dW1 per warp
    constexpr int T4 = 8 / SPLIT, T3 = 4 / SPLIT, T25 = 8 / NW;
    extern __shared__ __align__(16) __half sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    uint32_t nvalid = M;
    if (n_valid_ptr) {
        const int32_t nv = *n_valid_ptr;
        nvalid = nv < 0 ? 0u : ((uint32_t)nv < M ? (uint32_t)nv : M);
    }
    // persistent weight-gradient accumulators: warp w owns
    //   dW1: rows [16*(w/2), +16), k-in tiles [(w%2)*K1/16, +K1/16)      dW4: rows [16*(w/2), +16), tiles [(w%2)*4, +4)
    //   dW3: rows [16*(w/2), +16), tiles [(w%2)*2, +2)                   dW2, dW5: the single 16-row block, tile w
    float acc1[T1][4], acc4[T4][4], acc3[T3][4], acc2[T25][4], acc5[T25][4];
#pragma unroll
    for (int i = 0; i < T1; ++i) acc1[i][0] = acc1[i][1] = acc1[i][2] = acc1[i][3] = 0.f;
#pragma unroll
    for (int i = 0; i < T4; ++i) acc4[i][0] = acc4[i][1] = acc4[i][2] = acc4[i][3] = 0.f;
#pragma unroll
    for (int i = 0; i < T3; ++i) acc3[i][0] = acc3[i][1] = acc3[i][2] = acc3[i][3] = 0.f;
#pragma unroll
    for (int i = 0; i < T25; ++i) {
        acc2[i][0] = acc2[i][1] = acc2[i][2] = acc2[i][3] = 0.f;
        acc5[i][0] = acc5[i][1] = acc5[i][2] = acc5[i][3] = 0.f;
    }

    const uint32_t ntiles = ceil_div(nvalid, (uint32_t)SM::PTS);
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // ------------------------------ phase 1 ------------------------------
        const int row0 = warp * 16 + g;  // row inside the 128-point tile
        const uint32_t r0 = tile * SM::PTS + row0, r1 = r0 + 8;
        const bool v0 = r0 < nvalid, v1 = r1 < nvalid;
        TileFwd<K1, H, HC> s;
        if (FH) load_feat_frags_h<K1>(s.a1, static_cast<const __half*>(feat), r0, r1, v0, v1, t);
        else load_feat_frags<K1>(s.a1, static_cast<const float*>(feat), r0, r1, v0, v1, t);
        store_frags<K1 / 16>(sm + SM::O_F, SM::P_F, row0, s.a1, t);
        tile_forward<K1, H, HC, true>(s, L, wp, dirs, r0, r1, v0, v1, lane);
        store_frags<H / 16>(sm + SM::O_H1, SM::P_H, row0, s.a2, t);
        store_frags<2>(sm + SM::O_I2, SM::P_I, row0, s.a3, t);
        store_frags<HC / 16>(sm + SM::O_H3, SM::P_C, row0, s.a4, t);
        store_frags<HC / 16>(sm + SM::O_H4, SM::P_C, row0, s.a5, t);
        __syncwarp();

        // d5 = half(g_rgb) * s * (1 - s), fp16 (sigmoid backward under autocast); columns 3..15 are zero
        uint32_t d5[1][4];
        {
            float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f;
            if (t == 0) {
                if (v0) { e0 = r16(__ldg(g_rgb + 3 * (size_t)r0)); e1 = r16(__ldg(g_rgb + 3 * (size_t)r0 + 1)); }
                if (v1) { e2 = r16(__ldg(g_rgb + 3 * (size_t)r1)); e3 = r16(__ldg(g_rgb + 3 * (size_t)r1 + 1)); }
            } else if (t == 1) {
                if (v0) e0 = r16(__ldg(g_rgb + 3 * (size_t)r0 + 2));
                if (v1) e2 = r16(__ldg(g_rgb + 3 * (size_t)r1 + 2));
            }
            d5[0][0] = pack_h2(e0 * s.rgb[0] * (1.f - s.rgb[0]), e1 * s.rgb[1] * (1.f - s.rgb[1]));
            d5[0][1] = pack_h2(e2 * s.rgb[2] * (1.f - s.rgb[2]), e3 * s.rgb[3] * (1.f - s.rgb[3]));
            if (t >= 2) { d5[0][0] = 0u; d5[0][1] = 0u; }
            if (t == 1) { d5[0][0] &= 0x0000ffffu; d5[0][1] &= 0x0000ffffu; }  // column 3 is padding
            d5[0][2] = 0u;
            d5[0][3] = 0u;
        }
        store_frags<1>(sm + SM::O_D5, SM::P_S, row0, d5, t);

        // dh4 = (d5 W5) * [h4 > 0]
        uint32_t d4[HC / 16][4];
        {
            float acc[HC / 8][4];
            layer_mma<1, HC / 8>(acc, d5, wp, L.B5, lane);
            acc_to_frag<HC / 8, false>(acc, d4);
            {
                uint32_t hm[HC / 16][4];
                load_frags<HC / 16>(sm + SM::O_H4, SM::P_C, row0, hm, t);
                relu_mask<HC / 16>(d4, hm);
            }
        }
        store_frags<HC / 16>(sm + SM::O_D4, SM::P_C, row0, d4, t);
        // dh3 = (dh4 W4) * [h3 > 0]
        uint32_t d3[HC / 16][4];
        {
            float acc[HC / 8][4];
            layer_mma<HC / 16, HC / 8>(acc, d4, wp, L.B4, lane);
            acc_to_frag<HC / 8, false>(acc, d3);
            {
                uint32_t hm[HC / 16][4];
                load_frags<HC / 16>(sm + SM::O_H3, SM::P_C, row0, hm, t);
                relu_mask<HC / 16>(d3, hm);
            }
        }
        store_frags<HC / 16>(sm + SM::O_D3, SM::P_C, row0, d3, t);
        // d(in2) = dh3 W3 ; the geo half (internal columns 16..31) feeds dh2, the SH half (columns 0..15) only g_dirs
        uint32_t d2[1][4];
        {
            float acc[4][4];
            layer_mma<HC / 16, 4>(acc, d3, wp, L.B3, lane);
            if constexpr (DIRS) {
                // gather the point's 16 SH columns from the four lanes of its quad (row g: elements 0, 1; row g + 8: 2, 3),
                // rounded to fp16 as the autocast linear backward returns them; lane t = 0 finishes row r0, t = 1 row r1
                float sh0[16], sh1[16];
#pragma unroll
                for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                    for (int tt = 0; tt < 4; ++tt) {
                        const int src = (lane & ~3) | tt;
                        sh0[nt * 8 + 2 * tt] = r16(__shfl_sync(0xffffffffu, acc[nt][0], src));
                        sh0[nt * 8 + 2 * tt + 1] = r16(__shfl_sync(0xffffffffu, acc[nt][1], src));
                        sh1[nt * 8 + 2 * tt] = r16(__shfl_sync(0xffffffffu, acc[nt][2], src));
                        sh1[nt * 8 + 2 * tt + 1] = r16(__shfl_sync(0xffffffffu, acc[nt][3], src));
                    }
                const uint32_t r = t == 0 ? r0 : r1;
                if (t < 2 && (t == 0 ? v0 : v1)) {
                    float gd[3];
                    sh_backward<16>(__ldg(dirs + 3 * (size_t)r), __ldg(dirs + 3 * (size_t)r + 1), __ldg(dirs + 3 * (size_t)r + 2),
                                    t == 0 ? sh0 : sh1, gd);
#pragma unroll
                    for (int a = 0; a < 3; ++a) g_dirs[3 * (size_t)r + a] = gd[a];
                }
            }
            // dh2 tiles 0,1 <- d(in2) tiles 2,3 ; column 15 <- g_sigma * exp(clamp(logit, -15, 15)) (trunc_exp backward)
            float c1 = acc[3][1], c3 = acc[3][3];
            if (t == 3) {
                const float gs0 = v0 ? __ldg(g_sigma + r0) : 0.f, gs1 = v1 ? __ldg(g_sigma + r1) : 0.f;
                c1 = gs0 * expf(fminf(fmaxf(s.logit0, -15.f), 15.f));
                c3 = gs1 * expf(fminf(fmaxf(s.logit1, -15.f), 15.f));
            }
            d2[0][0] = pack_h2(acc[2][0], acc[2][1]);
            d2[0][1] = pack_h2(acc[2][2], acc[2][3]);
            d2[0][2] = pack_h2(acc[3][0], c1);
            d2[0][3] = pack_h2(acc[3][2], c3);
        }
        store_frags<1>(sm + SM::O_D2, SM::P_S, row0, d2, t);
        // dh1 = (dh2 W2) * [h1 > 0]
        uint32_t d1[H / 16][4];
        {
            float acc[H / 8][4];
            layer_mma<1, H / 8>(acc, d2, wp, L.B2, lane);
            acc_to_frag<H / 8, false>(acc, d1);
            {
                uint32_t hm[H / 16][4];
                load_frags<H / 16>(sm + SM::O_H1, SM::P_H, row0, hm, t);
                relu_mask<H / 16>(d1, hm);
            }
        }
        store_frags<H / 16>(sm + SM::O_D1, SM::P_H, row0, d1, t);
        // g_feat = dh1 W1 (fp16-rounded, as the autocast linear backward returns it)
        if (g_feat) {
            float acc[K1 / 8][4];
            layer_mma<H / 16, K1 / 8>(acc, d1, wp, L.B1, lane);
            if (FH) {
                uint32_t* q0 = reinterpret_cast<uint32_t*>(static_cast<__half*>(g_feat) + (size_t)r0 * K1) + t;
                uint32_t* q1 = reinterpret_cast<uint32_t*>(static_cast<__half*>(g_feat) + (size_t)r1 * K1) + t;
#pragma unroll
                for (int nt = 0; nt < K1 / 8; ++nt) {
                    if (r0 < M) q0[4 * nt] = v0 ? pack_h2(acc[nt][0], acc[nt][1]) : 0u;
                    if (r1 < M) q1[4 * nt] = v1 ? pack_h2(acc[nt][2], acc[nt][3]) : 0u;
                }
            } else {
                float2* q0 = reinterpret_cast<float2*>(static_cast<float*>(g_feat) + (size_t)r0 * K1) + t;
                float2* q1 = reinterpret_cast<float2*>(static_cast<float*>(g_feat) + (size_t)r1 * K1) + t;
#pragma unroll
                for (int nt = 0; nt < K1 / 8; ++nt) {
                    if (r0 < M) q0[4 * nt] = v0 ? make_float2(r16(acc[nt][0]), r16(acc[nt][1])) : make_float2(0.f, 0.f);
                    if (r1 < M) q1[4 * nt] = v1 ? make_float2(r16(acc[nt][2]), r16(acc[nt][3])) : make_float2(0.f, 0.f);
                }
            }
        }
        __syncthreads();
        // ------------------------------ phase 2 ------------------------------
        {
            const int nb = warp / SPLIT, hf = warp % SPLIT;
#pragma unroll 1
            for (int pt0 = 0; pt0 < SM::PTS; pt0 += 16) {
                dw_kstep<T1>(acc1, sm + SM::O_D1, SM::P_H, nb, sm + SM::O_F, SM::P_F, hf * T1, pt0, lane);
                dw_kstep<T4>(acc4, sm + SM::O_D4, SM::P_C, nb, sm + SM::O_H3, SM::P_C, hf * T4, pt0, lane);
                dw_kstep<T3>(acc3, sm + SM::O_D3, SM::P_C, nb, sm + SM::O_I2, SM::P_I, hf * T3, pt0, lane);
                dw_kstep<T25>(acc2, sm + SM::O_D2, SM::P_S, 0, sm + SM::O_H1, SM::P_H, warp * T25, pt0, lane);
                dw_kstep<T25>(acc5, sm + SM::O_D5, SM::P_S, 0, sm + SM::O_H4, SM::P_C, warp * T25, pt0, lane);
            }
        }
        __syncthreads();
    }
    // ------------------------------ flush weight gradients ------------------------------
    {
        if constexpr (DET) {   // this CTA's slot of the workspace
            const size_t o = (size_t)blockIdx.x * wgrad_slot(K1, H).size;
            gW1 += o; gW2 += o; gW3 += o; gW4 += o; gW5 += o;
        }
        const int nb = warp / SPLIT, hf = warp % SPLIT;
        const int n0 = nb * 16 + g, n1 = n0 + 8;
#pragma unroll
        for (int q = 0; q < T1; ++q) {
            const int k = (hf * T1 + q) * 8 + 2 * t;
            wgrad_add<DET>(gW1 + (size_t)n0 * K1 + k, acc1[q][0]);
            wgrad_add<DET>(gW1 + (size_t)n0 * K1 + k + 1, acc1[q][1]);
            wgrad_add<DET>(gW1 + (size_t)n1 * K1 + k, acc1[q][2]);
            wgrad_add<DET>(gW1 + (size_t)n1 * K1 + k + 1, acc1[q][3]);
        }
#pragma unroll
        for (int q = 0; q < T4; ++q) {
            const int k = (hf * T4 + q) * 8 + 2 * t;
            wgrad_add<DET>(gW4 + (size_t)n0 * HC + k, acc4[q][0]);
            wgrad_add<DET>(gW4 + (size_t)n0 * HC + k + 1, acc4[q][1]);
            wgrad_add<DET>(gW4 + (size_t)n1 * HC + k, acc4[q][2]);
            wgrad_add<DET>(gW4 + (size_t)n1 * HC + k + 1, acc4[q][3]);
        }
#pragma unroll
        for (int q = 0; q < T3; ++q) {
            const int k = (hf * T3 + q) * 8 + 2 * t;  // internal color_net[0] column: 0..15 SH, 16..30 geo, 31 padding
            if (k < 31) { wgrad_add<DET>(gW3 + (size_t)n0 * 31 + k, acc3[q][0]); wgrad_add<DET>(gW3 + (size_t)n1 * 31 + k, acc3[q][2]); }
            if (k + 1 < 31) { wgrad_add<DET>(gW3 + (size_t)n0 * 31 + k + 1, acc3[q][1]); wgrad_add<DET>(gW3 + (size_t)n1 * 31 + k + 1, acc3[q][3]); }
        }
#pragma unroll
        for (int q = 0; q < T25; ++q) {
            const int k = (warp * T25 + q) * 8 + 2 * t;
            {   // sigma_net[1]: internal row j < 15 -> reference row j+1, internal 15 -> row 0
                const int ra = g + 1;                    // internal row g  (< 8)
                const int rb = (g + 8 < 15) ? g + 9 : 0; // internal row g+8
                wgrad_add<DET>(gW2 + (size_t)ra * H + k, acc2[q][0]);
                wgrad_add<DET>(gW2 + (size_t)ra * H + k + 1, acc2[q][1]);
                wgrad_add<DET>(gW2 + (size_t)rb * H + k, acc2[q][2]);
                wgrad_add<DET>(gW2 + (size_t)rb * H + k + 1, acc2[q][3]);
            }
            if (g < 3) {  // color_net[2]: rows 0..2 real
                wgrad_add<DET>(gW5 + (size_t)g * HC + k, acc5[q][0]);
                wgrad_add<DET>(gW5 + (size_t)g * HC + k + 1, acc5[q][1]);
            }
        }
    }
}

// g_W += the sum of the per-CTA slots of a DET backward kernel, in slot order (wgrad_slot layout)
__global__ void __launch_bounds__(256)
k_wgrad_reduce(const float* __restrict__ slots, uint32_t nslots, WgradSlot L, float* __restrict__ gW1, float* __restrict__ gW2,
               float* __restrict__ gW3, float* __restrict__ gW4, float* __restrict__ gW5) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < L.size; i += (size_t)gridDim.x * blockDim.x) {
        float acc = 0.f;
        for (uint32_t b = 0; b < nslots; ++b) acc += slots[(size_t)b * L.size + i];
        float* dst = i < L.o2 ? gW1 + i : i < L.o3 ? gW2 + (i - L.o2) : i < L.o4 ? gW3 + (i - L.o3) : i < L.o5 ? gW4 + (i - L.o4) : gW5 + (i - L.o5);
        *dst += acc;
    }
}

}  // namespace tnl

using namespace tnl;

static bool dims_supported(const tnl_mlp_dims* d) {
    if (!d) return false;
    const bool k_ok = d->in_dim == 48 || d->in_dim == 96 || d->in_dim == 144;
    const bool h_ok = (d->hidden == 64 && d->hidden_c == 64) || (d->hidden == 128 && d->hidden_c == 128);
    return k_ok && h_ok;
}

// the packed block holds the mma.sync fragment layout followed (16-byte aligned) by the tcgen05 tile layout
static size_t legacy_packed_bytes(const tnl_mlp_dims* d) {
    const size_t b = sizeof(uint32_t) * (size_t)make_layout((int)d->in_dim, (int)d->hidden, (int)d->hidden_c).total;
    return (b + 255) & ~(size_t)255;
}
// tcgen05 path: fp16 feature stream (TNL_MLP_LEGACY=1 forces the mma.sync kernels)
static bool use_tc(const tnl_mlp_dims* d, int feat_fp16) {
    static const bool legacy = getenv("TNL_MLP_LEGACY") != nullptr;
    return !legacy && feat_fp16 && mlp_tc_supported(d->in_dim, d->hidden, d->hidden_c);
}

namespace tnl {
size_t mlp_tc_packed_offset(const tnl_mlp_dims* d) { return legacy_packed_bytes(d); }
bool mlp_tc_selected(const tnl_mlp_dims* d) { return dims_supported(d) && use_tc(d, 1); }
}  // namespace tnl

#define TNL_MLP_DISPATCH(DIMS, CALL)                                                        \
    do {                                                                                    \
        const uint32_t k_ = (DIMS)->in_dim, h_ = (DIMS)->hidden;                            \
        if (k_ == 48 && h_ == 64) { CALL(48, 64, 64); }                                     \
        else if (k_ == 96 && h_ == 64) { CALL(96, 64, 64); }                                \
        else if (k_ == 144 && h_ == 64) { CALL(144, 64, 64); }                              \
        else if (k_ == 48 && h_ == 128) { CALL(48, 128, 128); }                             \
        else if (k_ == 96 && h_ == 128) { CALL(96, 128, 128); }                             \
        else { CALL(144, 128, 128); }                                                       \
    } while (0)

extern "C" {

size_t tnl_mlp_packed_bytes(const tnl_mlp_dims* dims) {
    if (!dims_supported(dims)) return 0;
    return legacy_packed_bytes(dims) + (mlp_tc_supported(dims->in_dim, dims->hidden, dims->hidden_c) ? mlp_tc_packed_bytes(dims->in_dim, dims->hidden) : 0);
}

int tnl_mlp_pack_weights(const tnl_mlp_dims* dims, const float* W1, const float* W2, const float* W3, const float* W4,
                         const float* W5, void* packed, tnl_stream_t stream) {
    if (!dims_supported(dims)) {
        set_error("mlp: supported dims are in_dim in {48,96,144} (C = 16/32/48) and hidden = hidden_color in {64,128}");
        return TNL_ERR_UNSUPPORTED;
    }
    TNL_ARG_CHECK(W1 && W2 && W3 && W4 && W5 && packed, "null pointer");
    const MlpLayout L = make_layout((int)dims->in_dim, (int)dims->hidden, (int)dims->hidden_c);
    k_mlp_pack<<<ceil_div(L.total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        L, W1, W2, W3, W4, W5, static_cast<uint32_t*>(packed));
    if (mlp_tc_supported(dims->in_dim, dims->hidden, dims->hidden_c))
        mlp_tc_pack(dims->in_dim, dims->hidden, W1, W2, W3, W4, W5, static_cast<uint8_t*>(packed) + legacy_packed_bytes(dims),
                    reinterpret_cast<cudaStream_t>(stream));
    return finish_launch("mlp_pack_weights");
}

int tnl_mlp_forward(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                    uint32_t M, const int32_t* n_valid, float* sigma, float* rgb, float* geo, tnl_stream_t stream) {
    if (M == 0) return 0;
    if (!dims_supported(dims)) {
        set_error("mlp: unsupported dims");
        return TNL_ERR_UNSUPPORTED;
    }
    TNL_ARG_CHECK(packed && feat && sigma, "null pointer");
    TNL_ARG_CHECK(dirs == nullptr || rgb != nullptr, "rgb output required when dirs are given");
    TNL_ARG_CHECK(((uintptr_t)feat & 7) == 0, "feat must be 8-byte aligned");
    const uint32_t ntiles = ceil_div(M, 16u);
    const uint32_t blocks = min(ceil_div(ntiles, 4u), (uint32_t)(kNumSM * 16));
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (use_tc(dims, feat_fp16)) {
        TNL_ARG_CHECK(((uintptr_t)feat & 15) == 0, "feat must be 16-byte aligned");
        mlp_tc_forward(dims->in_dim, dims->hidden, static_cast<const uint8_t*>(packed) + legacy_packed_bytes(dims), feat, dirs, M, n_valid, sigma,
                       rgb, geo, s);
        return finish_launch("mlp_forward(tcgen05)");
    }
#define CALL(K, HH, HCC)                                                                                                  \
    do {                                                                                                                 \
        if (feat_fp16) k_mlp_fwd<K, HH, HCC, true><<<blocks, 128, 0, s>>>(static_cast<const uint32_t*>(packed), feat, dirs, M, n_valid, sigma, rgb, geo); \
        else k_mlp_fwd<K, HH, HCC, false><<<blocks, 128, 0, s>>>(static_cast<const uint32_t*>(packed), feat, dirs, M, n_valid, sigma, rgb, geo); \
    } while (0)
    TNL_MLP_DISPATCH(dims, CALL);
#undef CALL
    return finish_launch("mlp_forward");
}

}  // extern "C"

// CTAs of the mma.sync backward kernel: two independent 4-warp CTAs per SM -- while one is in its latency-bound recompute / dX
// phase the other runs the shared-memory-bound weight-gradient phase (TNL_MLP_BWD_NW=8 selects the single 8-warp CTA variant)
static int mlp_bwd_warps() {
    static const int nw = getenv("TNL_MLP_BWD_NW") ? atoi(getenv("TNL_MLP_BWD_NW")) : 4;
    return nw == 8 ? 8 : 4;
}
static uint32_t mlp_bwd_blocks(uint32_t M, int nw) {
    return min(ceil_div(M, (uint32_t)(16 * nw)), (uint32_t)(kNumSM * (nw == 4 ? 2 : 1)));
}
// slots of the deterministic weight-gradient reduction: one per CTA of the kernel mlp_backward launches for these arguments
static uint32_t mlp_det_slots(const tnl_mlp_dims* d, int feat_fp16, uint32_t M) {
#ifdef __CUDACC__
    if (use_tc(d, feat_fp16)) return mlp_tc_backward_blocks(d->hidden, M);
#endif
    return mlp_bwd_blocks(M, mlp_bwd_warps());
}

// tnl_mlp_backward (g_dirs == nullptr), tnl_mlp_backward_dirs, and with det_slots != nullptr tnl_mlp_backward_det
static int mlp_backward(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs, uint32_t M,
                        const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* g_W1, float* g_W2,
                        float* g_W3, float* g_W4, float* g_W5, float* g_dirs, float* det_slots, tnl_stream_t stream) {
    if (M == 0) return 0;
    if (!dims_supported(dims) || (dims->hidden != 64 && !use_tc(dims, feat_fp16))) {
        set_error("mlp_backward: the 128-wide heads take the fp16 feature stream (tcgen05 kernels); fp32 features: hidden = hidden_color = 64 only");
        return TNL_ERR_UNSUPPORTED;
    }
    TNL_ARG_CHECK(packed && feat && dirs && g_sigma && g_rgb && g_W1 && g_W2 && g_W3 && g_W4 && g_W5, "null pointer");
    TNL_ARG_CHECK(((uintptr_t)feat & 7) == 0 && ((uintptr_t)g_feat & 7) == 0, "feat/g_feat must be 8-byte aligned");
    const bool fh = feat_fp16 != 0;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (use_tc(dims, feat_fp16)) {
        TNL_ARG_CHECK(((uintptr_t)feat & 15) == 0 && ((uintptr_t)g_feat & 15) == 0, "feat/g_feat must be 16-byte aligned");
        const uint8_t* wpk = static_cast<const uint8_t*>(packed) + legacy_packed_bytes(dims);
#ifdef __CUDACC__
        if (det_slots) {
            mlp_tc_backward_det(dims->in_dim, dims->hidden, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, det_slots, g_dirs, s);
            return finish_launch("mlp_backward_det(tcgen05)");
        }
#endif
        if (!g_dirs) {
            mlp_tc_backward(dims->in_dim, dims->hidden, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, g_W1, g_W2, g_W3, g_W4, g_W5, s);
            return finish_launch("mlp_backward(tcgen05)");
        }
#ifdef __CUDACC__   // (host builds of this file have no tcgen05 implementation: use_tc() is false there)
        mlp_tc_backward_dirs(dims->in_dim, dims->hidden, wpk, feat, dirs, M, n_valid, g_sigma, g_rgb, g_feat, g_W1, g_W2, g_W3, g_W4, g_W5,
                             g_dirs, s);
#endif
        return finish_launch("mlp_backward_dirs(tcgen05)");
    }
    const int nw = mlp_bwd_warps();
    const uint32_t blocks = mlp_bwd_blocks(M, nw);
#define CALLB_DD(K, NW, FHV, DV, DETV, W1, W2, W3, W4, W5)                                                               \
    do {                                                                                                                \
        using SMB = BwdSmem<K, 64, 64, NW>;                                                                             \
        static bool attr = false;                                                                                       \
        if (!attr) {                                                                                                    \
            cudaFuncSetAttribute(k_mlp_bwd<K, 64, 64, NW, FHV, DV, DETV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMB::BYTES); \
            attr = true;                                                                                                \
        }                                                                                                               \
        k_mlp_bwd<K, 64, 64, NW, FHV, DV, DETV><<<blocks, NW * 32, SMB::BYTES, s>>>(static_cast<const uint32_t*>(packed), feat, dirs, \
                                                                                M, n_valid, g_sigma, g_rgb, g_feat, W1, W2, W3, W4, W5, \
                                                                                g_dirs);                                 \
    } while (0)
#define CALLB_D(K, NW, FHV, DV)                                                                                          \
    do {                                                                                                                \
        if (det_slots) {                                                                                                \
            const WgradSlot L = wgrad_slot(K, 64);                                                                      \
            CALLB_DD(K, NW, FHV, DV, true, det_slots, det_slots + L.o2, det_slots + L.o3, det_slots + L.o4, det_slots + L.o5); \
        } else {                                                                                                        \
            CALLB_DD(K, NW, FHV, DV, false, g_W1, g_W2, g_W3, g_W4, g_W5);                                              \
        }                                                                                                               \
    } while (0)
#define CALLB_FH(K, NW, FHV)                        \
    do {                                            \
        if (g_dirs) CALLB_D(K, NW, FHV, true);      \
        else CALLB_D(K, NW, FHV, false);            \
    } while (0)
#define CALLB_NW(K, NW)                  \
    do {                                 \
        if (fh) CALLB_FH(K, NW, true);   \
        else CALLB_FH(K, NW, false);     \
    } while (0)
#define CALLB(K)                  \
    do {                          \
        if (nw == 8) CALLB_NW(K, 8); \
        else CALLB_NW(K, 4);      \
    } while (0)
    if (dims->in_dim == 48) CALLB(48);
    else if (dims->in_dim == 96) CALLB(96);
    else CALLB(144);
#undef CALLB
#undef CALLB_NW
#undef CALLB_FH
#undef CALLB_D
#undef CALLB_DD
    return finish_launch(g_dirs ? "mlp_backward_dirs" : "mlp_backward");
}

extern "C" {

int tnl_mlp_backward(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                     uint32_t M, const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* g_W1,
                     float* g_W2, float* g_W3, float* g_W4, float* g_W5, tnl_stream_t stream) {
    return mlp_backward(dims, packed, feat, feat_fp16, dirs, M, n_valid, g_sigma, g_rgb, g_feat, g_W1, g_W2, g_W3, g_W4, g_W5, nullptr,
                        nullptr, stream);
}

int tnl_mlp_backward_dirs(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                          uint32_t M, const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* g_W1,
                          float* g_W2, float* g_W3, float* g_W4, float* g_W5, float* g_dirs, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_dirs, "null pointer");
    // rows the kernels do not visit (>= *n_valid) keep these zeros
    cudaMemsetAsync(g_dirs, 0, (size_t)M * 3 * sizeof(float), reinterpret_cast<cudaStream_t>(stream));   // (errors: finish_launch)
    return mlp_backward(dims, packed, feat, feat_fp16, dirs, M, n_valid, g_sigma, g_rgb, g_feat, g_W1, g_W2, g_W3, g_W4, g_W5, g_dirs,
                        nullptr, stream);
}

size_t tnl_mlp_backward_det_workspace(const tnl_mlp_dims* dims, int feat_fp16, uint32_t M) {
    if (!dims_supported(dims) || M == 0) return 0;
    return (size_t)mlp_det_slots(dims, feat_fp16, M) * wgrad_slot(dims->in_dim, dims->hidden).size * sizeof(float);
}

int tnl_mlp_backward_det(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs, uint32_t M,
                         const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat, float* g_W1, float* g_W2,
                         float* g_W3, float* g_W4, float* g_W5, float* g_dirs, void* workspace, size_t workspace_bytes,
                         tnl_stream_t stream) {
    if (M == 0) return 0;
    const size_t need = tnl_mlp_backward_det_workspace(dims, feat_fp16, M);
    TNL_ARG_CHECK(workspace != nullptr && need > 0 && workspace_bytes >= need && ((uintptr_t)workspace & 15) == 0,
                  "workspace: tnl_mlp_backward_det_workspace bytes, 16-byte aligned (supported dims)");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (g_dirs) cudaMemsetAsync(g_dirs, 0, (size_t)M * 3 * sizeof(float), s);   // rows the kernels do not visit (>= *n_valid)
    cudaMemsetAsync(workspace, 0, need, s);   // slots of CTAs without a tile stay zero
    float* slots = static_cast<float*>(workspace);
    const int rc = mlp_backward(dims, packed, feat, feat_fp16, dirs, M, n_valid, g_sigma, g_rgb, g_feat, g_W1, g_W2, g_W3, g_W4, g_W5,
                                g_dirs, slots, stream);
    if (rc != 0) return rc;
    const WgradSlot L = wgrad_slot(dims->in_dim, dims->hidden);
    k_wgrad_reduce<<<(unsigned)min(ceil_div(L.size, (size_t)256), (size_t)kNumSM * 4), 256, 0, s>>>(
        slots, mlp_det_slots(dims, feat_fp16, M), L, g_W1, g_W2, g_W3, g_W4, g_W5);
    return finish_launch("mlp_backward_det");
}


}  // extern "C"
