// Tri-plane bilinear sampling (gather) and its adjoint (scatter) -- sm_100a, channels-last planes.
//
// Behavioural contract: TriPlaneVolume.forward -> sample_from_planes_aux
// (/root/reference/reconstruction/triplaneencoder/triplane_encoder.py:314-332, 523-530):
//   u = coords / bound ; plane 0 samples (u_x,u_z), plane 1 (u_x,u_y), plane 2 (u_y,u_z) (:250-289);
//   F.grid_sample(bilinear, padding_mode='border', align_corners=True); concat -> feat[m][p*C + c].
// Arithmetic follows ATen's grid_sampler_2d (unnormalise ((g+1)/2)*(R-1), clip to [0,R-1], weights
// nw/ne/sw/se as products of differences, accumulate in that order, out-of-range corners skipped).
//
// Why channels-last: with planes [3][R][R][C] a texel's C features are one contiguous 4*C-byte run, so
// a bilinear tap is 2 x (two adjacent texels) = two contiguous 8*C-byte reads; every 32-byte sector
// fetched is fully used.  The reference's NCHW layout fetches 2 sectors per (plane, channel) for 16
// useful bytes (SURVEY.md 8a-2).
//
// Mapping: one thread per (point, plane, 4-channel group): four 128-bit loads (one per corner),
// lerp in registers, one 128-bit store into the contiguous feature row.  Backward: one 128-bit
// load of the feature gradient and four vector atomic adds (red.global.add.v4.f32).
#include "common.cuh"
#include "sample_coords.cuh"

namespace tnl {

// HALF: features are written as fp16 -- the rounding the first nn.Linear applies under autocast anyway (network.py:127),
// moved into the producer so that the feature stream costs half the bytes.
template <bool HALF>
__global__ void __launch_bounds__(256)
k_sample_fwd(const float* __restrict__ planes, const float* __restrict__ xyz, uint32_t M, int R, int C, float inv_bound,
             int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
             void* __restrict__ feat_) {
    const int cq_per = C >> 2;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t total = (uint64_t)M * 3 * cq_per;
    if (idx >= total) return;
    const int cq = (int)(idx % cq_per);
    const int p = (int)((idx / cq_per) % 3);
    uint32_t m = (uint32_t)(idx / ((uint64_t)3 * cq_per));
    if (perm) m = (uint32_t)__ldg(perm + m);
    const size_t q4 = ((size_t)m * 3 * C + (size_t)p * C) / 4 + cq;   // index of this thread's 4-channel group
    if (n_valid && (int32_t)m >= *n_valid) {
        if (HALF) reinterpret_cast<uint2*>(feat_)[q4] = make_uint2(0u, 0u);
        else reinterpret_cast<float4*>(feat_)[q4] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    const float4* base = reinterpret_cast<const float4*>(planes + (((size_t)p * R + t.y0) * R + t.x0) * C) + cq;
    const size_t dx = (size_t)cq_per, dy = (size_t)R * cq_per;
    float4 acc;
    {
        const float4 v = __ldg(base);
        acc.x = v.x * t.nw; acc.y = v.y * t.nw; acc.z = v.z * t.nw; acc.w = v.w * t.nw;
    }
    if (t.x1ok) {
        const float4 v = __ldg(base + dx);
        acc.x = fmaf(v.x, t.ne, acc.x); acc.y = fmaf(v.y, t.ne, acc.y); acc.z = fmaf(v.z, t.ne, acc.z); acc.w = fmaf(v.w, t.ne, acc.w);
    }
    if (t.y1ok) {
        const float4 v = __ldg(base + dy);
        acc.x = fmaf(v.x, t.sw, acc.x); acc.y = fmaf(v.y, t.sw, acc.y); acc.z = fmaf(v.z, t.sw, acc.z); acc.w = fmaf(v.w, t.sw, acc.w);
    }
    if (t.x1ok && t.y1ok) {
        const float4 v = __ldg(base + dy + dx);
        acc.x = fmaf(v.x, t.se, acc.x); acc.y = fmaf(v.y, t.se, acc.y); acc.z = fmaf(v.z, t.se, acc.z); acc.w = fmaf(v.w, t.se, acc.w);
    }
    if (HALF) reinterpret_cast<uint2*>(feat_)[q4] = pack4h(acc);
    else reinterpret_cast<float4*>(feat_)[q4] = acc;
}

__device__ __forceinline__ void red_add_v4(float* addr, float4 v, float w) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" ::"l"(addr), "f"(v.x * w), "f"(v.y * w), "f"(v.z * w),
                 "f"(v.w * w)
                 : "memory");
}

template <bool HALF>
__global__ void __launch_bounds__(256)
k_sample_bwd(const void* __restrict__ g_feat_, const float* __restrict__ xyz, uint32_t M, int R, int C, float inv_bound,
             int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
             float* __restrict__ g_planes) {
    const int cq_per = C >> 2;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t total = (uint64_t)M * 3 * cq_per;
    if (idx >= total) return;
    const int cq = (int)(idx % cq_per);
    const int p = (int)((idx / cq_per) % 3);
    uint32_t m = (uint32_t)(idx / ((uint64_t)3 * cq_per));
    if (perm) m = (uint32_t)__ldg(perm + m);
    if (n_valid && (int32_t)m >= *n_valid) return;
    const size_t q4 = ((size_t)m * 3 * C + (size_t)p * C) / 4 + cq;
    const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + q4))
                          : __ldg(reinterpret_cast<const float4*>(g_feat_) + q4);
    if (g.x == 0.f && g.y == 0.f && g.z == 0.f && g.w == 0.f) return;  // adding zeros is a no-op
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    float* base = g_planes + (((size_t)p * R + t.y0) * R + t.x0) * C + 4 * cq;
    const size_t dx = (size_t)C, dy = (size_t)R * C;
    red_add_v4(base, g, t.nw);
    if (t.x1ok) red_add_v4(base + dx, g, t.ne);
    if (t.y1ok) red_add_v4(base + dy, g, t.sw);
    if (t.x1ok && t.y1ok) red_add_v4(base + dy + dx, g, t.se);
}

// ------------------------------------------------------------------------------------------------
// Specialised variants for C in {16, 32, 48}: 8 channels per thread (two 128-bit loads per corner), thread -> (point,
// plane, channel group) decoded with compile-time constants (the generic kernels above spend most of their issue slots
// on 64-bit index arithmetic: ncu showed them issue-bound at 20-25 % of DRAM bandwidth once the visiting order is sorted).
// ------------------------------------------------------------------------------------------------
template <int TPP>  // threads per (point, plane) = C / 8
struct SampleCfg {
    static constexpr int C = 8 * TPP;
    static constexpr int PPB = 16;                     // points per block
    static constexpr int NT = PPB * 3 * TPP;           // threads per block
};

__device__ __forceinline__ void fma4(float4& acc, const float4 v, const float w) {
    acc.x = fmaf(v.x, w, acc.x); acc.y = fmaf(v.y, w, acc.y); acc.z = fmaf(v.z, w, acc.z); acc.w = fmaf(v.w, w, acc.w);
}

template <int TPP, bool HALF>
__global__ void __launch_bounds__(SampleCfg<TPP>::NT)
k_sample_fwd8(const float* __restrict__ planes, const float* __restrict__ xyz, uint32_t M, int R, float inv_bound,
              int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
              void* __restrict__ feat_) {
    using Cfg = SampleCfg<TPP>;
    constexpr int C = Cfg::C;
    const int tid = threadIdx.x;
    const int cg = tid % TPP, p = (tid / TPP) % 3, lp = tid / (3 * TPP);
    uint32_t m = blockIdx.x * Cfg::PPB + lp;
    if (m >= M) return;
    if (perm) m = (uint32_t)__ldg(perm + m);
    const size_t q8 = ((size_t)m * 3 + p) * TPP + cg;   // index of this thread's 8-channel group
    if (n_valid && (int32_t)m >= *n_valid) {
        if (HALF) reinterpret_cast<uint4*>(feat_)[q8] = make_uint4(0u, 0u, 0u, 0u);
        else { reinterpret_cast<float4*>(feat_)[2 * q8] = make_float4(0.f, 0.f, 0.f, 0.f); reinterpret_cast<float4*>(feat_)[2 * q8 + 1] = make_float4(0.f, 0.f, 0.f, 0.f); }
        return;
    }
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    const float4* base = reinterpret_cast<const float4*>(planes + (((size_t)p * R + t.y0) * R + t.x0) * C) + 2 * cg;
    const size_t dx = C / 4, dy = (size_t)R * (C / 4);
    float4 a0, a1;
    {
        const float4 v0 = __ldg(base), v1 = __ldg(base + 1);
        a0 = make_float4(v0.x * t.nw, v0.y * t.nw, v0.z * t.nw, v0.w * t.nw);
        a1 = make_float4(v1.x * t.nw, v1.y * t.nw, v1.z * t.nw, v1.w * t.nw);
    }
    if (t.x1ok) { fma4(a0, __ldg(base + dx), t.ne); fma4(a1, __ldg(base + dx + 1), t.ne); }
    if (t.y1ok) { fma4(a0, __ldg(base + dy), t.sw); fma4(a1, __ldg(base + dy + 1), t.sw); }
    if (t.x1ok && t.y1ok) { fma4(a0, __ldg(base + dy + dx), t.se); fma4(a1, __ldg(base + dy + dx + 1), t.se); }
    if (HALF) {
        const uint2 lo = pack4h(a0), hi = pack4h(a1);
        reinterpret_cast<uint4*>(feat_)[q8] = make_uint4(lo.x, lo.y, hi.x, hi.y);
    } else {
        reinterpret_cast<float4*>(feat_)[2 * q8] = a0;
        reinterpret_cast<float4*>(feat_)[2 * q8 + 1] = a1;
    }
}

// backward: 4 channels per thread (one vector atomic per corner) -- measured faster than 8 (more atomics in flight)
template <int TPP4>  // threads per (point, plane) = C / 4
struct ScatterCfg {
    static constexpr int C = 4 * TPP4;
    static constexpr int PPB = 8;
    static constexpr int NT = PPB * 3 * TPP4;
};

template <int TPP4, bool HALF>
__global__ void __launch_bounds__(ScatterCfg<TPP4>::NT)
k_sample_bwd4(const void* __restrict__ g_feat_, const float* __restrict__ xyz, uint32_t M, int R, float inv_bound,
              int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
              float* __restrict__ g_planes) {
    using Cfg = ScatterCfg<TPP4>;
    constexpr int C = Cfg::C;
    const int tid = threadIdx.x;
    const int cq = tid % TPP4, p = (tid / TPP4) % 3, lp = tid / (3 * TPP4);
    uint32_t m = blockIdx.x * Cfg::PPB + lp;
    if (m >= M) return;
    if (perm) m = (uint32_t)__ldg(perm + m);
    if (n_valid && (int32_t)m >= *n_valid) return;
    const size_t q4 = ((size_t)m * 3 + p) * TPP4 + cq;
    const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + q4))
                          : __ldg(reinterpret_cast<const float4*>(g_feat_) + q4);
    if (g.x == 0.f && g.y == 0.f && g.z == 0.f && g.w == 0.f) return;  // adding zeros is a no-op
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    float* base = g_planes + (((size_t)p * R + t.y0) * R + t.x0) * C + 4 * cq;
    const size_t dx = (size_t)C, dy = (size_t)R * C;
    red_add_v4(base, g, t.nw);
    if (t.x1ok) red_add_v4(base + dx, g, t.ne);
    if (t.y1ok) red_add_v4(base + dy, g, t.sw);
    if (t.x1ok && t.y1ok) red_add_v4(base + dy + dx, g, t.se);
}

// the same scatter restricted to ONE plane (thread <-> (point, 4 channels); 24 points per block): the multi-GPU step scatters plane
// by plane so that the exchange of plane p overlaps the scatter of plane p + 1 (parallel.PeerGradExchange)
template <int TPP4, bool HALF>
__global__ void __launch_bounds__(ScatterCfg<TPP4>::NT)
k_sample_bwd4_plane(const void* __restrict__ g_feat_, const float* __restrict__ xyz, uint32_t M, int R, float inv_bound,
                    int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
                    float* __restrict__ g_planes, int p) {
    using Cfg = ScatterCfg<TPP4>;
    constexpr int C = Cfg::C;
    const int tid = threadIdx.x;
    const int cq = tid % TPP4, lp = tid / TPP4;
    uint32_t m = blockIdx.x * (3 * Cfg::PPB) + lp;
    if (m >= M) return;
    if (perm) m = (uint32_t)__ldg(perm + m);
    if (n_valid && (int32_t)m >= *n_valid) return;
    const size_t q4 = ((size_t)m * 3 + p) * TPP4 + cq;
    const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + q4))
                          : __ldg(reinterpret_cast<const float4*>(g_feat_) + q4);
    if (g.x == 0.f && g.y == 0.f && g.z == 0.f && g.w == 0.f) return;
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    float* base = g_planes + (((size_t)p * R + t.y0) * R + t.x0) * C + 4 * cq;
    const size_t dx = (size_t)C, dy = (size_t)R * C;
    red_add_v4(base, g, t.nw);
    if (t.x1ok) red_add_v4(base + dx, g, t.ne);
    if (t.y1ok) red_add_v4(base + dy, g, t.sw);
    if (t.x1ok && t.y1ok) red_add_v4(base + dy + dx, g, t.se);
}


// ------------------------------------------------------------------------------------------------
// Gradient with respect to the sample POSITIONS: grid_sampler_2d_backward w.r.t. the grid, chained through the projection
// u = xyz * inv_bound.  Callers that differentiate the field in space need it (the super_resolution application's analytic
// normals, super_resolution/threestudio/models/geometry/implicit_volume.py:218-226, through the F.grid_sample call of
// super_resolution/threestudio/models/triplaneencoder/triplane_encoder.py:262); the NeRF training step never does.
// Block = 32 points x 3 planes.  Thread (point, plane) walks the C channels of its four corner texels (contiguous 4*C-byte
// runs, every sector fully used) with the term order of ATen's kernel; the three planes of a point meet in shared memory
// and thread (point, axis) writes one component, so the result is deterministic and needs no atomics.
// ------------------------------------------------------------------------------------------------
constexpr int XG_PPB = 32;

__device__ __forceinline__ float dot4(const float4 a, const float4 b) {
    return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)));
}

__global__ void __launch_bounds__(3 * XG_PPB)
k_sample_xyz_grad(const float* __restrict__ g_feat, const float* __restrict__ planes, const float* __restrict__ xyz,
                  uint32_t M, int R, int C, float inv_bound, int fp16_coords, float* __restrict__ g_xyz) {
    __shared__ float s_uv[XG_PPB][3][2];
    const int p = threadIdx.x % 3, lp = threadIdx.x / 3;
    const uint32_t m = blockIdx.x * XG_PPB + lp;
    float gu = 0.f, gv = 0.f;
    if (m < M) {
        float gx, gy, mx, my;
        plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
        const float ix = to_pixel_grad(gx, R, mx), iy = to_pixel_grad(gy, R, my);
        const float fx = floorf(ix), fy = floorf(iy);
        const int x0 = (int)fx, y0 = (int)fy;
        const bool x1ok = x0 + 1 <= R - 1, y1ok = y0 + 1 <= R - 1;
        const float wx0 = (fx + 1.0f) - ix, wx1 = ix - fx, wy0 = (fy + 1.0f) - iy, wy1 = iy - fy;
        const int cq_per = C >> 2;
        const float4* base = reinterpret_cast<const float4*>(planes + (((size_t)p * R + y0) * R + x0) * C);
        const float4* go = reinterpret_cast<const float4*>(g_feat + ((size_t)m * 3 + p) * C);
        const size_t dx = (size_t)cq_per, dy = (size_t)R * cq_per;
        for (int q = 0; q < cq_per; ++q) {
            const float4 g = __ldg(go + q);
            const float nw = dot4(__ldg(base + q), g);
            const float ne = x1ok ? dot4(__ldg(base + dx + q), g) : 0.f;
            const float sw = y1ok ? dot4(__ldg(base + dy + q), g) : 0.f;
            const float se = (x1ok && y1ok) ? dot4(__ldg(base + dy + dx + q), g) : 0.f;
            gu -= nw * wy0; gv -= nw * wx0;
            gu += ne * wy0; gv -= ne * wx1;
            gu -= sw * wy1; gv += sw * wx0;
            gu += se * wy1; gv += se * wx1;
        }
        gu *= mx;
        gv *= my;
    }
    s_uv[lp][p][0] = gu;
    s_uv[lp][p][1] = gv;
    __syncthreads();
    if (m < M) {
        // axis a = p of this thread: x <- u of planes 0, 1;  y <- v of plane 1, u of plane 2;  z <- v of planes 0, 2
        const float s = (p == 0) ? s_uv[lp][0][0] + s_uv[lp][1][0]
                      : (p == 1) ? s_uv[lp][1][1] + s_uv[lp][2][0]
                                 : s_uv[lp][0][1] + s_uv[lp][2][1];
        g_xyz[3 * (size_t)m + p] = s * inv_bound;
    }
}

// The same gradient for the NeRF sampler's streams: g_feat fp16 or fp32 (HALF), rows visited in `perm` order, rows >= *n_valid
// set to zero, and the fp16-autocast rounding of the reference's backward (fp16_coords): its projection matmul returns the grid
// gradient of each plane rounded to fp16, sums the two planes that read an axis in fp16 (the broadcast reduction of the matmul
// backward), and the division by bound scales that in fp32.  A caller that needs the plane gradient too launches
// tnl_sample_planes_backward separately: folding the scatter into this kernel's pass over the taps was measured slower than the two
// launches (profiles/README.md).
template <bool HALF>
__global__ void __launch_bounds__(3 * XG_PPB)
k_sample_xyz_grad_nerf(const void* __restrict__ g_feat_, const float* __restrict__ planes, const float* __restrict__ xyz, uint32_t M,
                       int R, int C, float inv_bound, int fp16_coords, const int32_t* __restrict__ n_valid,
                       const int32_t* __restrict__ perm, float* __restrict__ g_xyz) {
    __shared__ float s_uv[XG_PPB][3][2];
    const int p = threadIdx.x % 3, lp = threadIdx.x / 3;
    const uint32_t i = blockIdx.x * XG_PPB + lp;
    const uint32_t m = (i < M && perm) ? (uint32_t)__ldg(perm + i) : i;
    const bool valid = i < M && !(n_valid && (int32_t)m >= *n_valid);
    float gu = 0.f, gv = 0.f;
    if (valid) {
        float gx, gy, mx, my;
        plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
        const float ix = to_pixel_grad(gx, R, mx), iy = to_pixel_grad(gy, R, my);
        const float fx = floorf(ix), fy = floorf(iy);
        const int x0 = (int)fx, y0 = (int)fy;
        const bool x1ok = x0 + 1 <= R - 1, y1ok = y0 + 1 <= R - 1;
        const float wx0 = (fx + 1.0f) - ix, wx1 = ix - fx, wy0 = (fy + 1.0f) - iy, wy1 = iy - fy;
        const int cq_per = C >> 2;
        const size_t row = (size_t)m * 3 * C + (size_t)p * C;
        const float4* base = reinterpret_cast<const float4*>(planes + (((size_t)p * R + y0) * R + x0) * C);
        const size_t dx = (size_t)cq_per, dy = (size_t)R * cq_per;
        for (int q = 0; q < cq_per; ++q) {
            const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + row / 4 + q))
                                  : __ldg(reinterpret_cast<const float4*>(g_feat_) + row / 4 + q);
            const float nw = dot4(__ldg(base + q), g);
            const float ne = x1ok ? dot4(__ldg(base + dx + q), g) : 0.f;
            const float sw = y1ok ? dot4(__ldg(base + dy + q), g) : 0.f;
            const float se = (x1ok && y1ok) ? dot4(__ldg(base + dy + dx + q), g) : 0.f;
            gu -= nw * wy0; gv -= nw * wx0;
            gu += ne * wy0; gv -= ne * wx1;
            gu -= sw * wy1; gv += sw * wx0;
            gu += se * wy1; gv += se * wx1;
        }
        gu *= mx;
        gv *= my;
        if (fp16_coords) { gu = __half2float(__float2half_rn(gu)); gv = __half2float(__float2half_rn(gv)); }
    }
    s_uv[lp][p][0] = gu;
    s_uv[lp][p][1] = gv;
    __syncthreads();
    if (i < M) {
        // axis a = p of this thread: x <- u of planes 0, 1;  y <- v of plane 1, u of plane 2;  z <- v of planes 0, 2
        float s = (p == 0) ? s_uv[lp][0][0] + s_uv[lp][1][0]
                : (p == 1) ? s_uv[lp][1][1] + s_uv[lp][2][0]
                           : s_uv[lp][0][1] + s_uv[lp][2][1];
        if (fp16_coords) s = __half2float(__float2half_rn(s));
        g_xyz[3 * (size_t)m + p] = valid ? s * inv_bound : 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
// Deterministic scatter (torch.use_deterministic_algorithms): the same contributions c = g * w as k_sample_bwd4, added in
// 64-bit fixed point.  Integer addition is associative, so the sums do not depend on the visiting order (perm) or on the
// thread schedule.  Scale: m = max |g_feat| over the rows below *n_valid, 2^e > m, mu = ceil(log2 M), unit = 2^(e + mu - 62).
// Every bilinear weight is <= 1, so |c| <= m < 2^e, and a texel of one plane receives at most M contributions: no partial sum
// reaches 2^62 units.  Each contribution is rounded once to a multiple of the unit (error <= unit / 2), the texel's sum is
// rounded once to fp32.  A non-finite g_feat row turns the whole converted gradient into NaN, so that loss scaling skips the
// step as it does with the fp32 atomics.
// ------------------------------------------------------------------------------------------------
struct DetScale {
    int state;          // 0: every contribution is zero, 1: finite, 2: some g_feat value is inf or NaN
    double to_fixed;    // 2^(62 - e - mu)
    float unit;         // 2^(e + mu - 62)
};

__device__ __forceinline__ DetScale det_scale(uint32_t absmax_bits, uint32_t M) {
    DetScale s{0, 0.0, 0.f};
    if (absmax_bits == 0u) return s;
    if (absmax_bits >= 0x7f800000u) { s.state = 2; return s; }
    int e;
    frexpf(__uint_as_float(absmax_bits), &e);                 // m = f 2^e, f in [0.5, 1): 2^e > m
    const int mu = M > 1u ? 32 - __clz((int)(M - 1u)) : 0;     // 2^mu >= M
    s.state = 1;
    s.to_fixed = ldexp(1.0, 62 - e - mu);
    s.unit = ldexpf(1.f, e + mu - 62);
    return s;
}

// max |g_feat| over rows [0, min(*n_valid, M)) as the bit pattern of a non-negative float (order-free atomicMax; NaN > inf)
template <bool HALF>
__global__ void __launch_bounds__(256)
k_det_absmax(const void* __restrict__ g_feat_, uint32_t M, int C, const int32_t* __restrict__ n_valid, uint32_t* __restrict__ absmax) {
    uint32_t rows = M;
    if (n_valid) rows = *n_valid < 0 ? 0u : min((uint32_t)*n_valid, M);
    const size_t n4 = (size_t)rows * 3 * C / 4;
    uint32_t mx = 0u;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + i)) : __ldg(reinterpret_cast<const float4*>(g_feat_) + i);
        mx = max(mx, max(max(__float_as_uint(fabsf(g.x)), __float_as_uint(fabsf(g.y))), max(__float_as_uint(fabsf(g.z)), __float_as_uint(fabsf(g.w)))));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx != 0u) atomicMax(absmax, mx);
}

__device__ __forceinline__ void red_add_fixed(unsigned long long* addr, float4 v, float w, double to_fixed) {
    atomicAdd(addr, (unsigned long long)llrint((double)(v.x * w) * to_fixed));
    atomicAdd(addr + 1, (unsigned long long)llrint((double)(v.y * w) * to_fixed));
    atomicAdd(addr + 2, (unsigned long long)llrint((double)(v.z * w) * to_fixed));
    atomicAdd(addr + 3, (unsigned long long)llrint((double)(v.w * w) * to_fixed));
}

// thread <-> (point, plane, 4-channel group) as in k_sample_bwd4; TPP4 = C / 4, or 0 for a run-time C
template <int TPP4, bool HALF>
__global__ void __launch_bounds__(256)
k_sample_bwd_det(const void* __restrict__ g_feat_, const float* __restrict__ xyz, uint32_t M, int R, int C_rt, float inv_bound,
                 int fp16_coords, const int32_t* __restrict__ n_valid, const int32_t* __restrict__ perm,
                 const uint32_t* __restrict__ absmax, unsigned long long* __restrict__ acc) {
    const int C = TPP4 ? 4 * TPP4 : C_rt, cq_per = C >> 2;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)M * 3 * cq_per) return;
    const DetScale sc = det_scale(*absmax, M);
    if (sc.state != 1) return;
    const int cq = (int)(idx % cq_per);
    const int p = (int)((idx / cq_per) % 3);
    uint32_t m = (uint32_t)(idx / ((uint64_t)3 * cq_per));
    if (perm) m = (uint32_t)__ldg(perm + m);
    if (n_valid && (int32_t)m >= *n_valid) return;
    const size_t q4 = ((size_t)m * 3 + p) * cq_per + cq;
    const float4 g = HALF ? unpack4h(__ldg(reinterpret_cast<const uint2*>(g_feat_) + q4))
                          : __ldg(reinterpret_cast<const float4*>(g_feat_) + q4);
    if (g.x == 0.f && g.y == 0.f && g.z == 0.f && g.w == 0.f) return;  // adding zeros is a no-op
    float gx, gy;
    plane_coords(xyz, m, p, inv_bound, fp16_coords, gx, gy);
    const Tap t = make_tap(gx, gy, R);
    unsigned long long* base = acc + (((size_t)p * R + t.y0) * R + t.x0) * C + 4 * cq;
    const size_t dx = (size_t)C, dy = (size_t)R * C;
    red_add_fixed(base, g, t.nw, sc.to_fixed);
    if (t.x1ok) red_add_fixed(base + dx, g, t.ne, sc.to_fixed);
    if (t.y1ok) red_add_fixed(base + dy, g, t.sw, sc.to_fixed);
    if (t.x1ok && t.y1ok) red_add_fixed(base + dy + dx, g, t.se, sc.to_fixed);
}

// g_planes += acc * unit (one rounding: the int64 -> fp32 conversion; the unit is a power of two) over the listed T x T tiles of
// [3][R][R][C] (ids / *count as tnl_tiles_zero), or over the whole planes when ids == nullptr
__global__ void __launch_bounds__(256)
k_det_convert(const unsigned long long* __restrict__ acc, float* __restrict__ g_planes, const int32_t* __restrict__ ids,
              const int32_t* __restrict__ count, int R, int C, int T, const uint32_t* __restrict__ absmax, uint32_t M) {
    const DetScale sc = det_scale(*absmax, M);
    if (sc.state == 0) return;
    const float nan = __uint_as_float(0x7fffffffu);
    if (ids == nullptr) {
        const size_t n = (size_t)3 * R * R * C;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
            g_planes[i] = sc.state == 2 ? nan : g_planes[i] + (float)(long long)acc[i] * sc.unit;
        return;
    }
    if ((int)blockIdx.x >= __ldg(count)) return;
    const int id = __ldg(ids + blockIdx.x), nt = R / T;
    const int p = id / (nt * nt), ty = (id / nt) % nt, tx = id % nt;
    const int rows_per_cta = (T + gridDim.y - 1) / gridDim.y;
    const int row_end = min(T, (int)(blockIdx.y + 1) * rows_per_cta);
    for (int row = blockIdx.y * rows_per_cta; row < row_end; ++row) {
        const size_t o = (((size_t)p * R + (size_t)ty * T + row) * R + (size_t)tx * T) * C;
        for (int i = threadIdx.x; i < T * C; i += blockDim.x)
            g_planes[o + i] = sc.state == 2 ? nan : g_planes[o + i] + (float)(long long)acc[o + i] * sc.unit;
    }
}

template <int TPP>
static void launch_fwd8(const float* planes, const float* xyz, uint32_t M, uint32_t R, float inv_bound, int fp16_coords,
                        const int32_t* n_valid, const int32_t* perm, void* feat, int half, cudaStream_t s) {
    using Cfg = SampleCfg<TPP>;
    const unsigned blocks = ceil_div(M, (uint32_t)Cfg::PPB);
    if (half) k_sample_fwd8<TPP, true><<<blocks, Cfg::NT, 0, s>>>(planes, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, feat);
    else k_sample_fwd8<TPP, false><<<blocks, Cfg::NT, 0, s>>>(planes, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, feat);
}
template <int TPP4>
static void launch_bwd4(const void* g_feat, int half, const float* xyz, uint32_t M, uint32_t R, float inv_bound, int fp16_coords,
                        const int32_t* n_valid, const int32_t* perm, float* g_planes, cudaStream_t s) {
    using Cfg = ScatterCfg<TPP4>;
    const unsigned blocks = ceil_div(M, (uint32_t)Cfg::PPB);
    if (half) k_sample_bwd4<TPP4, true><<<blocks, Cfg::NT, 0, s>>>(g_feat, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, g_planes);
    else k_sample_bwd4<TPP4, false><<<blocks, Cfg::NT, 0, s>>>(g_feat, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, g_planes);
}

template <int TPP4>
static void launch_bwd4_plane(const void* g_feat, int half, const float* xyz, uint32_t M, uint32_t R, float inv_bound, int fp16_coords,
                              const int32_t* n_valid, const int32_t* perm, float* g_planes, int plane, cudaStream_t s) {
    using Cfg = ScatterCfg<TPP4>;
    const unsigned blocks = ceil_div(M, (uint32_t)(3 * Cfg::PPB));
    if (half) k_sample_bwd4_plane<TPP4, true><<<blocks, Cfg::NT, 0, s>>>(g_feat, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, g_planes, plane);
    else k_sample_bwd4_plane<TPP4, false><<<blocks, Cfg::NT, 0, s>>>(g_feat, xyz, M, (int)R, inv_bound, fp16_coords, n_valid, perm, g_planes, plane);
}

}  // namespace tnl

using namespace tnl;

extern "C" {

int tnl_sample_planes_forward(const float* planes, const float* xyz, uint32_t M, uint32_t R, uint32_t C, float inv_bound,
                              int fp16_coords, const int32_t* n_valid, const int32_t* perm, void* feat, int feat_fp16,
                              tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(planes && xyz && feat, "null pointer");
    TNL_ARG_CHECK(C >= 4 && C % 4 == 0 && R >= 2, "C must be a multiple of 4, R >= 2");
    TNL_ARG_CHECK(((uintptr_t)planes & 15) == 0 && ((uintptr_t)feat & 15) == 0, "planes/feat must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (C == 16 || C == 32 || C == 48) {
        if (C == 16) launch_fwd8<2>(planes, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, feat, feat_fp16, st);
        else if (C == 32) launch_fwd8<4>(planes, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, feat, feat_fp16, st);
        else launch_fwd8<6>(planes, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, feat, feat_fp16, st);
        return finish_launch("sample_planes_forward");
    }
    const uint64_t total = (uint64_t)M * 3 * (C / 4);
    if (feat_fp16)
        k_sample_fwd<true><<<(unsigned)ceil_div(total, (uint64_t)256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
            planes, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid, perm, feat);
    else
        k_sample_fwd<false><<<(unsigned)ceil_div(total, (uint64_t)256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
            planes, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid, perm, feat);
    return finish_launch("sample_planes_forward");
}

int tnl_sample_planes_backward(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                               float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                               float* g_planes, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_feat && xyz && g_planes, "null pointer");
    TNL_ARG_CHECK(C >= 4 && C % 4 == 0 && R >= 2, "C must be a multiple of 4, R >= 2");
    TNL_ARG_CHECK(((uintptr_t)g_planes & 15) == 0 && ((uintptr_t)g_feat & 15) == 0, "g_planes/g_feat must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (C == 16 || C == 32 || C == 48) {
        if (C == 16) launch_bwd4<4>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, st);
        else if (C == 32) launch_bwd4<8>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, st);
        else launch_bwd4<12>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, st);
        return finish_launch("sample_planes_backward");
    }
    const uint64_t total = (uint64_t)M * 3 * (C / 4);
    if (feat_fp16)
        k_sample_bwd<true><<<(unsigned)ceil_div(total, (uint64_t)256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
            g_feat, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid, perm, g_planes);
    else
        k_sample_bwd<false><<<(unsigned)ceil_div(total, (uint64_t)256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
            g_feat, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid, perm, g_planes);
    return finish_launch("sample_planes_backward");
}

int tnl_sample_planes_backward_plane(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                                     float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                     float* g_planes, uint32_t plane, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_feat && xyz && g_planes && plane < 3, "null pointer / plane index");
    TNL_ARG_CHECK(C == 16 || C == 32 || C == 48, "per-plane scatter: C in {16, 32, 48}");
    TNL_ARG_CHECK(((uintptr_t)g_planes & 15) == 0 && ((uintptr_t)g_feat & 15) == 0, "g_planes/g_feat must be 16-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (C == 16) launch_bwd4_plane<4>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, (int)plane, st);
    else if (C == 32) launch_bwd4_plane<8>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, (int)plane, st);
    else launch_bwd4_plane<12>(g_feat, feat_fp16, xyz, M, R, inv_bound, fp16_coords, n_valid, perm, g_planes, (int)plane, st);
    return finish_launch("sample_planes_backward_plane");
}

size_t tnl_sample_planes_backward_det_workspace(uint32_t R, uint32_t C) {
    return 256 + (size_t)3 * R * R * C * sizeof(unsigned long long);
}

int tnl_sample_planes_backward_det(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                                   float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                   const int32_t* tile_ids, const int32_t* tile_count, uint32_t tile_capacity, uint32_t T,
                                   float* g_planes, void* workspace, size_t workspace_bytes, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_feat && xyz && g_planes && workspace, "null pointer");
    TNL_ARG_CHECK(C >= 4 && C % 4 == 0 && R >= 2, "C must be a multiple of 4, R >= 2");
    TNL_ARG_CHECK(((uintptr_t)g_planes & 15) == 0 && ((uintptr_t)g_feat & (feat_fp16 ? 7 : 15)) == 0 && ((uintptr_t)workspace & 255) == 0,
                  "g_planes must be 16-byte aligned, g_feat 8 (fp16) or 16 (fp32), the workspace 256");
    TNL_ARG_CHECK(workspace_bytes >= tnl_sample_planes_backward_det_workspace(R, C), "workspace too small");
    TNL_ARG_CHECK(tile_ids == nullptr || (tile_count != nullptr && T > 0 && R % T == 0), "tile list: count and a tile edge dividing R");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint32_t* absmax = static_cast<uint32_t*>(workspace);
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(workspace) + 256);
    cudaMemsetAsync(absmax, 0, sizeof(uint32_t), st);
    if (tile_ids) {
        // the int64 accumulator viewed as fp32 planes of 2C channels: the same tiles, zeroed by the same kernel
        if (tile_capacity > 0) {
            const int rc = tnl_tiles_zero(reinterpret_cast<float*>(acc), tile_ids, tile_count, tile_capacity, R, 2 * C, T, stream);
            if (rc != 0) return rc;
        }
    } else {
        cudaMemsetAsync(acc, 0, (size_t)3 * R * R * C * sizeof(unsigned long long), st);
    }
    const uint32_t absmax_blocks = (uint32_t)min(ceil_div((uint64_t)M * 3 * C / 4, (uint64_t)256), (uint64_t)kNumSM * 8);
    if (feat_fp16) k_det_absmax<true><<<absmax_blocks, 256, 0, st>>>(g_feat, M, (int)C, n_valid, absmax);
    else k_det_absmax<false><<<absmax_blocks, 256, 0, st>>>(g_feat, M, (int)C, n_valid, absmax);
    const unsigned blocks = (unsigned)ceil_div((uint64_t)M * 3 * (C / 4), (uint64_t)256);
#define TNL_DET_SCATTER(TPP4)                                                                                                       \
    do {                                                                                                                            \
        if (feat_fp16) k_sample_bwd_det<TPP4, true><<<blocks, 256, 0, st>>>(g_feat, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, \
                                                                            n_valid, perm, absmax, acc);                            \
        else k_sample_bwd_det<TPP4, false><<<blocks, 256, 0, st>>>(g_feat, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid, \
                                                                   perm, absmax, acc);                                              \
    } while (0)
    if (C == 16) TNL_DET_SCATTER(4);
    else if (C == 32) TNL_DET_SCATTER(8);
    else if (C == 48) TNL_DET_SCATTER(12);
    else TNL_DET_SCATTER(0);
#undef TNL_DET_SCATTER
    if (tile_ids) {
        if (tile_capacity > 0)
            k_det_convert<<<dim3(tile_capacity, 4), 256, 0, st>>>(acc, g_planes, tile_ids, tile_count, (int)R, (int)C, (int)T, absmax, M);
    } else {
        k_det_convert<<<kNumSM * 8, 256, 0, st>>>(acc, g_planes, nullptr, nullptr, (int)R, (int)C, 1, absmax, M);
    }
    return finish_launch("sample_planes_backward_det");
}

int tnl_sample_planes_backward_coords(const float* g_feat, const float* planes, const float* xyz, uint32_t M, uint32_t R,
                                      uint32_t C, float inv_bound, int fp16_coords, float* g_xyz, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_feat && planes && xyz && g_xyz, "null pointer");
    TNL_ARG_CHECK(C >= 4 && C % 4 == 0 && R >= 2, "C must be a multiple of 4, R >= 2");
    TNL_ARG_CHECK(((uintptr_t)planes & 15) == 0 && ((uintptr_t)g_feat & 15) == 0, "planes/g_feat must be 16-byte aligned");
    k_sample_xyz_grad<<<ceil_div(M, (uint32_t)XG_PPB), 3 * XG_PPB, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        g_feat, planes, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, g_xyz);
    return finish_launch("sample_planes_backward_coords");
}

int tnl_sample_planes_backward_xyz(const void* g_feat, int feat_fp16, const float* planes, const float* xyz, uint32_t M, uint32_t R,
                                   uint32_t C, float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                   float* g_xyz, tnl_stream_t stream) {
    if (M == 0) return 0;
    TNL_ARG_CHECK(g_feat && planes && xyz && g_xyz, "null pointer");
    TNL_ARG_CHECK(C >= 4 && C % 4 == 0 && R >= 2, "C must be a multiple of 4, R >= 2");
    TNL_ARG_CHECK(((uintptr_t)planes & 15) == 0 && ((uintptr_t)g_feat & (feat_fp16 ? 7 : 15)) == 0,
                  "planes must be 16-byte aligned, g_feat 8 (fp16) or 16 (fp32)");
    const unsigned blocks = ceil_div(M, (uint32_t)XG_PPB);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (feat_fp16)
        k_sample_xyz_grad_nerf<true><<<blocks, 3 * XG_PPB, 0, st>>>(g_feat, planes, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid,
                                                                   perm, g_xyz);
    else
        k_sample_xyz_grad_nerf<false><<<blocks, 3 * XG_PPB, 0, st>>>(g_feat, planes, xyz, M, (int)R, (int)C, inv_bound, fp16_coords, n_valid,
                                                                    perm, g_xyz);
    return finish_launch("sample_planes_backward_xyz");
}

}  // extern "C"
