// Ray utilities, occupancy-grid marching, compositing, SH encoding -- sm_100a.
//
// Behavioural contract: /root/reference/aux_libs/raymarching/src/raymarching.cu (kernels :91-905) and
// aux_libs/shencoder/src/shencoder.cu:27-123.  Integer results (sample counts, cell indices, bits)
// and fp32 sample positions are bit-exact with the reference's nvcc build: every float operation whose
// rounding matters is written with an explicit round-to-nearest intrinsic in the order (and with the
// FMA contractions) the reference's SASS performs them, so no compiler version can re-associate them.
//
// Design differences (B200-first, not a port):
//   * march_rays_train is count -> deterministic device-wide exclusive scan -> write, so the sample
//     layout is ray-ordered and reproducible (the reference races on atomicAdd, :405-406);
//   * stream argument everywhere (the reference launches on the legacy default stream);
//   * alive-ray compaction runs on the device (kills the per-iteration D2H sync of renderer.py:364).
#include "common.cuh"
#include "mlp_math.cuh"
#include <float.h>

namespace tnl {

constexpr float kSqrt3x2 = 3.4641016151377544f;  // 2*sqrt(3) as the reference's fp32 product 2 * 1.7320508f
constexpr float kRPi = 0.3183098861837907f;

__device__ __forceinline__ float clampf(float x, float lo, float hi) { return fminf(hi, fmaxf(lo, x)); }

__host__ __device__ __forceinline__ uint32_t spread3(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
__host__ __device__ __forceinline__ uint32_t morton_encode(uint32_t x, uint32_t y, uint32_t z) {
    return spread3(x) | (spread3(y) << 1) | (spread3(z) << 2);
}
__host__ __device__ __forceinline__ uint32_t compact3(uint32_t x) {
    x &= 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

// ------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------
__global__ void k_near_far(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                           const float* __restrict__ aabb, uint32_t N, float min_near,
                           float* __restrict__ nears, float* __restrict__ fars) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float tn = 0.f, tf = 0.f;
    bool miss = false;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float o = rays_o[3 * (size_t)n + a];
        const float r = __fdiv_rn(1.0f, rays_d[3 * (size_t)n + a]);
        float t0 = __fmul_rn(__fsub_rn(aabb[a], o), r);
        float t1 = __fmul_rn(__fsub_rn(aabb[a + 3], o), r);
        if (t0 > t1) { const float s = t0; t0 = t1; t1 = s; }
        if (a == 0) { tn = t0; tf = t1; continue; }
        if (tn > t1 || t0 > tf) { miss = true; break; }
        if (t0 > tn) tn = t0;
        if (t1 < tf) tf = t1;
    }
    if (miss) { nears[n] = FLT_MAX; fars[n] = FLT_MAX; return; }
    if (tn < min_near) tn = min_near;
    nears[n] = tn;
    fars[n] = tf;
}

__global__ void k_sph_from_ray(const float* __restrict__ rays_o, const float* __restrict__ rays_d, float radius,
                               uint32_t N, float* __restrict__ coords) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float ox = rays_o[3 * (size_t)n], oy = rays_o[3 * (size_t)n + 1], oz = rays_o[3 * (size_t)n + 2];
    const float dx = rays_d[3 * (size_t)n], dy = rays_d[3 * (size_t)n + 1], dz = rays_d[3 * (size_t)n + 2];
    const float A = dx * dx + dy * dy + dz * dz;
    const float B = ox * dx + oy * dy + oz * dz;
    const float C = ox * ox + oy * oy + oz * oz - radius * radius;
    const float t = (-B + sqrtf(B * B - A * C)) / A;
    const float x = ox + t * dx, y = oy + t * dy, z = oz + t * dz;
    const float theta = atan2f(sqrtf(x * x + z * z), y);
    const float phi = atan2f(z, x);
    coords[2 * (size_t)n] = 2 * theta * kRPi - 1;
    coords[2 * (size_t)n + 1] = phi * kRPi;
}

__global__ void k_morton3d(const int32_t* __restrict__ coords, uint32_t N, int32_t* __restrict__ indices) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    indices[n] = (int32_t)morton_encode((uint32_t)coords[3 * (size_t)n], (uint32_t)coords[3 * (size_t)n + 1],
                                        (uint32_t)coords[3 * (size_t)n + 2]);
}

__global__ void k_morton3d_invert(const int32_t* __restrict__ indices, uint32_t N, int32_t* __restrict__ coords) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int32_t v = indices[n];  // signed shifts, as the reference (:249-253)
    coords[3 * (size_t)n + 0] = (int32_t)compact3((uint32_t)(v >> 0));
    coords[3 * (size_t)n + 1] = (int32_t)compact3((uint32_t)(v >> 1));
    coords[3 * (size_t)n + 2] = (int32_t)compact3((uint32_t)(v >> 2));
}

// One thread packs 4 bytes (32 cells): two 128-bit loads per byte, one 32-bit store. N = output bytes.
__global__ void k_packbits(const float* __restrict__ grid, uint32_t N, float thresh, uint8_t* __restrict__ bitfield) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;  // 32-bit word index
    const uint32_t nwords = N / 4;
    if (w < nwords) {
        const float4* g = reinterpret_cast<const float4*>(grid) + (size_t)w * 8;
        uint32_t bits = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 v = __ldg(g + q);
            bits |= (v.x > thresh ? 1u : 0u) << (4 * q + 0);
            bits |= (v.y > thresh ? 1u : 0u) << (4 * q + 1);
            bits |= (v.z > thresh ? 1u : 0u) << (4 * q + 2);
            bits |= (v.w > thresh ? 1u : 0u) << (4 * q + 3);
        }
        reinterpret_cast<uint32_t*>(bitfield)[w] = bits;
    } else if (w == nwords) {  // ragged tail bytes (N % 4)
        for (uint32_t b = nwords * 4; b < N; ++b) {
            uint8_t bits = 0;
            for (int i = 0; i < 8; ++i) bits |= (grid[(size_t)b * 8 + i] > thresh) ? (uint8_t)(1u << i) : 0;
            bitfield[b] = bits;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// marching core: one probe at parameter t (shared by training and inference marching)
// ------------------------------------------------------------------------------------------------
struct MarchRay {
    float ox, oy, oz, dx, dy, dz, rdx, rdy, rdz;
};
struct MarchParams {
    float bound, dt_gamma, dt_min, dt_max, rH, Hf, Hm1f, Cf;
    uint32_t H3;
    int H;
    const uint8_t* grid;
};

__device__ __forceinline__ MarchParams make_params(float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                                                   uint32_t H, const uint8_t* grid) {
    MarchParams p;
    p.bound = bound;
    p.dt_gamma = dt_gamma;
    p.dt_min = __fdiv_rn(kSqrt3x2, (float)max_steps);
    p.dt_max = __fdiv_rn(__fmul_rn(kSqrt3x2, (float)(1 << (C - 1))), (float)H);
    p.rH = __fdiv_rn(1.0f, (float)H);
    p.Hf = (float)H;
    p.Hm1f = (float)(H - 1);
    p.Cf = (float)C;
    p.H3 = H * H * H;
    p.H = (int)H;
    p.grid = grid;
    return p;
}

__device__ __forceinline__ MarchRay load_ray(const float* __restrict__ o, const float* __restrict__ d) {
    MarchRay r;
    r.ox = o[0]; r.oy = o[1]; r.oz = o[2];
    r.dx = d[0]; r.dy = d[1]; r.dz = d[2];
    r.rdx = __fdiv_rn(1.0f, r.dx); r.rdy = __fdiv_rn(1.0f, r.dy); r.rdz = __fdiv_rn(1.0f, r.dz);
    return r;
}

__device__ __forceinline__ int level_of(float v, float Cf) {
    int e;
    frexpf(v, &e);
    return (int)fminf(Cf - 1.0f, fmaxf(0.0f, (float)e));
}

__device__ __forceinline__ float exit_dist(int n, float d, float rd, float pos, float mip_bound, float rH) {
    // (((n + 0.5 + 0.5*sign(d)) * rH * 2 - 1) * mip_bound - pos) * rd   with the reference's contractions
    float v = __fadd_rn((float)n, 0.5f);
    v = __fmaf_rn(copysignf(1.0f, d), 0.5f, v);
    v = __fmul_rn(v, rH);
    v = __fmaf_rn(v, 2.0f, -1.0f);
    v = __fmaf_rn(mip_bound, v, -pos);
    return __fmul_rn(v, rd);
}

// Returns true if the cell containing the point at `t` is occupied; then (x,y,z,dt) describe the sample.
// Otherwise advances t past the cell boundary with the reference's repeated-increment loop.
__device__ __forceinline__ bool march_probe(const MarchParams& p, const MarchRay& r, float& t, float& x, float& y,
                                            float& z, float& dt) {
    x = clampf(__fmaf_rn(t, r.dx, r.ox), -p.bound, p.bound);
    y = clampf(__fmaf_rn(t, r.dy, r.oy), -p.bound, p.bound);
    z = clampf(__fmaf_rn(t, r.dz, r.oz), -p.bound, p.bound);
    dt = clampf(__fmul_rn(t, p.dt_gamma), p.dt_min, p.dt_max);
    const int la = level_of(fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z))), p.Cf);
    const int lb = level_of(__fmul_rn(__fmul_rn(dt, p.Hf), 0.5f), p.Cf);
    const int level = max(la, lb);
    const float mip_bound = fminf(scalbnf(1.0f, level), p.bound);
    const float mip_rbound = __fdiv_rn(1.0f, mip_bound);
    // 0.5 * (x * mip_rbound + 1) * H : fma in fp32, then two exact scalings (the reference widens to
    // double for them, :374-376; the products are exact either way), clamp, truncate.
    const int nx = __float2int_rz(clampf(__fmul_rn(__fmul_rn(0.5f, __fmaf_rn(x, mip_rbound, 1.0f)), p.Hf), 0.0f, p.Hm1f));
    const int ny = __float2int_rz(clampf(__fmul_rn(__fmul_rn(0.5f, __fmaf_rn(y, mip_rbound, 1.0f)), p.Hf), 0.0f, p.Hm1f));
    const int nz = __float2int_rz(clampf(__fmul_rn(__fmul_rn(0.5f, __fmaf_rn(z, mip_rbound, 1.0f)), p.Hf), 0.0f, p.Hm1f));
    const uint32_t index = (uint32_t)level * p.H3 + morton_encode((uint32_t)nx, (uint32_t)ny, (uint32_t)nz);
    const bool occ = (__ldg(p.grid + (index >> 3)) >> (index & 7)) & 1;
    if (occ) return true;
    const float tx = exit_dist(nx, r.dx, r.rdx, x, mip_bound, p.rH);
    const float ty = exit_dist(ny, r.dy, r.rdy, y, mip_bound, p.rH);
    const float tz = exit_dist(nz, r.dz, r.rdz, z, mip_bound, p.rH);
    const float tt = __fadd_rn(t, fmaxf(0.0f, fminf(tx, fminf(ty, tz))));
    do {
        t = __fadd_rn(t, clampf(__fmul_rn(t, p.dt_gamma), p.dt_min, p.dt_max));
    } while (t < tt);
    return false;
}

// pass 1: count samples per ray; rays[n] = (n, ?, count)
__global__ void k_march_train_count(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                    const uint8_t* __restrict__ grid, float bound, float dt_gamma, uint32_t max_steps,
                                    uint32_t N, uint32_t C, uint32_t H, const float* __restrict__ nears,
                                    const float* __restrict__ fars, const float* __restrict__ noises,
                                    int32_t* __restrict__ rays, float* __restrict__ ts) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const MarchParams p = make_params(bound, dt_gamma, max_steps, C, H, grid);
    const MarchRay r = load_ray(rays_o + 3 * (size_t)n, rays_d + 3 * (size_t)n);
    const float far = fars[n];
    float t = nears[n];
    t = __fmaf_rn(clampf(__fmul_rn(t, dt_gamma), p.dt_min, p.dt_max), noises[n], t);
    uint32_t num = 0;
    float x, y, z, dt;
    float* tn = ts ? ts + (size_t)n * max_steps : nullptr;    // optional: the parameter of every sample, for k_march_train_emit
    while (t < far && num < max_steps) {
        if (march_probe(p, r, t, x, y, z, dt)) {
            if (tn) tn[num] = t;
            ++num;
            t = __fadd_rn(t, dt);
        }
    }
    rays[3 * (size_t)n] = (int32_t)n;
    rays[3 * (size_t)n + 2] = (int32_t)num;
}

// pass 2: re-march and write the samples into [offset, offset+count).  TS: also write each row's ray parameter t to ts_out.
template <bool TS>
__device__ __forceinline__ void march_train_write(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                  const uint8_t* __restrict__ grid, float bound, float dt_gamma, uint32_t max_steps,
                                                  uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* __restrict__ nears,
                                                  const float* __restrict__ fars, const float* __restrict__ noises,
                                                  const int32_t* __restrict__ rays, float* __restrict__ xyzs,
                                                  float* __restrict__ dirs, float* __restrict__ deltas, float* __restrict__ ts_out) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const uint32_t offset = (uint32_t)rays[3 * (size_t)n + 1];
    const uint32_t num = (uint32_t)rays[3 * (size_t)n + 2];
    if (num == 0 || offset + num > M) return;  // overflowing rays are dropped silently, as the reference (:416)
    const MarchParams p = make_params(bound, dt_gamma, max_steps, C, H, grid);
    const MarchRay r = load_ray(rays_o + 3 * (size_t)n, rays_d + 3 * (size_t)n);
    const float far = fars[n];
    float t = nears[n];
    t = __fmaf_rn(clampf(__fmul_rn(t, dt_gamma), p.dt_min, p.dt_max), noises[n], t);
    float last_t = t;
    float* px = xyzs + 3 * (size_t)offset;
    float* pd = dirs + 3 * (size_t)offset;
    float* pl = deltas + 2 * (size_t)offset;
    float* pt = TS ? ts_out + offset : nullptr;
    uint32_t step = 0;
    float x, y, z, dt;
    while (t < far && step < num) {
        if (march_probe(p, r, t, x, y, z, dt)) {
            px[0] = x; px[1] = y; px[2] = z;
            pd[0] = r.dx; pd[1] = r.dy; pd[2] = r.dz;
            if (TS) *pt++ = t;
            t = __fadd_rn(t, dt);
            pl[0] = dt;
            pl[1] = __fsub_rn(t, last_t);
            last_t = t;
            px += 3; pd += 3; pl += 2;
            ++step;
        }
    }
}

__global__ void k_march_train_write(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                    const uint8_t* __restrict__ grid, float bound, float dt_gamma, uint32_t max_steps,
                                    uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* __restrict__ nears,
                                    const float* __restrict__ fars, const float* __restrict__ noises,
                                    const int32_t* __restrict__ rays, float* __restrict__ xyzs,
                                    float* __restrict__ dirs, float* __restrict__ deltas) {
    march_train_write<false>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, noises, rays, xyzs, dirs,
                             deltas, nullptr);
}

__global__ void k_march_train_write_ts(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                       const uint8_t* __restrict__ grid, float bound, float dt_gamma, uint32_t max_steps,
                                       uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* __restrict__ nears,
                                       const float* __restrict__ fars, const float* __restrict__ noises,
                                       const int32_t* __restrict__ rays, float* __restrict__ xyzs,
                                       float* __restrict__ dirs, float* __restrict__ deltas, float* __restrict__ ts_out) {
    march_train_write<true>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, noises, rays, xyzs, dirs,
                            deltas, ts_out);
}

// pass 2 without a second traversal: pass 1 recorded the parameter t of every sample (ts[n][k]); one warp per ray turns them into
// positions / directions / deltas with the very operations of the traversal (same roundings => bit-identical rows) and writes
// the ray's rows coalesced.  The occupancy grid is not touched again.  TS: also write each row's t to ts_out.
template <bool TS>
__device__ __forceinline__ void march_train_emit(const float* __restrict__ rays_o, const float* __restrict__ rays_d, float bound,
                                                 float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                                 const float* __restrict__ nears, const float* __restrict__ noises,
                                                 const int32_t* __restrict__ rays, const float* __restrict__ ts, float* __restrict__ xyzs,
                                                 float* __restrict__ dirs, float* __restrict__ deltas, float* __restrict__ ts_out) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t offset = (uint32_t)rays[3 * (size_t)n + 1];
    const uint32_t num = (uint32_t)rays[3 * (size_t)n + 2];
    if (num == 0 || offset + num > M) return;  // overflowing rays are dropped silently, as the reference (:416)
    const MarchParams p = make_params(bound, dt_gamma, max_steps, C, H, nullptr);
    const MarchRay r = load_ray(rays_o + 3 * (size_t)n, rays_d + 3 * (size_t)n);
    float t0 = nears[n];
    t0 = __fmaf_rn(clampf(__fmul_rn(t0, dt_gamma), p.dt_min, p.dt_max), noises[n], t0);      // last_t before the first sample
    const float* tn = ts + (size_t)n * max_steps;
    for (uint32_t k = lane; k < num; k += 32) {
        const float t = tn[k];
        const float dt = clampf(__fmul_rn(t, p.dt_gamma), p.dt_min, p.dt_max);
        float last_t = t0;
        if (k > 0) {
            const float tp = tn[k - 1];
            last_t = __fadd_rn(tp, clampf(__fmul_rn(tp, p.dt_gamma), p.dt_min, p.dt_max));
        }
        const size_t i = (size_t)offset + k;
        xyzs[3 * i] = clampf(__fmaf_rn(t, r.dx, r.ox), -p.bound, p.bound);
        xyzs[3 * i + 1] = clampf(__fmaf_rn(t, r.dy, r.oy), -p.bound, p.bound);
        xyzs[3 * i + 2] = clampf(__fmaf_rn(t, r.dz, r.oz), -p.bound, p.bound);
        dirs[3 * i] = r.dx; dirs[3 * i + 1] = r.dy; dirs[3 * i + 2] = r.dz;
        deltas[2 * i] = dt;
        deltas[2 * i + 1] = __fsub_rn(__fadd_rn(t, dt), last_t);
        if (TS) ts_out[i] = t;
    }
}

__global__ void __launch_bounds__(256)
k_march_train_emit(const float* __restrict__ rays_o, const float* __restrict__ rays_d, float bound, float dt_gamma, uint32_t max_steps,
                   uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* __restrict__ nears, const float* __restrict__ noises,
                   const int32_t* __restrict__ rays, const float* __restrict__ ts, float* __restrict__ xyzs, float* __restrict__ dirs,
                   float* __restrict__ deltas) {
    march_train_emit<false>(rays_o, rays_d, bound, dt_gamma, max_steps, N, C, H, M, nears, noises, rays, ts, xyzs, dirs, deltas, nullptr);
}

__global__ void __launch_bounds__(256)
k_march_train_emit_ts(const float* __restrict__ rays_o, const float* __restrict__ rays_d, float bound, float dt_gamma,
                      uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* __restrict__ nears,
                      const float* __restrict__ noises, const int32_t* __restrict__ rays, const float* __restrict__ ts,
                      float* __restrict__ xyzs, float* __restrict__ dirs, float* __restrict__ deltas, float* __restrict__ ts_out) {
    march_train_emit<true>(rays_o, rays_d, bound, dt_gamma, max_steps, N, C, H, M, nears, noises, rays, ts, xyzs, dirs, deltas, ts_out);
}

// ------------------------------------------------------------------------------------------------
// device-wide exclusive scan of uint32 values read with a stride (three small kernels)
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total, uint32_t* smem /*[33]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) smem[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = (lane < (int)(blockDim.x >> 5)) ? smem[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += u;
        }
        smem[lane] = wi - w;
        if (lane == 31) smem[32] = wi;
    }
    __syncthreads();
    const uint32_t res = smem[warp] + incl - v;
    *total = smem[32];
    __syncthreads();
    return res;
}

// mode 0: value = in[i*stride]; mode 1: value = (in[i*stride] >= 0) (alive flag)
template <int MODE>
__device__ __forceinline__ uint32_t scan_value(const int32_t* in, uint32_t i, uint32_t n, uint32_t stride) {
    if (i >= n) return 0u;
    const int32_t v = in[(size_t)i * stride];
    return MODE == 0 ? (uint32_t)v : (v >= 0 ? 1u : 0u);
}

template <int MODE>
__global__ void k_scan_block_sums(const int32_t* __restrict__ in, uint32_t n, uint32_t stride,
                                  uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t sm[33];
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t total;
    block_exclusive_scan(scan_value<MODE>(in, i, n, stride), &total, sm);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: in-place exclusive scan of block_sums (any length), grand total -> totals
__global__ void k_scan_of_sums(uint32_t* __restrict__ block_sums, uint32_t nblocks, int32_t* __restrict__ counter,
                               uint32_t n_items, int32_t* __restrict__ total_out) {
    __shared__ uint32_t sm[33];
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nblocks; base += kScanThreads) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? block_sums[i] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_scan(v, &total, sm);
        if (i < nblocks) block_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) {
        if (counter) {  // march_rays_train: counter[0] += total samples, counter[1] += rays
            counter[0] += (int32_t)carry;
            counter[1] += (int32_t)n_items;
        }
        if (total_out) *total_out = (int32_t)carry;
    }
}

__global__ void k_scan_offsets(const int32_t* __restrict__ in, uint32_t n, uint32_t stride,
                               const uint32_t* __restrict__ block_sums, int32_t* __restrict__ out) {
    __shared__ uint32_t sm[33];
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(scan_value<0>(in, i, n, stride), &total, sm);
    if (i < n) out[(size_t)i * stride] = (int32_t)(block_sums[blockIdx.x] + ex);
}

__global__ void k_compact_scatter(const int32_t* __restrict__ alive, uint32_t n, const uint32_t* __restrict__ block_sums,
                                  int32_t* __restrict__ out) {
    __shared__ uint32_t sm[33];
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    const uint32_t f = scan_value<1>(alive, i, n, 1);
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(f, &total, sm);
    if (f) out[block_sums[blockIdx.x] + ex] = alive[i];
}

// ------------------------------------------------------------------------------------------------
// compositing (training): one WARP per ray.  Lanes take 32 consecutive samples (coalesced loads), transmittance is an
// inclusive warp product scan, depth / colour prefix sums are warp sum scans, the early stop (T < T_thresh after
// including the sample, reference :557) is a ballot.  Same formulas as the reference kernels (:500-682); the order of
// the fp32 products / sums is a scan tree instead of a sequential chain (difference ~1e-7 relative, inside the stated
// tolerance of the composited values).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_scan_mul(float v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v *= u;
    }
    return v;
}
__device__ __forceinline__ float warp_scan_add(float v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

__global__ void __launch_bounds__(256)
k_composite_train_fwd(const float* __restrict__ sigmas, const float* __restrict__ rgbs, const float* __restrict__ deltas,
                      const int32_t* __restrict__ rays, uint32_t M, uint32_t N, float T_thresh,
                      float* __restrict__ weights_sum, float* __restrict__ depth, float* __restrict__ image) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t index = (uint32_t)rays[3 * (size_t)n];
    const uint32_t offset = (uint32_t)rays[3 * (size_t)n + 1];
    const uint32_t num = (uint32_t)rays[3 * (size_t)n + 2];
    float r = 0.f, g = 0.f, b = 0.f, ws = 0.f, d = 0.f;
    if (num != 0 && offset + num <= M) {
        float T = 1.0f, t = 0.f;  // carried across 32-sample chunks (uniform over the warp)
        for (uint32_t base = 0; base < num; base += 32) {
            const uint32_t k = base + lane;
            const bool act = k < num;
            const size_t i = (size_t)offset + k;
            const float sg = act ? __ldg(sigmas + i) : 0.f;
            const float2 dl = act ? __ldg(reinterpret_cast<const float2*>(deltas) + i) : make_float2(0.f, 0.f);
            const float c0 = act ? __ldg(rgbs + 3 * i) : 0.f, c1 = act ? __ldg(rgbs + 3 * i + 1) : 0.f,
                        c2 = act ? __ldg(rgbs + 3 * i + 2) : 0.f;
            const float alpha = act ? 1.0f - __expf(-sg * dl.x) : 0.f;
            const float incl = warp_scan_mul(1.0f - alpha, lane);      // prod_{j<=lane} (1 - alpha_j)
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            const float T_after = T * incl;
            const float tt = t + warp_scan_add(dl.y, lane);
            // first sample after which the transmittance drops below the threshold: it still contributes, later ones do not
            const uint32_t stop = __ballot_sync(0xffffffffu, act && T_after < T_thresh);
            const int last = stop ? (__ffs(stop) - 1) : 31;
            if (act && lane <= last) {
                const float w = alpha * (T * excl);
                r += w * c0; g += w * c1; b += w * c2;
                d += w * tt;
                ws += w;
            }
            if (stop) break;
            T = __shfl_sync(0xffffffffu, T_after, 31);
            t = __shfl_sync(0xffffffffu, tt, 31);
        }
        r = warp_sum(r); g = warp_sum(g); b = warp_sum(b); ws = warp_sum(ws); d = warp_sum(d);
    }
    if (lane == 0) {
        weights_sum[index] = ws;
        depth[index] = d;
        image[3 * (size_t)index] = r;
        image[3 * (size_t)index + 1] = g;
        image[3 * (size_t)index + 2] = b;
    }
}

__global__ void __launch_bounds__(256)
k_composite_train_bwd(const float* __restrict__ grad_ws, const float* __restrict__ grad_image,
                      const float* __restrict__ sigmas, const float* __restrict__ rgbs, const float* __restrict__ deltas,
                      const int32_t* __restrict__ rays, const float* __restrict__ weights_sum,
                      const float* __restrict__ image, uint32_t M, uint32_t N, float T_thresh,
                      float* __restrict__ grad_sigmas, float* __restrict__ grad_rgbs) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t index = (uint32_t)rays[3 * (size_t)n];
    const uint32_t offset = (uint32_t)rays[3 * (size_t)n + 1];
    const uint32_t num = (uint32_t)rays[3 * (size_t)n + 2];
    if (num == 0 || offset + num > M) return;
    const float gi0 = grad_image[3 * (size_t)index], gi1 = grad_image[3 * (size_t)index + 1],
                gi2 = grad_image[3 * (size_t)index + 2];
    const float tail = grad_ws[index] * (1.0f - weights_sum[index]);
    const float rf = image[3 * (size_t)index], gf = image[3 * (size_t)index + 1], bf = image[3 * (size_t)index + 2];
    float T = 1.0f, r = 0.f, g = 0.f, b = 0.f;  // carried across chunks
    bool done = false;                          // the ray has terminated: the remaining samples get zero gradient
    for (uint32_t base = 0; base < num; base += 32) {
        const uint32_t k = base + lane;
        const bool act = k < num;
        const size_t i = (size_t)offset + k;
        if (done) {                             // (the reference relies on zero-initialised outputs; here every row is written)
            if (act) { grad_rgbs[3 * i] = 0.f; grad_rgbs[3 * i + 1] = 0.f; grad_rgbs[3 * i + 2] = 0.f; grad_sigmas[i] = 0.f; }
            continue;
        }
        const float sg = act ? __ldg(sigmas + i) : 0.f;
        const float d0 = act ? __ldg(deltas + 2 * i) : 0.f;
        const float c0 = act ? __ldg(rgbs + 3 * i) : 0.f, c1 = act ? __ldg(rgbs + 3 * i + 1) : 0.f,
                    c2 = act ? __ldg(rgbs + 3 * i + 2) : 0.f;
        const float alpha = act ? 1.0f - __expf(-sg * d0) : 0.f;
        const float incl = warp_scan_mul(1.0f - alpha, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.0f;
        const float T_after = T * incl;
        const float w = alpha * (T * excl);
        const float ri = r + warp_scan_add(w * c0, lane), gi = g + warp_scan_add(w * c1, lane),
                    bi = b + warp_scan_add(w * c2, lane);   // colour accumulated up to and including this sample
        const uint32_t stop = __ballot_sync(0xffffffffu, act && T_after < T_thresh);
        const int last = stop ? (__ffs(stop) - 1) : 31;
        if (act && lane <= last) {
            grad_rgbs[3 * i] = gi0 * w;
            grad_rgbs[3 * i + 1] = gi1 * w;
            grad_rgbs[3 * i + 2] = gi2 * w;
            grad_sigmas[i] = d0 * (gi0 * (T_after * c0 - (rf - ri)) + gi1 * (T_after * c1 - (gf - gi)) +
                                   gi2 * (T_after * c2 - (bf - bi)) + tail);
        } else if (act) {
            grad_rgbs[3 * i] = 0.f; grad_rgbs[3 * i + 1] = 0.f; grad_rgbs[3 * i + 2] = 0.f; grad_sigmas[i] = 0.f;
        }
        if (stop) { done = true; continue; }
        T = __shfl_sync(0xffffffffu, T_after, 31);
        r = __shfl_sync(0xffffffffu, ri, 31);
        g = __shfl_sync(0xffffffffu, gi, 31);
        b = __shfl_sync(0xffffffffu, bi, 31);
    }
}

// Rows of the [M, *] sample buffers that no kept ray owns: [T, M) with T = offset of the first ray that does not fit
// (offset <= M < offset + count; the slots are allocated in ray order, so every later ray is dropped as well) or, when all rays
// fit, the total sample count.  The reference gets zeros there from zero-initialised buffers (raymarching.py:205-207, 283-284:
// about 190 MB of memset per step); here the few rows of the tail are cleared instead.  Up to three buffers of widths wa/wb/wc.
__global__ void __launch_bounds__(256)
k_zero_unowned_rows(const int32_t* __restrict__ rays, uint32_t N, uint32_t M, float* __restrict__ a, int wa, float* __restrict__ b, int wb,
                    float* __restrict__ c, int wc) {
    __shared__ uint32_t sT;
    if (threadIdx.x == 0) {
        uint32_t lo = 0, hi = N;     // first ray whose end exceeds M (ends are non-decreasing in ray order)
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            const uint32_t end = (uint32_t)rays[3 * (size_t)mid + 1] + (uint32_t)rays[3 * (size_t)mid + 2];
            if (end > M) hi = mid; else lo = mid + 1;
        }
        sT = lo < N ? (uint32_t)rays[3 * (size_t)lo + 1] : ((uint32_t)rays[3 * (size_t)(N - 1) + 1] + (uint32_t)rays[3 * (size_t)(N - 1) + 2]);
    }
    __syncthreads();
    const uint32_t T = sT < M ? sT : M;
    for (uint32_t row = T + blockIdx.x * blockDim.x + threadIdx.x; row < M; row += gridDim.x * blockDim.x) {
        if (a) for (int j = 0; j < wa; ++j) a[(size_t)row * wa + j] = 0.f;
        if (b) for (int j = 0; j < wb; ++j) b[(size_t)row * wb + j] = 0.f;
        if (c) for (int j = 0; j < wc; ++j) c[(size_t)row * wc + j] = 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
// inference marching / compositing (reference :700-905)
// ------------------------------------------------------------------------------------------------
// one alive ray: up to n_step samples into rows [n*n_step, (n+1)*n_step) of xyzs / dirs / deltas.  zero_tail: clear the rows
// the ray does not reach (the host-driven loop passes freshly zeroed buffers instead, as the reference does).
__device__ __forceinline__ void march_rays_one(uint32_t n, uint32_t n_step, const int32_t* __restrict__ rays_alive,
                                               const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                                               const float* __restrict__ rays_d, float bound, float dt_gamma, uint32_t max_steps,
                                               uint32_t C, uint32_t H, const uint8_t* __restrict__ grid,
                                               const float* __restrict__ fars, float* __restrict__ xyzs, float* __restrict__ dirs,
                                               float* __restrict__ deltas, const float* __restrict__ noises, bool zero_tail) {
    const int32_t index = rays_alive[n];
    const MarchParams p = make_params(bound, dt_gamma, max_steps, C, H, grid);
    const MarchRay r = load_ray(rays_o + 3 * (size_t)index, rays_d + 3 * (size_t)index);
    const float far = fars[index];
    float t = rays_t[index];
    if (noises != nullptr) t = __fmaf_rn(clampf(__fmul_rn(t, dt_gamma), p.dt_min, p.dt_max), noises[n], t);
    float last_t = t;
    float* px = xyzs + 3 * (size_t)n * n_step;
    float* pd = dirs + 3 * (size_t)n * n_step;
    float* pl = deltas + 2 * (size_t)n * n_step;
    uint32_t step = 0;
    float x, y, z, dt;
    while (t < far && step < n_step) {
        if (march_probe(p, r, t, x, y, z, dt)) {
            px[0] = x; px[1] = y; px[2] = z;
            pd[0] = r.dx; pd[1] = r.dy; pd[2] = r.dz;
            t = __fadd_rn(t, dt);
            pl[0] = dt;
            pl[1] = __fsub_rn(t, last_t);
            last_t = t;
            px += 3; pd += 3; pl += 2;
            ++step;
        }
    }
    if (zero_tail)
        for (; step < n_step; ++step) {
            px[0] = 0.f; px[1] = 0.f; px[2] = 0.f;
            pd[0] = 0.f; pd[1] = 0.f; pd[2] = 0.f;
            pl[0] = 0.f; pl[1] = 0.f;
            px += 3; pd += 3; pl += 2;
        }
}

__global__ void k_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* __restrict__ rays_alive,
                             const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                             const float* __restrict__ rays_d, float bound, float dt_gamma, uint32_t max_steps,
                             uint32_t C, uint32_t H, const uint8_t* __restrict__ grid, const float* __restrict__ fars,
                             float* __restrict__ xyzs, float* __restrict__ dirs, float* __restrict__ deltas,
                             const float* __restrict__ noises) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_alive) return;
    march_rays_one(n, n_step, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C, H, grid, fars, xyzs, dirs, deltas,
                   noises, false);
}

__device__ __forceinline__ void composite_rays_one(uint32_t n, uint32_t n_step, float T_thresh, int32_t* __restrict__ rays_alive,
                                                   float* __restrict__ rays_t, const float* __restrict__ sigmas,
                                                   const float* __restrict__ rgbs, const float* __restrict__ deltas,
                                                   float* __restrict__ weights_sum, float* __restrict__ depth,
                                                   float* __restrict__ image) {
    const int32_t index = rays_alive[n];
    const float* s = sigmas + (size_t)n * n_step;
    const float* c = rgbs + 3 * (size_t)n * n_step;
    const float* dl = deltas + 2 * (size_t)n * n_step;
    float t = rays_t[index], ws = weights_sum[index], d = depth[index];
    float r = image[3 * (size_t)index], g = image[3 * (size_t)index + 1], b = image[3 * (size_t)index + 2];
    uint32_t step = 0;
    while (step < n_step) {
        if (dl[2 * step] == 0) break;  // terminated ray (padding)
        const float alpha = 1.0f - __expf(-s[step] * dl[2 * step]);
        const float T = 1 - ws;
        const float w = alpha * T;
        ws += w;
        t += dl[2 * step + 1];
        d += w * t;
        r += w * c[3 * step];
        g += w * c[3 * step + 1];
        b += w * c[3 * step + 2];
        if (T < T_thresh) break;
        ++step;
    }
    if (step < n_step) rays_alive[n] = -1; else rays_t[index] = t;
    weights_sum[index] = ws;
    depth[index] = d;
    image[3 * (size_t)index] = r;
    image[3 * (size_t)index + 1] = g;
    image[3 * (size_t)index + 2] = b;
}

__global__ void k_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* __restrict__ rays_alive,
                                 float* __restrict__ rays_t, const float* __restrict__ sigmas,
                                 const float* __restrict__ rgbs, const float* __restrict__ deltas,
                                 float* __restrict__ weights_sum, float* __restrict__ depth, float* __restrict__ image) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_alive) return;
    composite_rays_one(n, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image);
}

// ------------------------------------------------------------------------------------------------
// device-driven inference loop (SURVEY.md 8f-3): the loop state of renderer.py:342-368 lives in `ctrl` on the device, so the
// host can issue several iterations without reading anything back.
//   ctrl[0] n_alive   rays in the current alive list            ctrl[1] n_step   samples per ray this iteration (0 = finished)
//   ctrl[2] step      samples per ray marched so far            ctrl[3] n_rows   n_alive * n_step = valid rows of this iteration
//   ctrl[4] iterations that did work                            ctrl[6] n_next   survivors left by the last compaction
// k_infer_plan is the only writer of ctrl[0..4]; the compaction writes ctrl[6].
// ------------------------------------------------------------------------------------------------
enum { kCtlAlive = 0, kCtlStep = 1, kCtlMarched = 2, kCtlRows = 3, kCtlIters = 4, kCtlNext = 6 };

__global__ void k_infer_plan(int32_t* __restrict__ ctrl, uint32_t N, uint32_t max_steps) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int32_t n_alive = ctrl[kCtlNext];
    const int32_t marched = ctrl[kCtlMarched];
    int32_t n_step = 0;
    if (n_alive > 0 && (uint32_t)marched < max_steps) {      // renderer.py:342-352
        n_step = (int32_t)(N / (uint32_t)n_alive);
        n_step = n_step > 8 ? 8 : (n_step < 1 ? 1 : n_step);
    }
    ctrl[kCtlAlive] = n_alive;
    ctrl[kCtlStep] = n_step;
    ctrl[kCtlRows] = n_alive * n_step;
    if (n_step > 0) {
        ctrl[kCtlMarched] = marched + n_step;                   // renderer.py:368
        ctrl[kCtlIters] += 1;
    }
}

__global__ void k_march_rays_dev(const int32_t* __restrict__ ctrl, const int32_t* __restrict__ rays_alive,
                                 const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                                 const float* __restrict__ rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                                 uint32_t H, const uint8_t* __restrict__ grid, const float* __restrict__ fars,
                                 float* __restrict__ xyzs, float* __restrict__ dirs, float* __restrict__ deltas,
                                 const float* __restrict__ noises) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_alive = (uint32_t)ctrl[kCtlAlive], n_step = (uint32_t)ctrl[kCtlStep];
    if (n_step == 0 || n >= n_alive) return;
    march_rays_one(n, n_step, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C, H, grid, fars, xyzs, dirs, deltas,
                   noises, true);
}

__global__ void k_composite_rays_dev(const int32_t* __restrict__ ctrl, float T_thresh, int32_t* __restrict__ rays_alive,
                                     float* __restrict__ rays_t, const float* __restrict__ sigmas, const float* __restrict__ rgbs,
                                     const float* __restrict__ deltas, float* __restrict__ weights_sum, float* __restrict__ depth,
                                     float* __restrict__ image) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_alive = (uint32_t)ctrl[kCtlAlive], n_step = (uint32_t)ctrl[kCtlStep];
    if (n_step == 0 || n >= n_alive) return;
    composite_rays_one(n, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image);
}

// compaction with the element count read from ctrl; grids are sized by the caller's upper bound `cap`.  A finished
// iteration (n_step == 0) leaves the list and ctrl[6] untouched.
__global__ void k_compact_sums_dev(const int32_t* __restrict__ ctrl, const int32_t* __restrict__ alive,
                                   uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t sm[33];
    const uint32_t n = ctrl[kCtlStep] > 0 ? (uint32_t)ctrl[kCtlAlive] : 0u;
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t total;
    block_exclusive_scan(scan_value<1>(alive, i, n, 1), &total, sm);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void k_compact_scan_dev(int32_t* __restrict__ ctrl, uint32_t* __restrict__ block_sums, uint32_t nblocks) {
    __shared__ uint32_t sm[33];
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nblocks; base += kScanThreads) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? block_sums[i] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_scan(v, &total, sm);
        if (i < nblocks) block_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0 && ctrl[kCtlStep] > 0) ctrl[kCtlNext] = (int32_t)carry;
}

__global__ void k_compact_scatter_dev(const int32_t* __restrict__ ctrl, const int32_t* __restrict__ alive,
                                      const uint32_t* __restrict__ block_sums, int32_t* __restrict__ out) {
    __shared__ uint32_t sm[33];
    const uint32_t n = ctrl[kCtlStep] > 0 ? (uint32_t)ctrl[kCtlAlive] : 0u;
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    const uint32_t f = scan_value<1>(alive, i, n, 1);
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(f, &total, sm);
    if (f) out[block_sums[blockIdx.x] + ex] = alive[i];
}

// ------------------------------------------------------------------------------------------------
// ray gradient of the training march (tnl_rays_backward): with every sample's t held fixed, xyz_k = clamp(o + t_k d) and
// dirs_k = d, so  g_o = sum_k mask_k g_xyz_k  and  g_d = sum_k t_k mask_k g_xyz_k + sum_k g_dirs_k  (mask: o + t_k d inside
// [-bound, bound] per component, borders included, as torch.clamp's backward).  One warp per ray: lane l adds the rows
// l, l + 32, ... in that order, then a fixed xor tree sums the lanes -- no atomics, the same bits on every run.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_rays_backward(const int32_t* __restrict__ rays, const float* __restrict__ ts, const float* __restrict__ rays_o,
                const float* __restrict__ rays_d, float bound, const float* __restrict__ g_xyz, const float* __restrict__ g_dirs,
                const int32_t* __restrict__ n_valid, uint32_t N, uint32_t M, float* __restrict__ g_rays_o,
                float* __restrict__ g_rays_d) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t index = (uint32_t)rays[3 * (size_t)n];
    const uint32_t offset = (uint32_t)rays[3 * (size_t)n + 1];
    const uint32_t num = (uint32_t)rays[3 * (size_t)n + 2];
    float go[3] = {0.f, 0.f, 0.f}, gd[3] = {0.f, 0.f, 0.f};
    if (num != 0 && offset + num <= M) {   // dropped rays (overflowing M) contribute nothing
        uint32_t end = offset + num;
        if (n_valid) {
            const int32_t nv = *n_valid;
            const uint32_t v = nv < 0 ? 0u : (uint32_t)nv;
            end = end < v ? end : v;
        }
        const float o[3] = {rays_o[3 * (size_t)n], rays_o[3 * (size_t)n + 1], rays_o[3 * (size_t)n + 2]};
        const float d[3] = {rays_d[3 * (size_t)n], rays_d[3 * (size_t)n + 1], rays_d[3 * (size_t)n + 2]};
        for (uint32_t i = offset + lane; i < end; i += 32) {
            // all loads first, independent of the mask: one memory round trip per iteration instead of two dependent ones
            const float t = __ldg(ts + i);
            float gx[3], gv[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                gx[a] = g_xyz ? __ldg(g_xyz + 3 * (size_t)i + a) : 0.f;
                gv[a] = g_dirs ? __ldg(g_dirs + 3 * (size_t)i + a) : 0.f;
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float u = __fmaf_rn(t, d[a], o[a]);          // the march's own unclamped coordinate
                if (g_xyz && u >= -bound && u <= bound) {
                    go[a] = __fadd_rn(go[a], gx[a]);
                    gd[a] = __fmaf_rn(t, gx[a], gd[a]);
                }
                if (g_dirs) gd[a] = __fadd_rn(gd[a], gv[a]);
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        go[a] = warp_sum(go[a]);
        gd[a] = warp_sum(gd[a]);
    }
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            g_rays_o[3 * (size_t)index + a] = go[a];
            g_rays_d[3 * (size_t)index + a] = gd[a];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// SH basis, degree <= 4 (shencoder.cu:50-68)
// ------------------------------------------------------------------------------------------------
__global__ void k_sh_encode(const float* __restrict__ inputs, float* __restrict__ outputs, uint32_t B, uint32_t degree) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float x = inputs[3 * (size_t)b], y = inputs[3 * (size_t)b + 1], z = inputs[3 * (size_t)b + 2];
    float* o = outputs + (size_t)b * degree * degree;
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    o[0] = 0.28209479177387814f;
    if (degree <= 1) return;
    o[1] = -0.48860251190291987f * y;
    o[2] = 0.48860251190291987f * z;
    o[3] = -0.48860251190291987f * x;
    if (degree <= 2) return;
    o[4] = 1.0925484305920792f * xy;
    o[5] = -1.0925484305920792f * yz;
    o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
    o[7] = -1.0925484305920792f * xz;
    o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
    if (degree <= 3) return;
    o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2);
    o[10] = 2.8906114426405538f * xy * z;
    o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
    o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
    o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
    o[14] = 1.4453057213202769f * z * (x2 - y2);
    o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
}

// input gradient of k_sh_encode: grad_inputs[b] = sum_ch grad[b][ch] d o[ch] / d inputs[b] (the reference's kernel_sh_backward)
template <int NCH>
__global__ void k_sh_encode_backward(const float* __restrict__ grad, const float* __restrict__ inputs, uint32_t B,
                                     float* __restrict__ grad_inputs) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float gd[3];
    sh_backward<NCH>(inputs[3 * (size_t)b], inputs[3 * (size_t)b + 1], inputs[3 * (size_t)b + 2], grad + (size_t)b * NCH, gd);
#pragma unroll
    for (int a = 0; a < 3; ++a) grad_inputs[3 * (size_t)b + a] = gd[a];
}

}  // namespace tnl

// ================================================================================================
// C ABI
// ================================================================================================
using namespace tnl;
static inline cudaStream_t S(tnl_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static constexpr uint32_t kT = 128;

extern "C" {

int tnl_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N, float min_near,
                           float* nears, float* fars, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(rays_o && rays_d && aabb && nears && fars, "null pointer");
    k_near_far<<<ceil_div(N, kT), kT, 0, S(stream)>>>(rays_o, rays_d, aabb, N, min_near, nears, fars);
    return finish_launch("near_far_from_aabb");
}

int tnl_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                     tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(rays_o && rays_d && coords, "null pointer");
    k_sph_from_ray<<<ceil_div(N, kT), kT, 0, S(stream)>>>(rays_o, rays_d, radius, N, coords);
    return finish_launch("sph_from_ray");
}

int tnl_morton3d(const int32_t* coords, uint32_t N, int32_t* indices, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(coords && indices, "null pointer");
    k_morton3d<<<ceil_div(N, 256u), 256, 0, S(stream)>>>(coords, N, indices);
    return finish_launch("morton3d");
}

int tnl_morton3d_invert(const int32_t* indices, uint32_t N, int32_t* coords, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(coords && indices, "null pointer");
    k_morton3d_invert<<<ceil_div(N, 256u), 256, 0, S(stream)>>>(indices, N, coords);
    return finish_launch("morton3d_invert");
}

int tnl_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(grid && bitfield, "null pointer");
    TNL_ARG_CHECK((reinterpret_cast<uintptr_t>(grid) & 15) == 0 && (reinterpret_cast<uintptr_t>(bitfield) & 3) == 0,
                  "grid must be 16-byte aligned, bitfield 4-byte aligned");
    const uint32_t nthreads = N / 4 + 1;
    k_packbits<<<ceil_div(nthreads, 256u), 256, 0, S(stream)>>>(grid, N, density_thresh, bitfield);
    return finish_launch("packbits");
}

size_t tnl_march_rays_train_workspace(uint32_t N) { return sizeof(uint32_t) * (ceil_div(N, (uint32_t)kScanThreads) + 1); }

// with room for one float per (ray, step) the second traversal is replaced by k_march_train_emit
static size_t march_scan_bytes(uint32_t N) { return (tnl_march_rays_train_workspace(N) + 255) & ~(size_t)255; }
size_t tnl_march_rays_train_workspace_fast(uint32_t N, uint32_t max_steps) {
    return march_scan_bytes(N) + sizeof(float) * (size_t)N * max_steps;
}

// ts_out == nullptr: tnl_march_rays_train; else also the ray parameter of every row (tnl_march_rays_train_ts)
static int march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                            uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* nears,
                            const float* fars, float* xyzs, float* dirs, float* deltas, int32_t* rays, int32_t* counter,
                            const float* noises, void* workspace, size_t workspace_bytes, float* ts_out, tnl_stream_t stream) {
    uint32_t* block_sums = static_cast<uint32_t*>(workspace);
    const uint32_t nb = ceil_div(N, (uint32_t)kScanThreads);
    const bool fast = M > 0 && workspace_bytes >= tnl_march_rays_train_workspace_fast(N, max_steps);
    float* ts = fast ? reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + march_scan_bytes(N)) : nullptr;
    k_march_train_count<<<ceil_div(N, kT), kT, 0, S(stream)>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H,
                                                                nears, fars, noises, rays, ts);
    k_scan_block_sums<0><<<nb, kScanThreads, 0, S(stream)>>>(rays + 2, N, 3, block_sums);
    k_scan_of_sums<<<1, kScanThreads, 0, S(stream)>>>(block_sums, nb, counter, N, nullptr);
    k_scan_offsets<<<nb, kScanThreads, 0, S(stream)>>>(rays + 2, N, 3, block_sums, rays + 1);
    if (M > 0) {
        if (fast && ts_out)
            k_march_train_emit_ts<<<ceil_div(N, 8u), 256, 0, S(stream)>>>(rays_o, rays_d, bound, dt_gamma, max_steps, N, C, H, M, nears,
                                                                          noises, rays, ts, xyzs, dirs, deltas, ts_out);
        else if (fast)
            k_march_train_emit<<<ceil_div(N, 8u), 256, 0, S(stream)>>>(rays_o, rays_d, bound, dt_gamma, max_steps, N, C, H, M, nears, noises,
                                                                       rays, ts, xyzs, dirs, deltas);
        else if (ts_out)
            k_march_train_write_ts<<<ceil_div(N, kT), kT, 0, S(stream)>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M,
                                                                           nears, fars, noises, rays, xyzs, dirs, deltas, ts_out);
        else
            k_march_train_write<<<ceil_div(N, kT), kT, 0, S(stream)>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N,
                                                                        C, H, M, nears, fars, noises, rays, xyzs, dirs, deltas);
        // rows no kept ray owns are zeros, as in the reference's zero-initialised buffers: the caller may pass uninitialised memory
        k_zero_unowned_rows<<<32, 256, 0, S(stream)>>>(rays, N, M, xyzs, 3, dirs, 3, deltas, 2);
        if (ts_out) k_zero_unowned_rows<<<32, 256, 0, S(stream)>>>(rays, N, M, ts_out, 1, nullptr, 0, nullptr, 0);
    }
    return finish_launch(ts_out ? "march_rays_train_ts" : "march_rays_train");
}

#define TNL_MARCH_TRAIN_CHECKS(what)                                                                                            \
    TNL_ARG_CHECK(rays_o && rays_d && grid && nears && fars && rays && counter && noises, "null pointer");                     \
    TNL_ARG_CHECK(M == 0 || (xyzs && dirs && deltas), "null output");                                                          \
    TNL_ARG_CHECK(C >= 1 && C <= 8 && H >= 2 && H <= 1024 && max_steps >= 1, "unsupported cascade / grid size");              \
    if (workspace == nullptr || workspace_bytes < tnl_march_rays_train_workspace(N)) {                                          \
        set_error(what ": workspace too small");                                                                                \
        return TNL_ERR_WORKSPACE;                                                                                               \
    }

int tnl_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                         uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* nears,
                         const float* fars, float* xyzs, float* dirs, float* deltas, int32_t* rays, int32_t* counter,
                         const float* noises, void* workspace, size_t workspace_bytes, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_MARCH_TRAIN_CHECKS("march_rays_train");
    return march_rays_train(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, xyzs, dirs, deltas, rays,
                            counter, noises, workspace, workspace_bytes, nullptr, stream);
}

int tnl_march_rays_train_ts(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                            uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* nears,
                            const float* fars, float* xyzs, float* dirs, float* deltas, float* ts, int32_t* rays,
                            int32_t* counter, const float* noises, void* workspace, size_t workspace_bytes, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_MARCH_TRAIN_CHECKS("march_rays_train_ts");
    TNL_ARG_CHECK(M == 0 || ts, "null output");
    return march_rays_train(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, xyzs, dirs, deltas, rays,
                            counter, noises, workspace, workspace_bytes, M > 0 ? ts : nullptr, stream);
}

int tnl_rays_backward(const int32_t* rays, const float* ts, const float* rays_o, const float* rays_d, float bound,
                      const float* g_xyz, const float* g_dirs, const int32_t* n_valid, uint32_t N, uint32_t M, float* g_rays_o,
                      float* g_rays_d, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(rays && rays_o && rays_d && g_rays_o && g_rays_d, "null pointer");
    TNL_ARG_CHECK(M == 0 || ts, "null ts");
    TNL_ARG_CHECK(bound > 0.f, "bound must be positive");
    k_rays_backward<<<ceil_div(N, 8u), 256, 0, S(stream)>>>(rays, ts, rays_o, rays_d, bound, M ? g_xyz : nullptr,
                                                             M ? g_dirs : nullptr, n_valid, N, M, g_rays_o, g_rays_d);
    return finish_launch("rays_backward");
}

int tnl_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas, const int32_t* rays,
                                     uint32_t M, uint32_t N, float T_thresh, float* weights_sum, float* depth,
                                     float* image, tnl_stream_t stream) {
    if (N == 0) return 0;
    TNL_ARG_CHECK(rays && weights_sum && depth && image, "null pointer");
    TNL_ARG_CHECK(M == 0 || (sigmas && rgbs && deltas), "null input");
    TNL_ARG_CHECK(((uintptr_t)deltas & 7) == 0, "deltas must be 8-byte aligned");
    k_composite_train_fwd<<<ceil_div(N, 8u), 256, 0, S(stream)>>>(sigmas, rgbs, deltas, rays, M, N, T_thresh, weights_sum,
                                                                   depth, image);
    return finish_launch("composite_rays_train_forward");
}

int tnl_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image, const float* sigmas,
                                      const float* rgbs, const float* deltas, const int32_t* rays,
                                      const float* weights_sum, const float* image, uint32_t M, uint32_t N,
                                      float T_thresh, float* grad_sigmas, float* grad_rgbs, tnl_stream_t stream) {
    if (N == 0 || M == 0) return 0;
    TNL_ARG_CHECK(grad_weights_sum && grad_image && sigmas && rgbs && deltas && rays && weights_sum && image &&
                      grad_sigmas && grad_rgbs, "null pointer");
    k_composite_train_bwd<<<ceil_div(N, 8u), 256, 0, S(stream)>>>(grad_weights_sum, grad_image, sigmas, rgbs, deltas, rays,
                                                                   weights_sum, image, M, N, T_thresh, grad_sigmas, grad_rgbs);
    // every row a kept ray owns has been written (zeros past the ray's termination); the rest of the buffers: the unowned tail
    k_zero_unowned_rows<<<32, 256, 0, S(stream)>>>(rays, N, M, grad_sigmas, 1, grad_rgbs, 3, nullptr, 0);
    return finish_launch("composite_rays_train_backward");
}

int tnl_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                   const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                   uint32_t H, const uint8_t* grid, const float* nears, const float* fars, float* xyzs, float* dirs,
                   float* deltas, const float* noises, tnl_stream_t stream) {
    (void)nears;
    if (n_alive == 0 || n_step == 0) return 0;
    TNL_ARG_CHECK(rays_alive && rays_t && rays_o && rays_d && grid && fars && xyzs && dirs && deltas && noises,
                  "null pointer");
    TNL_ARG_CHECK(C >= 1 && C <= 8 && H >= 2 && H <= 1024 && max_steps >= 1, "unsupported cascade / grid size");
    k_march_rays<<<ceil_div(n_alive, kT), kT, 0, S(stream)>>>(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound,
                                                               dt_gamma, max_steps, C, H, grid, fars, xyzs, dirs, deltas,
                                                               noises);
    return finish_launch("march_rays");
}

int tnl_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive, float* rays_t,
                       const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum, float* depth,
                       float* image, tnl_stream_t stream) {
    if (n_alive == 0 || n_step == 0) return 0;
    TNL_ARG_CHECK(rays_alive && rays_t && sigmas && rgbs && deltas && weights_sum && depth && image, "null pointer");
    k_composite_rays<<<ceil_div(n_alive, kT), kT, 0, S(stream)>>>(n_alive, n_step, T_thresh, rays_alive, rays_t, sigmas,
                                                                   rgbs, deltas, weights_sum, depth, image);
    return finish_launch("composite_rays");
}

int tnl_infer_plan(int32_t* ctrl, uint32_t N, uint32_t max_steps, tnl_stream_t stream) {
    TNL_ARG_CHECK(ctrl, "null pointer");
    TNL_ARG_CHECK(N >= 1 && max_steps >= 1, "N and max_steps must be positive");
    k_infer_plan<<<1, 32, 0, S(stream)>>>(ctrl, N, max_steps);
    return finish_launch("infer_plan");
}

int tnl_march_rays_dev(const int32_t* ctrl, uint32_t cap, const int32_t* rays_alive, const float* rays_t, const float* rays_o,
                       const float* rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                       const uint8_t* grid, const float* fars, float* xyzs, float* dirs, float* deltas, const float* noises,
                       tnl_stream_t stream) {
    if (cap == 0) return 0;
    TNL_ARG_CHECK(ctrl && rays_alive && rays_t && rays_o && rays_d && grid && fars && xyzs && dirs && deltas, "null pointer");
    TNL_ARG_CHECK(C >= 1 && C <= 8 && H >= 2 && H <= 1024 && max_steps >= 1, "unsupported cascade / grid size");
    k_march_rays_dev<<<ceil_div(cap, kT), kT, 0, S(stream)>>>(ctrl, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C,
                                                              H, grid, fars, xyzs, dirs, deltas, noises);
    return finish_launch("march_rays_dev");
}

int tnl_composite_rays_dev(const int32_t* ctrl, uint32_t cap, float T_thresh, int32_t* rays_alive, float* rays_t,
                           const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum, float* depth,
                           float* image, tnl_stream_t stream) {
    if (cap == 0) return 0;
    TNL_ARG_CHECK(ctrl && rays_alive && rays_t && sigmas && rgbs && deltas && weights_sum && depth && image, "null pointer");
    k_composite_rays_dev<<<ceil_div(cap, kT), kT, 0, S(stream)>>>(ctrl, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas,
                                                                  weights_sum, depth, image);
    return finish_launch("composite_rays_dev");
}

int tnl_compact_alive_dev(int32_t* ctrl, uint32_t cap, const int32_t* alive, int32_t* out, void* workspace,
                          size_t workspace_bytes, tnl_stream_t stream) {
    if (cap == 0) return 0;
    TNL_ARG_CHECK(ctrl && alive && out, "null pointer");
    if (workspace == nullptr || workspace_bytes < tnl_compact_alive_workspace(cap)) {
        set_error("compact_alive_dev: workspace too small");
        return TNL_ERR_WORKSPACE;
    }
    uint32_t* block_sums = static_cast<uint32_t*>(workspace);
    const uint32_t nb = ceil_div(cap, (uint32_t)kScanThreads);
    k_compact_sums_dev<<<nb, kScanThreads, 0, S(stream)>>>(ctrl, alive, block_sums);
    k_compact_scan_dev<<<1, kScanThreads, 0, S(stream)>>>(ctrl, block_sums, nb);
    k_compact_scatter_dev<<<nb, kScanThreads, 0, S(stream)>>>(ctrl, alive, block_sums, out);
    return finish_launch("compact_alive_dev");
}

size_t tnl_compact_alive_workspace(uint32_t n) { return sizeof(uint32_t) * (ceil_div(n, (uint32_t)kScanThreads) + 1); }

int tnl_compact_alive(const int32_t* alive, uint32_t n, int32_t* out, int32_t* n_out_dev, void* workspace,
                      size_t workspace_bytes, tnl_stream_t stream) {
    TNL_ARG_CHECK(n_out_dev, "null pointer");
    if (n == 0) {
        cudaMemsetAsync(n_out_dev, 0, sizeof(int32_t), S(stream));
        return finish_launch("compact_alive");
    }
    TNL_ARG_CHECK(alive && out, "null pointer");
    if (workspace == nullptr || workspace_bytes < tnl_compact_alive_workspace(n)) {
        set_error("compact_alive: workspace too small");
        return TNL_ERR_WORKSPACE;
    }
    uint32_t* block_sums = static_cast<uint32_t*>(workspace);
    const uint32_t nb = ceil_div(n, (uint32_t)kScanThreads);
    k_scan_block_sums<1><<<nb, kScanThreads, 0, S(stream)>>>(alive, n, 1, block_sums);
    k_scan_of_sums<<<1, kScanThreads, 0, S(stream)>>>(block_sums, nb, nullptr, n, n_out_dev);
    k_compact_scatter<<<nb, kScanThreads, 0, S(stream)>>>(alive, n, block_sums, out);
    return finish_launch("compact_alive");
}

int tnl_sh_encode_forward(const float* inputs, float* outputs, uint32_t B, uint32_t degree, tnl_stream_t stream) {
    if (B == 0) return 0;
    TNL_ARG_CHECK(inputs && outputs, "null pointer");
    if (degree < 1 || degree > 4) {
        set_error("sh_encode_forward: only degree 1..4 is on the hot path (reference uses 4)");
        return TNL_ERR_UNSUPPORTED;
    }
    k_sh_encode<<<ceil_div(B, 256u), 256, 0, S(stream)>>>(inputs, outputs, B, degree);
    return finish_launch("sh_encode_forward");
}

int tnl_sh_encode_backward(const float* grad, const float* inputs, uint32_t B, uint32_t degree, float* grad_inputs,
                           tnl_stream_t stream) {
    if (B == 0) return 0;
    TNL_ARG_CHECK(grad && inputs && grad_inputs, "null pointer");
    TNL_ARG_CHECK(degree >= 1 && degree <= 4, "sh_encode_backward: degree must be 1..4");
    const unsigned blocks = ceil_div(B, 256u);
    if (degree == 1) k_sh_encode_backward<1><<<blocks, 256, 0, S(stream)>>>(grad, inputs, B, grad_inputs);
    else if (degree == 2) k_sh_encode_backward<4><<<blocks, 256, 0, S(stream)>>>(grad, inputs, B, grad_inputs);
    else if (degree == 3) k_sh_encode_backward<9><<<blocks, 256, 0, S(stream)>>>(grad, inputs, B, grad_inputs);
    else k_sh_encode_backward<16><<<blocks, 256, 0, S(stream)>>>(grad, inputs, B, grad_inputs);
    return finish_launch("sh_encode_backward");
}

}  // extern "C"
