// Marching cubes over a dense fp32 volume -- sm_100a.
//
// Input: u [nx][ny][nz] (C-contiguous; the reference's u[x, y, z]), threshold thr; a lattice point is inside iff u >= thr.
// Output, in an order that does not depend on the thread schedule:
//   vertices  float64 [V][3], one per lattice edge whose end values straddle thr, ordered by (linear index of the edge's
//             lower lattice point, axis x < y < z); position p + t * e_axis, t = (thr - u_a) / (u_b - u_a) in float64 from the
//             lower end a to the upper end b (t = 1 when u_a is infinite);
//   triangles int64 [T][3] vertex ids, ordered by (linear cube index, order of the case table mc_tables.cuh).
//
// Two passes over the lattice in blocks of kPts consecutive points (256 threads, 8 chunks of 256):
//   k_mc_count  per point: the crossing edges it owns (mask, 3 bits) and the triangles of the cube it is the lower corner of;
//               writes (block-local exclusive vertex prefix << 3 | mask) as uint16 per point and the block's two totals;
//   k_mc_scan   one block: exclusive 64-bit prefix of the block totals -> per-block vertex / triangle offsets + the grand totals;
//   k_mc_emit   per point: its vertices, and its cube's triangles, whose vertex ids it reads from the uint16 words of the up to
//               8 lattice points of the cube.
// The caller reads the two totals (one 16-byte copy), allocates the outputs and launches the emit.
#include "common.cuh"
#include "mc_tables.cuh"

namespace tnl {

constexpr int kMcThreads = 256;
constexpr int kMcChunks = 8;
constexpr uint32_t kPts = kMcThreads * kMcChunks;  // lattice points per block; 3 * kPts < 2^13 (uint16 word = prefix << 3 | mask)
constexpr int kScanThreads = 1024;

struct McOffset {
    unsigned long long v, t;   // vertices / triangles before the block
};

struct McGeom {
    uint64_t n;            // nx * ny * nz
    uint64_t sx, sy;       // strides of x and y (z is contiguous)
    uint32_t nx, ny, nz;
};

// offset of cube corner c = x + 2y + 4z from the cube's lower lattice point
__device__ __forceinline__ uint64_t mc_corner_offset(const McGeom& g, int c) {
    return (c & 1 ? g.sx : 0) + (c & 2 ? g.sy : 0) + (c & 4 ? 1 : 0);
}

__device__ __forceinline__ bool mc_inside(float v, double thr) { return (double)v >= thr; }

// exclusive scan over the 256 threads of the block; `sm` holds 8 words
__device__ __forceinline__ uint32_t mc_block_scan(uint32_t v, uint32_t* sm, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) sm[warp] = incl;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kMcThreads / 32; ++w) {
        const uint32_t s = sm[w];
        before += (w < warp) ? s : 0u;
        tot += s;
    }
    __syncthreads();  // sm is reused by the next call
    total = tot;
    return before + incl - v;
}

// Everything one lattice point contributes: crossing mask of the edges it owns (bit a: edge along axis a), the case of the cube
// it is the lower corner of (-1 if none), and whether u[p] is NaN.
struct McPoint {
    uint32_t x, y, z;
    uint32_t mask;
    int cube_case;
    bool nan;
};

__device__ __forceinline__ McPoint mc_point(const float* __restrict__ u, uint64_t L, const McGeom& g, double thr) {
    McPoint r;
    r.z = (uint32_t)(L % g.nz);
    const uint64_t xy = L / g.nz;
    r.y = (uint32_t)(xy % g.ny);
    r.x = (uint32_t)(xy / g.ny);
    const float u0 = __ldg(u + L);
    r.nan = isnan(u0);
    const bool in0 = mc_inside(u0, thr);
    const bool hx = r.x + 1 < g.nx, hy = r.y + 1 < g.ny, hz = r.z + 1 < g.nz;
    r.mask = 0;
    if (hx && mc_inside(__ldg(u + L + g.sx), thr) != in0) r.mask |= 1u;
    if (hy && mc_inside(__ldg(u + L + g.sy), thr) != in0) r.mask |= 2u;
    if (hz && mc_inside(__ldg(u + L + 1), thr) != in0) r.mask |= 4u;
    r.cube_case = -1;
    if (hx && hy && hz) {
        int c = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            c |= (int)mc_inside(__ldg(u + L + mc_corner_offset(g, k)), thr) << k;
        }
        r.cube_case = c;
    }
    return r;
}

__global__ void __launch_bounds__(kMcThreads) k_mc_count(const float* __restrict__ u, McGeom g, double thr,
                                                         uint16_t* __restrict__ words, uint2* __restrict__ block_counts) {
    __shared__ uint8_t ntri_s[256];
    __shared__ uint32_t sm[kMcThreads / 32];
    __shared__ int nan_s;
    ntri_s[threadIdx.x] = kMcTriCount[threadIdx.x];
    if (threadIdx.x == 0) nan_s = 0;
    __syncthreads();
    uint32_t carry_v = 0, carry_t = 0;
    const uint64_t base = (uint64_t)blockIdx.x * kPts;
    for (int c = 0; c < kMcChunks; ++c) {
        const uint64_t L = base + (uint64_t)c * kMcThreads + threadIdx.x;
        uint32_t nv = 0, nt = 0, mask = 0;
        if (L < g.n) {
            const McPoint p = mc_point(u, L, g, thr);
            if (p.nan) nan_s = 1;
            mask = p.mask;
            nv = __popc(mask);
            nt = p.cube_case >= 0 ? ntri_s[p.cube_case] : 0u;
        }
        uint32_t total;
        const uint32_t ex = mc_block_scan(nv | (nt << 16), sm, total);   // chunk sums: < 2^10 vertices, < 2^11 triangles
        if (L < g.n) words[L] = (uint16_t)(((carry_v + (ex & 0xffffu)) << 3) | mask);
        carry_v += total & 0xffffu;
        carry_t += total >> 16;
    }
    if (threadIdx.x == 0) block_counts[blockIdx.x] = make_uint2(nan_s ? 0xffffffffu : carry_v, carry_t);
}

// one block: offsets[b] = (vertices, triangles) before block b; totals = (V, T), or (-1, -1) if any block saw a NaN
__global__ void __launch_bounds__(kScanThreads) k_mc_scan(const uint2* __restrict__ block_counts, uint32_t nb,
                                                          McOffset* __restrict__ offsets, int64_t* __restrict__ totals) {
    __shared__ unsigned long long sv[kScanThreads], st[kScanThreads];
    __shared__ int nan_s;
    if (threadIdx.x == 0) nan_s = 0;
    const uint32_t per = ceil_div(nb, (uint32_t)kScanThreads);
    const uint32_t b0 = min(nb, threadIdx.x * per), b1 = min(nb, b0 + per);
    unsigned long long v = 0, t = 0;
    bool nan = false;
    for (uint32_t b = b0; b < b1; ++b) {
        const uint2 c = block_counts[b];
        nan |= c.x == 0xffffffffu;
        v += c.x;
        t += c.y;
    }
    sv[threadIdx.x] = v;
    st[threadIdx.x] = t;
    __syncthreads();
    if (nan) nan_s = 1;
    // Hillis-Steele inclusive scan of the per-thread sums
    for (int o = 1; o < kScanThreads; o <<= 1) {
        const unsigned long long av = threadIdx.x >= (unsigned)o ? sv[threadIdx.x - o] : 0ull;
        const unsigned long long at = threadIdx.x >= (unsigned)o ? st[threadIdx.x - o] : 0ull;
        __syncthreads();
        sv[threadIdx.x] += av;
        st[threadIdx.x] += at;
        __syncthreads();
    }
    unsigned long long ov = sv[threadIdx.x] - v, ot = st[threadIdx.x] - t;
    for (uint32_t b = b0; b < b1; ++b) {
        const uint2 c = block_counts[b];
        offsets[b] = McOffset{ov, ot};
        ov += c.x;
        ot += c.y;
    }
    if (threadIdx.x == kScanThreads - 1) {
        totals[0] = nan_s ? -1 : (int64_t)sv[threadIdx.x];
        totals[1] = nan_s ? -1 : (int64_t)st[threadIdx.x];
    }
}

__device__ __forceinline__ uint64_t mc_vertex_id(const uint16_t* __restrict__ words, const McOffset* __restrict__ offsets,
                                                 uint64_t L, int axis) {
    const uint32_t w = words[L];
    return offsets[L / kPts].v + (w >> 3) + __popc(w & ((1u << axis) - 1u));
}

__global__ void __launch_bounds__(kMcThreads) k_mc_emit(const float* __restrict__ u, McGeom g, double thr,
                                                        const uint16_t* __restrict__ words, const McOffset* __restrict__ offsets,
                                                        int64_t n_vertices, int64_t n_triangles, double* __restrict__ vertices,
                                                        int64_t* __restrict__ triangles) {
    __shared__ int8_t tab_s[256][16];
    __shared__ uint8_t ntri_s[256];
    __shared__ uint32_t sm[kMcThreads / 32];
#pragma unroll
    for (int k = 0; k < 16; ++k) tab_s[threadIdx.x][k] = kMcTriTable[threadIdx.x][k];
    ntri_s[threadIdx.x] = kMcTriCount[threadIdx.x];
    __syncthreads();
    uint64_t carry_t = offsets[blockIdx.x].t;
    const uint64_t base = (uint64_t)blockIdx.x * kPts;
    for (int c = 0; c < kMcChunks; ++c) {
        const uint64_t L = base + (uint64_t)c * kMcThreads + threadIdx.x;
        McPoint p{};
        p.cube_case = -1;
        if (L < g.n) p = mc_point(u, L, g, thr);
        const uint32_t nt = p.cube_case >= 0 ? ntri_s[p.cube_case] : 0u;
        uint32_t total;
        const uint32_t ex = mc_block_scan(nt, sm, total);
        if (L < g.n && p.mask) {
            uint64_t id = mc_vertex_id(words, offsets, L, 0);
            const double ua = (double)__ldg(u + L);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (!(p.mask & (1u << a))) continue;
                const double ub = (double)__ldg(u + L + mc_corner_offset(g, 1 << a));
                const double t = isinf(ua) ? 1.0 : (thr - ua) / (ub - ua);
                if (id < (uint64_t)n_vertices) {
                    double* v = vertices + 3 * id;
                    v[0] = (double)p.x + (a == 0 ? t : 0.0);
                    v[1] = (double)p.y + (a == 1 ? t : 0.0);
                    v[2] = (double)p.z + (a == 2 ? t : 0.0);
                }
                ++id;
            }
        }
        if (nt) {
            uint64_t tid = carry_t + ex;
            const int8_t* row = tab_s[p.cube_case];
            for (uint32_t i = 0; i < nt; ++i, ++tid) {
                if (tid >= (uint64_t)n_triangles) break;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int e = row[3 * i + k];
                    triangles[3 * tid + k] = (int64_t)mc_vertex_id(words, offsets, L + mc_corner_offset(g, kMcEdgeCorner[e]), e >> 2);
                }
            }
        }
        carry_t += total;
    }
}

bool mc_geom(uint32_t nx, uint32_t ny, uint32_t nz, McGeom& g, uint32_t& nb) {
    if (nx < 2 || ny < 2 || nz < 2) return false;
    g.nx = nx;
    g.ny = ny;
    g.nz = nz;
    g.sy = nz;
    g.sx = (uint64_t)ny * nz;
    g.n = g.sx * nx;
    nb = (uint32_t)ceil_div(g.n, (uint64_t)kPts);
    return true;
}

// workspace: [uint16 word per lattice point, padded to 16 B][uint2 counts per block, padded][McOffset per block]
size_t mc_words_bytes(const McGeom& g) { return (2 * g.n + 15) / 16 * 16; }
size_t mc_counts_bytes(uint32_t nb) { return ((size_t)nb * 8 + 15) / 16 * 16; }

}  // namespace tnl

using namespace tnl;

extern "C" {

size_t tnl_mc_workspace(uint32_t nx, uint32_t ny, uint32_t nz) {
    McGeom g;
    uint32_t nb;
    if (!mc_geom(nx, ny, nz, g, nb)) return 0;
    return mc_words_bytes(g) + mc_counts_bytes(nb) + (size_t)nb * 16;
}

int tnl_mc_count(const float* volume, uint32_t nx, uint32_t ny, uint32_t nz, double threshold, void* workspace,
                 size_t workspace_bytes, int64_t* totals, tnl_stream_t stream) {
    TNL_ARG_CHECK(volume && workspace && totals, "null pointer");
    McGeom g;
    uint32_t nb;
    TNL_ARG_CHECK(mc_geom(nx, ny, nz, g, nb), "the volume needs at least 2 points along each axis");
    TNL_ARG_CHECK(!isnan(threshold), "threshold is NaN");
    if (workspace_bytes < tnl_mc_workspace(nx, ny, nz)) {
        set_error("mc_count: workspace too small");
        return TNL_ERR_WORKSPACE;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint16_t* words = reinterpret_cast<uint16_t*>(ws);
    uint2* counts = reinterpret_cast<uint2*>(ws + mc_words_bytes(g));
    McOffset* offsets = reinterpret_cast<McOffset*>(ws + mc_words_bytes(g) + mc_counts_bytes(nb));
    k_mc_count<<<nb, kMcThreads, 0, s>>>(volume, g, threshold, words, counts);
    k_mc_scan<<<1, kScanThreads, 0, s>>>(counts, nb, offsets, totals);
    return finish_launch("mc_count");
}

int tnl_mc_emit(const float* volume, uint32_t nx, uint32_t ny, uint32_t nz, double threshold, const void* workspace,
                size_t workspace_bytes, int64_t n_vertices, int64_t n_triangles, double* vertices, int64_t* triangles,
                tnl_stream_t stream) {
    TNL_ARG_CHECK(n_vertices >= 0 && n_triangles >= 0, "the volume contains NaN (the count returned negative totals)");
    TNL_ARG_CHECK(volume && workspace, "null pointer");
    TNL_ARG_CHECK((vertices || n_vertices == 0) && (triangles || n_triangles == 0), "null pointer");
    McGeom g;
    uint32_t nb;
    TNL_ARG_CHECK(mc_geom(nx, ny, nz, g, nb), "the volume needs at least 2 points along each axis");
    TNL_ARG_CHECK(!isnan(threshold), "threshold is NaN");
    if (workspace_bytes < tnl_mc_workspace(nx, ny, nz)) {
        set_error("mc_emit: workspace too small");
        return TNL_ERR_WORKSPACE;
    }
    if (n_vertices == 0 && n_triangles == 0) return 0;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const uint8_t* ws = static_cast<const uint8_t*>(workspace);
    const uint16_t* words = reinterpret_cast<const uint16_t*>(ws);
    const McOffset* offsets = reinterpret_cast<const McOffset*>(ws + mc_words_bytes(g) + mc_counts_bytes(nb));
    k_mc_emit<<<nb, kMcThreads, 0, s>>>(volume, g, threshold, words, offsets, n_vertices, n_triangles, vertices, triangles);
    return finish_launch("mc_emit");
}

}  // extern "C"
