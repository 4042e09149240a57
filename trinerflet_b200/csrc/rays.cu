// On-device step feeder (SURVEY.md 8f-2) -- sm_100a.  Replaces, for the per-step batch, the reference's
//   get_rays                       /root/reference/reconstruction/nerf/utils.py:64-149
//   shuffle_data / select_batch    nerf/utils.py:228-243   (index into the flattened [B*H*W] ray table)
//   the target gather of collate   nerf/provider.py:708-711
// The reference materialises rays_o / rays_d / images for ALL B*H*W rays (64 M rays = 1.5 GB + 0.77 GB for the Blender
// set), permutes the three tables on the host every epoch and copies a pageable slice to the device every step.  Here
// the poses (6.4 KB) and the images stay resident in HBM and a step's rays are generated from their flat ids.
#include "common.cuh"
#include "rays_core.cuh"

namespace tnl {

// thread <-> ray.  ids == nullptr: id = first_id + thread index (full frames, get_rays with N = -1).
template <int CI>
__global__ void k_rays_from_ids(const float* __restrict__ poses, RayIntrinsics k, uint32_t HW, uint32_t W,
                                const int64_t* __restrict__ ids, int64_t first_id, int64_t n_total, uint32_t n,
                                const float* __restrict__ images, float* __restrict__ rays_o, float* __restrict__ rays_d,
                                float* __restrict__ gt) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int64_t id = ids ? ids[t] : first_id + (int64_t)t;
    // out-of-range ids are clamped (the reference would raise an index error on the host; a kernel cannot)
    id = id < 0 ? 0 : (id >= n_total ? n_total - 1 : id);
    uint32_t img, pix;
    split_ray_id(id, HW, img, pix);
    float dir[3], o[3], d[3];
    pixel_direction(k, W, pix, dir);
    const float4* P4 = reinterpret_cast<const float4*>(poses + 16 * (size_t)img);
    const float4 r0 = __ldg(P4), r1 = __ldg(P4 + 1), r2 = __ldg(P4 + 2);
    const float pose[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
    ray_from_pose(pose, dir, o, d);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        rays_o[3 * (size_t)t + a] = o[a];
        rays_d[3 * (size_t)t + a] = d[a];
    }
    if (CI > 0) {
        const float* src = images + (size_t)id * CI;
#pragma unroll
        for (int c = 0; c < CI; ++c) gt[(size_t)t * CI + c] = __ldg(src + c);
    }
}


// Pose gradient of k_rays_from_ids (rays_d = R dir(pix), rays_o = pose[:3,3]): one CTA per image b scans the batch in a fixed
// order -- thread j takes the rays j, j + 256, ... (the whole batch for explicit ids, only the image's range for the implicit
// ones) -- and adds g_d[r] dir[c] into g_pose[b][r][c] and g_o[r] into g_pose[b][r][3]; a fixed shuffle tree and a warp-ordered
// sum finish the block.  No atomics: the same bits on every run.  The bottom row is 0; an image without rays gets 0.
constexpr int kPoseThreads = 256;

__global__ void __launch_bounds__(kPoseThreads)
k_rays_from_ids_backward(const float* __restrict__ g_rays_o, const float* __restrict__ g_rays_d, RayIntrinsics k, uint32_t HW,
                         uint32_t W, const int64_t* __restrict__ ids, int64_t first_id, int64_t n_total, uint32_t n,
                         float* __restrict__ g_poses) {
    __shared__ float part[kPoseThreads / 32][12];
    const uint32_t b = blockIdx.x;
    const int64_t lo = (int64_t)b * HW, hi = lo + HW;
    uint32_t t0 = 0, t1 = n;
    if (!ids) {     // id = first_id + t, in range (checked on the host): the image's rays are one contiguous slice
        const int64_t a = lo - first_id, e = hi - first_id;
        t0 = (uint32_t)(a < 0 ? 0 : (a > (int64_t)n ? (int64_t)n : a));
        t1 = (uint32_t)(e < 0 ? 0 : (e > (int64_t)n ? (int64_t)n : e));
    }
    float acc[12];
#pragma unroll
    for (int q = 0; q < 12; ++q) acc[q] = 0.f;
    for (uint32_t t = t0 + threadIdx.x; t < t1; t += kPoseThreads) {
        int64_t id = ids ? __ldg(ids + t) : first_id + (int64_t)t;
        id = id < 0 ? 0 : (id >= n_total ? n_total - 1 : id);   // the forward's clamp
        if (id < lo || id >= hi) continue;
        float dir[3];
        pixel_direction(k, W, (uint32_t)(id - lo), dir);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float gd = g_rays_d ? __ldg(g_rays_d + 3 * (size_t)t + r) : 0.f;
            const float go = g_rays_o ? __ldg(g_rays_o + 3 * (size_t)t + r) : 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) acc[4 * r + c] = __fmaf_rn(gd, dir[c], acc[4 * r + c]);
            acc[4 * r + 3] = __fadd_rn(acc[4 * r + 3], go);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 12; ++q) {
        const float v = warp_sum(acc[q]);
        if (lane == 0) part[warp][q] = v;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        const int q = threadIdx.x;
        float v = 0.f;
        if (q < 12)
            for (int w = 0; w < kPoseThreads / 32; ++w) v = __fadd_rn(v, part[w][q]);
        g_poses[16 * (size_t)b + q] = v;
    }
}

}  // namespace tnl

using namespace tnl;

extern "C" {

int tnl_rays_from_ids(const float* poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W,
                      const int64_t* ray_ids, int64_t first_id, uint32_t n, const float* images, uint32_t image_channels,
                      float* rays_o, float* rays_d, float* targets, tnl_stream_t stream) {
    if (n == 0) return 0;
    TNL_ARG_CHECK(poses && rays_o && rays_d, "null pointer");
    TNL_ARG_CHECK(B >= 1 && H >= 1 && W >= 1 && (uint64_t)H * W <= 0x7fffffffull, "bad image geometry");
    TNL_ARG_CHECK(fx != 0.f && fy != 0.f, "zero focal length");
    TNL_ARG_CHECK((images == nullptr) == (targets == nullptr), "images and targets must be given together");
    TNL_ARG_CHECK(images == nullptr || image_channels == 3 || image_channels == 4, "image_channels must be 3 or 4");
    TNL_ARG_CHECK((reinterpret_cast<uintptr_t>(poses) & 15) == 0, "poses must be 16-byte aligned");
    const uint32_t HW = H * W;
    const int64_t n_total = (int64_t)B * HW;
    TNL_ARG_CHECK(ray_ids || (first_id >= 0 && first_id + (int64_t)n <= n_total), "implicit id range outside the ray table");
    const RayIntrinsics k{fx, fy, cx, cy};
    const dim3 grid(ceil_div(n, 256u)), block(256);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const uint32_t ci = images ? image_channels : 0;
    if (ci == 0)
        k_rays_from_ids<0><<<grid, block, 0, s>>>(poses, k, HW, W, ray_ids, first_id, n_total, n, images, rays_o, rays_d, targets);
    else if (ci == 3)
        k_rays_from_ids<3><<<grid, block, 0, s>>>(poses, k, HW, W, ray_ids, first_id, n_total, n, images, rays_o, rays_d, targets);
    else
        k_rays_from_ids<4><<<grid, block, 0, s>>>(poses, k, HW, W, ray_ids, first_id, n_total, n, images, rays_o, rays_d, targets);
    return finish_launch("rays_from_ids");
}

int tnl_rays_from_ids_backward(const float* g_rays_o, const float* g_rays_d, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W, const int64_t* ray_ids, int64_t first_id, uint32_t n,
                               float* g_poses, tnl_stream_t stream) {
    TNL_ARG_CHECK(g_poses, "null pointer");
    TNL_ARG_CHECK(B >= 1 && H >= 1 && W >= 1 && (uint64_t)H * W <= 0x7fffffffull, "bad image geometry");
    TNL_ARG_CHECK(fx != 0.f && fy != 0.f, "zero focal length");
    const uint32_t HW = H * W;
    const int64_t n_total = (int64_t)B * HW;
    TNL_ARG_CHECK(ray_ids || (first_id >= 0 && first_id + (int64_t)n <= n_total), "implicit id range outside the ray table");
    const RayIntrinsics k{fx, fy, cx, cy};
    k_rays_from_ids_backward<<<B, kPoseThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(g_rays_o, g_rays_d, k, HW, W, ray_ids,
                                                                                              first_id, n_total, n, g_poses);
    return finish_launch("rays_from_ids_backward");
}

}  // extern "C"
