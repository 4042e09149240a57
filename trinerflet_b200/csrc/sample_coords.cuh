// Coordinate / tap arithmetic used by the plane-sampling kernels (sample.cu): everything
// that decides WHICH texels a point touches lives here, so that the binning and the samplers cannot disagree.
// Arithmetic follows ATen's grid_sampler_2d (unnormalise ((g+1)/2)*(R-1), clip to [0,R-1], weights nw/ne/sw/se as products
// of differences); see sample.cu for the behavioural contract.
#pragma once
#include "common.cuh"

namespace tnl {

struct Tap {
    int x0, y0;       // north-west texel
    float nw, ne, sw, se;
    bool x1ok, y1ok;  // south / east neighbours inside the plane
};

__device__ __forceinline__ float to_pixel(float g, int R) {
    float v = ((g + 1.0f) * 0.5f) * (float)(R - 1);
    return fminf((float)(R - 1), fmaxf(v, 0.0f));
}

// to_pixel plus d(pixel)/d(g): ATen's clip_coordinates_set_grad -- the derivative is (R-1)/2 strictly inside the plane and 0
// on or beyond its border (grid_sampler_2d_backward, padding_mode='border', align_corners=True).
__device__ __forceinline__ float to_pixel_grad(float g, int R, float& dg) {
    const float hi = (float)(R - 1);
    const float v = ((g + 1.0f) * 0.5f) * hi;
    if (!(v > 0.0f)) { dg = 0.0f; return 0.0f; }   // also NaN, which to_pixel maps to texel 0
    if (v >= hi) { dg = 0.0f; return hi; }
    dg = 0.5f * hi;
    return v;
}

__device__ __forceinline__ Tap make_tap(float gx, float gy, int R) {
    const float ix = to_pixel(gx, R), iy = to_pixel(gy, R);
    const float fx = floorf(ix), fy = floorf(iy);
    Tap t;
    t.x0 = (int)fx;
    t.y0 = (int)fy;
    const float ex = fx + 1.0f, ey = fy + 1.0f;  // south-east corner coordinates
    t.nw = (ex - ix) * (ey - iy);
    t.ne = (ix - fx) * (ey - iy);
    t.sw = (ex - ix) * (iy - fy);
    t.se = (ix - fx) * (iy - fy);
    t.x1ok = t.x0 + 1 <= R - 1;
    t.y1ok = t.y0 + 1 <= R - 1;
    return t;
}

// projected coordinate of a world coordinate x
__device__ __forceinline__ float project_coord(float x, float inv_bound, int fp16_coords) {
    float g = __fmul_rn(x, inv_bound);
    if (fp16_coords) g = __half2float(__float2half_rn(g));  // autocast rounds the projected coordinates to fp16 (triplane_encoder.py:299)
    return g;
}

// projected coordinate of point m on world axis a (0 = x, 1 = y, 2 = z)
__device__ __forceinline__ float axis_coord(const float* __restrict__ xyz, uint32_t m, int a, float inv_bound, int fp16_coords) {
    return project_coord(__ldg(xyz + 3 * (size_t)m + a), inv_bound, fp16_coords);
}

__device__ __forceinline__ void plane_coords(const float* __restrict__ xyz, uint32_t m, int p, float inv_bound,
                                             int fp16_coords, float& gx, float& gy) {
    const int a = (p == 2) ? 1 : 0;
    const int b = (p == 1) ? 1 : 2;
    gx = axis_coord(xyz, m, a, inv_bound, fp16_coords);
    gy = axis_coord(xyz, m, b, inv_bound, fp16_coords);
}

__device__ __forceinline__ uint2 pack4h(float4 v) {
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}
__device__ __forceinline__ float4 unpack4h(uint2 u) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

}  // namespace tnl
