/* trinerflet_b200 -- C ABI of the B200-native (sm_100a) TriNeRFLet reconstruction hot path.
 *
 * Drop-in boundary for the native layer the reference reaches through pybind11/torch:
 *   aux_libs/raymarching/src/raymarching.h:7-18  (10 functions, at::Tensor args, outputs pre-allocated)
 *   aux_libs/shencoder/src/shencoder.h:9-10      (sh_encode_forward / backward)
 * plus the library calls the reference makes for the encoder and MLP heads
 *   pytorch_wavelets DWTInverse      (reconstruction/triplaneencoder/triplane_encoder.py:394)
 *   F.grid_sample                    (triplane_encoder.py:329)
 *   nn.Linear x5 / trunc_exp / sigmoid (reconstruction/nerf/network.py:118-147)
 *   GradScaler.step/update + Adam    (reconstruction/nerf/utils.py:1170-1173, reconstruction/main_nerf.py:119)
 * and a few entry points without a reference counterpart that the B200 design adds on the same path: the sample
 * visit order (tnl_cell_sort), the tile set a training step can touch and its exchange between GPUs
 * (tnl_mark_dirty_tiles, tnl_tiles_*), the work-list variants of the IDWT (tnl_idwt_level_*_sparse), and diagnostics
 * that pin the tcgen05 conventions on hardware (tnl_umma_*).
 *
 * Conventions (all entry points):
 *   - plain device pointers + explicit element counts, no torch types; every output buffer is
 *     allocated by the caller (same ownership rule as the reference, SURVEY.md 8b);
 *   - `stream` is the caller's CUDA stream (cudaStream_t passed as void*); kernels never allocate,
 *     never synchronise, keep no state between calls;
 *   - return value: 0 = launched ok, >0 = cudaError_t, <0 = TNL_ERR_*; tnl_last_error() gives text;
 *   - fp32 everywhere unless the name says otherwise; int32 index tensors as in the reference.
 *
 * Memory layouts of the encoder ("channels-last", see DESIGN.md):
 *   plane tensor   x   [3][n][n][C]        (logical reference shape [3,C,n,n], C fastest)
 *   detail coefs   yh  [3][3][n][n][C]     (logical reference shape [3,C,3,n,n])
 */
#ifndef TRINERFLET_B200_H
#define TRINERFLET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TNL_ABI_VERSION 1
#define TNL_ERR_INVALID_ARGUMENT (-1)
#define TNL_ERR_UNSUPPORTED (-2)
#define TNL_ERR_WORKSPACE (-3)

typedef void* tnl_stream_t; /* cudaStream_t */

int tnl_abi_version(void);
const char* tnl_last_error(void);

/* ------------------------------------------------------------------ ray utilities ---------- */
/* replaces near_far_from_aabb  (raymarching.h:7, raymarching.cu:148-156) */
int tnl_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                           float min_near, float* nears, float* fars, tnl_stream_t stream);
/* replaces sph_from_ray        (raymarching.h:8, raymarching.cu:201-209) */
int tnl_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                     tnl_stream_t stream);
/* replaces morton3D / morton3D_invert (raymarching.h:9-10, raymarching.cu:229-260) */
int tnl_morton3d(const int32_t* coords, uint32_t N, int32_t* indices, tnl_stream_t stream);
int tnl_morton3d_invert(const int32_t* indices, uint32_t N, int32_t* coords, tnl_stream_t stream);
/* replaces packbits            (raymarching.h:11, raymarching.cu:292-300); N = number of output bytes */
int tnl_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, tnl_stream_t stream);

/* ------------------------------------------------------------------ training march ---------- */
/* replaces march_rays_train    (raymarching.h:13, raymarching.cu:482-490).
 * Same outputs; sample slots are allocated by a deterministic exclusive scan in ray order instead
 * of the reference's atomicAdd race (raymarching.cu:405-406), so rays[n] = (n, offset_n, count_n).
 * counter[0] += total samples, counter[1] += N (as the reference's atomics leave them).
 * xyzs/dirs/deltas may be uninitialised: rows no kept ray owns are zero-filled by the call (the reference zero-initialises
 * the whole buffers, raymarching.py:205-207; rays are dropped, from the first that does not fit, when offset + count > M).
 * workspace: >= tnl_march_rays_train_workspace(N) bytes of device scratch. */
size_t tnl_march_rays_train_workspace(uint32_t N);
/* >= this many bytes of workspace (one float per ray and step on top of the scan scratch) let the call record every sample's ray
 * parameter during the counting traversal and emit the rows from it, warp per ray and coalesced, instead of traversing the
 * occupancy grid a second time; bit-identical outputs. */
size_t tnl_march_rays_train_workspace_fast(uint32_t N, uint32_t max_steps);
int tnl_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                         float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                         const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                         int32_t* rays, int32_t* counter, const float* noises, void* workspace,
                         size_t workspace_bytes, tnl_stream_t stream);
/* tnl_march_rays_train plus ts [M] (fp32, overwritten): the ray parameter t of every emitted row, so that
 * xyzs[i] == clamp(fmaf(ts[i], rays_d, rays_o), -bound, bound) bit for bit; rows no ray owns get 0.  Same arguments and
 * outputs otherwise (bit-identical); ts may be NULL only when M == 0. */
int tnl_march_rays_train_ts(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                            uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* nears,
                            const float* fars, float* xyzs, float* dirs, float* deltas, float* ts, int32_t* rays,
                            int32_t* counter, const float* noises, void* workspace, size_t workspace_bytes,
                            tnl_stream_t stream);
/* Ray gradient of the training march with every sample's t held fixed (xyz = clamp(o + t d), dirs = d):
 *   g_rays_o[n] = sum_k mask_k g_xyz_k,   g_rays_d[n] = sum_k t_k mask_k g_xyz_k + sum_k g_dirs_k
 * over the rows k of ray n (rays [N][3] and ts [M] from tnl_march_rays_train_ts), mask_k per component: the march's unclamped
 * coordinate fmaf(t, d, o) lies in [-bound, bound] (borders included, torch.clamp's backward).  g_xyz / g_dirs [M][3] fp32, either
 * may be NULL (zero).  Rays with no sample or dropped for overflowing M, and rows >= *n_valid (DEVICE int32, NULL = M), contribute
 * nothing.  g_rays_o / g_rays_d [N][3] are overwritten.  One warp per ray, fixed summation order: the same bits on every run. */
int tnl_rays_backward(const int32_t* rays, const float* ts, const float* rays_o, const float* rays_d, float bound,
                      const float* g_xyz, const float* g_dirs, const int32_t* n_valid, uint32_t N, uint32_t M, float* g_rays_o,
                      float* g_rays_d, tnl_stream_t stream);
/* replaces composite_rays_train_forward / _backward (raymarching.h:14-15, raymarching.cu:580-693).
 * backward: grad_sigmas / grad_rgbs may be uninitialised; every row is written (zeros past a ray's termination and in rows no
 * kept ray owns -- what the reference leaves untouched in its zero-initialised outputs, raymarching.py:283-284). */
int tnl_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                     const int32_t* rays, uint32_t M, uint32_t N, float T_thresh,
                                     float* weights_sum, float* depth, float* image, tnl_stream_t stream);
int tnl_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                      const float* sigmas, const float* rgbs, const float* deltas,
                                      const int32_t* rays, const float* weights_sum, const float* image,
                                      uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas,
                                      float* grad_rgbs, tnl_stream_t stream);

/* ------------------------------------------------------------------ inference march ---------- */
/* replaces march_rays / composite_rays (raymarching.h:17-18, raymarching.cu:808-914) */
int tnl_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                   const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps,
                   uint32_t C, uint32_t H, const uint8_t* grid, const float* nears, const float* fars,
                   float* xyzs, float* dirs, float* deltas, const float* noises, tnl_stream_t stream);
int tnl_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive, float* rays_t,
                       const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                       float* depth, float* image, tnl_stream_t stream);
/* on-device stream compaction of rays_alive (replaces the boolean-index + D2H sync at
 * reconstruction/nerf/renderer.py:364): out[0..n_out) = alive[i] for alive[i] >= 0, order kept;
 * *n_out_dev receives the count.  workspace >= tnl_compact_alive_workspace(n) bytes. */
size_t tnl_compact_alive_workspace(uint32_t n);
int tnl_compact_alive(const int32_t* alive, uint32_t n, int32_t* out, int32_t* n_out_dev, void* workspace,
                      size_t workspace_bytes, tnl_stream_t stream);

/* Device-driven inference loop (SURVEY.md 8f-3): the loop state of NeRFRenderer.run_cuda's eval branch
 * (reconstruction/nerf/renderer.py:342-368: n_alive, n_step = max(min(N // n_alive, 8), 1), step += n_step, the
 * boolean-index compaction) lives in `ctrl` (device int32[8]) so that the host can issue several iterations back to back
 * and read the state only now and then (the reference synchronises once per iteration).
 *   ctrl[0] n_alive   ctrl[1] n_step (0 = loop finished)   ctrl[2] samples per ray marched so far
 *   ctrl[3] n_alive*n_step = valid rows of this iteration (pass ctrl+3 as `n_valid` to the sampling / MLP calls)
 *   ctrl[4] iterations that did work   ctrl[6] survivors left by the last compaction
 * Start state: all zero except ctrl[6] = N.  One iteration = tnl_infer_plan; tnl_march_rays_dev; field; tnl_composite_rays_dev;
 * tnl_compact_alive_dev (alive -> out, swap the two lists).  `cap` >= n_alive sizes the grids (any upper bound: N, or the
 * last n_alive the host has seen); buffers hold min(N, 8*cap) rows (+ alignment).  Rows a ray does not reach are zeroed by the
 * marcher (the host-driven calls rely on freshly zeroed buffers instead).  noises may be NULL (no perturbation).
 * Iterations issued after the loop has finished do nothing.  Results are identical to the host-driven calls. */
int tnl_infer_plan(int32_t* ctrl, uint32_t N, uint32_t max_steps, tnl_stream_t stream);
int tnl_march_rays_dev(const int32_t* ctrl, uint32_t cap, const int32_t* rays_alive, const float* rays_t,
                       const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                       uint32_t H, const uint8_t* grid, const float* fars, float* xyzs, float* dirs, float* deltas,
                       const float* noises, tnl_stream_t stream);
int tnl_composite_rays_dev(const int32_t* ctrl, uint32_t cap, float T_thresh, int32_t* rays_alive, float* rays_t,
                           const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum, float* depth,
                           float* image, tnl_stream_t stream);
int tnl_compact_alive_dev(int32_t* ctrl, uint32_t cap, const int32_t* alive, int32_t* out, void* workspace,
                          size_t workspace_bytes, tnl_stream_t stream);

/* ------------------------------------------------------------------ SH direction encoder ----- */
/* replaces sh_encode_forward (shencoder.h:9, shencoder.cu:387-398) for degree <= 4, dy_dx = NULL */
int tnl_sh_encode_forward(const float* inputs, float* outputs, uint32_t B, uint32_t degree, tnl_stream_t stream);
/* replaces sh_encode_backward (shencoder.h:10, shencoder.cu kernel_sh_backward): grad_inputs [B][3] (fp32, overwritten) =
 * sum_ch grad[b][ch] d(outputs[b][ch]) / d(inputs[b]), the analytic Jacobian of tnl_sh_encode_forward's polynomials summed in
 * channel order.  grad [B][degree^2].  degree outside 1..4 returns TNL_ERR_INVALID_ARGUMENT. */
int tnl_sh_encode_backward(const float* grad, const float* inputs, uint32_t B, uint32_t degree, float* grad_inputs,
                           tnl_stream_t stream);

/* ------------------------------------------------------------------ wavelet planes ----------- */
/* One level of the inverse 2-D DWT (bior6.8, zero mode; other wavelets: the *_wavelet calls below) exactly as TriPlaneVolume.build_planes chains
 * it (triplane_encoder.py:379-394):  out = IDWT(pad4(2*x), pad4(yh)),  n -> 2n.
 * x [3][n][n][C], yh [3][3][n][n][C] (yh[.,0]=high-pass along H, [.,1]=along W, [.,2]=both),
 * out [3][2n][2n][C].  C % 8 == 0, n % 8 == 0. */
/* abs_sum (device float*, may be NULL): += sum |yh| over the level -- the forward value of the wavelet L1
 * regulariser (reconstruction/nerf/utils.py:640-655) as a by-product of the pass that reads yh anyway. */
int tnl_idwt_level_forward(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                           tnl_stream_t stream);
/* Exact adjoint of the above: g_out [3][2n][2n][C] -> g_x [3][n][n][C], g_yh [3][3][n][n][C]
 * (what SFB2D.backward + pad backward + the 2*x factor produce in the reference's autograd graph).
 * Optional fused regulariser gradient: if yh and reg_grad (device float*) are non-NULL,
 * g_yh += reg_coef * (*reg_grad) * sign(yh)   (d/dyh of  sum|yh|, scaled by its upstream gradient).
 * plane0 / nplanes: process only planes [plane0, plane0 + nplanes) (the multi-GPU path pipelines the per-plane gradient
 * exchange against the backward of the previous plane); (0, 3) = all. */
int tnl_idwt_level_backward(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                            const float* reg_grad, float reg_coef, uint32_t plane0, uint32_t nplanes, tnl_stream_t stream);

/* Work-list variants of the two calls above for the training hot path, where the planes are only sampled (and only
 * receive gradient) inside the tiles the occupancy grid marks (tnl_mark_dirty_tiles); n % 16 == 0.
 *   active / clean: int32 [max][4] = {plane, m0, row_lo, row_hi}: blocks of 16 coarse columns [m0, m0+16) x rows
 *   [row_lo, row_hi); together the two lists tile the level exactly once.  counts (device int32[2]) = number of valid
 *   entries of (active, clean); the grids are sized by max_active / max_clean, so the lists may be rewritten in place
 *   between launches (and CUDA-graph replays) when the occupancy grid changes.
 * forward : active blocks are reconstructed exactly as by the dense call (their part of `out`, fine pixels
 *   [2*m0, 2*m0+32) x [2*row_lo, 2*row_hi)); the part of `out` that belongs to clean blocks is NOT written; clean
 *   blocks only contribute their |yh| to abs_sum.  The caller marks as active every block whose output is read later.
 * backward: active blocks as the dense call; clean blocks (g_out == 0 on their whole input window):
 *   g_x = 0, g_yh = reg_coef * (*reg_grad) * sign(yh) (or 0 without the regulariser).
 *   parts: bit 0 = process the active blocks, bit 1 = the clean blocks (3 = both).  The clean part does not depend on
 *   g_out (may be NULL), so the training step issues it early on a second stream.  abs_sum (may be NULL): the clean
 *   part adds sum |yh| over its blocks, so a forward that ran with parts = 1 (active blocks only) gets the complete
 *   regulariser value without a second pass over the coefficients.
 * forward parts: bit 0 = reconstruct the active blocks, bit 1 = add the clean blocks' |yh| to abs_sum. */
int tnl_idwt_level_forward_sparse(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                  const int32_t* active, const int32_t* clean, const int32_t* counts, uint32_t max_active,
                                  uint32_t max_clean, uint32_t parts, tnl_stream_t stream);
int tnl_idwt_level_backward_sparse(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                   const float* reg_grad, float reg_coef, const int32_t* active, const int32_t* clean,
                                   const int32_t* counts, uint32_t max_active, uint32_t max_clean, uint32_t parts,
                                   float* abs_sum, tnl_stream_t stream);

/* The four calls above for a chosen wavelet of the reference's pad table (triplane_encoder.py:174-180); the calls without
 * the suffix are the TNL_WAVELET_BIOR6_8 case.  Same arguments plus `wavelet`; unknown ids return TNL_ERR_INVALID_ARGUMENT.
 * Every bank has 4*pad = L - 2 (L = filter length), so a padded level maps n -> 2n and the shapes above hold for all of them. */
#define TNL_WAVELET_BIOR6_8 0 /* pad 4, L = 18 */
#define TNL_WAVELET_HAAR 1    /* pad 0, L = 2 */
#define TNL_WAVELET_BIOR2_2 2 /* pad 1, L = 6 */
#define TNL_WAVELET_BIOR2_6 3 /* pad 3, L = 14 */
#define TNL_WAVELET_BIOR4_4 4 /* pad 2, L = 10 */
int tnl_idwt_level_forward_wavelet(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                   uint32_t wavelet, tnl_stream_t stream);
int tnl_idwt_level_backward_wavelet(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                    const float* reg_grad, float reg_coef, uint32_t plane0, uint32_t nplanes, uint32_t wavelet,
                                    tnl_stream_t stream);
int tnl_idwt_level_forward_sparse_wavelet(const float* x, const float* yh, float* out, uint32_t n, uint32_t C, float* abs_sum,
                                          const int32_t* active, const int32_t* clean, const int32_t* counts, uint32_t max_active,
                                          uint32_t max_clean, uint32_t parts, uint32_t wavelet, tnl_stream_t stream);
int tnl_idwt_level_backward_sparse_wavelet(const float* g_out, float* g_x, float* g_yh, uint32_t n, uint32_t C, const float* yh,
                                           const float* reg_grad, float reg_coef, const int32_t* active, const int32_t* clean,
                                           const int32_t* counts, uint32_t max_active, uint32_t max_clean, uint32_t parts,
                                           float* abs_sum, uint32_t wavelet, tnl_stream_t stream);

/* Bilinear tri-plane sampling: replaces F.grid_sample(bilinear, border, align_corners=True) +
 * permute/concat of TriPlaneVolume.forward (triplane_encoder.py:314-332, 523-530).
 * planes [3][R][R][C]; xyz [M][3]; feat [M][3C] with feature index p*C + c.
 * u = xyz * inv_bound (inv_bound = 1/bound in fp32, CUDA's tensor/scalar rule); if fp16_coords != 0,
 * u is rounded to fp16 first (the autocast quirk of triplane_encoder.py:299, SURVEY.md 8a-2).
 * n_valid (device int32*, may be NULL): rows >= *n_valid are skipped (feat rows written as zeros).
 * perm (device int32 [M], may be NULL): visit order (tnl_cell_sort); row m of feat always belongs to point m.
 * feat_fp16 != 0: feat / g_feat are __half [M][3C] -- the rounding the first nn.Linear applies under autocast
 * (network.py:127) done by the producer, halving the bytes of the feature stream. */
int tnl_sample_planes_forward(const float* planes, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                              float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                              void* feat, int feat_fp16, tnl_stream_t stream);
/* Adjoint scatter (grid_sampler_2d_backward w.r.t. input): g_planes += ...; caller zero-fills g_planes. */
int tnl_sample_planes_backward(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                               float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                               float* g_planes, tnl_stream_t stream);
/* The same scatter for ONE plane (plane = 0, 1, 2; C in {16, 32, 48}): three calls equal tnl_sample_planes_backward.  The
 * multi-GPU training step issues them one by one and starts the exchange of a plane's gradient while the next plane scatters. */
int tnl_sample_planes_backward_plane(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                                     float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                     float* g_planes, uint32_t plane, tnl_stream_t stream);
/* Deterministic mode (torch.use_deterministic_algorithms): the scatter of tnl_sample_planes_backward with sums that do not depend on
 * the visiting order (perm) or the thread schedule.  Contributions are added in 64-bit fixed point: m = max |g_feat| over the rows
 * below *n_valid, 2^e > m, mu = ceil(log2 M), unit = 2^(e + mu - 62); each contribution is rounded to a multiple of the unit (no
 * partial sum can overflow), and each texel's sum is converted to fp32 once and added to g_planes.  Per texel the result is within
 * n * unit / 2 (n = its contributions) plus one fp32 rounding of the exact sum.  If a g_feat value below *n_valid is inf or NaN,
 * every converted g_planes element is NaN.  tile_ids == NULL: the whole planes; else only the listed T x T tiles (tile_ids /
 * tile_count / tile_capacity as tnl_tiles_zero) are accumulated and converted, contributions elsewhere are dropped (the
 * work-list IDWT backward reads only those tiles).  workspace: tnl_sample_planes_backward_det_workspace(R, C) bytes (int64 accumulator), 256-byte aligned. */
size_t tnl_sample_planes_backward_det_workspace(uint32_t R, uint32_t C);
int tnl_sample_planes_backward_det(const void* g_feat, int feat_fp16, const float* xyz, uint32_t M, uint32_t R, uint32_t C,
                                   float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                   const int32_t* tile_ids, const int32_t* tile_count, uint32_t tile_capacity, uint32_t T,
                                   float* g_planes, void* workspace, size_t workspace_bytes, tnl_stream_t stream);

/* Gradient with respect to the sample positions (grid_sampler_2d_backward w.r.t. the grid, chained through u = xyz * inv_bound):
 * g_xyz [M][3] = d(sum g_feat * feat)/d(xyz), written (not accumulated).  The derivative is zero along an axis whose projected
 * coordinate lies on or beyond the plane border (ATen's clip_coordinates_set_grad), and the fp16 rounding of fp16_coords is
 * passed straight through, as autograd does for a dtype cast.  fp32 features only.  Replaces what autograd derives from the
 * F.grid_sample call of super_resolution/threestudio/models/triplaneencoder/triplane_encoder.py:262 when the positions
 * require grad (analytic normals, super_resolution/threestudio/models/geometry/implicit_volume.py:218-226). */
int tnl_sample_planes_backward_coords(const float* g_feat, const float* planes, const float* xyz, uint32_t M, uint32_t R,
                                      uint32_t C, float inv_bound, int fp16_coords, float* g_xyz, tnl_stream_t stream);
/* Position gradient of the NeRF field's plane gather (TriPlaneVolume.forward with coordinates that require grad):
 * g_xyz [M][3] fp32 (every row written; rows >= *n_valid get 0) from g_feat [M][3C] (fp16 if feat_fp16, else fp32), with the
 * n_valid / perm conventions of tnl_sample_planes_backward.  fp16_coords reproduces the reference's fp16-autocast backward:
 * each plane's grid gradient is rounded to fp16, the per-axis sum of the two planes that read an axis is rounded to fp16 again,
 * and only then scaled by inv_bound.  planes [3][R][R][C] channels-last, as tnl_sample_planes_forward reads them. */
int tnl_sample_planes_backward_xyz(const void* g_feat, int feat_fp16, const float* planes, const float* xyz, uint32_t M, uint32_t R,
                                   uint32_t C, float inv_bound, int fp16_coords, const int32_t* n_valid, const int32_t* perm,
                                   float* g_xyz, tnl_stream_t stream);

/* Spatial binning of sample points: perm[i] = row of the i-th point in the order of a G^3 Morton grid over
 * [-bound, bound]^3 (rows >= *n_valid last).  Kernels taking `perm` visit points in that order, which makes the
 * plane gathers / gradient scatters of neighbouring threads hit the same texels (L2 locality); per-point results
 * are unchanged.  No reference counterpart (the reference evaluates samples in marching order). */
size_t tnl_cell_sort_workspace(uint32_t M, uint32_t G);
int tnl_cell_sort(const float* xyz, uint32_t M, const int32_t* n_valid, float inv_bound, uint32_t G, int32_t* perm,
                  void* workspace, size_t workspace_bytes, tnl_stream_t stream);

/* ------------------------------------------------------------------ sigma / color MLP heads -- */
/* NeRFNetwork.forward / .density (network.py:118-166) with the fp16-autocast arithmetic the reference
 * trains with: fp16 operands, fp32 accumulation, fp16 rounding of every layer output, fp32 exp/SH.
 * Weight masters are fp32 row-major [out][in] exactly as nn.Linear stores them:
 *   W1 [H][3C]  W2 [16][H]  W3 [Hc][31]  W4 [Hc][Hc]  W5 [3][Hc];  H, Hc in {64, 128}; 3C % 16 == 0.
 * `packed` (device, >= tnl_mlp_packed_bytes) receives the tensor-core fragment-ordered fp16 copy;
 * re-pack after every optimizer step. */
typedef struct tnl_mlp_dims {
    uint32_t in_dim;   /* 3C */
    uint32_t hidden;   /* H  */
    uint32_t hidden_c; /* Hc */
} tnl_mlp_dims;
size_t tnl_mlp_packed_bytes(const tnl_mlp_dims* dims);
int tnl_mlp_pack_weights(const tnl_mlp_dims* dims, const float* W1, const float* W2, const float* W3,
                         const float* W4, const float* W5, void* packed, tnl_stream_t stream);
/* feat [M][3C] fp32 (or __half if feat_fp16), dirs [M][3] fp32 (NULL => density only) -> sigma [M] fp32, rgb [M][3] fp32
 * (fp16-representable), geo [M][15] fp32 (may be NULL).  n_valid as above (skipped rows -> zeros). */
int tnl_mlp_forward(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                    uint32_t M, const int32_t* n_valid, float* sigma, float* rgb, float* geo,
                    tnl_stream_t stream);
/* Backward of tnl_mlp_forward: recomputes activations from feat; g_sigma [M], g_rgb [M][3] in;
 * g_feat [M][3C] out, same dtype as feat (may be NULL); g_W1..g_W5 fp32 accumulated with atomics (caller zero-fills).
 * H = Hc = 128 (the "large" config) requires the fp16 feature stream (feat_fp16 != 0: tcgen05 kernels, csrc/mlp_tc128.cu). */
int tnl_mlp_backward(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                     uint32_t M, const int32_t* n_valid, const float* g_sigma, const float* g_rgb,
                     void* g_feat, float* g_W1, float* g_W2, float* g_W3, float* g_W4, float* g_W5,
                     tnl_stream_t stream);
/* tnl_mlp_backward fused with tnl_sample_planes_backward for the training step (64-wide heads, tcgen05 kernels, fp16 feat,
 * in_dim = 3C with C in {16, 32}): rows are visited in the order perm [M] (tnl_cell_sort, required), and the input gradient,
 * rounded to fp16 as tnl_mlp_backward stores it, is scattered straight into g_planes [3][R][R][C] (channels-last, accumulated:
 * the caller zero-fills every texel the points touch) instead of being written to memory.  feat / dirs / g_sigma / g_rgb /
 * xyz are indexed by point, as for the two separate calls; R, C, inv_bound, fp16_coords, n_valid as for
 * tnl_sample_planes_backward.  Same results as the two calls up to the order of the fp32 atomic additions. */
int tnl_mlp_backward_scatter(const tnl_mlp_dims* dims, const void* packed, const void* feat, const float* dirs, uint32_t M,
                             const int32_t* n_valid, const int32_t* perm, const float* g_sigma, const float* g_rgb,
                             const float* xyz, uint32_t R, uint32_t C, float inv_bound, int fp16_coords, float* g_planes,
                             float* g_W1, float* g_W2, float* g_W3, float* g_W4, float* g_W5, tnl_stream_t stream);
/* tnl_mlp_backward plus the gradient with respect to the view directions: g_dirs [M][3] fp32 (every row written; rows >=
 * *n_valid get 0).  d(in3) = dh3 W3 is taken over all 32 columns; its SH part is rounded to fp16 (the autocast linear backward),
 * and the degree-4 SH Jacobian at dirs is applied as tnl_sh_encode_backward does.  Same dims and feature streams as
 * tnl_mlp_backward; g_feat and the weight gradients are the same. */
int tnl_mlp_backward_dirs(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                          uint32_t M, const int32_t* n_valid, const float* g_sigma, const float* g_rgb,
                          void* g_feat, float* g_W1, float* g_W2, float* g_W3, float* g_W4, float* g_W5, float* g_dirs,
                          tnl_stream_t stream);
/* Deterministic mode (torch.use_deterministic_algorithms): tnl_mlp_backward (g_dirs == NULL) or tnl_mlp_backward_dirs with weight
 * gradients that do not depend on the order in which the CTAs finish.  Each CTA of the same kernels writes its partial sums to its
 * own slot of `workspace` instead of adding them with fp32 atomics, and a reduction kernel adds the slots in index order to
 * g_W1..g_W5 (accumulated, as tnl_mlp_backward does).  The tile schedule is static, so the result depends on M, *n_valid and the
 * inputs only: the same bits on every call.  The workspace (16-byte aligned) holds tnl_mlp_backward_det_workspace(dims,
 * feat_fp16, M) bytes (0: unsupported dims); g_feat and g_dirs are the same as those of the default entry points. */
size_t tnl_mlp_backward_det_workspace(const tnl_mlp_dims* dims, int feat_fp16, uint32_t M);
int tnl_mlp_backward_det(const tnl_mlp_dims* dims, const void* packed, const void* feat, int feat_fp16, const float* dirs,
                         uint32_t M, const int32_t* n_valid, const float* g_sigma, const float* g_rgb, void* g_feat,
                         float* g_W1, float* g_W2, float* g_W3, float* g_W4, float* g_W5, float* g_dirs, void* workspace,
                         size_t workspace_bytes, tnl_stream_t stream);

/* Diagnostic: ONE tcgen05.mma product D[M x N] = A B^T with fp16 operands given as plain row-major matrices
 * (A: [a_rows][a_cols] = [M][K] if a_mn == 0, [K][M] if a_mn != 0; B likewise with N), staged in the un-swizzled
 * canonical shared-memory layout the fused MLP kernels use; out [128][ncols] = raw dump of the TMEM accumulator
 * (lane-major).  Pins the descriptor conventions of csrc/umma.cuh on real hardware (tests/test_gpu_umma.py). */
int tnl_umma_probe(const void* A, int a_rows, int a_cols, const void* B, int b_rows, int b_cols, int a_mn, int b_mn,
                   int M, int N, int K, float* out, int ncols, tnl_stream_t stream);

/* Diagnostic: tensor-pipe cost of one product shape / operand layout: `reps` x (K/16) tcgen05.mma issued back to back;
 * out2[0] = cycles until completion, out2[1] = cycles spent issuing. */
int tnl_umma_bench(int a_rows, int b_rows, int a_mn, int b_mn, int M, int N, int K, int reps, long long* out2,
                   tnl_stream_t stream);
/* Diagnostic: as tnl_umma_bench with free descriptor fields (LBO / SBO / K-step in 16-byte units, layout type 0 = none,
 * 2 = 128B swizzle, 4 = 64B, 6 = 32B), issued by a converged warp; zero operands. */
int tnl_umma_bench2(uint32_t a_lbo, uint32_t a_sbo, uint32_t a_step, uint32_t a_type, uint32_t b_lbo, uint32_t b_sbo,
                    uint32_t b_step, uint32_t b_type, int a_mn, int b_mn, int M, int N, int ksteps, int reps, long long* out2,
                    tnl_stream_t stream);
/* Diagnostic: counters64 = device buffer of 64 uint64 (zero-filled by the caller) that CTA 0 of the tcgen05 MLP
 * backward fills with cycle counts per pipeline stage ([0..9] warpgroup wait, [10..19] warpgroup epilogue,
 * [20..39] issuer wait (stage*2+wg), [40..59] issuer issue); NULL switches it off (default). */
int tnl_mlp_tc_profile(unsigned long long* counters64);

/* ------------------------------------------------------------------ optimizer epilogue -------- */
/* `scaler.step(optimizer); scaler.update()` of the reference loop (reconstruction/nerf/utils.py:1170-1173) with
 * torch.optim.Adam(betas, eps) (reconstruction/main_nerf.py:119), over flat fp32 arrays (any memory order, the same for
 * p / g / m / v).  All scalars that depend on earlier kernels stay on the device, so the epilogue needs no host sync.
 *   tnl_grad_nonfinite : *found_inf = 1 if any element of g is inf / NaN (caller zero-fills found_inf once per step)
 *   tnl_adam_prepare   : state3 = {step, 1 - beta1^step, sqrt(1 - beta2^step)}; step += 1 unless *found_inf != 0
 *   tnl_adam_step      : unless *found_inf != 0:  g' = g * (*inv_scale) (+ weight_decay * p);  m += (g' - m)(1 - beta1);
 *                        v = beta2 v + (1 - beta2) g'^2;  p -= lr / state3[1] * m / (sqrt(v) / state3[2] + eps)
 * inv_scale / found_inf may be NULL (no loss scaling). */
int tnl_grad_nonfinite(const float* g, uint64_t n, float* found_inf, tnl_stream_t stream);
int tnl_adam_prepare(float* state3, const float* found_inf, float beta1, float beta2, tnl_stream_t stream);
int tnl_adam_step(float* p, const float* g, float* m, float* v, uint64_t n, const float* inv_scale, const float* found_inf,
                  const float* state3, float lr, float beta1, float beta2, float eps, float weight_decay, tnl_stream_t stream);

/* ------------------------------------------------------------------ density grid ------------- */
/* Fused pieces of NeRFRenderer.update_extra_state (reconstruction/nerf/renderer.py:448-542). */
/* cell-centre sample positions for a list of Morton cells of one cascade (renderer.py:474-483):
 *   xyz = (2*coord/(H-1) - 1) * (bound_c - hgs) + (2*noise - 1) * hgs,  hgs = bound_c / H
 * indices [n] int32 Morton codes, noise [n][3] uniform [0,1) -> xyz [n][3] */
int tnl_grid_cell_positions(const int32_t* indices, uint32_t n, uint32_t H, float bound_c, const float* noise,
                            float* xyz, tnl_stream_t stream);
/* The tail of update_extra_state without a host round trip (renderer.py:526-534): grid = max(grid*decay, tmp_grid) where both >= 0, plus
 * *sum = sum_i max(grid[i], 0) in double (zeroed here); then mean = *sum / n_cells -> *mean_out, thresh = min(mean, thresh_cap),
 * bitfield = packbits(grid > thresh).  n_cells % 32 == 0. */
int tnl_grid_ema_update_sum(float* grid, const float* tmp_grid, uint32_t n, float decay, double* sum, tnl_stream_t stream);
int tnl_packbits_mean(const float* grid, uint32_t n_cells, const double* sum, float thresh_cap, float* mean_out,
                      uint8_t* bitfield, tnl_stream_t stream);
/* tmp_grid_cascade[indices[i]] = sigma[i] * scale   (renderer.py:486-488: `tmp_grid[cas, indices] = sigmas * density_scale`) */
int tnl_grid_scatter(const int32_t* indices, const float* sigma, uint32_t n, float scale, float* tmp_grid_cascade,
                     tnl_stream_t stream);

/* ------------------------------------------------------------------ step feeder (SURVEY.md 8f-2) -- */
/* replaces, for one step's batch, get_rays (reconstruction/nerf/utils.py:64-149), the index into the shuffled ray table
 * of shuffle_data / select_batch (utils.py:228-243) and the target gather of collate (nerf/provider.py:708-711).
 * poses [B][4][4] cam2world (row-major, 16-byte aligned); pixel centre + 0.5, dir = normalise((i-cx)/fx, (j-cy)/fy, 1),
 * rays_d = dir @ R^T, rays_o = t.  A ray id addresses the flattened [B*H*W] table: id = image * H*W + row * W + col.
 * ray_ids [n] int64 device pointer, or NULL for the contiguous range first_id .. first_id+n-1 (full frames, N = -1).
 * images [B][H*W][image_channels] fp32 (optional, channels 3 or 4) -> targets [n][image_channels]; both NULL to skip.
 * Ids outside [0, B*H*W) are clamped (the reference raises on the host). */
int tnl_rays_from_ids(const float* poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W,
                      const int64_t* ray_ids, int64_t first_id, uint32_t n, const float* images, uint32_t image_channels,
                      float* rays_o, float* rays_d, float* targets, tnl_stream_t stream);
/* Pose gradient of tnl_rays_from_ids (same B, intrinsics, H, W, ray_ids / first_id, n; ids clamped as there):
 *   g_poses[b][r][c] = sum_{rays t of image b} g_rays_d[t][r] dir_t[c]  (c < 3),   g_poses[b][r][3] = sum g_rays_o[t][r],
 * bottom row 0; an image without rays gets exactly 0.  dir_t is recomputed with the forward's per-pixel arithmetic.  The
 * gradient does not depend on the pose values, so the poses are not an argument.  g_rays_o / g_rays_d [n][3] fp32 (either may
 * be NULL: zero); g_poses [B][4][4] fp32 is overwritten.  One CTA per image scans the batch in a fixed order: no atomics, the
 * same bits on every run. */
int tnl_rays_from_ids_backward(const float* g_rays_o, const float* g_rays_d, uint32_t B, float fx, float fy, float cx, float cy,
                               uint32_t H, uint32_t W, const int64_t* ray_ids, int64_t first_id, uint32_t n, float* g_poses,
                               tnl_stream_t stream);

/* ------------------------------------------------------------------ multi-GPU gradient exchange ---- */
/* flags [3][R/T][R/T] (uint8): 1 where a tile of T x T texels can receive plane gradient, i.e. lies under the projection
 * of an occupied density-grid cell (+ margin texels).  Deterministic function of the bitfield: identical on all ranks. */
int tnl_mark_dirty_tiles(const uint8_t* bitfield, uint32_t cascade, uint32_t H, float bound, uint32_t R, uint32_t T,
                         uint32_t margin, uint8_t* flags, tnl_stream_t stream);
/* gather / scatter the listed tiles between planes [3][R][R][C] and a compact buffer [n_tiles][T][T][C]
 * (tile id = (p * R/T + ty) * R/T + tx); unpack multiplies by `scale` (1/world_size for an average).
 * bf16 != 0: the compact (transport) buffer is bfloat16 -- half the NVLink bytes; planes stay fp32. */
/* Zero the listed tiles of planes [3][R][R][C] (the part of the plane-gradient buffer the work-list IDWT backward reads);
 * *count (device) = number of valid ids, the grid is sized by `capacity`. */
int tnl_tiles_zero(float* planes, const int32_t* tile_ids, const int32_t* count, uint32_t capacity, uint32_t R, uint32_t C,
                   uint32_t T, tnl_stream_t stream);
int tnl_tiles_pack(const float* planes, const int32_t* tile_ids, uint32_t n_tiles, uint32_t R, uint32_t C, uint32_t T,
                   void* compact, int bf16, tnl_stream_t stream);
int tnl_tiles_unpack(const void* compact, const int32_t* tile_ids, uint32_t n_tiles, uint32_t R, uint32_t C, uint32_t T,
                     float scale, int bf16, float* planes, tnl_stream_t stream);

/* The same exchange IN PLACE over peer memory, without pack / unpack and in fp32: the plane-gradient buffers [3][R][R][C] of
 * all ranks are symmetric allocations (identical size, peer-mapped over NVLink; `multicast` != NULL: additionally mapped
 * through one NVSwitch multicast address).  Tile k of the (replicated) list is reduced by rank k % world:
 *   multicast != NULL   multimem.ld_reduce.add (sum formed in the switch) -> x scale -> multimem.st (broadcast by the switch);
 *   multicast == NULL   loads from every peers[r], sum in rank order, stores to every peers[r]  (peers: HOST array of `world`
 *                       device pointers, each rank's mapping of the same buffer; world <= 8).
 * tile_ids / count / capacity as tnl_tiles_zero (count read on the device).  The caller brackets the call with cross-rank
 * barriers.  tnl_flat_allreduce: the same for a flat fp32 buffer (n_floats % 4 == 0; the MLP weight gradients). */
int tnl_tiles_allreduce(void* multicast, const void* const* peers, const int32_t* tile_ids, const int32_t* count,
                        uint32_t capacity, uint32_t R, uint32_t C, uint32_t T, uint32_t rank, uint32_t world, float scale,
                        tnl_stream_t stream);
int tnl_flat_allreduce(void* multicast, const void* const* peers, uint32_t n_floats, uint32_t rank, uint32_t world,
                       float scale, tnl_stream_t stream);

/* ------------------------------------------------------------------ mesh extraction ---------- */
/* Marching cubes (replaces mcubes.marching_cubes in the reference's extract_geometry, nerf/utils.py) over a dense fp32 volume
 * [nx][ny][nz] (C-contiguous, u[x, y, z]; nx, ny, nz >= 2; +-inf allowed, NaN rejected).  A lattice point is inside iff
 * u >= threshold.  Case table: csrc/mc_tables.cuh (generated by csrc/gen_mc_tables.py; face-local, so no cracks between cubes).
 * Outputs, in an order that does not depend on the thread schedule:
 *   vertices  [V][3] float64, index space: one per lattice edge whose end values straddle the threshold, ordered by (linear
 *             index of the edge's lower lattice point, axis x < y < z); position p + t e_axis with
 *             t = (threshold - u_lower) / (u_upper - u_lower) in float64 (t = 1 if u_lower is infinite);
 *   triangles [T][3] int64 vertex ids, ordered by (linear cube index, table order); normals (v1-v0)x(v2-v0) point from the
 *             inside region to the outside one.
 * Two calls on one stream and workspace:
 *   tnl_mc_count  writes totals[2] (DEVICE int64) = (V, T), or (-1, -1) if the volume contains a NaN;
 *   tnl_mc_emit   takes the host copy of those totals (the capacities of the caller's outputs) and fills the outputs; negative
 *                 totals return TNL_ERR_INVALID_ARGUMENT.
 * Workspace: tnl_mc_workspace bytes, about 2.01 bytes per lattice point (a uint16 per point plus 24 bytes per 2048 points);
 * 2.0 GiB at 1024^3.  0 if an axis has fewer than 2 points. */
size_t tnl_mc_workspace(uint32_t nx, uint32_t ny, uint32_t nz);
int tnl_mc_count(const float* volume, uint32_t nx, uint32_t ny, uint32_t nz, double threshold, void* workspace,
                 size_t workspace_bytes, int64_t* totals, tnl_stream_t stream);
int tnl_mc_emit(const float* volume, uint32_t nx, uint32_t ny, uint32_t nz, double threshold, const void* workspace,
                size_t workspace_bytes, int64_t n_vertices, int64_t n_triangles, double* vertices, int64_t* triangles,
                tnl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TRINERFLET_B200_H */
