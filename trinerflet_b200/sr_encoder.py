"""The tri-plane encoders of the reference's super_resolution application over the same CUDA kernels -- drop-in for
super_resolution/threestudio/models/triplaneencoder/triplane_encoder.py (SURVEY.md 8 f-4):

    TriPlaneVolume             :26-436   wavelet tri-plane with a low- and a high-resolution reading of the same coefficients
    KPlaneVolume               :445-489  a pyramid of plain tri-planes, features concatenated or multiplied over the planes
    MultiscaleKPlaneVolume     :491-527  low-resolution pyramid (+ a high-resolution pyramid in 'high_res' mode), concatenated
    MultiscaleKPlaneMulVolume  :529-578  the same with every plane of every level multiplied together

Same constructor kwargs, attributes, method names (including `reset_cahce`) and state-dict keys, so the application's
`get_encoding` (super_resolution/threestudio/models/networks.py:142-177) can construct these instead.  What differs from the
reconstruction encoder (triplane_encoder.py in this package):

  * `get_planes()` stops the level loop at the first level whose side reaches plane_resolution / low_res_scale (and, in double
    mode, again at plane_resolution / high_res_scale), so a low-resolution render pays for the coarse levels only; the
    high-resolution planes continue from the low-resolution ones (one autograd chain, gradients of both renders add up in the
    shared coarse levels).  With `enable_cache` both readings are kept until `reset_cahce()`.
  * positions arrive in the unit cube (`input_pts_in_unit_cube`) and are mapped to [-lbound, lbound] first.
  * the positions may require grad (analytic normals, threestudio/models/geometry/implicit_volume.py:218-226): the sampling
    node returns d/d(xyz) from tnl_sample_planes_backward_coords.  As with the reference's F.grid_sample (:262), the backward
    is not differentiable again by default; `high_order_gradients = True` switches to an op with the capability of the
    reference's grid_backward.py (whose call is commented out at :263): gradients of any order between planes and features.
  * an empty batch returns zeros(0, 3C) (:431-434).

Storage is channels-last as everywhere in this package (see triplane_encoder.py); reference checkpoints load unchanged.
There is no CPU path: tensors must be CUDA tensors.
"""
import torch
import torch.nn as nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from ._lib import call, ptr, stream
from . import triplane_encoder as _te
from .triplane_encoder import _inv_bound, build_planes, cl_empty_planes, to_cl_planes


class _SamplePlanesXyz(Function):
    """feat [M,3C] = bilinear samples of planes [3,C,R,R] at xyz/bound; backward w.r.t. the planes (scatter) and the positions."""

    @staticmethod
    def forward(ctx, planes, coords, bound):
        _te._require_cuda_f32(planes, "planes")
        planes_cl = to_cl_planes(planes.detach())
        xyz = coords.detach().contiguous().float()
        M, C, R = xyz.shape[0], planes.shape[1], planes.shape[2]
        feat = torch.empty(M, 3 * C, device=planes.device, dtype=torch.float32)
        inv = _inv_bound(bound)
        call("tnl_sample_planes_forward", ptr(planes_cl), ptr(xyz), M, R, C, inv, 0, None, None, ptr(feat), 0, stream())
        ctx.save_for_backward(planes_cl, xyz)
        ctx.meta = (M, R, C, inv, coords.dtype)
        return feat

    @staticmethod
    @once_differentiable
    def backward(ctx, g_feat):
        planes_cl, xyz = ctx.saved_tensors
        M, R, C, inv, coords_dtype = ctx.meta
        g_feat = g_feat.contiguous().float()
        g_planes = g_xyz = None
        if ctx.needs_input_grad[0]:
            g_planes = cl_empty_planes(C, R, device=g_feat.device, zero=True)
            _te.scatter_planes(g_feat, False, xyz, M, R, C, inv, 0, None, None, g_planes)
        if ctx.needs_input_grad[1]:
            g_xyz = torch.empty(M, 3, device=g_feat.device, dtype=torch.float32)
            call("tnl_sample_planes_backward_coords", ptr(g_feat), ptr(planes_cl), ptr(xyz), M, R, C, inv, 0, ptr(g_xyz), stream())
            g_xyz = g_xyz.to(coords_dtype)
        return g_planes, g_xyz, None


class _SampleHighOrder(Function):
    """The sampling op with gradients of arbitrary order between the planes and the output -- the capability of the reference's
    grid_backward.py (:41-99, NVIDIA's grid_sample_gradfix; present in the reference but switched off at triplane_encoder.py:263):
    the backward pass is itself an autograd node whose derivative w.r.t. the incoming feature gradient is this op again, applied
    to the plane-shaped cotangent.  As there (:84-97), second-order terms through the positions are not provided."""

    @staticmethod
    def forward(ctx, planes, coords, bound):
        feat = _SamplePlanesXyz.forward(ctx, planes, coords, bound)
        ctx.bound = bound
        return feat

    @staticmethod
    def backward(ctx, g_feat):
        planes_cl, xyz = ctx.saved_tensors
        g_planes, g_xyz = _SampleHighOrderBackward.apply(g_feat, planes_cl, xyz, ctx.bound, ctx.meta, ctx.needs_input_grad[0],
                                                        ctx.needs_input_grad[1])
        return g_planes, g_xyz, None


class _SampleHighOrderBackward(Function):
    @staticmethod
    def forward(ctx, g_feat, planes_cl, xyz, bound, meta, need_planes, need_xyz):
        M, R, C, inv, coords_dtype = meta
        g_feat = g_feat.detach().contiguous().float()
        g_planes = g_xyz = None
        if need_planes:
            g_planes = cl_empty_planes(C, R, device=g_feat.device, zero=True)
            _te.scatter_planes(g_feat, False, xyz, M, R, C, inv, 0, None, None, g_planes)
        if need_xyz:
            g_xyz = torch.empty(M, 3, device=g_feat.device, dtype=torch.float32)
            call("tnl_sample_planes_backward_coords", ptr(g_feat), ptr(planes_cl), ptr(xyz), M, R, C, inv, 0, ptr(g_xyz), stream())
            g_xyz = g_xyz.to(coords_dtype)
        ctx.save_for_backward(xyz)
        ctx.bound = bound
        ctx.set_materialize_grads(False)
        return g_planes, g_xyz

    @staticmethod
    def backward(ctx, gg_planes, gg_xyz):
        xyz, = ctx.saved_tensors
        gg_feat = None
        if ctx.needs_input_grad[0] and gg_planes is not None:
            gg_feat = _SampleHighOrder.apply(gg_planes, xyz, ctx.bound)
        return gg_feat, None, None, None, None, None, None


def sample_planes_xyz(planes, coords, bound, high_order=False):
    """planes logical [3,C,R,R], coords [M,3] in [-bound, bound] -> features [M, 3C]; differentiable in both.  high_order:
    gradients of any order between planes and features (see _SampleHighOrder); default: once, like F.grid_sample."""
    if high_order:
        return _SampleHighOrder.apply(planes, coords, float(bound))
    return _SamplePlanesXyz.apply(planes, coords, float(bound))


class TriPlaneVolume(_te.TriPlaneVolume):
    """super_resolution/threestudio/models/triplaneencoder/triplane_encoder.py:26-436."""

    def __init__(self, number_of_features=3, plane_resolution=224, init_sigma=0.1, lbound=1, viewdir_plane_resolution=32,
                 two_planes_per_axis=False, planes_features=None, viewdir_plane=None, apply_activation_on_features=False,
                 inner_multi_res_scale=1, inner_multi_res_viewdir_scale=1, viewdir_mode='plane',
                 inner_multi_res_scale_current=1, low_res_scale=1, high_res_scale=1, input_pts_in_unit_cube=True,
                 wavelet_type='bior6.8', wavelet_base_resolution=0, init_fn=None):
        levels = _te.get_levels(inner_multi_res_scale) if inner_multi_res_scale > 1 else 0
        if levels > 0 and wavelet_base_resolution != 0:
            # :141 / :309 stop cropping the analysis / padding the synthesis below this side; no reference config sets it with levels
            raise NotImplementedError("trinerflet_b200.sr_encoder.TriPlaneVolume: wavelet_base_resolution != 0 with wavelet levels")
        if levels > 0 and wavelet_type != 'bior6.8':
            # the super-resolution readings keep the reference configuration's bior6.8
            raise NotImplementedError(f"trinerflet_b200.sr_encoder.TriPlaneVolume: wavelet_type={wavelet_type} with wavelet levels")
        if low_res_scale < high_res_scale:
            raise AssertionError("low_res_scale >= high_res_scale")                     # :73
        if planes_features is None and init_fn is not None and levels == 0:      # :91-96: only the plain planes use init_fn
            planes_features = init_fn(init_sigma * torch.randn(3, number_of_features, plane_resolution, plane_resolution))
        super().__init__(number_of_features=number_of_features, plane_resolution=plane_resolution, init_sigma=init_sigma,
                         lbound=lbound, viewdir_plane_resolution=viewdir_plane_resolution,
                         two_planes_per_axis=two_planes_per_axis, planes_features=planes_features, viewdir_plane=viewdir_plane,
                         apply_activation_on_features=apply_activation_on_features,
                         inner_multi_res_scale=inner_multi_res_scale,
                         inner_multi_res_viewdir_scale=inner_multi_res_viewdir_scale, viewdir_mode=viewdir_mode,
                         inner_multi_res_scale_current=inner_multi_res_scale_current,
                         # without levels the wavelet is never applied (KPlaneVolume passes 'haar'); any name will do
                         wavelet_type=wavelet_type if levels > 0 else 'bior6.8', wavelet_base_resolution=0)
        self.wavelet_type = wavelet_type
        self.planes_features_wavelet_pad = _te.PAD_DICT.get(wavelet_type, 0)
        self.wavelet_base_resolution = wavelet_base_resolution
        self.input_pts_in_unit_cube = input_pts_in_unit_cube
        self.n_output_dims = 3 * number_of_features
        self.n_input_dims = 3
        self.low_res_scale = low_res_scale
        self.high_res_scale = high_res_scale
        self.double_resolution_mode = False
        self.current_resolution_mode = 'low_res'
        self.enable_cache = False
        self.enable_grid_acc = False
        self.init_fn = init_fn
        # True: sample through the op that can be differentiated repeatedly w.r.t. the planes -- what the reference's
        # grid_backward.grid_sample offers (its call is commented out there, triplane_encoder.py:263, so the default is off)
        self.high_order_gradients = False

    # -- the two readings of the coefficient pyramid (:268-340) ----------------------------------------
    def _level_split(self):
        """(k_low, k_high): how many wavelet levels each reading applies.  The reference's loop tests the side of x BEFORE
        each level l (n0 * 2^l) against the two thresholds; a reading that is never reached uses all levels."""
        L = self.planes_features_wavelet_all_level
        n0 = self.planes_features.shape[2]
        low_res = self.plane_resolution / self.low_res_scale
        high_res = self.plane_resolution / self.high_res_scale
        k_low = next((l for l in range(L) if n0 * 2 ** l >= low_res), L)
        k_high = next((l for l in range(k_low, L) if n0 * 2 ** l >= high_res), L)
        return k_low, k_high

    def get_planes(self, max_res=-1, max_scale=-1):
        # max_res / max_scale are accepted and ignored, as in the reference (:268; get_grid_features passes max_res)
        if self.last_used_planes is not None:
            key = self.current_resolution_mode if self.double_resolution_mode else 'low_res'
            return self.last_used_planes[key]
        planes = x_low = self.planes_features     # (without levels the reference caches None here and fails on the next call)
        x_high = None
        if self.inner_wavelet_scale > 1:
            coefs = list(self.planes_features_wavelet_coefs)
            k_low, k_high = self._level_split()
            x_low = build_planes(self.planes_features, coefs[:k_low]) if k_low > 0 else self.planes_features
            if self.double_resolution_mode:
                x_high = build_planes(x_low, coefs[k_low:k_high]) if k_high > k_low else x_low
            planes = x_high if (self.double_resolution_mode and self.current_resolution_mode == 'high_res') else x_low
        if self.enable_cache:
            self.last_used_planes = {'low_res': x_low, 'high_res': x_high}
        return planes

    def set_resolution_mode(self, val):
        assert val in ['low_res', 'high_res']
        self.current_resolution_mode = val

    def set_double_mode(self, val: bool):
        self.double_resolution_mode = val

    def reset_cahce(self):  # (sic)
        self.last_used_planes = None

    reset_cache = reset_cahce

    def get_wavelet_features(self):
        return list(self.planes_features_wavelet_coefs) if self.inner_wavelet_scale > 1 else []

    def wavelet_l1(self, lam, abs_sums=None):
        raise NotImplementedError("the super_resolution application forms its regulariser from get_wavelet_features() "
                                  "(threestudio/systems/triplane_wavelet_sr.py:651-660)")

    def prefetch_planes(self, side, partial_zero=False):
        raise NotImplementedError("prefetch_planes belongs to the NeRF training step (trainer.TrainStep)")

    # -- sampling (:252-265, :347-369, :421-436) ------------------------------------------------------------
    def sample_from_planes(self, coordinates, plane_features=None, lbound=None):
        if plane_features is None:
            plane_features = self.get_planes()
        if lbound is None:
            lbound = self.lbound
        if self.input_pts_in_unit_cube:
            coordinates = (coordinates * 2 - 1) * lbound
        feat = sample_planes_xyz(plane_features, coordinates, lbound, high_order=self.high_order_gradients)
        return feat.view(feat.shape[0], 3, plane_features.shape[1])

    def forward(self, coordinates, bound=None):
        if coordinates.shape[0] == 0:
            return torch.zeros(0, self.number_of_features * 3, device=coordinates.device, dtype=coordinates.dtype)
        sampled = self.sample_from_planes(coordinates, lbound=bound)
        return sampled.view(sampled.shape[0], -1)

    def get_grid_features(self, grid_res, plane_features=None, grid=None):
        """:371-413 -- features on a regular grid_res^3 lattice of the cube (axes permuted to (z, x, y) as the reference does)."""
        if grid is None:
            axis = torch.arange(grid_res)
            gx, gy, gz = torch.meshgrid(axis, axis, axis, indexing='xy')
            grid = torch.stack([gx, gy, gz], dim=-1) / (grid_res - 1)
        assert grid.max() <= 1 and grid.min() >= 0
        grid = 2 * self.lbound * grid - self.lbound
        grid = grid[..., [2, 0, 1]]
        if plane_features is None:
            plane_features = self.get_planes(2 * grid_res)
        grid = grid.to(device=plane_features.device, dtype=plane_features.dtype)
        shape = grid.shape
        feats = self.sample_from_planes(grid.reshape(-1, 3), plane_features=plane_features)
        return self.lbound, feats.view(*shape[:-1], -1), grid


def kplanes_init_mul(x):
    """:442-444 -- uniform in [-1, 1): multiplied planes must not start near zero."""
    return 2 * torch.rand_like(x) - 1


class KPlaneVolume(nn.Module):
    """:445-489 -- `levels` plain tri-planes of side base_resolution * 2^l."""

    def __init__(self, base_resolution, levels, channels, features_mode, func_init=False):
        super().__init__()
        assert levels >= 1
        assert features_mode in ['mul', 'concatination']   # (sic)
        self.features_mode = features_mode
        tri = []
        for lvl in range(levels):
            res = base_resolution * (2 ** lvl)
            tri.append(TriPlaneVolume(number_of_features=channels, plane_resolution=res, init_sigma=0.1, lbound=1,
                                      viewdir_plane_resolution=-1, apply_activation_on_features=False, inner_multi_res_scale=1,
                                      inner_multi_res_scale_current=1, low_res_scale=1, high_res_scale=1, wavelet_type='haar',
                                      wavelet_base_resolution=res,
                                      init_fn=None if (features_mode == 'concatination' and not func_init) else kplanes_init_mul))
        self.triplane_lst = nn.ModuleList(tri)
        self.n_output_dims = levels * channels * (3 if features_mode == 'concatination' else 1)
        self.output_dim = self.n_output_dims
        self.n_input_dims = 3
        self.channels = channels

    def forward(self, coordinates, bound=None):
        res = []
        for tri in self.triplane_lst:
            f = tri(coordinates, bound=bound)
            if self.features_mode == 'mul':
                f = f.view(f.shape[0], 3, self.channels)
                f = f[:, 0] * f[:, 1] * f[:, 2]
            res.append(f)
        return torch.cat(res, dim=-1)


class _Multiscale(nn.Module):
    def __init__(self, base_resolution, low_res_levels, high_res_levels, channels, features_mode, func_init):
        super().__init__()
        assert high_res_levels >= low_res_levels
        self.low_res_vol = KPlaneVolume(base_resolution, low_res_levels, channels, features_mode, func_init=func_init)
        self.high_res_vol = KPlaneVolume(base_resolution * (2 ** low_res_levels), high_res_levels - low_res_levels, channels,
                                         features_mode, func_init=func_init)
        self.enable_cache = True
        self.double_mode = False
        self.resolution_mode = 'low_res'
        self.n_input_dims = 3

    def reset_cahce(self):  # (sic)
        pass

    def set_double_mode(self, val):
        self.double_mode = val

    def set_resolution_mode(self, val):
        assert val in ['low_res', 'high_res']
        self.resolution_mode = val

    def get_planes(self):
        return torch.zeros(1, 3, 50, 50)     # placeholder the application only logs (:518, :556)

    def get_wavelet_features(self):
        return []

    def _high(self):
        return self.double_mode and self.resolution_mode == 'high_res'


class MultiscaleKPlaneVolume(_Multiscale):
    """:491-527."""

    def __init__(self, base_resolution, low_res_levels, high_res_levels, channels, features_mode):
        super().__init__(base_resolution, low_res_levels, high_res_levels, channels, features_mode, func_init=False)
        self.n_output_dims = self.low_res_vol.n_output_dims
        self.n_output_dims_high_res = self.low_res_vol.n_output_dims + self.high_res_vol.n_output_dims

    def forward(self, coordinates, bound=None):
        res = self.low_res_vol(coordinates, bound=bound)
        if self._high():
            res = torch.cat([res, self.high_res_vol(coordinates, bound=bound)], dim=-1)
        return res


class MultiscaleKPlaneMulVolume(_Multiscale):
    """:529-578 -- needs features_mode='concatination': the product over planes and levels is taken here."""

    def __init__(self, base_resolution, low_res_levels, high_res_levels, channels, features_mode):
        super().__init__(base_resolution, low_res_levels, high_res_levels, channels, features_mode, func_init=True)
        self.n_output_dims = channels * 3

    @staticmethod
    def mul_tensor(x):
        res = x[..., 0, :]
        for i in range(1, x.shape[-2]):
            res = res * x[..., i, :]
        return res

    def forward(self, coordinates, bound=None):
        res = self.low_res_vol(coordinates, bound=bound)
        res = self.mul_tensor(res.view(res.shape[0], -1, self.n_output_dims))
        if self._high():
            hi = self.high_res_vol(coordinates, bound=bound)
            res = res * self.mul_tensor(hi.view(res.shape[0], -1, self.n_output_dims))
        return res
