"""NeRFNetwork -- drop-in for reconstruction/nerf/network.py:10-243 with encoding='triplane_wavelet':
TriPlaneVolume encoder -> sigma MLP (3C -> H -> 16, ReLU, no bias) -> trunc_exp density + 15 geo features ->
color MLP ([SH16(d), geo] -> Hc -> Hc -> 3, sigmoid).  Same constructor arguments, sub-module / parameter names
(`encoder.*`, `sigma_net.{0,1}.weight`, `color_net.{0,1,2}.weight`), `forward`, `density`, `color`, `get_params`.

Under CUDA fp16 autocast (how every reference command trains, --fp16) the five nn.Linear calls, both
activations, trunc_exp and the SH encoder run as ONE fused tensor-core kernel per direction
(tnl_mlp_forward / tnl_mlp_backward) with the autocast rounding points reproduced.  Without autocast the
layers run as plain fp32 torch ops on the nn.Linear weights, exactly as the reference's would.
"""
import ctypes

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function

from . import _lib
from ._lib import MlpDims, call, ptr, stream
from .activation import trunc_exp
from .encoding import get_encoder
from .renderer import NeRFRenderer
from .triplane_encoder import gather_features, take_grad_buffer


def fused_dims_supported(in_dim, hidden, hidden_color):
    """the fused kernels cover the reference's configurations: C in {16, 32, 48}, hidden = hidden_color in {64, 128}
    (forward and backward; the 128-wide heads on the tcgen05 kernels of csrc/mlp_tc128.cu)"""
    return in_dim in (48, 96, 144) and hidden == hidden_color and hidden in (64, 128)


def pack_mlp_weights(dims, weights):
    lib = _lib.load()
    nbytes = lib.tnl_mlp_packed_bytes(ctypes.byref(dims))
    if nbytes == 0:
        raise RuntimeError("trinerflet_b200: unsupported MLP dimensions for the fused kernel")
    packed = torch.empty(nbytes, dtype=torch.uint8, device=weights[0].device)
    ws = [w.detach().contiguous().float() for w in weights]
    call("tnl_mlp_pack_weights", ctypes.byref(dims), *[ptr(w) for w in ws], ptr(packed), stream())
    return packed


_warned_library_path = False


def _warn_library_path(net, x):
    """The fused kernels implement the fp16-autocast arithmetic every reference command trains with (--fp16).  Outside CUDA fp16
    autocast, or with head sizes other than 64 / 128, the heads run the reference's literal op sequence through torch's
    library GEMMs: a documented precision switch, never silent."""
    global _warned_library_path
    if not _warned_library_path and x.is_cuda:
        import warnings
        why = ("MLP dimensions outside the fused kernels" if not fused_dims_supported(net.in_dim, net.hidden_dim, net.hidden_dim_color)
               else "no CUDA fp16 autocast is active")
        warnings.warn(f"trinerflet_b200.NeRFNetwork: {why}; the sigma/color heads run as plain torch ops (library GEMMs), not the "
                      "fused sm_100a kernels. Wrap the call in torch.autocast('cuda', dtype=torch.float16) as the reference's --fp16 does.")
        _warned_library_path = True


def _mlp_forward(feat, dirs, n_valid, W):
    """tnl_mlp_forward -> (sigma, rgb, fp32 contiguous dirs, packed weights, dims)"""
    dirs = dirs.detach().contiguous().float()
    M = feat.shape[0]
    dims = MlpDims(W[0].shape[1], W[0].shape[0], W[3].shape[0])
    packed = pack_mlp_weights(dims, W)
    sigma = torch.empty(M, device=feat.device, dtype=torch.float32)
    rgb = torch.empty(M, 3, device=feat.device, dtype=torch.float32)
    call("tnl_mlp_forward", ctypes.byref(dims), ptr(packed), ptr(feat), int(feat.dtype == torch.float16), ptr(dirs), M, ptr(n_valid),
         ptr(sigma), ptr(rgb), None, stream())
    return sigma, rgb, dirs, packed, dims


class _FieldMLP(Function):
    """(feat [M,3C], dirs [M,3]) -> sigma [M] fp32, rgb [M,3] fp32 (fp16-representable values).  When dirs require grad the
    backward is tnl_mlp_backward_dirs, which also returns their gradient."""

    @staticmethod
    def forward(ctx, feat, dirs, n_valid, W1, W2, W3, W4, W5):
        feat = feat.contiguous()
        ctx.in_dtype = feat.dtype
        ctx.dirs_dtype = dirs.dtype
        if W1.shape[0] != 64:
            feat = feat.half()          # 128-wide heads: tcgen05 kernels only, fp16 feature stream (the first Linear's own rounding)
        elif feat.dtype != torch.float16:
            feat = feat.float()
        sigma, rgb, dirs, packed, dims = _mlp_forward(feat, dirs, n_valid, (W1, W2, W3, W4, W5))
        ctx.save_for_backward(feat, dirs, packed, n_valid if n_valid is not None else torch.empty(0))
        ctx.dims = (dims.in_dim, dims.hidden, dims.hidden_c, n_valid is not None)
        ctx.wshapes = [tuple(w.shape) for w in (W1, W2, W3, W4, W5)]
        return sigma, rgb

    @staticmethod
    def backward(ctx, g_sigma, g_rgb):
        feat, dirs, packed, n_valid = ctx.saved_tensors
        in_dim, hidden, hidden_c, has_nv = ctx.dims
        dims = MlpDims(in_dim, hidden, hidden_c)
        M = feat.shape[0]
        g_sigma = g_sigma.contiguous().float()
        g_rgb = g_rgb.contiguous().float()
        g_feat = torch.empty_like(feat)
        gW = [torch.zeros(s, device=feat.device, dtype=torch.float32) for s in ctx.wshapes]
        args = (ctypes.byref(dims), ptr(packed), ptr(feat), int(feat.dtype == torch.float16), ptr(dirs), M,
                ptr(n_valid) if has_nv else None, ptr(g_sigma), ptr(g_rgb), ptr(g_feat), *[ptr(g) for g in gW])
        g_dirs = None
        if ctx.needs_input_grad[1]:
            g_dirs = torch.empty(M, 3, device=feat.device, dtype=torch.float32)
        if _lib.deterministic():
            # the same kernels with the weight gradients reduced over per-CTA slots in a fixed order
            nbytes = _lib.load().tnl_mlp_backward_det_workspace(ctypes.byref(dims), int(feat.dtype == torch.float16), M)
            ws = _lib.workspace("mlp_backward_det", nbytes, feat.device)
            call("tnl_mlp_backward_det", *args, ptr(g_dirs), ptr(ws), ws.numel(), stream())
        elif g_dirs is not None:
            call("tnl_mlp_backward_dirs", *args, ptr(g_dirs), stream())
        else:
            call("tnl_mlp_backward", *args, stream())
        if g_dirs is not None:
            g_dirs = g_dirs.to(ctx.dirs_dtype)
        # (rows >= *n_valid of g_feat are never read: the sampling backward skips them with the same counter)
        if g_feat.dtype != ctx.in_dtype:
            g_feat = g_feat.to(ctx.in_dtype)
        return (g_feat, g_dirs, None, *gW)


class _Field(Function):
    """The field of a training step on the fused path (fp16 autocast, 64-wide heads, cell-sorted samples): (planes [3,C,R,R],
    coords [M,3], dirs [M,3], W1..W5) -> sigma [M], rgb [M,3].  The forward makes the two calls of the unfused path (plane gather
    in cell order into fp16 features, tnl_mlp_forward), so it computes the same bits; the backward is ONE
    tnl_mlp_backward_scatter, which scatters the feature gradient into the planes from inside the MLP backward instead of
    writing it out and reading it back.  Same gradient-buffer contract as _SamplePlanes (grad_buf of prefetch_planes)."""

    @staticmethod
    def forward(ctx, planes, coords, dirs, bound, n_valid, perm, grad_buf, W1, W2, W3, W4, W5):
        ctx.grad_buf = grad_buf
        # fp16 coordinates: the path runs under fp16 autocast, which rounds the projected coordinates (sample_planes)
        feat, coords, ctx.meta = gather_features(planes, coords, bound, True, n_valid, perm, True)
        sigma, rgb, dirs, packed, dims = _mlp_forward(feat, dirs, n_valid, (W1, W2, W3, W4, W5))
        ctx.save_for_backward(feat, coords, dirs, packed, n_valid if n_valid is not None else torch.empty(0), perm)
        ctx.dims = (dims.in_dim, dims.hidden, dims.hidden_c)
        ctx.wshapes = [tuple(w.shape) for w in (W1, W2, W3, W4, W5)]
        return sigma, rgb

    @staticmethod
    def backward(ctx, g_sigma, g_rgb):
        feat, coords, dirs, packed, n_valid, perm = ctx.saved_tensors
        M, R, C, inv, fp16_coords, has_nv, _, _ = ctx.meta
        dims = MlpDims(*ctx.dims)
        g_planes, external, plane_hook = take_grad_buffer(ctx, C, R, feat.device)
        assert plane_hook is None, "the plane-by-plane exchange scatters through _SamplePlanes"
        g_sigma = g_sigma.contiguous().float()
        g_rgb = g_rgb.contiguous().float()
        gW = [torch.zeros(s, device=feat.device, dtype=torch.float32) for s in ctx.wshapes]
        call("tnl_mlp_backward_scatter", ctypes.byref(dims), ptr(packed), ptr(feat), ptr(dirs), M, ptr(n_valid) if has_nv else None,
             ptr(perm), ptr(g_sigma), ptr(g_rgb), ptr(coords), R, C, inv, fp16_coords, ptr(g_planes), *[ptr(g) for g in gW], stream())
        return (None if external else g_planes, None, None, None, None, None, None, *gW)


class _DensityMLP(Function):
    """feat -> sigma [M], geo [M,15]; forward only (the density grid update runs under no_grad)."""

    @staticmethod
    def forward(ctx, feat, W1, W2, W3, W4, W5):
        feat = feat.contiguous()
        if feat.dtype != torch.float16:
            feat = feat.float()
        M = feat.shape[0]
        dims = MlpDims(W1.shape[1], W1.shape[0], W4.shape[0])
        packed = pack_mlp_weights(dims, (W1, W2, W3, W4, W5))
        sigma = torch.empty(M, device=feat.device, dtype=torch.float32)
        geo = torch.empty(M, 15, device=feat.device, dtype=torch.float32)
        call("tnl_mlp_forward", ctypes.byref(dims), ptr(packed), ptr(feat), int(feat.dtype == torch.float16), None, M, None,
             ptr(sigma), None, ptr(geo), stream())
        ctx.mark_non_differentiable(sigma, geo)
        return sigma, geo

    @staticmethod
    def backward(ctx, *g):
        raise RuntimeError("trinerflet_b200: density() is forward-only on the fused path")


class NeRFNetwork(NeRFRenderer):
    def __init__(self, encoding="triplane_wavelet", encoding_dir="sphere_harmonics", encoding_bg="hashgrid",
                 num_layers=2, hidden_dim=64, geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64, num_layers_bg=2,
                 hidden_dim_bg=64, bound=1, density_blob_scale=0, density_blob_std=0.5, mlp_weight_decay=0,
                 nerfacc_renderer=False, **kwargs):
        super().__init__(bound, **kwargs)
        if encoding != "triplane_wavelet" or encoding_dir != "sphere_harmonics":
            raise NotImplementedError("trinerflet_b200.NeRFNetwork covers encoding='triplane_wavelet' + SH directions")
        if num_layers != 2 or num_layers_color != 3 or geo_feat_dim != 15:
            raise NotImplementedError("MLP depth / geo_feat_dim other than the reference defaults (2 / 3 / 15)")
        if density_blob_scale > 1e-5 or nerfacc_renderer:
            raise NotImplementedError("density_blob / nerfacc renderer are outside the hot path")
        self.num_layers, self.hidden_dim, self.geo_feat_dim = num_layers, hidden_dim, geo_feat_dim
        self.encoder, self.in_dim = get_encoder(encoding, desired_resolution=2048 * bound, bound=bound, **kwargs)
        self.sigma_net = nn.ModuleList([nn.Linear(self.in_dim, hidden_dim, bias=False),
                                        nn.Linear(hidden_dim, 1 + geo_feat_dim, bias=False)])
        self.num_layers_color, self.hidden_dim_color = num_layers_color, hidden_dim_color
        self.encoder_dir, self.in_dim_dir = get_encoder(encoding_dir)
        self.color_net = nn.ModuleList([nn.Linear(self.in_dim_dir + geo_feat_dim, hidden_dim_color, bias=False),
                                        nn.Linear(hidden_dim_color, hidden_dim_color, bias=False),
                                        nn.Linear(hidden_dim_color, 3, bias=False)])
        self.bg_net = None
        self.density_blob_scale = density_blob_scale
        self.density_blob_std = density_blob_std
        self.mlp_weight_decay = mlp_weight_decay

    # ------------------------------------------------------------------------------------------
    def _weights(self):
        return (self.sigma_net[0].weight, self.sigma_net[1].weight, self.color_net[0].weight, self.color_net[1].weight,
                self.color_net[2].weight)

    def _fused(self):
        return (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.float16
                and fused_dims_supported(self.in_dim, self.hidden_dim, self.hidden_dim_color))

    # visit the samples of a training step in the order of a coarse 3-D grid (L2 locality of the plane gather /
    # gradient scatter, see csrc/sort.cu); per-point results do not depend on it
    spatial_sort_min_points = 1 << 18

    def forward(self, x, d, n_valid=None):
        """x [M,3] in [-bound, bound], d [M,3] unit dirs -> sigma [M] fp32, color [M,3]."""
        perm = None
        if x.is_cuda and x.shape[0] >= self.spatial_sort_min_points and torch.is_grad_enabled():
            from .triplane_encoder import cell_sort
            perm = cell_sort(x, self.bound, n_valid, 64)
        fused = self._fused()
        if (fused and perm is not None and self.hidden_dim == 64 and self.in_dim in (48, 96)
                and self.encoder.scatter_plane_hook is None and not x.requires_grad and not d.requires_grad
                and not _lib.deterministic()):
            # training step: one fused MLP-backward + plane scatter (the plane-by-plane exchange of the multi-GPU step scatters
            # through _SamplePlanes instead; input gradients go through _SamplePlanes / _FieldMLP; deterministic mode takes
            # _SamplePlanes + _FieldMLP, whose results per row do not depend on perm)
            planes, gbuf = self.encoder.planes_and_grad_buffer()
            return _Field.apply(planes, x, d, self.bound, n_valid, perm, gbuf, *self._weights())
        # fused path: the feature stream between the gather and the MLP kernels is fp16 (the first Linear's own rounding)
        feat = self.encoder(x, bound=self.bound, n_valid=n_valid, perm=perm, half_out=fused)
        if fused:
            return _FieldMLP.apply(feat, d, n_valid, *self._weights())
        _warn_library_path(self, x)
        # reference op sequence (network.py:125-147); precision follows the ambient autocast state
        h = F.relu(self.sigma_net[0](feat))
        h = self.sigma_net[1](h)
        sigma = trunc_exp(h[..., 0])
        geo_feat = h[..., 1:]
        h = torch.cat([self.encoder_dir(d), geo_feat], dim=-1)
        h = F.relu(self.color_net[0](h))
        h = F.relu(self.color_net[1](h))
        color = torch.sigmoid(self.color_net[2](h))
        return sigma, color

    def density(self, x):
        fused = not torch.is_grad_enabled() and self._fused()
        feat = self.encoder(x, bound=self.bound, half_out=fused)
        if fused:
            sigma, geo = _DensityMLP.apply(feat, *self._weights())
            return {'sigma': sigma, 'geo_feat': geo}
        h = F.relu(self.sigma_net[0](feat))
        h = self.sigma_net[1](h)
        return {'sigma': trunc_exp(h[..., 0]), 'geo_feat': h[..., 1:]}

    def color(self, x, d, mask=None, geo_feat=None, **kwargs):
        """network.py:186-214 (only the non-cuda_ray sampler calls it; kept for API completeness)."""
        if mask is not None:
            rgbs = torch.zeros(mask.shape[0], 3, dtype=x.dtype, device=x.device)
            if not mask.any():
                return rgbs
            d, geo_feat = d[mask], geo_feat[mask]
        h = torch.cat([self.encoder_dir(d), geo_feat], dim=-1)
        h = F.relu(self.color_net[0](h))
        h = F.relu(self.color_net[1](h))
        h = torch.sigmoid(self.color_net[2](h))
        if mask is not None:
            rgbs[mask] = h.to(rgbs.dtype)
            return rgbs
        return h

    def get_params(self, lr):
        """network.py:217-243."""
        params = [{'params': self.encoder.parameters(), 'lr': lr}, {'params': self.encoder_dir.parameters(), 'lr': lr}]
        extra = {'weight_decay': self.mlp_weight_decay} if self.mlp_weight_decay > 0 else {}
        params += [{'params': self.sigma_net.parameters(), 'lr': lr, **extra},
                   {'params': self.color_net.parameters(), 'lr': lr, **extra}]
        return params
