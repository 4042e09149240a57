"""TriPlaneVolume -- drop-in for reconstruction/triplaneencoder/triplane_encoder.py:26-530 on the path every
README command uses (wavelet-parameterised planes, all levels learnable, no rotation / dropout / auto-scale / upscale),
with every wavelet of the reference's pad table (bior6.8, the README's choice, and bior2.6, bior4.4, bior2.2, haar).  Same constructor kwargs, attributes, method names and state-dict keys:

    planes_features                    logical [3, C, n0, n0]
    planes_features_wavelet_coefs.{l}  logical [3, C, 3, n0*2^l, n0*2^l]
    plane_axes [3,3,2], plane_normals [3,3,1] (buffers)

B200-first differences (DESIGN.md "data layout"):
  * parameters, gradients and planes keep the reference's logical shapes but are STORED channels-last
    (C fastest: strides of a `[3,n,n,C]` / `[3,3,n,n,C]` tensor permuted back), so that one texel's C features are
    one contiguous run for the sampling gather/scatter and pixel rows are contiguous for the IDWT kernels;
    `load_state_dict` / `state_dict` / optimizers are stride-agnostic, so reference checkpoints load unchanged;
  * `build_planes` is one fused CUDA kernel per level (tnl_idwt_level_forward) instead of 2 pads +
    6 conv_transpose2d + 3 adds per level; its backward is the exact adjoint kernel;
  * `sample_from_planes` is one gather kernel (tnl_sample_planes_forward); backward one scatter kernel.
There is no CPU path: tensors must be CUDA tensors.
"""
import math

import numpy as np
import torch
import torch.nn as nn
from torch.autograd import Function

from . import _lib
from ._lib import call, ptr, stream
from .idwt_plan import idwt_call

PAD_DICT = {'bior6.8': 4, 'bior2.6': 3, 'bior4.4': 2, 'bior2.2': 1, 'haar': 0}  # triplane_encoder.py:174-180


def get_levels(upscale_factor):
    """reconstruction/triplaneencoder/utils.py:274-279."""
    wavelet_levels = math.log2(upscale_factor)
    if abs(wavelet_levels - round(wavelet_levels)) > 1e-5:
        raise ValueError('Unsupported res. should be 2^')
    return round(wavelet_levels)


# ----------------------------------------------------------------------------------------------
# channels-last helpers
# ----------------------------------------------------------------------------------------------
def cl_empty_planes(C, n, device=None, dtype=torch.float32, zero=False):
    """Logical [3, C, n, n] tensor stored as [3][n][n][C]."""
    f = torch.zeros if zero else torch.empty
    return f(3, n, n, C, device=device, dtype=dtype).permute(0, 3, 1, 2)


def cl_empty_coefs(C, n, device=None, dtype=torch.float32, zero=False):
    """Logical [3, C, 3, n, n] tensor stored as [3][3][n][n][C]."""
    f = torch.zeros if zero else torch.empty
    return f(3, 3, n, n, C, device=device, dtype=dtype).permute(0, 4, 1, 2, 3)


def is_cl_planes(t):
    return t.dim() == 4 and t.permute(0, 2, 3, 1).is_contiguous()


def is_cl_coefs(t):
    return t.dim() == 5 and t.permute(0, 2, 3, 4, 1).is_contiguous()


def to_cl_planes(t):
    if is_cl_planes(t):
        return t
    out = cl_empty_planes(t.shape[1], t.shape[2], device=t.device, dtype=t.dtype)
    out.copy_(t)
    return out


def to_cl_coefs(t):
    if is_cl_coefs(t):
        return t
    out = cl_empty_coefs(t.shape[1], t.shape[3], device=t.device, dtype=t.dtype)
    out.copy_(t)
    return out


def _require_cuda_f32(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"trinerflet_b200: {what} must be a CUDA tensor (no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"trinerflet_b200: {what} must be float32")


# ----------------------------------------------------------------------------------------------
# multilevel inverse DWT  (build_planes, triplane_encoder.py:364-405)
# ----------------------------------------------------------------------------------------------
class _BuildPlanes(Function):
    """planes = IDWT_L(...IDWT_1(2*x0, yh_0)..., yh_{L-1}) with the wavelet's zero padding per level, plus abs_sums[l] = sum|yh_l|
    (the forward value of the wavelet L1 regulariser, a free by-product of the pass that reads yh).  Linear in all
    inputs, so backward needs no saved activations: it is the chain of adjoint level kernels, with the regulariser
    gradient  g_abs[l] * sign(yh_l)  folded into the coefficient-gradient store."""

    @staticmethod
    def forward(ctx, planes_features, plan, wave, *coefs):
        """plan: None = dense (reference semantics); an idwt_plan.IdwtPlan = reconstruct only the blocks the training-step
        sampler reads (the rest of the returned planes is undefined) and restrict the adjoint to where gradient arrives."""
        _require_cuda_f32(planes_features, "planes_features")
        x = to_cl_planes(planes_features.detach())
        C, n = x.shape[1], x.shape[2]
        ctx.n0, ctx.C, ctx.levels = n, C, len(coefs)
        if plan is not None and (plan.levels != len(coefs) or plan.n0 != n or plan.C != C):
            raise RuntimeError("IdwtPlan does not match the encoder geometry")
        ctx.plan, ctx.wave = plan, wave
        ctx.set_materialize_grads(False)   # an unused abs_sums output must not cost a pass over the coefficients
        # deterministic mode: the kernels' per-CTA atomic |yh| sums are replaced by torch's deterministic reductions (below)
        det = _lib.deterministic()
        abs_sums = torch.zeros(max(len(coefs), 1), device=x.device, dtype=torch.float32)
        saved = []
        for l, yh in enumerate(coefs):
            _require_cuda_f32(yh, "wavelet coefficients")
            if yh.shape != (3, C, 3, n, n):
                raise RuntimeError(f"wavelet level has shape {tuple(yh.shape)}, expected {(3, C, 3, n, n)}")
            yh = to_cl_coefs(yh.detach())
            saved.append(yh)
            out = cl_empty_planes(C, 2 * n, device=x.device)
            a = None if det else abs_sums[l:l + 1]
            if plan is None:
                idwt_call("tnl_idwt_level_forward", wave, ptr(x), ptr(yh), ptr(out), n, C, ptr(a), stream())
            else:
                plan.forward_level(l, x, yh, out, n, a, parts=1, wave=wave)
            x, n = out, 2 * n
        if plan is not None:
            if plan.on_planes_ready is not None and plan.defer_clean_abs:
                plan.on_planes_ready()               # the planes are complete and nothing else of this call is awaited
            plan.on_planes_ready = None
            n = ctx.n0
            for l, yh in enumerate(saved if not det else []):   # |yh| of the blocks that were not reconstructed (regulariser value)
                if plan.defer_clean_abs:             # ... except those the backward's clean part will read anyway
                    plan.forward_gap_abs(l, yh, n, abs_sums[l:l + 1])
                else:
                    plan.forward_level(l, saved[l], yh, saved[l], n, abs_sums[l:l + 1], parts=2, wave=wave)   # x / out untouched
                n *= 2
        if det and saved:
            abs_sums = torch.stack([yh.abs().sum() for yh in saved])
        ctx.save_for_backward(*saved)
        return x, abs_sums

    @staticmethod
    def backward(ctx, g, g_abs):
        C = ctx.C
        n = ctx.n0 * (2 ** ctx.levels)
        yhs = ctx.saved_tensors
        if g is None:
            g = cl_empty_planes(C, n, device=yhs[0].device, zero=True)
        g = to_cl_planes(g)
        if g_abs is not None:
            g_abs = g_abs.contiguous().float()
        grads = []
        for l in reversed(range(ctx.levels)):
            n //= 2
            g_x = cl_empty_planes(C, n, device=g.device)
            g_yh = cl_empty_coefs(C, n, device=g.device)
            if ctx.plan is not None:
                if g_abs is not None:
                    ctx.plan.backward_level(l, g, g_x, g_yh, n, yhs[l], g_abs[l:l + 1], 1.0, wave=ctx.wave)
                else:
                    ctx.plan.backward_level(l, g, g_x, g_yh, n, None, None, 0.0, wave=ctx.wave)
            elif g_abs is not None:
                idwt_call("tnl_idwt_level_backward", ctx.wave, ptr(g), ptr(g_x), ptr(g_yh), n, C, ptr(yhs[l]), ptr(g_abs[l:l + 1]),
                          1.0, 0, 3, stream())
            else:
                idwt_call("tnl_idwt_level_backward", ctx.wave, ptr(g), ptr(g_x), ptr(g_yh), n, C, None, None, 0.0, 0, 3, stream())
            grads.append(g_yh)
            g = g_x
        return (g, None, None, *reversed(grads))


class PlanewiseIdwtBackward:
    """The adjoint of build_planes driven plane by plane (multi-GPU path): `run(plane)` pushes the gradient of one of the
    three planes through all levels, so plane p can be processed while the gradient of plane p+1 is still being
    exchanged.  Writes straight into freshly allocated .grad tensors of the encoder parameters."""

    def __init__(self, encoder, g_planes, reg_scale=None, reg_coef=0.0):
        self.enc = encoder
        self.C, self.levels = encoder.number_of_features, len(encoder.planes_features_wavelet_coefs)
        self.n0 = encoder.planes_features.shape[2]
        self.g = to_cl_planes(g_planes)
        self.reg_scale, self.reg_coef = reg_scale, float(reg_coef)
        dev = self.g.device
        self.g_x = [cl_empty_planes(self.C, self.n0 * 2 ** l, device=dev) for l in range(self.levels)]
        self.g_yh = [cl_empty_coefs(self.C, self.n0 * 2 ** l, device=dev) for l in range(self.levels)]

    def run(self, plane):
        g = self.g
        for l in reversed(range(self.levels)):
            n = self.n0 * 2 ** l
            yh = self.enc.planes_features_wavelet_coefs[l]
            use_reg = self.reg_scale is not None and self.reg_coef != 0.0
            idwt_call("tnl_idwt_level_backward", self.enc.wavelet_type, ptr(g), ptr(self.g_x[l]), ptr(self.g_yh[l]), n, self.C,
                      ptr(yh.detach()) if use_reg else None, ptr(self.reg_scale) if use_reg else None, self.reg_coef, plane, 1,
                      stream())
            g = self.g_x[l]

    def assign(self):
        """Install the results as parameter gradients (zero_grad(set_to_none=True) semantics)."""
        self.enc.planes_features.grad = self.g_x[0]
        for p, g in zip(self.enc.planes_features_wavelet_coefs, self.g_yh):
            p.grad = g


class SplitIdwtBackward:
    """The adjoint of a work-list plane reconstruction in two parts (multi-GPU path): `run_clean()` covers the blocks that
    receive no plane gradient (regulariser gradient / zeros only) and needs nothing from the render backward, so it runs
    while the plane gradient is still being exchanged between the ranks; `run_active(g_planes)` pushes the exchanged
    gradient through the remaining blocks.  `assign()` installs the results as parameter gradients."""

    def __init__(self, encoder, plan, reg_scale=None, reg_coef=0.0):
        self.enc, self.plan = encoder, plan
        self.C, self.levels = encoder.number_of_features, len(encoder.planes_features_wavelet_coefs)
        self.n0 = encoder.planes_features.shape[2]
        self.reg_scale, self.reg_coef = reg_scale, float(reg_coef)
        self.abs_sums = None   # [L] tensor the clean part completes with sum |yh| of its blocks (plan.defer_clean_abs)
        dev = encoder.planes_features.device
        self.g_x = [cl_empty_planes(self.C, self.n0 * 2 ** l, device=dev) for l in range(self.levels)]
        self.g_yh = [cl_empty_coefs(self.C, self.n0 * 2 ** l, device=dev) for l in range(self.levels)]

    def _level(self, l, g, parts):
        use_reg = self.reg_scale is not None and self.reg_coef != 0.0
        yh = self.enc.planes_features_wavelet_coefs[l].detach()
        abs_sum = self.abs_sums[l:l + 1] if (self.abs_sums is not None and (parts & 2)) else None
        self.plan.backward_level(l, g, self.g_x[l], self.g_yh[l], self.n0 * 2 ** l, yh if use_reg else None,
                                 self.reg_scale if use_reg else None, self.reg_coef, parts, abs_sum, wave=self.enc.wavelet_type)

    def run_clean(self):
        for l in range(self.levels):
            self._level(l, None, 2)
        self.clean_done = True

    def run_active(self, g_planes):
        g = to_cl_planes(g_planes)
        for l in reversed(range(self.levels)):
            self._level(l, g, 1)
            g = self.g_x[l]

    def assign(self):
        self.enc.planes_features.grad = self.g_x[0]
        for p, g in zip(self.enc.planes_features_wavelet_coefs, self.g_yh):
            p.grad = g


def build_planes_with_abs(planes_features, coefs, plan=None, wave='bior6.8'):
    """-> (planes [3,C,R,R], abs_sums [L] with abs_sums[l] = sum |coefs[l]|), both differentiable."""
    return _BuildPlanes.apply(planes_features, plan, wave, *coefs)


def build_planes(planes_features, coefs, plan=None, wave='bior6.8'):
    return _BuildPlanes.apply(planes_features, plan, wave, *coefs)[0]


# ----------------------------------------------------------------------------------------------
# tri-plane bilinear sampling (sample_from_planes_aux, triplane_encoder.py:314-332)
# ----------------------------------------------------------------------------------------------
def _inv_bound(bound):
    # CUDA evaluates `tensor / python_scalar` as tensor * fp32(1/scalar)
    return float(np.float32(1.0) / np.float32(bound))


def gather_features(planes, coords, bound, fp16_coords, n_valid, perm, half_out):
    """The plane gather (tnl_sample_planes_forward) -> (feat [M, 3C], the fp32 contiguous coords it read, meta tuple of the
    backward: M, R, C, inv_bound, fp16_coords, has n_valid, has perm, half_out)."""
    _require_cuda_f32(planes, "planes")
    planes_cl = to_cl_planes(planes.detach())
    coords = coords.detach().contiguous().float()
    M = coords.shape[0]
    C, R = planes.shape[1], planes.shape[2]
    feat = torch.empty(M, 3 * C, device=planes.device, dtype=torch.float16 if half_out else torch.float32)
    inv = _inv_bound(bound)
    call("tnl_sample_planes_forward", ptr(planes_cl), ptr(coords), M, R, C, inv, int(bool(fp16_coords)),
         ptr(n_valid), ptr(perm), ptr(feat), int(bool(half_out)), stream())
    return feat, coords, (M, R, C, inv, int(bool(fp16_coords)), n_valid is not None, perm is not None, bool(half_out))


def take_grad_buffer(ctx, C, R, device):
    """-> (g_planes, external, plane_hook): where a sampling backward scatters.  The buffer of ctx.grad_buf (zero-filled ahead of
    time on the prefetch stream, TriPlaneVolume.prefetch_planes) is taken once, after the current stream waits for it; without
    one a zero-filled channels-last buffer.  external: the caller owns the buffer and the backward returns no plane gradient.
    Sets ctx.grad_tiles: the idwt_plan.IdwtPlan tile list of a buffer zeroed only there, else None."""
    ctx.grad_tiles = None
    if ctx.grad_buf is None:
        return cl_empty_planes(C, R, device=device, zero=True), False, None
    g_planes, ready, external, plane_hook, ctx.grad_tiles = ctx.grad_buf
    ctx.grad_buf = None
    torch.cuda.current_stream().wait_event(ready)
    return g_planes, external, plane_hook


def scatter_planes(g_feat, half, coords, M, R, C, inv, fp16_coords, nv, pm, g_planes, tiles=None):
    """g_planes += the adjoint of the plane gather (tnl_sample_planes_backward).  In deterministic mode the fixed-point scatter
    tnl_sample_planes_backward_det, restricted to the tiles of `tiles` (an IdwtPlan.zero list) when given."""
    if not _lib.deterministic():
        call("tnl_sample_planes_backward", ptr(g_feat), int(half), ptr(coords), M, R, C, inv, fp16_coords, nv, pm, ptr(g_planes), stream())
        return
    nbytes = _lib.load().tnl_sample_planes_backward_det_workspace(R, C)
    ws = _lib.workspace("sample_planes_backward_det", nbytes, g_feat.device)
    ids, count, cap = (ptr(tiles["ids"]), ptr(tiles["count"]), tiles["cap"]) if tiles is not None else (None, None, 0)
    from .idwt_plan import TILE
    call("tnl_sample_planes_backward_det", ptr(g_feat), int(half), ptr(coords), M, R, C, inv, fp16_coords, nv, pm, ids, count, cap, TILE,
         ptr(g_planes), ptr(ws), ws.numel(), stream())


class _SamplePlanes(Function):
    @staticmethod
    def forward(ctx, planes, coords, bound, fp16_coords, n_valid, perm=None, half_out=False, grad_buf=None):
        ctx.grad_buf = grad_buf
        feat, coords, ctx.meta = gather_features(planes, coords, bound, fp16_coords, n_valid, perm, half_out)
        # the position gradient reads the planes (the gather's channels-last copy: no copy when they are stored that way)
        ctx.save_for_backward(coords, n_valid if n_valid is not None else torch.empty(0),
                              perm if perm is not None else torch.empty(0),
                              to_cl_planes(planes.detach()) if ctx.needs_input_grad[1] else None)
        return feat

    @staticmethod
    def backward(ctx, g_feat):
        coords, n_valid, perm, planes_cl = ctx.saved_tensors
        M, R, C, inv, fp16_coords, has_nv, has_perm, half = ctx.meta
        g_feat = g_feat.contiguous().half() if half else g_feat.contiguous().float()
        nv, pm = (ptr(n_valid) if has_nv else None), (ptr(perm) if has_perm else None)
        g_planes, external = None, False
        if ctx.needs_input_grad[0]:
            g_planes, external, plane_hook = take_grad_buffer(ctx, C, R, g_feat.device)
            if plane_hook is not None and C in (16, 32, 48):
                # multi-GPU step: plane by plane, so that the caller can start exchanging plane p while plane p + 1 scatters
                _lib.alert_nondeterministic("the plane-by-plane scatter of the multi-GPU step (tnl_sample_planes_backward_plane)")
                for p in range(3):
                    call("tnl_sample_planes_backward_plane", ptr(g_feat), int(half), ptr(coords), M, R, C, inv, fp16_coords, nv, pm,
                         ptr(g_planes), p, stream())
                    plane_hook(p)
            else:
                scatter_planes(g_feat, half, coords, M, R, C, inv, fp16_coords, nv, pm, g_planes, ctx.grad_tiles)
        g_xyz = None
        if ctx.needs_input_grad[1]:
            g_xyz = torch.empty(M, 3, device=g_feat.device, dtype=torch.float32)
            call("tnl_sample_planes_backward_xyz", ptr(g_feat), int(half), ptr(planes_cl), ptr(coords), M, R, C, inv, fp16_coords, nv, pm,
                 ptr(g_xyz), stream())
        # external: the caller's persistent (symmetric-memory) buffer holds the plane gradient; autograd must not clone 1.6 GB of it
        return None if external else g_planes, g_xyz, None, None, None, None, None, None


def cell_sort(coords, bound, n_valid=None, G=64):
    """perm [M] int32: visit order of the points by a G^3 Morton grid (tnl_cell_sort)."""
    from . import _lib
    coords = coords.detach().contiguous().float()
    M = coords.shape[0]
    perm = torch.empty(M, dtype=torch.int32, device=coords.device)
    ws = torch.empty(max(int(_lib.load().tnl_cell_sort_workspace(M, G)), 16), dtype=torch.uint8, device=coords.device)
    call("tnl_cell_sort", ptr(coords), M, ptr(n_valid), _inv_bound(bound), G, ptr(perm), ptr(ws), ws.numel(), stream())
    return perm


def sample_planes(planes, coords, bound, fp16_coords=None, n_valid=None, perm=None, half_out=False, grad_buf=None):
    """planes logical [3,C,R,R] -> features [M, 3C] (fp32). fp16_coords=None follows the autocast state, as the
    reference's projection matmul does (SURVEY.md 8a-2)."""
    if fp16_coords is None:
        fp16_coords = torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.float16
    return _SamplePlanes.apply(planes, coords, float(bound), bool(fp16_coords), n_valid, perm, bool(half_out), grad_buf)


# ----------------------------------------------------------------------------------------------
# module
# ----------------------------------------------------------------------------------------------
class TriPlaneVolume(nn.Module):
    def __init__(self, number_of_features=3, plane_resolution=224, init_sigma=0.1, lbound=1,
                 viewdir_plane_resolution=32, two_planes_per_axis=False, planes_features=None, viewdir_plane=None,
                 apply_activation_on_features=False, inner_multi_res_scale=1, inner_multi_res_viewdir_scale=1,
                 viewdir_mode='plane', inner_multi_res_scale_current=1, learn_rotation_axis=False, dropout=0,
                 wavelet_type='bior6.8', lbound_auto_scale=False, upscale_ratio_bound=-1, upscale_levels=2,
                 wavelet_base_resolution=0):
        super().__init__()
        unsupported = []
        if two_planes_per_axis: unsupported.append("two_planes_per_axis")
        if apply_activation_on_features: unsupported.append("apply_activation_on_features")
        if learn_rotation_axis: unsupported.append("learn_rotation_axis")
        if 0 < dropout < 1: unsupported.append("dropout")
        if lbound_auto_scale: unsupported.append("lbound_auto_scale")
        if 0 < upscale_ratio_bound < 1: unsupported.append("upscale_ratio_bound")
        if wavelet_base_resolution not in (0,): unsupported.append("wavelet_base_resolution")
        if inner_multi_res_scale_current != 1: unsupported.append("inner_multi_res_scale_current != 1")
        if inner_multi_res_scale > 1 and wavelet_type not in PAD_DICT: unsupported.append(f"wavelet_type={wavelet_type}")
        if unsupported:
            raise NotImplementedError("trinerflet_b200.TriPlaneVolume: options outside the hot path (no reference config "
                                      f"uses them, SURVEY.md 8a-2): {unsupported}")
        self.number_of_features = number_of_features
        self.plane_resolution = plane_resolution
        self.init_sigma = init_sigma
        self.lbound = lbound
        self.lbound_viewdir = 1
        self.output_dim = 3 * number_of_features
        self.viewdir_plane_resolution = viewdir_plane_resolution
        self.two_planes_per_axis = False
        self.apply_activation_on_features = False
        self.wavelet_type = wavelet_type
        self.inner_wavelet_scale = inner_multi_res_scale
        self.inner_wavelet_viewdir_scale = inner_multi_res_viewdir_scale
        self.inner_multi_res_scale_current = inner_multi_res_scale_current
        self.wavelet_base_resolution = wavelet_base_resolution
        self.learn_rotation_axis = False
        self.rotation_matrix = None
        self.dropout = None
        self.lbound_auto_scale = False
        self.lbound_scale = None
        self.upscale_ratio_bound = upscale_ratio_bound
        self.upscale_levels = upscale_levels
        self.upscale_enabled = False
        self.plane_direction = ['up', 'front', 'right']

        # plane bases, triplane_encoder.py:250-289 : up=(x,z), front=(x,y), right=(y,z)
        eye = torch.eye(3)
        axes = torch.stack([torch.cat([eye[:, 0:1], eye[:, 2:3]], dim=1),
                            torch.cat([eye[:, 0:1], eye[:, 1:2]], dim=1),
                            torch.cat([eye[:, 1:2], eye[:, 2:3]], dim=1)], dim=0)
        normals = torch.stack([eye[:, 1:2], eye[:, 2:3], eye[:, 0:1]], dim=0)
        self.register_buffer('plane_axes', axes.clone())
        self.register_buffer('plane_normals', normals.clone())

        self.last_used_planes = None
        self._last_abs_sums = None
        # training hot path only: an idwt_plan.IdwtPlan restricts the next reconstructions to the occupied tiles
        # (see idwt_plan.py); None = dense planes, the reference's semantics
        self.idwt_plan = None
        self.external_grad_buffer = None      # set by the multi-GPU training step: where the sampling backward scatters (see prefetch_planes)
        self.scatter_plane_hook = None        # ... and a callback after each plane's scatter (starts that plane's exchange)
        self._init_plane_features(planes_features)

    # -- parameters (triplane_encoder.py:155-231) --------------------------------------------------
    def _init_plane_features(self, planes_features):
        C, R = self.number_of_features, self.plane_resolution
        if self.inner_wavelet_scale <= 1:
            levels, n0 = 0, R
        else:
            levels = get_levels(self.inner_wavelet_scale)
            if R % (2 ** levels) != 0:
                raise ValueError("plane_resolution must be divisible by the wavelet upscale factor")
            n0 = R // (2 ** levels)
        self.planes_features_wavelet_all_level = levels
        self.planes_features_wavelet_current_level = 0
        self.planes_features_wavelet_pad = PAD_DICT.get(self.wavelet_type, 0)
        self.planes_features_wavelet_yh_shapes = [torch.Size([3, C, 3, n0 * 2 ** l, n0 * 2 ** l]) for l in range(levels)]
        if planes_features is None:
            planes_features = self.init_sigma * torch.randn(3, C, n0, n0)  # same RNG call as the reference (:212 / :162)
        base = cl_empty_planes(C, n0)
        base.copy_(planes_features.detach())
        self.planes_features = nn.Parameter(base)
        coefs = []
        for l in range(levels):
            coefs.append(nn.Parameter(cl_empty_coefs(C, n0 * 2 ** l, zero=True)))  # zero-init, :220
        self.planes_features_wavelet_coefs = nn.ParameterList(coefs)

    def _apply(self, fn, *args, **kwargs):
        # nn.Module._apply (e.g. .to(device)) preserves strides for dense non-overlapping tensors; nothing to do,
        # but drop the plane cache because it lives on the old device.
        self.last_used_planes = None
        return super()._apply(fn, *args, **kwargs)

    # -- reference API -----------------------------------------------------------------------------
    def get_wavelet_features(self):
        return list(self.planes_features_wavelet_coefs) if self.inner_wavelet_scale > 1 else []

    def get_wavelet_features_upscaled(self):
        return []

    def get_lbound_scale(self):
        return None

    def get_params(self, opt_cfg):
        return self.parameters()

    def get_params2(self, lr):
        return [{'params': [], 'lr': 10 * lr}, {'params': list(self.parameters()), 'lr': lr}]

    def reset_cahce(self):  # (sic) -- reference spelling, nerf/utils.py:1139,1162
        self.last_used_planes = None
        self._last_abs_sums = None

    reset_cache = reset_cahce

    def prefetch_planes(self, side, partial_zero=False):
        """Reconstruct the planes on stream `side` while the caller's stream goes on with work that does not need them
        (ray marching, the cell sort); the first sampling call waits for them.  Also zero-fills the plane-gradient buffer
        of this step's sampling backward there.  Same result as get_planes(); the autograd node of the reconstruction
        runs its backward on `side` too (torch's stream-aware engine orders it after the sampling backward)."""
        main = torch.cuda.current_stream()
        side.wait_stream(main)
        plan = self.idwt_plan
        with torch.cuda.stream(side):
            ready = torch.cuda.Event()
            fired = []
            if plan is not None:
                plan.on_planes_ready = lambda: (ready.record(side), fired.append(1))
            planes = self.get_planes()
            if not fired:
                ready.record(side)
            gbuf = None
            if torch.is_grad_enabled() and planes.requires_grad:
                ext = self.external_grad_buffer     # multi-GPU: the persistent symmetric-memory buffer of parallel.PeerGradExchange
                if plan is not None and partial_zero:
                    # the work-list backward only reads the tiles around the occupied ones: zero those, leave the rest undefined
                    gbuf = ext if ext is not None else cl_empty_planes(self.number_of_features, self.plane_resolution, device=planes.device)
                    plan.zero_gradient_tiles(gbuf.permute(0, 2, 3, 1))
                elif ext is not None:
                    gbuf = ext
                    gbuf.zero_()
                else:
                    gbuf = cl_empty_planes(self.number_of_features, self.plane_resolution, device=planes.device, zero=True)
                gready = torch.cuda.Event()
                gready.record(side)
                gbuf = (gbuf, gready, ext is not None, self.scatter_plane_hook if ext is not None else None,
                        plan.zero if (plan is not None and partial_zero) else None)
        self._prefetch = (ready, gbuf)
        return planes

    def _join_prefetch(self):
        """-> the pre-zeroed gradient buffer (once per prefetch) after making the current stream wait for the planes."""
        pf = getattr(self, "_prefetch", None)
        if pf is None:
            return None
        ready, gbuf = pf
        torch.cuda.current_stream().wait_event(ready)
        self._prefetch = None
        return gbuf

    def build_planes(self, planes_features=None, coefs=None):
        planes_features = self.planes_features if planes_features is None else planes_features
        coefs = list(self.planes_features_wavelet_coefs) if coefs is None else coefs
        if self.inner_wavelet_scale <= 1 or len(coefs) == 0:
            return planes_features
        planes, abs_sums = build_planes_with_abs(planes_features, coefs, self.idwt_plan, self.wavelet_type)
        self._last_abs_sums = abs_sums
        return planes

    def get_planes(self, max_res=-1, max_scale=-1, get_all_resolutions=False):
        if self.last_used_planes is not None:
            return self.last_used_planes               # whatever the arguments, as the reference (:409-410)
        if max_res > 0 or max_scale > 0 or get_all_resolutions:
            return self._get_planes_limited(max_res, max_scale, get_all_resolutions)
        planes = self.build_planes()
        if isinstance(planes, nn.Parameter):           # no wavelet levels: cache an alias (assigning a Parameter would register it)
            planes = planes.view_as(planes)
        self.last_used_planes = planes
        return planes

    def _get_planes_limited(self, max_res, max_scale, get_all_resolutions):
        """The coarser / per-level readings of build_planes (:376-398), used by the reference's tooling (save_triplane,
        nerf/utils.py:1649; get_grid_features, :500), not by a training step: the level loop stops at the first level whose input
        side has reached `max_res` or whose accumulated upscale factor has reached `max_scale`, and the planes come back at that
        side; `get_all_resolutions` returns the input of every level visited and the final planes (after a stop the last entry
        appears twice, as in the reference).  Dense, level by level."""
        x, all_res, scale = self.planes_features, [], 1
        if self.inner_wavelet_scale > 1:
            for yh in self.planes_features_wavelet_coefs:
                if get_all_resolutions:
                    all_res.append(x)
                if (max_res > 0 and min(x.shape[2:]) >= max_res) or (max_scale > 0 and scale >= max_scale):
                    break
                x = build_planes(x, [yh], wave=self.wavelet_type)
                scale *= 2
            if get_all_resolutions:
                all_res.append(x)
        if isinstance(x, nn.Parameter):                # stopped before the first level: cache an alias, not the Parameter itself
            x = x.view_as(x)
            if get_all_resolutions:
                all_res[-1] = x
        self.last_used_planes = x
        self._last_abs_sums = None
        return all_res if get_all_resolutions else x

    def wavelet_l1(self, lam, abs_sums=None):
        """lam * (sum_l mean|yh_l| * numel_l / numel_all) / L -- the regulariser of nerf/utils.py:640-655 (unweighted
        branch), taken from the |yh| sums the plane reconstruction produced; its gradient is applied inside the IDWT
        backward kernels (no extra pass over the coefficients).  Call after get_planes() of the same step, or pass the
        |yh| sums of that reconstruction."""
        self._join_prefetch()
        feats = self.get_wavelet_features()
        if len(feats) == 0:
            return None
        if abs_sums is None:
            if self.last_used_planes is None or getattr(self, "_last_abs_sums", None) is None:
                self.get_planes()
            abs_sums = self._last_abs_sums
            if abs_sums is None:      # the cached planes came from a band-limited query, which keeps no |yh| sums
                abs_sums = torch.stack([v.abs().sum() for v in feats])
        total = sum(v.numel() for v in feats)
        return lam * abs_sums.sum() / (total * len(feats))

    def sample_from_planes(self, coordinates, plane_features=None, lbound=None, n_valid=None):
        if plane_features is None:
            plane_features = self.get_planes()
        if lbound is None:
            lbound = self.lbound
        feat = sample_planes(plane_features, coordinates, lbound, n_valid=n_valid)
        return feat.view(feat.shape[0], 3, self.number_of_features)

    def get_grid_features(self, grid_res, plane_features=None, grid=None):
        """:485-512 -- features on a regular grid_res^3 lattice of [-lbound, lbound]^3 (axes permuted to (z, x, y) as the
        reference does); the planes default to the first level whose side reaches 2 * grid_res."""
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
        return self.lbound, feats.reshape(*shape[:-1], -1), grid

    def planes_and_grad_buffer(self):
        """-> (planes, the gradient buffer of this step's sampling backward or None): what a sampling call of the step needs."""
        planes = self.get_planes()
        gbuf = self._join_prefetch()
        if gbuf is not None and not torch.is_grad_enabled():
            gbuf = None
        return planes, gbuf

    def forward(self, coordinates, bound, n_valid=None, perm=None, half_out=False):
        """coordinates [M,3] in [-bound, bound] -> features [M, 3C] (index p*C + c); fp32 as the reference's
        grid_sample, or fp16 (half_out) for the fused MLP path, which rounds its input to fp16 anyway."""
        planes, gbuf = self.planes_and_grad_buffer()
        return sample_planes(planes, coordinates, bound, n_valid=n_valid, perm=perm, half_out=half_out, grad_buf=gbuf)

    # -- checkpoints: accept reference (NCHW-contiguous) tensors, keep channels-last storage -------------
    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)  # Tensor.copy_ keeps our strides
        self.last_used_planes = None
