"""Input gradients of the field on the host build of the kernels (tests/emu): the SH encoder backward, the position gradient of
the plane gather and the direction gradient of the mma.sync MLP backward, each
against fp64 autograd of the reference's op sequence (tests/field_truth.py, oracle/field.py); and the argument checks of the
new entry points."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import field as of
from tests import field_truth as ft
from tests import kemu

BOUND = 1.5


def _rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _cl(planes):
    return np.ascontiguousarray(planes.permute(0, 2, 3, 1).numpy())


def _inv():
    return float(np.float32(1.0) / np.float32(BOUND))


@pytest.mark.parametrize("degree", [1, 2, 3, 4])
def test_sh_backward_matches_fp64_autograd(degree):
    g = torch.Generator().manual_seed(degree)
    B = 2000
    d = torch.randn(B, 3, generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    d[:3] = torch.tensor([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0]])
    grad = torch.randn(B, degree ** 2, generator=g)
    dd = d.double().requires_grad_(True)
    (want,) = torch.autograd.grad(of.sh16(dd)[:, :degree ** 2], dd, grad.double())
    out = np.full((B, 3), np.nan, np.float32)
    kemu.call("tnl_sh_encode_backward", kemu.f32(grad.numpy()), kemu.f32(d.numpy()), B, degree, out, None)
    assert _rel_l2(out, want.numpy()) <= 1e-6
    if degree == 1:
        assert (out == 0).all()


def _points(M, g):
    xyz = (torch.rand(M, 3, generator=g) * 2 - 1) * BOUND
    xyz[:4] = torch.tensor([[-1.5, -1.5, -1.5], [1.5, 1.5, 1.5], [0.3, -1.6, 0.2], [1.4999, 0.0, -1.4999]])   # border / outside
    return xyz


def _perm(xyz, M, nv):
    perm = np.empty(M, np.int32)
    work = np.zeros(max(kemu.lib().tnl_cell_sort_workspace(M, 16), 16), np.uint8)
    kemu.call("tnl_cell_sort", xyz.numpy(), M, nv, _inv(), 16, perm, work, work.size, None)
    return perm


@pytest.mark.parametrize("C,R,half,use_perm", [(16, 48, False, False), (32, 64, True, True), (48, 40, True, False), (8, 32, False, True)])
def test_position_gradient_matches_fp64_autograd(C, R, half, use_perm):
    """fp32 coordinates: the kernel against fp64 autograd of the literal gather; rows >= n_valid get exactly zero"""
    g = torch.Generator().manual_seed(C + R)
    M = 1501
    planes = torch.randn(3, C, R, R, generator=g)
    xyz = _points(M, g)
    nv = np.array([M - 77], np.int32)
    perm = _perm(xyz, M, nv) if use_perm else None
    G = torch.randn(M, 3 * C, generator=g)
    Gk = G.numpy().astype(np.float16) if half else G.numpy()
    Gt = torch.from_numpy(Gk.astype(np.float32)).double()
    x64 = xyz.double().requires_grad_(True)
    (want,) = torch.autograd.grad(ft.sample(planes.double(), x64, BOUND), x64, Gt)
    want = want.numpy()
    g_xyz = np.full((M, 3), np.nan, np.float32)
    kemu.call("tnl_sample_planes_backward_xyz", Gk, int(half), _cl(planes), xyz.numpy(), M, R, C, _inv(), 0, nv, perm, g_xyz, None)
    assert (g_xyz[M - 77:] == 0).all()
    assert _rel_l2(g_xyz[:M - 77], want[:M - 77]) <= 1e-5


def test_position_gradient_fp16_coordinate_rounding():
    """fp16_coords: the reference's autocast backward rounds each plane's grid gradient to fp16, rounds the sum of the two planes
    that read an axis to fp16 again, then scales by fp32(1/bound).  Emulated here on the grid itself, in fp32 as ATen's CPU
    grid_sample backward computes it."""
    g = torch.Generator().manual_seed(11)
    C, R, M = 16, 64, 1200
    planes = torch.randn(3, C, R, R, generator=g)
    xyz = _points(M, g)
    G = torch.randn(M, 3 * C, generator=g)
    u = of.project_coords(xyz, BOUND, fp16=True)
    grid = torch.stack([torch.stack([u[:, a], u[:, b]], dim=-1) for a, b in of.PLANE_AXES], dim=0).requires_grad_(True)
    s = torch.nn.functional.grid_sample(planes, grid.unsqueeze(2), mode="bilinear", padding_mode="border", align_corners=True)
    (gg,) = torch.autograd.grad(s.permute(2, 0, 1, 3).reshape(M, -1), grid, G)
    gg = gg.half().float()                                                        # [3, M, 2] per-plane grid gradient
    ax = [gg[0, :, 0] + gg[1, :, 0], gg[1, :, 1] + gg[2, :, 0], gg[0, :, 1] + gg[2, :, 1]]
    want = torch.stack([a.half().float() for a in ax], dim=-1) * np.float32(_inv())
    g_xyz = np.full((M, 3), np.nan, np.float32)
    kemu.call("tnl_sample_planes_backward_xyz", G.numpy(), 0, _cl(planes), xyz.numpy(), M, R, C, _inv(), 1, None, None, g_xyz, None)
    # the per-plane sums may differ in the last fp32 bits from ATen's, which can move an fp16 rounding by one step
    assert _rel_l2(g_xyz, want.numpy()) <= 2e-3
    assert (np.abs(g_xyz - want.numpy()) <= 2 * np.abs(want.numpy()) * 2.0 ** -10 + 1e-30).mean() >= 0.99


def _mlp_pack(C, W):
    from trinerflet_b200._lib import MlpDims
    dims = MlpDims(3 * C, 64, 64)
    packed = np.zeros(kemu.lib().tnl_mlp_packed_bytes(ctypes.byref(dims)), np.uint8)
    kemu.call("tnl_mlp_pack_weights", ctypes.byref(dims), *[kemu.f32(w.numpy()) for w in W], packed, None)
    return dims, packed


@pytest.mark.parametrize("C,M,half", [(16, 300, False), (32, 150, True), (48, 77, False)])
def test_mlp_direction_gradient_matches_oracle(C, M, half):
    """tnl_mlp_backward_dirs (mma.sync kernels): g_dirs against autograd of the oracle's fp16-autocast emulation; g_feat and the
    weight gradients are tnl_mlp_backward's; rows >= n_valid get zero"""
    g = torch.Generator().manual_seed(7 + C)
    W = of.init_mlp_weights(C, 64, 64, gen=g)
    feat = 0.5 * torch.randn(M, 3 * C, generator=g)
    d = torch.randn(M, 3, generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    gs, grgb = torch.randn(M, generator=g) * 64.0, torch.randn(M, 3, generator=g) * 64.0
    d_o = d.clone().requires_grad_(True)
    _, rgb_o, _ = of.mlp_forward(feat, d_o, W, fp16=True)
    (want,) = torch.autograd.grad(rgb_o, d_o, grgb)                   # (sigma does not depend on the direction)
    dims, packed = _mlp_pack(C, W)
    fk = feat.numpy().astype(np.float16) if half else feat.numpy()
    nv = np.array([M - 5], np.int32)
    outs = []
    for name in ("tnl_mlp_backward", "tnl_mlp_backward_dirs"):
        g_feat = np.zeros((M, 3 * C), fk.dtype)
        gW = [np.zeros(tuple(w.shape), np.float32) for w in W]
        extra = [np.full((M, 3), np.nan, np.float32)] if name.endswith("dirs") else []
        kemu.call(name, ctypes.byref(dims), packed, fk, int(half), d.numpy(), M, nv, gs.numpy(), grgb.numpy(), g_feat, *gW, *extra, None)
        outs.append((g_feat, gW, extra))
    (gf0, gW0, _), (gf1, gW1, (g_dirs,)) = outs
    assert np.array_equal(gf0, gf1) and all(np.array_equal(a, b) for a, b in zip(gW0, gW1))
    assert (g_dirs[M - 5:] == 0).all()
    assert _rel_l2(g_dirs[:M - 5], want.numpy()[:M - 5]) <= 1e-2


def test_abi_argument_checks():
    lib = kemu.lib()
    a = np.zeros(64, np.float32)
    p = kemu.p(a)
    # SH backward: null pointers, degree outside 1..4
    assert lib.tnl_sh_encode_backward(None, p, 4, 4, p, None) == -1
    assert lib.tnl_sh_encode_backward(p, p, 4, 4, None, None) == -1
    assert lib.tnl_sh_encode_backward(p, p, 4, 0, p, None) == -1
    assert lib.tnl_sh_encode_backward(p, p, 4, 5, p, None) == -1
    # position gradient: null pointers, C not a multiple of 4, misaligned buffers
    buf = np.zeros(4096 + 8, np.float32)
    al, mis = kemu.p(buf), ctypes.c_void_p(buf.ctypes.data + 4)
    f = ctypes.c_float(1.0)
    args = lambda gf=al, pl=al, gx=al, C=16: (gf, 0, pl, al, 4, 8, C, f, 0, None, None, gx, None)   # noqa: E731
    assert lib.tnl_sample_planes_backward_xyz(*args(gf=None)) == -1
    assert lib.tnl_sample_planes_backward_xyz(*args(gx=None)) == -1
    assert lib.tnl_sample_planes_backward_xyz(*args(C=6)) == -1
    assert lib.tnl_sample_planes_backward_xyz(*args(pl=mis)) == -1
    assert lib.tnl_sample_planes_backward_xyz(*args(gf=mis)) == -1
    # MLP direction gradient: g_dirs required, misaligned features rejected like tnl_mlp_backward
    g = torch.Generator().manual_seed(0)
    dims, packed = _mlp_pack(16, of.init_mlp_weights(16, 64, 64, gen=g))
    M = 16
    feat = np.zeros(M * 48 + 2, np.float32)
    z = [kemu.p(np.zeros(n, np.float32)) for n in (3 * M, M, 3 * M, 64 * 48, 16 * 64, 64 * 31, 64 * 64, 3 * 64, 3 * M)]
    dirs, gs, grgb, gW1, gW2, gW3, gW4, gW5, gd = z
    gf = kemu.p(np.zeros(M * 48, np.float32))
    assert lib.tnl_mlp_backward_dirs(ctypes.byref(dims), kemu.p(packed), kemu.p(feat), 0, dirs, M, None, gs, grgb, gf, gW1, gW2, gW3,
                                     gW4, gW5, None, None) == -1
    assert lib.tnl_mlp_backward_dirs(ctypes.byref(dims), kemu.p(packed), ctypes.c_void_p(feat.ctypes.data + 4), 0, dirs, M, None, gs,
                                     grgb, gf, gW1, gW2, gW3, gW4, gW5, gd, None) == -1
    assert lib.tnl_mlp_backward_dirs(ctypes.byref(dims), kemu.p(packed), kemu.p(feat), 0, None, M, None, gs, grgb, gf, gW1, gW2, gW3,
                                     gW4, gW5, gd, None) == -1
