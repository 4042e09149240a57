"""CPU: the deterministic-mode kernels (tnl_sample_planes_backward_det, tnl_mlp_backward_det on the mma.sync kernels) through the
host build of their sources (tests/kemu.py), and the Python switches of torch.use_deterministic_algorithms.

The fixed-point scatter must not depend on the visiting order or on the thread schedule: the same bits with and without `perm`,
with the points permuted, and under TNL_EMU_SCHED=reverse / random (read once per process, so those runs are subprocesses)."""
import ctypes
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch

from oracle import field as of
from tests import kemu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def deterministic_mode():
    """torch.use_deterministic_algorithms(True) for one test; the previous state (and warn_only) is restored."""
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


def _aligned(nbytes, align=256):
    raw = np.zeros(nbytes + align, np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + nbytes]


def _lattice_case(C, M, seed, fp16):
    """Points on a lattice whose bilinear weights are multiples of 1/16 and feature gradients with 11 significant bits: every
    contribution g * w is exact in fp32, so an fp64 sum of them is the exact texel sum."""
    g = torch.Generator().manual_seed(seed)
    R = 33                                               # bound 1: pixel coordinate (x + 1) / 2 * 32 = j / 4
    xyz = (-1.0 + torch.randint(0, 129, (M, 3), generator=g).float() / 64.0).numpy()
    G = torch.randn(M, 3 * C, generator=g).half().float()
    G[M - 40:] = 0.0
    Gin = G.numpy().copy()
    Gin[M - 40:] = np.nan                                # rows >= n_valid are never read
    Gin = Gin.astype(np.float16) if fp16 else Gin
    return R, xyz, G, Gin


def _det_scatter(Gin, fp16, xyz, M, R, C, nv, perm=None):
    ws = _aligned(kemu.lib().tnl_sample_planes_backward_det_workspace(R, C))
    gp = np.zeros((3, R, R, C), np.float32)
    kemu.call("tnl_sample_planes_backward_det", Gin, int(fp16), xyz, M, R, C, 1.0, 0, nv, perm, None, None, 0, 0, gp, ws, ws.size, None)
    return gp


@pytest.mark.parametrize("C,fp16", [(16, True), (32, False), (48, True), (48, False)])
def test_det_scatter_within_bound_of_exact_sum_and_order_free(C, fp16):
    M = 1500
    R, xyz, G, Gin = _lattice_case(C, M, C + int(fp16), fp16)
    nv = np.array([M - 40], np.int32)
    gp = _det_scatter(Gin, fp16, xyz, M, R, C, nv)
    pl = torch.zeros(3, C, R, R, dtype=torch.float64, requires_grad=True)
    (of.sample_planes(pl, torch.from_numpy(xyz), 1.0) * G.double()).sum().backward()
    ref = np.ascontiguousarray(pl.grad.permute(0, 2, 3, 1).numpy())
    m = float(np.abs(G.numpy()).max())
    e = np.frexp(m)[1]
    mu = int(np.ceil(np.log2(M)))
    unit = 2.0 ** (e + mu - 62)
    tol = M * unit / 2 + 2.0 ** -24 * np.abs(ref)
    assert (np.abs(gp.astype(np.float64) - ref) <= tol).all()
    # visiting order: perm, and the points themselves permuted, give the same bits
    perm = np.random.default_rng(C).permutation(M).astype(np.int32)
    assert np.array_equal(_det_scatter(Gin, fp16, xyz, M, R, C, nv, perm).view(np.uint32), gp.view(np.uint32))
    q = np.random.default_rng(C + 1).permutation(M - 40)
    q = np.concatenate([q, np.arange(M - 40, M)])
    gq = _det_scatter(np.ascontiguousarray(Gin[q]), fp16, np.ascontiguousarray(xyz[q]), M, R, C, nv)
    assert np.array_equal(gq.view(np.uint32), gp.view(np.uint32))


def test_det_scatter_tile_list_and_nonfinite():
    C, M = 16, 800
    R, xyz, G, Gin = _lattice_case(C, M, 5, True)
    R = 32                                               # tiles of 16 x 16 texels: 2 x 2 per plane
    xyz = np.clip(xyz, -1.0, 1.0)
    nv = np.array([M - 40], np.int32)
    dense = _det_scatter(Gin, True, xyz, M, R, C, nv)
    ids, count = np.array([0, 3, 5, 10], np.int32), np.array([4], np.int32)
    ws = _aligned(kemu.lib().tnl_sample_planes_backward_det_workspace(R, C))
    ws[:] = 0xff                                         # the call zeroes what it accumulates into
    gp = np.full((3, R, R, C), np.nan, np.float32)
    tiles = gp.reshape(3, 2, 16, 2, 16, C)
    for t in ids:
        tiles[t // 4, (t // 2) % 2, :, t % 2] = 0.0
    kemu.call("tnl_sample_planes_backward_det", Gin, 1, xyz, M, R, C, 1.0, 0, nv, None, ids, count, 8, 16, gp, ws, ws.size, None)
    dense_t = dense.reshape(3, 2, 16, 2, 16, C)
    for t in ids:
        a, b = tiles[t // 4, (t // 2) % 2, :, t % 2], dense_t[t // 4, (t // 2) % 2, :, t % 2]
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # an inf below n_valid: every converted element is NaN (the optimizer then skips the step); NaN rows past n_valid are ignored
    Gbad = Gin.copy()
    Gbad[7, 3] = np.inf
    assert np.isnan(_det_scatter(Gbad, True, xyz, M, R, C, nv)).all()
    assert np.isfinite(dense).all()


def test_det_scatter_argument_checks():
    lib = kemu.lib()
    C, M, R = 16, 10, 8
    g = np.zeros((M, 3 * C), np.float32)
    xyz = np.zeros((M, 3), np.float32)
    gp = np.zeros((3, R, R, C), np.float32)
    need = lib.tnl_sample_planes_backward_det_workspace(R, C)
    assert need == 256 + 3 * R * R * C * 8
    ws = _aligned(need)
    args = lambda w, wsz, ids=None, cnt=None, T=0, Cc=C: (kemu.p(g), 0, kemu.p(xyz), M, R, Cc, ctypes.c_float(1.0), 0, None, None,  # noqa: E731
                                                          kemu.p(ids), kemu.p(cnt), 4, T, kemu.p(gp), w, wsz, None)
    assert lib.tnl_sample_planes_backward_det(*args(kemu.p(ws), need)) == 0
    assert lib.tnl_sample_planes_backward_det(*args(kemu.p(ws), need - 1)) == -1          # workspace too small
    assert lib.tnl_sample_planes_backward_det(*args(None, need)) == -1                    # no workspace
    assert lib.tnl_sample_planes_backward_det(*args(kemu.p(ws), need, Cc=6)) == -1        # C not a multiple of 4
    ids, cnt = np.zeros(4, np.int32), np.zeros(1, np.int32)
    assert lib.tnl_sample_planes_backward_det(*args(kemu.p(ws), need, ids, cnt, T=3)) == -1   # tile edge must divide R
    assert lib.tnl_sample_planes_backward_det(*args(kemu.p(ws), need, ids, None, T=4)) == -1  # tile list without its count


def _mlp_case(C, M):
    from trinerflet_b200._lib import MlpDims
    g = torch.Generator().manual_seed(3 + C)
    W = of.init_mlp_weights(C, 64, 64, gen=g)
    feat = (0.5 * torch.randn(M, 3 * C, generator=g)).numpy()
    d = torch.randn(M, 3, generator=g)
    d = (d / d.norm(dim=-1, keepdim=True)).numpy()
    gs = (torch.randn(M, generator=g) * 64.0).numpy()
    grgb = (torch.randn(M, 3, generator=g) * 64.0).numpy()
    dims = MlpDims(3 * C, 64, 64)
    packed = np.zeros(kemu.lib().tnl_mlp_packed_bytes(ctypes.byref(dims)), np.uint8)
    kemu.call("tnl_mlp_pack_weights", ctypes.byref(dims), *[kemu.f32(w.numpy()) for w in W], packed, None)
    return W, dims, packed, feat, d, gs, grgb


def _mlp_det(C, M, dirs_grad):
    W, dims, packed, feat, d, gs, grgb = _mlp_case(C, M)
    nv = np.array([M - 9], np.int32)
    ws = _aligned(kemu.lib().tnl_mlp_backward_det_workspace(ctypes.byref(dims), 0, M), 16)
    gW = [np.zeros(tuple(w.shape), np.float32) for w in W]
    g_feat = np.zeros((M, 3 * C), np.float32)
    g_dirs = np.full((M, 3), np.nan, np.float32) if dirs_grad else None
    kemu.call("tnl_mlp_backward_det", ctypes.byref(dims), packed, feat, 0, d, M, nv, gs, grgb, g_feat, *gW, g_dirs, ws, ws.size, None)
    ref = [np.zeros(tuple(w.shape), np.float32) for w in W]
    g_feat_ref = np.zeros((M, 3 * C), np.float32)
    kemu.call("tnl_mlp_backward", ctypes.byref(dims), packed, feat, 0, d, M, nv, gs, grgb, g_feat_ref, *ref, None)
    return gW, ref, g_feat, g_feat_ref, g_dirs


@pytest.mark.parametrize("C,dirs_grad", [(16, False), (48, True)])
def test_mlp_backward_det_matches_atomic_version(C, dirs_grad):
    M = 700                                              # several CTAs (128 points each)
    gW, ref, g_feat, g_feat_ref, g_dirs = _mlp_det(C, M, dirs_grad)
    assert np.array_equal(g_feat, g_feat_ref)
    for a, b in zip(gW, ref):
        assert np.allclose(a, b, rtol=1e-5, atol=1e-5 * np.abs(b).max()), a.shape
    if dirs_grad:
        assert np.isfinite(g_dirs).all() and (g_dirs[M - 9:] == 0).all()


def test_mlp_backward_det_argument_checks():
    from trinerflet_b200._lib import MlpDims
    lib = kemu.lib()
    W, dims, packed, feat, d, gs, grgb = _mlp_case(16, 100)
    need = lib.tnl_mlp_backward_det_workspace(ctypes.byref(dims), 0, 100)
    assert need > 0 and lib.tnl_mlp_backward_det_workspace(ctypes.byref(MlpDims(40, 64, 64)), 0, 100) == 0
    ws = _aligned(need, 16)
    gW = [np.zeros(tuple(w.shape), np.float32) for w in W]
    g_feat = np.zeros((100, 48), np.float32)
    args = lambda w, wsz: (ctypes.byref(dims), kemu.p(packed), kemu.p(feat), 0, kemu.p(d), 100, None, kemu.p(gs), kemu.p(grgb),  # noqa: E731
                           kemu.p(g_feat), *[kemu.p(x) for x in gW], None, w, wsz, None)
    assert lib.tnl_mlp_backward_det(*args(kemu.p(ws), need)) == 0
    assert lib.tnl_mlp_backward_det(*args(kemu.p(ws), need - 4)) == -1
    assert lib.tnl_mlp_backward_det(*args(None, need)) == -1


_SCHED_SCRIPT = r"""
import hashlib, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_deterministic_emu as t
R, xyz, G, Gin = t._lattice_case(32, 1200, 1, True)
nv = np.array([1160], np.int32)
h = hashlib.sha256(t._det_scatter(Gin, True, xyz, 1200, R, 32, nv).tobytes())
gW = t._mlp_det(16, 500, True)[0]
for w in gW:
    h.update(w.tobytes())
print(h.hexdigest())
"""


def test_det_kernels_bit_identical_under_other_thread_schedules():
    kemu.lib()   # build once before the subprocesses load it
    digests = []
    for sched in (None, "reverse", "random:7"):
        env = dict(os.environ)
        env.pop("TNL_EMU_SCHED", None)
        if sched:
            env["TNL_EMU_SCHED"] = sched
        out = subprocess.run([sys.executable, "-c", _SCHED_SCRIPT, ROOT], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        digests.append(out.stdout.strip().splitlines()[-1])
    assert digests[0] == digests[1] == digests[2], digests


def test_multi_gpu_step_is_refused_in_deterministic_mode(deterministic_mode):
    from trinerflet_b200 import _lib, trainer
    with pytest.raises(RuntimeError, match="deterministic"):
        trainer.TrainStep(None, world_size=2)       # before any distributed call (or anything of the model)
    torch.use_deterministic_algorithms(True, warn_only=True)
    with pytest.warns(UserWarning, match="deterministic"):
        _lib.alert_nondeterministic("a multi-GPU TrainStep (world_size > 1)")


def test_alert_is_silent_with_the_flag_off():
    from trinerflet_b200 import _lib
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(False)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            _lib.alert_nondeterministic("anything")
        assert not _lib.deterministic()
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
