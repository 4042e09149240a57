"""Camera pose refinement on the host build of the kernels (tests/emu): the ray parameters of the training march
(tnl_march_rays_train_ts), the ray gradient of the march (tnl_rays_backward) and the pose gradient of the ray feeder
(tnl_rays_from_ids_backward), each against an fp64 restatement; their schedule independence; CameraPoses' exp map against fp64
central differences; the autograd wiring of raymarching / rays on CPU tensors; and the argument checks of the new entry points."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import kemu
from tests.util import random_bitfield, synthetic_rays

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUND, CAS, H = 1.5, 2, 128
AABB = np.array([-BOUND] * 3 + [BOUND] * 3, np.float32)


def _rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------ march with ts
@pytest.fixture(scope="module")
def scene():
    o, d = synthetic_rays(512, 0)
    _, bits = random_bitfield(0)
    bits = bits.numpy()
    N = len(o)
    nears, fars = np.empty(N, np.float32), np.empty(N, np.float32)
    kemu.call("tnl_near_far_from_aabb", o, d, AABB, N, 0.2, nears, fars, None)
    noises = np.random.default_rng(3).random(N).astype(np.float32)
    return o, d, bits, nears, fars, noises


def _march(scene, M, fast, with_ts, max_steps=1024):
    o, d, bits, nears, fars, noises = scene
    N = len(o)
    xyzs, dirs, deltas = (np.full((M, w), np.nan, np.float32) for w in (3, 3, 2))
    ts = np.full(M, np.nan, np.float32)
    rays, counter = np.empty((N, 3), np.int32), np.zeros(2, np.int32)
    lib = kemu.lib()
    wsz = lib.tnl_march_rays_train_workspace_fast(N, max_steps) if fast else lib.tnl_march_rays_train_workspace(N)
    ws = np.zeros(wsz, np.uint8)
    if with_ts:
        kemu.call("tnl_march_rays_train_ts", o, d, bits, BOUND, 0.0, max_steps, N, CAS, H, M, nears, fars, xyzs, dirs, deltas, ts,
                  rays, counter, noises, ws, wsz, None)
    else:
        kemu.call("tnl_march_rays_train", o, d, bits, BOUND, 0.0, max_steps, N, CAS, H, M, nears, fars, xyzs, dirs, deltas,
                  rays, counter, noises, ws, wsz, None)
    return xyzs, dirs, deltas, rays, counter, ts


@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("mean_count", [400, 20])          # 20: rays overflow M and are dropped
def test_march_ts_is_the_plain_march_plus_t(scene, fast, mean_count):
    o, d = scene[0], scene[1]
    M = len(o) * mean_count
    plain = _march(scene, M, fast, False)
    *outs, ts = _march(scene, M, fast, True)
    for a, b in zip(plain[:5], outs):
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
    xyzs, rays = outs[0], outs[3]
    owned = np.zeros(M, bool)
    for n, off, cnt in rays:
        if cnt and off + cnt <= M:
            owned[off:off + cnt] = True
    assert (mean_count == 20) == (not owned.all() and owned.sum() < rays[:, 2].sum())
    assert (ts[~owned] == 0).all() and np.isfinite(ts).all()
    ray_of = np.full(M, -1)
    for n, off, cnt in rays:
        if cnt and off + cnt <= M:
            ray_of[off:off + cnt] = n
    r = ray_of[owned]
    u = (ts[owned, None].astype(np.float64) * d[r].astype(np.float64) + o[r].astype(np.float64)).astype(np.float32)
    assert np.array_equal(_bits(np.clip(u, -BOUND, BOUND)), _bits(xyzs[owned]))


# ------------------------------------------------------------------------------------------------ ray gradient
def _ray_case(seed=0, N=300, M=4000):
    """hand-made march output: zero-count rays, rays overflowing M, clamped components on both borders (exactly at +-bound too)"""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, 40, N)
    counts[::17] = 0
    offs = np.concatenate([[0], np.cumsum(counts)[:-1]])
    rays = np.stack([np.arange(N), offs, counts], 1).astype(np.int32)
    o = rng.uniform(-1.2, 1.2, (N, 3)).astype(np.float32)
    d = rng.normal(size=(N, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    ts = np.zeros(M, np.float32)
    for n, off, cnt in rays:
        if cnt and off + cnt <= M:
            ts[off:off + cnt] = np.sort(rng.uniform(0.0, 3.5, cnt)).astype(np.float32)   # far enough to leave the box
    # exact borders: o = bound - 1, d = 1, t = 1 -> fmaf = +bound; o = -bound + 0.5, d = -0.5, t = 1 -> -bound
    o[1] = [BOUND - 1, -BOUND + 0.5, 0.25]
    d[1] = [1.0, -0.5, 0.0]
    if counts[1] and offs[1] + counts[1] <= M:
        ts[offs[1]] = 1.0
        ts[offs[1] + min(1, counts[1] - 1)] = np.nextafter(np.float32(1.0), np.float32(2.0))
    g_xyz = rng.normal(size=(M, 3)).astype(np.float32)
    g_dirs = rng.normal(size=(M, 3)).astype(np.float32)
    return rays, ts, o, d, g_xyz, g_dirs


def _ray_truth(rays, ts, o, d, g_xyz, g_dirs, n_valid, M):
    N = len(rays)
    go, gd = np.zeros((N, 3)), np.zeros((N, 3))
    for n, off, cnt in rays:
        if cnt == 0 or off + cnt > M:
            continue
        for i in range(off, min(off + cnt, n_valid)):
            t = np.float64(ts[i])
            if g_xyz is not None:
                u = (t * d[n].astype(np.float64) + o[n].astype(np.float64)).astype(np.float32)
                m = (u >= -BOUND) & (u <= BOUND)
                go[n] += m * g_xyz[i]
                gd[n] += t * m * g_xyz[i]
            if g_dirs is not None:
                gd[n] += g_dirs[i]
    return go, gd


def _ray_kernel(rays, ts, o, d, g_xyz, g_dirs, n_valid, M):
    N = len(rays)
    go, gd = np.full((N, 3), np.nan, np.float32), np.full((N, 3), np.nan, np.float32)
    nv = None if n_valid is None else np.array([n_valid], np.int32)
    kemu.call("tnl_rays_backward", rays, ts, o, d, BOUND, g_xyz, g_dirs, nv, N, M, go, gd, None)
    return go, gd


@pytest.mark.parametrize("which", ["both", "xyz", "dirs"])
@pytest.mark.parametrize("n_valid", [None, 2500])
def test_rays_backward_matches_fp64_sum(which, n_valid):
    M = 4000
    rays, ts, o, d, g_xyz, g_dirs = _ray_case(M=M)
    assert (rays[:, 1] + rays[:, 2] > M).any() and (rays[:, 2] == 0).any()
    gx = g_xyz if which in ("both", "xyz") else None
    gdir = g_dirs if which in ("both", "dirs") else None
    go, gd = _ray_kernel(rays, ts, o, d, gx, gdir, n_valid, M)
    tgo, tgd = _ray_truth(rays, ts, o, d, gx, gdir, M if n_valid is None else n_valid, M)
    if gx is None:
        assert (go == 0).all()
    else:
        assert _rel_l2(go, tgo) <= 2e-6
    assert _rel_l2(gd, tgd) <= 2e-6
    dead = (rays[:, 2] == 0) | (rays[:, 1] + rays[:, 2] > M)
    if n_valid is not None:
        dead |= rays[:, 1] >= n_valid
    assert (go[dead] == 0).all() and (gd[dead] == 0).all()
    # ray 1: its first row sits exactly on +bound (x) and -bound (y) and passes (torch.clamp's backward); the next row's x is one
    # ulp beyond and does not, its y rounds back onto -bound and does
    if gx is not None:
        off = rays[1, 1]
        u0 = np.float32(np.float64(ts[off]) * d[1, 0] + o[1, 0])
        u1 = np.float32(np.float64(ts[off + 1]) * d[1, 0] + o[1, 0])
        assert u0 == BOUND and u1 > BOUND and rays[1, 2] >= 2
        assert np.float32(np.float64(ts[off]) * d[1, 1] + o[1, 1]) == -BOUND
        r1 = rays[1:2].copy()
        r1[0, 0] = 0
        one, _ = _ray_kernel(r1, ts, o[1:2], d[1:2], gx, None, off + 2, M)
        assert one[0, 0] == g_xyz[off, 0] and one[0, 1] == np.float32(np.float64(g_xyz[off, 1]) + g_xyz[off + 1, 1])


# ------------------------------------------------------------------------------------------------ pose gradient
INTR = (23.0, 21.5, 15.7, 12.2)
PH, PW = 24, 32


def _dirs64(pix):
    fx, fy, cx, cy = INTR
    i = (pix % PW).astype(np.float64) + 0.5
    j = (pix // PW).astype(np.float64) + 0.5
    xs, ys = (i - cx) / fx, (j - cy) / fy
    v = torch.from_numpy(np.stack([xs, ys, np.ones_like(xs)], -1))
    return v / v.norm(dim=-1, keepdim=True)


def _pose_truth(poses, ids, g_o, g_d):
    """fp64 autograd of the reference's get_rays expression (rays_d = dirs @ R^T, rays_o = pose[:3,3]) per ray"""
    P = torch.from_numpy(poses.astype(np.float64)).requires_grad_(True)
    n_total = len(poses) * PH * PW
    ids = np.clip(ids, 0, n_total - 1)
    img, pix = ids // (PH * PW), ids % (PH * PW)
    dirs = _dirs64(pix)
    R = P[img, :3, :3]
    rays_d = (dirs.unsqueeze(1) * R).sum(-1)
    rays_o = P[img, :3, 3]
    (g,) = torch.autograd.grad([rays_o, rays_d], [P], [torch.from_numpy(g_o.astype(np.float64)),
                                                        torch.from_numpy(g_d.astype(np.float64))])
    return g.numpy()


def _poses(B, seed):
    rng = np.random.default_rng(seed)
    q = rng.normal(size=(B, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    R = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                  2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                  2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1).reshape(B, 3, 3)
    P = np.zeros((B, 4, 4), np.float32)
    P[:, :3, :3] = R
    P[:, :3, 3] = rng.uniform(-2, 2, (B, 3))
    P[:, 3, 3] = 1
    return P


def _pose_kernel(B, ids, first_id, n, g_o, g_d):
    out = np.full((B, 4, 4), np.nan, np.float32)
    fx, fy, cx, cy = INTR
    kemu.call("tnl_rays_from_ids_backward", g_o, g_d, B, fx, fy, cx, cy, PH, PW, ids, first_id, n, out, None)
    return out


def test_pose_backward_ray_ids_matches_fp64_autograd():
    B, n = 7, 3000
    rng = np.random.default_rng(5)
    poses = _poses(B, 5)
    ids = rng.integers(0, (B - 1) * PH * PW, n).astype(np.int64)      # image B-1 has no ray
    ids[:3] = [-5, B * PH * PW + 9, 0]                                   # clamped as the forward clamps them
    g_o = rng.normal(size=(n, 3)).astype(np.float32)
    g_d = rng.normal(size=(n, 3)).astype(np.float32)
    got = _pose_kernel(B, ids, 0, n, g_o, g_d)
    want = _pose_truth(poses, ids, g_o, g_d)
    assert _rel_l2(got, want) <= 1e-5
    assert (got[:, 3] == 0).all()
    clamped_last = np.clip(ids, 0, B * PH * PW - 1) // (PH * PW) == B - 1
    assert clamped_last.sum() == 1            # only the clamped id lands on the last image
    # NULL gradients are zeros
    only_d = _pose_kernel(B, ids, 0, n, None, g_d)
    assert (only_d[:, :3, 3] == 0).all() and _rel_l2(only_d, _pose_truth(poses, ids, np.zeros_like(g_o), g_d)) <= 1e-5


def test_pose_backward_first_id_matches_fp64_autograd_and_empty_images_are_zero():
    B = 6
    first, n = 2 * PH * PW + 100, PH * PW + 50           # images 0, 1 and 5 get no ray
    poses = _poses(B, 6)
    rng = np.random.default_rng(6)
    g_o = rng.normal(size=(n, 3)).astype(np.float32)
    g_d = rng.normal(size=(n, 3)).astype(np.float32)
    got = _pose_kernel(B, None, first, n, g_o, g_d)
    want = _pose_truth(poses, np.arange(first, first + n), g_o, g_d)
    assert _rel_l2(got, want) <= 1e-5
    assert (got[[0, 1, 4, 5]] == 0).all() and (got[2, :3] != 0).any() and (got[3, :3] != 0).any()
    assert got[4].sum() == 0 and np.array_equal(got[5], np.zeros((4, 4), np.float32))


_SCHED_SCRIPT = r"""
import hashlib, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_pose_grads_emu as t
rays, ts, o, d, gx, gdir = t._ray_case(M=4000)
h = hashlib.sha256()
for a in t._ray_kernel(rays, ts, o, d, gx, gdir, 2500, 4000):
    h.update(a.tobytes())
rng = np.random.default_rng(5)
ids = rng.integers(0, 7 * t.PH * t.PW, 3000).astype(np.int64)
go, gd = rng.normal(size=(3000, 3)).astype(np.float32), rng.normal(size=(3000, 3)).astype(np.float32)
h.update(t._pose_kernel(7, ids, 0, 3000, go, gd).tobytes())
h.update(t._pose_kernel(7, None, 500, 3000, go, gd).tobytes())
print(h.hexdigest())
"""


def test_backward_kernels_bit_identical_under_other_thread_schedules():
    kemu.lib()
    digests = []
    for sched in (None, "reverse", "random:11"):
        env = dict(os.environ)
        env.pop("TNL_EMU_SCHED", None)
        if sched:
            env["TNL_EMU_SCHED"] = sched
        out = subprocess.run([sys.executable, "-c", _SCHED_SCRIPT, ROOT], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        digests.append(out.stdout.strip().splitlines()[-1])
    assert digests[0] == digests[1] == digests[2], digests


# ------------------------------------------------------------------------------------------------ CameraPoses
def test_camera_poses_identity_at_zero_and_fp64_gradients():
    from trinerflet_b200.poses import CameraPoses, se3_exp
    P = torch.from_numpy(_poses(5, 7))
    cams = CameraPoses(P)
    out = cams()
    assert out.dtype == torch.float32 and torch.equal(out.view(torch.int32), P.view(torch.int32))
    assert torch.equal(se3_exp(torch.zeros(3, 6)), torch.eye(4).expand(3, 4, 4))
    c64 = CameraPoses(P.double(), fixed=[3])

    def f(delta):
        c64.delta.data = delta
        return c64()

    for xi in (torch.zeros(5, 6, dtype=torch.float64),
               torch.randn(5, 6, dtype=torch.float64, generator=torch.Generator().manual_seed(1)) * 0.4,
               torch.full((5, 6), 0.05, dtype=torch.float64)):           # |omega|^2 = 0.0075: the series branch away from 0
        x = xi.clone().requires_grad_(True)
        out = c64.poses.unsqueeze(-1) * se3_exp(torch.where(c64.free.unsqueeze(-1), x, torch.zeros_like(x))).unsqueeze(-3)
        out = out.sum(-2)
        w = torch.randn_like(out)
        (g,) = torch.autograd.grad((out * w).sum(), x)
        num = torch.zeros_like(xi)
        eps = 1e-6
        for b in range(5):
            for k in range(6):
                e = torch.zeros_like(xi)
                e[b, k] = eps
                num[b, k] = ((f(xi + e) * w).sum() - (f(xi - e) * w).sum()) / (2 * eps)
        assert torch.allclose(g, num, rtol=1e-7, atol=1e-8), (g - num).abs().max()
        assert (g[3] == 0).all()
    # the module's own parameter path: fixed images get exactly zero gradient
    c64.delta.data = torch.zeros(5, 6, dtype=torch.float64)
    (c64() * torch.randn(5, 4, 4, dtype=torch.float64)).sum().backward()
    assert (c64.delta.grad[3] == 0).all() and (c64.delta.grad[[0, 1, 2, 4]] != 0).any()
    groups = c64.get_params(1e-3)
    assert groups[0]['params'][0] is c64.delta and groups[0]['lr'] == 1e-3


def test_se3_exp_is_a_rigid_transform_and_matches_the_matrix_exponential():
    from trinerflet_b200.poses import _hat, se3_exp
    xi = torch.randn(16, 6, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    xi[:4, :3] *= 1e-3                                                  # series branch
    T = se3_exp(xi)
    X = torch.zeros(16, 4, 4, dtype=torch.float64)
    X[:, :3, :3] = _hat(xi[:, :3])
    X[:, :3, 3] = xi[:, 3:]
    assert torch.allclose(T, torch.linalg.matrix_exp(X), atol=1e-12)


# ------------------------------------------------------------------------------------------------ autograd wiring (CPU tensors)
def test_python_wiring_on_the_host_build(monkeypatch, scene):
    from tests import emu_backend
    emu_backend.install(monkeypatch)
    from trinerflet_b200 import raymarching, rays as R
    from trinerflet_b200.poses import CameraPoses
    o, d, bits, nears, fars, noises = scene
    ro = torch.from_numpy(o).requires_grad_(True)
    rd = torch.from_numpy(d).requires_grad_(True)
    bitfield = torch.from_numpy(bits)
    nn_, ff = raymarching.near_far_from_aabb(ro, rd, torch.from_numpy(AABB), 0.2)
    assert not nn_.requires_grad and not ff.requires_grad
    counter = torch.zeros(2, dtype=torch.int32)
    xyzs, dirs, deltas, rays = raymarching.march_rays_train(ro, rd, BOUND, bitfield, CAS, H, nn_, ff, counter, len(o) * 40,
                                                            False, 128, False, 0.0, 1024)
    assert xyzs.requires_grad and dirs.requires_grad and not deltas.requires_grad and not rays.requires_grad
    # grad mode off: the plain entry point, no ray parameters recorded, nothing differentiable
    called = []
    real_call = raymarching.call
    monkeypatch.setattr(raymarching, "call", lambda name, *a: (called.append(name), real_call(name, *a))[1])
    with torch.no_grad():
        ng = raymarching.march_rays_train(ro, rd, BOUND, bitfield, CAS, H, nn_, ff, torch.zeros(2, dtype=torch.int32), len(o) * 40,
                                          False, 128, False, 0.0, 1024)
    assert called == ["tnl_march_rays_train"] and not ng[0].requires_grad
    monkeypatch.setattr(raymarching, "call", real_call)
    plain = raymarching.march_rays_train(ro.detach(), rd.detach(), BOUND, bitfield, CAS, H, nn_, ff, torch.zeros(2, dtype=torch.int32),
                                         len(o) * 40, False, 128, False, 0.0, 1024)
    for a, b in zip((xyzs, dirs, deltas, rays), plain):
        assert torch.equal(a.detach(), b)
    gx, gdir = torch.randn_like(xyzs), torch.randn_like(dirs)
    go, gd = torch.autograd.grad([xyzs, dirs], [ro, rd], [gx, gdir])
    M = xyzs.shape[0]
    # reconstruct ts from the march (t = the row's parameter) through the _ts entry point directly
    ts = np.zeros(M, np.float32)
    x2, d2, l2 = (np.zeros((M, w), np.float32) for w in (3, 3, 2))
    r2, c2 = np.empty((len(o), 3), np.int32), np.zeros(2, np.int32)
    wsz = kemu.lib().tnl_march_rays_train_workspace_fast(len(o), 1024)
    kemu.call("tnl_march_rays_train_ts", o, d, bits, BOUND, 0.0, 1024, len(o), CAS, H, M, nn_.numpy(), ff.numpy(), x2, d2, l2, ts,
              r2, c2, np.zeros(len(o), np.float32), np.zeros(wsz, np.uint8), wsz, None)
    want = _ray_kernel(r2, ts, o, d, gx.numpy(), gdir.numpy(), None, M)
    assert np.array_equal(go.numpy(), want[0]) and np.array_equal(gd.numpy(), want[1])
    # the feeder: pose gradient through select_batch(poses=CameraPoses()) equals the kernel on the same ray gradients
    P = torch.from_numpy(_poses(4, 9))
    feeder = R.RayFeeder(P, INTR, PH, PW, images=torch.rand(4, PH, PW, 3, generator=torch.Generator().manual_seed(0)), seed=0)
    cams = CameraPoses(P)
    data = feeder.select_batch(0, 500, poses=cams())
    assert data['rays_o'].requires_grad and not data['images'].requires_grad
    plain = feeder.select_batch(0, 500)
    assert torch.equal(data['rays_o'].detach(), plain['rays_o']) and torch.equal(data['rays_d'].detach(), plain['rays_d'])
    g_o, g_d = torch.randn(1, 500, 3), torch.randn(1, 500, 3)
    (gP,) = torch.autograd.grad([data['rays_o'], data['rays_d']], [cams.delta], [g_o, g_d])
    assert gP.shape == (4, 6) and torch.isfinite(gP).all() and (gP != 0).any()
    with pytest.raises(RuntimeError, match="out"):
        R.rays_from_ids(cams(), INTR, PH, PW, ray_ids=feeder.batch_ids(0, 10), out=(torch.empty(10, 3), torch.empty(10, 3)))


# ------------------------------------------------------------------------------------------------ argument checks
def test_new_entry_points_reject_bad_arguments():
    lib = kemu.lib()
    p = kemu.p
    a = np.zeros(64, np.float32)
    r = np.zeros((4, 3), np.int32)
    assert lib.tnl_rays_backward(None, p(a), p(a), p(a), 1.0, p(a), p(a), None, 4, 4, p(a), p(a), None) == -1
    assert lib.tnl_rays_backward(p(r), None, p(a), p(a), 1.0, p(a), p(a), None, 4, 4, p(a), p(a), None) == -1
    assert lib.tnl_rays_backward(p(r), p(a), p(a), p(a), 0.0, p(a), p(a), None, 4, 4, p(a), p(a), None) == -1
    assert lib.tnl_rays_backward(p(r), p(a), p(a), p(a), 1.0, p(a), p(a), None, 4, 4, None, p(a), None) == -1
    assert b"null" in lib.tnl_last_error()
    assert lib.tnl_rays_from_ids_backward(p(a), p(a), 2, 1.0, 1.0, 0.0, 0.0, 4, 4, None, 0, 8, None, None) == -1
    assert lib.tnl_rays_from_ids_backward(p(a), p(a), 2, 0.0, 1.0, 0.0, 0.0, 4, 4, None, 0, 8, p(a), None) == -1
    assert lib.tnl_rays_from_ids_backward(p(a), p(a), 0, 1.0, 1.0, 0.0, 0.0, 4, 4, None, 0, 8, p(a), None) == -1
    assert lib.tnl_rays_from_ids_backward(p(a), p(a), 2, 1.0, 1.0, 0.0, 0.0, 4, 4, None, 30, 8, p(a), None) == -1
    assert b"implicit id range" in lib.tnl_last_error()
    bits = np.zeros(2 * 32 ** 3 // 8, np.uint8)
    ws = np.zeros(1024, np.uint8)
    c = np.zeros(2, np.int32)
    args = [p(a), p(a), p(bits), 1.0, 0.0, 64, 4, 2, 32, 16, p(a), p(a), p(a), p(a), p(a)]
    assert lib.tnl_march_rays_train_ts(*args, None, p(r), p(c), p(a), p(ws), ws.size, None) == -1      # M > 0 needs ts
    assert lib.tnl_march_rays_train_ts(*args, p(a), p(r), p(c), p(a), p(ws), 0, None) < 0              # workspace too small
