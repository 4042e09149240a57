"""GPU: camera pose refinement.  The training march with ray parameters (tnl_march_rays_train_ts) against the plain march; ray
gradients through NeRFNetwork.render against a literal torch graph (march positions with t held fixed, the reference's field
from tests/field_truth.py, compositing restated in torch with the T < T_thresh stop); pose gradients through the ray feeder and
get_rays against fp64 autograd of the reference's get_rays; pose-refinement steps through TrainStep (dense and work-list IDWT,
bit-reproducible in deterministic mode); and the unchanged training path when no ray requires grad."""
import math

import pytest
import torch

from tests import field_truth as ft
from tests.util import rel_l2

pytestmark = pytest.mark.gpu

BOUND = 1.5


def _net(C=16, R=128, S=2, seed=0, smooth=False):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    net = NeRFNetwork(bound=BOUND, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=C, triplane_resolution=R,
                      triplane_wavelet_levels=S, hidden_dim=64, hidden_dim_color=64).cuda()
    scene.init_model_(net, seed=seed)
    if smooth:                                   # finer wavelet levels zeroed: the planes are the upsampled base planes
        with torch.no_grad():
            for p in net.encoder.planes_features_wavelet_coefs:
                p.zero_()
        net.encoder.reset_cahce()
    scene.install_ball_occupancy(net, 0.75)
    return net


def _rays(n, seed):
    from trinerflet_b200 import scene
    ro, rd, tgt = scene.sample_batch(scene.make_scene(), n, torch.Generator().manual_seed(seed))
    return ro.cuda(), rd.cuda(), tgt.cuda()


def _march(net, ro, rd, M, with_ts, fast=True):
    """one direct ABI call of the training march -> xyzs, dirs, deltas, rays, counter (, ts)"""
    from trinerflet_b200 import _lib, raymarching
    N = ro.shape[0]
    nears, fars = raymarching.near_far_from_aabb(ro, rd, net.aabb_train, net.min_near)
    out = [torch.full((M, w), float("nan"), device="cuda") for w in (3, 3, 2)]
    rays, counter = torch.empty(N, 3, dtype=torch.int32, device="cuda"), torch.zeros(2, dtype=torch.int32, device="cuda")
    ts = torch.full((M,), float("nan"), device="cuda")
    lib = _lib.load()
    wsz = lib.tnl_march_rays_train_workspace_fast(N, 1024) if fast else lib.tnl_march_rays_train_workspace(N)
    ws = torch.zeros(wsz, dtype=torch.uint8, device="cuda")
    noises = torch.zeros(N, device="cuda")
    p = _lib.ptr
    head = (p(ro), p(rd), p(net.density_bitfield), BOUND, 0.0, 1024, N, net.cascade, net.grid_size, M, p(nears), p(fars),
            p(out[0]), p(out[1]), p(out[2]))
    tail = (p(rays), p(counter), p(noises), p(ws), wsz, _lib.stream())
    if with_ts:
        _lib.call("tnl_march_rays_train_ts", *head, p(ts), *tail)
        return (*out, rays, counter, ts)
    _lib.call("tnl_march_rays_train", *head, *tail)
    return (*out, rays, counter)


def _owner(rays, M):
    """row -> ray index (-1: no ray owns the row)"""
    own = torch.full((M,), -1, dtype=torch.long, device=rays.device)
    r = rays.long()
    keep = (r[:, 2] > 0) & (r[:, 1] + r[:, 2] <= M)
    idx = torch.repeat_interleave(torch.arange(len(r), device=rays.device)[keep], r[keep, 2])
    rows = torch.repeat_interleave(r[keep, 1], r[keep, 2]) + (torch.arange(len(idx), device=rays.device)
                                                              - torch.repeat_interleave(torch.cumsum(r[keep, 2], 0) - r[keep, 2], r[keep, 2]))
    own[rows] = idx
    return own


@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("frac", [2.0, 0.6])           # 0.6: M below the sample count, rays are dropped
def test_march_ts_bit_identical_and_ts_reproduces_xyzs(fast, frac):
    net = _net()
    ro, rd, _ = _rays(6000, 1)
    total = int(_march(net, ro, rd, 0, False)[4][0])
    M = int(total * frac) // 128 * 128
    plain = _march(net, ro, rd, M, False, fast)
    *outs, ts = _march(net, ro, rd, M, True, fast)
    for a, b in zip(plain, outs):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    own = _owner(outs[3], M)
    dropped = (outs[3][:, 1] + outs[3][:, 2] > M) & (outs[3][:, 2] > 0)
    assert (frac < 1) == bool(dropped.any()) and (ts[own < 0] == 0).all()
    r = own[own >= 0]
    t = ts[own >= 0].double()
    u = (t[:, None] * rd[r].double() + ro[r].double()).float()        # t*d exact in fp64: the fma's single rounding
    assert torch.equal(u.clamp(-BOUND, BOUND).view(torch.int32), outs[0][own >= 0].view(torch.int32))


def _composite_truth(sigma, rgb, deltas, own, N, T_thresh=1e-4):
    """compositing of the training render restated in torch (reference raymarching.cu:500-682): per ray, in sample order,
    w = alpha T with T the transmittance before the sample; samples after the first one with T (1 - alpha) < T_thresh get 0"""
    rows = torch.nonzero(own >= 0).squeeze(1)
    ray = own[rows]
    K = int(torch.bincount(ray, minlength=N).max())
    start = torch.zeros(N, dtype=torch.long, device=own.device)
    first = torch.ones_like(ray, dtype=torch.bool)
    first[1:] = ray[1:] != ray[:-1]
    start[ray[first]] = rows[first]
    k = rows - start[ray]
    A = torch.zeros(N, K, device=own.device, dtype=sigma.dtype)
    alpha = 1 - torch.exp(-sigma[rows] * deltas[rows, 0])
    A = A.index_put((ray, k), alpha)
    C = torch.zeros(N, K, 3, device=own.device, dtype=rgb.dtype).index_put((ray, k), rgb[rows])
    Tcum = torch.cumprod(1 - A, dim=1)
    T_ex = torch.cat([torch.ones_like(Tcum[:, :1]), Tcum[:, :-1]], 1)
    stop_before = torch.cat([torch.zeros_like(Tcum[:, :1], dtype=torch.bool), (Tcum < T_thresh)[:, :-1]], 1)
    keep = ~(torch.cumsum(stop_before.int(), 1) > 0)
    w = A * T_ex * keep
    tt = torch.zeros(N, K, device=own.device).index_put((ray, k), deltas[rows, 1]).cumsum(1)
    return w.sum(1), (w.detach() * tt).sum(1), (w.unsqueeze(-1) * C).sum(1)


def _literal_ray_grads(net, ro, rd, tgt, M, autocast, lam_depth):
    """autograd.grad(loss, (rays_o, rays_d)) of the literal graph"""
    xyzs, dirs, deltas, rays, counter, ts = _march(net, ro, rd, M, True)
    own = _owner(rays, M)
    ro = ro.detach().clone().requires_grad_(True)
    rd = rd.detach().clone().requires_grad_(True)
    valid = own >= 0
    r = own.clamp(min=0)
    u = ro[r] + ts[:, None] * rd[r]
    xyz = torch.where(valid[:, None], xyzs + (u.clamp(-BOUND, BOUND) - u.clamp(-BOUND, BOUND).detach()), xyzs)
    dd = torch.where(valid[:, None], dirs + (rd[r] - rd[r].detach()), dirs)
    planes = net.encoder.get_planes().detach()
    W = [w.detach() for w in net._weights()]
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        sigma, rgb = ft.field(planes, xyz[valid], dd[valid], W, BOUND)
    sig = torch.zeros(M, device="cuda").index_put((torch.nonzero(valid).squeeze(1),), sigma.float())
    col = torch.zeros(M, 3, device="cuda").index_put((torch.nonzero(valid).squeeze(1),), rgb.float())
    ws, depth, image = _composite_truth(sig, col, deltas, own, ro.shape[0])
    from trinerflet_b200 import raymarching
    nears, fars = raymarching.near_far_from_aabb(ro.detach(), rd.detach(), net.aabb_train, net.min_near)
    image = image + (1 - ws).unsqueeze(-1) * 0.0
    depth = torch.clamp(depth - nears, min=0) / (fars - nears)
    loss = ((image - tgt) ** 2).mean() + lam_depth * torch.nan_to_num(depth).mean()
    return torch.autograd.grad(loss, (ro, rd)), int((own >= 0).sum())


def _product_ray_grads(net, ro, rd, tgt, mean_count, autocast, lam_depth):
    ro = ro.detach().clone().requires_grad_(True)
    rd = rd.detach().clone().requires_grad_(True)
    net.train()
    net.mean_count = mean_count
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        out = net.render(ro.unsqueeze(0), rd.unsqueeze(0), staged=False, bg_color=0.0, perturb=False, force_all_rays=False,
                         dt_gamma=0, max_steps=1024)
        loss = ((out['image'].view(-1, 3).float() - tgt) ** 2).mean() + lam_depth * torch.nan_to_num(out['depth']).mean()
    return torch.autograd.grad(loss, (ro, rd))


@pytest.mark.parametrize("autocast,tol", [(False, 1e-4), (True, 1e-2)])
@pytest.mark.parametrize("drop", [False, True])
@pytest.mark.parametrize("lam_depth", [0.0, 0.5])
def test_ray_gradients_through_render_match_the_literal_graph(autocast, tol, drop, lam_depth):
    net = _net()
    ro, rd, tgt = _rays(3000, 2)
    total = int(_march(net, ro, rd, 0, False)[4][0])
    mean_count = int(total * 0.6) if drop else 0
    M = total if not drop else mean_count + 128 - mean_count % 128
    (go, gd), used = _literal_ray_grads(net, ro, rd, tgt, M, autocast, lam_depth)
    assert (used < total) == drop
    po, pd = _product_ray_grads(net, ro, rd, tgt, mean_count, autocast, lam_depth)
    assert rel_l2(po, go) <= tol and rel_l2(pd, gd) <= tol, (rel_l2(po, go), rel_l2(pd, gd))
    if drop:
        dead = _march(net, ro, rd, M, False)[3]
        dead = (dead[:, 1] + dead[:, 2] > M) | (dead[:, 2] == 0)
        assert dead.any() and (po[dead] == 0).all() and (pd[dead] == 0).all()


# ------------------------------------------------------------------------------------------------ pose gradients
def _restated_get_rays64(P, intr, H, W, ids):
    """the reference's get_rays per ray in fp64: dir = normalise((i+0.5-cx)/fx, (j+0.5-cy)/fy, 1), rays_d = dir @ R^T"""
    fx, fy, cx, cy = intr
    ids = ids.clamp(0, P.shape[0] * H * W - 1)
    img, pix = ids // (H * W), ids % (H * W)
    i = (pix % W).double() + 0.5
    j = (pix // W).double() + 0.5
    v = torch.stack([(i - cx) / fx, (j - cy) / fy, torch.ones_like(i)], -1)
    v = v / v.norm(dim=-1, keepdim=True)
    return P[img, :3, 3], (v.unsqueeze(1) * P[img, :3, :3]).sum(-1)


def _cams(B=8, H=48, W=64, seed=0, fov=0.25):
    from trinerflet_b200 import scene
    P = scene.make_poses(B, seed).cuda()
    f = 0.5 * W / math.tan(0.5 * fov)
    return P, (f, f * 1.01, W / 2 + 0.3, H / 2 - 0.2), H, W


def test_pose_gradients_through_the_feeder_and_get_rays():
    from trinerflet_b200 import rays as R
    P, intr, H, W = _cams()
    images = torch.rand(8, H, W, 3, device="cuda")
    feeder = R.RayFeeder(P, intr, H, W, images, seed=3)
    g = torch.Generator(device="cuda").manual_seed(0)
    for b, bs in ((0, 5000), (3, 7000)):
        Pg = P.clone().requires_grad_(True)
        data = feeder.select_batch(b, bs, poses=Pg)
        plain = feeder.select_batch(b, bs)
        assert torch.equal(data['rays_o'].detach(), plain['rays_o']) and torch.equal(data['rays_d'].detach(), plain['rays_d'])
        assert not data['images'].requires_grad
        n = data['rays_o'].shape[1]
        g_o, g_d = torch.randn(1, n, 3, device="cuda", generator=g), torch.randn(1, n, 3, device="cuda", generator=g)
        (gP,) = torch.autograd.grad([data['rays_o'], data['rays_d']], [Pg], [g_o, g_d])
        P64 = P.double().requires_grad_(True)
        o64, d64 = _restated_get_rays64(P64, intr, H, W, feeder.batch_ids(b, bs))
        (want,) = torch.autograd.grad([o64, d64], [P64], [g_o[0].double(), g_d[0].double()])
        assert rel_l2(gP, want) <= 1e-5 and (gP[:, 3] == 0).all()
    # get_rays: random pixels shared by the B poses, and the full frame (first_id form)
    for N in (300, -1):
        Pg = P.clone().requires_grad_(True)
        res = R.get_rays(Pg, intr, H, W, N=N)
        n = res['rays_o'].shape[1]
        g_o, g_d = torch.randn(8, n, 3, device="cuda", generator=g), torch.randn(8, n, 3, device="cuda", generator=g)
        (gP,) = torch.autograd.grad([res['rays_o'], res['rays_d']], [Pg], [g_o, g_d])
        ids = (res['inds'] + (torch.arange(8, device="cuda") * H * W).unsqueeze(1)).reshape(-1)
        P64 = P.double().requires_grad_(True)
        o64, d64 = _restated_get_rays64(P64, intr, H, W, ids)
        (want,) = torch.autograd.grad([o64, d64], [P64], [g_o.reshape(-1, 3).double(), g_d.reshape(-1, 3).double()])
        assert rel_l2(gP, want) <= 1e-5
    # an image with no ray in the batch gets exactly zero
    Pg = P.clone().requires_grad_(True)
    ro, rd = R.rays_from_ids(Pg, intr, H, W, ray_ids=torch.arange(2 * H * W, 3 * H * W, device="cuda"))
    (gP,) = torch.autograd.grad([ro, rd], [Pg], [torch.ones_like(ro), torch.ones_like(rd)])
    assert (gP[torch.arange(8) != 2] == 0).all() and (gP[2, :3] != 0).all()


def test_backward_kernels_repeat_bit_for_bit_with_the_flag_off():
    from trinerflet_b200 import _lib
    assert not torch.are_deterministic_algorithms_enabled()
    net = _net()
    ro, rd, _ = _rays(20000, 4)
    total = int(_march(net, ro, rd, 0, False)[4][0])
    xyzs, dirs, deltas, rays, counter, ts = _march(net, ro, rd, total, True)
    gx, gdir = torch.randn_like(xyzs), torch.randn_like(dirs)
    res = []
    for _ in range(3):
        go, gd = torch.empty_like(ro), torch.empty_like(rd)
        _lib.call("tnl_rays_backward", _lib.ptr(rays), _lib.ptr(ts), _lib.ptr(ro), _lib.ptr(rd), BOUND, _lib.ptr(gx), _lib.ptr(gdir),
                  None, ro.shape[0], total, _lib.ptr(go), _lib.ptr(gd), _lib.stream())
        gP = torch.empty(100, 4, 4, device="cuda")
        ids = torch.randint(0, 100 * 800 * 800, (ro.shape[0],), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
        _lib.call("tnl_rays_from_ids_backward", _lib.ptr(go), _lib.ptr(gd), 100, 1111.0, 1111.0, 400.0, 400.0, 800, 800, _lib.ptr(ids),
                  0, ro.shape[0], _lib.ptr(gP), _lib.stream())
        res.append(torch.cat([go.view(-1), gd.view(-1), gP.view(-1)]))
    assert all(torch.equal(r.view(torch.int32), res[0].view(torch.int32)) for r in res)


# ------------------------------------------------------------------------------------------------ refinement steps through TrainStep
def _refine_setup(seed=0, fp16=True, radius=None, fov=0.25, H=48, W=64, contrast=1.0, rot_deg=(0.2, 0.4), trans=(0.0045, 0.009),
                  lr=2e-4, n_avg=1):
    """frozen field + 8 cameras looking at it + targets rendered at the true poses + CameraPoses at perturbed poses.
    radius: camera distance from the origin (None: the scene's 4.03); contrast scales the base planes (texture); rotation
    perturbation angles uniform in rot_deg (degrees), translation lengths uniform in trans (scene units); n_avg > 1: the targets
    are the mean of n_avg jittered training renders, i.e. what the jittered training render gives on average"""
    from trinerflet_b200 import rays as R, trainer
    from trinerflet_b200.poses import CameraPoses, se3_exp
    net = _net(smooth=True, seed=seed)
    if contrast != 1.0:
        with torch.no_grad():
            net.encoder.planes_features.mul_(contrast)
        net.encoder.reset_cahce()
    P, intr, H, W = _cams(8, H, W, seed=5, fov=fov)
    if radius is not None:
        P[:, :3, 3] *= radius / P[:, :3, 3].norm(dim=-1, keepdim=True)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=fp16):
        net.train()
        ro, rd = R.rays_from_ids(P, intr, H, W, first_id=0, n=8 * H * W)
        img = sum(net.render(ro.unsqueeze(0), rd.unsqueeze(0), staged=False, bg_color=0.0, perturb=n_avg > 1, force_all_rays=True,
                             max_steps=1024)['image'].view(8, H, W, 3).float() for _ in range(n_avg)) / n_avg
    feeder = R.RayFeeder(P, intr, H, W, img, seed=seed)
    g = torch.Generator().manual_seed(11 + seed)
    ang = (torch.rand(8, generator=g) * (rot_deg[1] - rot_deg[0]) + rot_deg[0]) * math.pi / 180
    axis = torch.randn(8, 3, generator=g)
    axis = axis / axis.norm(dim=-1, keepdim=True)
    dt = torch.randn(8, 3, generator=g)
    dt = dt / dt.norm(dim=-1, keepdim=True) * (torch.rand(8, 1, generator=g) * (trans[1] - trans[0]) + trans[0])
    xi = torch.cat([axis * ang[:, None], dt], -1)
    noisy = P @ se3_exp(xi).cuda()
    cams = CameraPoses(noisy)
    opt = torch.optim.Adam(cams.get_params(lr), betas=(0.9, 0.99), eps=1e-15)
    step = trainer.TrainStep(net, trainer.default_opt(fp16=fp16, wavelet_regularization=0.0), opt)
    step.perturbation = xi
    return net, P, cams, feeder, step


def _pose_errors(P, Q):
    """per camera: rotation error (degrees, fp64) and camera-centre distance"""
    Rr = P[:, :3, :3].double().transpose(1, 2) @ Q[:, :3, :3].double()
    skew = torch.stack([Rr[:, 2, 1] - Rr[:, 1, 2], Rr[:, 0, 2] - Rr[:, 2, 0], Rr[:, 1, 0] - Rr[:, 0, 1]], -1)
    cos = (Rr.diagonal(dim1=1, dim2=2).sum(-1) - 1) / 2
    ang = torch.atan2(0.5 * skew.norm(dim=-1), cos)
    return ang * 180 / math.pi, (P[:, :3, 3].double() - Q[:, :3, 3].double()).norm(dim=-1)


def _refine(net, cams, feeder, step, n_steps, bs=4096):
    sched = torch.optim.lr_scheduler.LambdaLR(step.optimizer, lambda i: 0.02 ** min(i / n_steps, 1))
    for i in range(n_steps):
        b = i % feeder.steps_per_epoch(bs)
        if b == 0:
            feeder.shuffle()
        data = feeder.select_batch(b, bs, poses=cams())
        net.zero_grad(set_to_none=True)
        step.forward_backward(data['rays_o'][0], data['rays_d'][0], data['images'][0], update_grid=False)
        step.optimizer_step()
        sched.step()


# cameras at 1.6 scene units from the origin with a 1.5 rad field of view: the ball of occupied space (radius 0.75) spans depths
# 0.85 .. 2.35, so a small rotation and a sideways translation move the image differently (parallax).  With the scene's far,
# narrow cameras (4.03 units, 0.25 rad) the two are nearly the same image shift, the problem is ill-conditioned and Adam does
# not separate them.  The base planes are scaled by 10: the random init's colours and densities are nearly uniform.
RECOVERY = dict(radius=1.6, fov=1.5, H=96, W=128, contrast=10.0, lr=2e-4)


def test_perturbed_cameras_are_recovered():
    """8 cameras of 96x128 pixels around a frozen smooth field (finer wavelet levels zeroed, ball occupancy), perturbed by
    0.23-0.40 degrees and 0.0046-0.0090 scene units (0.3-0.6 % of the bound); 1500 steps of 16384 rays through
    TrainStep.forward_backward (fp16 autocast, work-list IDWT, jittered march) + Adam (lr 2e-4 decayed to 4e-6) on CameraPoses
    alone.  Measured on a B200, the largest ratio of final to initial error over the cameras after 300 / 600 / 900 / 1200 / 1500
    steps: rotation 0.47 / 0.20 / 0.16 / 0.14 / 0.14, translation 0.30 / 0.14 / 0.13 / 0.14 / 0.14.  Per camera, rotation
    0.230 0.297 0.397 0.234 0.317 0.339 0.317 0.226 deg -> 0.0091 0.0067 0.0041 0.030 0.011 0.013 0.013 0.031 deg, translation
    0.0046 0.0069 0.0059 0.0068 0.0057 0.0065 0.0080 0.0090 -> 0.00023 0.00024 0.00025 0.00093 0.00049 0.00038 0.00053 0.00083.
    Bar: every camera's rotation and translation error <= 1/4 of its initial value (measured <= 0.14)."""
    torch.manual_seed(0)
    net, P, cams, feeder, step = _refine_setup(**RECOVERY)
    r0, t0 = _pose_errors(P, cams().detach())
    _refine(net, cams, feeder, step, 1500, bs=16384)
    r1, t1 = _pose_errors(P, cams().detach())
    assert (r1 <= 0.25 * r0).all() and (t1 <= 0.25 * t0).all(), (r1 / r0, t1 / t0)


def test_seeded_pose_refinement_is_bit_reproducible_in_deterministic_mode():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        outs = []
        for _ in range(2):
            torch.manual_seed(3)
            net, P, cams, feeder, step = _refine_setup(seed=1)
            _refine(net, cams, feeder, step, 12)
            outs.append(torch.cat([cams.delta.detach().view(-1), cams().detach().view(-1)] +
                                  [s.view(-1) for s in step.optimizer.state[cams.delta].values() if torch.is_tensor(s) and s.dim()]))
        assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    finally:
        torch.use_deterministic_algorithms(prev)


def test_dense_and_work_list_steps_give_the_same_pose_gradient():
    torch.manual_seed(0)
    net, P, cams, feeder, step = _refine_setup()
    data = feeder.select_batch(0, 4096, poses=None)
    grads = []
    for sparse in (True, False):
        step.sparse_idwt = sparse
        net.zero_grad(set_to_none=True)
        cams.zero_grad(set_to_none=True)
        torch.manual_seed(7)      # the march's jitter
        d = feeder.select_batch(0, 4096, poses=cams())
        step.forward_backward(d['rays_o'][0], d['rays_d'][0], d['images'][0], update_grid=False)
        grads.append(cams.delta.grad.clone())
    assert grads[0].abs().sum() > 0 and rel_l2(grads[1], grads[0]) <= 1e-5
    with pytest.raises(RuntimeError, match="capture"):
        step.capture(data['rays_o'][0].clone().requires_grad_(True), data['rays_d'][0], data['images'][0])


def test_rays_without_grad_keep_the_fused_training_path_and_its_bits(monkeypatch):
    from trinerflet_b200 import network, trainer
    calls = []
    orig = network._Field.apply
    with monkeypatch.context() as m:
        m.setattr(network._Field, "apply", lambda *a: (calls.append(1), orig(*a))[1])
        net = _net(C=32, R=256, S=4)
        ro, rd, tgt = _rays(1 << 17, 6)
        step = trainer.TrainStep(net, trainer.default_opt(), None)
        step.forward_backward(ro, rd, tgt, update_grid=False)
        assert calls
    # deterministic mode: a default step gives the same loss and gradients whether the step before it on the same model and
    # TrainStep was a default one or a pose-refinement one (rays that require grad, the _ts march and both backward kernels)
    from trinerflet_b200.poses import CameraPoses
    from trinerflet_b200 import rays as R
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        res = []
        for refine_first in (False, True):
            net = _net(C=32, R=256, S=4)
            step = trainer.TrainStep(net, trainer.default_opt(), None)
            P, intr, H, W = _cams(8, 96, 128, fov=1.0)
            cams = CameraPoses(P)
            images = torch.rand(8, H, W, 3, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
            data = R.RayFeeder(P, intr, H, W, images, seed=0).select_batch(0, 1 << 16, poses=cams() if refine_first else None)
            assert data['rays_o'].requires_grad == refine_first
            torch.manual_seed(4)
            step.forward_backward(data['rays_o'][0], data['rays_d'][0], data['images'][0], update_grid=False)
            assert (cams.delta.grad is not None) == refine_first
            net.zero_grad(set_to_none=True)
            torch.manual_seed(5)
            loss = step.forward_backward(ro, rd, tgt, update_grid=False)
            res.append(torch.cat([loss.reshape(-1)] + [p.grad.reshape(-1) for p in net.parameters() if p.grad is not None]))
        assert torch.equal(res[0].view(torch.int32), res[1].view(torch.int32))
    finally:
        torch.use_deterministic_algorithms(prev)
