"""GPU parity: trinerflet_b200.raymarching (C ABI -> sm_100a kernels) against
  (1) the plain-C oracle restatement (oracle/raymarch.c), and
  (2) the UNMODIFIED reference kernels compiled from /root/reference (oracle/_ref/_raymarching_ref.so), when present.
Integer results and fp32 sample positions must be bit-exact; composited floats carry the tolerance written below
(the GPU uses ex2.approx for __expf, the C oracle expf)."""
import os

import numpy as np
import pytest
import torch

from tests.util import random_bitfield, synthetic_rays

pytestmark = pytest.mark.gpu

BOUND, CAS, H = 1.5, 2, 128
COMPOSITE_ATOL = 2e-5   # fp32 composited rgb / depth / weights vs C oracle (expf vs ex2.approx, ~300 terms)
COMPOSITE_ATOL_REF = 1e-6  # vs the reference kernel itself (same __expf): identical up to FMA-contraction choices


def _setup(n=4096, seed=0, max_steps=1024):
    from trinerflet_b200 import raymarching as rm
    o, d = synthetic_rays(n, seed)
    _, bits = random_bitfield(seed)
    dev = torch.device("cuda")
    ro, rd, bf = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev), bits.to(dev)
    aabb = torch.tensor([-BOUND] * 3 + [BOUND] * 3, device=dev)
    nears, fars = rm.near_far_from_aabb(ro, rd, aabb, 0.2)
    return rm, o, d, bits, ro, rd, bf, aabb, nears, fars


def _ref():
    from oracle import build_ref
    return build_ref.load_ref("raymarching")


def test_near_far_morton_packbits_bitexact():
    from oracle import raymarch as orc
    rm, o, d, bits, ro, rd, bf, aabb, nears, fars = _setup()
    n_o, f_o = orc.near_far_from_aabb(o, d, aabb.cpu().numpy(), 0.2)
    assert np.array_equal(nears.cpu().numpy(), n_o) and np.array_equal(fars.cpu().numpy(), f_o)
    rng = np.random.default_rng(1)
    c = rng.integers(0, 128, (100000, 3)).astype(np.int32)
    idx = rm.morton3D(torch.from_numpy(c).cuda())
    assert np.array_equal(idx.cpu().numpy(), orc.morton3D(c))
    back = rm.morton3D_invert(idx)
    assert np.array_equal(back.cpu().numpy(), c)
    grid = torch.from_numpy(rng.random((2, 128 ** 3)).astype(np.float32))
    for thresh in (0.0, 0.3, 0.999):
        pb = rm.packbits(grid.cuda(), thresh)
        assert np.array_equal(pb.cpu().numpy(), orc.packbits(grid.numpy(), thresh))
        assert np.array_equal(pb.cpu().numpy(), np.packbits(grid.numpy().reshape(-1) > thresh, bitorder='little'))
    ref = _ref()
    if ref is not None:
        n_r, f_r = torch.empty_like(nears), torch.empty_like(fars)
        ref.near_far_from_aabb(ro, rd, aabb, ro.shape[0], 0.2, n_r, f_r)
        assert torch.equal(n_r, nears) and torch.equal(f_r, fars)
        pb_r = torch.empty(2 * 128 ** 3 // 8, dtype=torch.uint8, device="cuda")
        ref.packbits(grid.cuda(), pb_r.numel(), 0.3, pb_r)
        assert torch.equal(pb_r, rm.packbits(grid.cuda(), 0.3))


@pytest.mark.parametrize("max_steps,dt_gamma", [(1024, 0.0), (512, 1.0 / 128)])
def test_march_rays_train_bitexact(max_steps, dt_gamma):
    from oracle import raymarch as orc
    rm, o, d, bits, ro, rd, bf, aabb, nears, fars = _setup(max_steps=max_steps)
    N = o.shape[0]
    torch.manual_seed(3)
    noises = torch.rand(N, device="cuda")
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    # go through the C ABI directly so that the noises are shared with the oracle
    from trinerflet_b200 import _lib
    lib = _lib.load()
    M = N * 256
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); deltas = torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda")
    # both forms of the second pass: re-traversal (small workspace) first, then emission from the recorded sample parameters;
    # the outputs start as NaN (the call zero-fills the rows no ray owns) and must come out bit-identical
    outs = []
    for wsz in (lib.tnl_march_rays_train_workspace(N), lib.tnl_march_rays_train_workspace_fast(N, max_steps)):
        xyzs.fill_(float("nan")); dirs.fill_(float("nan")); deltas.fill_(float("nan")); counter.zero_()
        ws = torch.empty(wsz, dtype=torch.uint8, device="cuda")
        _lib.call("tnl_march_rays_train", _lib.ptr(ro), _lib.ptr(rd), _lib.ptr(bf), BOUND, dt_gamma, max_steps, N, CAS, H, M,
                  _lib.ptr(nears), _lib.ptr(fars), _lib.ptr(xyzs), _lib.ptr(dirs), _lib.ptr(deltas), _lib.ptr(rays),
                  _lib.ptr(counter), _lib.ptr(noises), _lib.ptr(ws), ws.numel(), _lib.stream())
        outs.append([t.clone() for t in (xyzs, dirs, deltas, rays, counter)])
    for a, b in zip(*outs):
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)
    x_o, d_o, l_o, r_o, c_o = orc.march_rays_train(o, d, BOUND, bits.numpy(), CAS, H, nears.cpu().numpy(),
                                                   fars.cpu().numpy(), noises.cpu().numpy(), M, dt_gamma, max_steps)
    assert np.array_equal(counter.cpu().numpy(), c_o)
    assert np.array_equal(rays.cpu().numpy(), r_o)          # ray order, offsets and counts
    total = int(c_o[0])
    assert total > N  # the scene is not empty
    assert np.array_equal(xyzs.cpu().numpy().view(np.uint32), x_o.view(np.uint32))
    assert np.array_equal(dirs.cpu().numpy().view(np.uint32), d_o.view(np.uint32))
    assert np.array_equal(deltas.cpu().numpy().view(np.uint32), l_o.view(np.uint32))
    ref = _ref()
    if ref is not None:  # the reference kernel: slot order is a race, compare per ray after sorting by ray id
        xr = torch.zeros_like(xyzs); dr = torch.zeros_like(dirs); lr = torch.zeros_like(deltas)
        rr = torch.empty_like(rays); cr = torch.zeros_like(counter)
        ref.march_rays_train(ro, rd, bf, BOUND, dt_gamma, max_steps, N, CAS, H, M, nears, fars, xr, dr, lr, rr, cr, noises)
        assert torch.equal(cr, counter)
        rr = rr.cpu().numpy(); rr = rr[np.argsort(rr[:, 0])]
        mine = rays.cpu().numpy()
        assert np.array_equal(rr[:, 0], mine[:, 0]) and np.array_equal(rr[:, 2], mine[:, 2])
        xr, lr, xm, lm = xr.cpu().numpy(), lr.cpu().numpy(), xyzs.cpu().numpy(), deltas.cpu().numpy()
        for n in np.random.default_rng(0).choice(N, 512, replace=False):
            a, b, k = rr[n, 1], mine[n, 1], mine[n, 2]
            assert np.array_equal(xr[a:a + k].view(np.uint32), xm[b:b + k].view(np.uint32))
            assert np.array_equal(lr[a:a + k].view(np.uint32), lm[b:b + k].view(np.uint32))


def test_march_overflow_and_empty_and_full():
    from trinerflet_b200 import raymarching as rm
    _, o, d, bits, ro, rd, bf, aabb, nears, fars = _setup(1024)
    N = ro.shape[0]
    empty = torch.zeros_like(bf)
    c = torch.zeros(2, dtype=torch.int32, device="cuda")
    x, dd, dl, rays = rm.march_rays_train(ro, rd, BOUND, empty, CAS, H, nears, fars, c, -1, False, 128, True, 0, 1024)
    assert int(c[0]) == 0 and int(c[1]) == N and x.shape[0] == 128 and int(rays[:, 2].sum()) == 0
    full = torch.full_like(bf, 255)
    c.zero_()
    x, dd, dl, rays = rm.march_rays_train(ro, rd, BOUND, full, CAS, H, nears, fars, c, -1, False, 128, True, 0, 64)
    from oracle import raymarch as orc
    r_o = orc.march_rays_train(o, d, BOUND, full.cpu().numpy(), CAS, H, nears.cpu().numpy(), fars.cpu().numpy(),
                               np.zeros(N, np.float32), 0, 0.0, 64)[3]
    assert np.array_equal(rays.cpu().numpy(), r_o) and int(rays[:, 2].max()) == 64   # long chords saturate max_steps
    # overflow: M smaller than needed -> late rays dropped silently, earlier ones intact
    c.zero_()
    x2, _, _, rays2 = rm.march_rays_train(ro, rd, BOUND, full, CAS, H, nears, fars, c, 128 * 50, False, 128, False, 0, 64)
    M = x2.shape[0]
    assert M == 128 * 51 and torch.equal(rays2, rays)
    keep = (rays2[:, 1] + rays2[:, 2] <= M).cpu().numpy()
    last = int((rays2[:, 1] + rays2[:, 2])[torch.from_numpy(keep).cuda()].max())
    assert torch.equal(x2[:last], x[:last]) and float(x2[last:].abs().sum()) == 0.0


def test_composite_train_fwd_bwd():
    from oracle import raymarch as orc
    from trinerflet_b200 import raymarching as rm
    _, o, d, bits, ro, rd, bf, aabb, nears, fars = _setup(2048)
    N = ro.shape[0]
    c = torch.zeros(2, dtype=torch.int32, device="cuda")
    torch.manual_seed(0)
    xyzs, dirs, deltas, rays = rm.march_rays_train(ro, rd, BOUND, bf, CAS, H, nears, fars, c, -1, True, 128, True, 0, 1024)
    M = xyzs.shape[0]
    sig = (torch.rand(M, device="cuda") * 40).requires_grad_(True)
    rgb = torch.rand(M, 3, device="cuda").requires_grad_(True)
    ws, depth, img = rm.composite_rays_train(sig, rgb, deltas, rays, 1e-4)
    ws_o, dp_o, im_o = orc.composite_rays_train_forward(sig.detach().cpu().numpy(), rgb.detach().cpu().numpy(),
                                                         deltas.cpu().numpy(), rays.cpu().numpy(), 1e-4)
    assert np.abs(ws.detach().cpu().numpy() - ws_o).max() <= COMPOSITE_ATOL
    assert np.abs(img.detach().cpu().numpy() - im_o).max() <= COMPOSITE_ATOL
    assert np.abs(depth.detach().cpu().numpy() - dp_o).max() <= 10 * COMPOSITE_ATOL
    gws, gim = torch.randn(N, device="cuda"), torch.randn(N, 3, device="cuda")
    (ws * gws).sum().backward(retain_graph=True)
    g_s1 = sig.grad.clone(); sig.grad = None; g_r1 = rgb.grad.clone(); rgb.grad = None
    ((ws * gws).sum() + (img * gim).sum()).backward()
    gs_o, gc_o = orc.composite_rays_train_backward(gws.cpu().numpy(), gim.cpu().numpy(), sig.detach().cpu().numpy(),
                                                   rgb.detach().cpu().numpy(), deltas.cpu().numpy(), rays.cpu().numpy(),
                                                   ws_o, im_o, 1e-4)
    assert np.abs(rgb.grad.cpu().numpy() - gc_o).max() <= COMPOSITE_ATOL
    denom = np.abs(gs_o).max()
    assert np.abs(sig.grad.cpu().numpy() - gs_o).max() / denom <= 1e-4   # grad_sigma: stated rel tolerance 1e-4 (fp32)
    ref = _ref()
    if ref is not None:
        ws_r, dp_r, im_r = torch.empty_like(ws), torch.empty_like(depth), torch.empty_like(img)
        ref.composite_rays_train_forward(sig.detach(), rgb.detach(), deltas, rays, M, N, 1e-4, ws_r, dp_r, im_r)
        assert (ws_r - ws).abs().max().item() <= COMPOSITE_ATOL_REF and (im_r - img).abs().max().item() <= COMPOSITE_ATOL_REF
        assert (dp_r - depth).abs().max().item() <= 10 * COMPOSITE_ATOL_REF
        gs_r, gc_r = torch.zeros_like(sig), torch.zeros_like(rgb)
        ref.composite_rays_train_backward(gws, gim, sig.detach(), rgb.detach(), deltas, rays, ws_r, im_r, M, N, 1e-4, gs_r, gc_r)
        assert (gc_r - rgb.grad).abs().max().item() <= COMPOSITE_ATOL_REF
        assert ((gs_r - sig.grad).abs().max() / gs_r.abs().max()).item() <= 1e-5


def test_kernels_against_reference_kernel_fixture(golden_dir):
    """The product kernels on the inputs of tests/golden/raymarch_ref.npz against the outputs the reference's own CUDA kernels
    gave on them: the same bit-exact / COMPOSITE_ATOL_REF checks as the live comparisons above, without the reference build."""
    from trinerflet_b200 import _lib
    from trinerflet_b200 import raymarching as rm
    g = np.load(os.path.join(golden_dir, "raymarch_ref.npz"))
    dev = torch.device("cuda")
    ro, rd = torch.from_numpy(g["rays_o"]).to(dev), torch.from_numpy(g["rays_d"]).to(dev)
    bf, noises = torch.from_numpy(g["bitfield"]).to(dev), torch.from_numpy(g["noises"]).to(dev)
    N, M, max_steps, dt_gamma = ro.shape[0], int(g["M"]), int(g["max_steps"]), float(g["dt_gamma"])
    aabb = torch.tensor([-BOUND] * 3 + [BOUND] * 3, device=dev)
    nears, fars = rm.near_far_from_aabb(ro, rd, aabb, 0.2)
    assert np.array_equal(nears.cpu().numpy().view(np.uint32), g["nears"].view(np.uint32))
    assert np.array_equal(fars.cpu().numpy().view(np.uint32), g["fars"].view(np.uint32))
    lib = _lib.load()
    xyzs, dirs, deltas = (torch.zeros(M, k, device=dev) for k in (3, 3, 2))
    rays = torch.empty(N, 3, dtype=torch.int32, device=dev)
    counter = torch.zeros(2, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.tnl_march_rays_train_workspace(N), dtype=torch.uint8, device=dev)
    _lib.call("tnl_march_rays_train", _lib.ptr(ro), _lib.ptr(rd), _lib.ptr(bf), BOUND, dt_gamma, max_steps, N, CAS, H, M,
              _lib.ptr(nears), _lib.ptr(fars), _lib.ptr(xyzs), _lib.ptr(dirs), _lib.ptr(deltas), _lib.ptr(rays),
              _lib.ptr(counter), _lib.ptr(noises), _lib.ptr(ws), ws.numel(), _lib.stream())
    assert np.array_equal(counter.cpu().numpy(), g["counter"])
    # the reference kernel's slot order is a race: compare per ray, its rows sorted by ray id
    rr, mine = g["rays"][np.argsort(g["rays"][:, 0])], rays.cpu().numpy()
    assert np.array_equal(rr[:, 0], mine[:, 0]) and np.array_equal(rr[:, 2], mine[:, 2])
    xm, lm = xyzs.cpu().numpy(), deltas.cpu().numpy()
    for n in range(N):
        a, b, k = rr[n, 1], mine[n, 1], mine[n, 2]
        assert np.array_equal(g["xyzs"][a:a + k].view(np.uint32), xm[b:b + k].view(np.uint32))
        assert np.array_equal(g["deltas"][a:a + k].view(np.uint32), lm[b:b + k].view(np.uint32))
    w, _, img = rm.composite_rays_train(torch.from_numpy(g["sigmas"]).to(dev), torch.from_numpy(g["rgbs"]).to(dev),
                                        torch.from_numpy(g["deltas"]).to(dev), torch.from_numpy(g["rays"]).to(dev), 1e-4)
    assert np.abs(w.detach().cpu().numpy() - g["weights_sum"]).max() <= COMPOSITE_ATOL_REF
    assert np.abs(img.detach().cpu().numpy() - g["image"]).max() <= COMPOSITE_ATOL_REF
    packed = rm.packbits(torch.from_numpy(g["grid"]).to(dev), float(g["thresh"]))
    assert np.array_equal(packed.cpu().numpy(), g["packed"])
    assert np.array_equal(rm.morton3D(torch.from_numpy(g["coords"]).to(dev)).cpu().numpy(), g["morton"])


def _hash_field(x):
    """sigma [n], rgb [n,3] as a pure integer function of the BITS of the sample positions (numpy): the same sample gets the
    same values in both loops, whatever slot it occupies"""
    u = np.ascontiguousarray(x).view(np.uint32).astype(np.uint64)
    h = (u[:, 0] * np.uint64(73856093)) ^ (u[:, 1] * np.uint64(19349663)) ^ (u[:, 2] * np.uint64(83492791))
    h = (h ^ (h >> np.uint64(13))) * np.uint64(0x9E3779B1)
    sig = ((h >> np.uint64(8)) & np.uint64(0xFFFF)).astype(np.float32) / np.float32(65535) * np.float32(30)
    rgb = np.stack([((h >> np.uint64(s)) & np.uint64(0xFF)).astype(np.float32) / np.float32(255) for s in (24, 32, 40)], -1)
    return sig, np.ascontiguousarray(rgb)


def test_inference_march_composite_loop():
    """march_rays / composite_rays / device compaction driven as renderer.py:342-368 does, vs the C oracle.  The two loops run
    with SEPARATE state from start to end (no re-synchronisation): sample positions / deltas are compared bit for bit while
    the alive lists agree; a ray whose transmittance sits within float noise of T_thresh may terminate one chunk apart
    (__expf vs expf), which changes the other loop's chunk schedule but not any ray's own sample sequence."""
    from oracle import raymarch as orc
    from trinerflet_b200 import raymarching as rm
    _, o, d, bits, ro, rd, bf, aabb, nears, fars = _setup(3000)
    N = ro.shape[0]
    # ---- device loop
    ws = torch.zeros(N, device="cuda"); dp = torch.zeros(N, device="cuda"); im = torch.zeros(N, 3, device="cuda")
    alive = torch.arange(N, dtype=torch.int32, device="cuda"); rt = nears.clone()
    n_alive, step, trace_g = N, 0, []
    while step < 1024 and n_alive > 0:
        n_step = max(min(N // n_alive, 8), 1)
        x, dd, dl = rm.march_rays(n_alive, n_step, alive, rt, ro, rd, BOUND, bf, CAS, H, nears, fars, 128, False, 0, 1024)
        sig, rgb = _hash_field(x.cpu().numpy())
        trace_g.append((alive.cpu().numpy().copy(), x.cpu().numpy(), dl.cpu().numpy()))
        rm.composite_rays(n_alive, n_step, alive, rt, torch.from_numpy(sig).cuda(), torch.from_numpy(rgb).cuda(), dl, ws, dp, im, 1e-4)
        alive, cnt = rm.compact_rays_alive(alive, n_alive)
        n_alive = int(cnt.item())
        alive = alive[:n_alive]
        step += n_step
    # ---- oracle loop, its own state
    ws_o, dp_o, im_o = np.zeros(N, np.float32), np.zeros(N, np.float32), np.zeros((N, 3), np.float32)
    alive_o, rt_o = np.arange(N, dtype=np.int32), nears.cpu().numpy().copy()
    n_alive, step, it, lockstep, compared = N, 0, 0, True, 0
    diverged = set()
    while step < 1024 and n_alive > 0:
        n_step = max(min(N // n_alive, 8), 1)
        x_o, d_o, l_o = orc.march_rays(n_alive, n_step, alive_o, rt_o, o, d, BOUND, bits.numpy(), CAS, H,
                                       nears.cpu().numpy(), fars.cpu().numpy(), np.zeros(n_alive, np.float32), 128, 0.0, 1024)
        if lockstep and it < len(trace_g) and np.array_equal(trace_g[it][0], alive_o):
            assert np.array_equal(trace_g[it][1].view(np.uint32), x_o.view(np.uint32))
            assert np.array_equal(trace_g[it][2].view(np.uint32), l_o.view(np.uint32))
            compared += 1
        elif lockstep:
            lockstep = False
            diverged = set(trace_g[it][0].tolist()) ^ set(alive_o.tolist()) if it < len(trace_g) else set(alive_o.tolist())
        sig, rgb = _hash_field(x_o)
        orc.composite_rays(n_alive, n_step, alive_o, rt_o, sig, rgb, l_o, ws_o, dp_o, im_o, 1e-4)
        alive_o = alive_o[alive_o >= 0].copy()
        n_alive = alive_o.shape[0]
        step += n_step
        it += 1
    assert compared >= 20                                   # the bit-exact part covered a substantial prefix of the loop
    # per-ray results do not depend on the chunk schedule; rays that terminated a sample apart differ by < T_thresh-weighted terms
    bad = np.zeros(N, bool)
    for a, b in ((ws.cpu().numpy(), ws_o), (im.cpu().numpy(), im_o), (dp.cpu().numpy(), dp_o)):
        diff = np.abs(a - b).reshape(N, -1).max(-1)
        bad |= diff > 5e-5
        assert diff.max() <= 1e-3                           # extra samples carry weight < T_thresh = 1e-4 (depth: x t <= 6)
    assert int(bad.sum()) <= max(1, N // 1000)              # <= 0.1 % of the rays 


def test_sh_encoder():
    from oracle import field as of
    from trinerflet_b200.shencoder import SHEncoder
    d = torch.randn(5000, 3)
    d = d / d.norm(dim=-1, keepdim=True)
    out = SHEncoder(3, 4)(d.cuda())
    assert (out.cpu() - of.sh16(d)).abs().max().item() <= 1e-6
    from oracle import build_ref
    ref = build_ref.load_ref("shencoder")
    if ref is not None:
        o_r = torch.empty(5000, 16, device="cuda")
        ref.sh_encode_forward(d.cuda(), o_r, 5000, 3, 4, None)
        assert (o_r - out).abs().max().item() <= 1e-6
