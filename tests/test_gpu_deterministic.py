"""GPU: torch.use_deterministic_algorithms(True) -- bit-reproducible single-GPU training steps.

The flag is global: every test here that sets it does so through the `deterministic_mode` fixture, which restores the previous
state (and warn_only)."""
import ctypes

import numpy as np
import pytest
import torch

from tests.test_deterministic_emu import _lattice_case
from tests.util import rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture
def deterministic_mode():
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


def _model(cfg, seed=0):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS[cfg]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"],
                      triplane_resolution=c["R"], triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"],
                      hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=seed)
    scene.install_ball_occupancy(net, 0.75)
    return net


def _bits(t):
    return t.detach().contiguous().view(torch.int32) if t.dtype == torch.float32 else t.detach().contiguous()


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _scatter(G, half, xyz, M, R, C, nv, perm):
    from trinerflet_b200._lib import ptr
    from trinerflet_b200.triplane_encoder import cl_empty_planes, scatter_planes
    gp = cl_empty_planes(C, R, device="cuda", zero=True)
    scatter_planes(G, half, xyz, M, R, C, 1.0, 0, ptr(nv), ptr(perm), gp)
    return gp


@pytest.mark.parametrize("C,half", [(16, True), (32, False), (48, True)])
def test_det_scatter_order_free_and_within_bound(C, half, deterministic_mode):
    from oracle import field as of
    M = 200000
    R, xyz, G, Gin = _lattice_case(C, M, C, half)
    xyz_d = torch.from_numpy(xyz).cuda()
    Gd = torch.from_numpy(Gin).cuda()
    nv = torch.tensor([M - 40], dtype=torch.int32, device="cuda")
    a = _scatter(Gd, half, xyz_d, M, R, C, nv, None)
    perm = torch.randperm(M, device="cuda").int()
    assert _same_bits(_scatter(Gd, half, xyz_d, M, R, C, nv, perm), a)
    q = torch.cat([torch.randperm(M - 40), torch.arange(M - 40, M)]).cuda()
    assert _same_bits(_scatter(Gd[q].contiguous(), half, xyz_d[q].contiguous(), M, R, C, nv, None), a)
    pl = torch.zeros(3, C, R, R, dtype=torch.float64, requires_grad=True)   # (on the CPU: grid_sample's CUDA backward adds atomically)
    (of.sample_planes(pl, torch.from_numpy(xyz), 1.0) * G.double()).sum().backward()
    ref = pl.grad.permute(0, 2, 3, 1).cuda()
    a = a.permute(0, 2, 3, 1)
    e = int(np.frexp(float(G.abs().max()))[1])
    unit = 2.0 ** (e + int(np.ceil(np.log2(M))) - 62)
    assert ((a.double() - ref).abs() <= M * unit / 2 + 2.0 ** -24 * ref.abs()).all()
    Gbad = Gd.clone()
    Gbad[11, 2] = float("inf")
    assert not torch.isfinite(_scatter(Gbad, half, xyz_d, M, R, C, nv, None)).all()


@pytest.mark.parametrize("C,hidden,half,dirs_grad", [(16, 64, True, False), (32, 64, True, True), (48, 128, True, False),
                                                     (48, 128, True, True), (16, 64, False, True), (32, 64, False, False)])
def test_mlp_backward_det_bit_identical(C, hidden, half, dirs_grad):
    from oracle import field as of
    from trinerflet_b200 import _lib
    from trinerflet_b200._lib import MlpDims, call, ptr, stream
    from trinerflet_b200.network import pack_mlp_weights
    M = 300000
    g = torch.Generator().manual_seed(C + hidden)
    W = [w.cuda() for w in of.init_mlp_weights(C, hidden, hidden, gen=g)]
    feat = (0.5 * torch.randn(M, 3 * C, generator=g)).cuda().to(torch.float16 if half else torch.float32)
    d = torch.nn.functional.normalize(torch.randn(M, 3, generator=g), dim=-1).cuda()
    gs, grgb = (torch.randn(M, generator=g) * 64).cuda(), (torch.randn(M, 3, generator=g) * 64).cuda()
    nv = torch.tensor([M - 1000], dtype=torch.int32, device="cuda")
    dims = MlpDims(3 * C, hidden, hidden)
    packed = pack_mlp_weights(dims, W)
    ws = torch.empty(_lib.load().tnl_mlp_backward_det_workspace(ctypes.byref(dims), int(half), M), dtype=torch.uint8, device="cuda")
    runs = []
    for name in ("tnl_mlp_backward_det", "tnl_mlp_backward_det", "default"):
        gW = [torch.zeros_like(w) for w in W]
        g_feat = torch.empty_like(feat)
        g_dirs = torch.empty(M, 3, device="cuda") if dirs_grad else None
        args = (ctypes.byref(dims), ptr(packed), ptr(feat), int(half), ptr(d), M, ptr(nv), ptr(gs), ptr(grgb), ptr(g_feat), *[ptr(x) for x in gW])
        if name == "default":
            if dirs_grad:
                call("tnl_mlp_backward_dirs", *args, ptr(g_dirs), stream())
            else:
                call("tnl_mlp_backward", *args, stream())
        else:
            call(name, *args, ptr(g_dirs), ptr(ws), ws.numel(), stream())
        runs.append((gW, g_feat, g_dirs))
    for a, b in zip(runs[0][0], runs[1][0]):
        assert _same_bits(a, b)
    for a, b in zip(runs[0][0], runs[2][0]):
        assert rel_l2(a, b) <= 1e-5
    assert _same_bits(runs[0][1][:M - 1000], runs[2][1][:M - 1000])
    if dirs_grad:
        assert _same_bits(runs[0][2], runs[2][2])


def _run_steps(cfg, n_steps, seed=0, graph=False):
    from trinerflet_b200 import scene, trainer
    net = _model(cfg, seed)
    opt = trainer.default_opt(update_extra_interval=5)
    ts = trainer.TrainStep(net, opt, trainer.make_optimizer(net, 1e-2, fused=True), world_size=1)
    sc = scene.make_scene()
    g = torch.Generator().manual_seed(seed + 1)
    losses = []
    for i in range(n_steps):
        ro, rd, tgt = (t.cuda() for t in scene.sample_batch(sc, scene.CONFIGS[cfg]["rays"], g))
        torch.manual_seed(100 + i)
        losses.append(ts.step(ro, rd, tgt, update_grid=(i % 5 == 4)))
    state = [p.detach().clone() for p in net.parameters()]
    moments = [v.clone() for st in ts.optimizer.state.values() for v in st.values() if torch.is_tensor(v)]
    return torch.stack(losses), state, moments, net.density_grid.clone(), net.density_bitfield.clone()


def test_training_steps_bit_reproducible_small(deterministic_mode):
    a = _run_steps("small", 20)
    b = _run_steps("small", 20)
    assert _same_bits(a[0], b[0])
    for x, y in zip(a[1] + a[2], b[1] + b[2]):
        assert _same_bits(x, y)
    assert len(a[2]) > 0
    assert _same_bits(a[3], b[3]) and torch.equal(a[4], b[4])


def _one_step_grads(cfg, sparse=True, batch_seed=3):
    from trinerflet_b200 import scene, trainer
    sc = scene.make_scene()
    ro, rd, tgt = (t.cuda() for t in scene.sample_batch(sc, scene.CONFIGS[cfg]["rays"], torch.Generator().manual_seed(batch_seed)))
    net = _model(cfg)
    ts = trainer.TrainStep(net, trainer.default_opt(), None, world_size=1)
    ts.sparse_idwt = sparse
    torch.manual_seed(0)
    loss = ts.forward_backward(ro, rd, tgt, update_grid=False)
    return loss, [p.grad.detach().clone() for p in net.parameters()], ts


def test_dense_and_worklist_steps_bit_identical(deterministic_mode):
    la, ga, _ = _one_step_grads("cpu", sparse=False)
    lb, gb, ts = _one_step_grads("cpu", sparse=True)
    assert 0.0 < ts._plan.stats["tile_fraction"] < 0.9
    assert _same_bits(la, lb)
    for a, b in zip(ga, gb):
        assert _same_bits(a, b)


def test_large_step_twice_same_bits(deterministic_mode):
    la, ga, _ = _one_step_grads("large")
    lb, gb, _ = _one_step_grads("large")
    assert _same_bits(la, lb)
    for a, b in zip(ga, gb):
        assert _same_bits(a, b)


def test_deterministic_gradients_agree_with_default_mode_small():
    """Only the order of the sums differs from the default mode: same tolerance as the fused-scatter path (rel-L2 <= 1e-5)."""
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        l0, g0, _ = _one_step_grads("small")
        torch.use_deterministic_algorithms(True)
        l1, g1, _ = _one_step_grads("small")
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    assert abs(float(l0) - float(l1)) <= 1e-5 * abs(float(l0))
    for a, b in zip(g0, g1):
        assert rel_l2(b, a) <= 1e-5


def test_graph_replay_equals_eager_bits(deterministic_mode):
    from trinerflet_b200 import scene, trainer
    sc = scene.make_scene()
    g = torch.Generator().manual_seed(11)
    b = [tuple(t.cuda() for t in scene.sample_batch(sc, 4096, g)) for _ in range(3)]
    out = []
    for graph in (False, True):
        net = _model("tiny")
        ts = trainer.TrainStep(net, trainer.default_opt(), None, world_size=1)
        torch.manual_seed(0)
        ts.forward_backward(*b[0], update_grid=False)
        net.mean_count = int(net.step_counter[0, 0].item())
        net.local_step = 0
        net.zero_grad(set_to_none=True)
        if graph:
            ts.capture(*b[1], warmup=1)
            torch.manual_seed(5)
            loss = ts.replay(*b[2])
        else:
            for _ in range(2):
                net.zero_grad(set_to_none=True)
                ts.forward_backward(*b[1], update_grid=False)
            net.zero_grad(set_to_none=True)
            torch.manual_seed(5)
            loss = ts.forward_backward(*b[2], update_grid=False)
        out.append((loss.clone(), [p.grad.detach().clone() for p in net.parameters()]))
    assert _same_bits(out[0][0], out[1][0])
    for a, c in zip(out[0][1], out[1][1]):
        assert _same_bits(a, c)


def test_grid_refresh_duplicates_follow_index_put(deterministic_mode):
    net = _model("tiny")
    H = net.grid_size
    idx = torch.randint(0, H ** 3, (50000,), device="cuda").int()
    idx[1::2] = idx[0::2]                                   # every cell twice: the refresh's partial sweep has duplicates
    tmp = torch.full_like(net.density_grid, -1.0)
    torch.manual_seed(3)
    net._sweep_cells(0, idx, tmp)
    torch.manual_seed(3)
    noise = torch.rand(idx.shape[0], 3, device="cuda")
    from trinerflet_b200._lib import call, ptr, stream
    xyz = torch.empty(idx.shape[0], 3, device="cuda")
    call("tnl_grid_cell_positions", ptr(idx), idx.shape[0], H, float(min(1, net.bound)), ptr(noise), ptr(xyz), stream())
    sig = net.density(xyz)["sigma"].reshape(-1).float()
    want = torch.full_like(net.density_grid, -1.0)
    want[0].index_put_((idx.long(),), sig * float(net.density_scale))
    assert _same_bits(tmp, want)


def test_field_dispatch_follows_the_flag(monkeypatch):
    from trinerflet_b200 import network
    net = _model("tiny")
    net.spatial_sort_min_points = 1
    seen = []
    orig = network._Field.apply
    monkeypatch.setattr(network._Field, "apply", lambda *a: (seen.append(1), orig(*a))[1])
    x = (torch.rand(4096, 3, device="cuda") * 2 - 1)
    d = torch.nn.functional.normalize(torch.randn(4096, 3, device="cuda"), dim=-1)
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        with torch.autocast("cuda", dtype=torch.float16):
            net(x, d)
        assert seen == [1]
        torch.use_deterministic_algorithms(True)
        with torch.autocast("cuda", dtype=torch.float16):
            s, c = net(x, d)
        assert seen == [1] and s.shape == (4096,)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
