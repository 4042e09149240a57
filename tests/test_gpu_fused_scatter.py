"""GPU: the fused training path (one tnl_mlp_backward_scatter: MLP backward + plane-gradient scatter) against the unfused one
(tnl_mlp_backward writing g_feat, then tnl_sample_planes_backward) on the same seeded inputs.  The forward is the same calls,
so its values are bit-identical; the gradients differ only by the order of fp32 additions (atomics, tile order of the weight
gradients)."""
import pytest
import torch

from tests.util import rel_l2

pytestmark = pytest.mark.gpu


class _CallLog:
    """records the names of the ABI calls network.py makes"""

    def __init__(self, monkeypatch):
        from trinerflet_b200 import network
        self.names = []
        inner = network.call

        def call(name, *args):
            self.names.append(name)
            return inner(name, *args)
        monkeypatch.setattr(network, "call", call)


def _inputs(C, M, n_valid, seed=0, R=256, bound=1.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    planes = (0.5 * torch.randn(3, R, R, C, device="cuda", generator=g)).permute(0, 3, 1, 2).detach().requires_grad_()
    coords = (torch.rand(M, 3, device="cuda", generator=g) * 2 - 1) * bound
    dirs = torch.nn.functional.normalize(torch.randn(M, 3, device="cuda", generator=g), dim=-1)
    shapes = [(64, 3 * C), (16, 64), (64, 31), (64, 64), (3, 64)]
    W = [(torch.randn(s, device="cuda", generator=g) / s[1] ** 0.5).requires_grad_() for s in shapes]
    gs = torch.randn(M, device="cuda", generator=g)
    grgb = torch.randn(M, 3, device="cuda", generator=g)
    gs[n_valid - 5000:] = 0.0            # samples past ray termination: all-zero gradient rows
    grgb[n_valid - 5000:] = 0.0
    nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
    return planes, coords, dirs, W, gs, grgb, nv, bound


@pytest.mark.parametrize("C", [16, 32])
def test_field_function_matches_sample_plus_mlp(C, monkeypatch):
    """_Field against _SamplePlanes + _FieldMLP: cell-sorted points, an n_valid tail that is not a multiple of the 128-point
    tile, padding rows whose gradient must not reach the planes, and zero-gradient rows."""
    from trinerflet_b200.network import _Field, _FieldMLP
    from trinerflet_b200.triplane_encoder import cell_sort, sample_planes
    log = _CallLog(monkeypatch)
    M = 300_001
    n_valid = M - 1_000
    out = []
    for fused in (False, True):
        planes, coords, dirs, W, gs, grgb, nv, bound = _inputs(C, M, n_valid)
        perm = cell_sort(coords, bound, nv, 64)
        with torch.autocast("cuda", dtype=torch.float16):
            if fused:
                sigma, rgb = _Field.apply(planes, coords, dirs, bound, nv, perm, None, *W)
            else:
                feat = sample_planes(planes, coords, bound, n_valid=nv, perm=perm, half_out=True)
                sigma, rgb = _FieldMLP.apply(feat, dirs, nv, *W)
        ((sigma * gs).sum() + (rgb * grgb).sum()).backward()
        torch.cuda.synchronize()
        out.append((sigma, rgb, planes.grad, [w.grad for w in W]))
    assert log.names.count("tnl_mlp_backward_scatter") == 1
    (s0, c0, gp0, gw0), (s1, c1, gp1, gw1) = out
    assert torch.equal(s0, s1) and torch.equal(c0, c1)
    assert gp0.abs().sum() > 0
    assert rel_l2(gp1, gp0) <= 1e-5
    for a, b in zip(gw1, gw0):
        assert rel_l2(a, b) <= 1e-5


def _model(cfg):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS[cfg]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"],
                      triplane_resolution=c["R"], triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"],
                      hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=0)
    scene.install_ball_occupancy(net, 0.75)
    net.spatial_sort_min_points = 0      # cell-sort (and so take the fused path) at this test's batch size too
    return net


def _unfused(net):
    # a per-plane scatter hook sends the step through _SamplePlanes; without an external gradient buffer it is never called
    net.encoder.scatter_plane_hook = lambda plane: None


@pytest.mark.parametrize("cfg", ["small", "base_light"])
@pytest.mark.parametrize("sparse_idwt", [True, False])
def test_training_step_fused_equals_unfused(cfg, sparse_idwt, monkeypatch):
    """Steady-state training steps as bench.py runs them (fixed sample buffer with an n_valid tail, planes prefetched on the side
    stream, work-list or dense plane reconstruction): same loss bits, gradients equal to fp32 reordering."""
    from trinerflet_b200 import scene, trainer
    log = _CallLog(monkeypatch)
    sc = scene.make_scene()
    ro, rd, tgt = (t.cuda() for t in scene.sample_batch(sc, 8192, torch.Generator().manual_seed(3)))
    out = []
    for fused in (False, True):
        net = _model(cfg)
        if not fused:
            _unfused(net)
        ts = trainer.TrainStep(net, trainer.default_opt(), None, world_size=1)
        ts.sparse_idwt = sparse_idwt
        torch.manual_seed(0)
        ts.forward_backward(ro, rd, tgt, update_grid=False)
        net.mean_count = int(net.step_counter[0, 0].item())
        net.local_step = 0
        net.zero_grad(set_to_none=True)
        n0 = log.names.count("tnl_mlp_backward_scatter")
        torch.manual_seed(1)
        loss = ts.forward_backward(ro, rd, tgt, update_grid=False)
        assert log.names.count("tnl_mlp_backward_scatter") - n0 == int(fused)
        out.append((loss.clone(), {n: p.grad.detach().clone() for n, p in net.named_parameters()}))
        del net, ts
    assert torch.equal(out[0][0], out[1][0])
    for n, g in out[0][1].items():
        assert rel_l2(out[1][1][n], g) <= 1e-5, n


def test_fused_step_graph_replay_equals_eager(monkeypatch):
    """TrainStep.capture()/replay() of the fused step against the same step launched eagerly."""
    from trinerflet_b200 import scene, trainer
    log = _CallLog(monkeypatch)
    sc = scene.make_scene()
    g = torch.Generator().manual_seed(11)
    b = [tuple(t.cuda() for t in scene.sample_batch(sc, 8192, g)) for _ in range(3)]
    out = []
    for graph in (False, True):
        net = _model("small")
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
        out.append((float(loss), [p.grad.detach().clone() for p in net.parameters()]))
    assert "tnl_mlp_backward_scatter" in log.names and "tnl_mlp_backward" not in log.names
    assert abs(out[0][0] - out[1][0]) <= 1e-5 * abs(out[0][0])
    for a, c in zip(out[0][1], out[1][1]):
        assert rel_l2(c, a) <= 1e-5
