"""GPU: every wavelet of the reference's pad table (bior6.8, haar, bior2.2, bior2.6, bior4.4) through the device build --
level kernels against the oracle, work-list equal to dense, a whole training step of the `small` geometry against
the oracle's training step (tests/wavelet_oracle.py), graph replay equal to eager, and an eval render with the device-driven loop.  bior6.8's own
versions of the step, replay and render tests live in test_gpu_baseline_sizes.py / test_gpu_train.py /
test_gpu_x_infer_loop.py; tolerances as stated there."""
import pytest
import torch

from tests import wavelet_oracle
from tests.util import cl_coefs, cl_planes, rel_l2, rel_linf

pytestmark = pytest.mark.gpu
WAVES = ["bior6.8", "haar", "bior2.2", "bior2.6", "bior4.4"]


def _rand_coefs(C, n0, levels, seed):
    g = torch.Generator().manual_seed(seed)
    pf = 0.1 * torch.randn(3, C, n0, n0, generator=g)
    coefs = [0.05 * torch.randn(3, C, 3, n0 * 2 ** l, n0 * 2 ** l, generator=g) for l in range(levels)]
    return pf, coefs


def _net(cfg, wave, radius=0.75, **kw):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    c = dict(scene.CONFIGS[cfg], **kw)
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"], triplane_resolution=c["R"],
                      triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"], hidden_dim_color=c["hidden"], wavelet_type=wave).cuda()
    assert net.encoder.wavelet_type == wave
    scene.init_model_(net, seed=0)
    scene.install_ball_occupancy(net, radius)
    return net


@pytest.mark.parametrize("wave", WAVES)
def test_level_kernels_match_oracle(wave):
    """C=16, 64 -> 512 (3 levels), all three planes: planes rel-L_inf <= 1e-5, adjoint rel-L2 <= 1e-4"""
    from oracle import wavelet as ow
    from trinerflet_b200.triplane_encoder import build_planes
    C, n0, levels = 16, 64, 3
    pf, coefs = _rand_coefs(C, n0, levels, seed=7)
    R = n0 * 2 ** levels
    gout = torch.randn(3, C, R, R, generator=torch.Generator().manual_seed(1))
    pf_o = pf.clone().requires_grad_(True)
    coefs_o = [c.clone().requires_grad_(True) for c in coefs]
    ref = ow.build_planes(pf_o, coefs_o, wave)
    ref.backward(gout)
    pf_g = cl_planes(pf.cuda()).requires_grad_(True)
    coefs_g = [cl_coefs(c.cuda()).requires_grad_(True) for c in coefs]
    out = build_planes(pf_g, coefs_g, wave=wave)
    assert out.shape == ref.shape and rel_linf(out, ref) <= 1e-5
    out.backward(gout.cuda())
    assert rel_l2(pf_g.grad, pf_o.grad) <= 1e-4
    for a, b in zip(coefs_g, coefs_o):
        assert rel_l2(a.grad, b.grad) <= 1e-4


@pytest.mark.parametrize("wave", WAVES)
def test_worklist_equals_dense(wave):
    """work-list forward bit-identical to dense inside the marked tiles; the adjoint of a tile-supported gradient bit-identical"""
    from trinerflet_b200.idwt_plan import IdwtPlan
    from trinerflet_b200.triplane_encoder import build_planes
    C, n0, levels = 32, 64, 3
    R, T = n0 * 2 ** levels, n0 * 2 ** levels // 32
    pf, coefs = _rand_coefs(C, n0, levels, seed=8)
    g = torch.Generator().manual_seed(2)
    flags = torch.rand(3, T, T, generator=g) < 0.15
    flags[:, 4:8, 5:9] = True
    mask = flags.repeat_interleave(32, 1).repeat_interleave(32, 2)[:, None].cuda()
    gout = (torch.randn(3, C, R, R, generator=g).cuda() * mask).contiguous()
    plan = IdwtPlan(R, n0, levels, C, "cuda").update(flags.cuda())
    res = []
    for p in (None, plan):
        pf_g = cl_planes(pf.cuda()).requires_grad_(True)
        coefs_g = [cl_coefs(c.cuda()).requires_grad_(True) for c in coefs]
        out = build_planes(pf_g, coefs_g, p, wave=wave)
        out.backward(gout)
        res.append((torch.where(mask, out.detach(), 0.0), pf_g.grad, [c.grad for c in coefs_g]))
    (o_d, gp_d, gc_d), (o_s, gp_s, gc_s) = res
    assert torch.equal(o_s, o_d) and torch.equal(gp_s, gp_d)
    for a, b in zip(gc_s, gc_d):
        assert torch.equal(a, b)


@pytest.mark.parametrize("wave", WAVES[1:])
def test_whole_training_step_small_config_matches_oracle(wave):
    """`small` geometry (C=16, 1024^2 planes, 4 levels), 2 048 rays, the steady-state step bench.py times (fp16 autocast +
    GradScaler, work-list IDWT + split backward) against the oracle's training step with the same wavelet: loss within 2e-3,
    every parameter gradient within rel-L2 1e-2 (bior6.8: test_gpu_baseline_sizes.py)"""
    from trinerflet_b200 import scene, trainer
    net = _net("small", wave, C=16, R=1024, S=16, hidden=64)
    net.train()
    sc = scene.make_scene()
    N = 2048
    ro, rd, tgt = scene.sample_batch(sc, N, torch.Generator().manual_seed(0))
    opt = trainer.default_opt(fp16=True)
    ts = trainer.TrainStep(net, opt, None)
    ts.sparse_idwt = True
    torch.manual_seed(5)
    loss = ts.forward_backward(ro.cuda(), rd.cuda(), tgt.cuda(), update_grid=False)
    M = int(net.step_counter[0, 0])
    assert M > 50_000 and ts._plan is not None
    scale = float(ts.scaler.get_scale())
    torch.manual_seed(5)
    noises = torch.rand(N, device="cuda").cpu().numpy()
    pf = net.encoder.planes_features.detach().cpu().contiguous().requires_grad_(True)
    coefs = [p.detach().cpu().contiguous().requires_grad_(True) for p in net.encoder.planes_features_wavelet_coefs]
    W = [w.detach().cpu().clone().requires_grad_(True) for w in net._weights()]
    loss_o, M_o = wavelet_oracle.train_step(pf, coefs, W, ro, rd, tgt, net.density_bitfield.cpu().numpy(), noises, wave,
                                            lam=opt.wavelet_regularization, loss_scale=scale, fp16=True)
    assert M_o == M
    assert abs(float(loss) - loss_o) <= 2e-3 * abs(loss_o)
    ours = [net.encoder.planes_features.grad] + [p.grad for p in net.encoder.planes_features_wavelet_coefs] + [w.grad for w in net._weights()]
    theirs = [pf.grad] + [c.grad for c in coefs] + [w.grad for w in W]
    for a, b in zip(ours, theirs):
        assert rel_l2(a, b) <= 1e-2, (tuple(a.shape), rel_l2(a, b))


def test_cuda_graph_replay_equals_eager_step_bior26():
    """TrainStep.capture()/replay() against the eager step with a non-default wavelet: same loss, same gradients"""
    from trinerflet_b200 import scene, trainer
    sc = scene.make_scene()
    g = torch.Generator().manual_seed(11)
    b = [tuple(t.cuda() for t in scene.sample_batch(sc, 4096, g)) for _ in range(3)]
    out = []
    for graph in (False, True):
        net = _net("tiny", "bior2.6")
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
    assert abs(out[0][0] - out[1][0]) <= 1e-5 * abs(out[0][0])
    for a, c in zip(out[0][1], out[1][1]):
        assert rel_l2(c, a) <= 1e-5


@pytest.mark.parametrize("wave", WAVES)
def test_eval_render_with_device_loop(wave):
    """inference render (fp16 autocast, device-driven loop) on the wavelet's planes: the device loop equals the host loop,
    and the planes it samples are the oracle's reconstruction with that wavelet"""
    from oracle import wavelet as ow
    from trinerflet_b200 import scene
    net = _net("tiny", wave)
    net.eval()
    planes = net.encoder.get_planes()
    ref = ow.build_planes(net.encoder.planes_features.detach().cpu(), [p.detach().cpu() for p in net.encoder.planes_features_wavelet_coefs],
                          wave)
    assert rel_linf(planes, ref) <= 1e-5
    sc = scene.make_scene()
    ro, rd = scene.full_frame(sc, 3)
    pick = torch.arange(0, ro.shape[0], 97)[:5000]
    ro, rd = ro[pick].cuda(), rd[pick].cuda()
    outs = []
    for chunk in (0, 8):
        net.infer_chunk = chunk
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            outs.append(net.render(ro.unsqueeze(0), rd.unsqueeze(0), staged=True, bg_color=1, perturb=False, max_steps=512))
    assert net.last_infer_loop.reads < net.last_infer_loop.iterations_done
    a, b = outs
    assert float(a["weights_sum"].sum()) > 10.0
    for k in ("image", "weights_sum"):
        assert (a[k].float() - b[k].float()).abs().max().item() <= 1e-6, k
