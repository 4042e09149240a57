"""CPU: the IDWT level kernels for every wavelet of the reference's pad table (tnl_idwt_level_*_wavelet) on the host build of
the product kernels (tests/kemu.py) against the oracle -- dense forward and backward, exact adjointness, work-list variants
bit-identical to dense -- plus TriPlaneVolume's wavelet handling and one emulated training step with a non-default wavelet
(dense and work-list) against the oracle pipeline (tests/wavelet_oracle.py)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import wavelet as ow
from tests import emu_backend, kemu, wavelet_oracle
from tests.util import rel_l2

WAVES = ["bior6.8", "haar", "bior2.2", "bior2.6", "bior4.4"]
IDS = {"bior6.8": 0, "haar": 1, "bior2.2": 2, "bior2.6": 3, "bior4.4": 4}


def _cl(t):
    return np.ascontiguousarray(t.detach().permute(0, 2, 3, 1).numpy())


def _cl_coefs(t):
    return np.ascontiguousarray(t.detach().permute(0, 2, 3, 4, 1).numpy())


def _fwd(wave, pf, coefs, plan=None):
    x = _cl(pf)
    C, n = x.shape[3], x.shape[1]
    abs_sums = np.zeros(len(coefs), np.float32)
    for l, yh in enumerate(coefs):
        out = np.full((3, 2 * n, 2 * n, C), np.nan, np.float32)
        if plan is None:
            kemu.call("tnl_idwt_level_forward_wavelet", x, _cl_coefs(yh), out, n, C, abs_sums[l:l + 1], IDS[wave], None)
        else:
            s = plan.fwd[l]
            kemu.call("tnl_idwt_level_forward_sparse_wavelet", x, _cl_coefs(yh), out, n, C, abs_sums[l:l + 1], s["active"].numpy(),
                      s["clean"].numpy(), s["counts"].numpy(), s["cap_active"], s["cap_clean"], 3, IDS[wave], None)
        x, n = out, 2 * n
    return x, abs_sums


def _bwd(wave, gout, coefs, n0, reg, plan=None):
    g, C = gout, gout.shape[3]
    g_yh = [None] * len(coefs)
    reg_grad = np.array([reg], np.float32)
    for l in reversed(range(len(coefs))):
        n = n0 * 2 ** l
        gx = np.full((3, n, n, C), np.nan, np.float32)
        gy = np.full((3, 3, n, n, C), np.nan, np.float32)
        yh = _cl_coefs(coefs[l])
        if plan is None:
            kemu.call("tnl_idwt_level_backward_wavelet", g, gx, gy, n, C, yh, reg_grad, 0.25, 0, 3, IDS[wave], None)
        else:
            s = plan.bwd[l]
            kemu.call("tnl_idwt_level_backward_sparse_wavelet", g, gx, gy, n, C, yh, reg_grad, 0.25, s["active"].numpy(),
                      s["clean"].numpy(), s["counts"].numpy(), s["cap_active"], s["cap_clean"], 3, None, IDS[wave], None)
        g_yh[l] = gy
        g = gx
    return g, g_yh


@pytest.mark.parametrize("wave", WAVES)
@pytest.mark.parametrize("C,n0,levels", [(8, 8, 2), (24, 16, 1)])
def test_dense_level_kernels_match_oracle_and_are_exact_adjoints(wave, C, n0, levels):
    g = torch.Generator().manual_seed(C + n0 + IDS[wave])
    pf = torch.randn(3, C, n0, n0, generator=g, requires_grad=True)
    coefs = [torch.randn(3, C, 3, n0 * 2 ** l, n0 * 2 ** l, generator=g, requires_grad=True) for l in range(levels)]
    ref = ow.build_planes(pf, coefs, wave)
    planes, abs_sums = _fwd(wave, pf, coefs)
    assert np.abs(planes - _cl(ref)).max() <= 1e-5 * ref.abs().max().item()
    for l, c in enumerate(coefs):
        assert abs(abs_sums[l] - c.detach().abs().sum().item()) <= 1e-4 * abs_sums[l]
    gout = torch.randn(ref.shape, generator=g)
    (ref * gout).sum().backward()
    gx, gyh = _bwd(wave, _cl(gout), coefs, n0, 0.0)
    assert np.abs(gx - _cl(pf.grad)).max() <= 1e-4 * pf.grad.abs().max().item()
    for l, c in enumerate(coefs):
        assert np.abs(gyh[l] - _cl_coefs(c.grad)).max() <= 1e-4 * c.grad.abs().max().item()
    # <g, fwd(x, yh)> == <bwd_x(g), x> + sum_l <bwd_yh_l(g), yh_l>, the kernels' outputs on both sides
    lhs = float((_cl(gout).astype(np.float64) * planes).sum())
    rhs = float((gx.astype(np.float64) * _cl(pf)).sum()) + sum(float((a.astype(np.float64) * _cl_coefs(c)).sum()) for a, c in zip(gyh, coefs))
    assert abs(lhs - rhs) <= 1e-5 * (np.abs(_cl(gout)).astype(np.float64) * np.abs(planes)).sum()
    # fused regulariser gradient
    _, gyh_r = _bwd(wave, _cl(gout), coefs, n0, 0.5)
    for a, b, c in zip(gyh_r, gyh, coefs):
        assert np.abs(a - (b + _cl_coefs(0.125 * torch.sign(c.detach())))).max() <= 1e-6 * np.abs(a).max()


@pytest.mark.parametrize("wave", WAVES[1:])
def test_worklist_level_kernels_equal_dense(wave):
    from trinerflet_b200.idwt_plan import IdwtPlan
    C, n0, levels = 16, 16, 2
    R = n0 * 2 ** levels
    T = R // 32
    g = torch.Generator().manual_seed(11 + IDS[wave])
    flags = torch.rand(3, T, T, generator=g) < 0.1
    flags[:, 0:2, 1:3] = True
    plan = IdwtPlan(R, n0, levels, C, "cpu").update(flags)
    pf = torch.randn(3, C, n0, n0, generator=g)
    coefs = [0.1 * torch.randn(3, C, 3, n0 * 2 ** l, n0 * 2 ** l, generator=g) for l in range(levels)]
    coefs[-1][:, :, :, ::3, ::4] = 0.0
    dense, abs_d = _fwd(wave, pf, coefs)
    sparse, abs_s = _fwd(wave, pf, coefs, plan)
    mask = np.repeat(np.repeat(flags.numpy(), 32, axis=1), 32, axis=2)[..., None]
    assert np.array_equal(np.where(mask, sparse, 0).view(np.uint32), np.where(mask, dense, 0).view(np.uint32))
    assert np.abs(abs_s - abs_d).max() <= 1e-5 * abs_d.max()
    gout = (np.random.default_rng(1).standard_normal(dense.shape).astype(np.float32) * mask).astype(np.float32)
    gx_d, gy_d = _bwd(wave, gout, coefs, n0, 0.7)
    gx_s, gy_s = _bwd(wave, gout, coefs, n0, 0.7, plan)
    assert np.array_equal(gx_s.view(np.uint32), gx_d.view(np.uint32))
    for a, b in zip(gy_s, gy_d):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_bior68_id_is_the_existing_entry_points_and_unknown_ids_are_rejected():
    g = torch.Generator().manual_seed(2)
    C, n = 16, 16
    x, yh = _cl(torch.randn(3, C, n, n, generator=g)), _cl_coefs(torch.randn(3, C, 3, n, n, generator=g))
    a, b = np.zeros((3, 2 * n, 2 * n, C), np.float32), np.zeros((3, 2 * n, 2 * n, C), np.float32)
    kemu.call("tnl_idwt_level_forward", x, yh, a, n, C, None, None)
    kemu.call("tnl_idwt_level_forward_wavelet", x, yh, b, n, C, None, 0, None)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    lib, p = kemu.lib(), kemu.p
    assert lib.tnl_idwt_level_forward_wavelet(p(x), p(yh), p(b), n, C, None, 5, None) == -1
    assert b"unknown wavelet" in lib.tnl_last_error()
    gx, gy = np.zeros((3, n, n, C), np.float32), np.zeros((3, 3, n, n, C), np.float32)
    assert lib.tnl_idwt_level_backward_wavelet(p(a), p(gx), p(gy), n, C, None, None, 0.0, 0, 3, 7, None) == -1
    cnt = np.zeros(2, np.int32)
    items = np.zeros((1, 4), np.int32)
    assert lib.tnl_idwt_level_forward_sparse_wavelet(p(x), p(yh), p(a), n, C, None, p(items), p(items), p(cnt), 1, 1, 3, 99, None) == -1
    assert lib.tnl_idwt_level_backward_sparse_wavelet(p(a), p(gx), p(gy), n, C, None, None, 0.0, p(items), p(items), p(cnt), 1, 1, 3,
                                                      None, 0xFFFFFFFF, None) == -1


def test_triplane_volume_accepts_the_pad_table_and_checkpoints_do_not_depend_on_the_wavelet():
    from trinerflet_b200.triplane_encoder import TriPlaneVolume
    shapes = None
    for wave, pad in [("bior6.8", 4), ("bior2.6", 3), ("bior4.4", 2), ("bior2.2", 1), ("haar", 0)]:
        enc = TriPlaneVolume(number_of_features=8, plane_resolution=64, inner_multi_res_scale=4, wavelet_type=wave)
        assert enc.wavelet_type == wave and enc.planes_features_wavelet_pad == pad
        sd = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
        assert shapes is None or sd == shapes
        shapes = sd
    for wave in ("db4", "bior3.3", "sym2", "coif1"):
        with pytest.raises(NotImplementedError):
            TriPlaneVolume(number_of_features=8, plane_resolution=64, inner_multi_res_scale=4, wavelet_type=wave)
    TriPlaneVolume(number_of_features=8, plane_resolution=64, wavelet_type="db4")     # no levels: the wavelet is never applied


@pytest.fixture
def emu(monkeypatch):
    return emu_backend.install(monkeypatch)


@pytest.mark.parametrize("sparse", [False, True])
def test_training_step_with_bior44_matches_oracle_pipeline(emu, sparse):
    """NeRFNetwork(wavelet_type='bior4.4') through TrainStep.forward_backward (dense IDWT, or work-list IDWT with
    SplitIdwtBackward) against the oracle's training step with the same wavelet"""
    from trinerflet_b200 import scene, trainer
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS["tiny"]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"], triplane_resolution=c["R"],
                      triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"], hidden_dim_color=c["hidden"], wavelet_type="bior4.4")
    assert net.encoder.wavelet_type == "bior4.4"
    scene.init_model_(net, seed=0)
    with torch.no_grad():
        for p in net.encoder.planes_features_wavelet_coefs:
            p.normal_(0.0, 0.05, generator=torch.Generator().manual_seed(p.shape[-1]))    # non-zero detail coefficients
    scene.install_ball_occupancy(net, 0.45 if sparse else 0.75)
    net.train()
    sc = scene.make_scene()
    N = 300
    ro, rd, tgt = scene.sample_batch(sc, N, torch.Generator().manual_seed(0))
    opt = trainer.default_opt(fp16=False)
    ts = trainer.TrainStep(net, opt, None)
    ts.sparse_idwt = sparse
    ts.plan_on_any_device = True
    torch.manual_seed(5)
    loss = ts.forward_backward(ro, rd, tgt, update_grid=False)
    assert (ts._plan is not None) == sparse
    M = int(net.step_counter[0, 0])
    torch.manual_seed(5)
    noises = torch.rand(N).numpy()
    pf = net.encoder.planes_features.detach().clone().contiguous().requires_grad_(True)
    coefs = [p.detach().clone().contiguous().requires_grad_(True) for p in net.encoder.planes_features_wavelet_coefs]
    W = [w.detach().clone().requires_grad_(True) for w in net._weights()]
    loss_o, M_o = wavelet_oracle.train_step(pf, coefs, W, ro, rd, tgt, net.density_bitfield.numpy(), noises, "bior4.4",
                                            lam=opt.wavelet_regularization)
    assert M_o == M
    assert abs(float(loss) - loss_o) <= 1e-5 * abs(loss_o)
    assert rel_l2(net.encoder.planes_features.grad, pf.grad) <= 1e-4
    for p, c in zip(net.encoder.planes_features_wavelet_coefs, coefs):
        assert rel_l2(p.grad, c.grad) <= 1e-4
    for w, wo in zip(net._weights(), W):
        assert rel_l2(w.grad, wo.grad) <= 1e-4


def test_planewise_adjoint_and_band_limited_queries_with_haar(emu):
    """PlanewiseIdwtBackward (the multi-GPU per-plane adjoint) and get_planes(max_res / get_all_resolutions) carry the wavelet"""
    from trinerflet_b200.triplane_encoder import PlanewiseIdwtBackward, TriPlaneVolume
    torch.manual_seed(0)
    enc = TriPlaneVolume(number_of_features=8, plane_resolution=64, inner_multi_res_scale=4, wavelet_type="haar")
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for p in enc.planes_features_wavelet_coefs:
            p.copy_(torch.randn(p.shape, generator=g))
    pf = enc.planes_features.detach().clone().requires_grad_(True)
    coefs = [p.detach().clone().requires_grad_(True) for p in enc.planes_features_wavelet_coefs]
    ref = ow.build_planes(pf, coefs, "haar")
    assert rel_l2(enc.get_planes(), ref) <= 1e-6
    enc.reset_cache()
    half, all_res = enc.get_planes(max_res=32), None
    assert half.shape[-1] == 32 and rel_l2(half, ow.build_planes(pf, coefs[:1], "haar")) <= 1e-6
    enc.reset_cache()
    all_res = enc.get_planes(get_all_resolutions=True)
    _, all_ref = ow.build_planes_limited(pf, coefs, get_all_resolutions=True, wave="haar")
    assert len(all_res) == len(all_ref) and all(rel_l2(a, b) <= 1e-6 for a, b in zip(all_res, all_ref))
    gout = torch.randn(ref.shape, generator=g)
    ref.backward(gout)
    bw = PlanewiseIdwtBackward(enc, gout)
    for p in range(3):
        bw.run(p)
    bw.assign()
    assert rel_l2(enc.planes_features.grad, pf.grad) <= 1e-5
    for p, c in zip(enc.planes_features_wavelet_coefs, coefs):
        assert rel_l2(p.grad, c.grad) <= 1e-5
