"""Boundary proof (SURVEY.md 8b): the REFERENCE's own host code -- reconstruction/nerf/renderer.py (NeRFRenderer.run_cuda
train + eval branches, update_extra_state, mark_untrained_grid; :257-381, :383-446, :448-542), nerf/network.py (NeRFNetwork)
and encoding.py (get_encoder) -- imported UNMODIFIED from a checkout of the original project and run over this package's
drop-in modules:

    import raymarching                                  ->  trinerflet_b200.raymarching       (renderer.py:9)
    from shencoder import SHEncoder                     ->  trinerflet_b200.shencoder         (encoding.py:61)
    from triplaneencoder.triplane_encoder import ...    ->  trinerflet_b200.triplane_encoder  (encoding.py:76)

i.e. the four-import patch of INTEGRATION.md, then compared with trinerflet_b200.NeRFNetwork / NeRFRenderer on the same
parameters, rays and RNG seed.  The kernels run as their host build (tests/emu): this is a test of the INTERFACE -- names,
argument order, return conventions, in-place semantics, RNG call order -- not of device code.  Runs only where the
environment variable TRINERFLET_REFERENCE names such a checkout."""
import importlib
import os
import sys
import types
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import reference_path
from tests import emu_backend

REF = reference_path("reconstruction")
pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original project (TRINERFLET_REFERENCE)")


@pytest.fixture
def ref_modules(monkeypatch):
    """the reference's nerf.renderer / nerf.network with the three extension imports shadowed by the drop-in modules"""
    emu_backend.install(monkeypatch)
    import trinerflet_b200.raymarching as rm
    import trinerflet_b200.shencoder as sh
    import trinerflet_b200.triplane_encoder as te
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("nerf", "encoding", "activation", "triplaneencoder")}
    for k in saved:
        del sys.modules[k]
    monkeypatch.setitem(sys.modules, "raymarching", rm)
    monkeypatch.setitem(sys.modules, "shencoder", sh)
    pkg = types.ModuleType("triplaneencoder")
    pkg.__path__ = []
    monkeypatch.setitem(sys.modules, "triplaneencoder", pkg)
    monkeypatch.setitem(sys.modules, "triplaneencoder.triplane_encoder", te)
    for name in ["trimesh", "cv2", "tensorboardX", "mcubes", "lpips", "torch_ema", "torchmetrics", "torchmetrics.functional", "imageio",
                 "torchvision", "matplotlib", "matplotlib.pyplot", "nerfacc"]:
        try:
            importlib.import_module(name)
        except Exception:
            monkeypatch.setitem(sys.modules, name, mock.MagicMock())
    monkeypatch.syspath_prepend(REF)
    renderer = importlib.import_module("nerf.renderer")
    network = importlib.import_module("nerf.network")
    assert renderer.__file__.startswith(REF) and network.__file__.startswith(REF)
    assert renderer.raymarching is rm                      # the reference's `import raymarching` resolved to the drop-in
    yield renderer, network
    for k in [k for k in sys.modules if k.split(".")[0] in ("nerf", "encoding", "activation", "triplaneencoder")]:
        del sys.modules[k]
    sys.modules.update(saved)


KW = dict(triplane_channels=16, triplane_resolution=128, triplane_wavelet_levels=2, learn_rotation_axis=False, dropout=0,
          wavelet_type="bior6.8", lbound_auto_scale=False, upscale_ratio_bound=-1, upscale_levels=2, wavelet_base_resolution=0)


def _pair(network):
    """(reference NeRFNetwork over the drop-in modules, trinerflet_b200 NeRFNetwork) with identical parameters / occupancy"""
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    ref = network.NeRFNetwork(encoding="triplane_wavelet", bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, **KW)
    ours = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, **KW)
    scene.init_model_(ours, seed=0)
    missing = ref.load_state_dict(ours.state_dict(), strict=True)      # same parameter / buffer names on both sides
    assert not missing.missing_keys and not missing.unexpected_keys
    for m in (ref, ours):
        grid = scene.ball_density_grid(1.5, 0.75)
        m.density_grid.copy_(grid)
        m.density_bitfield.copy_(scene.packbits_cpu(grid, 0.5))
        m.mean_density = float(grid.clamp(min=0).mean())
        m.iter_density = 16
    return ref, ours


def test_reference_run_cuda_train_and_eval_over_the_dropin_modules(ref_modules):
    renderer, network = ref_modules
    from trinerflet_b200 import scene
    ref, ours = _pair(network)
    assert type(ref).__mro__[1] is renderer.NeRFRenderer
    sc = scene.make_scene()
    ro, rd, _ = scene.sample_batch(sc, 300, torch.Generator().manual_seed(0))
    outs = []
    for m in (ref, ours):                                   # training branch (renderer.py:269-321): march -> field -> composite
        m.train()
        torch.manual_seed(3)
        o = m.render(ro.unsqueeze(0), rd.unsqueeze(0), staged=False, bg_color=None, perturb=True, force_all_rays=False,
                     dt_gamma=0, max_steps=256)
        loss = o["image"].sum() + o["weights_sum"].sum() if "weights_sum" in o else o["image"].sum()
        loss.backward()
        outs.append((o, [p.grad.clone() for p in m.parameters()], int(m.step_counter[0, 0]), m.local_step))
    (o_r, g_r, cnt_r, ls_r), (o_o, g_o, cnt_o, ls_o) = outs
    assert cnt_r == cnt_o > 1000 and ls_r == ls_o == 1
    assert torch.equal(o_r["image"], o_o["image"])
    fin = torch.isfinite(o_r["depth"])
    assert torch.equal(fin, torch.isfinite(o_o["depth"])) and torch.equal(o_r["depth"][fin], o_o["depth"][fin])
    for a, b in zip(g_r, g_o):
        assert torch.equal(a, b)                            # same kernels, same order: bit-identical gradients
    ro2, rd2 = scene.full_frame(sc, 7)
    pick = torch.arange(0, ro2.shape[0], 1201)
    ro2, rd2 = ro2[pick].contiguous(), rd2[pick].contiguous()
    res = []
    for m in (ref, ours):                                   # inference branch (renderer.py:324-374): the march/composite loop
        m.eval()
        with torch.no_grad():
            res.append(m.render(ro2.unsqueeze(0), rd2.unsqueeze(0), staged=True, bg_color=1, perturb=False, dt_gamma=0, max_steps=256))
    assert float(res[0]["weights_sum"].sum() if "weights_sum" in res[0] else res[0]["image"].sum()) > 0
    assert torch.equal(res[0]["image"], res[1]["image"])
    fin = torch.isfinite(res[0]["depth"])
    assert torch.equal(res[0]["depth"][fin], res[1]["depth"][fin])


def test_reference_update_extra_state_and_mark_untrained_grid_over_the_dropin_modules(ref_modules):
    renderer, network = ref_modules
    from trinerflet_b200 import scene
    ref, ours = _pair(network)
    # (the partial sweep writes duplicate cell indices, "allow for duplication" renderer.py:503: which duplicate wins is a race
    #  inside index_put_ -- in the reference itself -- unless the assignment runs sequentially)
    monkeypatch_threads = torch.get_num_threads()
    torch.set_num_threads(1)
    for it in (0, 16):                                      # full sweep, then the partial (uniform + occupied) sweep
        for m in (ref, ours):
            m.iter_density = it
            m.local_step = 3
            m.step_counter[:3, 0] = torch.tensor([100, 200, 330], dtype=torch.int32)
            torch.manual_seed(21 + it)
            m.update_extra_state()
        assert ref.iter_density == ours.iter_density == it + 1
        assert ref.mean_count == ours.mean_count == 210 and ref.local_step == ours.local_step == 0
        assert abs(ref.mean_density - ours.mean_density) <= 1e-6 * abs(ref.mean_density)
        # cell positions: the reference forms them with separate torch ops, the drop-in with one kernel (one fused multiply-add
        # more or less): sigma agrees to float rounding, and a bit can only flip where a cell sits on the threshold
        err = ((ref.density_grid - ours.density_grid).abs() / ref.density_grid.abs().clamp_min(1e-6)).max().item()
        flips = int((ref.density_bitfield ^ ours.density_bitfield).to(torch.int32).apply_(lambda v: bin(v).count("1")).sum())
        print(f"update_extra_state it={it}: max rel |grid diff| = {err:.2e}, bit flips = {flips} of {ref.density_bitfield.numel() * 8}")
        assert err <= 1e-5 and flips <= 4
    torch.set_num_threads(monkeypatch_threads)
    sc = scene.make_scene()
    poses = sc.poses[:6]
    for m in (ref, ours):
        m.density_grid.zero_()
        m.mark_untrained_grid(poses, sc.intrinsics)
    assert torch.equal(ref.density_grid, ours.density_grid) and int((ours.density_grid < 0).sum()) > 0


# one stage of the README command (/root/reference/README.md:46), scaled down and without --fp16 (the host build computes fp32)
CLI = ("main_nerf.py --path data --workspace out --cuda_ray --bound 1.5 --scale 1 --dt_gamma 0 --iters 1000 --num_rays 300 "
       "--background_color 0 --triplane_wavelet --triplane_channels 16 --triplane_wavelet_levels 2 --triplane_resolution 128 "
       "--wavelet_regularization 0.2 --downscale 1 --ckpt latest_model --ema_decay -1 --training_evaluate_test --warmup_steps 0 "
       "--fast_training --max_steps 256")
STAGED = ['iters', 'num_rays', 'triplane_resolution', 'triplane_wavelet_levels', 'downscale', 'warmup_steps', 'lr',
          'wavelet_regularization', 'upscale_ratio_bound', 'upscale_levels']                     # main_nerf.py:168-170
PASSED_TO_NERF = ['triplane_channels', 'triplane_resolution', 'triplane_wavelet_levels', 'wavelet_type', 'hidden_dim',
                  'hidden_dim_color', 'hidden_dim_bg', 'learn_rotation_axis', 'dropout', 'inner_bound', 'lbound_auto_scale',
                  'upscale_ratio_bound', 'upscale_levels', 'density_blob_scale', 'density_blob_std', 'mlp_weight_decay',
                  'wavelet_base_resolution', 'nerfacc_renderer']                                  # main_nerf.py:44-58


def test_reference_trainer_train_step_from_its_own_command_line(ref_modules, monkeypatch):
    """The reference's option parser (run_utils.get_params) on a README-shaped command line, its model construction
    (main_nerf.py:44-72) and its Trainer.train_step (nerf/utils.py:532-679: render with **vars(opt), MSE, the wavelet
    regulariser expression) -- all unmodified -- over (a) the reference NeRFNetwork on the drop-in modules and (b) this
    package's NeRFNetwork built from the SAME keyword arguments; then the fast path INTEGRATION.md offers in its place,
    TrainStep.forward_backward, on the same rays.  Loss and every parameter gradient must agree."""
    import argparse
    from trinerflet_b200 import scene, trainer as our_trainer
    from trinerflet_b200.network import NeRFNetwork as OurNet
    renderer, network = ref_modules
    run_utils = importlib.import_module("run_utils")
    utils = importlib.import_module("nerf.utils")
    assert run_utils.__file__.startswith(REF) and utils.__file__.startswith(REF)
    monkeypatch.setattr(sys, "argv", CLI.split())
    opt = run_utils.get_params()
    for key in STAGED:                                                   # run(): one stage (main_nerf.py:190-199)
        vars(opt)[key] = vars(opt)[key][0]
    assert opt.triplane_wavelet and opt.cuda_ray and opt.wavelet_regularization == 0.2 and opt.patch_size == 1
    extra = {k: vars(opt)[k] for k in PASSED_TO_NERF}
    build = dict(encoding="triplane_wavelet", bound=opt.bound, cuda_ray=opt.cuda_ray, density_scale=opt.density_scale,
                 min_near=opt.min_near, density_thresh=opt.density_thresh, bg_radius=opt.bg_radius, **extra)
    ref, ours, fast = network.NeRFNetwork(**build), OurNet(**build), OurNet(**build)
    scene.init_model_(ours, seed=0)
    with torch.no_grad():
        for p in ours.encoder.planes_features_wavelet_coefs:            # non-zero detail coefficients: the regulariser has a gradient
            p.copy_(0.05 * torch.randn(p.shape, generator=torch.Generator().manual_seed(5)))
    grid = scene.ball_density_grid(1.5, 0.75)
    for m in (ref, ours, fast):
        if m is not ours:
            m.load_state_dict(ours.state_dict(), strict=True)
        m.density_grid.copy_(grid)
        m.density_bitfield.copy_(scene.packbits_cpu(grid, 0.5))
        m.mean_density = float(grid.clamp(min=0).mean())
        m.iter_density = 16
        m.train()
    sc = scene.make_scene()
    ro, rd, tgt = scene.sample_batch(sc, opt.num_rays, torch.Generator().manual_seed(0))
    data = {"rays_o": ro.unsqueeze(0), "rays_d": rd.unsqueeze(0), "images": tgt.unsqueeze(0)}
    results = []
    for m in (ref, ours):
        me = argparse.Namespace(model=m, opt=opt, criterion=torch.nn.MSELoss(reduction='none'), error_map=None, nerfacc_renderer=None)
        torch.manual_seed(11)
        pred, gt, loss, aux = utils.Trainer.train_step(me, {k: v.clone() for k, v in data.items()})
        loss.backward()
        results.append((pred.detach(), float(loss.detach()), aux, [p.grad.clone() for p in m.parameters()]))
    (pred_r, loss_r, aux_r, g_r), (pred_o, loss_o, aux_o, g_o) = results
    assert aux_r.keys() == aux_o.keys() == {"mse", "wavelet_reg"} and aux_r["wavelet_reg"] > 0
    assert torch.equal(pred_r, pred_o) and loss_r == loss_o
    for a, b in zip(g_r, g_o):
        assert torch.equal(a, b)
    # the replacement for train_step + backward: same rays, same jitter draw
    step = our_trainer.TrainStep(fast, opt, None)
    torch.manual_seed(11)
    loss_f = step.forward_backward(ro, rd, tgt, update_grid=False)
    assert abs(float(loss_f) - loss_r) <= 1e-6 * abs(loss_r)
    for p, g in zip(fast.parameters(), g_r):
        assert float((p.grad - g).norm() / g.norm().clamp_min(1e-30)) <= 1e-5


def test_reference_epoch_loop_against_the_fast_path(ref_modules, monkeypatch):
    """Four optimizer steps of the reference's Trainer.train_one_epoch2 (nerf/utils.py:1115-1177: shuffle_data, select_batch,
    reset_cahce / get_planes, train_step, scaler.scale(loss).backward(), scaler.step(optimizer), LambdaLR(decay_function)),
    unmodified, over this package's NeRFNetwork -- against the loop INTEGRATION.md describes: the same batches through
    TrainStep.step with FusedAdam and the same schedule.  The two parameter trajectories must stay together."""
    import argparse
    import functools
    from trinerflet_b200 import scene, trainer as our_trainer
    from trinerflet_b200.network import NeRFNetwork as OurNet
    from trinerflet_b200.optim import FusedAdam
    run_utils = importlib.import_module("run_utils")
    utils = importlib.import_module("nerf.utils")
    monkeypatch.setattr(sys, "argv", (CLI + " --update_extra_interval 1000 --warmup_steps 2").split())
    opt = run_utils.get_params()
    for key in STAGED:
        vars(opt)[key] = vars(opt)[key][-1]
    build = dict(encoding="triplane_wavelet", bound=opt.bound, cuda_ray=opt.cuda_ray, density_scale=opt.density_scale,
                 min_near=opt.min_near, density_thresh=opt.density_thresh, bg_radius=opt.bg_radius,
                 **{k: vars(opt)[k] for k in PASSED_TO_NERF})
    theirs_loop, fast = OurNet(**build), OurNet(**build)
    scene.init_model_(theirs_loop, seed=0)
    fast.load_state_dict(theirs_loop.state_dict(), strict=True)
    grid = scene.ball_density_grid(1.5, 0.75)
    for m in (theirs_loop, fast):
        m.density_grid.copy_(grid)
        m.density_bitfield.copy_(scene.packbits_cpu(grid, 0.5))
        m.mean_density = float(grid.clamp(min=0).mean())
        m.iter_density = 16
        m.mark_bitfield_changed()
    sc = scene.make_scene()
    n_steps = 4
    ro, rd, tgt = scene.sample_batch(sc, n_steps * opt.num_rays, torch.Generator().manual_seed(2))
    all_data = {"rays_o": ro.view(1, -1, 3), "rays_d": rd.view(1, -1, 3), "images": tgt.view(1, -1, 3)}    # collate_all layout [B, N, C]
    sched = lambda optimizer: torch.optim.lr_scheduler.LambdaLR(optimizer, lambda it: utils.decay_function(it, opt))   # main_nerf.py:131

    # (a) the reference's loop, its own optimizer construction (main_nerf.py:119)
    optimizer = torch.optim.Adam(theirs_loop.get_params(opt.lr), betas=(0.9, 0.99), eps=1e-15)
    me = argparse.Namespace(model=theirs_loop, opt=opt, criterion=torch.nn.MSELoss(reduction='none'), error_map=None, nerfacc_renderer=None,
                            log=lambda *a, **k: None, epoch=1, optimizer=optimizer, local_rank=1, report_metric_at_train=False, metrics=[],
                            local_step=0, global_step=1, device=torch.device("cpu"), fp16=False, use_tensorboardX=False,
                            scaler=torch.amp.GradScaler("cuda", enabled=False), scheduler_update_every_step=True,
                            lr_scheduler=sched(optimizer), stats={"loss": []}, ema=None)
    me.train_step = functools.partial(utils.Trainer.train_step, me)
    me.clear_grad = functools.partial(utils.Trainer.clear_grad, me)
    torch.manual_seed(21)
    utils.Trainer.train_one_epoch2(me, {k: v.clone() for k, v in all_data.items()})
    assert me.global_step == 1 + n_steps and len(me.stats["loss"]) == 1

    # (b) the fast path on the same shuffled batches and jitter draws
    fused = FusedAdam(fast.get_params(opt.lr), betas=(0.9, 0.99), eps=1e-15)
    lr_sched = sched(fused)
    step = our_trainer.TrainStep(fast, opt, fused)
    fast.train()
    torch.manual_seed(21)
    shuffled = utils.shuffle_data({k: v.clone() for k, v in all_data.items()})
    losses = []
    for b in range(n_steps):
        d = utils.select_batch(shuffled, b, opt.num_rays, torch.device("cpu"))
        losses.append(float(step.step(d["rays_o"][0], d["rays_d"][0], d["images"][0], update_grid=False)))
        lr_sched.step()
    assert abs(sum(losses) / n_steps - me.stats["loss"][0]) <= 1e-5 * me.stats["loss"][0]
    assert optimizer.param_groups[0]["lr"] == fused.param_groups[0]["lr"] != opt.lr            # the warm-up schedule moved both
    start = OurNet(**build)
    scene.init_model_(start, seed=0)
    for (name, a), b, a0 in zip(theirs_loop.named_parameters(), fast.parameters(), start.parameters()):
        travelled = float((a - a0).norm())
        assert travelled > 0.0, name                                              # four Adam steps moved every tensor ...
        assert float((a - b).norm()) <= 1e-4 * travelled, name      # ... and both loops moved it to the same place (measured: 2e-7)
