"""GPU: the marching cubes of csrc/mesh.cu on the device against the numpy restatement oracle/mesh.py, bit for bit (analytic
volumes, random noise, the density volume of a `small` NeRFNetwork); the device sweep extract_fields against the reference's
chunked loop with a .cpu() per chunk; extract_geometry end to end; determinism; a 1024^3 ball (64-bit indexing)."""
import importlib
import os
import sys
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import mesh as om
from oracle import reference_path
from tests.test_mesh_emu import (_assert_same, assert_closed_oriented, assert_on_lattice_edges, ball, euler, noise, signed_volume,
                                 torus, touching_balls)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,u,thr", [
    ("ball64", ball(64, 25.0), 0.0),
    ("torus48", torus(48, 13.0, 5.5), 0.0),
    ("touching_balls40", touching_balls(40, 9.0), 0.0),
    ("equal_to_threshold", np.random.default_rng(3).integers(0, 3, (33, 31, 29)).astype(np.float32), 1.0),
])
def test_device_matches_the_oracle_on_analytic_volumes(name, u, thr):
    from trinerflet_b200 import mesh
    got = mesh.marching_cubes(torch.from_numpy(u).cuda(), thr)
    _assert_same(got, om.marching_cubes(u, thr))
    if name != "equal_to_threshold":
        assert_closed_oriented(got[1])


def test_device_matches_the_oracle_on_noise_128():
    from trinerflet_b200 import mesh
    u = noise(128, seed=1)
    got = mesh.marching_cubes(u, 0.25)                   # numpy input: moved to the device
    _assert_same(got, om.marching_cubes(u, 0.25))
    assert len(got[1]) > 1_000_000
    _assert_same(mesh.marching_cubes(u, 0.25), got)      # two calls, identical arrays


def test_nan_raises_on_the_device():
    from trinerflet_b200 import mesh
    u = ball(40, 9.0)
    u[39, 0, 17] = np.nan
    with pytest.raises(ValueError):
        mesh.marching_cubes(torch.from_numpy(u).cuda(), 0.0)
    v, t = mesh.marching_cubes(torch.full((9, 8, 7), -1.0, device="cuda"), 0.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)


@pytest.fixture(scope="module")
def small_net():
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS["small"]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"],
                      triplane_resolution=c["R"], triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"],
                      hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=0)
    net.eval()
    return net


def _query(net):
    def query_func(pts):                                 # the reference Trainer.save_mesh's query_func
        with torch.no_grad():
            with torch.autocast("cuda", dtype=torch.float16):
                return net.density(pts.to("cuda"))["sigma"]
    return query_func


def test_sweep_and_extract_geometry_match_the_reference_loop(small_net):
    from trinerflet_b200 import mesh
    bmin, bmax = small_net.aabb_infer[:3], small_net.aabb_infer[3:]
    q = _query(small_net)
    u_ref = om.extract_fields(bmin, bmax, 256, q)                 # .cpu() per chunk into a numpy volume
    u_dev = mesh.extract_fields(bmin, bmax, 256, q)
    assert u_dev.is_cuda and u_dev.dtype == torch.float32
    assert np.array_equal(u_dev.cpu().numpy(), u_ref)
    thr = float(np.median(u_ref))
    got = mesh.marching_cubes(u_dev, thr)
    _assert_same(got, om.marching_cubes(u_ref, thr))
    assert len(got[1]) > 10_000
    v, t = mesh.extract_geometry(bmin, bmax, 256, thr, q)
    vo, to = om.marching_cubes(u_ref, thr)
    _assert_same((v, t), (om.world_transform(vo, bmin, bmax, 256), to))
    _assert_same(mesh.extract_geometry(bmin, bmax, 256, thr, q), (v, t))


def test_ball_1024_is_a_closed_oriented_sphere():
    from trinerflet_b200 import mesh
    n, r = 1024, 400.0
    a = torch.arange(n, device="cuda", dtype=torch.float32) - (n - 1) / 2 - 0.137
    u = r - torch.sqrt(a[:, None, None] ** 2 + a[None, :, None] ** 2 + a[None, None, :] ** 2)
    v, t = mesh.marching_cubes(u, 0.0)
    del u
    torch.cuda.empty_cache()
    assert v.shape[0] > 2 ** 21
    assert_closed_oriented(t)
    assert euler(v, t) == 2
    assert_on_lattice_edges(v, (n, n, n))
    assert abs(signed_volume(v, t) / (4.0 / 3.0 * np.pi * r ** 3) - 1) < 0.01


REF = reference_path("reconstruction")


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original project (TRINERFLET_REFERENCE)")
def test_reference_extract_fields_over_the_dropin(small_net, monkeypatch):
    """the reference's own nerf/utils.py extract_fields over the drop-in's density() gives our device volume"""
    from trinerflet_b200 import mesh
    for name in ["trimesh", "cv2", "tensorboardX", "mcubes", "lpips", "torch_ema", "torchmetrics", "torchmetrics.functional", "imageio",
                 "torchvision", "matplotlib", "matplotlib.pyplot", "nerfacc", "raymarching", "shencoder"]:
        try:
            importlib.import_module(name)
        except Exception:
            monkeypatch.setitem(sys.modules, name, mock.MagicMock())
    monkeypatch.syspath_prepend(REF)
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "nerf"}
    for k in saved:
        del sys.modules[k]
    try:
        utils = importlib.import_module("nerf.utils")
        bmin, bmax = small_net.aabb_infer[:3], small_net.aabb_infer[3:]
        q = _query(small_net)
        assert np.array_equal(utils.extract_fields(bmin, bmax, 160, q), mesh.extract_fields(bmin, bmax, 160, q).cpu().numpy())
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] == "nerf"]:
            del sys.modules[k]
        sys.modules.update(saved)
