"""CPU: the super_resolution encoders (trinerflet_b200/sr_encoder.py, SURVEY.md 8 f-4) over the host build of the product
kernels (tests/emu_backend.py), against
  * the reference's own fp32 results (tests/golden/sr_encoder_fp32.npz, written by tests/golden/make_sr_golden.py from the
    reference module imported out of /root/reference),
  * the oracle restatement (oracle/sr_encoder.py), which is pinned against the same file here,
  * and, when /root/reference is present (this container), the reference module itself, live, on a larger random case."""
import numpy as np
import pytest
import torch

from tests import emu_backend, sr_cases
from tests.golden import make_sr_golden as G
from tests.util import rel_l2


@pytest.fixture
def emu(monkeypatch):
    return emu_backend.install(monkeypatch)


def test_oracle_restatement_matches_reference_golden():
    """oracle/sr_encoder.py (fp32, same ops) against what the reference classes produced: planes of both readings for every
    (low_res_scale, high_res_scale) of the fixture, features, and the plain-plane pyramids"""
    from oracle import sr_encoder as osr
    z = sr_cases.golden()
    x = torch.from_numpy(z["x"])
    pf = torch.from_numpy(z["wavelet/state/planes_features"])
    coefs = [torch.from_numpy(z[f"wavelet/state/planes_features_wavelet_coefs.{l}"]) for l in range(2)]
    R = G.WAVELET["plane_resolution"]
    for lo, hi in G.SCALES:
        tag = f"wavelet/{lo}_{hi}/"
        single, none = osr.two_readings(pf, coefs, R, lo, hi, False)
        assert none is None
        assert tuple(single.shape) == tuple(z[tag + "planes_single_shape"])
        np.testing.assert_array_equal(single.numpy(), z[tag + "planes_low"])
        low, high = osr.two_readings(pf, coefs, R, lo, hi, True)
        np.testing.assert_array_equal(low.numpy(), z[tag + "planes_low"])
        np.testing.assert_array_equal(high.numpy(), z[tag + "planes_high"])
        np.testing.assert_array_equal(osr.encode(low, x).numpy(), z[tag + "feat_low"])
        np.testing.assert_array_equal(osr.encode(high, x).numpy(), z[tag + "feat_high"])
    for mode in ("concatination", "mul"):
        tag = f"kplanes/{mode}/"
        planes = [torch.from_numpy(z[tag + f"state/triplane_lst.{l}.planes_features"]) for l in range(G.KPLANES["levels"])]
        np.testing.assert_array_equal(osr.kplanes(planes, x, mode).numpy(), z[tag + "feat"])
    for name, fn in (("multiscale", osr.multiscale), ("multiscale_mul", osr.multiscale_mul)):
        tag = name + "/state/"
        low = [torch.from_numpy(z[tag + "low_res_vol.triplane_lst.0.planes_features"])]
        high = [torch.from_numpy(z[tag + f"high_res_vol.triplane_lst.{l}.planes_features"]) for l in range(2)]
        np.testing.assert_array_equal(fn(low, high, x, "concatination", False).numpy(), z[name + "/feat_low"])
        np.testing.assert_array_equal(fn(low, high, x, "concatination", True).numpy(), z[name + "/feat_high"])


def test_wavelet_two_readings_match_reference_golden(emu):
    sr_cases.check_wavelet_golden("cpu")


def test_plane_pyramids_match_reference_golden(emu):
    sr_cases.check_kplanes_golden("cpu")


def test_two_render_step_matches_oracle(emu):
    sr_cases.check_against_oracle("cpu", C=8, R=64, scale=8, low=4, high=1, M=300)
    sr_cases.check_against_oracle("cpu", C=24, R=32, scale=2, low=2, high=2, M=100, seed=1)   # C outside {16, 32, 48}: generic kernels


def test_position_gradient_properties(emu):
    sr_cases.check_position_gradient_properties("cpu")


def test_high_order_gradients_like_grid_backward(emu):
    sr_cases.check_high_order_gradients("cpu")


def test_low_resolution_phase_runs_coarse_levels_only(emu):
    sr_cases.check_low_resolution_phase_cost("cpu", R=128)


def test_constructor_surface_and_rejections():
    from trinerflet_b200 import sr_encoder
    enc = sr_encoder.TriPlaneVolume(number_of_features=8, plane_resolution=32, inner_multi_res_scale=4, low_res_scale=2)
    assert enc.n_output_dims == enc.output_dim == 24 and enc.n_input_dims == 3
    assert enc.double_resolution_mode is False and enc.current_resolution_mode == 'low_res' and enc.enable_cache is False
    assert enc._level_split() == (1, 2)
    assert [tuple(p.shape) for p in enc.get_wavelet_features()] == [(3, 8, 3, 8, 8), (3, 8, 3, 16, 16)]
    with pytest.raises(AssertionError):
        sr_encoder.TriPlaneVolume(low_res_scale=1, high_res_scale=2)
    with pytest.raises(AssertionError):
        enc.set_resolution_mode('mid_res')
    with pytest.raises(NotImplementedError):
        sr_encoder.TriPlaneVolume(plane_resolution=32, inner_multi_res_scale=4, wavelet_base_resolution=16)
    with pytest.raises(NotImplementedError):
        sr_encoder.TriPlaneVolume(plane_resolution=32, inner_multi_res_scale=4, wavelet_type='haar')
    # plain planes take any wavelet name and base resolution (KPlaneVolume passes 'haar' / the plane side), and init_fn
    torch.manual_seed(0)
    plain = sr_encoder.TriPlaneVolume(number_of_features=4, plane_resolution=8, wavelet_type='haar', wavelet_base_resolution=8,
                                      init_fn=sr_encoder.kplanes_init_mul)
    torch.manual_seed(0)
    torch.randn(3, 4, 8, 8)
    assert torch.equal(plain.planes_features.detach(), 2 * torch.rand(3, 4, 8, 8) - 1)
    assert plain.get_wavelet_features() == [] and len(plain.state_dict()) == 3
    # no CUDA extension call is made on CPU tensors: the product has no CPU path
    with pytest.raises(RuntimeError):
        enc(torch.rand(4, 3))


@pytest.mark.skipif(not G.reference_available(), reason="needs a checkout of the original project (TRINERFLET_REFERENCE)")
def test_against_the_reference_module_live(emu):
    """the reference's TriPlaneVolume (its configs' shape: low_res_scale 4, high_res_scale 1) and ours from the same state dict,
    through the application's step sequence; then the reverse direction of the checkpoint: our state dict into the reference"""
    from trinerflet_b200 import sr_encoder
    ref = G.load_reference_module()
    kw = dict(number_of_features=8, plane_resolution=128, inner_multi_res_scale=16, low_res_scale=4, high_res_scale=1,
              wavelet_type='bior6.8', wavelet_base_resolution=0, init_sigma=0.1, lbound=1, viewdir_plane_resolution=-1,
              apply_activation_on_features=False, inner_multi_res_scale_current=1)      # networks.py:143-156
    gen = torch.Generator().manual_seed(7)
    theirs = G.quiet(ref.TriPlaneVolume, **kw)
    G.randomise_(theirs, gen)
    ours = sr_encoder.TriPlaneVolume(**kw)
    ours.load_state_dict(theirs.state_dict(), strict=True)
    assert list(ours.state_dict().keys()) == list(theirs.state_dict().keys())
    x = G.test_points(400, gen)
    w_low, w_high = torch.randn(400, 24, generator=gen), torch.randn(400, 24, generator=gen)
    a = G.two_render_step(theirs, x, w_low, w_high)
    b = G.two_render_step(ours, x, w_low, w_high)
    assert rel_l2(b[0], a[0]) <= sr_cases.TOL and rel_l2(b[1], a[1]) <= sr_cases.TOL
    assert rel_l2(b[3], a[3]) <= sr_cases.TOL_X
    for name in a[2]:
        assert rel_l2(b[2][name], a[2][name]) <= sr_cases.TOL, name
    # low-resolution-only phase of the application (double mode off): coarse levels only
    for enc in (theirs, ours):
        enc.enable_cache = False
        enc.set_double_mode(False)
    with torch.no_grad():
        assert tuple(ours.get_planes().shape) == tuple(theirs.get_planes().shape) == (3, 8, 32, 32)
        assert rel_l2(ours(x), theirs(x)) <= sr_cases.TOL
    # get_grid_features (:371-413): the lattice, its axis permutation and the features on it
    with torch.no_grad():
        lb_a, feat_a, grid_a = theirs.get_grid_features(6)
        lb_b, feat_b, grid_b = ours.get_grid_features(6)
    assert lb_a == lb_b and torch.equal(grid_a, grid_b) and tuple(feat_a.shape) == tuple(feat_b.shape) == (6, 6, 6, 24)
    assert rel_l2(feat_b, feat_a) <= sr_cases.TOL
    G.randomise_(ours, gen)
    theirs.load_state_dict(ours.state_dict(), strict=True)
    with torch.no_grad():
        assert rel_l2(ours(x), theirs(x)) <= sr_cases.TOL
