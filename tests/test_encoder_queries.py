"""CPU: the tooling queries of the reconstruction encoder -- TriPlaneVolume.get_planes(max_res / max_scale /
get_all_resolutions) and get_grid_features (reconstruction/triplaneencoder/triplane_encoder.py:364-416, :485-512; callers
nerf/utils.py:1649 save_triplane and :500) -- over the host build of the kernels, against the oracle restatement
(oracle/wavelet.build_planes_limited) and, given a checkout of the original project (TRINERFLET_REFERENCE), the reference
module itself."""
import contextlib
import importlib.util
import io
import os
import sys
import types

import pytest
import torch

from oracle import field as of
from oracle import reference_path
from oracle import wavelet as ow
from tests import emu_backend
from tests.util import rel_l2

REF = reference_path("reconstruction")
KW = dict(number_of_features=8, plane_resolution=64, init_sigma=0.1, lbound=1.5, inner_multi_res_scale=8)   # 8 -> 16 -> 32 -> 64


@pytest.fixture
def emu(monkeypatch):
    return emu_backend.install(monkeypatch)


def _ours(seed=0):
    from trinerflet_b200.triplane_encoder import TriPlaneVolume
    enc = TriPlaneVolume(**KW)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in enc.parameters():
            p.copy_(0.2 * torch.randn(p.shape, generator=g))
    return enc


def _params(enc):
    return enc.planes_features.detach().contiguous(), [p.detach().contiguous() for p in enc.planes_features_wavelet_coefs]


@pytest.mark.parametrize("kw,side", [(dict(max_res=16), 16), (dict(max_res=32), 32), (dict(max_res=7), 8), (dict(max_scale=2), 16),
                                     (dict(max_scale=4), 32), (dict(max_res=32, max_scale=2), 16), (dict(max_res=1000), 64)])
def test_coarser_readings_match_oracle(emu, kw, side):
    enc = _ours()
    pf, coefs = _params(enc)
    want, _ = ow.build_planes_limited(pf, coefs, **kw)
    got = enc.get_planes(**kw)
    assert tuple(got.shape) == tuple(want.shape) == (3, 8, side, side) and rel_l2(got, want) <= 1e-5
    # the result is cached like any other reading: the next query returns it whatever its arguments (:409-410)
    assert enc.get_planes() is got and enc.get_planes(max_res=8) is got
    enc.reset_cahce()
    full = enc.get_planes()
    assert rel_l2(full, ow.build_planes(pf, coefs)) <= 1e-5
    # gradient reaches only the levels that were applied
    enc.reset_cahce()
    enc.get_planes(**kw).square().sum().backward()
    pfo = pf.clone().requires_grad_(True)
    co = [c.clone().requires_grad_(True) for c in coefs]
    ow.build_planes_limited(pfo, co, **kw)[0].square().sum().backward()
    assert rel_l2(enc.planes_features.grad, pfo.grad) <= 1e-5
    for p, c in zip(enc.planes_features_wavelet_coefs, co):
        if c.grad is None:
            assert p.grad is None
        else:
            assert rel_l2(p.grad, c.grad) <= 1e-5


def test_all_resolutions_and_grid_features_match_oracle(emu):
    enc = _ours(1)
    pf, coefs = _params(enc)
    planes, want = ow.build_planes_limited(pf, coefs, get_all_resolutions=True)
    got = enc.get_planes(get_all_resolutions=True)
    assert [tuple(t.shape) for t in got] == [(3, 8, n, n) for n in (8, 16, 32, 64)]
    for a, b in zip(got, want):
        assert rel_l2(a, b) <= 1e-5
    assert enc.last_used_planes is got[-1]           # the cache holds the final planes, not the list (:415, :437-438)
    # the fused regulariser still works after a query that kept no |yh| sums
    lam = 0.2
    total = sum(c.numel() for c in coefs)
    want_reg = lam * sum(c.abs().mean() * (c.numel() / total) for c in coefs) / len(coefs)
    assert abs(float(enc.wavelet_l1(lam).detach()) - float(want_reg)) <= 1e-6 * float(want_reg)
    enc.reset_cahce()
    # stopped early, the list repeats its last entry (the reference appends inside the loop and again after it)
    got = enc.get_planes(max_res=16, get_all_resolutions=True)
    assert [t.shape[-1] for t in got] == [8, 16, 16] and got[1] is got[2]
    enc.reset_cahce()
    # get_grid_features: lattice of 5^3 points on the first reading whose side reaches 2 * 5 = 10, i.e. the 16^2 planes
    lb, feats, grid = enc.get_grid_features(5)
    limited, _ = ow.build_planes_limited(pf, coefs, max_res=10)
    assert limited.shape[-1] == 16
    axis = torch.arange(5)
    gx, gy, gz = torch.meshgrid(axis, axis, axis, indexing='xy')
    lattice = (2 * 1.5 * (torch.stack([gx, gy, gz], dim=-1) / 4) - 1.5)[..., [2, 0, 1]]
    want_f = of.sample_planes(limited, lattice.reshape(-1, 3), 1.5, recip_mul=False).view(5, 5, 5, 24)
    assert lb == 1.5 and torch.equal(grid, lattice) and tuple(feats.shape) == (5, 5, 5, 24)
    assert rel_l2(feats, want_f) <= 1e-5


def _reference_class(monkeypatch):
    """the reference's reconstruction TriPlaneVolume, loaded from its file under a private module name (the reference's package
    names must not stay in sys.modules: tests/test_reference_host_over_dropin.py binds them to the drop-in modules)"""
    pw = types.ModuleType("pytorch_wavelets")
    pw.DWTForward, pw.DWTInverse = ow.DWTForward, ow.DWTInverse
    monkeypatch.setitem(sys.modules, "pytorch_wavelets", pw)
    pkg = types.ModuleType("triplaneencoder")
    pkg.__path__ = [REF + "/triplaneencoder"]
    monkeypatch.setitem(sys.modules, "triplaneencoder", pkg)
    monkeypatch.delitem(sys.modules, "triplaneencoder.utils", raising=False)
    spec = importlib.util.spec_from_file_location("_ref_reconstruction_triplane_encoder", REF + "/triplaneencoder/triplane_encoder.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    monkeypatch.delitem(sys.modules, "triplaneencoder.utils", raising=False)
    return mod.TriPlaneVolume


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original project (TRINERFLET_REFERENCE)")
def test_queries_against_the_reference_module_live(emu, monkeypatch):
    Ref = _reference_class(monkeypatch)
    with contextlib.redirect_stdout(io.StringIO()):
        theirs = Ref(viewdir_plane_resolution=-1, apply_activation_on_features=False, inner_multi_res_scale_current=1,
                     learn_rotation_axis=False, dropout=0, wavelet_type="bior6.8", lbound_auto_scale=False, upscale_ratio_bound=-1,
                     upscale_levels=2, wavelet_base_resolution=0, **KW)
    ours = _ours(2)
    theirs.load_state_dict(ours.state_dict(), strict=True)
    pf, coefs = _params(ours)
    with torch.no_grad():
        for kw in (dict(max_res=16), dict(max_scale=4), dict(max_res=32, max_scale=2)):
            theirs.reset_cahce(); ours.reset_cahce()
            a, b = theirs.get_planes(**kw), ours.get_planes(**kw)
            assert torch.equal(a, ow.build_planes_limited(pf, coefs, **kw)[0])          # pins the restatement
            assert rel_l2(b, a) <= 1e-5
        theirs.reset_cahce(); ours.reset_cahce()
        la, lb = theirs.get_planes(get_all_resolutions=True), ours.get_planes(get_all_resolutions=True)
        assert len(la) == len(lb) == 4 and all(rel_l2(y, x) <= 1e-5 for x, y in zip(la, lb))
        theirs.reset_cahce(); ours.reset_cahce()
        la, lb = theirs.get_planes(max_scale=2, get_all_resolutions=True), ours.get_planes(max_scale=2, get_all_resolutions=True)
        assert [t.shape[-1] for t in la] == [t.shape[-1] for t in lb] == [8, 16, 16]
        theirs.reset_cahce(); ours.reset_cahce()
        ra, rb = theirs.get_grid_features(6), ours.get_grid_features(6)
        assert ra[0] == rb[0] and torch.equal(ra[2], rb[2]) and rel_l2(rb[1], ra[1]) <= 1e-5


def test_plane_cache_never_registers_a_parameter(emu):
    """without wavelet levels (or when a query stops before the first level) the planes ARE the base parameter; the cache must
    hold an alias -- assigning the Parameter itself to a module attribute registers it under the cache's name, after which the
    next ordinary assignment of a tensor raises (the reference module has exactly this trap)"""
    from trinerflet_b200.triplane_encoder import TriPlaneVolume
    plain = TriPlaneVolume(number_of_features=8, plane_resolution=16, inner_multi_res_scale=1)
    keys = list(plain.state_dict().keys())
    p = plain.get_planes()
    assert p.data_ptr() == plain.planes_features.data_ptr() and not isinstance(p, torch.nn.Parameter)
    p.sum().backward()
    assert plain.planes_features.grad is not None
    plain.reset_cahce()
    enc = _ours()
    enc.get_planes(max_res=8)                       # stops before the first level
    enc.reset_cahce()
    enc.get_planes()                                # a tensor is assignable again
    assert list(plain.state_dict().keys()) == keys and "encoder.last_used_planes" not in dict(enc.named_parameters())
    assert [n for n, _ in enc.named_parameters()] == ["planes_features"] + [f"planes_features_wavelet_coefs.{l}" for l in range(3)]
