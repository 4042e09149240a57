"""GPU: gradients of the field with respect to its inputs (positions x, view directions d) through NeRFNetwork, density(),
TriPlaneVolume and SHEncoder, against torch.autograd.grad of the reference's literal op sequence (tests/field_truth.py) run
under the same precision: real CUDA fp16 autocast (rel-L2 <= 1e-2) or fp32 (rel-L2 <= 1e-4)."""
import pytest
import torch

from tests import field_truth as ft
from tests.util import rel_l2

pytestmark = pytest.mark.gpu

BOUND = 1.5


def _net(C, hidden, R=128, S=2, wave="bior6.8"):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    net = NeRFNetwork(bound=BOUND, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=C, triplane_resolution=R,
                      triplane_wavelet_levels=S, hidden_dim=hidden, hidden_dim_color=hidden, wavelet_type=wave).cuda()
    scene.init_model_(net, seed=C + hidden)
    return net


def _inputs(M, seed, n_tail=0):
    g = torch.Generator().manual_seed(seed)
    x = ((torch.rand(M, 3, generator=g) * 2 - 1) * BOUND * 0.95).cuda()
    d = torch.randn(M, 3, generator=g)
    d = (d / d.norm(dim=-1, keepdim=True)).cuda()
    gs, grgb = (torch.randn(M, generator=g) * 64.0).cuda(), (torch.randn(M, 3, generator=g) * 64.0).cuda()
    nv = torch.tensor([M - n_tail], dtype=torch.int32, device="cuda") if n_tail else None
    return x, d, gs, grgb, nv


def _net_grads(net, x, d, gs, grgb, nv=None, autocast=True):
    x = x.clone().requires_grad_(True)
    d = d.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        sigma, rgb = net(x, d, n_valid=nv)
        assert type(sigma.grad_fn).__name__ != "_FieldBackward"
        return torch.autograd.grad((sigma, rgb), (x, d), (gs, grgb))


def _truth(net, x, d, gs, grgb, autocast=True):
    planes = net.encoder.get_planes().detach()
    W = [w.detach() for w in net._weights()]
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        return ft.input_grads(planes, x, d, W, BOUND, gs, grgb)


@pytest.mark.parametrize("C,hidden", [(16, 64), (32, 64), (48, 64), (16, 128), (32, 128), (48, 128)])
@pytest.mark.parametrize("M,n_tail", [(5000, 0), (5000, 123), ((1 << 18) + 4321, 1000)])
def test_network_input_grads_fp16_autocast(C, hidden, M, n_tail):
    """fused kernels (the position gradient of the gather, the direction gradient from the MLP backward's epilogue) against the
    literal graph under real autocast; M above spatial_sort_min_points visits the samples in cell order; tail rows get zero"""
    net = _net(C, hidden)
    assert (M >= net.spatial_sort_min_points) == (M > 5000)
    x, d, gs, grgb, nv = _inputs(M, seed=C + hidden + M, n_tail=n_tail)
    gx, gd = _net_grads(net, x, d, gs, grgb, nv)
    V = M - n_tail
    tx, td = _truth(net, x[:V], d[:V], gs[:V], grgb[:V])
    assert rel_l2(gx[:V], tx) <= 1e-2, rel_l2(gx[:V], tx)
    assert rel_l2(gd[:V], td) <= 1e-2, rel_l2(gd[:V], td)
    if n_tail:
        assert (gx[V:] == 0).all() and (gd[V:] == 0).all()


@pytest.mark.parametrize("C,hidden", [(16, 64), (48, 128)])
def test_network_input_grads_fp32(C, hidden):
    """library path (no autocast): the gather's position gradient and SHEncoder's backward inside torch's graph"""
    net = _net(C, hidden)
    x, d, gs, grgb, _ = _inputs(4000, seed=C)
    gx, gd = _net_grads(net, x, d, gs, grgb, autocast=False)
    tx, td = _truth(net, x, d, gs, grgb, autocast=False)
    assert rel_l2(gx, tx) <= 1e-4 and rel_l2(gd, td) <= 1e-4, (rel_l2(gx, tx), rel_l2(gd, td))


@pytest.mark.parametrize("autocast", [True, False])
def test_density_position_gradient(autocast):
    net = _net(32, 64)
    x, _, gs, _, _ = _inputs(3000, seed=5)
    xr = x.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        (gx,) = torch.autograd.grad(net.density(xr)["sigma"], xr, gs)
        x2 = x.clone().requires_grad_(True)
        sigma, _ = ft.density(net.encoder.get_planes().detach(), x2, [w.detach() for w in net._weights()], BOUND)
        (tx,) = torch.autograd.grad(sigma, x2, gs)
    assert rel_l2(gx, tx) <= (1e-2 if autocast else 1e-4), rel_l2(gx, tx)


@pytest.mark.parametrize("wave", ["bior6.8", "bior4.4", "bior2.6", "bior2.2", "haar"])
def test_triplane_volume_position_gradient(wave):
    """TriPlaneVolume.forward alone, planes reconstructed with each wavelet: the position gradient against the literal gather, and
    the parameter gradients the same whether or not the positions require grad"""
    net = _net(16, 64, wave=wave)
    enc = net.encoder
    x, _, _, _, _ = _inputs(6000, seed=9)
    G = torch.randn(6000, 48, generator=torch.Generator().manual_seed(1)).cuda()
    grads = []
    for with_x in (True, False):
        enc.reset_cache()
        for p in enc.parameters():
            p.grad = None
        xr = x.clone().requires_grad_(with_x)
        feat = enc(xr, bound=BOUND)
        (feat * G).sum().backward()
        grads.append(([p.grad.clone() for p in enc.parameters()], xr.grad))
    (gp_x, gx), (gp, _) = grads
    for a, b in zip(gp_x, gp):
        assert rel_l2(a, b) <= 1e-5
    x2 = x.clone().requires_grad_(True)
    (tx,) = torch.autograd.grad(ft.sample(enc.get_planes().detach(), x2, BOUND), x2, G)
    assert rel_l2(gx, tx) <= 1e-4, rel_l2(gx, tx)


@pytest.mark.parametrize("degree", [1, 2, 3, 4])
def test_sh_encoder_backward(degree):
    from oracle import field as of
    from trinerflet_b200.shencoder import SHEncoder
    g = torch.Generator().manual_seed(degree)
    d = torch.randn(5000, 3, generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    grad = torch.randn(5000, degree ** 2, generator=g)
    dc = d.cuda().requires_grad_(True)
    (gd,) = torch.autograd.grad(SHEncoder(3, degree)(dc), dc, grad.cuda())
    dd = d.double().requires_grad_(True)
    (want,) = torch.autograd.grad(of.sh16(dd)[:, :degree ** 2], dd, grad.double())
    assert rel_l2(gd, want) <= 1e-6, rel_l2(gd, want)
    from oracle import build_ref
    ref = build_ref.load_ref("shencoder")
    if ref is None:
        pytest.skip("the reference's shencoder extension is not built")
    o_r = torch.empty(5000, degree ** 2, device="cuda")
    dy_dx = torch.empty(5000, 3 * degree ** 2, device="cuda")
    ref.sh_encode_forward(d.cuda(), o_r, 5000, 3, degree, dy_dx)
    g_r = torch.zeros(5000, 3, device="cuda")
    ref.sh_encode_backward(grad.cuda(), d.cuda(), 5000, 3, degree, dy_dx, g_r)
    assert (g_r - gd).abs().max().item() <= 1e-6 * max(1.0, g_r.abs().max().item())


def test_training_forward_still_dispatches_to_fused_field():
    """positions and directions without grad: the training step's one fused MLP backward with plane scatter (_Field); with either
    requiring grad: the gather and MLP autograd functions that return input gradients"""
    net = _net(32, 64)
    M = net.spatial_sort_min_points + 1000
    x, d, gs, grgb, _ = _inputs(M, seed=3)
    with torch.autocast("cuda", dtype=torch.float16):
        sigma, _ = net(x, d)
        assert type(sigma.grad_fn).__name__ == "_FieldBackward"
        for xr, dr in ((True, False), (False, True)):
            sigma, _ = net(x.clone().requires_grad_(xr), d.clone().requires_grad_(dr))
            assert type(sigma.grad_fn).__name__ == "_FieldMLPBackward"
