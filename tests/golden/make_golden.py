"""Generates tests/golden/*.npz by importing the REFERENCE's own Python modules from
/root/reference (read-only) and running them on CPU in fp32.  Run in the build container only;
the GPU box has no /root/reference, so the resulting small fixtures are committed.

    python tests/golden/make_golden.py

What is the real reference here and what is substituted (cannot be avoided in this container):
  * reconstruction/triplaneencoder/triplane_encoder.py::TriPlaneVolume   -- REAL (level loop, 2*x, pad 4,
    plane axes, grid_sample call, feature concat order)
  * reconstruction/nerf/network.py::NeRFNetwork, activation.py::trunc_exp, encoding.py::get_encoder -- REAL
  * pytorch_wavelets (absent, no network) -> oracle/wavelet.py restatement (so the IDWT arithmetic
    itself is "parity unpinned"; see oracle/wavelet.py header)
  * shencoder (CUDA-only extension) -> oracle/field.py::sh16 (restates shencoder.cu:50-68);
    pinned separately on the GPU box against the compiled reference kernel (oracle/_ref)
  * raymarching (CUDA-only) and UI/IO imports of nerf/utils.py (trimesh, cv2, lpips, ...) -> inert stubs
"""
import os
import sys
import types
import importlib
from unittest import mock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import reference_path, require_reference  # noqa: E402
from oracle import wavelet as ow  # noqa: E402
from oracle import field as of  # noqa: E402

REF = reference_path("reconstruction")


def _install_stubs():
    pw = types.ModuleType("pytorch_wavelets")
    pw.DWTForward, pw.DWTInverse = ow.DWTForward, ow.DWTInverse
    sys.modules["pytorch_wavelets"] = pw

    sh = types.ModuleType("shencoder")

    class SHEncoder(torch.nn.Module):
        def __init__(self, input_dim=3, degree=4):
            super().__init__()
            assert degree == 4
            self.output_dim = 16

        def forward(self, inputs, size=1):
            return of.sh16(inputs / size)

    sh.SHEncoder = SHEncoder
    sys.modules["shencoder"] = sh
    sys.modules["raymarching"] = mock.MagicMock()
    for name in ["trimesh", "cv2", "tensorboardX", "mcubes", "lpips", "torch_ema", "torchmetrics",
                 "torchmetrics.functional", "imageio", "torchvision", "matplotlib", "matplotlib.pyplot"]:
        try:
            importlib.import_module(name)
        except Exception:
            sys.modules[name] = mock.MagicMock()


def main():
    _install_stubs()
    sys.path.insert(0, require_reference(REF))
    from triplaneencoder.triplane_encoder import TriPlaneVolume
    from nerf.network import NeRFNetwork

    torch.manual_seed(1234)
    g = torch.Generator().manual_seed(1234)

    # ---------------- encoder: C=4, R=64, S=4 (base 16, 2 levels) ----------------
    C, R, S, bound = 4, 64, 4, 1.5
    enc = TriPlaneVolume(number_of_features=C, plane_resolution=R, init_sigma=0.1, lbound=bound,
                         viewdir_plane_resolution=-1, apply_activation_on_features=False,
                         inner_multi_res_scale=S, inner_multi_res_scale_current=1,
                         learn_rotation_axis=False, dropout=0, wavelet_type="bior6.8",
                         lbound_auto_scale=False, upscale_ratio_bound=-1, upscale_levels=2,
                         wavelet_base_resolution=0)
    with torch.no_grad():
        for p in enc.planes_features_wavelet_coefs:
            p.copy_(0.05 * torch.randn(p.shape, generator=g))
    M = 257
    xyz = (torch.rand(M, 3, generator=g) * 2 - 1) * bound
    xyz[:8] = torch.tensor([[-1.5, -1.5, -1.5], [1.5, 1.5, 1.5], [0, 0, 0], [1.5, -1.5, 0.3],
                            [-1.4999, 1.4999, 0], [0.75, 0.75, 0.75], [1.5, 0, 0], [0, 0, -1.5]])
    wfeat = torch.randn(M, 3 * C, generator=g)
    planes = enc.get_planes()
    feat = enc(xyz, bound)
    (feat * wfeat).sum().backward()
    out = dict(C=C, R=R, S=S, bound=bound, xyz=xyz.numpy(), wfeat=wfeat.numpy(),
               planes_features=enc.planes_features.detach().numpy(),
               planes=planes.detach().numpy(), feat=feat.detach().numpy(),
               g_planes_features=enc.planes_features.grad.numpy())
    for i, p in enumerate(enc.planes_features_wavelet_coefs):
        out[f"coef{i}"] = p.detach().numpy()
        out[f"g_coef{i}"] = p.grad.numpy()
    np.savez_compressed(os.path.join(HERE, "encoder_fp32.npz"), **out)
    print("encoder_fp32.npz: planes", tuple(planes.shape), "feat", tuple(feat.shape))

    # ---------------- full field: NeRFNetwork.forward / .density ----------------
    net = NeRFNetwork(encoding="triplane_wavelet", bound=bound, cuda_ray=False, density_scale=1,
                      min_near=0.2, density_thresh=10, bg_radius=-1,
                      triplane_channels=C, triplane_resolution=R, triplane_wavelet_levels=S,
                      hidden_dim=64, hidden_dim_color=64, learn_rotation_axis=False, dropout=0,
                      wavelet_type="bior6.8", lbound_auto_scale=False, upscale_ratio_bound=-1,
                      upscale_levels=2, density_blob_scale=0, density_blob_std=0.5,
                      mlp_weight_decay=-1, wavelet_base_resolution=0, nerfacc_renderer=False)
    with torch.no_grad():
        for p in net.encoder.planes_features_wavelet_coefs:
            p.copy_(0.05 * torch.randn(p.shape, generator=g))
    dirs = torch.randn(M, 3, generator=g)
    dirs = dirs / dirs.norm(dim=-1, keepdim=True)
    wsig = torch.randn(M, generator=g)
    wrgb = torch.randn(M, 3, generator=g)
    sigma, color = net(xyz, dirs)
    dens = net.density(xyz)
    (sigma * wsig).sum().backward(retain_graph=True)
    (color * wrgb).sum().backward()
    out = dict(C=C, R=R, S=S, bound=bound, xyz=xyz.numpy(), dirs=dirs.numpy(), wsig=wsig.numpy(),
               wrgb=wrgb.numpy(), sigma=sigma.detach().numpy(), color=color.detach().numpy(),
               dens_sigma=dens["sigma"].detach().numpy(), dens_geo=dens["geo_feat"].detach().numpy(),
               planes_features=net.encoder.planes_features.detach().numpy(),
               g_planes_features=net.encoder.planes_features.grad.numpy())
    for i, p in enumerate(net.encoder.planes_features_wavelet_coefs):
        out[f"coef{i}"] = p.detach().numpy()
        out[f"g_coef{i}"] = p.grad.numpy()
    names = ["sigma_net.0", "sigma_net.1", "color_net.0", "color_net.1", "color_net.2"]
    sd = dict(net.named_parameters())
    for i, n in enumerate(names):
        out[f"W{i + 1}"] = sd[n + ".weight"].detach().numpy()
        out[f"g_W{i + 1}"] = sd[n + ".weight"].grad.numpy()
    out["state_dict_keys"] = np.array(sorted(net.state_dict().keys()))
    np.savez_compressed(os.path.join(HERE, "field_fp32.npz"), **out)
    print("field_fp32.npz: sigma", tuple(sigma.shape), "color", tuple(color.shape))
    print("state_dict keys:", sorted(net.state_dict().keys()))


if __name__ == "__main__":
    main()
