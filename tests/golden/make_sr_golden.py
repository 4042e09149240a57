"""Generates tests/golden/sr_encoder_fp32.npz by importing the REFERENCE's own super_resolution encoder module from
/root/reference (read-only) and running it on CPU in fp32.  Run in the build container only; the GPU box has no
/root/reference, so the resulting small fixture is committed.

    python tests/golden/make_sr_golden.py

Real: super_resolution/threestudio/models/triplaneencoder/triplane_encoder.py (TriPlaneVolume, KPlaneVolume,
MultiscaleKPlaneVolume, MultiscaleKPlaneMulVolume) with its own utils.py / grid_backward.py.  Substituted: pytorch_wavelets
(absent, no network) -> oracle/wavelet.py, as in make_golden.py; the `threestudio` package __init__ files (they import
lightning, diffusers ...) are bypassed by registering bare namespace modules whose __path__ points at the real directories.
"""
import contextlib
import importlib
import io
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import reference_path, require_reference  # noqa: E402

REF = reference_path("super_resolution", "threestudio")
OUT = os.path.join(HERE, "sr_encoder_fp32.npz")

# one parameter set (C = 8 -- the IDWT kernels take multiples of 8 --, R = 32, two wavelet levels: sides 8 -> 16 -> 32), three pairs of (low_res_scale, high_res_scale):
#   (2, 1): low reading after one level, high reading after both          (the shape of the reference's configs)
#   (4, 2): low reading = the base planes themselves, high reading stops one level early
#   (1, 1): both readings are the full reconstruction
WAVELET = dict(number_of_features=8, plane_resolution=32, inner_multi_res_scale=4, wavelet_type="bior6.8")
SCALES = [(2, 1), (4, 2), (1, 1)]
KPLANES = dict(base_resolution=8, levels=2, channels=4)
MULTISCALE = dict(base_resolution=4, low_res_levels=1, high_res_levels=3, channels=4)


def reference_available():
    return os.path.isdir(REF)


def load_reference_module():
    """-> the reference module threestudio.models.triplaneencoder.triplane_encoder, imported from /root/reference."""
    require_reference(REF)
    from oracle import wavelet as ow
    if "pytorch_wavelets" not in sys.modules:
        pw = types.ModuleType("pytorch_wavelets")
        pw.DWTForward, pw.DWTInverse = ow.DWTForward, ow.DWTInverse
        sys.modules["pytorch_wavelets"] = pw
    for name, path in [("threestudio", REF), ("threestudio.models", REF + "/models"),
                       ("threestudio.models.triplaneencoder", REF + "/models/triplaneencoder")]:
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [path]
            sys.modules[name] = m
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")        # pkg_resources deprecation notice of grid_backward.py
        return importlib.import_module("threestudio.models.triplaneencoder.triplane_encoder")


def quiet(fn, *a, **k):
    """the reference constructors print their level shapes"""
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def test_points(n, gen):
    """unit-cube positions: interior, a few outside the cube (border clamp), and some exactly on faces / corners"""
    x = torch.rand(n, 3, generator=gen)
    x[: n // 8] = x[: n // 8] * 1.4 - 0.2
    x[n // 8] = torch.tensor([0.0, 0.5, 1.0])
    x[n // 8 + 1] = torch.tensor([1.0, 1.0, 1.0])
    x[n // 8 + 2] = torch.tensor([0.0, 0.0, 0.0])
    x[n // 8 + 3] = torch.tensor([0.5, 0.5, 0.5])
    return x


def randomise_(module, gen, scale=0.3):
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(scale * torch.randn(p.shape, generator=gen))


def two_render_step(enc, x, w_low, w_high):
    """what one training step of the application does with the encoder (threestudio/systems/triplane_wavelet_sr.py:364-476):
    cache on, double mode, a low-resolution and a high-resolution render from the same cached planes, one backward.
    -> (feat_low, feat_high, {param name: grad}, d loss / d x)"""
    enc.enable_cache = True
    enc.reset_cahce()
    enc.set_double_mode(True)
    enc.set_resolution_mode('low_res')
    enc.get_planes()
    x = x.clone().requires_grad_(True)
    f_low = enc(x)
    enc.set_resolution_mode('high_res')
    f_high = enc(x)
    enc.set_resolution_mode('low_res')
    loss = (f_low * w_low).sum() + (f_high * w_high).sum()
    for p in enc.parameters():
        p.grad = None
    loss.backward()
    # a level neither reading reaches gets no gradient (None); stored as zeros
    grads = {n: (torch.zeros_like(p) if p.grad is None else p.grad.detach().clone()) for n, p in enc.named_parameters()}
    enc.reset_cahce()
    return f_low.detach(), f_high.detach(), grads, x.grad.detach()


def main():
    ref = load_reference_module()
    gen = torch.Generator().manual_seed(1234)
    out = {}
    x = test_points(160, gen)
    out["x"] = x.numpy()
    C = WAVELET["number_of_features"]
    w_low = torch.randn(160, 3 * C, generator=gen)
    w_high = torch.randn(160, 3 * C, generator=gen)
    out["w_low"], out["w_high"] = w_low.numpy(), w_high.numpy()
    state = None
    for lo, hi in SCALES:
        enc = quiet(ref.TriPlaneVolume, low_res_scale=lo, high_res_scale=hi, **WAVELET)
        if state is None:
            randomise_(enc, gen)
            state = {k: v.clone() for k, v in enc.state_dict().items()}
            for k, v in state.items():
                out["wavelet/state/" + k] = v.numpy()
        else:
            enc.load_state_dict(state)
        tag = f"wavelet/{lo}_{hi}/"
        # single-resolution reading (double mode off): the loop stops at the low-resolution level
        enc.enable_cache = False
        enc.set_double_mode(False)
        with torch.no_grad():
            out[tag + "planes_single_shape"] = np.array(enc.get_planes().shape)     # (the values equal planes_low)
            out[tag + "feat_single"] = enc(x).numpy()
        f_low, f_high, grads, gx = two_render_step(enc, x, w_low, w_high)
        enc.enable_cache = True
        enc.set_double_mode(True)
        with torch.no_grad():
            enc.set_resolution_mode('low_res')
            out[tag + "planes_low"] = enc.get_planes().numpy()
            enc.set_resolution_mode('high_res')
            out[tag + "planes_high"] = enc.get_planes().numpy()
        out[tag + "feat_low"], out[tag + "feat_high"], out[tag + "grad_x"] = f_low.numpy(), f_high.numpy(), gx.numpy()
        for k, g in grads.items():
            out[tag + "grad/" + k] = g.numpy()

    # plain-plane pyramids
    for mode in ("concatination", "mul"):
        kp = quiet(ref.KPlaneVolume, features_mode=mode, **KPLANES)
        randomise_(kp, gen, 0.7)
        tag = f"kplanes/{mode}/"
        for k, v in kp.state_dict().items():
            out[tag + "state/" + k] = v.numpy()
        xg = x.clone().requires_grad_(True)
        f = kp(xg)
        w = torch.randn(f.shape, generator=gen)
        (f * w).sum().backward()
        out[tag + "feat"], out[tag + "w"], out[tag + "grad_x"] = f.detach().numpy(), w.numpy(), xg.grad.numpy()
        for n, p in kp.named_parameters():
            out[tag + "grad/" + n] = p.grad.numpy()
    for name, cls in (("multiscale", ref.MultiscaleKPlaneVolume), ("multiscale_mul", ref.MultiscaleKPlaneMulVolume)):
        ms = quiet(cls, features_mode="concatination", **MULTISCALE)
        randomise_(ms, gen, 0.7)
        tag = name + "/"
        for k, v in ms.state_dict().items():
            out[tag + "state/" + k] = v.numpy()
        with torch.no_grad():
            out[tag + "feat_low"] = ms(x).numpy()
            ms.set_double_mode(True)
            ms.set_resolution_mode('high_res')
            out[tag + "feat_high"] = ms(x).numpy()
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT}: {len(out)} arrays, {os.path.getsize(OUT) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
