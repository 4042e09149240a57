"""Mesh extraction from a trained field on the GPU: the reference's extract_fields / extract_geometry (torch-ngp nerf/utils.py,
called by Trainer.save_mesh) with the density sweep kept on the device and the marching cubes in CUDA (csrc/mesh.cu).

A user of the reference Trainer can rebind

    import nerf.utils, trinerflet_b200.mesh
    nerf.utils.extract_geometry = trinerflet_b200.mesh.extract_geometry

and save_mesh keeps working unchanged (same signature and return convention; export stays the host's code)."""
import numpy as np
import torch

from . import _lib
from ._lib import call, ptr, stream


def marching_cubes(volume, threshold):
    """mcubes.marching_cubes(volume, threshold) on the GPU.

    volume: a CUDA tensor or a numpy array [nx, ny, nz] (moved to the current device), read as float32; a point is inside iff
    its value >= threshold.  Returns (vertices [V, 3] float64 in index space, triangles [T, 3] int64) as numpy arrays, in the
    order csrc/mesh.cu documents: vertices by (linear index of the edge's lower lattice point, axis), triangles by (linear cube
    index, case-table order); triangle normals point from the inside region to the outside one.  The vertex positions follow
    mcubes' linear interpolation; the triangulation is this package's crack-free table, not mcubes'.
    Raises ValueError if the volume contains a NaN."""
    if isinstance(volume, np.ndarray):
        volume = torch.from_numpy(np.ascontiguousarray(volume, np.float32)).cuda()
    u = volume.detach().to(torch.float32).contiguous()
    if u.dim() != 3 or min(u.shape) < 2:
        raise ValueError(f"marching_cubes: expected a volume [nx, ny, nz] with at least 2 points per axis, got {tuple(u.shape)}")
    thr = float(threshold)
    if thr != thr:
        raise ValueError("marching_cubes: threshold is NaN")
    nx, ny, nz = u.shape
    ws = torch.empty(_lib.load().tnl_mc_workspace(nx, ny, nz), dtype=torch.uint8, device=u.device)
    totals = torch.empty(2, dtype=torch.int64, device=u.device)
    call("tnl_mc_count", ptr(u), nx, ny, nz, thr, ptr(ws), ws.numel(), ptr(totals), stream())
    n_v, n_t = (int(v) for v in totals.cpu())             # the one device-to-host read before the outputs exist
    if n_v < 0:
        raise ValueError("marching_cubes: the volume contains NaN")
    vertices = torch.empty(n_v, 3, dtype=torch.float64, device=u.device)
    triangles = torch.empty(n_t, 3, dtype=torch.int64, device=u.device)
    call("tnl_mc_emit", ptr(u), nx, ny, nz, thr, ptr(ws), ws.numel(), n_v, n_t, ptr(vertices) if n_v else None,
         ptr(triangles) if n_t else None, stream())
    return vertices.cpu().numpy(), triangles.cpu().numpy()


def extract_fields(bound_min, bound_max, resolution, query_func, S=128):
    """The reference's extract_fields with the volume on the device: the same linspace / split / meshgrid('ij') positions,
    query_func(pts [n, 3]) per chunk of S^3 points, each chunk's values written into a float32 volume [resolution]^3 on the
    device query_func returns them on, without a synchronisation.  Returns that tensor (the reference returns a numpy array).
    The points are built on bound_min's device (the reference's Trainer passes its aabb_infer, which lives on the model's)."""
    dev = bound_min.device if isinstance(bound_min, torch.Tensor) else torch.device("cpu")
    # linspace on the host as in the reference (bit-identical positions), copied to the points' device once
    X = torch.linspace(bound_min[0], bound_max[0], resolution).to(dev).split(S)
    Y = torch.linspace(bound_min[1], bound_max[1], resolution).to(dev).split(S)
    Z = torch.linspace(bound_min[2], bound_max[2], resolution).to(dev).split(S)
    u = None
    with torch.no_grad():
        for xi, xs in enumerate(X):
            for yi, ys in enumerate(Y):
                for zi, zs in enumerate(Z):
                    xx, yy, zz = torch.meshgrid(xs, ys, zs, indexing="ij")
                    pts = torch.cat([xx.reshape(-1, 1), yy.reshape(-1, 1), zz.reshape(-1, 1)], dim=-1)
                    val = query_func(pts).reshape(len(xs), len(ys), len(zs)).detach()
                    if u is None:
                        u = torch.empty(resolution, resolution, resolution, dtype=torch.float32, device=val.device)
                    u[xi * S: xi * S + len(xs), yi * S: yi * S + len(ys), zi * S: zi * S + len(zs)] = val
    return u


def _host(b):
    return b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, np.float32)


def extract_geometry(bound_min, bound_max, resolution, threshold, query_func):
    """The reference's extract_geometry: sweep, marching cubes, then the float64 world transform on the host.
    Returns (vertices [V, 3] float64 in world space, triangles [T, 3] int64) as numpy arrays."""
    u = extract_fields(bound_min, bound_max, resolution, query_func)
    vertices, triangles = marching_cubes(u, threshold)
    b_max_np, b_min_np = _host(bound_max), _host(bound_min)
    vertices = vertices / (resolution - 1.0) * (b_max_np - b_min_np)[None, :] + b_min_np[None, :]
    return vertices, triangles
