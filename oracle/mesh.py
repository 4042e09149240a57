"""TEST INFRASTRUCTURE ONLY (oracle) -- plain-numpy restatement of the marching cubes of trinerflet_b200/csrc/mesh.cu, the arbiter
of the exact comparisons: the same generated case table (parsed from csrc/mc_tables.cuh), the same float64 interpolation and the
same output order (vertices by (linear index of the edge's lower lattice point, axis), triangles by (linear cube index, table
order)).  Also the reference's extract_fields / world transform (torch-ngp nerf/utils.py) restated literally, with a .cpu()
per chunk.  Never imported by the product package."""
import os
import re

import numpy as np
import torch

TABLES = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "trinerflet_b200", "csrc", "mc_tables.cuh")


def load_tables(path=TABLES):
    """-> (edge_corner [12] int, tri_table [256, 16] int, -1 padded)"""
    src = open(path).read()

    def array(name):
        body = re.search(name + r"\[[^=]*=\s*\{(.*?)\};", src, re.S).group(1)
        return np.array([int(v) for v in re.findall(r"-?\d+", body)], np.int64)

    return array("kMcEdgeCorner"), array("kMcTriTable").reshape(256, 16)


def _inside(u, thr):
    return u.astype(np.float64) >= thr


def marching_cubes(u, threshold):
    """u [nx, ny, nz] float32 -> (vertices [V, 3] float64 index space, triangles [T, 3] int64)"""
    u = np.ascontiguousarray(u, np.float32)
    if np.isnan(u).any():
        raise ValueError("volume contains NaN")
    thr = float(threshold)
    nx, ny, nz = u.shape
    ins = _inside(u, thr)
    ud = u.astype(np.float64)
    # vertices: key = 3 * linear index of the lower point + axis, sorted
    keys, pos = [], []
    for a in range(3):
        lo = [slice(None)] * 3
        hi = [slice(None)] * 3
        lo[a] = slice(0, u.shape[a] - 1)
        hi[a] = slice(1, None)
        cross = ins[tuple(lo)] != ins[tuple(hi)]
        idx = np.nonzero(cross)
        ua, ub = ud[tuple(lo)][idx], ud[tuple(hi)][idx]
        with np.errstate(invalid="ignore", divide="ignore"):
            t = np.where(np.isinf(ua), 1.0, (thr - ua) / (ub - ua))
        p = np.stack(idx, -1).astype(np.float64)
        p[:, a] = p[:, a] + t
        lin = (idx[0].astype(np.int64) * ny + idx[1]) * nz + idx[2]
        keys.append(3 * lin + a)
        pos.append(p)
    keys = np.concatenate(keys)
    pos = np.concatenate(pos)
    order = np.argsort(keys, kind="stable")
    keys, vertices = keys[order], pos[order]
    # triangles: cubes in linear order, table rows in order
    edge_corner, table = load_tables()
    case = np.zeros((nx - 1, ny - 1, nz - 1), np.int64)
    for c in range(8):
        dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
        case |= ins[dx:nx - 1 + dx, dy:ny - 1 + dy, dz:nz - 1 + dz].astype(np.int64) << c
    cx, cy, cz = np.nonzero(case)
    cases = case[cx, cy, cz]
    cx, cy, cz = (np.asarray(v, np.int64) for v in (cx, cy, cz))
    rows = table[cases]                                           # [n, 16]
    valid = rows >= 0
    e = np.where(valid, rows, 0)
    c0 = edge_corner[e]
    lin = ((cx[:, None] + (c0 & 1)) * ny + cy[:, None] + ((c0 >> 1) & 1)) * nz + cz[:, None] + ((c0 >> 2) & 1)
    k = 3 * lin + e // 4
    vid = np.searchsorted(keys, k[valid])                         # row-major: cube order, then table order
    assert np.array_equal(keys[vid], k[valid])
    return vertices.reshape(-1, 3), vid.astype(np.int64).reshape(-1, 3)


def extract_fields(bound_min, bound_max, resolution, query_func, S=128):
    """the reference's extract_fields, with its per-chunk .cpu() into a host volume"""
    X = torch.linspace(bound_min[0], bound_max[0], resolution).split(S)
    Y = torch.linspace(bound_min[1], bound_max[1], resolution).split(S)
    Z = torch.linspace(bound_min[2], bound_max[2], resolution).split(S)
    u = np.zeros([resolution, resolution, resolution], dtype=np.float32)
    with torch.no_grad():
        for xi, xs in enumerate(X):
            for yi, ys in enumerate(Y):
                for zi, zs in enumerate(Z):
                    xx, yy, zz = torch.meshgrid(xs, ys, zs, indexing="ij")
                    pts = torch.cat([xx.reshape(-1, 1), yy.reshape(-1, 1), zz.reshape(-1, 1)], dim=-1)
                    val = query_func(pts).reshape(len(xs), len(ys), len(zs)).detach().cpu().numpy()
                    u[xi * S: xi * S + len(xs), yi * S: yi * S + len(ys), zi * S: zi * S + len(zs)] = val
    return u


def world_transform(vertices, bound_min, bound_max, resolution):
    """the reference's vertices / (resolution - 1) * (b_max - b_min) + b_min on the host"""
    b_max_np = bound_max.detach().cpu().numpy()
    b_min_np = bound_min.detach().cpu().numpy()
    return vertices / (resolution - 1.0) * (b_max_np - b_min_np)[None, :] + b_min_np[None, :]
