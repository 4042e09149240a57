"""CPU: the marching cubes of csrc/mesh.cu (host build of the product kernel source, tests/kemu_mesh.py) against the numpy restatement
oracle/mesh.py, bit for bit, plus properties of the surface that do not depend on the case table, and the generator of the
table (csrc/gen_mc_tables.py) against the checked-in csrc/mc_tables.cuh."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import mesh as om
from tests import kemu_mesh as kemu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "trinerflet_b200", "csrc")


def _gen():
    spec = importlib.util.spec_from_file_location("gen_mc_tables", os.path.join(CSRC, "gen_mc_tables.py"))
    g = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(g)
    return g


# ------------------------------------------------------------------------------------------ volumes (index space, float32)
def _grid(n):
    return np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing="ij")


def ball(n, r, c=None):
    x, y, z = _grid(n)
    c = (n - 1) / 2 + 0.137 if c is None else c
    return (r - np.sqrt((x - c) ** 2 + (y - c) ** 2 + (z - c) ** 2)).astype(np.float32)


def torus(n, R, r):
    x, y, z = _grid(n)
    c = (n - 1) / 2 + 0.21
    q = np.sqrt((x - c) ** 2 + (y - c) ** 2) - R
    return (r - np.sqrt(q ** 2 + (z - c) ** 2)).astype(np.float32)


def touching_balls(n, r):
    c = (n - 1) / 2 + 0.31
    x, y, z = _grid(n)
    d1 = np.sqrt((x - (c - r)) ** 2 + (y - c) ** 2 + (z - c) ** 2)
    d2 = np.sqrt((x - (c + r)) ** 2 + (y - c) ** 2 + (z - c) ** 2)
    return np.maximum(r - d1, r - d2).astype(np.float32)


def noise(n, seed=0):
    return np.random.default_rng(seed).standard_normal((n, n, n)).astype(np.float32)


# ------------------------------------------------------------------------------------------ host build of the kernels
def mc_emu(u, thr):
    u = np.ascontiguousarray(u, np.float32)
    nx, ny, nz = u.shape
    lib = kemu.lib()
    nbytes = lib.tnl_mc_workspace(nx, ny, nz)
    ws = np.zeros(nbytes, np.uint8)
    totals = np.zeros(2, np.int64)
    kemu.call("tnl_mc_count", u, nx, ny, nz, float(thr), ws, nbytes, totals, None)
    nv, nt = int(totals[0]), int(totals[1])
    if nv < 0:
        raise ValueError("NaN")
    v = np.full((nv, 3), np.nan)
    t = np.full((nt, 3), -7, np.int64)
    kemu.call("tnl_mc_emit", u, nx, ny, nz, float(thr), ws, nbytes, nv, nt, v if nv else None, t if nt else None, None)
    return v, t


def _assert_same(a, b):
    va, ta = a
    vb, tb = b
    assert va.shape == vb.shape and ta.shape == tb.shape
    assert np.array_equal(va.view(np.uint64), vb.view(np.uint64))          # bit for bit, signed zeros included
    assert np.array_equal(ta, tb)


# ------------------------------------------------------------------------------------------ table-independent properties
def _undirected_counts(t):
    """-> (directed edge keys, undirected keys, unique undirected keys, their counts); key = a * n + b"""
    e = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]]).astype(np.int64)
    n = int(t.max()) + 1 if len(t) else 1
    directed = e[:, 0] * n + e[:, 1]
    und = np.minimum(e[:, 0], e[:, 1]) * n + np.maximum(e[:, 0], e[:, 1])
    uniq, cnt = np.unique(und, return_counts=True)
    return directed, und, uniq, cnt, n


def assert_closed_oriented(t):
    directed, _, _, cnt, _ = _undirected_counts(t)
    assert (cnt == 2).all(), np.bincount(cnt)
    assert len(np.unique(directed)) == len(directed)     # no directed edge twice: the two uses run in opposite directions


def euler(v, t):
    _, _, uniq, _, _ = _undirected_counts(t)
    return len(v) - len(uniq) + len(t)


def signed_volume(v, t):
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0)


def assert_on_lattice_edges(v, shape):
    frac = v - np.floor(v)
    assert ((frac != 0).sum(1) <= 1).all()
    assert (v >= 0).all() and (v <= np.array(shape) - 1).all()


# ------------------------------------------------------------------------------------------ generator
def test_checked_in_table_is_the_generators_output():
    assert open(os.path.join(CSRC, "mc_tables.cuh")).read() == _gen().render()


def test_generated_cases_are_face_local_and_cover_every_crossing():
    g = _gen()
    rows = g.table()
    edge_corner, table = om.load_tables()
    assert edge_corner.tolist() == g.EDGE_CORNER
    n_amb = 0
    for case in range(256):
        inside = [(case >> c) & 1 for c in range(8)]
        crossing = {e for e in range(12) if inside[g.EDGE_CORNER[e]] != inside[g.EDGE_CORNER[e] + (1 << (e // 4))]}
        segs = g.oriented_segments(case)
        used = [e for lp in g.loops(case) for e in lp]
        assert sorted(used) == sorted(crossing)                                     # each crossing edge exactly once
        for a, b in segs:                                                          # every segment lies on a cube face
            assert g._FS[a] & g._FS[b]
        segset = {frozenset(s) for s in segs}
        tris = rows[case]
        flat = [e for tr in tris for e in tr]
        assert table[case].tolist() == flat + [-1] * (16 - len(flat))
        assert set(flat) == crossing
        for tr in tris:
            for i in range(3):
                a, b = tr[i], tr[(i + 1) % 3]
                if g._FS[a] & g._FS[b]:
                    assert frozenset((a, b)) in segset, (case, tr)
        n_amb += any(sorted(inside[c] for c in cyc) == [0, 0, 1, 1] and inside[cyc[0]] == inside[cyc[2]] for cyc, _ in g.FACES)
        assert len(tris) <= 5
    assert n_amb == 120


# ------------------------------------------------------------------------------------------ exact equality with the oracle
@pytest.mark.parametrize("name,u,thr,chi", [
    ("ball32", ball(32, 11.3), 0.0, 2),
    ("ball64", ball(64, 25.0), 0.0, 2),
    ("torus48", torus(48, 13.0, 5.5), 0.0, 0),
    ("touching_balls40", touching_balls(40, 9.0), 0.0, None),
])
def test_closed_surfaces_match_the_oracle_and_are_closed(name, u, thr, chi):
    got = mc_emu(u, thr)
    _assert_same(got, om.marching_cubes(u, thr))
    v, t = got
    assert len(t) > 0
    assert_closed_oriented(t)
    assert_on_lattice_edges(v, u.shape)
    if chi is not None:
        assert euler(v, t) == chi
    assert signed_volume(v, t) > 0
    if name == "ball64":
        exact = 4.0 / 3.0 * np.pi * 25.0 ** 3
        assert abs(signed_volume(v, t) / exact - 1) < 0.01


def test_random_noise_covers_every_case_and_matches_the_oracle():
    u = noise(24)
    ins = u >= 0.0
    case = np.zeros((23, 23, 23), np.int64)
    for c in range(8):
        dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
        case |= ins[dx:23 + dx, dy:23 + dy, dz:23 + dz].astype(np.int64) << c
    assert len(np.unique(case)) == 256
    got = mc_emu(u, 0.0)
    _assert_same(got, om.marching_cubes(u, 0.0))
    v, t = got
    assert_on_lattice_edges(v, u.shape)
    directed, _, uniq, cnt, n = _undirected_counts(t)
    # interior edges: two triangles, opposite directions; the others (one triangle) lie on an outer face of the lattice
    assert len(np.unique(directed)) == len(directed)
    assert set(np.unique(cnt).tolist()) <= {1, 2}
    hi = np.array(u.shape) - 1
    once = uniq[cnt == 1]
    a, b = v[once // n], v[once % n]
    on_face = ((a == b) & ((a == 0) | (a == hi))).any(1)
    assert once.size > 0 and on_face.all()


def test_lattice_values_equal_to_the_threshold():
    u = np.random.default_rng(3).integers(0, 3, (12, 13, 14)).astype(np.float32)
    got = mc_emu(u, 1.0)
    _assert_same(got, om.marching_cubes(u, 1.0))
    v, _ = got
    assert (v == np.floor(v)).any()                       # t = 0 at the points that equal the threshold


def test_infinite_values():
    u = ball(20, 6.0)
    u[10, 10, 10] = np.inf
    u[0, 0, 0] = -np.inf
    u[10, 10, 4] = np.inf
    got = mc_emu(u, 0.0)
    _assert_same(got, om.marching_cubes(u, 0.0))
    assert np.isfinite(got[0]).all()
    assert_on_lattice_edges(got[0], u.shape)


def test_non_cubic_shape_and_threshold_order():
    u = ball(17, 5.0)[:, :15, :11].copy()
    for thr in (-1.5, 0.0, 2.25):
        _assert_same(mc_emu(u, thr), om.marching_cubes(u, thr))


# ------------------------------------------------------------------------------------------ errors and edge cases
def test_nan_is_rejected():
    u = ball(10, 3.0)
    u[9, 9, 9] = np.nan                                   # a corner that takes part in no crossing edge
    lib = kemu.lib()
    nbytes = lib.tnl_mc_workspace(10, 10, 10)
    ws = np.zeros(nbytes, np.uint8)
    totals = np.zeros(2, np.int64)
    kemu.call("tnl_mc_count", u, 10, 10, 10, 0.0, ws, nbytes, totals, None)
    assert totals.tolist() == [-1, -1]
    assert lib.tnl_mc_emit(kemu.p(u), 10, 10, 10, 0.0, kemu.p(ws), nbytes, -1, -1, None, None, None) == -1
    assert b"NaN" in lib.tnl_last_error()
    with pytest.raises(ValueError):
        mc_emu(u, 0.0)
    with pytest.raises(ValueError):
        om.marching_cubes(u, 0.0)


def test_argument_errors():
    lib = kemu.lib()
    u = ball(4, 1.0)
    ws = np.zeros(lib.tnl_mc_workspace(4, 4, 4), np.uint8)
    totals = np.zeros(2, np.int64)
    P = kemu.p
    assert lib.tnl_mc_workspace(1, 4, 4) == 0
    assert lib.tnl_mc_count(None, 4, 4, 4, 0.0, P(ws), ws.size, P(totals), None) == -1
    assert lib.tnl_mc_count(P(u), 4, 4, 4, 0.0, None, ws.size, P(totals), None) == -1
    assert lib.tnl_mc_count(P(u), 4, 4, 4, 0.0, P(ws), ws.size, None, None) == -1
    for shape in ((1, 4, 4), (4, 1, 4), (4, 4, 1), (0, 4, 4)):
        assert lib.tnl_mc_count(P(u), *shape, 0.0, P(ws), ws.size, P(totals), None) == -1
        assert lib.tnl_mc_emit(P(u), *shape, 0.0, P(ws), ws.size, 0, 0, None, None, None) == -1
    assert lib.tnl_mc_count(P(u), 4, 4, 4, float("nan"), P(ws), ws.size, P(totals), None) == -1
    assert lib.tnl_mc_count(P(u), 4, 4, 4, 0.0, P(ws), ws.size - 1, P(totals), None) == -3     # TNL_ERR_WORKSPACE
    assert lib.tnl_mc_emit(None, 4, 4, 4, 0.0, P(ws), ws.size, 0, 0, None, None, None) == -1
    assert lib.tnl_mc_emit(P(u), 4, 4, 4, 0.0, P(ws), ws.size, 5, 2, None, None, None) == -1   # outputs missing


@pytest.mark.parametrize("fill", [-1.0, 1.0])
def test_empty_results(fill):
    u = np.full((5, 6, 7), fill, np.float32)
    v, t = mc_emu(u, 0.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)
    v, t = om.marching_cubes(u, 0.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)


def test_workspace_is_about_two_bytes_per_point():
    lib = kemu.lib()
    assert lib.tnl_mc_workspace(1024, 1024, 1024) == 2 * 1024 ** 3 + 24 * (1024 ** 3 // 2048)
    assert lib.tnl_mc_workspace(2, 2, 2) == 16 + 16 + 16


# ------------------------------------------------------------------------------------------ the package's host code
def test_python_api_on_the_host_build(monkeypatch):
    from tests import emu_backend
    from trinerflet_b200 import _lib, mesh
    emu_backend.install(monkeypatch)
    monkeypatch.setattr(_lib, "_lib", kemu.lib())              # the library with the mesh kernels
    u = torus(24, 6.0, 2.5)
    got = mesh.marching_cubes(u, 0.0)
    _assert_same(got, om.marching_cubes(u, 0.0))
    assert got[0].dtype == np.float64 and got[1].dtype == np.int64
    _assert_same(mesh.marching_cubes(torch.from_numpy(u), 0.0), got)
    v, t = mesh.marching_cubes(np.zeros((3, 3, 3), np.float32), 1.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)
    bad = u.copy()
    bad[3, 4, 5] = np.nan
    with pytest.raises(ValueError):
        mesh.marching_cubes(bad, 0.0)
    with pytest.raises(ValueError):
        mesh.marching_cubes(np.zeros((1, 3, 3), np.float32), 0.0)

    # extract_geometry over an analytic query_func: the reference's chunked sweep + the oracle + the world transform
    bmin, bmax = torch.tensor([-1.0, -0.9, -1.1]), torch.tensor([1.0, 1.2, 0.8])

    def query(p):
        return 0.7 - p.norm(dim=-1)

    res = 21
    u_ref = om.extract_fields(bmin, bmax, res, query, S=8)
    u_dev = mesh.extract_fields(bmin, bmax, res, query, S=8)
    assert np.array_equal(u_dev.numpy(), u_ref)
    v, t = mesh.extract_geometry(bmin, bmax, res, 0.0, query)
    vo, to = om.marching_cubes(om.extract_fields(bmin, bmax, res, query), 0.0)
    _assert_same((v, t), (om.world_transform(vo, bmin, bmax, res), to))
