"""Generates mc_tables.cuh, the marching-cubes case table of csrc/mesh.cu (and of oracle/mesh.py, which parses the same file).

    python trinerflet_b200/csrc/gen_mc_tables.py            rewrite mc_tables.cuh next to this script
    python trinerflet_b200/csrc/gen_mc_tables.py --check    exit 1 if the checked-in file differs from the output

Construction (face-local, so two cubes that share a face always cut it the same way and the mesh has no cracks):
  * corners c = x + 2y + 4z; cube edge e = 4 * axis + k joins corner EDGE_CORNER[e] (its bit `axis` clear; k-th such corner in
    increasing order) to EDGE_CORNER[e] + (1 << axis).  A corner is inside iff u >= threshold; an edge crosses iff exactly one
    of its corners is inside.
  * each of the 6 faces with 2 crossing edges gives one segment between them; a face with 4 crossing edges (the ambiguous
    diagonal pattern) gives two segments, each cutting off one inside corner.  The rule reads only the face's four corners.
  * every crossing edge lies on two faces, so the segments chain into disjoint loops.  Each loop is oriented so that the normals
    (v1 - v0) x (v2 - v0) of its triangles point from the inside region to the outside one.
  * each loop is triangulated without a diagonal between two crossing points of a common face unless that pair is a segment
    (the neighbouring cube could draw that diagonal too, and the edge would then belong to four triangles).  Among the allowed
    triangulations the one found first by a recursion that prefers fans from the loop's lowest edge index is taken.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "mc_tables.cuh")


def corner_pos(c):
    return np.array([c & 1, (c >> 1) & 1, (c >> 2) & 1], np.float64)


EDGE_CORNER = [c for a in range(3) for c in range(8) if not (c >> a) & 1]
EDGE_AXIS = [e // 4 for e in range(12)]


def edge_of(c0, c1):
    lo, hi = min(c0, c1), max(c0, c1)
    a = (hi ^ lo).bit_length() - 1
    return 4 * a + [c for c in range(8) if not (c >> a) & 1].index(lo)


def edge_mid(e):
    p = corner_pos(EDGE_CORNER[e])
    p[EDGE_AXIS[e]] = 0.5
    return p


# faces (axis, side): corners in cyclic order around the face, outward normal
FACES = []
for a in range(3):
    b, c = [x for x in range(3) if x != a]
    for side in (0, 1):
        base = side << a
        cyc = [base, base | (1 << b), base | (1 << b) | (1 << c), base | (1 << c)]
        n = np.zeros(3)
        n[a] = 1.0 if side else -1.0
        FACES.append((cyc, n))


def face_segments(case):
    """-> list of (edge_a, edge_b, N): N points, within the face, from the segment's inside side to its outside side"""
    segs = []
    for cyc, n in FACES:
        ins = [(case >> c) & 1 for c in cyc]
        cross = [edge_of(cyc[i], cyc[(i + 1) % 4]) for i in range(4) if ins[i] != ins[(i + 1) % 4]]
        if len(cross) == 2:
            pin = [corner_pos(c) for c, i in zip(cyc, ins) if i]
            pout = [corner_pos(c) for c, i in zip(cyc, ins) if not i]
            segs.append((cross[0], cross[1], np.mean(pout, 0) - np.mean(pin, 0), n))
        elif len(cross) == 4:
            for i in range(4):
                if ins[i]:
                    ea, eb = edge_of(cyc[i], cyc[(i - 1) % 4]), edge_of(cyc[i], cyc[(i + 1) % 4])
                    m = 0.5 * (edge_mid(ea) + edge_mid(eb))
                    segs.append((ea, eb, m - corner_pos(cyc[i]), n))
    return segs


def oriented_segments(case):
    """segments as directed pairs (a -> b): walking a -> b, the surface normal N, the face normal n and the walk satisfy
    d = N x n (the boundary of a patch inside the cube, traversed counter-clockwise seen from N's tip)"""
    out = []
    for ea, eb, N, n in face_segments(case):
        d = np.cross(N, n)
        s = float(np.dot(edge_mid(eb) - edge_mid(ea), d))
        assert abs(s) > 1e-9, (case, ea, eb)
        out.append((ea, eb) if s > 0 else (eb, ea))
    return out


def loops(case):
    nxt = {}
    for a, b in oriented_segments(case):
        assert a not in nxt, ("edge leaves twice", case, a)
        nxt[a] = b
    assert sorted(nxt) == sorted(nxt.values()), ("open chain", case)
    out, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        loop, e = [], start
        while e not in seen:
            seen.add(e)
            loop.append(e)
            e = nxt[e]
        out.append(loop)          # starts at the loop's lowest edge index
    return out


def face_sets():
    """edge -> set of the two faces it lies on"""
    fs = {e: set() for e in range(12)}
    for f, (cyc, _) in enumerate(FACES):
        for i in range(4):
            fs[edge_of(cyc[i], cyc[(i + 1) % 4])].add(f)
    return fs


_FS = face_sets()


def triangulate(loop, segs):
    L = len(loop)

    def allowed(i, j):
        if (j - i) % L in (1, L - 1):
            return True
        a, b = loop[i], loop[j]
        return not (_FS[a] & _FS[b]) or (a, b) in segs or (b, a) in segs

    memo = {}

    def tri(i, j):                # triangulation of loop[i..j] closed by the chord (i, j), or None
        if j - i < 2:
            return []
        if (i, j) in memo:
            return memo[(i, j)]
        res = None
        for k in range(j - 1, i, -1):        # k = j-1 first: fans from loop[i]
            if allowed(i, k) and allowed(k, j):
                left, right = tri(i, k), tri(k, j)
                if left is not None and right is not None:
                    res = left + right + [(loop[i], loop[k], loop[j])]
                    break
        memo[(i, j)] = res
        return res

    t = tri(0, L - 1)
    assert t is not None, ("no admissible triangulation", loop)
    return t


def table():
    rows = []
    for case in range(256):
        segs = set(oriented_segments(case))
        tris = []
        for loop in loops(case):
            tris += triangulate(loop, segs)
        rows.append(tris)
    return rows


def render():
    rows = table()
    lines = ["// GENERATED by trinerflet_b200/csrc/gen_mc_tables.py -- do not edit; see that script for the construction.",
             "// Corners c = x + 2y + 4z.  Cube edge e runs from corner kMcEdgeCorner[e] along axis e / 4 (x, y, z).",
             "// kMcTriTable[case][3 * i + k] = cube edge of vertex k of triangle i, -1 terminated; case bit c = (u[corner c] >= threshold).",
             "#pragma once", "#include <stdint.h>", "", "namespace tnl {", "",
             f"constexpr int kMcMaxTris = {max(len(r) for r in rows)};",
             "__device__ const uint8_t kMcEdgeCorner[12] = {" + ", ".join(str(c) for c in EDGE_CORNER) + "};",
             "__device__ const uint8_t kMcTriCount[256] = {"]
    for i in range(0, 256, 32):
        lines.append("    " + ", ".join(str(len(r)) for r in rows[i:i + 32]) + ",")
    lines.append("};")
    lines.append("__device__ const int8_t kMcTriTable[256][16] = {")
    for case, r in enumerate(rows):
        flat = [e for tr in r for e in tr]
        flat += [-1] * (16 - len(flat))
        lines.append("    {" + ", ".join(str(e) for e in flat) + "},")
    lines += ["};", "", "}  // namespace tnl", ""]
    return "\n".join(lines)


if __name__ == "__main__":
    text = render()
    if "--check" in sys.argv:
        same = os.path.exists(OUT) and open(OUT).read() == text
        print("mc_tables.cuh is " + ("up to date" if same else "STALE"))
        sys.exit(0 if same else 1)
    with open(OUT, "w") as f:
        f.write(text)
