"""Generate the marching-cubes case tables (xrdslam_b200/csrc/mc_tables.cuh).

Conventions shared by the kernel (csrc/mesh.cu) and the numpy oracle (oracle/marching_cubes.py):

* Cube corner n = dx | dy << 1 | dz << 2 sits at lattice point (i + dx, j + dy, k + dz).
  Case index bit n is set when that corner is inside (value < level).
* Cube edge e runs along axis a = e // 4 from the corner whose other two offsets are
  (b0, b1) = (e & 1, (e >> 1) & 1), in increasing axis order.  Its vertex is the crossing
  of the lattice edge (lower end point, axis a).
* For each case: cut every edge whose ends differ, join the cut points into closed polygons
  by walking the six cube faces, and fan-triangulate each polygon from its smallest edge id.
  On a face with two diagonal inside corners (an ambiguous face) each inside corner is cut
  off on its own: the two inside corners are kept apart.  The choice depends only on the
  four corner signs of that face, so two cubes sharing the face produce the same segments
  there and the mesh has no cracks.
* Winding: the right-hand normal (v1 - v0) x (v2 - v0) of every triangle points from the
  inside corners toward the outside ones, i.e. toward increasing field values.

Run `python scripts/gen_mc_tables.py` to rewrite the header; tests check that the committed
header equals what this script produces.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                      'xrdslam_b200', 'csrc', 'mc_tables.cuh')


def corner_pos(n):
    return np.array([n & 1, (n >> 1) & 1, (n >> 2) & 1], dtype=np.float64)


def edge_corners(e):
    """(lower corner, upper corner) of cube edge e."""
    a, b0, b1 = e // 4, e & 1, (e >> 1) & 1
    others = [d for d in range(3) if d != a]
    off = [0, 0, 0]
    off[others[0]], off[others[1]] = b0, b1
    lo = off[0] | off[1] << 1 | off[2] << 2
    return lo, lo | (1 << a)


EDGES = [edge_corners(e) for e in range(12)]
EDGE_ID = {frozenset(c): e for e, c in enumerate(EDGES)}


def faces():
    """The six faces: (outward normal, the four corners in cyclic order)."""
    out = []
    for a in range(3):
        u, v = [d for d in range(3) if d != a]
        for side in (0, 1):
            cyc = []
            for bu, bv in ((0, 0), (1, 0), (1, 1), (0, 1)):
                off = [0, 0, 0]
                off[a], off[u], off[v] = side, bu, bv
                cyc.append(off[0] | off[1] << 1 | off[2] << 2)
            n = np.zeros(3)
            n[a] = 1.0 if side else -1.0
            out.append((n, cyc))
    return out


FACES = faces()


def edge_mid(e):
    lo, hi = EDGES[e]
    return 0.5 * (corner_pos(lo) + corner_pos(hi))


def face_segments(case, normal, cyc):
    """Oriented segments (edge_from, edge_to) the surface leaves on one face."""
    inside = [bool(case >> c & 1) for c in cyc]
    cut = [EDGE_ID[frozenset((cyc[q], cyc[(q + 1) % 4]))] for q in range(4)
           if inside[q] != inside[(q + 1) % 4]]
    if not cut:
        return []
    if len(cut) == 4:  # ambiguous: cut off each inside corner on its own
        pairs = []
        for q in range(4):
            if inside[q]:
                ea = EDGE_ID[frozenset((cyc[q], cyc[(q + 1) % 4]))]
                eb = EDGE_ID[frozenset((cyc[q], cyc[(q + 3) % 4]))]
                pairs.append((ea, eb, corner_pos(cyc[q]), None))
    else:
        ins = [corner_pos(c) for c, i in zip(cyc, inside) if i]
        outs = [corner_pos(c) for c, i in zip(cyc, inside) if not i]
        pairs = [(cut[0], cut[1], np.mean(ins, 0), np.mean(outs, 0))]
    segs = []
    for ea, eb, pin, pout in pairs:
        a, b = edge_mid(ea), edge_mid(eb)
        # in-face direction from the inside corner(s) toward the outside ones
        d = (0.5 * (a + b) if pout is None else pout) - pin
        # orient so that normal x (b - a) points toward the outside corners
        if np.dot(np.cross(normal, b - a), d) < 0:
            ea, eb = eb, ea
        segs.append((ea, eb))
    return segs


def case_polygons(case):
    """Closed, oriented polygons of edge ids, each starting at its smallest edge id."""
    nxt = {}
    for normal, cyc in FACES:
        for ea, eb in face_segments(case, normal, cyc):
            assert ea not in nxt
            nxt[ea] = eb
    polys, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        poly, e = [], start
        while e not in seen:
            seen.add(e)
            poly.append(e)
            e = nxt[e]
        assert e == start
        polys.append(poly)
    return polys


def case_triangles(case):
    tris = []
    for poly in case_polygons(case):
        for q in range(1, len(poly) - 1):
            tris.append((poly[0], poly[q], poly[q + 1]))
    return tris


def tables():
    """-> (tri_count [256] int, tri_table [256][3 * max_tris] int, -1 padded)."""
    all_tris = [case_triangles(c) for c in range(256)]
    max_t = max(len(t) for t in all_tris)
    count = np.array([len(t) for t in all_tris], dtype=np.int32)
    table = np.full((256, 3 * max_t), -1, dtype=np.int32)
    for c, t in enumerate(all_tris):
        if t:
            table[c, :3 * len(t)] = np.array(t).reshape(-1)
    return count, table


def render_header():
    count, table = tables()
    max_t = table.shape[1] // 3
    lines = [
        '// Generated by scripts/gen_mc_tables.py -- do not edit.',
        '// Marching-cubes case tables: corner n = dx | dy << 1 | dz << 2, case bit n set when',
        '// the corner is inside (value < level); edge e runs along axis e / 4 from the corner',
        '// with the other two offsets (e & 1, (e >> 1) & 1).  See the script for the',
        '// polygon walk, the ambiguous-face rule and the winding.',
        '#pragma once',
        '',
        f'#define XRD_MC_MAX_TRIS {max_t}',
        '',
        'namespace xrd {',
        'namespace mc {',
        '',
        '__constant__ unsigned char c_tri_count[256] = {',
    ]
    for r in range(0, 256, 16):
        lines.append('    ' + ', '.join(str(int(v)) for v in count[r:r + 16]) + ',')
    lines += ['};', '', f'__constant__ signed char c_tri_table[256][{3 * max_t}] = {{']
    for c in range(256):
        lines.append('    {' + ', '.join(str(int(v)) for v in table[c]) + '},')
    lines += ['};', '', '}  // namespace mc', '}  // namespace xrd', '']
    return '\n'.join(lines)


if __name__ == '__main__':
    text = render_header()
    if '--check' in sys.argv:
        with open(HEADER) as f:
            sys.exit(0 if f.read() == text else 1)
    with open(HEADER, 'w') as f:
        f.write(text)
    print(HEADER)
