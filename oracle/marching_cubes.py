"""numpy restatement of csrc/mesh.cu (xrd_mc_count / xrd_mc_emit), for the tests.

Same case tables (scripts/gen_mc_tables.py is imported, not copied), same inside rule
(value < level), same output order -- vertices by (volume, i, j, k, axis), faces by
(volume, cube, table order) -- and the same vertex formula:
    t = (level - v0) / (v1 - v0)                        fp32
    world_d = origin_d + (i_d + t * e_d) * spacing_d    fp64 (numpy never contracts to FMA),
                                                        stored as fp32.
"""
from __future__ import annotations

import importlib.util
import os

import numpy as np

_GEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'scripts',
                    'gen_mc_tables.py')


def load_generator():
    spec = importlib.util.spec_from_file_location('gen_mc_tables', _GEN)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_TABLES = None


def tables():
    global _TABLES
    if _TABLES is None:
        _TABLES = load_generator().tables()
    return _TABLES


def marching_cubes(field, level=0.0, origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0)):
    """field: [B, nx, ny, nz] (or [nx, ny, nz]) fp32; origin / spacing: [3] shared or [B, 3].
    -> (verts f32 [V,3], faces i32 [F,3])."""
    f = np.asarray(field, dtype=np.float32)
    if f.ndim == 3:
        f = f[None]
    B, nx, ny, nz = f.shape
    org = np.broadcast_to(np.asarray(origin, dtype=np.float64).reshape(-1, 3), (B, 3))
    spc = np.broadcast_to(np.asarray(spacing, dtype=np.float64).reshape(-1, 3), (B, 3))
    lv = np.float32(level)
    count, table = tables()
    ins = f < lv

    # crossing flags of the +x, +y, +z edge of every lattice point
    flags = np.zeros((B, nx, ny, nz), dtype=np.int64)
    flags[:, :-1] |= (ins[:, :-1] != ins[:, 1:]) * 1
    flags[:, :, :-1] |= (ins[:, :, :-1] != ins[:, :, 1:]) * 2
    flags[:, :, :, :-1] |= (ins[:, :, :, :-1] != ins[:, :, :, 1:]) * 4
    nv = ((flags & 1) > 0).astype(np.int64) + ((flags & 2) > 0) + ((flags & 4) > 0)
    voff = np.concatenate([[0], np.cumsum(nv.reshape(-1))[:-1]]).reshape(flags.shape)

    # vertices, point-major then axis
    verts = np.empty((int(nv.sum()), 3), dtype=np.float32)
    b, i, j, k = np.nonzero(flags)
    idx = np.stack([i, j, k], -1)
    for a in range(3):
        sel = (flags[b, i, j, k] >> a & 1) > 0
        bb, ii = b[sel], idx[sel]
        v0 = f[bb, ii[:, 0], ii[:, 1], ii[:, 2]]
        n1 = ii.copy()
        n1[:, a] += 1
        v1 = f[bb, n1[:, 0], n1[:, 1], n1[:, 2]]
        t = (lv - v0) / (v1 - v0)  # fp32
        pos = ii.astype(np.float64)
        pos[:, a] = pos[:, a] + t.astype(np.float64)
        w = (org[bb] + pos * spc[bb]).astype(np.float32)
        rank = np.zeros(len(bb), dtype=np.int64)
        for a2 in range(a):
            rank += (flags[bb, ii[:, 0], ii[:, 1], ii[:, 2]] >> a2) & 1
        verts[voff[bb, ii[:, 0], ii[:, 1], ii[:, 2]] + rank] = w

    # faces, cube-major then table order
    cs = np.zeros((B, nx - 1, ny - 1, nz - 1), dtype=np.int64)
    for n in range(8):
        dx, dy, dz = n & 1, (n >> 1) & 1, (n >> 2) & 1
        cs |= ins[:, dx:nx - 1 + dx, dy:ny - 1 + dy, dz:nz - 1 + dz].astype(np.int64) << n
    faces = []
    cb, ci, cj, ck = np.nonzero(count[cs])  # C order = (volume, i, j, k)
    for c in range(len(cb)):
        case = cs[cb[c], ci[c], cj[c], ck[c]]
        for e in table[case, :3 * count[case]]:
            a, b0, b1 = e >> 2, e & 1, (e >> 1) & 1
            off = [b0, b1]
            d = [0, 0, 0]
            others = [x for x in range(3) if x != a]
            d[others[0]], d[others[1]] = off
            p = (cb[c], ci[c] + d[0], cj[c] + d[1], ck[c] + d[2])
            fl = flags[p]
            faces.append(voff[p] + sum((fl >> a2) & 1 for a2 in range(a)))
    faces = np.asarray(faces, dtype=np.int32).reshape(-1, 3)
    return verts, faces
