"""Marching-cubes tables, the numpy oracle (oracle/marching_cubes.py) on analytic fields, and the
host logic of the mesher (xrdslam_b200/mesher.py) -- no GPU needed."""
import itertools
import os

import numpy as np
import pytest
import torch

from oracle.marching_cubes import load_generator, marching_cubes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gen = load_generator()


# ---- tables --------------------------------------------------------------------------------
def test_committed_header_matches_generator():
    with open(os.path.join(ROOT, 'xrdslam_b200', 'csrc', 'mc_tables.cuh')) as f:
        assert f.read() == gen.render_header()


def _face_of_edges(ea, eb):
    """Faces (index into gen.FACES) containing both cube edges."""
    out = []
    for fi, (_, cyc) in enumerate(gen.FACES):
        fe = {gen.EDGE_ID[frozenset((cyc[q], cyc[(q + 1) % 4]))] for q in range(4)}
        if ea in fe and eb in fe:
            out.append(fi)
    return out


def _boundary_edges(tris):
    """Directed triangle edges whose undirected edge is used once in the case."""
    cnt = {}
    for t in tris:
        for a, b in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])):
            cnt[frozenset((a, b))] = cnt.get(frozenset((a, b)), 0) + 1
    return [(a, b) for t in tris for a, b in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0]))
            if cnt[frozenset((a, b))] == 1]


def test_boundary_edges_lie_on_cube_faces():
    for case in range(256):
        tris = gen.case_triangles(case)
        for a, b in _boundary_edges(tris):
            assert _face_of_edges(a, b), (case, a, b)
        # every cut edge is a vertex of exactly one polygon
        cut = {e for e, (lo, hi) in enumerate(gen.EDGES) if (case >> lo & 1) != (case >> hi & 1)}
        used = [e for p in gen.case_polygons(case) for e in p]
        assert sorted(used) == sorted(cut)


def _edge_world(e, shift):
    lo, hi = gen.EDGES[e]
    return (tuple(gen.corner_pos(lo) + shift), tuple(gen.corner_pos(hi) + shift))


def _face_segments_world(case, axis, side, shift):
    """Boundary segments the case leaves on one cube face, as directed pairs of world edges."""
    fi = 2 * axis + side
    segs = set()
    for a, b in _boundary_edges(gen.case_triangles(case)):
        if fi in _face_of_edges(a, b):
            segs.add((_edge_world(a, shift), _edge_world(b, shift)))
    return segs


@pytest.mark.parametrize('axis', [0, 1, 2])
def test_shared_faces_produce_matching_segments(axis):
    """Every sign assignment of two cubes sharing a face: the segments both leave on that face
    are the same, with opposite direction (consistent orientation across cubes)."""
    shift = np.zeros(3)
    shift[axis] = 1.0
    lower_face = [n for n in range(8) if n >> axis & 1]      # side 1 of the lower cube
    upper_face = [n ^ (1 << axis) for n in lower_face]       # the same points, side 0 above
    free_lo = [n for n in range(8) if not n >> axis & 1]
    free_up = [n for n in range(8) if n >> axis & 1]
    for fbits in range(16):
        for lbits, ubits in itertools.product(range(16), range(16)):
            lo = sum(((fbits >> q) & 1) << lower_face[q] for q in range(4)) | \
                sum(((lbits >> q) & 1) << free_lo[q] for q in range(4))
            up = sum(((fbits >> q) & 1) << upper_face[q] for q in range(4)) | \
                sum(((ubits >> q) & 1) << free_up[q] for q in range(4))
            sa = _face_segments_world(lo, axis, 1, np.zeros(3))
            sb = _face_segments_world(up, axis, 0, shift)
            assert {(b, a) for a, b in sb} == sa, (axis, lo, up)


# ---- oracle on analytic fields ---------------------------------------------------------------
def _lattice(n=(64, 64, 64), lo=-1.0, hi=1.0):
    axes = [np.linspace(lo, hi, k) for k in n]
    X, Y, Z = np.meshgrid(*axes, indexing='ij')
    return X, Y, Z, axes


def _mesh_checks(v, f, euler=None):
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).astype(np.int64)
    key = e[:, 0] * (len(v) + 1) + e[:, 1]
    assert len(np.unique(key)) == len(key), 'a directed edge appears twice'
    und = np.sort(e, 1)
    _, cnt = np.unique(und[:, 0] * (len(v) + 1) + und[:, 1], return_counts=True)
    assert (cnt == 2).all(), 'not a closed 2-manifold'
    assert len(np.unique(f)) == len(v)
    if euler is not None:
        assert len(v) - len(cnt) + len(f) == euler


def _volume(v, f):
    a, b, c = (v[f[:, q]].astype(np.float64) for q in range(3))
    return float(np.einsum('ij,ij->i', a, np.cross(b, c)).sum() / 6)


def _check_vertices_and_normals(fld, v, f, origin, spacing, grad):
    idx = (v.astype(np.float64) - origin) / spacing
    frac = np.abs(idx - np.round(idx))
    on_axis = frac > 1e-4
    assert (on_axis.sum(1) <= 1).all()
    for r in np.nonzero(on_axis.sum(1) == 1)[0][:2000]:
        a = int(np.argmax(on_axis[r]))
        i0 = np.round(idx[r]).astype(int)
        i0[a] = int(np.floor(idx[r][a]))
        i1 = i0.copy()
        i1[a] += 1
        v0, v1 = fld[tuple(i0)], fld[tuple(i1)]
        assert (v0 < 0) != (v1 < 0)
        t = (0 - v0) / (v1 - v0)
        assert abs(idx[r][a] - i0[a] - t) < 1e-4
    p0, p1, p2 = (v[f[:, q]].astype(np.float64) for q in range(3))
    n = np.cross(p1 - p0, p2 - p0)
    g = grad((p0 + p1 + p2) / 3)
    assert (np.einsum('ij,ij->i', n, g) > 0).mean() > 0.999


def _run(fld, axes):
    origin = np.array([a[0] for a in axes])
    spacing = np.array([a[1] - a[0] for a in axes])
    v, f = marching_cubes(fld.astype(np.float32), 0.0, origin, spacing)
    return v, f, origin, spacing


def test_oracle_sphere():
    X, Y, Z, axes = _lattice()
    r = 0.7
    fld = np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - r
    v, f, o, s = _run(fld, axes)
    _mesh_checks(v, f, euler=2)
    assert abs(_volume(v, f) / (4 / 3 * np.pi * r ** 3) - 1) < 0.01
    _check_vertices_and_normals(fld.astype(np.float32), v, f, o, s, lambda p: p)


def test_oracle_torus():
    X, Y, Z, axes = _lattice()
    R, r = 0.6, 0.25
    q = np.sqrt(X ** 2 + Y ** 2)
    fld = np.sqrt((q - R) ** 2 + Z ** 2) - r
    v, f, o, s = _run(fld, axes)
    _mesh_checks(v, f, euler=0)
    assert abs(_volume(v, f) / (2 * np.pi ** 2 * R * r ** 2) - 1) < 0.01

    def grad(p):
        qq = np.sqrt(p[:, 0] ** 2 + p[:, 1] ** 2)
        return np.stack([p[:, 0] * (qq - R) / qq, p[:, 1] * (qq - R) / qq, p[:, 2]], -1)
    _check_vertices_and_normals(fld.astype(np.float32), v, f, o, s, grad)


def test_oracle_box():
    X, Y, Z, axes = _lattice()
    h = np.array([0.55, 0.4, 0.3])
    fld = np.maximum(np.maximum(np.abs(X) - h[0], np.abs(Y) - h[1]), np.abs(Z) - h[2])
    v, f, _, _ = _run(fld, axes)
    _mesh_checks(v, f, euler=2)
    assert abs(_volume(v, f) / (8 * h.prod()) - 1) < 0.01


def _ambiguous_faces(ins):
    """Lattice faces whose two diagonal corners are inside and the other two outside."""
    n = 0
    for a, b in ((0, 1), (0, 2), (1, 2)):
        def sl(da, db):
            s = [slice(None)] * 3
            s[a] = slice(da, ins.shape[a] - 1 + da)
            s[b] = slice(db, ins.shape[b] - 1 + db)
            return tuple(s)
        c00, c11, c10, c01 = ins[sl(0, 0)], ins[sl(1, 1)], ins[sl(1, 0)], ins[sl(0, 1)]
        n += int(((c00 & c11 & ~c10 & ~c01) | (~c00 & ~c11 & c10 & c01)).sum())
    return n


def two_spheres(X, Y, Z, step, r=0.4, gap=0.2):
    """Two spheres on the xy diagonal whose gap is below one lattice step."""
    d = (r + gap * step) / np.sqrt(2)
    return np.minimum(np.sqrt((X - d) ** 2 + (Y - d) ** 2 + Z ** 2),
                      np.sqrt((X + d) ** 2 + (Y + d) ** 2 + Z ** 2)) - r


def test_oracle_two_nearly_touching_spheres():
    X, Y, Z, axes = _lattice((48, 48, 48))
    fld = two_spheres(X, Y, Z, axes[0][1] - axes[0][0])
    assert _ambiguous_faces(fld < 0) > 0
    v, f, _, _ = _run(fld, axes)
    _mesh_checks(v, f)


def test_oracle_non_cubic_lattice():
    X, Y, Z, axes = _lattice((21, 33, 46))
    fld = (X / 0.8) ** 2 + (Y / 0.6) ** 2 + (Z / 0.7) ** 2 - 1
    v, f, o, s = _run(fld, axes)
    _mesh_checks(v, f, euler=2)
    assert abs(_volume(v, f) / (4 / 3 * np.pi * 0.8 * 0.6 * 0.7) - 1) < 0.03
    _check_vertices_and_normals(fld.astype(np.float32), v, f, o, s,
                                lambda p: p / np.array([0.64, 0.36, 0.49]))


def test_oracle_order_and_batch():
    """Vertices ordered by (volume, i, j, k, axis); volumes never share vertices; faces of
    volume b only reference volume b's vertices."""
    g = np.random.default_rng(0)
    fld = g.standard_normal((3, 5, 6, 7)).astype(np.float32)
    fld[1] = 1.0  # no crossing
    v, f = marching_cubes(fld, 0.0, np.zeros((3, 3)), np.ones((3, 3)))
    nv0 = len(marching_cubes(fld[0])[0])
    v2, f2 = marching_cubes(fld[2])
    assert np.array_equal(v[nv0:], v2)
    assert np.array_equal(f[f.min(1) >= nv0] - nv0, f2)


# ---- mesher host logic ----------------------------------------------------------------------
def test_mesher_lattice_matches_reference_layout():
    """The device lattice order [i][j][k] equals the reference's meshgrid / reshape(ny,nx,nz) /
    transpose(1,0,2) volume, coordinates equal np.linspace bit for bit, and points not
    strictly inside the bounding box get 100."""
    from xrdslam_b200.mesher import Mesher, MesherConfig
    mc_bound = torch.from_numpy(np.array([[-1.1, 0.9], [-0.7, 1.3], [-0.5, 0.45]]))
    bbox = torch.from_numpy(np.array([[-1.0, 0.8], [-0.6, 1.2], [-0.45, 0.4]]))
    res = 11
    m = Mesher(MesherConfig(resolution=res, points_batch_size=97), None, bbox, mc_bound)
    c = 3.25

    def query_fn(p):
        return (p[:, 0] + 10 * p[:, 1] + 100 * p[:, 2] - c)[:, None]

    fld, xyz = m.get_field(query_fn, torch.device('cpu'))
    for d in range(3):
        ref = np.linspace(float(mc_bound[d][0]), float(mc_bound[d][1]), res)
        assert np.array_equal(xyz[d], ref) and xyz[d].dtype == np.float64
    # the reference (mesher.py:41-66, 138-167, 203-214)
    x, y, z = xyz
    xx, yy, zz = np.meshgrid(x, y, z)
    pts = torch.tensor(np.vstack([xx.ravel(), yy.ravel(), zz.ravel()]).T, dtype=torch.float)
    ret = query_fn(pts)
    mask = ((pts[:, 0] < bbox[0][1]) & (pts[:, 0] > bbox[0][0]) & (pts[:, 1] < bbox[1][1]) &
            (pts[:, 1] > bbox[1][0]) & (pts[:, 2] < bbox[2][1]) & (pts[:, 2] > bbox[2][0]))
    ret[~mask, :] = 100
    ref = ret.numpy()[:, -1].astype(np.float32).reshape(res, res, res).transpose([1, 0, 2])
    assert 0 < int(mask.sum()) < mask.numel()
    assert np.array_equal(fld.numpy(), ref)


def test_mesher_use_mask_not_provided():
    from xrdslam_b200.mesher import Mesher, MesherConfig
    m = Mesher(MesherConfig(), None, None, None)
    with pytest.raises(NotImplementedError):
        m.get_mesh([], lambda p: p, use_mask=True)


def test_mesh_export_roundtrip(tmp_path):
    from xrdslam_b200.io_formats import read_ply
    from xrdslam_b200.mesher import Mesh
    X, Y, Z, axes = _lattice((16, 16, 16))
    v, f, _, _ = _run(np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - 0.6, axes)
    col = (np.arange(len(v) * 3) % 256).astype(np.uint8).reshape(-1, 3)
    path = Mesh(v, f, col).export(str(tmp_path / 'final_mesh.ply'))
    v2, f2, c2 = read_ply(path)
    assert np.array_equal(v2, v) and np.array_equal(f2, f) and np.array_equal(c2, col)


def test_workspace_bound_at_256():
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    assert 0 < lib.xrd_mc_workspace_bytes(1, 256, 256, 256) < (1 << 30)
    assert lib.xrd_mc_workspace_bytes(1, 1, 5, 5) == 0
