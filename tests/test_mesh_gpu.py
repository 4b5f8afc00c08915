"""Marching cubes (csrc/mesh.cu), the Vox-Fusion point query and the algorithms' get_mesh on the
device against the numpy oracle (oracle/marching_cubes.py) and the decoder oracles."""
import numpy as np
import pytest
import torch

from helpers import BOUND, max_abs
from oracle.marching_cubes import marching_cubes as mc_oracle
from test_mesh_cpu import _lattice, _mesh_checks, two_spheres

pytestmark = pytest.mark.gpu


def _cam():
    from xrdslam_b200.camera import Camera
    return Camera(320., 320., 319.5, 239.5, 640, 480)


def _mc_dev(fld, level=0.0, origin=(0., 0., 0.), spacing=(1., 1., 1.), origins=None,
            spacings=None):
    from xrdslam_b200.mesher import MarchingCubes
    t = lambda a: None if a is None else torch.from_numpy(np.asarray(a, np.float64)).cuda()
    mc = MarchingCubes(torch.from_numpy(np.ascontiguousarray(fld, np.float32)).cuda(), level,
                       origin, spacing, t(origins), t(spacings))
    v, f = mc.run()
    return v.cpu().numpy(), f.cpu().numpy()


def _same(dev, ora):
    (v, f), (vo, fo) = dev, ora
    assert f.shape == fo.shape and np.array_equal(f, fo)
    assert v.shape == vo.shape and np.array_equal(v.view(np.uint32), vo.view(np.uint32))


def _fields():
    X, Y, Z, ax = _lattice((40, 40, 40))
    step = ax[0][1] - ax[0][0]
    q = np.sqrt(X ** 2 + Y ** 2)
    Xn, Yn, Zn, axn = _lattice((21, 33, 46))
    return {
        'sphere': (np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - 0.7, ax),
        'torus': (np.sqrt((q - 0.6) ** 2 + Z ** 2) - 0.25, ax),
        'two_spheres': (two_spheres(X, Y, Z, step), ax),
        'non_cubic': ((Xn / 0.8) ** 2 + (Yn / 0.6) ** 2 + (Zn / 0.7) ** 2 - 1, axn),
        # many values exactly at the level (inside is value < level)
        'on_level': (np.round((np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - 0.5) * 8) / 8, ax),
        # surface cut open by the volume boundary
        'cut_open': (np.sqrt((X + 1) ** 2 + (Y + 1) ** 2 + (Z + 1) ** 2) - 0.9, ax),
        'empty': (np.ones_like(X), ax),
        'all_inside': (-np.ones_like(X), ax),
    }


@pytest.mark.parametrize('name', list(_fields()))
def test_mc_matches_oracle(cuda_dev, name):
    fld, ax = _fields()[name]
    fld = fld.astype(np.float32)
    origin = tuple(float(a[0]) for a in ax)
    spacing = tuple(float(a[2] - a[1]) for a in ax)
    dev = _mc_dev(fld, 0.0, origin, spacing)
    _same(dev, mc_oracle(fld, 0.0, origin, spacing))
    _same(dev, _mc_dev(fld, 0.0, origin, spacing))  # run to run
    if name in ('empty', 'all_inside'):
        assert dev[0].shape == (0, 3) and dev[1].shape == (0, 3)
    elif name not in ('cut_open',):
        _mesh_checks(*dev)


def test_mc_level_set(cuda_dev):
    fld, ax = _fields()['sphere']
    fld = fld.astype(np.float32)
    _same(_mc_dev(fld, 0.1, (0.5, -2., 1.), (0.1, 0.2, 0.3)),
          mc_oracle(fld, 0.1, (0.5, -2., 1.), (0.1, 0.2, 0.3)))


def test_mc_batched_small_volumes(cuda_dev):
    """Vox-Fusion's shape: many 8^3 volumes with their own origin / spacing, some without a
    crossing; vertices are never welded across volumes."""
    g = np.random.default_rng(3)
    B = 300
    c = g.uniform(-0.6, 0.6, (B, 3))
    x = np.linspace(-0.5, 0.5, 8)
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    fld = np.sqrt((X[None] - c[:, 0, None, None, None]) ** 2 + (Y[None] - c[:, 1, None, None, None]) ** 2
                  + (Z[None] - c[:, 2, None, None, None]) ** 2) - 0.35
    fld[::7] = 1.0
    fld[3::11] = -1.0
    fld = fld.astype(np.float32)
    origins = g.uniform(-5, 5, (B, 3))
    spacings = np.full((B, 3), 0.2 / 7)
    dev = _mc_dev(fld, 0.0, origins=origins, spacings=spacings)
    _same(dev, mc_oracle(fld, 0.0, origins, spacings))
    _same(dev, _mc_dev(fld, 0.0, origins=origins, spacings=spacings))
    assert dev[1].shape[0] > 0


def test_mc_workspace_and_shape_errors(cuda_dev):
    from xrdslam_b200 import _cabi
    from xrdslam_b200.mesher import MarchingCubes
    assert _cabi.lib().xrd_mc_workspace_bytes(1, 256, 256, 256) < (1 << 30)
    with pytest.raises(_cabi.XrdError):
        MarchingCubes(torch.zeros(1, 1, 5, 5, device=cuda_dev)).run()


def _vox_oracle_raw(model, pts, ids, centres, vertex_idx):
    """get_features + Decoder.get_values (voxel_helpers_voxfusion.py:106-153,
    decoder_voxfusion.py:122-140) on the CPU."""
    from oracle.voxfusion import VoxDecoder, offset_points_q
    dec = VoxDecoder()
    dec.load_state_dict({k: v.cpu() for k, v in model.decoder.state_dict().items()})
    vs = model.config.voxel_size
    ids = ids.long().cpu()
    point_xyz = centres.cpu()[ids]
    feats = model.embeddings.detach().cpu()[vertex_idx.long().cpu()[ids]].view(len(ids), -1)
    p = ((pts.cpu() - point_xyz) / vs + 0.5).unsqueeze(1)
    q = offset_points_q().unsqueeze(0)
    w = (p * q + (1 - p) * (1 - q)).prod(dim=-1, keepdim=True)
    emb = (w * feats.view(len(ids), 8, -1)).sum(1).float()
    with torch.no_grad():
        rgb, sdf = dec(emb)
    return torch.cat([rgb, sdf[:, None]], -1)


def _vox_algo(cuda_dev, mapping_iters=30):
    from test_algorithms_gpu import _frames
    from xrdslam_b200.voxfusion import VoxFusionConfig
    torch.manual_seed(0)
    np.random.seed(0)
    cam, poses, fr = _frames(2, rot_rep='quat', offset=(10.0, 10.0, 10.0))
    algo = VoxFusionConfig().setup(camera=cam, device=cuda_dev)
    algo.add_keyframe(fr[0])
    algo.optimize_update(mapping_iters, [fr[0]], is_mapping=True)
    return algo


def _vox_filtered(algo):
    voxels, _, features = algo.model.octree_tables()
    keep = ~features.eq(-1).any(-1)
    voxels, features = voxels[keep], features[keep]
    return voxels, features, (voxels[:, :3] + voxels[:, -1:] / 2) * algo.model.config.voxel_size


def test_voxfusion_query_matches_oracle(cuda_dev):
    algo = _vox_algo(cuda_dev, mapping_iters=5)
    m = algo.model
    voxels, features, centres = _vox_filtered(algo)
    g = torch.Generator().manual_seed(2)
    P = 5000
    ids = torch.randint(0, centres.shape[0], (P,), generator=g).to(cuda_dev)
    pts = centres[ids] + (torch.rand(P, 3, generator=g).to(cuda_dev) - 0.5) * m.config.voxel_size
    raw = m.query(pts, ids, centres, features)
    ref = _vox_oracle_raw(m, pts, ids, centres, features)
    assert raw.shape == (P, 4)
    assert max_abs(raw, ref) < 2e-4
    assert m.query(pts[:0], ids[:0], centres, features).shape == (0, 4)


def test_voxfusion_get_mesh(cuda_dev):
    algo = _vox_algo(cuda_dev)
    m = algo.model
    vs, res = m.config.voxel_size, 8
    voxels, features, centres = _vox_filtered(algo)
    mesh = algo.get_mesh()
    # the field the device meshes == the oracle decoder on the reference's lattice
    x = torch.linspace(-.5, .5, res)
    lat = torch.stack(torch.meshgrid(x, x, x, indexing='ij'), -1).float().to(cuda_dev) * vs
    pts = (lat.reshape(1, -1, 3) + centres.unsqueeze(1)).reshape(-1, 3)
    ids = torch.arange(centres.shape[0], device=cuda_dev)[:, None].expand(-1, res ** 3).reshape(-1)
    sdf = m.query(pts, ids, centres, features)[:, 3]
    assert mesh is not None and mesh.faces.shape[0] > 0, (
        centres.shape[0], float(sdf.min()), float(sdf.max()))
    sel = torch.randperm(pts.shape[0], generator=torch.Generator().manual_seed(0))[:20000]
    sel = sel.to(cuda_dev)
    assert max_abs(sdf[sel], _vox_oracle_raw(m, pts[sel], ids[sel], centres, features)[:, 3]) < 2e-4
    # oracle marching cubes on the device's field: identical mesh
    origins = (centres.double() - vs / 2).cpu().numpy()
    spacings = np.full_like(origins, vs / (res - 1))
    vo, fo = mc_oracle(sdf.reshape(-1, res, res, res).cpu().numpy(), 0.0, origins, spacings)
    _same((mesh.vertices, mesh.faces), (vo, fo))
    # colours: first voxel (list order) whose grid coordinates equal v // voxel_size
    grid = voxels[:, :3].cpu().numpy()
    first = {}
    for i, key in enumerate(map(tuple, grid)):
        first.setdefault(key, i)
    vpos = (torch.from_numpy(vo).to(cuda_dev) // vs).cpu().numpy()
    match = np.array([first.get(tuple(p), -1) for p in vpos])
    col = np.zeros((len(vo), 3), np.float32)
    ok = match >= 0
    col[ok] = _vox_oracle_raw(m, torch.from_numpy(vo[ok]), torch.from_numpy(match[ok]), centres,
                              features)[:, :3].numpy()
    assert mesh.vertex_colors.shape == (len(vo), 3)
    assert max_abs(mesh.vertex_colors, col) < 2e-4
    assert (mesh.vertex_colors[~ok] == 0).all()
    # a vertex in no voxel of the map gets colour 0
    far = torch.tensor([[-50.0, -50.0, -50.0], [float(centres[0, 0]), float(centres[0, 1]),
                                                float(centres[0, 2])]], device=cuda_dev)
    c = algo.vertex_colors(far, voxels, centres, features)
    assert (c[0] == 0).all() and max_abs(
        c[1:], _vox_oracle_raw(m, far[1:], torch.tensor([first[tuple((far[1:] // vs).cpu().numpy()[0])]]),
                               centres, features)[:, :3]) < 2e-4


def _coslam_algo(cuda_dev, resolution):
    from test_algorithms_gpu import _frames
    from xrdslam_b200.coslam import CoSLAMConfig
    from xrdslam_b200.mesher import MesherConfig
    torch.manual_seed(0)
    np.random.seed(0)
    cam, poses, fr = _frames(3, separate_LR=True)
    algo = CoSLAMConfig(mapping_sample=512, tracking_sample=256, tracking_Wedge=5,
                        tracking_Hedge=5, mapping_bound=BOUND.tolist(),
                        mesher=MesherConfig(resolution=resolution)).setup(camera=cam, device=cuda_dev)
    algo.optimize_update(10, [fr[0]], True)
    return algo


def _mask(p, bound):
    b = torch.as_tensor(bound)
    return ((p[:, 0] < b[0][1]) & (p[:, 0] > b[0][0]) & (p[:, 1] < b[1][1]) & (p[:, 1] > b[1][0])
            & (p[:, 2] < b[2][1]) & (p[:, 2] > b[2][0]))


def _check_algo_mesh(algo, mesh, field_o, color_o, tol):
    """Device field vs the oracle's, oracle MC on the device's field, colours within 1 step."""
    dev = algo.device
    fld, xyz = algo.mesher.get_field(algo.model.query_fn, dev)
    lat = algo.mesher.lattice_points([torch.from_numpy(v.astype(np.float32)) for v in xyz], 0,
                                     fld.numel())
    fo = field_o(lat)
    fo = torch.where(_mask(lat, algo.bounding_box), fo, torch.full_like(fo, 100))
    assert max_abs(fld.reshape(-1), fo) < tol
    vo, fco = mc_oracle(fld.cpu().numpy(), 0.0, tuple(float(v[0]) for v in xyz),
                        tuple(float(v[2] - v[1]) for v in xyz))
    _same((mesh.vertices, mesh.faces), (vo, fco))
    v = torch.from_numpy(vo)
    co = color_o(v)
    co = torch.where(_mask(v, algo.bounding_box)[:, None], co, torch.full_like(co, 100))
    co = (co.clamp(0, 1) * 255).to(torch.uint8)
    assert mesh.vertex_colors.dtype == np.uint8
    assert np.abs(mesh.vertex_colors.astype(int) - co.numpy().astype(int)).max() <= 1


def test_coslam_get_mesh(cuda_dev):
    from oracle.coslam import CoslamOracle
    algo = _coslam_algo(cuda_dev, 48)
    model = algo.model
    ora = CoslamOracle(BOUND)
    with torch.no_grad():
        ora.embed_fn.params.copy_(model.embed_fn.params.detach().cpu())
        ora.sdf0.weight.copy_(model.decoder.sdf_net.model[0].weight.cpu())
        ora.sdf1.weight.copy_(model.decoder.sdf_net.model[2].weight.cpu())
        ora.col0.weight.copy_(model.decoder.color_net.model[0].weight.cpu())
        ora.col1.weight.copy_(model.decoder.color_net.model[2].weight.cpu())
    bb = torch.as_tensor(BOUND, dtype=torch.float64)

    def raw_o(p):
        with torch.no_grad():
            return ora.query_color_sdf((p - bb[:, 0]) / (bb[:, 1] - bb[:, 0]))

    mesh = algo.get_mesh()
    assert mesh is not None and algo.cur_mesh is mesh and mesh.faces.shape[0] > 0
    _check_algo_mesh(algo, mesh, lambda p: raw_o(p)[:, 3].float(),
                     lambda p: torch.sigmoid(raw_o(p)[:, :3]).float(), 2e-5)


def test_nice_get_mesh(cuda_dev):
    """NICE-SLAM with the parity tests' paired model (oracle/nice.py restates its decoders)."""
    from test_nice_gpu import BOUND as NB, nice_pair
    from xrdslam_b200.mesher import MesherConfig
    from xrdslam_b200.nice_slam import NiceSLAMConfig
    ora, model = nice_pair(cuda_dev)
    bound = NB.tolist()
    mc_bound = [[-2.3, 2.3], [-2.3, 2.3], [-2.3, 2.3]]  # part of the lattice is masked
    algo = NiceSLAMConfig(mapping_bound=bound, marching_cubes_bound=mc_bound,
                          mesher=MesherConfig(resolution=48)).setup(camera=_cam(), device=cuda_dev)
    algo.model = model

    def dec(p, stage):
        with torch.no_grad():
            return ora.decode(p, stage)

    mesh = algo.get_mesh()
    assert mesh is not None and mesh.faces.shape[0] > 0
    _check_algo_mesh(algo, mesh, lambda p: dec(p, 'fine')[:, -1], lambda p: dec(p, 'color')[:, :3],
                     2e-4)


def test_point_slam_has_no_mesher(cuda_dev):
    from xrdslam_b200.algorithm import Algorithm
    from xrdslam_b200.point_slam import PointSLAM
    assert PointSLAM.get_mesh is Algorithm.get_mesh


def test_coslam_get_mesh_256(cuda_dev, tmp_path):
    from xrdslam_b200.io_formats import read_ply
    algo = _coslam_algo(cuda_dev, 256)
    mesh = algo.get_mesh()
    assert mesh is not None and mesh.faces.shape[0] > 0
    assert mesh.faces.max() < mesh.vertices.shape[0]
    v, f, c = read_ply(mesh.export(str(tmp_path / 'final_mesh.ply')))
    assert np.array_equal(v, mesh.vertices) and np.array_equal(f, mesh.faces)
    assert np.array_equal(c, mesh.vertex_colors)
