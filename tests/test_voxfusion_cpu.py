"""CPU tests for the Vox-Fusion map structure: this package's octree (csrc/octree.cpp) against
the reference's own svo.Octree compiled from its sources, through the digests stored in
tests/golden/reference_cpu.json (tests/golden/make_golden.py reference_cpu)."""
import numpy as np
import torch

from helpers import GOLDEN, digest, load_golden_json


def octree_inserts():
    g = torch.Generator().manual_seed(4)
    for it in range(4):
        pts = (torch.rand(2500, 3, generator=g) * 25 + 30 + 7 * it).int().contiguous()
        if it == 0:
            pts[0] = torch.tensor([0, 0, 0])
            pts[1] = torch.tensor([254, 254, 254])
            pts[2] = pts[3]  # duplicates
        yield pts


def test_octree_bit_exact_vs_reference_svo():
    """Centres, children and features after every insert equal the reference svo.Octree's
    (the first tree of its process, so the node ids coincide), bit for bit."""
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    ref = load_golden_json('reference_cpu.json')['octree']
    t = lib.xrd_octree_create(256)
    try:
        for pts, want in zip(octree_inserts(), ref):
            n = lib.xrd_octree_insert(t, pts.data_ptr(), pts.shape[0])
            assert n == lib.xrd_octree_num_nodes(t)
            mv = torch.empty(n, 4)
            mc = torch.empty(n, 8)
            mf = torch.empty(n, 8, dtype=torch.int32)
            assert lib.xrd_octree_export(t, mv.data_ptr(), mc.data_ptr(), mf.data_ptr()) == n
            assert [digest(mv), digest(mc), digest(mf)] == want
    finally:
        lib.xrd_octree_destroy(t)


def test_model_map_states_match_reference_formulas():
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.sparse_voxel import SparseVoxelConfig
    m = SparseVoxelConfig().setup(camera=Camera(320, 320, 319.5, 239.5, 640, 480))
    g = torch.Generator().manual_seed(0)
    pts = torch.rand(800, 3, generator=g) * 3 + 24.1
    m.insert_points(pts)
    ms = m.map_states
    N = ms['voxel_center_xyz'].shape[0]
    assert ms['voxel_structure'].shape == (N, 9) and ms['voxel_vertex_idx'].shape == (N, 8)
    leaf = ms['voxel_structure'][:, 8] == 1
    surf = leaf & (ms['voxel_vertex_idx'][:, 0] >= 0)
    # every inserted point lies inside a SURFACE leaf: centre = (floor(p/0.2) + 0.5) * 0.2
    want = {tuple(v) for v in torch.div(pts, 0.2, rounding_mode='floor').int().tolist()}
    have = {tuple(v) for v in torch.round(ms['voxel_center_xyz'][surf] / 0.2 - 0.5).int().tolist()}
    assert want <= have and len(have) == len(want)
    assert int(ms['voxel_vertex_idx'].max()) < m.config.num_embeddings


def vox_case():
    """A wall of voxels at z ~ 12.0 m (offset world), rays from above, marched by the oracle.
    The map comes from this package's octree (bit-exact vs the reference's svo above)."""
    from oracle.voxfusion import VoxOracle
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.sparse_voxel import SparseVoxelConfig
    g = torch.Generator().manual_seed(3)
    xy = torch.rand(3000, 2, generator=g) * 2.0 + 11.0
    pts = torch.cat([xy, torch.full((3000, 1), 12.05) + torch.rand(3000, 1, generator=g) * 0.3], 1)
    builder = SparseVoxelConfig().setup(camera=Camera(320, 320, 319.5, 239.5, 640, 480))
    builder.insert_points(pts)
    voxels, children, features = builder.export_octree()
    torch.manual_seed(5)  # the decoder keeps torch's default init
    ora = VoxOracle(seed=5)
    ora.set_map(voxels, children, features)
    with torch.no_grad():
        ora.embeddings.mul_(30.0)
    R = 96
    ro = torch.cat([torch.rand(R, 2, generator=g) * 1.6 + 11.2, torch.full((R, 1), 10.5)], 1)
    rd = torch.nn.functional.normalize(
        torch.cat([torch.randn(R, 2, generator=g) * 0.15, torch.ones(R, 1)], 1), dim=-1)
    rd[::13] = torch.tensor([0.0, 0.0, -1.0])  # rays that miss the map
    marched = ora.march(ro, rd, lambda shape: torch.rand(shape, generator=g))
    assert marched is not None
    inter, hits, samples = marched
    assert hits.any() and not hits.all()
    td = torch.full((R, 1), 1.62) + torch.rand(R, 1, generator=g) * 0.2
    td[5::11] = 0
    ts = torch.rand(R, 3, generator=g)
    ms = {'voxel_vertex_idx': ora.vertex_idx, 'voxel_center_xyz': ora.centres,
          'voxel_structure': ora.children}
    full_inter = {k: torch.zeros((R,) + v.shape[1:], dtype=v.dtype) for k, v in inter.items()}
    for k in full_inter:
        full_inter[k][hits] = inter[k]
    return ora, ro, rd, ts, td, marched, ms, full_inter


def test_vox_oracle_torch_part_matches_reference_python(one_thread):
    """oracle/voxfusion.py's features / decoder / sdf2weights / losses against the reference's
    own SparseVoxel.render_rays + get_loss_dict run on CPU on the same map, decoder, embeddings,
    intersections and samples (its two CUDA ops replaced by the oracle's intersections and
    samples, which the GPU tests pin bit-for-bit against the reference's compiled kernels)."""
    import os
    g = load_golden_json('reference_cpu.json')['vox']
    a = np.load(os.path.join(GOLDEN, 'reference_cpu.npz'))
    r = lambda k: torch.from_numpy(a['vox.' + k])
    ora, ro, rd, ts, td, marched, _, _ = vox_case()
    od = ora.decoder
    out_o, ld_o = ora.render(ro, rd, ts, td, marched)
    assert digest(out_o['ray_mask']) == g['ray_mask']
    assert (r('depth') - out_o['depth']).abs().max() < 1e-6
    assert (r('rgb') - out_o['rgb']).abs().max() < 1e-6
    assert (r('sdf') - out_o['sdf']).abs().max() < 1e-6
    assert set(ld_o) == set(g['losses'])
    for k, v in g['losses'].items():
        assert abs(v - float(ld_o[k].detach())) <= 1e-5 * max(1e-3, abs(v)), k
    # gradients of the summed loss w.r.t. embeddings and decoder
    sum(ld_o.values()).backward()
    ge_r = torch.zeros_like(ora.embeddings)
    ge_r[r('d_embeddings_rows')] = r('d_embeddings')
    assert (ora.embeddings.grad - ge_r).abs().max() <= 1e-5 * ge_r.abs().max()
    assert (od.sdf_out.weight.grad - r('d_sdf_out_w')).abs().max() <= \
        1e-5 * r('d_sdf_out_w').abs().max()


def test_device_octree_equals_host_octree_numbering():
    """octree_device.DeviceOctree (data-parallel build: unique / sort / searchsorted) produces
    the SAME node ids, codes, child tables and corner-leaf tables as the host C++ octree (which
    is bit-exact against the reference's compiled svo.Octree, test above) -- over duplicate
    voxels, two successive insert calls, coordinates at the grid edge (wrap quirk) and an
    empty second call.  Runs on the host here; the same tensor program runs on the GPU."""
    from xrdslam_b200 import _cabi
    from xrdslam_b200.octree_device import DeviceOctree
    lib = _cabi.lib()

    def host(vlist):
        t = lib.xrd_octree_create(256)
        for v in vlist:
            v = v.int().contiguous()
            lib.xrd_octree_insert(t, v.data_ptr(), v.shape[0])
        N = lib.xrd_octree_num_nodes(t)
        vo, ch, fe = torch.empty(N, 4), torch.empty(N, 8), torch.empty(N, 8, dtype=torch.int32)
        lib.xrd_octree_export(t, vo.data_ptr(), ch.data_ptr(), fe.data_ptr())
        lib.xrd_octree_destroy(t)
        return vo, ch, fe
    g = torch.Generator().manual_seed(0)
    for trial, (n1, n2) in enumerate([(50, 30), (2000, 1500), (1, 1), (5000, 5000), (300, 0)]):
        base = torch.randint(100, 150, (max(n1 // 4, 1), 3), generator=g)
        v1 = base[torch.randint(0, base.shape[0], (n1,), generator=g)] + \
            torch.randint(-2, 3, (n1, 3), generator=g)
        v2 = base[torch.randint(0, base.shape[0], (max(n2, 1),), generator=g)][:n2] + \
            torch.randint(-6, 7, (n2, 3), generator=g)
        if trial == 3:
            v1[:5] = torch.tensor([[255, 255, 255], [0, 0, 0], [255, 0, 128], [254, 255, 3],
                                   [128, 128, 128]])
        ref = host([v1, v2] if n2 else [v1])
        t = DeviceOctree(256)
        t.insert(v1)
        t.insert(v2)
        got = t.export()
        assert t.num_nodes() == ref[0].shape[0]
        for a, b in zip(ref, got):
            assert a.dtype == b.dtype and torch.equal(a, b), trial
