"""CPU tests (no GPU): the oracle is pinned to the reference's own classes through the
committed golden vectors and digests (tests/golden/make_golden.py); the C-ABI library loads and exports every declared symbol."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from helpers import (BOUND, digest, load_golden_coslam, load_golden_json, make_rays, max_abs,
                     rel_err, set_coslam_params)


def _oracle_from_golden():
    from oracle.coslam import CoslamOracle
    g = load_golden_coslam()
    ora = CoslamOracle(BOUND)
    set_coslam_params(ora, g, 'oracle')
    return ora, g


def test_oracle_matches_golden_reference_vectors():
    """oracle/coslam.py == vectors produced by the reference's JointEncoding."""
    ora, g = _oracle_from_golden()
    t = lambda k: torch.from_numpy(g[k])
    rays_o = t('rays_o').requires_grad_(True)
    rays_d = t('rays_d').requires_grad_(True)
    out, ld, tot = ora.step(rays_o, rays_d, t('target_s'), t('target_d'), t('noise'),
                            True, False, smooth_rand=t('smooth_rand').reshape(2, 3))
    tot.backward()
    assert np.array_equal(out['z_vals'].detach().numpy(), g['z_vals'])
    assert np.array_equal(out['raw'].detach().numpy(), g['raw'])
    assert np.array_equal(out['rgb'].detach().numpy(), g['rgb'])
    assert np.array_equal(out['depth'].detach().numpy(), g['depth'])
    got = [float(ld[k].detach()) for k in
           ('rgb_loss', 'depth_loss', 'sdf_loss', 'fs_loss', 'smooth_loss')]
    assert np.allclose(got, g['losses'], rtol=1e-6, atol=0)
    assert np.allclose(rays_o.grad.numpy(), g['d_rays_o'], rtol=1e-5, atol=1e-9)
    assert np.allclose(ora.sdf0.weight.grad.numpy(), g['d_w_sdf0'], rtol=1e-5, atol=1e-9)
    assert abs(float(ora.embed_fn.params.grad.double().norm()) - float(g['d_table_norm'])) \
        <= 1e-6 * float(g['d_table_norm'])
    assert int((ora.embed_fn.params.grad != 0).sum()) == int(g['d_table_nnz'])


def coslam_live_case():
    """Oracle with seeded parameters (table x 3000 of the reference's init scale: non-trivial
    sdf sign changes), rays and the noise the reference draws after torch.manual_seed(9)."""
    from oracle.coslam import CoslamOracle
    ora = CoslamOracle(BOUND)
    g = torch.Generator().manual_seed(21)
    with torch.no_grad():
        ora.embed_fn.params.copy_((torch.rand(ora.embed_fn.params.shape, generator=g) * 2 - 1) * 0.3)
        for lin in (ora.sdf0, ora.sdf1, ora.col0, ora.col1):
            lin.weight.copy_(torch.randn(lin.weight.shape, generator=g) / np.sqrt(lin.weight.shape[1]))
    R = 80
    rays_o, rays_d, ts, td, _ = make_rays(R, seed=3)
    torch.manual_seed(9)
    noise = torch.rand(R, 43)
    r1, r2 = torch.rand(3), torch.rand((1, 1, 1, 3))
    torch.manual_seed(4)
    n256 = torch.rand(R, 256)
    return ora, (rays_o, rays_d, ts, td), noise, torch.stack([r1, r2.reshape(3)]), n256


COSLAM_OUT_KEYS = ('rgb', 'depth', 'z_vals', 'raw', 'depth_var', 'disp_map', 'acc_map')


def test_oracle_matches_reference_class_live(one_thread):
    """The reference's JointEncoding on the same parameters, rays and noise: outputs and losses
    bit-identical (tests/golden/reference_cpu.json, written by make_golden.py reference_cpu)."""
    g = load_golden_json('reference_cpu.json')['coslam']
    ora, (rays_o, rays_d, ts, td), noise, smooth_rand, n256 = coslam_live_case()
    out_o, ld_o, _ = ora.step(rays_o, rays_d, ts, td, noise, True, False, smooth_rand=smooth_rand)
    for k in COSLAM_OUT_KEYS:
        assert digest(out_o[k]) == g['out'][k], k
    assert set(ld_o) == set(g['losses'])
    for k in ld_o:
        assert float(ld_o[k].detach()) == g['losses'][k], k
    # render-only path (target_d=None -> 256 uniform samples)
    o3 = ora.render_rays(rays_o, rays_d, None, n256)
    assert digest(o3['rgb']) == g['render']['rgb'] and digest(o3['depth']) == g['render']['depth']


def test_pose_roundtrip_like_frame_assert():
    """slam/common/frame.py:40-43: |pose - from_matrix(pose).matrix()| < 1e-3, for the
    matrix the reference's own __main__ check uses (opt_pose.py:112-124)."""
    from xrdslam_b200.opt_pose import OptimizablePose
    before = torch.tensor([[-0.955421, 0.119616, -0.269932, 2.655830],
                           [0.295248, 0.388339, -0.872939, 2.981598],
                           [0.000408, -0.913720, -0.406343, 1.368648],
                           [0.000000, 0.000000, 0.000000, 1.000000]])
    for rep in ('axis_angle', 'quat'):
        for sep in (True, False):
            p = OptimizablePose.from_matrix(before, separate_LR=sep, rot_rep=rep)
            assert torch.allclose(before, p.matrix().detach(), atol=1e-3)
    # and against the oracle's restatement of the pytorch3d functions
    from oracle import transforms_restated as tr
    from xrdslam_b200 import transforms as mine
    q = mine.matrix_to_quaternion(before[:3, :3])
    assert torch.allclose(q, tr.matrix_to_quaternion(before[:3, :3]), atol=1e-6)
    assert torch.allclose(mine.quaternion_to_matrix(q), tr.quaternion_to_matrix(q), atol=1e-6)
    assert torch.allclose(mine.quaternion_to_axis_angle(q), tr.quaternion_to_axis_angle(q),
                          atol=1e-6)


def test_cabi_exports_every_declared_symbol():
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, 'include', 'xrdslam_b200.h')).read()
    declared = set(re.findall(r'\b(xrd_[a-z0-9_]+)\s*\(', hdr))
    assert declared, 'no declarations parsed'
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in the header but not exported'
        assert name in _cabi.SYMBOLS, f'{name} has no ctypes signature'
    assert lib.xrd_abi_version() == 1


def test_linspace_matches_torch():
    """xrd_linspace_f32 is ATen's *scalar* formula.  torch's vectorised CPU path adds the
    lane offset to a per-vector base, so some elements differ in the last bit depending on
    the host's SIMD width -- the plugin therefore always passes torch.linspace tables to the
    kernel (bit-identical to the reference on the same host); the C function serves C callers."""
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    for (a, b, n) in [(0.0, 5.0, 32), (-0.1, 0.1, 11), (0.0, 5.0, 11), (0.0, 5.0, 256),
                      (0.01, 7.3, 33), (1.0, 1.0, 1), (-2.5, 9.75, 48)]:
        out = (C.c_float * n)()
        assert lib.xrd_linspace_f32(a, b, n, out) == 0
        mine = np.frombuffer(out, dtype=np.float32)
        ref = torch.linspace(a, b, n).numpy()
        ulp = np.spacing(np.maximum(np.abs(ref), np.float32(abs(b - a) / 8)))
        assert np.all(np.abs(mine - ref) <= 2 * ulp), (a, b, n)
        assert mine[0] == ref[0] and mine[-1] == ref[-1]


def test_hashgrid_layout_matches_oracle():
    from oracle.tcnn_restated import hashgrid_level_table
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    for desired, log2_t in [(325, 16), (512, 19), (128, 14), (2048, 19)]:
        pls = np.exp2(np.log2(desired / 16) / 15)
        g = _cabi.XrdHashGrid()
        assert lib.xrd_hashgrid_layout(C.byref(g), 16, log2_t, 16,
                                       float(np.float32(pls))) == 0
        t = hashgrid_level_table(16, 2, log2_t, 16, pls)
        assert g.n_entries == t['n_entries']
        for l in range(16):
            assert g.scale[l] == t['scale'][l] and g.resolution[l] == t['resolution'][l]
            assert g.size[l] == t['size'][l] and g.offset[l] == t['offset'][l]
            assert bool(g.hashed[l]) == bool(t['hashed'][l])


def test_model_refuses_cpu():
    """No CPU fallback: the product path fails loudly without a CUDA device."""
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.joint_encoding import JointEncodingConfig
    m = JointEncodingConfig().setup(camera=Camera(320., 320., 319.5, 239.5, 640, 480),
                                    bounding_box=BOUND)
    ro, rd, ts, td, _ = make_rays(8)
    with pytest.raises(RuntimeError):
        m(dict(rays_o=ro, rays_d=rd, target_s=ts, target_d=td, first=True))


def test_synthetic_scene_and_host_sampling():
    from xrdslam_b200.common import get_rays, get_samples
    from xrdslam_b200.synthetic import make_sequence
    cam, poses, frames = make_sequence(2, width=120, height=90)
    rgb, depth = frames[0]
    assert rgb.shape == (90, 120, 3) and depth.shape == (90, 120)
    assert 0.005 < (depth == 0).mean() < 0.05 and depth.max() < 10
    idx = torch.arange(0, 50) * 7
    ro, rd, d, c = get_samples(cam, 50, torch.from_numpy(poses[0]), depth, rgb, 'cpu',
                               Hedge=5, Wedge=5, indices=idx)
    assert ro.shape == (50, 3) and d.shape == (50, 1) and c.shape == (50, 3)
    # pixel (i,j) bookkeeping: row-major inside the cropped window
    w = 120 - 10
    jj, ii = idx // w + 5, idx % w + 5
    assert np.allclose(d.reshape(-1).numpy(), depth[jj.numpy(), ii.numpy()])
    full_o, full_d = get_rays(cam, torch.from_numpy(poses[0]), 'cpu')
    assert torch.allclose(rd, full_d[jj, ii], atol=1e-6)


def test_nice_oracle_matches_golden_reference_vectors():
    """oracle/nice.py == vectors produced by the reference's ConvOnet (stage color)."""
    from helpers import load_golden_nice, nice_from_golden
    g = load_golden_nice()
    ora = nice_from_golden(g, 'oracle')
    t = lambda k: torch.from_numpy(g[k])
    for tag, is_mapping in (('map', True), ('trk', False)):
        ora.zero_grad()
        rays_o = t('rays_o').requires_grad_(True)
        rays_d = t('rays_d').requires_grad_(True)
        out, ld, tot = ora.step(rays_o, rays_d, t('target_s'), t('target_d'), is_mapping, 'color')
        tot.backward()
        assert np.array_equal(out['rgb'].detach().numpy(), g[tag + '.rgb'])
        assert np.array_equal(out['depth'].detach().numpy(), g[tag + '.depth'])
        assert np.array_equal(out['uncertainty'].detach().numpy(), g[tag + '.uncertainty'])
        got = [float(ld['depth_loss'].detach()), float(ld['rgb_loss'].detach())]
        assert np.allclose(got, g[tag + '.losses'], rtol=1e-7, atol=0)
        assert np.allclose(rays_o.grad.numpy(), g[tag + '.d_rays_o'], rtol=1e-5, atol=1e-7)
        assert np.allclose(ora.color.B.grad.numpy(), g[tag + '.d_B'], rtol=1e-5, atol=1e-6)
        assert np.allclose(ora.color.pts[3].weight.grad.numpy(), g[tag + '.d_pts3_w'],
                           rtol=1e-5, atol=1e-6)
        gc = ora.grids['grid_color'].grad
        assert abs(float(gc.double().norm()) - float(g[tag + '.d_grid_color_norm'])) \
            <= 1e-6 * float(g[tag + '.d_grid_color_norm'])


NICE_COARSE_BOUND = np.array([[-2.0, 2.0], [-2.5, 2.0], [-2.0, 2.3]])
NICE_BOUND = np.array([[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]])
OFFICE0_BOUND = np.array([[-5.5, 5.9], [-6.7, 5.4], [-4.7, 5.3]])


def _nice_rays(R, seed):
    g = torch.Generator().manual_seed(seed)
    rays_o = (torch.rand(R, 3, generator=g) - 0.5) * 0.5
    rays_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    td = torch.rand(R, 1, generator=g) * 1.5 + 0.3
    td[3::7] = 0
    ts = torch.rand(R, 3, generator=g)
    return rays_o, rays_d, ts, td


def nice_coarse_case():
    """Seeded oracle with the coarse level: coarse grid x 30 and biases + 0.05 (non-trivial
    occupancies), 50 rays."""
    from oracle.nice import NiceOracle
    torch.manual_seed(3)  # fc_c layers keep torch's default init
    ora = NiceOracle(NICE_COARSE_BOUND, coarse=True, seed=3)
    with torch.no_grad():
        ora.grids['grid_coarse'].mul_(30)
        for lin in list(ora.coarse.pts) + [ora.coarse.out]:
            lin.bias.add_(0.05)
    return ora, _nice_rays(50, 4)


def test_nice_oracle_coarse_stage_matches_reference_class_live(one_thread):
    """Stage 'coarse' (MLP_no_xyz on the 2 m grid over the doubled bound, 32 uniform samples,
    no depth guidance): the reference's own ConvOnet(coarse=True) on the same parameters vs
    oracle/nice.py, outputs, loss and the coarse-grid gradient bit-identical."""
    g = load_golden_json('reference_cpu.json')['nice_coarse']
    ora, (rays_o, rays_d, ts, td) = nice_coarse_case()
    assert list(ora.grids['grid_coarse'].shape) == g['grid_coarse_shape']
    assert digest(ora.coarse_bound) == g['coarse_bound']
    out_o = ora.render(rays_o, rays_d, td, 'coarse')
    assert out_o['z_vals'].shape == (50, 32)
    for k in ('depth', 'uncertainty'):
        assert digest(out_o[k]) == g['out'][k], k
    ld_o = ora.loss_dict(out_o, ts, td, True, 'coarse')
    assert set(ld_o) == {'depth_loss'}
    assert float(ld_o['depth_loss'].detach()) == g['depth_loss']
    ld_o['depth_loss'].backward()
    assert digest(ora.grids['grid_coarse'].grad) == g['d_grid_coarse']


def nice_case():
    """Seeded oracle, grids x 30 (non-trivial occupancies), 64 rays."""
    from oracle.nice import NiceOracle
    torch.manual_seed(1)  # fc_c layers keep torch's default init
    ora = NiceOracle(NICE_BOUND, seed=1)
    with torch.no_grad():
        for k in ora.grids:
            ora.grids[k].mul_(30)
    return ora, _nice_rays(64, 2)


def test_nice_oracle_matches_reference_class_live(one_thread):
    """The reference's ConvOnet on the same parameters: stages color, middle and fine,
    outputs and mapping / tracking losses bit-identical."""
    from oracle.nice import NiceOracle
    g = load_golden_json('reference_cpu.json')['nice']
    ora, (rays_o, rays_d, ts, td) = nice_case()
    assert digest(ora.bound) == g['bound']
    out_o = ora.render(rays_o, rays_d, td, 'color')
    for k in ('rgb', 'depth', 'uncertainty'):
        assert digest(out_o[k]) == g['color']['out'][k], k
    for m in (True, False):
        ld_o = ora.loss_dict(out_o, ts, td, m, 'color')
        ref = g['color']['losses'][str(m)]
        assert set(ld_o) == set(ref)
        for k in ld_o:
            assert float(ld_o[k].detach()) == ref[k], (m, k)
    # stages middle / fine are CUDA-only in the reference (Q5: device = f'cuda:{p.get_device()}');
    # the stored values come from its own class run on the host with that string neutralised
    for stage in ('middle', 'fine'):
        out_o = ora.render(rays_o, rays_d, td, stage)
        for k in ('depth', 'uncertainty'):
            assert digest(out_o[k]) == g[stage]['out'][k], (stage, k)
        for m in (True, False):
            ld_o = ora.loss_dict(out_o, ts, td, m, stage)
            ref = g[stage]['losses'][str(m)]
            assert set(ld_o) == set(ref)
            for k in ld_o:
                assert float(ld_o[k].detach()) == ref[k], (stage, m, k)
    # the reference's grid-shape hazard (SURVEY Q2) at the default office0 bound
    assert g['office0_shapes'] == {'grid_middle': [1, 32, 31, 37, 35],
                                   'grid_fine': [1, 32, 63, 75, 71]}
    o2 = NiceOracle(OFFICE0_BOUND)
    for k, shp in g['office0_shapes'].items():
        assert list(o2.grids[k].shape) == shp, k


@pytest.mark.parametrize('tag,is_mapping', [('map', True), ('trk', False)])
def test_pointslam_oracle_matches_golden_reference_vectors(tag, is_mapping):
    """oracle/pointslam.py vs the reference's ConvOnet2 + NeuralPointCloud outputs and
    gradients (tests/golden/make_golden.py:pointslam; faiss -> exact kNN)."""
    from helpers import load_golden_pointslam, max_abs, pointslam_from_golden, rel_err
    g = load_golden_pointslam()
    ora = pointslam_from_golden(g, 'oracle')
    ro = torch.from_numpy(g['rays_o']).requires_grad_(True)
    rd = torch.from_numpy(g['rays_d']).requires_grad_(True)
    td = torch.from_numpy(g['target_d'])
    out = ora.render(ro, rd, td, torch.from_numpy(g['radius']), torch.from_numpy(g['rand_feat']))
    loss = ora.loss(out, td, is_mapping)
    loss.backward()
    assert torch.equal(out['valid_ray_mask'], torch.from_numpy(g[tag + '.valid']))
    assert max_abs(out['depth'], g[tag + '.depth']) < 1e-6
    assert max_abs(out['uncertainty'], g[tag + '.uncertainty']) < 1e-7
    assert abs(float(loss.detach()) - float(g[tag + '.loss'])) < 1e-5 * max(1, abs(float(loss.detach())))
    assert rel_err(ora.geo_feats.grad, g[tag + '.d_geo_feats']) < 1e-5
    # ray grads go through 1 / (D + 1e-10) weights: fp32 op-order noise ~1e-5 relative
    assert rel_err(ro.grad, g[tag + '.d_rays_o']) < 1e-4
    assert rel_err(rd.grad, g[tag + '.d_rays_d']) < 1e-4


def test_exact_knn_sentinels_and_ties():
    from oracle.pointslam import FLT_MAX, exact_knn
    cloud = torch.tensor([[0., 0, 0], [1, 0, 0], [-1, 0, 0]])
    D, I = exact_knn(cloud, torch.zeros(1, 3), 8)
    assert I[0].tolist() == [0, 1, 2, -1, -1, -1, -1, -1]  # tie 1 vs 2 -> lower id first
    assert D[0, 3:].eq(FLT_MAX).all() and D[0, :3].tolist() == [0.0, 1.0, 1.0]


@pytest.mark.parametrize('tag,is_mapping', [('cmap', True), ('ctrk', False)])
def test_pointslam_oracle_color_stage_matches_golden(tag, is_mapping):
    """Stage 'color' of oracle/pointslam.py vs the reference ConvOnet2 (MLP_color,
    MLP_col_neighbor, colour compositing + loss) incl. every colour-decoder gradient."""
    from helpers import (load_golden_pointslam, max_abs, oracle_cdec_grads,
                         pointslam_from_golden, rel_err)
    g = load_golden_pointslam()
    ora = pointslam_from_golden(g, 'oracle')
    ro = torch.from_numpy(g['rays_o']).requires_grad_(True)
    rd = torch.from_numpy(g['rays_d']).requires_grad_(True)
    td, ts = torch.from_numpy(g['target_d']), torch.from_numpy(g['target_s'])
    out = ora.render(ro, rd, td, torch.from_numpy(g['radius']), torch.from_numpy(g['rand_feat']),
                     'color', torch.from_numpy(g['rand_feat_color']))
    ld = ora.loss_dict(out, td, ts, is_mapping)
    sum(ld.values()).backward()
    assert max_abs(out['depth'], g[tag + '.depth']) < 1e-6
    assert max_abs(out['rgb'], g[tag + '.rgb']) < 1e-5
    assert abs(float(ld['geo_loss'].detach()) - float(g[tag + '.losses'][0])) < 1e-5 * max(1, float(g[tag + '.losses'][0]))
    assert abs(float(ld['rgb_loss'].detach()) - float(g[tag + '.losses'][1])) < 1e-4 * max(1, float(g[tag + '.losses'][1]))
    assert rel_err(ora.geo_feats.grad, g[tag + '.d_geo_feats']) < 1e-4
    assert rel_err(ora.col_feats.grad, g[tag + '.d_col_feats']) < 1e-4
    assert rel_err(ro.grad, g[tag + '.d_rays_o']) < 1e-3
    assert rel_err(rd.grad, g[tag + '.d_rays_d']) < 1e-3
    for k, v in oracle_cdec_grads(ora).items():
        assert rel_err(v, g[tag + '.d_cdec.' + k]) < 1e-3, k


def test_stage_schedulers_and_stage_selection():
    """B4: LambdaLR factors = stage learning rates; stage boundaries of nice / point."""
    from xrdslam_b200.schedulers import (LRconfig, NiceSLAMSchedulerConfig,
                                         PointSLAMSchedulerConfig)
    p = torch.nn.Parameter(torch.zeros(3))
    opt = torch.optim.Adam([p], lr=5.0)  # lr = factor 5.0 (mapping_lr_first_factor)
    cfg = NiceSLAMSchedulerConfig(coarse=False, stage_lr=LRconfig(0.0, 0.1, 0.005, 0.002),
                                  max_steps=10)
    sch = cfg.setup().get_scheduler(opt, 5.0)
    lrs = []
    for _ in range(10):
        lrs.append(opt.param_groups[0]['lr'])
        opt.step()
        sch.step()
    assert np.allclose(lrs, [0.5] * 5 + [0.025] * 2 + [0.01] * 3)
    pc = PointSLAMSchedulerConfig(start_lr=0.03, end_lr=0.005, max_steps=10, geo_iter_ratio=0.4)
    assert [pc.setup().factor(s) for s in (0, 4, 5, 9)] == [0.03, 0.03, 0.005, 0.005]


def test_remap_linear_bilinear_and_border():
    from xrdslam_b200.keyframe_selection import remap_linear
    img = torch.arange(12.).reshape(3, 4)
    uv = torch.tensor([[0., 0.], [1.5, 0.5], [3.0, 2.0], [3.5, 2.0], [-0.5, 0.], [1.03, 1.0]])
    out = remap_linear(img, uv)
    # 1.03 -> 33/32: OpenCV's 1/32-pixel coordinate quantisation
    assert torch.allclose(out, torch.tensor([0., 3.5, 11., 5.5, 0., 5. + 1. / 32]))


def test_pose_matrices_batched_equals_per_frame():
    """opt_pose.pose_matrices (one batched evaluation for the window) == stacking
    OptimizablePose.matrix() per frame, values and gradients, both rotation reps, including
    the identity-rotation branch and a detached (fixed) frame."""
    from xrdslam_b200.opt_pose import OptimizablePose, pose_matrices
    from xrdslam_b200.transforms import quaternion_to_matrix
    g = torch.Generator().manual_seed(0)
    for rep in ('axis_angle', 'quat'):
        ps = []
        for k in range(5):
            M = torch.eye(4)
            if k != 2:  # frame 2 keeps the identity rotation
                q = torch.randn(4, generator=g)
                M[:3, :3] = quaternion_to_matrix(q / q.norm())
            M[:3, 3] = torch.randn(3, generator=g)
            ps.append(OptimizablePose.from_matrix(M, rot_rep=rep))
        A = torch.stack([p.matrix() for p in ps])
        B = pose_matrices(ps, [True, False, False, False, False])
        assert torch.allclose(A, B, atol=1e-7)
        W = torch.randn(5, 4, 4, generator=g)
        params = [q for p in ps[1:] for q in p.parameters()]
        # the identity-rotation frame: matrix() returns eye(3) without touching data_r
        ga = torch.autograd.grad((A * W).sum(), params, allow_unused=True)
        gb = torch.autograd.grad((B * W).sum(), params, allow_unused=True)
        zero = lambda x, p: torch.zeros_like(p) if x is None else x
        for a, b, p in zip(ga, gb, params):
            assert torch.allclose(zero(a, p), zero(b, p), atol=1e-6)
        # the fixed frame receives no gradient through the batched form
        g0 = torch.autograd.grad((pose_matrices(ps, [True] + [False] * 4) * W).sum(),
                                 list(ps[0].parameters()), allow_unused=True)
        assert all(x is None or x.abs().sum() == 0 for x in g0)


def test_dynamic_radius_sobel_matches_scipy():
    """point_slam.sobel_magnitude restates skimage.filters.sobel_h/_v on rgb2gray
    (scipy.ndimage.convolve, mode='reflect'); the radius map follows interp1d's knots."""
    from scipy import ndimage as ndi
    from xrdslam_b200.point_slam import sobel_magnitude
    rng = np.random.default_rng(0)
    rgb = rng.random((37, 53, 3)).astype(np.float32)
    gray = rgb.astype(np.float64) @ np.array([0.2125, 0.7154, 0.0721])
    H = np.array([[1, 2, 1], [0, 0, 0], [-1, -2, -1]]) / 4.0
    mag = np.sqrt(ndi.convolve(gray, H)**2 + ndi.convolve(gray, H.T)**2)
    assert np.abs(sobel_magnitude(torch.from_numpy(rgb)).numpy() - mag).max() < 1e-12
    from scipy.interpolate import interp1d
    thr, rmax, rmin = 0.15, 0.08, 0.02
    m = np.clip(mag, 0.0, thr)
    ref = interp1d([0, 0.01, thr], [rmax, rmax, rmin])(m)
    mt = torch.from_numpy(m)
    mine = torch.where(mt <= 0.01, torch.full_like(mt, rmax), rmax + (mt - 0.01) * (rmin - rmax) / (thr - 0.01))
    assert np.abs(mine.numpy() - ref).max() < 1e-12


def test_keyframe_selection_overlap_on_host():
    """common.py:343-426: keyframes that see the current frame's back-projected samples are
    kept, a keyframe looking the other way is dropped (host tensors: the torch branch of
    rays_from_poses)."""
    from xrdslam_b200.frame import Frame
    from xrdslam_b200.keyframe_selection import keyframe_selection_overlap
    from xrdslam_b200.synthetic import CENTRE, look_at, make_camera, render_frame
    torch.manual_seed(0)
    np.random.seed(0)
    cam = make_camera(160, 120)
    eye = CENTRE + np.array([0.5, 0.0, 0.1])
    tgt = CENTRE + np.array([-1.5, 0.3, -0.2])
    poses = [look_at(eye, tgt),                                   # current view
             look_at(eye + np.array([0.1, 0.05, 0.0]), tgt),      # nearly the same view
             look_at(eye, eye + (eye - tgt)),                     # looks the opposite way
             look_at(eye + np.array([0.0, -0.2, 0.05]), tgt)]     # overlapping view
    frames = []
    for k, p in enumerate(poses):
        rgb, depth = render_frame(cam, p, seed=k)
        frames.append(Frame(k, rgb, depth, init_pose=p, rot_rep='quat'))
    sel = keyframe_selection_overlap(cam, frames[0], frames[1:], k=3, device='cpu')
    ids = sorted(f.fid for f in sel)
    assert ids == [1, 3], ids
    assert len(keyframe_selection_overlap(cam, frames[0], frames[1:], k=1, device='cpu')) == 1


FRONTEND_KW = (dict(Hedge=0, Wedge=0), dict(Hedge=7, Wedge=11),
               dict(Hedge=3, Wedge=5, depth_filter=True, return_index=True))


def test_host_frontend_bit_identical_to_reference_functions(one_thread):
    """common.get_samples / get_rays / get_camera_rays (host tensors) against the reference's
    own slam.common.common / slam.utils.utils functions under the same torch seed: identical
    pixel draws, rays, depth / colour gathers and index outputs (rows A1-A5)."""
    import xrdslam_b200.common as mc
    from xrdslam_b200.synthetic import make_sequence
    g = load_golden_json('reference_cpu.json')['frontend']
    cam, poses, fr = make_sequence(1, width=160, height=120)
    c2w = torch.from_numpy(poses[0])
    rgb, depth = fr[0]
    for kw, ref in zip(FRONTEND_KW, g['get_samples']):
        torch.manual_seed(5)
        b = mc.get_samples(cam, 333, c2w, depth, rgb, device='cpu', **kw)
        assert [digest(y) for y in b] == ref, kw
    assert [digest(y) for y in mc.get_rays(cam, c2w, 'cpu')] == g['get_rays']
    assert digest(mc.get_camera_rays(120, 160, cam.fx, cam.fy, cam.cx, cam.cy)) == g['get_camera_rays']


def optimizers_case(mod):
    A = mod.AdamOptimizerConfig
    torch.manual_seed(0)
    p = {'a': [torch.nn.Parameter(torch.randn(5))], 'pose': [torch.nn.Parameter(torch.randn(3))]}
    cfg = {'a': {'optimizer': A(lr=1e-2, weight_decay=1e-6, betas=(0.9, 0.99)), 'scheduler': None},
           'pose': {'optimizer': A(lr=1e-3, accum_step=5), 'scheduler': None}}
    opt = mod.Optimizers(cfg, p)
    g = torch.Generator().manual_seed(1)
    for step in range(12):
        opt.zero_grad_all()
        for k in p:
            gr = torch.randn(p[k][0].shape, generator=g)
            p[k][0].grad = gr if p[k][0].grad is None else p[k][0].grad + gr
        opt.optimizer_step_all(step=step)
    return {k: digest(v[0]) for k, v in p.items()}


def test_optimizers_match_reference_engine_incl_accum_step():
    """xrdslam_b200.optimizers.Optimizers (zero_grad_all / optimizer_step_all, accum_step = 5,
    weight decay, custom betas) against the reference's own slam.engine.optimizers on host
    parameters: bit-identical after 12 steps (rows B2 / B3, Q11)."""
    import xrdslam_b200.optimizers as mo
    assert optimizers_case(mo) == load_golden_json('reference_cpu.json')['optimizers']


def keyframe_case():
    from xrdslam_b200.frame import Frame
    from xrdslam_b200.synthetic import CENTRE, look_at, make_camera, render_frame
    cam = make_camera(160, 120)
    eye = CENTRE + np.array([0.5, 0.0, 0.1])
    tgt = CENTRE + np.array([-1.5, 0.3, -0.2])
    rng = np.random.default_rng(0)
    poses = [look_at(eye, tgt)] + [look_at(eye + rng.normal(size=3) * 0.3, tgt + rng.normal(size=3) * 0.8)
                                   for _ in range(7)] + [look_at(eye, eye + (eye - tgt))]
    frames = []
    for k, p in enumerate(poses):
        rgb, depth = render_frame(cam, p, seed=k)
        frames.append(Frame(k, rgb, depth, init_pose=p, rot_rep='quat'))
    return cam, frames


def test_keyframe_selection_overlap_matches_reference_function():
    """Same seeds -> the same keyframes in the same order as the reference's own
    slam.common.common.keyframe_selection_overlap (host tensors)."""
    from xrdslam_b200.keyframe_selection import keyframe_selection_overlap
    g = load_golden_json('reference_cpu.json')['keyframes']
    cam, frames = keyframe_case()
    for k in (2, 4, 8):
        torch.manual_seed(3)
        np.random.seed(3)
        b = keyframe_selection_overlap(cam, frames[0], frames[1:], k, device='cpu')
        assert [f.fid for f in b] == g[str(k)], k
    assert 8 not in [f.fid for f in b]  # the frame looking the other way has no overlap


def test_convonet_load_pretrain_key_mapping(tmp_path):
    """conv_onet.py:293-322: 'decoder.coarse.*' of the middle_fine checkpoint feeds the MIDDLE
    decoder, 'decoder.fine.*' the fine decoder, 'decoder.*' of the coarse checkpoint the coarse
    decoder; encoder keys are dropped; a set path must load."""
    import warnings
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.conv_onet import MLP, MLP_no_xyz, ConvOnetConfig
    torch.manual_seed(0)
    mid, fine, coarse = MLP('middle', 32, False), MLP('fine', 64, False), MLP_no_xyz('coarse', 32)
    ck = {'model': {'encoder.x': torch.zeros(1)}}
    ck['model'].update({'decoder.coarse.' + k: v.clone() for k, v in mid.state_dict().items()})
    ck['model'].update({'decoder.fine.' + k: v.clone() for k, v in fine.state_dict().items()})
    torch.save(ck, tmp_path / 'middle_fine.pt')
    ck2 = {'model': {'decoder.' + k: v.clone() for k, v in coarse.state_dict().items()}}
    ck2['model']['encoder.y'] = torch.zeros(1)
    torch.save(ck2, tmp_path / 'coarse.pt')
    cam = Camera(320., 320., 319.5, 239.5, 640, 480)
    bound = np.array([[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]])
    with warnings.catch_warnings():
        warnings.simplefilter('error')  # both checkpoints given: nothing stays random
        m = ConvOnetConfig(coarse=True, pretrained_decoders_coarse=tmp_path / 'coarse.pt',
                           pretrained_decoders_middle_fine=tmp_path / 'middle_fine.pt'
                           ).setup(camera=cam, bounding_box=bound)
    for got, ref in ((m.decoder.middle_decoder, mid), (m.decoder.fine_decoder, fine),
                     (m.decoder.coarse_decoder, coarse)):
        for k, v in ref.state_dict().items():
            assert torch.equal(got.state_dict()[k], v), k
    assert 'grid_coarse' in m.grids and 'grid_coarse' in m.get_param_groups()
    with pytest.warns(RuntimeWarning, match='randomly initialised'):
        ConvOnetConfig().setup(camera=cam, bounding_box=bound)
    with pytest.raises(Exception):
        ConvOnetConfig(pretrained_decoders_middle_fine=tmp_path / 'missing.pt').setup(
            camera=cam, bounding_box=bound)


PIXEL_GRAD_KW = (dict(), dict(Hedge=4, Wedge=6, depth_limit=3.0))


def test_pixel_grad_sampler_bit_identical_to_reference_function(one_thread):
    """common.get_sample_uv_with_grad / get_samples_with_pixel_grad (Point-SLAM colour-gradient
    pixels, default mapping_pixels_based_on_color_grad = 1000) against the reference's own
    functions under the same numpy seed.  skimage is handed to the reference as the
    scipy.ndimage restatement the mirror uses -- "parity unpinned" at rgb2gray / sobel; the
    selection logic (argpartition top ratio*n, region mask, np.random.choice, depth filter, ray
    construction) is the reference's own code."""
    import xrdslam_b200.common as mc
    from xrdslam_b200.synthetic import make_sequence
    g = load_golden_json('reference_cpu.json')['pixel_grad']
    cam, poses, fr = make_sequence(1, width=160, height=120)
    c2w = torch.from_numpy(poses[0])
    rgb, depth = fr[0]
    np.random.seed(3)
    b = mc.get_sample_uv_with_grad(5, 115, 7, 150, 40, rgb)
    assert digest(b) == g['uv'] and len(set(b.tolist())) == 40
    for kw, ref in zip(PIXEL_GRAD_KW, g['samples']):
        np.random.seed(11)
        rb = mc.get_samples_with_pixel_grad(cam, 60, c2w, depth, rgb, device='cpu', **kw)
        assert len(rb) == 6
        assert [digest(y) for y in rb] == ref, kw


def test_convonet2_load_pretrain(tmp_path):
    """conv_onet_pointslam.py:228-246: geometry decoder <- 'decoder.coarse.*' (strict=False)."""
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.conv_onet_pointslam import ConvOnet2Config
    cam = Camera(320., 320., 319.5, 239.5, 640, 480)
    with pytest.warns(RuntimeWarning, match='randomly initialised'):
        src = ConvOnet2Config().setup(camera=cam)
    sd = src.decoder.geo_decoder.state_dict()
    torch.manual_seed(3)
    ck = {'model': {'decoder.coarse.' + k: torch.randn_like(v) for k, v in sd.items()}}
    ck['model']['decoder.fine.fc_c.0.weight'] = torch.zeros(32, 64)
    ck['model']['encoder.z'] = torch.zeros(2)
    torch.save(ck, tmp_path / 'middle_fine.pt')
    m = ConvOnet2Config(pretrained_decoders_middle_fine=tmp_path / 'middle_fine.pt').setup(camera=cam)
    for k, v in m.decoder.geo_decoder.state_dict().items():
        assert torch.equal(v, ck['model']['decoder.coarse.' + k]), k
    torch.save({'model': {'encoder.z': torch.zeros(2)}}, tmp_path / 'bad.pt')
    with pytest.raises(RuntimeError):
        ConvOnet2Config(pretrained_decoders_middle_fine=tmp_path / 'bad.pt').setup(camera=cam)
