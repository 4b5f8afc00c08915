"""Generate the committed golden vectors by running the REFERENCE's own classes
(imported from a reference checkout through oracle/ref_harness.py) on CPU.

    python tests/golden/make_golden.py [coslam nice pointslam reference_cpu]
    python tests/golden/make_golden.py vox_grid     # on a B200, after oracle/build_ref.py

Needs the reference checkout (XRDSLAM_REFERENCE); the tests only read what this writes, so
they run without it.  reference_cpu needs oracle/_ref/svo.so, vox_grid oracle/_ref/grid.so
(both built by oracle/build_ref.py).  The tinycudann
encodings inside the reference model are the restated ones (parity unpinned there, see
DESIGN.md section 2); everything else -- sampling, decoders, sdf2weights, raw2outputs, losses,
smoothness -- is the reference's code, executed unmodified.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from helpers import BOUND, make_rays  # noqa: E402
from oracle import ref_harness  # noqa: E402


def coslam(R=96, seed=7):
    bb = torch.from_numpy(BOUND)
    ref = ref_harness.ref_joint_encoding(bb)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        ref.embed_fn.params.copy_(
            (torch.rand(ref.embed_fn.params.shape, generator=g) * 2 - 1) * 0.3)
        for seq in (ref.decoder.sdf_net.model, ref.decoder.color_net.model):
            for lin in (seq[0], seq[2]):
                lin.weight.copy_(torch.randn(lin.weight.shape, generator=g) /
                                 np.sqrt(lin.weight.shape[1]))
    rays_o, rays_d, ts, td, noise = make_rays(R, seed=seed)
    rays_o.requires_grad_(True)
    rays_d.requires_grad_(True)
    # the reference draws torch.rand(z_vals.shape) then (mapping) rand(3), rand(1,1,1,3)
    torch.manual_seed(seed)
    noise = torch.rand(R, 43)
    r1 = torch.rand(3)
    r2 = torch.rand((1, 1, 1, 3))
    torch.manual_seed(seed)
    inp = dict(rays_o=rays_o, rays_d=rays_d, target_s=ts, target_d=td, first=False)
    out = ref(inp)
    ld = ref.get_loss_dict(out, inp, True, 0)
    total = sum(ld.values())
    total.backward()
    sd = ref.state_dict()
    np.savez_compressed(
        os.path.join(HERE, 'coslam_map_step.npz'),
        rays_o=rays_o.detach().numpy(), rays_d=rays_d.detach().numpy(),
        target_s=ts.numpy(), target_d=td.numpy(), noise=noise.numpy(),
        smooth_rand=torch.cat([r1, r2.reshape(3)]).numpy(),
        w_sdf0=sd['decoder.sdf_net.model.0.weight'].numpy(),
        w_sdf1=sd['decoder.sdf_net.model.2.weight'].numpy(),
        w_col0=sd['decoder.color_net.model.0.weight'].numpy(),
        w_col1=sd['decoder.color_net.model.2.weight'].numpy(),
        table_seed=np.int64(seed),  # the 6.5 MB table is regenerated from the seed
        table_checksum=np.float64(sd['embed_fn.params'].double().sum().item()),
        z_vals=out['z_vals'].detach().numpy(), raw=out['raw'].detach().numpy(),
        rgb=out['rgb'].detach().numpy(), depth=out['depth'].detach().numpy(),
        depth_var=out['depth_var'].detach().numpy(), acc=out['acc_map'].detach().numpy(),
        losses=np.array([float(ld[k].detach()) for k in
                         ('rgb_loss', 'depth_loss', 'sdf_loss', 'fs_loss', 'smooth_loss')]),
        d_rays_o=rays_o.grad.numpy(), d_rays_d=rays_d.grad.numpy(),
        d_w_sdf0=ref.decoder.sdf_net.model[0].weight.grad.numpy(),
        d_w_col1=ref.decoder.color_net.model[2].weight.grad.numpy(),
        d_table_norm=np.float64(ref.embed_fn.params.grad.double().norm().item()),
        d_table_nnz=np.int64((ref.embed_fn.params.grad != 0).sum().item()),
        d_table_head=ref.embed_fn.params.grad[:4096].numpy())
    print('wrote coslam_map_step.npz')


def nice(R=120, seed=3):
    """Reference ConvOnet (slam/models/conv_onet.py), stage 'color' -- the one stage that
    runs on CPU (SURVEY Q5) -- mapping and tracking losses, with gradients."""
    bound = np.array([[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]])
    torch.manual_seed(seed)
    ref = ref_harness.ref_conv_onet(bound)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for i, k in enumerate(sorted(ref.grid_c)):
            # regenerated from the seed by the tests (keeps the fixture small)
            gg = torch.Generator().manual_seed(1000 + i)
            ref.grid_c[k] = (torch.randn(ref.grid_c[k].shape, generator=gg) * 0.3
                             ).requires_grad_(True)
        for dec in (ref.decoder.middle_decoder, ref.decoder.fine_decoder,
                    ref.decoder.color_decoder):
            dec.embedder._B.mul_(0.2)
            for lin in list(dec.fc_c) + list(dec.pts_linears) + [dec.output_linear]:
                lin.bias.copy_(torch.randn(lin.bias.shape, generator=g) * 0.1)
    rays_o = ((torch.rand(R, 3, generator=g) - 0.5) * 0.6).requires_grad_(True)
    rays_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g),
                                           dim=-1).requires_grad_(True)
    td = torch.rand(R, 1, generator=g) * 1.5 + 0.3
    td[3::7] = 0
    ts = torch.rand(R, 3, generator=g)
    blob = dict(bound=bound, rays_o=rays_o.detach().numpy(), rays_d=rays_d.detach().numpy(),
                target_s=ts.numpy(), target_d=td.numpy())
    sd = ref.decoder.state_dict()
    for k, v in sd.items():
        blob['dec.' + k] = v.numpy()
    for k, v in ref.grid_c.items():
        blob[k + '.shape'] = np.array(v.shape)
        blob[k + '.checksum'] = np.float64(v.detach().double().sum().item())
    for tag, is_mapping in (('map', True), ('trk', False)):
        for t in [rays_o, rays_d] + list(ref.grid_c.values()) + list(ref.decoder.parameters()):
            t.grad = None
        inp = dict(rays_o=rays_o, rays_d=rays_d, target_s=ts, target_d=td, stage='color')
        out = ref(inp)
        ld = ref.get_loss_dict(out, inp, is_mapping, 'color')
        sum(ld.values()).backward()
        blob[tag + '.rgb'] = out['rgb'].detach().numpy()
        blob[tag + '.depth'] = out['depth'].detach().numpy()
        blob[tag + '.uncertainty'] = out['uncertainty'].detach().numpy()
        blob[tag + '.losses'] = np.array([float(ld['depth_loss'].detach()),
                                          float(ld['rgb_loss'].detach())])
        blob[tag + '.d_rays_o'] = rays_o.grad.numpy().copy()
        blob[tag + '.d_rays_d'] = rays_d.grad.numpy().copy()
        gcg = ref.grid_c['grid_color'].grad
        blob[tag + '.d_grid_color_norm'] = np.float64(gcg.double().norm().item())
        blob[tag + '.d_grid_color_slice'] = gcg[0, :, 10:14, 10:14, 10:14].numpy().copy()
        blob[tag + '.d_grid_middle_norm'] = np.float64(
            ref.grid_c['grid_middle'].grad.double().norm().item())
        cd = ref.decoder.color_decoder
        blob[tag + '.d_B'] = cd.embedder._B.grad.numpy().copy()
        blob[tag + '.d_pts3_w'] = cd.pts_linears[3].weight.grad.numpy().copy()
        blob[tag + '.d_fcc0_w'] = cd.fc_c[0].weight.grad.numpy().copy()
    np.savez_compressed(os.path.join(HERE, 'nice_color_step.npz'), **blob)
    print('wrote nice_color_step.npz')


def pointslam(R0=300, R=80, seed=11):
    """Reference ConvOnet2 (slam/models/conv_onet_pointslam.py) + NeuralPointCloud, stage
    'geometry', on CPU with the exact-kNN stand-in for faiss (oracle/ref_harness.py):
    point-adding, mapping and tracking losses with gradients."""
    torch.manual_seed(seed)
    ref = ref_harness.ref_conv_onet2()
    g = torch.Generator().manual_seed(seed)
    ro0 = torch.zeros(R0, 3)
    rd0 = torch.nn.functional.normalize(
        torch.randn(R0, 3, generator=g) * torch.tensor([0.3, 0.3, 0.05]) +
        torch.tensor([0, 0, -1.0]), dim=-1)
    d0 = torch.rand(R0, generator=g) * 0.5 + 1.5
    e = torch.zeros(0)
    ref.model_update(dict(batch_rays_o=ro0, batch_rays_d=rd0, batch_gt_depth=d0,
                          batch_gt_color=torch.rand(R0, 3, generator=g),
                          batch_dynamic_r=torch.full((R0,), 0.04),
                          batch_rays_o_grad=ro0[:0], batch_rays_d_grad=rd0[:0],
                          batch_gt_depth_grad=e, batch_gt_color_grad=torch.rand(0, 3),
                          batch_dynamic_r_grad=e))
    npc = ref.neural_point_cloud
    gd = ref.decoder.geo_decoder
    cd = ref.decoder.color_decoder
    with torch.no_grad():
        gd.embedder._B.mul_(0.05)
        for lin in list(gd.fc_c) + list(gd.pts_linears) + [gd.output_linear]:
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=g) * 0.1)
        npc.geo_feats.mul_(5.0)
        # colour decoder: moderate sin() arguments, non-zero biases, wider activations so the
        # softplus(beta=100) kinks are exercised
        cd.embedder._B.mul_(0.05)
        cd.embedder_rel_pos._B.mul_(0.3)
        for lin in list(cd.pts_linears) + [cd.output_linear]:
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=g) * 0.05)
        npc.col_feats.mul_(5.0)
    rays_o = (torch.randn(R, 3, generator=g) * 0.01).requires_grad_(True)
    rays_d = rd0[:R].clone().requires_grad_(True)
    td = (d0[:R] + torch.randn(R, generator=g) * 0.01).reshape(-1, 1)
    td[5::9] = 0
    radius = torch.rand(R, generator=g) * 0.08 + 0.04
    blob = dict(add_rays_d=rd0.numpy(), add_depth=d0.numpy(),
                cloud_pos=np.asarray(npc._cloud_pos, np.float32),
                geo_feats=npc.geo_feats.detach().numpy().copy(),
                rays_o=rays_o.detach().numpy(), rays_d=rays_d.detach().numpy(),
                target_d=td.numpy(), radius=radius.numpy())
    for k, v in gd.state_dict().items():
        blob['dec.' + k] = v.numpy().copy()
    for k, v in cd.state_dict().items():
        blob['cdec.' + k] = v.numpy().copy()
    blob['cdec.embedder._B'] = cd.embedder._B.numpy().copy()  # plain attribute, not in state_dict
    blob['col_feats'] = npc.col_feats.detach().numpy().copy()
    target_s = torch.rand(R, 3, generator=g)
    blob['target_s'] = target_s.numpy()
    for tag, is_mapping in (('map', True), ('trk', False)):
        for t in [rays_o, rays_d, npc.geo_feats] + list(gd.parameters()):
            t.grad = None
        inp = dict(rays_o=rays_o, rays_d=rays_d, target_d=td, target_s=torch.zeros(R, 3),
                   stage='geometry', batch_dynamic_r=radius)
        torch.manual_seed(777)  # the decoders' N(0, 0.01) features (Q6) = the draws below
        out = ref(inp)
        ld = ref.get_loss_dict(out, inp, is_mapping)
        ld['geo_loss'].backward()
        blob[tag + '.depth'] = out['depth'].detach().numpy()
        blob[tag + '.uncertainty'] = out['uncertainty'].detach().numpy()
        blob[tag + '.valid'] = out['valid_ray_mask'].numpy()
        blob[tag + '.loss'] = np.float32(ld['geo_loss'].item())
        blob[tag + '.d_geo_feats'] = npc.geo_feats.grad.numpy().copy()
        blob[tag + '.d_rays_o'] = rays_o.grad.numpy().copy()
        blob[tag + '.d_rays_d'] = rays_d.grad.numpy().copy()
    torch.manual_seed(777)  # geometry decoder draws first, then the colour decoder
    blob['rand_feat'] = torch.zeros(32).normal_(mean=0, std=0.01).numpy()
    blob['rand_feat_color'] = torch.zeros(32).normal_(mean=0, std=0.01).numpy()
    # stage 'color'
    for tag, is_mapping in (('cmap', True), ('ctrk', False)):
        ps = [rays_o, rays_d, npc.geo_feats, npc.col_feats] + list(cd.parameters())
        for t in ps:
            t.grad = None
        inp = dict(rays_o=rays_o, rays_d=rays_d, target_d=td, target_s=target_s, stage='color',
                   batch_dynamic_r=radius)
        torch.manual_seed(777)
        out = ref(inp)
        ld = ref.get_loss_dict(out, inp, is_mapping)
        sum(ld.values()).backward()
        blob[tag + '.depth'] = out['depth'].detach().numpy()
        blob[tag + '.rgb'] = out['rgb'].detach().numpy()
        blob[tag + '.losses'] = np.array([ld['geo_loss'].item(), ld['rgb_loss'].item()],
                                         np.float32)
        blob[tag + '.d_geo_feats'] = npc.geo_feats.grad.numpy().copy()
        blob[tag + '.d_col_feats'] = npc.col_feats.grad.numpy().copy()
        blob[tag + '.d_rays_o'] = rays_o.grad.numpy().copy()
        blob[tag + '.d_rays_d'] = rays_d.grad.numpy().copy()
        for k, v in cd.named_parameters():
            blob[tag + '.d_cdec.' + k] = v.grad.numpy().copy()
    # two files, each under 1 MB: inputs + stage 'geometry', and the stage 'color' outputs
    color = {k: v for k, v in blob.items() if k.startswith(('cmap.', 'ctrk.'))}
    np.savez_compressed(os.path.join(HERE, 'pointslam_geo_step.npz'),
                        **{k: v for k, v in blob.items() if k not in color})
    np.savez_compressed(os.path.join(HERE, 'pointslam_color_step.npz'), **color)
    print('wrote pointslam_geo_step.npz, pointslam_color_step.npz', npc.pts_num(), 'points')


def _nice_oracle_to_ref(ora, ref):
    """Copy decoders + grids of oracle.nice.NiceOracle into a reference ConvOnet."""
    with torch.no_grad():
        for name in ('middle', 'fine', 'color'):
            r, o = getattr(ref.decoder, name + '_decoder'), getattr(ora, name)
            r.embedder._B.copy_(o.B)
            for i in range(5):
                for a, b in ((r.fc_c[i], o.fc_c[i]), (r.pts_linears[i], o.pts[i])):
                    a.weight.copy_(b.weight)
                    a.bias.copy_(b.bias)
            r.output_linear.weight.copy_(o.out.weight)
            r.output_linear.bias.copy_(o.out.bias)
        for k in ora.grids:
            ref.grid_c[k] = ora.grids[k].detach().clone()
        if ora.coarse is not None:
            r, o = ref.decoder.coarse_decoder, ora.coarse
            for i in range(5):
                r.pts_linears[i].weight.copy_(o.pts[i].weight)
                r.pts_linears[i].bias.copy_(o.pts[i].bias)
            r.output_linear.weight.copy_(o.out.weight)
            r.output_linear.bias.copy_(o.out.bias)


def reference_cpu():
    """Digests and scalars of the reference's own classes and functions on the seeded inputs
    of the tests in tests/test_oracle_cpu.py and tests/test_voxfusion_cpu.py (CPU only).
    Bit-exact comparisons are stored as SHA-256 digests, tolerance comparisons as arrays
    (reference_cpu.npz)."""
    import json
    from types import SimpleNamespace
    from scipy import ndimage
    from helpers import digest
    import test_oracle_cpu as T
    torch.set_num_threads(1)  # reduction order independent of the host's core count
    out, arrays = {}, {}
    out['octree'] = _svo_octree()  # first svo.Octree of the process: node ids coincide
    ref_harness.install()
    # Co-SLAM JointEncoding
    ora, (rays_o, rays_d, ts, td), noise, smooth_rand, n256 = T.coslam_live_case()
    ref = ref_harness.ref_joint_encoding(torch.from_numpy(BOUND))
    with torch.no_grad():
        ref.embed_fn.params.copy_(ora.embed_fn.params)
        ref.decoder.sdf_net.model[0].weight.copy_(ora.sdf0.weight)
        ref.decoder.sdf_net.model[2].weight.copy_(ora.sdf1.weight)
        ref.decoder.color_net.model[0].weight.copy_(ora.col0.weight)
        ref.decoder.color_net.model[2].weight.copy_(ora.col1.weight)
    torch.manual_seed(9)
    inp = dict(rays_o=rays_o, rays_d=rays_d, target_s=ts, target_d=td, first=False)
    out_r = ref(inp)
    ld_r = ref.get_loss_dict(out_r, inp, True, 0)
    torch.manual_seed(4)
    o2 = ref(dict(rays_o=rays_o, rays_d=rays_d, target_s=None, target_d=None))
    out['coslam'] = {'out': {k: digest(out_r[k]) for k in T.COSLAM_OUT_KEYS},
                     'losses': {k: float(v.detach()) for k, v in ld_r.items()},
                     'render': {'rgb': digest(o2['rgb']), 'depth': digest(o2['depth'])}}
    # NICE-SLAM ConvOnet, stage coarse
    ora, (rays_o, rays_d, ts, td) = T.nice_coarse_case()
    ref = ref_harness.ref_conv_onet(T.NICE_COARSE_BOUND, coarse=True)
    coarse_shape = list(ref.grid_c['grid_coarse'].shape)  # the reference's own construction
    _nice_oracle_to_ref(ora, ref)
    ref.grid_c['grid_coarse'].requires_grad_(True)
    inp = dict(rays_o=rays_o, rays_d=rays_d, target_s=ts, target_d=td, stage='coarse')
    with ref_harness.cuda_calls_are_noops():
        o = ref(inp)
    ld = ref.get_loss_dict(o, inp, True, 'coarse')
    ld['depth_loss'].backward()
    out['nice_coarse'] = {
        'grid_coarse_shape': coarse_shape,
        'coarse_bound': digest(ref.decoder.coarse_decoder.bound),
        'out': {k: digest(o[k]) for k in ('depth', 'uncertainty')},
        'depth_loss': float(ld['depth_loss'].detach()),
        'd_grid_coarse': digest(ref.grid_c['grid_coarse'].grad)}
    # NICE-SLAM ConvOnet, stages color / middle / fine
    ora, (rays_o, rays_d, ts, td) = T.nice_case()
    ref = ref_harness.ref_conv_onet(T.NICE_BOUND)
    _nice_oracle_to_ref(ora, ref)
    nice = {'bound': digest(ref.bounding_box)}
    for stage in ('color', 'middle', 'fine'):
        inp = dict(rays_o=rays_o, rays_d=rays_d, target_s=ts, target_d=td, stage=stage)
        with ref_harness.cuda_calls_are_noops():
            o = ref(inp)
            keys = ('rgb', 'depth', 'uncertainty') if stage == 'color' else ('depth', 'uncertainty')
            nice[stage] = {'out': {k: digest(o[k]) for k in keys}, 'losses': {
                str(m): {k: float(v.detach()) for k, v in ref.get_loss_dict(o, inp, m, stage).items()}
                for m in (True, False)}}
    ref2 = ref_harness.ref_conv_onet(T.OFFICE0_BOUND)
    nice['office0_shapes'] = {k: list(ref2.grid_c[k].shape) for k in ('grid_middle', 'grid_fine')}
    out['nice'] = nice
    # host front end
    import slam.common.common as rc
    import slam.utils.utils as ru
    from slam.common.camera import Camera as RCam
    from xrdslam_b200.synthetic import make_sequence
    cam, poses, fr = make_sequence(1, width=160, height=120)
    rcam = RCam(cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height)
    c2w = torch.from_numpy(poses[0])
    rgb, depth = fr[0]
    fe = {'get_samples': []}
    for kw in T.FRONTEND_KW:
        torch.manual_seed(5)
        fe['get_samples'].append([digest(x) for x in
                                  rc.get_samples(rcam, 333, c2w, depth, rgb, device='cpu', **kw)])
    fe['get_rays'] = [digest(x) for x in rc.get_rays(rcam, c2w, 'cpu')]
    fe['get_camera_rays'] = digest(torch.as_tensor(
        ru.get_camera_rays(120, 160, cam.fx, cam.fy, cam.cx, cam.cy)))
    out['frontend'] = fe
    # optimizers
    import slam.engine.optimizers as ro
    out['optimizers'] = T.optimizers_case(ro)
    # keyframe selection
    cam, frames = T.keyframe_case()
    rcam = RCam(cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height)
    out['keyframes'] = {}
    for k in (2, 4, 8):
        torch.manual_seed(3)
        np.random.seed(3)
        a = rc.keyframe_selection_overlap(rcam, frames[0], frames[1:], k, device='cpu')
        out['keyframes'][str(k)] = [f.fid for f in a]
    # Point-SLAM colour-gradient pixel sampler (skimage -> the scipy restatement the mirror uses)
    import xrdslam_b200.common as mc
    hs = np.array([[1, 2, 1], [0, 0, 0], [-1, -2, -1]], dtype=np.float64) / 4.0
    rc.rgb2gray = mc.rgb2gray_np
    rc.filters = SimpleNamespace(sobel_h=lambda im: ndimage.convolve(im, hs, mode='reflect'),
                                 sobel_v=lambda im: ndimage.convolve(im, hs.T, mode='reflect'))
    cam, poses, fr = make_sequence(1, width=160, height=120)
    rcam = RCam(cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height)
    c2w = torch.from_numpy(poses[0])
    rgb, depth = fr[0]
    np.random.seed(3)
    pg = {'uv': digest(rc.get_sample_uv_with_grad(5, 115, 7, 150, 40, rgb)), 'samples': []}
    for kw in T.PIXEL_GRAD_KW:
        np.random.seed(11)
        pg['samples'].append([digest(x) for x in rc.get_samples_with_pixel_grad(
            rcam, 60, c2w, depth, rgb, device='cpu', **kw)])
    out['pixel_grad'] = pg
    out['vox'], arrays = _vox_torch_part()
    with open(os.path.join(HERE, 'reference_cpu.json'), 'w') as f:
        json.dump(out, f, indent=1)
    np.savez_compressed(os.path.join(HERE, 'reference_cpu.npz'), **arrays)
    print('wrote reference_cpu.json, reference_cpu.npz')


def _svo_octree():
    """The reference's svo.Octree (oracle/_ref/svo.so) on the inserts of
    tests/test_voxfusion_cpu.py::test_octree_bit_exact_vs_reference_svo."""
    from helpers import digest
    import test_voxfusion_cpu as V
    torch.classes.load_library(os.path.join(os.path.dirname(os.path.dirname(HERE)), 'oracle',
                                            '_ref', 'svo.so'))
    ref = torch.classes.svo.Octree()
    ref.init(256, 16, 0.2)
    v0, _, _ = ref.get_centres_and_children()
    assert int(v0.shape[0]) == 1, 'not the first octree of the process'
    steps = []
    for pts in V.octree_inserts():
        ref.insert(pts)
        steps.append([digest(x) for x in ref.get_centres_and_children()])
    return steps


def _vox_torch_part():
    """The reference's SparseVoxel.render_rays + get_loss_dict on CPU (see
    tests/test_voxfusion_cpu.py::test_vox_oracle_torch_part_matches_reference_python)."""
    from helpers import digest
    import test_voxfusion_cpu as V
    ora, ro, rd, ts, td, marched, ms, full_inter = V.vox_case()
    inter, hits, samples = marched
    ref, sv = ref_harness.ref_sparse_voxel_cpu(ms, ora.embeddings.detach(), (full_inter, hits, samples))
    od = ora.decoder
    with torch.no_grad():
        r = ref.decoder
        for a, b in ((r.pts_linears[0], od.pts_linears[0]), (r.pts_linears[1], od.pts_linears[1]),
                     (r.sdf_out, od.sdf_out), (r.color_out[0], od.color_out[0]),
                     (r.color_out[2], od.color_out[2])):
            a.weight.copy_(b.weight)
            a.bias.copy_(b.bias)
    with ref_harness.cuda_calls_are_noops():
        out_r = ref.render_rays(ro.unsqueeze(0), rd.unsqueeze(0), target_d=td.unsqueeze(0))
    ld_r = ref.get_loss_dict(out_r, {'target_d': td, 'target_s': ts}, True)
    sum(ld_r.values()).backward()
    ge = ref.embeddings.grad
    rows = torch.nonzero(ge.abs().sum(-1)).reshape(-1)
    arrays = {'vox.depth': out_r['depth'].detach().numpy(), 'vox.rgb': out_r['rgb'].detach().numpy(),
              'vox.sdf': out_r['sdf'].detach().numpy(),
              'vox.d_embeddings_rows': rows.numpy(), 'vox.d_embeddings': ge[rows].numpy(),
              'vox.d_sdf_out_w': ref.decoder.sdf_out.weight.grad.numpy()}
    return {'ray_mask': digest(out_r['ray_mask']),
            'losses': {k: float(v.detach()) for k, v in ld_r.items()}}, arrays


def vox_grid():
    """Digests of the reference's own `grid` CUDA extension (oracle/_ref/grid.so, built by
    oracle/build_ref.py) on the seeded scenes of tests/test_voxfusion_gpu.py.  Needs a B200."""
    import importlib.machinery
    import importlib.util
    import json
    import test_voxfusion_gpu as T
    path = os.path.join(os.path.dirname(os.path.dirname(HERE)), 'oracle', '_ref', 'grid.so')
    loader = importlib.machinery.ExtensionFileLoader('grid', path)
    spec = importlib.util.spec_from_loader('grid', loader)
    grid = importlib.util.module_from_spec(spec)
    loader.exec_module(grid)
    dev = torch.device('cuda:0')
    out = {}
    rec = T.Recorder(grid)
    T.intersect_case(rec, dev)
    out['intersect'] = rec.digests
    rec = T.Recorder(grid)
    args = T.sampling_case(rec, dev)
    out['sampling'] = {'intersect': rec.digests}
    rec.digests = []
    rec.inverse_cdf_sampling(*args)
    out['sampling']['samples'] = rec.digests
    out['chained'] = {}
    for R in (300, 5 * 1024):
        model, ora, rays_o, rays_d, ts, td, noise_rank, noise_fn = T.chained_case(dev, R)
        rec = T.Recorder(grid)
        T._march_through_grid(rec, ora, rays_o, rays_d, noise_fn, dev)
        out['chained'][str(R)] = rec.digests
    dst = os.environ.get('GOLDEN_OUT', HERE)
    with open(os.path.join(dst, 'vox_grid_ref.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print('wrote vox_grid_ref.json')


if __name__ == '__main__':
    which = sys.argv[1:] or ['coslam', 'nice', 'pointslam']
    if 'vox_grid' not in which:
        assert ref_harness.available(), 'needs the reference checkout (XRDSLAM_REFERENCE)'
    for w in which:
        globals()[w]()
