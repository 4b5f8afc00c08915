"""Shared builders for the parity tests (oracle <-> CUDA path)."""
import hashlib
import json
import os

import numpy as np
import torch

BOUND = np.array([[-3, 3], [-4, 2.5], [-2, 2.5]], dtype=np.float64)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def make_rays(R, seed=0, zero_depth_every=7):
    g = torch.Generator().manual_seed(seed)
    rays_o = (torch.rand(R, 3, generator=g) - 0.5) * 1.0
    rays_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g),
                                           dim=-1)
    rays_d = rays_d * (1.0 + 0.2 * torch.rand(R, 1, generator=g))
    target_d = torch.rand(R, 1, generator=g) * 3 + 0.3
    if zero_depth_every:
        target_d[3::zero_depth_every] = 0
    target_s = torch.rand(R, 3, generator=g)
    noise = torch.rand(R, 43, generator=g)
    return rays_o, rays_d, target_s, target_d, noise


def coslam_pair(device, table_amp=0.3, seed=1, **cfg):
    """(oracle on CPU, B200 model on device) with identical parameters."""
    from oracle.coslam import CoslamOracle
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.joint_encoding import JointEncodingConfig
    ora = CoslamOracle(BOUND)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        ora.embed_fn.params.copy_(
            (torch.rand(ora.embed_fn.params.shape, generator=g) * 2 - 1) *
            table_amp)
        for lin in (ora.sdf0, ora.sdf1, ora.col0, ora.col1):
            lin.weight.copy_(torch.randn(lin.weight.shape, generator=g) *
                             (1.0 / np.sqrt(lin.weight.shape[1])))
    model = JointEncodingConfig(**cfg).setup(
        camera=Camera(320., 320., 319.5, 239.5, 640, 480), bounding_box=BOUND)
    with torch.no_grad():
        model.embed_fn.params.copy_(ora.embed_fn.params)
        model.decoder.sdf_net.model[0].weight.copy_(ora.sdf0.weight)
        model.decoder.sdf_net.model[2].weight.copy_(ora.sdf1.weight)
        model.decoder.color_net.model[0].weight.copy_(ora.col0.weight)
        model.decoder.color_net.model[2].weight.copy_(ora.col1.weight)
    model.to(device)
    return ora, model


def _t(x):
    return torch.from_numpy(np.asarray(x)) if not torch.is_tensor(x) else x


def digest(x):
    """SHA-256 of a tensor's dtype, shape and bytes: a bit-exact comparison against a stored
    reference output without storing the output itself."""
    t = _t(x).detach().cpu().contiguous()
    h = hashlib.sha256(f'{t.dtype} {tuple(t.shape)} '.encode())
    h.update(t.numpy().tobytes())
    return h.hexdigest()


def load_golden_json(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def rel_err(a, b):
    a, b = _t(a), _t(b)
    a = a.detach().double().cpu().reshape(-1)
    b = b.detach().double().cpu().reshape(-1)
    return float((a - b).norm() / (b.norm() + 1e-30))


def max_abs(a, b):
    a, b = _t(a), _t(b)
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max())


def load_golden_coslam():
    """Golden vectors written by tests/golden/make_golden.py (reference classes)."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'coslam_map_step.npz'))
    g = {k: g[k] for k in g.files}
    gen = torch.Generator().manual_seed(int(g['table_seed']))
    from oracle.tcnn_restated import hashgrid_level_table
    n = hashgrid_level_table(16, 2, 16, 16, np.exp2(np.log2(325 / 16) / 15))['n_params']
    g['table'] = ((torch.rand(n, generator=gen) * 2 - 1) * 0.3)
    assert abs(float(g['table'].double().sum()) - float(g['table_checksum'])) < 1e-9
    return g


def set_coslam_params(obj, g, kind):
    """Load golden parameters into an oracle (kind='oracle') or B200 model."""
    with torch.no_grad():
        t = lambda k: torch.from_numpy(g[k])
        if kind == 'oracle':
            obj.embed_fn.params.copy_(g['table'])
            obj.sdf0.weight.copy_(t('w_sdf0')); obj.sdf1.weight.copy_(t('w_sdf1'))
            obj.col0.weight.copy_(t('w_col0')); obj.col1.weight.copy_(t('w_col1'))
        else:
            obj.embed_fn.params.copy_(g['table'])
            obj.decoder.sdf_net.model[0].weight.copy_(t('w_sdf0'))
            obj.decoder.sdf_net.model[2].weight.copy_(t('w_sdf1'))
            obj.decoder.color_net.model[0].weight.copy_(t('w_col0'))
            obj.decoder.color_net.model[2].weight.copy_(t('w_col1'))


def load_golden_nice():
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'nice_color_step.npz'))
    g = {k: g[k] for k in g.files}
    for i, k in enumerate(sorted(['grid_middle', 'grid_fine', 'grid_color'])):
        gg = torch.Generator().manual_seed(1000 + i)
        g[k] = torch.randn(tuple(int(v) for v in g[k + '.shape']), generator=gg) * 0.3
        assert abs(float(g[k].double().sum()) - float(g[k + '.checksum'])) < 1e-6
    return g


def nice_from_golden(g, kind, device=None):
    """Build an oracle (kind='oracle') or B200 model from the golden parameters."""
    t = lambda k: torch.from_numpy(g[k])
    if kind == 'oracle':
        from oracle.nice import NiceOracle
        obj = NiceOracle(g['bound'])
        decs = {'middle': obj.middle, 'fine': obj.fine, 'color': obj.color}
    else:
        from xrdslam_b200.camera import Camera
        from xrdslam_b200.conv_onet import ConvOnetConfig
        obj = ConvOnetConfig(mapping_frustum_feature_selection=False).setup(
            camera=Camera(320., 320., 319.5, 239.5, 640, 480), bounding_box=g['bound'])
        decs = {n: getattr(obj.decoder, n + '_decoder') for n in ('middle', 'fine', 'color')}
    with torch.no_grad():
        for n, d in decs.items():
            pre = f'dec.{n}_decoder.'
            if kind == 'oracle':
                d.B.copy_(t(pre + 'embedder._B'))
                for i in range(5):
                    d.fc_c[i].weight.copy_(t(pre + f'fc_c.{i}.weight'))
                    d.fc_c[i].bias.copy_(t(pre + f'fc_c.{i}.bias'))
                    d.pts[i].weight.copy_(t(pre + f'pts_linears.{i}.weight'))
                    d.pts[i].bias.copy_(t(pre + f'pts_linears.{i}.bias'))
                d.out.weight.copy_(t(pre + 'output_linear.weight'))
                d.out.bias.copy_(t(pre + 'output_linear.bias'))
            else:
                sd = {k[len(pre):]: t(k) for k in g if k.startswith(pre)}
                d.load_state_dict(sd)  # same state_dict keys as the reference decoder
        for k in ('grid_middle', 'grid_fine', 'grid_color'):
            if kind == 'oracle':
                obj.grids[k].copy_(g[k])
            else:
                obj.set_grid(k, g[k])
    if device is not None:
        obj.to(device)
    return obj


def load_golden_pointslam():
    """Inputs + stage 'geometry' (pointslam_geo_step.npz) and stage 'color' outputs
    (pointslam_color_step.npz, keys cmap.* / ctrk.*)."""
    out = {}
    for name in ('pointslam_geo_step.npz', 'pointslam_color_step.npz'):
        g = np.load(os.path.join(GOLDEN, name))
        out.update({k: g[k] for k in g.files})
    return out


def pointslam_from_golden(g, kind, device=None):
    """Oracle (kind='oracle') or B200 ConvOnet2 with the golden decoder + point cloud."""
    t = lambda k: torch.from_numpy(g[k])
    pre = 'dec.'
    if kind == 'oracle':
        from oracle.pointslam import PointOracle
        obj = PointOracle()
        d = obj.geo
        with torch.no_grad():
            d.B.copy_(t(pre + 'embedder._B'))
            for i in range(5):
                d.fc_c[i].weight.copy_(t(pre + f'fc_c.{i}.weight'))
                d.fc_c[i].bias.copy_(t(pre + f'fc_c.{i}.bias'))
                d.pts[i].weight.copy_(t(pre + f'pts_linears.{i}.weight'))
                d.pts[i].bias.copy_(t(pre + f'pts_linears.{i}.bias'))
            d.out.weight.copy_(t(pre + 'output_linear.weight'))
            d.out.bias.copy_(t(pre + 'output_linear.bias'))
            c, cp = obj.col, 'cdec.'
            c.B.copy_(t(cp + 'embedder._B'))
            c.B_rel.copy_(t(cp + 'embedder_rel_pos._B'))
            for i in range(5):
                c.fc_c[i].weight.copy_(t(cp + f'fc_c.{i}.weight'))
                c.fc_c[i].bias.copy_(t(cp + f'fc_c.{i}.bias'))
                c.pts[i].weight.copy_(t(cp + f'pts_linears.{i}.weight'))
                c.pts[i].bias.copy_(t(cp + f'pts_linears.{i}.bias'))
            for name, lin in (('linear1', c.nb1), ('linear2', c.nb2)):
                lin.weight.copy_(t(cp + f'mlp_col_neighbor.{name}.weight'))
                lin.bias.copy_(t(cp + f'mlp_col_neighbor.{name}.bias'))
            c.out.weight.copy_(t(cp + 'output_linear.weight'))
            c.out.bias.copy_(t(cp + 'output_linear.bias'))
        obj.set_cloud(t('cloud_pos'), t('geo_feats'), col_feats=t('col_feats'))
        return obj
    from xrdslam_b200.camera import Camera
    from xrdslam_b200.conv_onet_pointslam import ConvOnet2Config
    obj = ConvOnet2Config().setup(camera=Camera(320., 320., 319.5, 239.5, 640, 480))
    # same keys as the reference decoder (whose geometry MLP also carries unused colour-only
    # members embedder_rel_pos / mlp_col_neighbor: dropped)
    own = obj.decoder.geo_decoder.state_dict().keys()
    sd = {k[len(pre):]: t(k) for k in g if k.startswith(pre) and k[len(pre):] in own}
    obj.decoder.geo_decoder.load_state_dict(sd)
    csd = {k[len('cdec.'):]: t(k) for k in g if k.startswith('cdec.') and k != 'cdec.embedder._B'}
    obj.decoder.color_decoder.load_state_dict(csd)  # the reference MLP_color's own keys
    obj.decoder.color_decoder.embedder._B.copy_(t('cdec.embedder._B'))
    obj.to(device)
    npc = obj.model_update(device)
    npc.set_cloud(t('cloud_pos'), t('geo_feats'), t('col_feats'))
    return obj


# oracle ColorDecoder parameter name -> reference MLP_color parameter name
def oracle_cdec_grads(ora):
    c = ora.col
    out = {'embedder_rel_pos._B': c.B_rel.grad}
    for i in range(5):
        out[f'fc_c.{i}.weight'], out[f'fc_c.{i}.bias'] = c.fc_c[i].weight.grad, c.fc_c[i].bias.grad
        out[f'pts_linears.{i}.weight'] = c.pts[i].weight.grad
        out[f'pts_linears.{i}.bias'] = c.pts[i].bias.grad
    for name, lin in (('linear1', c.nb1), ('linear2', c.nb2)):
        out[f'mlp_col_neighbor.{name}.weight'] = lin.weight.grad
        out[f'mlp_col_neighbor.{name}.bias'] = lin.bias.grad
    out['output_linear.weight'], out['output_linear.bias'] = c.out.weight.grad, c.out.bias.grad
    return out
