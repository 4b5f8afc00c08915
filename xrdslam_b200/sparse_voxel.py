"""Vox-Fusion model behind the reference's ``Model`` plugin surface, B200-native.

Host-side mirror of slam/models/sparse_voxel.py (reference @ f0366f20): same class / config
names, ``forward / get_loss_dict / get_param_groups / insert_points / update_map_states``
signatures, parameter groups ``decoder`` and ``embeddings``, decoder state_dict keys of
slam/model_components/decoder_voxfusion.py (``pts_linears.{0,1}``, ``sdf_out``,
``color_out.{0,2}``).  The octree is this package's own C++ structure (csrc/octree.cpp, node
ids identical to the reference's svo.Octree); ray/voxel intersection, sampling, feature
interpolation, decoder, compositing, losses and their gradients run in csrc/vox.cu through
the C-ABI.  No PyTorch fallback exists.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Type, Union

import numpy as np
import torch
from torch import nn
from torch.nn import Parameter

from . import _cabi
from ._cabi import (XrdRays, XrdVoxDecoder, XrdVoxDecoderGrads, XrdVoxGrads, XrdVoxMap,
                    XrdVoxMarch, XrdVoxMarchCfg, XrdVoxOut, XrdVoxRenderCfg, check, ptr)
from .base_model import Model, ModelConfig, scale_grads, upstream_scale

MAX_DEPTH = 10.0  # voxel_helpers_voxfusion.py:11


@dataclass
class SparseVoxelConfig(ModelConfig):
    """slam/models/sparse_voxel.py:38-72 (field names and defaults kept)."""
    _target: Type = field(default_factory=lambda: SparseVoxel)
    voxels_each_dim: int = 256
    voxel_size: float = 0.2
    num_embeddings: int = 20000
    embed_dim: int = 16
    max_distance: int = 10
    max_dpeth: float = 10
    training_trunc: float = 0.05
    trainging_rgb_weight: float = .5
    trainging_depth_weight: float = 1.0
    trainging_sdf_weight: float = 5000
    trainging_fs_weight: float = 10.0
    depth: int = 2
    width: int = 128
    in_dim: int = 16
    embedder: str = 'none'
    step_size: float = 0.05
    max_voxel_hit: int = 20
    num_iterations: int = 30
    overlap_th: float = 0.7
    keyframe_th: int = 30
    keyframe_selection: str = 'random'
    data_sc_factor: int = 1
    # --- B200 path knobs ---
    max_samples_per_ray: int = 256  # capacity of the per-ray sample arrays
    seed: int = 0
    device_octree: bool = True  # grow the octree on the device (octree_device.py)


class Decoder(nn.Module):
    """Parameter container of decoder_voxfusion.py:76-149 (depth 2, width 128, 'none')."""
    def __init__(self, width=128, in_dim=16, sdf_dim=128):
        super().__init__()
        self.pts_linears = nn.ModuleList([nn.Linear(in_dim, width), nn.Linear(width, width)])
        self.sdf_out = nn.Linear(width, 1 + sdf_dim)
        self.color_out = nn.Sequential(nn.Linear(sdf_dim + in_dim, width), nn.ReLU(),
                                       nn.Linear(width, 3), nn.Sigmoid())

    def tensors(self):
        return [self.pts_linears[0].weight, self.pts_linears[0].bias,
                self.pts_linears[1].weight, self.pts_linears[1].bias, self.sdf_out.weight,
                self.sdf_out.bias, self.color_out[0].weight, self.color_out[0].bias,
                self.color_out[2].weight, self.color_out[2].bias]


def _dec_struct(tensors, cls):
    d = cls()
    for n, t in zip(('w0', 'b0', 'w1', 'b1', 'ws', 'bs', 'wc0', 'bc0', 'wc1', 'bc1'), tensors):
        setattr(d, n, ptr(t))
    return d


class _VoxStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, target_s, target_d, noise, rays_o, rays_d, emb, *dec):
        need_rays = ctx.needs_input_grad[4] or ctx.needs_input_grad[5]
        need_map = any(ctx.needs_input_grad[6:])
        outs, grads = model._launch(rays_o, rays_d, target_s, target_d, noise,
                                    need_rays or need_map, need_rays, need_map)
        ctx.grads = grads
        if outs is None:
            raise RuntimeError('render_rays: no ray hit any voxel')
        ret = (outs['losses'], outs['rgb'], outs['depth'], outs['ray_mask'])
        ctx.mark_non_differentiable(*ret[1:])
        return ret

    @staticmethod
    def backward(ctx, g_losses, *_):
        g = ctx.grads
        ro, rd, emb, dec = scale_grads([g['d_rays_o'], g['d_rays_d'], g['d_emb'], list(g['d_dec'])],
                                       upstream_scale(g_losses))
        return (None, None, None, None, ro, rd, emb, *dec)


class SparseVoxel(Model):
    """Model class (slam/models/sparse_voxel.py:75-358)."""

    config: SparseVoxelConfig

    def __init__(self, config: SparseVoxelConfig, camera, bounding_box=None, **kwargs) -> None:
        super().__init__(config=config, camera=camera, bounding_box=bounding_box, **kwargs)
        self.config.step_size = self.config.voxel_size * self.config.step_size
        self.pose_offset = int(self.config.voxels_each_dim / 2.0 * self.config.voxel_size)

    def populate_modules(self):
        super().populate_modules()
        cfg = self.config
        if (cfg.depth, cfg.width, cfg.in_dim, cfg.embed_dim, cfg.embedder) != (2, 128, 16, 16, 'none'):
            raise NotImplementedError('decoder shape fixed to the reference vox-fusion config')
        self._dev_svo = None
        self.get_octree()
        self.get_decoder()
        self.map_states = None
        self._step_count = 0

    def get_octree(self):
        lib = _cabi.lib()
        self._svo = lib.xrd_octree_create(self.config.voxels_each_dim)
        if not self._svo:
            raise RuntimeError('xrd_octree_create failed')
        emb = torch.zeros((self.config.num_embeddings, self.config.embed_dim), dtype=torch.float32)
        torch.nn.init.normal_(emb, std=0.01)
        self.embeddings = nn.Parameter(emb)

    def __del__(self):
        svo = getattr(self, '_svo', None)
        if svo:
            try:
                _cabi.lib().xrd_octree_destroy(svo)
            except Exception:
                pass

    def get_decoder(self):
        self.decoder = Decoder(width=self.config.width, in_dim=self.config.embed_dim)

    # ---------------------------------------------------------- map update ---
    def insert_points(self, points):
        """sparse_voxel.py:325-332: voxel coords = floor(p / voxel_size), int32.  With the map on
        a CUDA device the octree is grown ON THE DEVICE (octree_device.DeviceOctree: same node
        ids as the reference's host insertion, no D2H of the ~300 k points per mapping frame and
        no H2D of the exported tables); otherwise by the host C++ octree (csrc/octree.cpp)."""
        voxels = torch.div(points, self.config.voxel_size, rounding_mode='floor')
        if self.config.device_octree and self.embeddings.device.type == 'cuda':
            if self._dev_svo is None:
                from .octree_device import DeviceOctree
                if _cabi.lib().xrd_octree_num_nodes(self._svo) != 1:
                    raise RuntimeError('octree already holds host-inserted voxels')
                self._dev_svo = DeviceOctree(self.config.voxels_each_dim, self.embeddings.device)
            n = self._dev_svo.insert(voxels.to(torch.int64))
            if n > self.config.num_embeddings:
                raise RuntimeError(f'octree has {n} nodes > num_embeddings='
                                   f'{self.config.num_embeddings} (the reference indexes past '
                                   'the table here, SURVEY Q4)')
            self.update_map_states()
            return
        self.insert_voxels(voxels.cpu().int())

    def insert_voxels(self, voxels_i32):
        if self._dev_svo is not None:
            raise RuntimeError('octree lives on the device: use insert_points')
        v = voxels_i32.contiguous()
        n = _cabi.lib().xrd_octree_insert(self._svo, v.data_ptr(), v.shape[0])
        if n < 0:
            check('xrd_octree_insert', n)
        if n > self.config.num_embeddings:
            raise RuntimeError(f'octree has {n} nodes > num_embeddings={self.config.num_embeddings} '
                               '(the reference indexes past the table here, SURVEY Q4)')
        self.update_map_states()

    def export_octree(self):
        """voxels f32 [N,4], children f32 [N,8], features i32 [N,8] (HOST tensors)."""
        if self._dev_svo is not None:
            return tuple(t.cpu() for t in self._dev_svo.export())
        lib = _cabi.lib()
        N = lib.xrd_octree_num_nodes(self._svo)
        voxels = torch.empty(N, 4)
        children = torch.empty(N, 8)
        features = torch.empty(N, 8, dtype=torch.int32)
        lib.xrd_octree_export(self._svo, voxels.data_ptr(), children.data_ptr(), features.data_ptr())
        return voxels, children, features

    def update_map_states(self):
        """sparse_voxel.py:334-351."""
        if self._dev_svo is not None:
            voxels, children, features = self._dev_svo.export()  # stays on the device
        else:
            voxels, children, features = self.export_octree()
        centres = (voxels[:, :3] + voxels[:, -1:] / 2) * self.config.voxel_size
        children = torch.cat([children, voxels[:, -1:]], -1)
        dev = self.embeddings.device
        self.map_states = {
            'voxel_vertex_idx': features.to(dev).contiguous(),
            'voxel_center_xyz': centres.to(dev).float().contiguous(),
            'voxel_structure': children.to(dev).int().contiguous(),
            'voxel_vertex_emb': self.embeddings,
        }

    def get_map_states(self):
        return dict(self.map_states)

    def octree_tables(self):
        """voxels f32 [N,4], children f32 [N,8], features i32 [N,8] on the map's device."""
        if self._dev_svo is not None:
            return self._dev_svo.export()
        return tuple(t.to(self.embeddings.device) for t in self.export_octree())

    @torch.no_grad()
    def query(self, points, voxel_ids, centres, vertex_idx):
        """voxel_helpers_voxfusion.py:15-95 (get_scores / eval_points): decoder outputs
        raw [P,4] = (rgb, sdf) at device points [P,3], each interpolated inside voxel
        ``voxel_ids[p]`` -- a row of ``centres`` [N,3] / ``vertex_idx`` [N,8] (the mesher's
        filtered voxel list)."""
        dev = self.embeddings.device
        P = points.shape[0]
        raw = torch.empty(P, 4, dtype=torch.float32, device=dev)
        if P == 0:
            return raw
        lib = _cabi.lib()
        emb = self.embeddings.detach()
        centres = centres.to(dev, torch.float32).contiguous()
        vertex_idx = vertex_idx.to(dev, torch.int32).contiguous()
        mp = XrdVoxMap(centres.shape[0], ptr(centres), None, ptr(vertex_idx), ptr(emb),
                       emb.shape[0])
        dec = _dec_struct([t.detach() for t in self.decoder.tensors()], XrdVoxDecoder)
        pts = points.to(dev, torch.float32).contiguous()
        ids = voxel_ids.to(dev, torch.int32).contiguous()
        nb = lib.xrd_voxfusion_query_workspace_bytes(P)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            st = lib.xrd_voxfusion_query(C.byref(mp), C.byref(dec), self.config.voxel_size,
                                         ptr(pts), ptr(ids), P, ptr(raw), ptr(ws), nb,
                                         torch.cuda.current_stream(dev).cuda_stream)
        check('xrd_voxfusion_query', st)
        return raw

    # -------------------------------------------------------------- C-ABI ---
    def _map_struct(self, emb):
        ms = self.map_states
        return XrdVoxMap(ms['voxel_center_xyz'].shape[0], ptr(ms['voxel_center_xyz']),
                         ptr(ms['voxel_structure']), ptr(ms['voxel_vertex_idx']), ptr(emb),
                         emb.shape[0])

    def march(self, rays_o, rays_d, noise=None, rays_per_block=0):
        """Intersections + samples (device tensors) and the host copy of the 5 stats."""
        cfg = self.config
        dev = self.embeddings.device
        lib = _cabi.lib()
        R = rays_o.shape[0]
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        H, Sc = 50, cfg.max_samples_per_ray
        m = dict(hit_idx=torch.empty(R, H, **i32), hit_tmin=torch.empty(R, H, **f32),
                 hit_tmax=torch.empty(R, H, **f32), smp_idx=torch.full((R, Sc), -1, **i32),
                 smp_depth=torch.full((R, Sc), MAX_DEPTH, **f32), smp_dist=torch.zeros(R, Sc, **f32),
                 smp_count=torch.empty(R, **i32), smp_base=torch.empty(R, **i32),
                 ray_mask=torch.empty(R, dtype=torch.uint8, device=dev),
                 stats=torch.zeros(8 + 2 * R, **i32))
        self._step_count += 1
        mc = XrdVoxMarchCfg(cfg.voxel_size, cfg.step_size, H, float(cfg.max_distance), Sc,
                            rays_per_block, (cfg.seed << 32) + self._step_count)
        ms = XrdVoxMarch(*[ptr(m[k]) for k in ('hit_idx', 'hit_tmin', 'hit_tmax', 'smp_idx',
                                               'smp_depth', 'smp_dist', 'smp_count', 'smp_base',
                                               'ray_mask', 'stats')])
        rays = XrdRays(R, ptr(rays_o), ptr(rays_d), None, None)
        mp = self._map_struct(self.embeddings.detach())
        with torch.cuda.device(dev):
            st = lib.xrd_voxfusion_march(C.byref(rays), C.byref(mp), C.byref(mc), ptr(noise),
                                         C.byref(ms), torch.cuda.current_stream(dev).cuda_stream)
        check('xrd_voxfusion_march', st)
        stats = m['stats'][:8].cpu().tolist()  # the one host read (reference: hits.sum() == 0)
        m['_cfg'], m['_struct'] = mc, ms
        m['n_hit_rays'], m['n_points'], m['s_max'], m['p_max'], m['overflow'] = stats[:5]
        return m

    def _launch(self, rays_o, rays_d, target_s, target_d, noise, with_grads, need_rays=False,
                need_map=False):
        cfg = self.config
        dev = self.embeddings.device
        if dev.type != 'cuda':
            raise RuntimeError('xrdslam_b200 has no CPU path: model must be on a CUDA device')
        if self.map_states is None:
            raise RuntimeError('empty map: call insert_points first')
        lib = _cabi.lib()
        f32 = dict(dtype=torch.float32, device=dev)
        rays_o = rays_o.detach().to(**f32).contiguous()
        rays_d = rays_d.detach().to(**f32).contiguous()
        R = rays_o.shape[0]
        if noise is not None:
            noise = noise.detach().to(**f32).contiguous()
        m = self.march(rays_o, rays_d, noise)
        self.last_march = m
        if m['n_hit_rays'] == 0 or m['n_points'] == 0:
            return None, None
        td = target_d.detach().to(**f32).reshape(-1).contiguous() if target_d is not None else None
        ts = target_s.detach().to(**f32).contiguous() if target_s is not None else None
        rays = XrdRays(R, ptr(rays_o), ptr(rays_d), ptr(ts), ptr(td))
        dts = [t.detach() for t in self.decoder.tensors()]
        dec = _dec_struct(dts, XrdVoxDecoder)
        emb = self.embeddings.detach()
        mp = self._map_struct(emb)
        rc = XrdVoxRenderCfg(cfg.voxel_size, cfg.training_trunc * cfg.data_sc_factor,
                             cfg.max_dpeth, MAX_DEPTH, cfg.trainging_rgb_weight,
                             cfg.trainging_depth_weight, cfg.trainging_sdf_weight,
                             cfg.trainging_fs_weight, m['n_points'], m['s_max'], m['n_hit_rays'])
        o = dict(rgb=torch.empty(R, 3, **f32), depth=torch.empty(R, **f32),
                 losses=torch.zeros(4, **f32), ray_mask=m['ray_mask'].bool())
        out = XrdVoxOut(ptr(o['rgb']), ptr(o['depth']), ptr(o['losses']))
        g, gs, keep = None, None, []
        if with_grads:
            if ts is None or td is None:
                raise RuntimeError('gradients need target_s and target_d')
            d_dec = [torch.zeros_like(t) for t in dts] if need_map else [None] * 10
            g = dict(d_emb=torch.zeros_like(emb) if need_map else None, d_dec=d_dec,
                     d_rays_o=torch.empty(R, 3, **f32) if need_rays else None,
                     d_rays_d=torch.empty(R, 3, **f32) if need_rays else None)
            gs = XrdVoxGrads()
            gs.d_embeddings = ptr(g['d_emb'])
            if need_map:
                dg = _dec_struct(d_dec, XrdVoxDecoderGrads)
                keep.append(dg)
                gs.d_decoder = C.pointer(dg)
            gs.d_rays_o, gs.d_rays_d = ptr(g['d_rays_o']), ptr(g['d_rays_d'])
        nb = lib.xrd_voxfusion_render_workspace_bytes(R, m['n_points'], int(with_grads))
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            st = lib.xrd_voxfusion_render(C.byref(rays), C.byref(mp), C.byref(m['_struct']),
                                          C.byref(m['_cfg']), C.byref(dec), C.byref(rc),
                                          C.byref(out), C.byref(gs) if gs is not None else None,
                                          ptr(ws), nb, torch.cuda.current_stream(dev).cuda_stream)
        check('xrd_voxfusion_render', st)
        return o, g

    # --------------------------------------------------------- Model API ---
    def get_outputs(self, input) -> Dict[str, Union[torch.Tensor, List]]:
        """sparse_voxel.py:152-159 (returns None when no ray hits a voxel, :179-181)."""
        rays_o, rays_d = input['rays_o'], input['rays_d']
        target_d, target_s = input.get('target_d'), input.get('target_s')
        noise = input.get('noise')
        fused = torch.is_grad_enabled() and target_s is not None and target_d is not None
        if fused:
            try:
                emb, dec = self.embeddings, self.decoder.tensors()
                if getattr(self, 'freeze_map_grads', False):  # tracking: pose gradients only
                    emb, dec = emb.detach(), [t.detach() for t in dec]
                losses, rgb, depth, ray_mask = _VoxStep.apply(
                    self, target_s, target_d, noise, rays_o, rays_d, emb, *dec)
            except RuntimeError as e:
                if 'no ray hit' in str(e):
                    print('\n\n', '!' * 20, 'render_rays. no hit', '!' * 20, '\n\n')
                    return None
                raise
            return {'depth': depth, 'rgb': rgb, 'ray_mask': ray_mask, '_losses': losses}
        o, _ = self._launch(rays_o, rays_d, target_s, target_d, noise, False)
        if o is None:
            return None
        o.pop('losses')
        return o

    def get_loss_dict(self, outputs, inputs, is_mapping, stage=None) -> Dict[str, torch.Tensor]:
        """sparse_voxel.py:103-143."""
        ls = outputs['_losses']
        return {'rgb_loss': ls[0], 'depth_loss': ls[1], 'sdf_loss': ls[2], 'fs_loss': ls[3]}

    def get_param_groups(self) -> Dict[str, List[Parameter]]:
        return {'decoder': list(self.decoder.parameters()), 'embeddings': [self.embeddings]}
