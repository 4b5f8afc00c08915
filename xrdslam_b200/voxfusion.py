"""Vox-Fusion algorithm (host-side mirror of slam/algorithms/voxfusion.py): octree growth
from every valid depth pixel of the mapping frame, per-frame pixel sampling -- around the
CUDA march + render step in sparse_voxel.py."""
from __future__ import annotations

import functools
from dataclasses import dataclass, field
from typing import Any, Dict, Type

import numpy as np
import torch

from .algorithm import Algorithm, AlgorithmConfig
from .common import get_camera_rays
from .mesher import MarchingCubes, Mesh
from .optimizers import AdamOptimizerConfig
from .sparse_voxel import SparseVoxelConfig


def _vox_optimizers():
    """slam/configs/input_config.py:178-195."""
    A = AdamOptimizerConfig
    return {
        'decoder': {'optimizer': A(lr=5e-3), 'scheduler': None},
        'embeddings': {'optimizer': A(lr=5e-3), 'scheduler': None},
        'tracking_pose': {'optimizer': A(lr=1e-2), 'scheduler': None},
        'mapping_pose': {'optimizer': A(lr=1e-3), 'scheduler': None},
    }


@dataclass
class VoxFusionConfig(AlgorithmConfig):
    """voxfusion.py:18-28 + the vox-fusion entry of input_config.py:159-201."""
    _target: Type = field(default_factory=lambda: VoxFusion)
    model: SparseVoxelConfig = field(default_factory=SparseVoxelConfig)
    keyframe_selection_method: str = 'random'
    tracking_n_iters: int = 30
    mapping_n_iters: int = 15
    mapping_first_n_iters: int = 30
    mapping_window_size: int = 5
    mapping_sample: int = 1024
    min_sample_pixels: int = 100
    tracking_sample: int = 1024
    ray_batch_size: int = 3000
    optimizers: Dict[str, Any] = field(default_factory=_vox_optimizers)


class VoxFusion(Algorithm):
    config: VoxFusionConfig

    def __init__(self, config: VoxFusionConfig, camera, device: str) -> None:
        super().__init__(config, camera, device)
        self.model = self.config.model.setup(camera=camera, bounding_box=None)
        self.model.to(device)
        # voxfusion.py:38-52 precompute: camera-frame directions of every pixel (resident)
        self.rays_d = get_camera_rays(camera.height, camera.width, camera.fx, camera.fy,
                                      camera.cx, camera.cy).float().to(device)
        self.bundle_adjust = True

    # voxfusion.py:55-94
    def get_model_input(self, optimize_frames, is_mapping):
        n = self.config.mapping_sample if is_mapping else self.config.tracking_sample
        rays_o, rays_d, gt_depth, gt_color = self._sample_window(optimize_frames, n)
        return {'rays_o': rays_o, 'rays_d': rays_d, 'target_s': gt_color, 'target_d': gt_depth}

    # voxfusion.py:96-106
    def create_voxels(self, frame):
        depth = self._frame_tensor(frame, 'depth')
        points = (self.rays_d * depth[..., None])[depth > 0].reshape(-1, 3)
        pose = frame.get_pose().detach().to(self.device)
        points = points @ pose[:3, :3].transpose(-1, -2) + pose[:3, 3]
        self.model.insert_points(points)

    def pre_precessing(self, cur_frame, is_mapping):
        if is_mapping:
            self.create_voxels(cur_frame)

    def get_loss(self, optimize_frames, is_mapping, step=None, n_iters=None, coarse=False):
        self.model.freeze_map_grads = not is_mapping  # tracking optimises the pose only
        model_input = self.get_model_input(optimize_frames, is_mapping)
        model_outputs = self.model(model_input)
        if model_outputs is None:  # no ray hit the map (sparse_voxel.py:197-199)
            raise RuntimeError('no ray intersects the voxel map')
        loss_dict = self.model.get_loss_dict(model_outputs, model_input, is_mapping, step)
        return functools.reduce(torch.add, loss_dict.values())

    def render_img(self, c2w, gt_depth=None, idx=None):
        with self.lock, torch.no_grad():
            return self._render_full(c2w, gt_depth)

    # voxfusion.py:173-177
    def get_mesh(self):
        with self.lock, torch.no_grad():
            return self.extract_mesh(clean_mesh=False, require_color=True, res=8)

    # Points per decoder call of the mesher (bounds the query workspace, ~2 KB a point).
    query_chunk = 1 << 18

    @torch.no_grad()
    def extract_mesh(self, res=8, clean_mesh=False, require_color=False):
        """voxfusion.py:179-251: per-voxel lattices of res^3 points, one batched marching-cubes
        call, colours queried in the voxel each vertex falls in.  -> Mesh, or None when no
        voxel holds a surface (where the reference's concatenate of nothing raises)."""
        if clean_mesh:
            raise NotImplementedError('clean_mesh needs depth and poses (not provided)')
        model = self.model
        vs = model.config.voxel_size
        voxels, _, features = model.octree_tables()
        keep = ~features.eq(-1).any(-1)
        voxels, features = voxels[keep], features[keep]
        centres = (voxels[:, :3] + voxels[:, -1:] / 2) * vs
        if centres.shape[0] == 0:
            return None
        # get_scores: torch.linspace on the host, * voxel_size, + centre (fp32, same op order)
        x = torch.linspace(-.5, .5, res)
        lat = torch.stack(torch.meshgrid(x, x, x, indexing='ij'), -1).float().to(self.device)
        lat *= vs
        pts = (lat.reshape(1, -1, 3) + centres.unsqueeze(1)).reshape(-1, 3)
        ids = torch.arange(centres.shape[0], device=self.device, dtype=torch.int32)
        ids = ids[:, None].expand(-1, res ** 3).reshape(-1)
        sdf = torch.empty(pts.shape[0], dtype=torch.float32, device=self.device)
        for s in range(0, pts.shape[0], self.query_chunk):
            e = s + self.query_chunk
            sdf[s:e] = model.query(pts[s:e], ids[s:e], centres, features)[:, 3]
        verts, faces = self.marching_cubes(centres, sdf.reshape(-1, res, res, res))
        if faces.shape[0] == 0:
            return None
        colors = None
        if require_color:
            colors = self.vertex_colors(verts, voxels, centres, features)
        return Mesh(verts.cpu().numpy(), faces.cpu().numpy(),
                    None if colors is None else colors.cpu().numpy())

    @torch.no_grad()
    def marching_cubes(self, voxels, sdf):
        """voxfusion.py:253-279 as one batched call: volume i has origin centre - voxel_size/2
        and spacing voxel_size / (res - 1); vertices are welded inside a voxel only."""
        vs = self.model.config.voxel_size
        res = sdf.shape[1]
        origins = voxels[:, :3].double() - vs / 2
        spacings = torch.full_like(origins, vs / (res - 1))
        return MarchingCubes(sdf, 0.0, origins=origins, spacings=spacings).run()

    def vertex_colors(self, verts, voxels, centres, features):
        """voxfusion.py:200-240: the voxel holding each vertex is the first filtered voxel
        whose grid coordinates equal verts // voxel_size (a sorted-key search in place of the
        reference's [1000, N_voxels] comparison); colour = decoder rgb there, 0 without a
        match."""
        vs = self.model.config.voxel_size
        pos = verts // vs
        grid = voxels[:, :3]
        bias, lim = 1 << 20, 1 << 21

        def pack(g):
            q = g.to(torch.int64) + bias
            return (q[:, 0] << 42) | (q[:, 1] << 21) | q[:, 2]

        packable = torch.isfinite(pos).all(-1) & (pos >= -bias).all(-1) & (pos < lim - bias).all(-1)
        key = pack(torch.where(packable[:, None], pos, torch.zeros_like(pos)))
        vkey, order = torch.sort(pack(grid), stable=True)  # ties keep list order: first match
        at = torch.searchsorted(vkey, key).clamp(max=vkey.shape[0] - 1)
        valid = packable & (vkey[at] == key)
        colors = torch.zeros_like(verts)
        sel = valid.nonzero().squeeze(1)
        idx = order[at[sel]]
        for s in range(0, int(sel.shape[0]), self.query_chunk):
            rows = sel[s:s + self.query_chunk]
            colors[rows] = self.model.query(verts[rows], idx[s:s + self.query_chunk], centres,
                                            features)[:, :3]
        return colors

