"""NICE-SLAM algorithm (host-side mirror of slam/algorithms/nice_slam.py): stage schedule
middle -> fine -> color, per-frame pixel sampling with the bounding-box far-plane pre-filter,
frustum feature selection, LambdaLR stage learning rates -- around the CUDA step in
conv_onet.py."""
from __future__ import annotations

import functools
from dataclasses import dataclass, field
from typing import Any, Dict, List, Type

import numpy as np
import torch

from .algorithm import Algorithm, AlgorithmConfig
from .conv_onet import ConvOnetConfig
from .mesher import MesherConfig
from .optimizers import AdamOptimizerConfig
from .schedulers import LRconfig, NiceSLAMSchedulerConfig


def _nice_optimizers():
    """slam/configs/input_config.py:105-152."""
    A, S, L = AdamOptimizerConfig, NiceSLAMSchedulerConfig, LRconfig
    return {
        'decoder': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.0, 0.0, 0.0, 0.005))},
        'grid_coarse': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.001, 0.0, 0.0, 0.0))},
        'grid_middle': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.0, 0.1, 0.005, 0.005))},
        'grid_fine': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.0, 0.0, 0.005, 0.005))},
        'grid_color': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.0, 0.0, 0.0, 0.005))},
        'tracking_pose': {'optimizer': A(lr=1e-3), 'scheduler': None},
        'mapping_pose': {'optimizer': A(), 'scheduler': S(stage_lr=L(0.0, 0.0, 0.0, 0.001))},
    }


@dataclass
class NiceSLAMConfig(AlgorithmConfig):
    """nice_slam.py:14-47 + the nice-slam entry of input_config.py:45-157 (coarse=True there:
    a coarse mapper runs after every mapping call, nice_slam.py:102-109)."""
    _target: Type = field(default_factory=lambda: NiceSLAM)
    model: ConvOnetConfig = field(default_factory=ConvOnetConfig)
    mesher: MesherConfig = field(default_factory=MesherConfig)
    coarse: bool = True
    tracking_n_iters: int = 10
    mapping_n_iters: int = 60
    mapping_first_n_iters: int = 1500
    mapping_window_size: int = 5
    mapping_sample: int = 1000
    min_sample_pixels: int = 200
    tracking_sample: int = 200
    ray_batch_size: int = 100000
    marching_cubes_bound: List[List[float]] = field(
        default_factory=lambda: [[-5.5, 5.9], [-6.7, 5.4], [-4.7, 5.3]])
    mapping_bound: List[List[float]] = field(
        default_factory=lambda: [[-5.5, 5.9], [-6.7, 5.4], [-4.7, 5.3]])
    tracking_Wedge: int = 100
    tracking_Hedge: int = 100
    mapping_middle_iter_ratio: float = 0.4
    mapping_fine_iter_ratio: float = 0.6
    mapping_lr_factor: float = 1.0
    mapping_lr_first_factor: float = 5.0
    mapping_color_refine: bool = True
    optimizers: Dict[str, Any] = field(default_factory=_nice_optimizers)


class NiceSLAM(Algorithm):
    config: NiceSLAMConfig

    def __init__(self, config: NiceSLAMConfig, camera, device: str) -> None:
        super().__init__(config, camera, device)
        self.stage = 'color'
        self.marching_cube_bound = torch.from_numpy(np.array(self.config.marching_cubes_bound))
        self.bounding_box = torch.from_numpy(np.array(self.config.mapping_bound))
        self.config.model.coarse = self.config.coarse
        self.model = self.config.model.setup(camera=camera, bounding_box=self.bounding_box)
        self.model.to(device)
        self.mesher = self.config.mesher.setup(camera=camera, bounding_box=self.bounding_box,
                                               marching_cubes_bound=self.marching_cube_bound)
        self.cur_mesh = None

    # nice_slam.py:72-112
    def do_mapping(self, cur_frame):
        n_iters = (self.config.mapping_n_iters if self.is_initialized() else
                   self.config.mapping_first_n_iters)
        outer = 1
        if cur_frame.is_final_frame and self.config.mapping_color_refine:
            outer = 5
            self.config.mapping_window_size *= 2
            self.config.mapping_middle_iter_ratio = 0.0
            self.config.mapping_fine_iter_ratio = 0.0
            self.model.config.mapping_fix_color = True
            self.model.config.mapping_frustum_feature_selection = False
        for _ in range(outer):
            with torch.no_grad():
                frames = self.select_optimize_frames(
                    cur_frame, self.config.keyframe_selection_method)
            self.optimize_update(n_iters, frames, is_mapping=True, coarse=False)
        if self.config.coarse:  # coarse mapper (nice_slam.py:102-109)
            frames = self.select_optimize_frames(cur_frame, 'random')
            self.optimize_update(n_iters, frames, is_mapping=True, coarse=True)
        if not self.is_initialized():
            self.set_initialized()

    # nice_slam.py:114-131
    def optimizer_config_update(self, max_iters, coarse=False):
        self.bundle_adjust = len(self.keyframe_graph) > 4 and not coarse
        for name, params in self.config.optimizers.items():
            factor = self.config.mapping_lr_factor if (self.is_initialized() or 'pose' in name) \
                else self.config.mapping_lr_first_factor
            if params['scheduler'] is not None:
                params['optimizer'].lr = factor
                sc = params['scheduler']
                sc.max_steps = max_iters
                sc.coarse = coarse
                sc.middle_iter_ratio = self.config.mapping_middle_iter_ratio
                sc.fine_iter_ratio = self.config.mapping_fine_iter_ratio

    def pre_precessing(self, cur_frame, is_mapping):
        if is_mapping:
            self.model.pre_precessing(cur_frame)

    def post_processing(self, step, is_mapping, optimizer=None, coarse=False):
        if is_mapping:
            self.model.post_processing(coarse)

    # nice_slam.py:141-202
    def get_model_input(self, optimize_frames, is_mapping):
        n, Hedge, Wedge = self.config.tracking_sample, self.config.tracking_Hedge, \
            self.config.tracking_Wedge
        if is_mapping:
            n = int(np.maximum(self.config.mapping_sample // len(optimize_frames),
                               self.config.min_sample_pixels))
            Hedge = Wedge = 0
        rays_o, rays_d, gt_depth, gt_color = self._sample_window(optimize_frames, n, Hedge, Wedge)
        with torch.no_grad():  # pre-filter depths beyond the bounding box exit
            det_o = rays_o.detach().unsqueeze(-1)
            det_d = rays_d.detach().unsqueeze(-1)
            t = (self._bbox_dev() - det_o) / det_d
            t, _ = torch.min(torch.max(t, dim=2)[0], dim=1)
            keep = (t >= gt_depth.squeeze(-1)).nonzero().squeeze(1)  # one host sync
        sel = lambda x: x.index_select(0, keep)
        return {'rays_o': sel(rays_o), 'rays_d': sel(rays_d), 'target_s': sel(gt_color),
                'target_d': sel(gt_depth), 'stage': self.stage, 'is_mapping': is_mapping}

    def _bbox_dev(self):
        b = self.__dict__.get('_bbox_dev_t')
        if b is None:
            b = self.bounding_box.unsqueeze(0).to(self.device)
            self.__dict__['_bbox_dev_t'] = b
        return b

    # nice_slam.py:204-216
    def set_stage(self, is_mapping, step, n_iters, coarse=False):
        if not is_mapping:
            self.stage = 'color'
        elif self.model.config.coarse and coarse:
            self.stage = 'coarse'
        elif step <= self.config.mapping_middle_iter_ratio * n_iters:
            self.stage = 'middle'
        elif step <= self.config.mapping_fine_iter_ratio * n_iters:
            self.stage = 'fine'
        else:
            self.stage = 'color'

    def get_loss(self, optimize_frames, is_mapping, step, n_iters, coarse=False):
        self.set_stage(is_mapping, step, n_iters, coarse=coarse)
        if is_mapping:
            self.model.grid_processing(coarse=coarse)
        self.model.freeze_map_grads = not is_mapping  # tracking optimises the pose only
        model_input = self.get_model_input(optimize_frames, is_mapping)
        model_outputs = self.model(model_input)
        loss_dict = self.model.get_loss_dict(model_outputs, model_input, is_mapping, self.stage)
        return functools.reduce(torch.add, loss_dict.values())

    def render_img(self, c2w, gt_depth=None, idx=None):
        with self.lock, torch.no_grad():
            return self._render_full(c2w, gt_depth, extra={'stage': 'color'})

    # nice_slam.py:281-288
    def get_mesh(self):
        with self.lock:
            self.cur_mesh = self.mesher.get_mesh(keyframe_graph=self.keyframe_graph,
                                                 query_fn=self.model.query_fn,
                                                 color_func=self.model.color_func,
                                                 device=self.device)
            return self.cur_mesh
