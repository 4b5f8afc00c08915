"""Algorithm base: the optimisation loop around the fused step (host-side mirror
of slam/algorithms/base_algorithm.py:17-302; same hooks, same loop order)."""
from __future__ import annotations

import random
import threading
from abc import abstractmethod
from dataclasses import dataclass, field
from typing import Any, Dict, Type

import torch

from .base_model import InstantiateConfig, ModelConfig
from .optimizers import OptimizerConfig, Optimizers


@dataclass
class AlgorithmConfig(InstantiateConfig):
    _target: Type = field(default_factory=lambda: Algorithm)
    model: ModelConfig = field(default_factory=ModelConfig)
    keyframe_selection_method: str = 'overlap'
    keyframe_use_ray_sample: bool = True
    tracking_n_iters: int = 10
    mapping_n_iters: int = 60
    mapping_first_n_iters: int = 200
    coarse: bool = False
    mapping_window_size: int = 5
    separate_LR: bool = False
    rot_rep: str = 'quat'
    retain_graph: bool = False
    optimizers: Dict[str, Any] = field(default_factory=lambda: {
        'model': {'optimizer': OptimizerConfig(lr=1e-2), 'scheduler': None},
        'tracking_pose': {'optimizer': OptimizerConfig(lr=1e-2), 'scheduler': None},
        'mapping_pose': {'optimizer': OptimizerConfig(lr=1e-3), 'scheduler': None},
    })

    def setup(self, **kwargs):
        return self._target(self, **kwargs)


class Algorithm():
    def __init__(self, config: AlgorithmConfig, camera, device: str) -> None:
        self.config = config
        self.camera = camera
        self.initialized = False
        self.finished = False
        self.lock = threading.RLock()
        self.gt_c2w_list = []
        self.gt_c2w_list_ori = []
        self.estimate_c2w_list = []
        self.keyframe_graph = []
        self.bundle_adjust = False

    # ---- hooks (docs/adding_a_new_algorithm.md) ---------------------------
    @abstractmethod
    def get_model_input(self, optimize_frames, is_mapping):
        pass

    @abstractmethod
    def get_loss(self, optimize_frames, is_mapping, step=None, n_iters=None,
                 coarse=False):
        pass

    def pre_precessing(self, cur_frame, is_mapping):
        pass

    def post_processing(self, step, is_mapping, optimizer=None, coarse=False):
        pass

    def render_img(self, c2w, gt_depth=None, idx=None):
        return None, None

    def get_mesh(self):
        """base_algorithm.py:89-91: algorithms without a mesher return None."""
        return None

    def optimizer_config_update(self, max_iters, coarse=False):
        pass

    @property
    def device(self):
        return self.model.device

    def _frame_tensor(self, frame, which):
        """Upload a frame's image once and keep it resident on the device (the reference
        re-uploads the full image every iteration, common.py:67-68 -- SURVEY row f1)."""
        import numpy as np
        key = '_dev_' + which
        t = frame.__dict__.get(key)
        if t is None:
            t = torch.as_tensor(np.asarray(getattr(frame, which), dtype=np.float32)
                                ).to(self.device)
            frame.__dict__[key] = t
        return t

    def _sample_window(self, frames, n, Hedge=0, Wedge=0, return_index=False):
        """All frames of the window at once: one batched pose evaluation, one H2D, three
        launches (csrc/rays.cu) -- instead of ~150 ATen launches and a host Rodrigues /
        quaternion chain per frame."""
        from .common import sample_window
        from .opt_pose import pose_matrices
        poses = pose_matrices([f.pose for f in frames]).to(self.device)
        return sample_window(self.camera, [self._frame_tensor(f, 'depth') for f in frames],
                             [self._frame_tensor(f, 'rgb') for f in frames], poses, n, Hedge,
                             Wedge, return_index=return_index)

    def _render_full(self, c2w, gt_depth, extra=None, per_pixel=None):
        """render_img body shared by the algorithms: all H*W rays in ray_batch_size chunks."""
        import numpy as np
        from .common import get_rays
        dev = self.device
        rays_o, rays_d = get_rays(self.camera, torch.as_tensor(c2w), device=dev)
        rays_o, rays_d = rays_o.reshape(-1, 3), rays_d.reshape(-1, 3)
        if gt_depth is not None:
            gt_depth = torch.as_tensor(np.asarray(gt_depth), dtype=torch.float32).to(dev
                                                                                     ).reshape(-1, 1)
        depths, colors = [], []
        bs = self.config.ray_batch_size
        for i in range(0, rays_d.shape[0], bs):
            batch = {'rays_o': rays_o[i:i + bs], 'rays_d': rays_d[i:i + bs], 'target_s': None,
                     'target_d': gt_depth[i:i + bs] if gt_depth is not None else None}
            batch.update(extra or {})
            for k, v in (per_pixel or {}).items():
                batch[k] = v[i:i + bs]
            out = self.model(batch)
            depths.append(out['depth'].double())
            colors.append(out['rgb'])
        H, W = self.camera.height, self.camera.width
        return (torch.cat(colors, 0).reshape(H, W, 3).cpu().numpy(),
                torch.cat(depths, 0).reshape(H, W).cpu().numpy())

    # ---- bookkeeping ------------------------------------------------------
    def add_framepose(self, c2w, gt_c2w, gt_c2w_ori):
        with self.lock:
            self.estimate_c2w_list.append(c2w)
            self.gt_c2w_list.append(gt_c2w)
            self.gt_c2w_list_ori.append(gt_c2w_ori)

    def update_framepose(self, idx, c2w):
        with self.lock:
            self.estimate_c2w_list[idx] = c2w

    def get_keyframes(self):
        return self.keyframe_graph

    def add_keyframe(self, keyframe):
        with self.lock:
            self.keyframe_graph.append(keyframe)

    # accessors the pipeline processes call through the Manager proxy
    # (base_algorithm.py:116-158; slam/pipeline/{tracker,mapper,xrdslam}.py)
    def get_estimate_c2w_list(self):
        with self.lock:
            return self.estimate_c2w_list

    def get_gt_c2w_list(self):
        with self.lock:
            return self.gt_c2w_list

    def get_gt_c2w_list_ori(self):
        with self.lock:
            return self.gt_c2w_list_ori

    def save_eval(self, out_dir, idx):
        """The trajectory checkpoint `ds-eval` reads (tracker.py:269-278, 410-420)."""
        from .io_formats import save_eval_tar
        return save_eval_tar(self, out_dir, idx)

    def is_separate_LR(self):
        with self.lock:
            return self.config.separate_LR

    def get_rot_rep(self):
        with self.lock:
            return self.config.rot_rep

    def is_initialized(self):
        with self.lock:
            return self.initialized

    def set_initialized(self):
        with self.lock:
            self.initialized = True

    def is_finished(self):
        with self.lock:
            return self.finished

    def set_finished(self):
        with self.lock:
            self.finished = True

    @staticmethod
    def release_frame_tensors(frame):
        """Drop the device-resident copies of a frame's images (_frame_tensor).  Called for
        frames that leave the optimisation window without becoming keyframes; keyframe
        containers that keep their images decide for themselves."""
        for k in ('_dev_depth', '_dev_rgb', '_ray_table'):
            frame.__dict__.pop(k, None)

    # ---- optimisation -----------------------------------------------------
    def setup_optimizers(self, n_iters, optimize_frames, is_mapping=True,
                         coarse=False) -> Optimizers:
        """base_algorithm.py:160-209."""
        self.optimizer_config_update(n_iters, coarse)
        cfg = dict(self.config.optimizers)
        sep = self.config.separate_LR
        if not is_mapping:
            frame = optimize_frames[0]
            if sep:
                r, t = frame.get_params()[:2]
                return Optimizers(cfg, {'tracking_pose_r': [r],
                                        'tracking_pose_t': [t]})
            return Optimizers(cfg, {'tracking_pose': frame.get_params()})
        model_params = self.model.get_param_groups()
        if not self.bundle_adjust or len(optimize_frames) == 1:
            return Optimizers(cfg, {**model_params})
        pose_params = ({'mapping_pose_r': [], 'mapping_pose_t': []}
                       if sep else {'mapping_pose': []})
        oldest = min(f.fid for f in optimize_frames)
        for kf in optimize_frames:
            if kf.fid == oldest:
                continue  # fixed to avoid drift
            if sep:
                pose_params['mapping_pose_r'].append(kf.get_params()[0])
                pose_params['mapping_pose_t'].append(kf.get_params()[1])
            else:
                pose_params['mapping_pose'].extend(kf.get_params())
        return Optimizers(cfg, {**pose_params, **model_params})

    def do_tracking(self, cur_frame):
        if self.is_initialized():
            return self.optimize_update(self.config.tracking_n_iters,
                                        [cur_frame], is_mapping=False)

    def finish_frame(self, frame):
        """The pipeline is done with `frame` (tracked, and mapped if it was a map frame):
        free its device images unless a keyframe container still needs them."""
        if not any(frame is kf for kf in self.keyframe_graph):
            self.release_frame_tensors(frame)

    def do_mapping(self, cur_frame):
        n_iters = (self.config.mapping_n_iters if self.is_initialized() else
                   self.config.mapping_first_n_iters)
        with torch.no_grad():
            frames = self.select_optimize_frames(
                cur_frame, self.config.keyframe_selection_method)
        self.optimize_update(n_iters, frames, is_mapping=True, coarse=False)
        if not self.is_initialized():
            self.set_initialized()

    def optimize_update(self, n_iters, optimize_frames, is_mapping,
                        coarse=False):
        """The hot loop (base_algorithm.py:239-275)."""
        with self.lock:
            self.pre_precessing(optimize_frames[-1], is_mapping)
            optimizers = self.setup_optimizers(n_iters, optimize_frames,
                                               is_mapping, coarse=coarse)
            candidate_c2w = None
            current_min_loss = 10000000000.
            for step in range(n_iters):
                optimizers.zero_grad_all()
                loss = self.get_loss(optimize_frames, is_mapping, step,
                                     n_iters, coarse=coarse)
                if not is_mapping:
                    lv = loss.detach().cpu().item()
                    if lv < current_min_loss:
                        current_min_loss = lv
                        candidate_c2w = optimize_frames[-1].get_pose().detach(
                        ).clone().cpu().numpy()
                loss.backward(
                    retain_graph=(self.config.retain_graph and is_mapping))
                self.post_processing(step, is_mapping, optimizers.optimizers,
                                     coarse=coarse)
                optimizers.optimizer_step_all(step=step)
                optimizers.scheduler_step_all()
            return candidate_c2w

    def select_optimize_frames(self, cur_frame, keyframe_selection_method):
        """base_algorithm.py:277-302 ('overlap' -> keyframe_selection_overlap is
        SURVEY row f3; 'random' / 'all' are the methods used by co-slam)."""
        window = self.config.mapping_window_size
        kfs = self.keyframe_graph
        if len(kfs) <= window or keyframe_selection_method == 'all':
            frames = list(kfs)
        elif keyframe_selection_method == 'random':
            frames = random.sample(kfs[:-1], window - 2) + [kfs[-1]]
        elif keyframe_selection_method == 'overlap':
            from .keyframe_selection import keyframe_selection_overlap
            frames = keyframe_selection_overlap(
                self.camera, cur_frame, kfs[:-1], window - 2,
                use_ray_sample=self.config.keyframe_use_ray_sample,
                device=self.device) + [kfs[-1]]
        else:
            raise ValueError(keyframe_selection_method)
        if cur_frame is not None:
            frames = frames + [cur_frame]
        return frames
