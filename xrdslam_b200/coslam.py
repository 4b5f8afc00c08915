"""Co-SLAM algorithm (host-side mirror of slam/algorithms/coslam.py): global
keyframe ray bank, per-ray pose gather for bundle adjustment, persistent model
optimizers -- driving the fused B200 step in joint_encoding.py."""
from __future__ import annotations

import functools
import random
from dataclasses import dataclass, field
from typing import Any, Dict, List, Type

import numpy as np
import torch

from .algorithm import Algorithm, AlgorithmConfig
from .common import get_camera_rays, get_rays, get_samples, rays_from_poses
from .joint_encoding import JointEncodingConfig
from .mesher import MesherConfig
from .opt_pose import pose_matrices
from .optimizers import AdamOptimizerConfig, Optimizers


def _coslam_optimizers():
    """slam/configs/input_config.py:255-292."""
    A = AdamOptimizerConfig
    return {
        'decoder': {'optimizer': A(lr=1e-2, weight_decay=1e-6, betas=(0.9, 0.99)),
                    'scheduler': None},
        'embed_fn': {'optimizer': A(lr=1e-2, eps=1e-15, betas=(0.9, 0.99)),
                     'scheduler': None},
        'embed_fn_color': {'optimizer': A(lr=1e-2, eps=1e-15, betas=(0.9, 0.99)),
                           'scheduler': None},
        'tracking_pose_r': {'optimizer': A(lr=1e-3), 'scheduler': None},
        'tracking_pose_t': {'optimizer': A(lr=1e-3), 'scheduler': None},
        'mapping_pose_r': {'optimizer': A(lr=1e-3, accum_step=5), 'scheduler': None},
        'mapping_pose_t': {'optimizer': A(lr=1e-3, accum_step=5), 'scheduler': None},
    }


@dataclass
class CoSLAMConfig(AlgorithmConfig):
    """coslam.py:17-38 + the co-slam entry of input_config.py:203-296."""
    _target: Type = field(default_factory=lambda: CoSLAM)
    model: JointEncodingConfig = field(default_factory=lambda: JointEncodingConfig(
        cam_depth_trunc=100.0, tcnn_encoding=True))
    mesher: MesherConfig = field(default_factory=MesherConfig)
    separate_LR: bool = True
    retain_graph: bool = True
    rot_rep: str = 'axis_angle'
    tracking_n_iters: int = 10
    mapping_n_iters: int = 10
    mapping_first_n_iters: int = 200
    keyframe_selection_method: str = 'all'
    rays_to_save_ratio: float = 0.05
    tracking_Wedge: int = 20
    tracking_Hedge: int = 20
    mapping_sample: int = 2048
    min_sample_pixels: int = 100
    tracking_sample: int = 1024
    ray_batch_size: int = 30000
    marching_cubes_bound: List[List[float]] = field(
        default_factory=lambda: [[-2.2, 2.6], [-3.4, 2.1], [-1.4, 2.0]])
    mapping_bound: List[List[float]] = field(
        default_factory=lambda: [[-3, 3], [-4, 2.5], [-2, 2.5]])
    optimizers: Dict[str, Any] = field(default_factory=_coslam_optimizers)
    # B200: run the mapping iterations as one CUDA graph each (coslam_graph.py)
    graph_mapping: bool = True


class _PinnedStaging:
    """Ring of pinned host blocks for the per-iteration ray rows [n,7] + pose ids [n]: the
    host gathers into a block, two async copies move it to the device, an event per block
    guards its reuse (iterations are not synchronised with the host)."""
    def __init__(self, depth=4):
        self.depth, self.slots, self.k, self.cur = depth, [], 0, None

    def acquire(self, n):
        if len(self.slots) < self.depth:
            self.slots.append(dict(rows=torch.empty(0, 7).pin_memory(),
                                   ids=torch.empty(0, dtype=torch.int64).pin_memory(),
                                   ev=None))
        sl = self.slots[self.k % self.depth]
        self.k += 1
        if sl['ev'] is not None:
            sl['ev'].synchronize()
        if sl['rows'].shape[0] < n:
            sl['rows'] = torch.empty(n, 7).pin_memory()
            sl['ids'] = torch.empty(n, dtype=torch.int64).pin_memory()
        self.cur = (sl, n)
        return sl['rows'][:n], sl['ids'][:n]

    def upload(self, dev):
        sl, n = self.cur
        rows = sl['rows'][:n].to(dev, non_blocking=True)
        ids = sl['ids'][:n].to(dev, non_blocking=True)
        if sl['ev'] is None:
            sl['ev'] = torch.cuda.Event()
        sl['ev'].record(torch.cuda.current_stream(dev))
        return rows, ids


class CoSLAM(Algorithm):
    def __init__(self, config: CoSLAMConfig, camera, device: str) -> None:
        super().__init__(config, camera, device)
        self.bounding_box = torch.from_numpy(np.array(self.config.mapping_bound))
        self.marching_cube_bound = torch.from_numpy(
            np.array(self.config.marching_cubes_bound))
        self.model = self.config.model.setup(camera=camera,
                                             bounding_box=self.bounding_box)
        self.model.to(device)
        self.mesher = self.config.mesher.setup(camera=camera, bounding_box=self.bounding_box,
                                               marching_cubes_bound=self.marching_cube_bound)
        self.cur_mesh = None
        self.bundle_adjust = True
        self.num_rays_to_save = int(self.camera.width * self.camera.height *
                                    self.config.rays_to_save_ratio)
        self.rays = None  # [n_kf * num_rays_to_save, 7] pinned host memory
        self._staging = _PinnedStaging()
        self.model_optimizers = None
        self._rng = np.random.default_rng(random.getrandbits(63))
        self._cam_dirs = get_camera_rays(camera.height, camera.width, camera.fx,
                                         camera.fy, camera.cx, camera.cy)

    # coslam.py:66-112
    def setup_optimizers(self, n_iters, optimize_frames, is_mapping=True,
                         coarse=False) -> Optimizers:
        cfg = dict(self.config.optimizers)
        if not is_mapping:
            return super().setup_optimizers(n_iters, optimize_frames, False)
        if self.model_optimizers is None:
            self.model_optimizers = Optimizers(cfg, {**self.model.get_param_groups()})
        if not self.bundle_adjust or len(optimize_frames) == 1:
            return self.model_optimizers
        sep = self.config.separate_LR
        pose_params = ({'mapping_pose_r': [], 'mapping_pose_t': []}
                       if sep else {'mapping_pose': []})
        for kf in optimize_frames[1:]:  # first frame's pose stays fixed
            if sep:
                pose_params['mapping_pose_r'].append(kf.get_params()[0])
                pose_params['mapping_pose_t'].append(kf.get_params()[1])
            else:
                pose_params['mapping_pose'].extend(kf.get_params())
        return Optimizers(cfg, {**pose_params}) + self.model_optimizers

    # coslam.py:114-125
    def _sample_ids(self, n, bs):
        """bs distinct indices in [0,n) -- random.sample's distribution
        (coslam.py:122,147) drawn with numpy's Floyd sampler (O(bs))."""
        return torch.from_numpy(self._rng.choice(n, size=bs, replace=False,
                                                 shuffle=False))

    def _frame_rays(self, keyframe):
        """[H*W,7] (dir_cam, rgb, depth) table of a frame, built once."""
        t = keyframe.__dict__.get('_ray_table')
        if t is None:
            depth = torch.from_numpy(np.asarray(keyframe.depth, dtype=np.float32))
            color = torch.from_numpy(np.asarray(keyframe.rgb, dtype=np.float32))
            t = torch.cat([self._cam_dirs, color, depth[..., None]],
                          dim=-1).reshape(-1, 7)
            keyframe.__dict__['_ray_table'] = t
        return t

    def sample_single_keyframe_rays(self, keyframe, bs):
        rays = self._frame_rays(keyframe)
        return rays[self._sample_ids(rays.shape[0], bs)]

    def add_keyframe(self, keyframe):
        with self.lock:
            rays = self.sample_single_keyframe_rays(keyframe, self.num_rays_to_save)
            self.rays = rays if self.rays is None else torch.cat([self.rays, rays], 0)
            if torch.cuda.is_available():
                self.rays = self.rays.pin_memory()
            keyframe.rgb = None
            keyframe.depth = None
            # the full-resolution copies made for sampling / tracking are dropped with the
            # images (the reference keeps only the ray bank, coslam.py:133-137)
            for k in ('_ray_table', '_dev_depth', '_dev_rgb'):
                keyframe.__dict__.pop(k, None)
            self.keyframe_graph.append(keyframe)

    def sample_global_rays(self, bs):
        n_kf = len(self.keyframe_graph)
        idxs = self._sample_ids(n_kf * self.num_rays_to_save, bs)
        return self.rays[idxs], idxs // self.num_rays_to_save

    # coslam.py:152-230
    def get_model_input(self, optimize_frames, is_mapping):
        cur_frame = optimize_frames[-1]
        dev = self.device
        if is_mapping:
            # host side: choose rows (random.sample semantics) and gather them straight
            # into a pinned staging block; device side: ONE copy of the rows, one of the
            # pose ids, rays built by csrc/rays.cu (per-ray pose gather + its backward).
            n_kf = len(self.keyframe_graph)
            n_bank = self.config.mapping_sample if n_kf > 0 else 0
            n_cur = self.config.mapping_sample
            if n_kf > 0:
                n_cur = int(np.maximum(self.config.mapping_sample // n_kf,
                                       self.config.min_sample_pixels))
            n = n_bank + n_cur
            rows, ids = self._staging.acquire(n) if dev.type == 'cuda' else (
                torch.empty(n, 7), torch.empty(n, dtype=torch.int64))
            pose_list, detach = [], []
            if n_kf > 0:
                if len(optimize_frames) != n_kf + 1:
                    # bank ids index the whole keyframe graph; the reference's
                    # poses_all[ids_all] (coslam.py:208) raises the same way when the
                    # window is a subset (keyframe_selection_method != 'all')
                    raise IndexError(
                        f'co-slam mapping window has {len(optimize_frames) - 1} keyframes but '
                        f'the ray bank indexes {n_kf}: use keyframe_selection_method="all"')
                idxs = self._sample_ids(n_kf * self.num_rays_to_save, n_bank)
                torch.index_select(self.rays, 0, idxs, out=rows[:n_bank])
                torch.div(idxs, self.num_rays_to_save, rounding_mode='floor',
                          out=ids[:n_bank])
                for frame in optimize_frames[:-1]:
                    pose_list.append(frame.pose)
                    detach.append(frame.fid == 0)
            cur_tab = self._frame_rays(cur_frame)
            torch.index_select(cur_tab, 0, self._sample_ids(cur_tab.shape[0], n_cur),
                               out=rows[n_bank:])
            ids[n_bank:] = -1  # the current frame's pose is appended last
            pose_list.append(cur_frame.pose)
            detach.append(False)
            poses_all = pose_matrices(pose_list, detach).to(dev)
            if dev.type == 'cuda':
                rays_all, ids_all = self._staging.upload(dev)
            else:
                rays_all, ids_all = rows, ids
            target_s = rays_all[..., 3:6]
            target_d = rays_all[..., 6:7]
            rays_o, rays_d = rays_from_poses(rays_all[..., :3], ids_all, poses_all)
            first_flag = len(self.keyframe_graph) == 0
        else:
            rays_o, rays_d, target_d, target_s = self._sample_window(
                [cur_frame], self.config.tracking_sample, self.config.tracking_Hedge,
                self.config.tracking_Wedge)
            first_flag = False
        return {
            'rays_o': rays_o.float(),
            'rays_d': rays_d.float(),
            'target_s': target_s.float(),
            'target_d': target_d.float(),
            'first': first_flag,
        }

    # ---- CUDA-graph mapping (row f1) -------------------------------------------------
    def _graph_ok(self, optimize_frames):
        cfg = self.config
        if not (cfg.graph_mapping and self.device.type == 'cuda' and cfg.separate_LR
                and cfg.rot_rep == 'axis_angle'):
            return False
        n_kf = len(self.keyframe_graph)
        return n_kf == 0 or len(optimize_frames) == n_kf + 1  # ids index the window 1:1

    def mapping_session(self, optimize_frames):
        """The captured iteration for this window shape (cached by shape)."""
        from .coslam_graph import MappingGraphSession
        n_kf = len(self.keyframe_graph)
        first = n_kf == 0
        n_bank = 0 if first else self.config.mapping_sample
        n_cur = self.config.mapping_sample if first else int(np.maximum(
            self.config.mapping_sample // n_kf, self.config.min_sample_pixels))
        ba = self.bundle_adjust and len(optimize_frames) > 1
        key = (n_bank, n_cur, len(optimize_frames), first, ba)
        # ONE live session: under keyframe_selection 'all' the window grows with every keyframe,
        # so the shape key changes for good -- the previous session (flat gradient bucket the
        # size of the hash table, raw outputs, workspace, the graph's private pool) is released
        # before the new one is captured instead of piling up over a sequence.
        cache = self.__dict__.setdefault('_graph_sessions', {})
        for k in [k for k in cache if k != key]:
            cache.pop(k).release()
        if key in cache and (cache[key].stale() or
                             cache[key].opt_groups[0][0] is not self.model_optimizers.optimizers['embed_fn']):
            cache.pop(key).release()  # optimiser state / parameters were replaced: re-capture
        if key not in cache:
            cache[key] = MappingGraphSession(self, n_bank, n_cur, len(optimize_frames), first, ba)
        return cache[key]

    def tracking_session(self):
        from .coslam_graph import TrackingGraphSession
        key = (self.config.tracking_sample, self.config.tracking_Hedge, self.config.tracking_Wedge)
        s = self.__dict__.get('_track_session')
        if s is None or s.key != key:  # the sample count / crop are baked into the graph
            s = self.__dict__['_track_session'] = TrackingGraphSession(self)
            s.key = key
        return s

    def optimize_update(self, n_iters, optimize_frames, is_mapping, coarse=False):
        cfg = self.config
        if not is_mapping and cfg.graph_mapping and self.device.type == 'cuda' and \
                cfg.separate_LR and cfg.rot_rep == 'axis_angle':
            with self.lock:
                sess = self.tracking_session()
                sess.begin(optimize_frames[-1])
                for _ in range(n_iters):
                    sess.step()
                return sess.end(optimize_frames[-1])
        if not is_mapping or not self._graph_ok(optimize_frames):
            return super().optimize_update(n_iters, optimize_frames, is_mapping, coarse=coarse)
        with self.lock:
            self.pre_precessing(optimize_frames[-1], True)
            self.setup_optimizers(n_iters, optimize_frames, True, coarse=coarse)
            sess = self.mapping_session(optimize_frames)
            sess.begin(optimize_frames)
            for step in range(n_iters):
                sess.step(step, optimize_frames)
            sess.end(optimize_frames)
            return None

    def get_loss(self, optimize_frames, is_mapping, step=None, n_iters=None,
                 coarse=False):
        # tracking optimises the pose only: no map gradients are needed
        self.model.freeze_map_grads = not is_mapping
        model_input = self.get_model_input(optimize_frames, is_mapping)
        model_outputs = self.model(model_input)
        loss_dict = self.model.get_loss_dict(model_outputs, model_input,
                                             is_mapping, step)
        return functools.reduce(torch.add, loss_dict.values())

    # coslam.py:245-289
    def render_img(self, c2w, gt_depth=None, idx=None):
        with self.lock, torch.no_grad():
            dev = self.device
            rays_o, rays_d = get_rays(self.camera, c2w, device=dev)
            rays_o, rays_d = rays_o.reshape(-1, 3), rays_d.reshape(-1, 3)
            if gt_depth is not None:
                gt_depth = torch.as_tensor(gt_depth, dtype=torch.float32
                                           ).to(dev).reshape(-1, 1)
            depths, colors = [], []
            bs = self.config.ray_batch_size
            for i in range(0, rays_d.shape[0], bs):
                batch = {'rays_o': rays_o[i:i + bs], 'rays_d': rays_d[i:i + bs],
                         'target_s': None, 'target_d': None}
                if gt_depth is not None:
                    batch['target_d'] = gt_depth[i:i + bs]
                out = self.model(batch)
                depths.append(out['depth'].double())
                colors.append(out['rgb'])
            depth = torch.cat(depths, 0).reshape(self.camera.height,
                                                 self.camera.width)
            color = torch.cat(colors, 0).reshape(self.camera.height,
                                                 self.camera.width, 3)
            return color.cpu().numpy(), depth.cpu().numpy()

    # coslam.py:291-298
    def get_mesh(self):
        with self.lock:
            self.cur_mesh = self.mesher.get_mesh(keyframe_graph=self.keyframe_graph,
                                                 query_fn=self.model.query_fn,
                                                 color_func=self.model.color_func,
                                                 device=self.device)
            return self.cur_mesh
