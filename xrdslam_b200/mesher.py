"""Mesh extraction on the device (host-side mirror of slam/common/mesher.py).

The reference evaluates the field on a uniform lattice in 500 k-point chunks, copies the whole
field to the host and runs skimage's marching cubes there.  Here the lattice is generated on
the device, the field stays there, marching cubes runs in csrc/mesh.cu (xrd_mc_count /
xrd_mc_emit) and only the counts (V, F) and the finished mesh cross to the host.
The TSDF / convex-hull mask of the reference (``use_mask=True``, get_bound_from_frames) needs
open3d and is not provided.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Type

import numpy as np
import torch

from . import _cabi
from ._cabi import XrdMcVolumes, check, ptr
from .base_model import InstantiateConfig
from .io_formats import write_ply


class Mesh:
    """The parts of ``trimesh.Trimesh`` the pipeline uses (tracker.py:247-257): host arrays
    vertices f32 [V,3], faces i32 [F,3], vertex_colors [V,3] (uint8, or float in [0,1] which
    ``write_ply`` quantises) or None."""

    def __init__(self, vertices, faces, vertex_colors=None):
        self.vertices = vertices
        self.faces = faces
        self.vertex_colors = vertex_colors

    def export(self, path):
        return write_ply(path, self.vertices, self.faces, self.vertex_colors)


class MarchingCubes:
    """xrd_mc_count + xrd_mc_emit over a batch of device volumes ``field`` [B,nx,ny,nz] fp32.
    ``origin`` / ``spacing``: 3 floats shared by all volumes, or ``origins`` / ``spacings``:
    device float64 [B,3] per volume."""

    def __init__(self, field, level=0.0, origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0),
                 origins=None, spacings=None):
        if field.dim() == 3:
            field = field[None]
        if field.dtype != torch.float32 or field.device.type != 'cuda':
            raise ValueError('marching cubes needs an fp32 field on a CUDA device')
        self.field = field.contiguous()
        self.dev = field.device
        self.origins = None if origins is None else origins.to(self.dev, torch.float64).contiguous()
        self.spacings = None if spacings is None else spacings.to(self.dev, torch.float64).contiguous()
        B, nx, ny, nz = self.field.shape
        self.level = float(level)
        self.vol = XrdMcVolumes(ptr(self.field), B, nx, ny, nz, (C.c_double * 3)(*origin),
                                (C.c_double * 3)(*spacing), ptr(self.origins), ptr(self.spacings))
        self.ws_bytes = _cabi.lib().xrd_mc_workspace_bytes(B, nx, ny, nz)
        self.ws = torch.empty(max(self.ws_bytes, 1), dtype=torch.uint8, device=self.dev)
        self.counts = torch.zeros(2, dtype=torch.int32, device=self.dev)

    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def count(self):
        """Enqueue the count phase; returns the device tensor (V, F)."""
        with torch.cuda.device(self.dev):
            st = _cabi.lib().xrd_mc_count(C.byref(self.vol), self.level, ptr(self.counts),
                                          ptr(self.ws), self.ws_bytes, self._stream())
        check('xrd_mc_count', st)
        return self.counts

    def emit(self, n_verts, n_faces):
        """Enqueue the emit phase into freshly allocated device outputs."""
        verts = torch.empty(n_verts, 3, dtype=torch.float32, device=self.dev)
        faces = torch.empty(n_faces, 3, dtype=torch.int32, device=self.dev)
        with torch.cuda.device(self.dev):
            st = _cabi.lib().xrd_mc_emit(C.byref(self.vol), self.level, ptr(verts), ptr(faces),
                                         ptr(self.ws), self.ws_bytes, self._stream())
        check('xrd_mc_emit', st)
        return verts, faces

    def run(self):
        """-> device (verts [V,3] f32, faces [F,3] i32); one host read of (V, F)."""
        n_verts, n_faces = self.count().tolist()
        return self.emit(n_verts, n_faces)


@dataclass
class MesherConfig(InstantiateConfig):
    """slam/common/mesher.py:19-29 (field names and defaults kept; the last three belong to the
    reference's mesh cleaning, kept for config compatibility)."""
    _target: Type = field(default_factory=lambda: Mesher)
    points_batch_size: int = 500000
    resolution: int = 130
    level_set: int = 0
    remove_small_geometry_threshold: float = 0.2
    clean_mesh_bound_scale: float = 1.02
    get_largest_components: bool = False


class Mesher:
    """slam/common/mesher.py:32-263."""

    def __init__(self, config: MesherConfig, camera, bounding_box, marching_cubes_bound) -> None:
        self.config = config
        self.bounding_box = bounding_box
        self.marching_cubes_bound = marching_cubes_bound
        self.camera = camera
        self.scale = 1.0

    def get_grid_uniform(self, resolution):
        """mesher.py:41-66 without the host point table: the three axis vectors (float64, as
        np.linspace makes them)."""
        b = np.asarray(self.marching_cubes_bound, dtype=np.float64)
        return {'xyz': [np.linspace(b[d][0], b[d][1], resolution) for d in range(3)]}

    def lattice_points(self, xyz32, start, end):
        """Lattice points [start, end) in [i][j][k] order (k fastest), fp32 -- the rows of the
        reference's meshgrid point table reordered by reshape(ny,nx,nz).transpose(1,0,2)."""
        x, y, z = xyz32
        ny, nz = y.shape[0], z.shape[0]
        idx = torch.arange(start, end, device=x.device)
        k = idx % nz
        j = (idx // nz) % ny
        i = idx // (nz * ny)
        return torch.stack([x[i], y[j], z[k]], -1)

    def eval_points(self, p, query_fn):
        """mesher.py:138-167 on one chunk: query, then 100 where the point is not strictly
        inside the bounding box."""
        bound = self.bounding_box
        mask_x = (p[:, 0] < bound[0][1]) & (p[:, 0] > bound[0][0])
        mask_y = (p[:, 1] < bound[1][1]) & (p[:, 1] > bound[1][0])
        mask_z = (p[:, 2] < bound[2][1]) & (p[:, 2] > bound[2][0])
        mask = mask_x & mask_y & mask_z
        ret = query_fn(p).reshape(p.shape[0], -1)
        return torch.where(mask[:, None], ret, torch.full_like(ret, 100))

    def get_field(self, query_fn, device, resolution=None):
        """The masked field [nx,ny,nz] fp32 on the device and the axis vectors."""
        res = self.config.resolution if resolution is None else resolution
        xyz = self.get_grid_uniform(res)['xyz']
        xyz32 = [torch.from_numpy(v.astype(np.float32)).to(device) for v in xyz]
        n = res ** 3
        fld = torch.empty(n, dtype=torch.float32, device=device)
        bs = self.config.points_batch_size
        for s in range(0, n, bs):
            e = min(s + bs, n)
            fld[s:e] = self.eval_points(self.lattice_points(xyz32, s, e), query_fn)[:, -1]
        return fld.reshape(res, res, res), xyz

    def marching_cubes(self, fld, xyz):
        """mesher.py:203-233: spacing x[2] - x[1] per axis, origin (x[0], y[0], z[0])."""
        return MarchingCubes(fld, self.config.level_set,
                             origin=tuple(float(v[0]) for v in xyz),
                             spacing=tuple(float(v[2] - v[1]) for v in xyz))

    def get_colors(self, verts, color_func):
        """mesher.py:235-253: clip(color[..., :3], 0, 1) * 255 -> uint8, on the device."""
        out = torch.empty(verts.shape[0], 3, dtype=torch.uint8, device=verts.device)
        bs = self.config.points_batch_size
        for s in range(0, verts.shape[0], bs):
            c = self.eval_points(verts[s:s + bs], color_func)[:, :3]
            out[s:s + bs] = (c.clamp(0, 1) * 255).to(torch.uint8)
        return out

    @torch.no_grad()
    def get_mesh(self, keyframe_graph, query_fn, color_func=None, device='cuda:0',
                 use_mask=False):
        """mesher.py:169-263 -> Mesh, or None when the level set is empty."""
        if use_mask:
            raise NotImplementedError('use_mask=True needs the TSDF / convex-hull bound '
                                      '(open3d), which this package does not provide')
        device = torch.device(device)
        fld, xyz = self.get_field(query_fn, device)
        verts, faces = self.marching_cubes(fld, xyz).run()
        if faces.shape[0] == 0:
            return None  # the reference's marching_cubes error branch
        colors = self.get_colors(verts, color_func) if color_func is not None else None
        verts = verts / self.scale
        return Mesh(verts.cpu().numpy(), faces.cpu().numpy(),
                    None if colors is None else colors.cpu().numpy())
