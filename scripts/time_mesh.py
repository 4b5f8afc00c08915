"""Mesh extraction timing on a B200 (one JSON line on stdout).

Co-SLAM and NICE-SLAM: Algorithm.get_mesh() at lattice resolution 256 (16.8 M query points);
Vox-Fusion: get_mesh() (8^3 lattice per voxel) -- each after a few mapping iterations on the
640x480 synthetic sequence of bench_workloads.py.  Per algorithm: device ms by CUDA events of
the lattice query, xrd_mc_count, xrd_mc_emit and the colour query (median over the timed calls)
and end-to-end ms of get_mesh() by the host clock, including the copies of the finished mesh.

    python scripts/time_mesh.py [--calls 3] [--resolution 256] [--map-iters 30]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


class Spans:
    """CUDA-event spans around wrapped callables; a call nested in another span counts there."""

    def __init__(self):
        self.ev = defaultdict(list)
        self.active = []

    def wrap(self, obj, attr, label):
        f = getattr(obj, attr)

        def w(*a, **k):
            if self.active:
                return f(*a, **k)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.active.append(label)
            s.record()
            try:
                return f(*a, **k)
            finally:
                e.record()
                self.active.pop()
                self.ev[label].append((s, e))
        setattr(obj, attr, w)

    def take(self):
        torch.cuda.synchronize()
        out = {k: sum(s.elapsed_time(e) for s, e in v) for k, v in self.ev.items()}
        self.ev.clear()
        return out


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader',
                             '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return name, pl


def time_algo(algo, wrap, calls):
    from xrdslam_b200.mesher import MarchingCubes
    sp = Spans()
    wrap(sp)
    sp.wrap(MarchingCubes, 'count', 'mc_count')
    sp.wrap(MarchingCubes, 'emit', 'mc_emit')
    mesh = algo.get_mesh()  # warm-up
    sp.take()
    stages, e2e = defaultdict(list), []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mesh = algo.get_mesh()
        e2e.append((time.perf_counter() - t0) * 1e3)
        for k, v in sp.take().items():
            stages[k].append(v)
    out ={f'{k}_ms': float(np.median(v)) for k, v in stages.items()}
    out['e2e_ms'] = float(np.median(e2e))
    out['V'] = 0 if mesh is None else int(mesh.vertices.shape[0])
    out['F'] = 0 if mesh is None else int(mesh.faces.shape[0])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=3)
    ap.add_argument('--resolution', type=int, default=256)
    ap.add_argument('--map-iters', type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('time_mesh.py needs a CUDA device')
    dev = torch.device('cuda:0')
    import bench_workloads as bw
    from xrdslam_b200 import mesher
    from xrdslam_b200.coslam import CoSLAMConfig
    orig = {k: getattr(mesher.MarchingCubes, k) for k in ('count', 'emit')}
    res = {}

    def mesher_spans(algo):
        def wrap(sp):
            sp.wrap(algo.mesher, 'get_field', 'lattice_query')
            sp.wrap(algo.mesher, 'get_colors', 'colour_query')
        return wrap

    torch.manual_seed(0)
    cam, frs = bw._frames(5, rot_rep='axis_angle', separate_LR=True)
    co = CoSLAMConfig().setup(camera=cam, device=dev)
    co.optimize_update(args.map_iters, [frs[0]], True)
    co.mesher.config.resolution = args.resolution
    res['coslam'] = time_algo(co, mesher_spans(co), args.calls)
    for k, f in orig.items():
        setattr(mesher.MarchingCubes, k, f)
    del co

    nw = bw.NiceWorkload(dev)
    nw.build()
    nw.begin(args.map_iters)
    for i in range(args.map_iters):
        nw.step(i)
    nw.algo.mesher.config.resolution = args.resolution
    res['nice'] = time_algo(nw.algo, mesher_spans(nw.algo), args.calls)
    for k, f in orig.items():
        setattr(mesher.MarchingCubes, k, f)
    del nw

    vw = bw.VoxWorkload(dev)
    vw.build()
    vw.begin(args.map_iters)
    for i in range(args.map_iters):
        vw.step(i)
    va = vw.algo

    def vox_wrap(sp):
        sp.wrap(va, 'vertex_colors', 'colour_query')
        sp.wrap(va.model, 'query', 'lattice_query')
    res['vox'] = time_algo(va, vox_wrap, args.calls)
    res['vox']['voxels'] = int(va.model.map_states['voxel_center_xyz'].shape[0])
    for k, f in orig.items():
        setattr(mesher.MarchingCubes, k, f)

    name, pl = card()
    print(json.dumps({'card': name, 'power_limit': pl, 'resolution': args.resolution,
                      'map_iters': args.map_iters, 'calls': args.calls, 'results': res}))


if __name__ == '__main__':
    main()
