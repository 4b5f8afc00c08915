#!/usr/bin/env python
"""Benchmark of the xrdslam render-and-optimise hot path on B200.

    python bench.py [--config coslam|nice|vox|point] --gpus N --steps K --warmup W
                    [--impl reference] [--scaling weak|strong]

--config selects the BASELINE.json configuration: coslam = cfg 2 (the default: the
configuration the headline metric is quoted on), vox = cfg 3, nice = cfg 4 (cfg 1 is its
CPU-plumbing shape), point = cfg 5; the three non-default workloads live in
bench_workloads.py.  Everything below describes the default.

Workload (BASELINE.json configs[1]): co-slam hash grid + OneBlob, 640x480
synthetic Replica-shaped RGB-D sequence.  One *step* = one mapping iteration of
the reference loop body (slam/algorithms/base_algorithm.py:255-273): assemble a
ray batch (2048 keyframe-bank rays + 2048 current-frame rays), fused
forward + loss + backward on the GPU (incl. the smoothness term), optimizer step.

  value   rays/s with the ray batches already resident in HBM (device timed,
          CUDA events per step, L2 flushed between steps, max over ranks).
  e2e     rays/s through the plugin call a user makes
          (CoSLAM.get_loss -> backward -> Optimizers.optimizer_step_all) with the
          keyframe ray bank in pinned HOST memory: per-step H2D copy of the
          sampled batch and D2H read of the loss are inside the timed region.
  N > 1   mapping rays are sharded: every rank owns a fixed 4096-ray batch
          (weak scaling), one NCCL all-reduce over the flat gradient bucket
          (hash table + MLP) per iteration, Adam replicated.

--impl reference times the CPU oracle port (torch, all host threads) of the same
step on rank 0 -- the reference's own code cannot travel to the GPU box (python
3.12 import failure + tinycudann/faiss absent, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_RAY = 88064  # SURVEY 8d: 43 samples x (1024 B gather + 1024 B scatter)
SMOOTH_BYTES = 29791 * 2048  # smoothness lattice, per mapping iteration
MAP_KF, MAP_CUR = 2048, 2048
N_KEYFRAMES = 5
METRIC = ('rays/s (co-slam mapping iteration: sample+march+hash gather+decode+'
          'composite+loss+backward+Adam, 640x480 synthetic RGB-D)')
WORKLOAD = ('co-slam hash-grid(16 lvl x 2 feat, 2^16) + OneBlob16, 640x480 synthetic room, '
            f'mapping iteration, {MAP_KF} keyframe-bank + {MAP_CUR} current-frame rays per GPU, '
            f'43 samples/ray, smoothness 31^3, {N_KEYFRAMES} keyframes')


# --steps / --warmup when not given: the CPU ports of --impl reference take seconds per step
DEFAULT_STEPS = {'ours': (200, 10), 'reference': (10, 2), 'reference_workload': (5, 0)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None,
                    help='timed steps (default 200; --impl reference: 10 for coslam, 5 otherwise)')
    ap.add_argument('--warmup', type=int, default=None,
                    help='untimed steps before them (default 10; --impl reference: 2 for coslam, '
                         '0 otherwise)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='coslam', choices=['coslam', 'nice', 'vox', 'point'])
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='N > 1: weak = fixed rays per GPU, strong = the single-GPU batch split over N')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-torch-gpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed as DIR/<name>.npy (float32); '
                         'default workload only (--impl ours --config coslam)')
    args = ap.parse_args()
    kind = args.impl if args.impl == 'ours' or args.config == 'coslam' else 'reference_workload'
    steps, warmup = DEFAULT_STEPS[kind]
    args.steps = steps if args.steps is None else args.steps
    args.warmup = warmup if args.warmup is None else args.warmup
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and (args.impl != 'ours' or args.config != 'coslam'):
        ap.error('--dump-outputs is implemented for the default workload '
                 '(--impl ours --config coslam)')
    return args


DUMP_LIMIT = 64 * 1024 * 1024


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy in float32 (float64 kept), at most DUMP_LIMIT
    bytes in all, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
        a = a if a.dtype == np.float64 else a.astype(np.float32)
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise RuntimeError(f'--dump-outputs: more than {DUMP_LIMIT} bytes at {name}')
        np.save(os.path.join(path, name + '.npy'), a)


def coslam_outputs(model, frames, sess, last):
    """What one mapping iteration hands its caller: the loss and its terms, the per-ray
    renders, and the parameters and poses after the optimiser step with the gradients they
    were stepped with."""
    out = {'loss': last['loss']}
    if sess is not None:
        renders = sess.out
        out['loss_terms'] = torch.cat([sess.losses, sess.smooth_loss])
        out['pose_rot'], out['pose_trans'] = sess.rot, sess.trans
    else:
        renders = last['out']
        out['loss_terms'] = torch.stack([v.detach() for v in last['loss_dict'].values()])
        out['pose_rot'] = torch.stack([f.pose.data_r.detach() for f in frames])
        out['pose_trans'] = torch.stack([f.pose.data_t.detach() for f in frames])
    for k, v in renders.items():
        if torch.is_tensor(v) and v.is_floating_point():
            out['render_' + k] = v
    named = [('table', model.embed_fn.params)] + [
        ('decoder_' + n.replace('.', '_'), p) for n, p in model.decoder.named_parameters()]
    for n, p in named:
        out[n] = p
        out['grad_' + n] = p.grad
    return out


# ------------------------------------------------------------------ clocks ---
class ClockSampler:
    """SM clock + throttle reasons sampled in-process through NVML every 5 ms
    while the timed region runs (the nvidia-smi recipe's fields)."""
    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.ok = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(',')[self.index])
                except ValueError:
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # noqa
            self.err = repr(e)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        bits = {
            'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown,
            'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
            'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown,
            'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap,
        }
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, b in bits.items():
                    if r & b:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        if not self.ok:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable']}
        self.stop_flag = True
        self.t.join(timeout=1)
        return {'sm_mhz': float(np.median(self.samples)) if self.samples else None,
                'sm_max_mhz': self.sm_max, 'reasons': sorted(self.reasons),
                'samples': len(self.samples)}


# ------------------------------------------------------------------ set-up ---
def build_algorithm(device, seed):
    from xrdslam_b200.coslam import CoSLAMConfig
    from xrdslam_b200.frame import Frame
    from xrdslam_b200.synthetic import make_sequence
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    cam, poses, frames = make_sequence(N_KEYFRAMES + 1)
    cfg = CoSLAMConfig()
    cfg.model.precision = 1  # 3xTF32 forward (fp32-level outputs/losses), TF32 backward
    algo = cfg.setup(camera=cam, device=device)
    kfs = []
    for k in range(N_KEYFRAMES):
        f = Frame(k, frames[k][0], frames[k][1], init_pose=poses[k],
                  separate_LR=True, rot_rep='axis_angle')
        algo.add_keyframe(f)
        kfs.append(f)
    cur = Frame(N_KEYFRAMES, frames[-1][0], frames[-1][1], init_pose=poses[-1],
                separate_LR=True, rot_rep='axis_angle')
    algo.set_initialized()
    return algo, kfs, cur


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one 4096-ray k_fused launch from the
    committed `ncu --set full` capture of this round (profiles/r02_coslam_kfused_traffic.json,
    written by scripts/ncu_summary.py); None when no capture of the current kernel exists."""
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'r02_coslam_kfused_traffic.json')))
        return int(d['dram_bytes_read'] + d['dram_bytes_write'])
    except Exception:
        return None


def flat_params(model):
    return [model.embed_fn.params] + list(model.decoder.parameters())


def allreduce_grads(dp):
    """ONE NCCL all-reduce over the flat gradient bucket (hash table + decoder).  The loss
    normalisers inside the kernels are already batch-global (model.dp), so the sum of the
    per-rank gradients IS the gradient of the all-rank batch: no division."""
    dp.all_reduce_grads()


def dp_preflight(model, dp, dev, R=1024):
    """Sharded == single-GPU check on the live process group (what tests/test_dp_gpu.py
    asserts on a 2-GPU box): every rank renders the SAME seeded batch once whole and once as
    its shard + all-reduce; the summed gradients must match the whole-batch gradients."""
    g = torch.Generator().manual_seed(77)
    rays_o = (torch.rand(R, 3, generator=g) - 0.5)
    rays_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    td = torch.rand(R, 1, generator=g) * 3 + 0.3
    ts = torch.rand(R, 3, generator=g)
    noise = torch.rand(R, 43, generator=g)
    full = dict(rays_o=rays_o.to(dev), rays_d=rays_d.to(dev), target_s=ts.to(dev),
                target_d=td.to(dev), first=True, noise=noise.to(dev))
    params = dp.params
    saved = [p.detach().clone() for p in params]
    gp = torch.Generator().manual_seed(5)
    with torch.no_grad():  # a non-trivial table, identical on every rank
        params[0].copy_(((torch.rand(params[0].shape, generator=gp) * 2 - 1) * 0.1).to(dev))
    model.dp = None
    for p in params:
        p.grad = None
    ld = model.get_loss_dict(model(full), full, True, 0)
    sum(ld.values()).backward()
    ref = [p.grad.detach().clone() for p in params]
    for p in params:
        p.grad = None
    model.dp = dp
    sl = dp.shard(R)
    part = {k: (v[sl] if torch.is_tensor(v) else v) for k, v in full.items()}
    ld = model.get_loss_dict(model(part), part, True, 0)
    sum(ld.values()).backward()
    dp.all_reduce_grads()
    rel = max(float((p.grad - r).norm() / (r.norm() + 1e-30)) for p, r in zip(params, ref))
    t = torch.tensor([rel], device=dev, dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    with torch.no_grad():
        for p, s_ in zip(params, saved):
            p.copy_(s_)
            p.grad = None
    rel = float(t.item())
    return {'ok': bool(rel < 1e-4), 'grad_rel_l2_max_over_ranks': rel, 'rays': R,
            'world': dp.world}


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    _cabi.check('xrd_check_device', lib.xrd_check_device(local))

    algo, kfs, cur = build_algorithm(dev, seed=1234 + rank)
    model = algo.model
    frames = kfs + [cur]
    K, W = args.steps, args.warmup
    # weak scaling: every rank renders the full single-GPU batch; strong: that batch is split
    strong = args.scaling == 'strong' and world > 1
    map_kf = MAP_KF // world if strong else MAP_KF
    map_cur = MAP_CUR // world if strong else MAP_CUR
    algo.config.mapping_sample = map_kf
    R = map_kf + map_cur
    params = flat_params(model)
    from xrdslam_b200.dp import MappingDataParallel
    dp = MappingDataParallel(params)
    dp.broadcast_params(0)  # identical replicas
    dp_parity = dp_preflight(model, dp, dev) if world > 1 else None
    model.dp = dp
    optim = algo.setup_optimizers(K, frames, is_mapping=True)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def make_batch():
        """What CoSLAM.get_model_input builds, with the current-frame share raised
        to 2048 rays (the reference's first-keyframe shape) so R is fixed."""
        algo.config.min_sample_pixels = map_cur
        inp = algo.get_model_input(frames, True)
        inp['smooth_rand'] = torch.rand(6)
        return inp

    last = {}

    def device_step(inp):
        optim.zero_grad_all()
        out = model(inp)
        loss_dict = model.get_loss_dict(out, inp, True, 0)
        loss = sum(loss_dict.values())
        loss.backward()
        allreduce_grads(dp)
        optim.optimizer_step_all(step=0)
        last.update(out=out, loss_dict=loss_dict)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: batches resident in HBM -----------------------
    # the mapping iteration is a CUDA graph (xrdslam_b200/coslam_graph.py) replayed from a
    # device-resident batch; N > 1: the two NCCL all-reduces (loss-normaliser counts, then ONE
    # flat bucket of all gradients + loss terms) are nodes of the same graph.
    use_graph = algo._graph_ok(frames)
    sess = None
    batches = []
    if use_graph:
        algo.config.min_sample_pixels = map_cur
        algo.bundle_adjust = True
        sess = algo.mapping_session(frames)
        sess.begin(frames)
        batches = [sess.make_resident_batch(frames) for _ in range(K + W)]
        run_step = lambda i: sess.step_resident(i, batches[i])
    else:
        for _ in range(K + W):
            b = make_batch()
            b = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in b.items()}
            b['rays_o'].requires_grad_(True)  # bundle adjustment: pose gradients are
            b['rays_d'].requires_grad_(True)  # part of the step (d loss / d rays)
            batches.append(b)
        run_step = lambda i: device_step(batches[i])
    for i in range(W):
        run_step(i)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(K)]
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        flush.zero_()  # L2 flush (256 MB > 126 MB L2), outside the timed events
        ev[i][0].record()
        last['loss'] = run_step(W + i)
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, coslam_outputs(model, frames, sess, last))
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    clk = clocks.stop() if rank == 0 else None
    value = world * R * K / (ms_total * 1e-3)
    if use_graph:  # the roofline leg below goes through Model.forward: needs autograd batches
        gen = []
        for _ in range(K + W):
            b = make_batch()
            b = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in b.items()}
            b['rays_o'].requires_grad_(True)
            b['rays_d'].requires_grad_(True)
            gen.append(b)
        batches = gen

    # ---------------- roofline: the fused kernel alone ---------------------
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(K)]
    for i in range(K):
        flush.zero_()
        optim.zero_grad_all()
        kev[i][0].record()  # materialise the lazily-created handles
        kev[i][1].record()  # (both are re-recorded by the library around k_fused)
        lib.xrd_debug_kernel_events(kev[i][0].cuda_event, kev[i][1].cuda_event)
        out = model(batches[W + i])
        lib.xrd_debug_kernel_events(None, None)
    torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    achieved = R * BYTES_PER_RAY / (k_ms * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'kernel': 'xrd::coslam::k_fused_g<true> (grouped persistent fused kernel)',
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak,
                'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback 6650',
                # dram__bytes_read.sum + dram__bytes_write.sum of one 4096-ray launch
                # (ncu --set full, profiles/r02_coslam_fused_g_4096rays_ncu.txt)
                'traffic': ncu_traffic(), 'kernel_ms': k_ms,
                'algorithmic_bytes_per_launch': R * BYTES_PER_RAY,
                'note': 'table (6.56 MB) is L2-resident: DRAM traffic is far below '
                        'the algorithmic bytes, see profiles/'}

    # ---------------- e2e: through the plugin, host ray bank ---------------
    algo.config.min_sample_pixels = map_cur
    h2d = R * 7 * 4 + R * 8 + 128  # sampled rows + pose ids + per-iteration scalar block
    d2h = 4
    if use_graph:
        # the session is asynchronous (pinned staging ring of depth 4, like CoSLAM's own mapping
        # loop which never reads the loss): every step's loss is copied D2H into a pinned ring
        # and read on the host two steps later, so host sampling + H2D of step i+1 overlap the
        # graph of step i.  The final barrier()/synchronize closes the timed region.
        loss_ring = [torch.zeros(1).pin_memory() for _ in range(4)]
        loss_ev = [torch.cuda.Event() for _ in range(4)]
        host_losses = []

        def e2e_step(i):
            lt = sess.step(i, frames)   # H2D rows/ids/scalars + the captured iteration
            k = i % 4
            loss_ring[k].copy_(lt.detach().reshape(1), non_blocking=True)  # D2H loss, every step
            loss_ev[k].record()
            j = i - 2
            if j >= 0:
                loss_ev[j % 4].synchronize()
                host_losses.append(float(loss_ring[j % 4][0]))
            return lt
    else:
        h2d = R * 7 * 4 + R * 8 + len(frames) * 16 * 4

        def e2e_step(i):
            optim.zero_grad_all()
            loss = algo.get_loss(frames, True, i, K)
            loss.backward()
            allreduce_grads(dp)
            optim.optimizer_step_all(step=i)
            return loss.item()  # D2H read of the step's result
    for i in range(W):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        lv = e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    if use_graph:
        sess.end(frames)
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * R * K / float(t.item())

    # ---------------- tracking iterations (reported beside) ----------------
    trk = None
    if rank == 0:
        # CoSLAM.optimize_update(..., is_mapping=False): one captured iteration per step,
        # image upload at begin(), best-pose read-back at end() -- per tracked frame
        n_it, n_frames = algo.config.tracking_n_iters, 20
        for i in range(3):
            algo.optimize_update(n_it, [cur], False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n_frames):
            cand = algo.optimize_update(n_it, [cur], False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        trk = {'tracking_iters_per_s': n_frames * n_it / dt,
               'tracking_frames_per_s': n_frames / dt, 'tracking_iters_per_frame': n_it,
               'tracking_rays': algo.config.tracking_sample,
               'tracking_rays_per_s': n_frames * n_it * algo.config.tracking_sample / dt}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_baseline(iters=2)
    tgb = None
    if rank == 0 and not args.no_torch_gpu_baseline:
        tgb = torch_gpu_baseline(dev)

    if rank == 0:
        line = {
            'metric': METRIC,
            'value': value, 'unit': 'rays/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_total / K, 'higher_is_better': True,
            'scaling': 'strong' if strong else 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'precision': 'fp32 gathers/compositing/loss; decoder GEMMs 3xTF32 forward, TF32 backward (fp32 accumulate)',
                       'workload': WORKLOAD,
                       'rays_per_step_per_gpu': R, 'parallelism': f'dp{world}',
                       'l2': 'flushed between timed steps (256 MB write); ray batches differ every step'},
            'e2e': {'value': e2e_value, 'unit': 'rays/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h,
                    'loss_readback': 'async D2H into a pinned ring every step, consumed by the host 2 steps later',
                    'path': ('CoSLAM.mapping_session(frames).step(): host pinned ray bank, '
                             'random.sample, H2D, one CUDA graph (poses, rays, sample, fused '
                             'fwd/loss/bwd, smoothness, pose grads, Adam)' +
                             ((' with the 2 NCCL all-reduces captured inside it' if getattr(sess, 'single_graph', True)
                               else ' in 3 captured segments around 2 NCCL all-reduces') if world > 1 else '') +
                             ', async D2H of the loss')
                    if use_graph else
                    ('CoSLAM.get_loss (host pinned ray bank, random.sample, H2D) -> '
                     'loss.backward -> all-reduce -> Optimizers.optimizer_step_all -> loss.item()')},
            'gpu_launches': K * ((11 if world == 1 else 12) if use_graph else 9) + (K // 5 if use_graph else 0),
            'gpu_launches_note': ('per step (one graph): pose::k_fwd, rays::k_fwd, k_sample, '
                                  'k_fused_g<true>, k_finalize, k_smooth_fwd, k_smooth_bwd, '
                                  'k_smooth_finalize, rays::k_bwd, pose::k_bwd, k_adam (+ k_adam on '
                                  'the poses every 5th step)') if use_graph else
                                 ('per step: rays::k_fwd, k_sample, k_fused_g<true>, k_finalize, '
                                  'k_smooth_fwd/bwd/finalize, rays::k_bwd, k_adam x2 (torch glue '
                                  'not counted)'),
            'clocks': clk, 'roofline': roofline, 'cpu_baseline': cpu,
            'torch_gpu_baseline': tgb, 'dp_parity': dp_parity,
            'iters': {'mapping_iters_per_s': K / (ms_total * 1e-3),
                      **(trk or {})},
            'wall_s_value_leg': wall,
        }
        print(json.dumps(line))
    _finish(world)


def _finish(world):
    """Multi-rank exit: captured graphs hold NCCL nodes and rank 0 runs single-GPU legs after
    the other ranks are done, so tearing the communicator down collectively can stall; the
    JSON line is out -- flush and leave (the OS reclaims the NCCL resources)."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


# ------------------------------------------------------------ CPU baseline ---
def coslam_ref_step_factory(R_bank, R_cur, device='cpu'):
    """One Co-SLAM mapping iteration of the oracle port (fwd + bwd + Adam) on `device`, on the
    SAME workload as the B200 arm: the keyframe ray bank and the per-iteration sampler are
    CoSLAM.get_model_input's own host path (random.sample rows of the bank + current-frame
    pixels, per-ray pose gather), R_bank + R_cur rays, smoothness term, Adam on table +
    decoder."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from oracle.coslam import CoslamOracle
    from helpers import BOUND
    dev = torch.device(device)
    algo, kfs, cur = build_algorithm(torch.device('cpu'), seed=1234)  # host sampler only
    frames = kfs + [cur]
    algo.config.mapping_sample = R_bank
    algo.config.min_sample_pixels = R_cur
    torch.manual_seed(0)
    ora = CoslamOracle(BOUND)
    if dev.type == 'cuda':
        ora.to(dev)
        ora.bounding_box = ora.bounding_box.to(dev) if hasattr(ora, 'bounding_box') else None
    opt = torch.optim.Adam([
        {'params': [ora.embed_fn.params], 'lr': 1e-2, 'eps': 1e-15, 'betas': (0.9, 0.99)},
        {'params': [ora.sdf0.weight, ora.sdf1.weight, ora.col0.weight, ora.col1.weight],
         'lr': 1e-2, 'weight_decay': 1e-6, 'betas': (0.9, 0.99)}])

    def step():
        with torch.no_grad():
            inp = algo.get_model_input(frames, True)  # host: rows, ids, poses -> rays
        t = lambda k: inp[k].detach().to(dev)
        R = inp['rays_o'].shape[0]
        opt.zero_grad(set_to_none=True)
        noise = torch.rand(R, 43).to(dev)
        _, _, tot = ora.step(t('rays_o'), t('rays_d'), t('target_s'), t('target_d'), noise, True,
                             False, smooth_rand=torch.rand(2, 3).to(dev))
        tot.backward()
        opt.step()
        return float(tot.detach())
    return step


def pick_threads(step):
    """The oracle ports are many small torch ops: past a few dozen threads the intra-op pool
    only adds contention.  Calibrate once on one step each."""
    cores = os.cpu_count() or 1
    best, best_t = cores, None
    t_all = time.perf_counter()
    for n in sorted({min(cores, c) for c in (8, 16, 32, cores)}, reverse=True):
        torch.set_num_threads(n)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
        if time.perf_counter() - t_all > 20.0:  # slow ports (Point-SLAM: ~15 s per step): bound
            break                               # the calibration, keep the best count seen so far
    torch.set_num_threads(best)
    return best


def cpu_baseline(iters=2):
    """Bounded sample of the SAME workload: `iters` full 4096-ray iterations (~10-30 s)."""
    step = coslam_ref_step_factory(MAP_KF, MAP_CUR)
    cores = pick_threads(step)
    t0 = time.perf_counter()
    for _ in range(iters):
        step()
    dt = time.perf_counter() - t0
    R = MAP_KF + MAP_CUR
    return {'value': R * iters / dt, 'unit': 'rays/s', 'cores': cores,
            'kind': 'port',
            'sample': f'{iters} mapping iterations x {R} rays x 43 samples, same sampler and '
                      'batch as the B200 arm (oracle/coslam.py torch-CPU port incl. smoothness '
                      '+ Adam)',
            'ms_per_iter': dt / iters * 1e3}


def torch_gpu_baseline(dev, iters=10):
    """The restated reference PyTorch path (oracle/coslam.py: restated-tcnn hash grid + OneBlob
    in torch ops, autograd, torch Adam) run on the B200 itself -- BASELINE.md section 5's
    'reference PyTorch path on the GPU', what north_star's >= 10x is quoted against."""
    try:
        step = coslam_ref_step_factory(MAP_KF, MAP_CUR, device=str(dev))
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        R = MAP_KF + MAP_CUR
        return {'value': R * iters / dt, 'unit': 'rays/s', 'ms_per_iter': dt / iters * 1e3,
                'kind': 'restated reference PyTorch path (oracle/coslam.py) on cuda, eager '
                        'autograd + torch.optim.Adam, host ray bank -> H2D per iteration',
                'iters': iters}
    except Exception as e:  # noqa
        return {'unavailable': repr(e)[:300]}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.config != 'coslam':
        return run_reference_workload(args)
    R = MAP_KF + MAP_CUR
    step = coslam_ref_step_factory(MAP_KF, MAP_CUR)
    cores = pick_threads(step)
    K, W = args.steps, args.warmup
    for _ in range(W):
        step()
    t0 = time.perf_counter()
    for _ in range(K):
        step()
    dt = time.perf_counter() - t0
    v = R * K / dt
    line = {
        'impl': 'reference',
        'metric': METRIC,
        'value': v, 'unit': 'rays/s', 'n_gpus': int(os.environ.get('WORLD_SIZE', '1')),
        'steps': K, 'warmup': W, 'ms_per_step': dt / K * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        # same workload, same batch, same sampler as the B200 arm; fewer steps
        'config': {'workload': WORKLOAD, 'rays_per_step_per_gpu': R,
                   'precision': 'fp32 (torch CPU)',
                   'sample': f'{K} full steps of {R} rays (same frames, ray bank, sampler, decoder, '
                             'losses, smoothness, Adam); the reference\'s own python cannot run on '
                             'the box (py3.12 + tinycudann absent): CPU oracle port, all host threads'},
        'cpu_baseline': {'value': v, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{K} steps x {R} rays'},
        'e2e': {'value': v, 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ------------------------------------------------- nice / vox / point (cfg 3-5) ---
def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


def run_workload(args):
    import torch.distributed as dist
    from bench_workloads import WORKLOADS
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    from xrdslam_b200 import _cabi
    lib = _cabi.lib()
    _cabi.check('xrd_check_device', lib.xrd_check_device(local))
    random.seed(1234 + rank)
    np.random.seed(1234 + rank)
    torch.manual_seed(1234 + rank)
    wl = WORKLOADS[args.config](dev, rank, world)
    wl.build()
    K, W = args.steps, args.warmup
    R = wl.rays_per_step()
    n_sched = wl.n_iters_schedule
    wl.begin(n_sched)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the timed steps walk through the stage schedule exactly like one mapping call does
    sched = [int(j * n_sched / K) for j in range(K)]
    for i in range(W):
        wl.step(sched[i % K])
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(K)]
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        flush.zero_()  # L2 flush between timed steps (outside the events)
        ev[i][0].record()
        wl.step(sched[i])
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - t0
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    clk = clocks.stop() if rank == 0 else None
    value = world * R * K / (ms_total * 1e-3)

    # ---- dominant kernel, timed by the library with events around its launches
    peaks = _peaks()
    kms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps_r = wl.roofline_steps() if hasattr(wl, 'roofline_steps') else list(range(8))
    for i in steps_r:
        flush.zero_()
        e0.record(); e1.record()
        lib.xrd_debug_kernel_events(e0.cuda_event, e1.cuda_event)
        wl.step(i)
        lib.xrd_debug_kernel_events(None, None)
        torch.cuda.synchronize()
        kms.append(e0.elapsed_time(e1))
    k_ms = float(np.median(kms))
    if args.config == 'vox':
        n_pts = int(wl.algo.model.last_march.get('n_points', 0)) or None
        roofline = wl.kernel_roofline(k_ms, float(peaks.get('bf16_tflops_sustained', 1400.0)),
                                      n_pts or 1)
    else:
        roofline = wl.kernel_roofline(k_ms, float(peaks.get('hbm_gbs', 6650.0)))
    roofline['peak_source'] = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback'

    # ---- e2e through the plugin call
    Ke = max(10, min(K, n_sched))
    wl.e2e(Ke)  # warm-up call (optimizer set-up paths, allocator)
    barrier()
    dt, h2d, d2h, _ = wl.e2e(Ke)
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * R * Ke / float(t.item())

    n_launch = count_launches(wl, min(K, 5))  # every rank: the step holds collectives
    barrier()
    trk = wl.tracking() if rank == 0 else None
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_baseline_workload(wl)
    if rank == 0:
        line = {
            'metric': wl.metric, 'value': value, 'unit': 'rays/s', 'n_gpus': world, 'steps': K,
            'warmup': W, 'ms_per_step': ms_total / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': wl.dtype, 'data': 'synthetic',
            'config': {'workload': wl.workload, 'rays_per_step_per_gpu': R,
                       'parallelism': f'dp{world}', 'precision': wl.precision,
                       'l2': 'flushed between timed steps (256 MB write)', 'map': wl.map_info},
            'e2e': {'value': e2e_value, 'unit': 'rays/s', 'h2d_bytes_per_step': h2d / Ke,
                    'd2h_bytes_per_step': d2h / Ke + 8,
                    'path': f'{type(wl.algo).__name__}.optimize_update({Ke}, window, is_mapping=True): '
                            'current frame as host arrays (upload inside), per-iteration device '
                            'sampling + fused step + autograd hand-off + Adam, one host read per '
                            'iteration (ray filter count), final D2H read'},
            'gpu_launches': None, 'clocks': clk, 'roofline': roofline, 'cpu_baseline': cpu,
            'iters': {'mapping_iters_per_s': K / (ms_total * 1e-3), **(trk or {})},
            'wall_s_value_leg': wall,
        }
        line['gpu_launches'] = n_launch
        print(json.dumps(line))
    _finish(world)


def count_launches(wl, n):
    """Launches of OUR kernels (names in namespace xrd::) inside n steps, counted with the
    torch profiler (CUPTI) outside every timed region."""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n):
                wl.step(i)
            torch.cuda.synchronize()
        tot = sum(e.count for e in prof.key_averages() if 'xrd::' in e.key)
        return int(round(tot / n)) if tot else None
    except Exception:
        return None


def cpu_baseline_workload(wl, budget_s=20.0):
    step, R, what = wl.cpu_step_factory()
    cores = pick_threads(step)
    t0 = time.perf_counter()
    n = 0
    while n < 1 or (time.perf_counter() - t0 < budget_s and n < 20):
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {'value': R * n / dt, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
            'sample': f'{n} mapping iterations x {R} rays, same frames / window / batch as the '
                      f'B200 arm: {what}', 'ms_per_iter': dt / n * 1e3}


def run_reference_workload(args):
    from bench_workloads import WORKLOADS
    dev = torch.device('cuda', 0) if torch.cuda.is_available() else torch.device('cpu')
    wl = WORKLOADS[args.config](dev, 0, 1)
    if args.config in ('vox', 'point'):
        wl.build()  # the map (octree / point cloud) is built by the product's own maintenance code
    step, R, what = wl.cpu_step_factory()
    cores = pick_threads(step)
    K, W = args.steps, args.warmup
    for _ in range(W):
        step()
    t0 = time.perf_counter()
    for _ in range(K):
        step()
    dt = time.perf_counter() - t0
    v = R * K / dt
    print(json.dumps({
        'impl': 'reference', 'metric': wl.metric, 'value': v, 'unit': 'rays/s',
        'n_gpus': int(os.environ.get('WORLD_SIZE', '1')), 'steps': K, 'warmup': W,
        'ms_per_step': dt / K * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl.workload, 'rays_per_step_per_gpu': R,
                   'sample': f'{K} full steps: {what}'},
        'cpu_baseline': {'value': v, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{K} steps x {R} rays'},
        'e2e': {'value': v, 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    elif a.config == 'coslam':
        run_ours(a)
    else:
        run_workload(a)
