"""Vox-Fusion GPU parity: (1) the raw intersection / sampling kernels bit-for-bit against the
reference's OWN `grid` CUDA extension, (2) the full march + render step against
oracle/voxfusion.py.  The reference extension's outputs on these seeded scenes are stored as
SHA-256 digests in tests/golden/vox_grid_ref.json (tests/golden/make_golden.py vox_grid runs
the extension, compiled from the reference sources by oracle/build_ref.py, on a B200)."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import digest, load_golden_json, max_abs, rel_err

pytestmark = pytest.mark.gpu
OFFSET = 25.6  # voxels_each_dim / 2 * voxel_size: keeps coordinates inside [0, 256) voxels


def golden():
    return load_golden_json('vox_grid_ref.json')


class OwnGrid:
    """This package's raw intersection / sampling kernels behind the call signatures of the
    reference's `grid` extension (svo_intersect, inverse_cdf_sampling)."""

    def __init__(self, dev):
        from xrdslam_b200 import _cabi
        self.dev, self.cabi, self.lib = dev, _cabi, _cabi.lib()

    def svo_intersect(self, ro, rd, cen, ch, vs, n_max):
        ro, rd = ro[0].float().contiguous(), rd[0].float().contiguous()
        cen, ch = cen[0].float().contiguous(), ch[0].int().contiguous()
        R = ro.shape[0]
        idx = torch.empty(R, n_max, dtype=torch.int32, device=self.dev)
        lo = torch.empty(R, n_max, device=self.dev)
        hi = torch.empty(R, n_max, device=self.dev)
        rays = self.cabi.XrdRays(R, ro.data_ptr(), rd.data_ptr(), None, None)
        mp = self.cabi.XrdVoxMap(cen.shape[0], cen.data_ptr(), ch.data_ptr(), None, None, 0)
        self.cabi.check('xrd_voxfusion_intersect_raw', self.lib.xrd_voxfusion_intersect_raw(
            C.byref(rays), C.byref(mp), vs, n_max, idx.data_ptr(), lo.data_ptr(), hi.data_ptr(),
            None))
        return idx[None], lo[None], hi[None]

    def inverse_cdf_sampling(self, pi, mn, mx, noise, pr, stp, fixed):
        G, K, P = pi.shape
        ms = noise.shape[-1]
        s_idx = torch.empty(G * K, ms, dtype=torch.int32, device=self.dev)
        s_depth = torch.empty(G * K, ms, device=self.dev)
        s_dist = torch.empty(G * K, ms, device=self.dev)
        c = lambda t: t.contiguous().data_ptr()
        self.cabi.check('xrd_voxfusion_sample_raw', self.lib.xrd_voxfusion_sample_raw(
            G * K, P, ms, K, c(pi), c(mn), c(mx), c(noise), c(pr), c(stp), s_idx.data_ptr(),
            s_depth.data_ptr(), s_dist.data_ptr(), None))
        return s_idx.reshape(G, K, ms), s_depth.reshape(G, K, ms), s_dist.reshape(G, K, ms)


class Recorder:
    """Wraps a `grid` implementation and keeps the digests of every output it returns, in call
    order (intersection t values only where a voxel was hit)."""

    def __init__(self, grid):
        self.grid, self.digests = grid, []

    def svo_intersect(self, *a):
        idx, lo, hi = self.grid.svo_intersect(*a)
        m = idx >= 0
        self.digests += [digest(idx), digest(lo[m]), digest(hi[m])]
        return idx, lo, hi

    def inverse_cdf_sampling(self, *a):
        out = self.grid.inverse_cdf_sampling(*a)
        self.digests += [digest(t) for t in out]
        return out


def scene(device, n_frames=2, R=700, seed=0):
    """Model with a map built from synthetic depth frames + a ray batch from the last pose."""
    from xrdslam_b200.sparse_voxel import SparseVoxelConfig
    from xrdslam_b200.synthetic import make_sequence
    cam, poses, frames = make_sequence(n_frames, width=160, height=120, offset=(OFFSET,) * 3)
    torch.manual_seed(seed)
    model = SparseVoxelConfig().setup(camera=cam).to(device)
    H, W = cam.height, cam.width
    j, i = torch.meshgrid(torch.arange(H, dtype=torch.float32),
                          torch.arange(W, dtype=torch.float32), indexing='ij')
    dirs = torch.stack([(i - cam.cx) / cam.fx, -(j - cam.cy) / cam.fy, -torch.ones_like(i)], -1)
    for (rgb, depth), c2w in zip(frames, poses):
        c2w = torch.from_numpy(c2w)
        d = torch.from_numpy(depth)
        pts = (dirs * d[..., None])[d > 0].reshape(-1, 3)
        pts = pts @ c2w[:3, :3].T + c2w[:3, 3]
        model.insert_points(pts)
    g = torch.Generator().manual_seed(seed)
    pix = torch.randint(0, H * W, (R,), generator=g)
    c2w = torch.from_numpy(poses[-1])
    rays_d = (dirs.reshape(-1, 3)[pix] @ c2w[:3, :3].T).contiguous()
    rays_o = c2w[:3, 3].expand(R, 3).contiguous()
    # a few rays that miss everything
    rays_d[:5] = torch.tensor([0.0, 0.0, 1.0])
    rays_o[:5] = torch.tensor([1.0, 1.0, 1.0])
    td = torch.from_numpy(frames[-1][1]).reshape(-1, 1)[pix].contiguous()
    ts = torch.from_numpy(frames[-1][0]).reshape(-1, 3)[pix].contiguous()
    return model, rays_o, rays_d, ts, td


def intersect_case(grid, dev):
    """The reference call exactly as voxel_helpers_voxfusion.py:237-255 would issue it with
    G = 1, on the map and rays of scene(dev)."""
    model, rays_o, rays_d, _, _ = scene(dev)
    ms = model.map_states
    ro, rd = rays_o.to(dev), rays_d.to(dev)
    return grid.svo_intersect(ro[None].contiguous(), rd[None].contiguous(),
                              ms['voxel_center_xyz'][None].contiguous(),
                              ms['voxel_structure'][None].contiguous(), 0.2, 50)


def sampling_case(grid, dev):
    """Intersections through `grid`, then the inputs of ray_sample + InverseCDFRaySampling.forward
    (voxel_helpers_voxfusion.py:399-481,690-714) for scene(dev, R=900)."""
    from oracle.voxfusion import ray_intersect
    model, rays_o, rays_d, _, _ = scene(dev, R=900)
    ms = model.map_states

    def gpu_intersect(ro, rd, cen, ch, vs, n_max):
        i, a, b = grid.svo_intersect(ro[None].to(dev).contiguous(), rd[None].to(dev).contiguous(),
                                     cen[None].contiguous(), ch[None].contiguous(), vs, n_max)
        return i[0].cpu(), a[0].cpu(), b[0].cpu()
    inter, hits = ray_intersect(rays_o, rays_d, ms['voxel_center_xyz'], ms['voxel_structure'],
                                0.2, intersect_fn=gpu_intersect)
    inter = {k: v[hits].to(dev) for k, v in inter.items()}
    dists = (inter['max_depth'] - inter['min_depth']).masked_fill(
        inter['intersected_voxel_idx'].eq(-1), 0)
    probs = dists / dists.sum(dim=-1, keepdim=True)
    steps = dists.sum(-1) / 0.01
    pts_idx = inter['intersected_voxel_idx']
    G, N, P = 200, pts_idx.size(0), pts_idx.size(1)
    Hh = int(np.ceil(N / G)) * G
    pad = lambda t: torch.cat([t, t[:1].expand(Hh - N, *t.shape[1:])], 0) if Hh > N else t
    pi, mn, mx, pr, stp = map(pad, (pts_idx, inter['min_depth'], inter['max_depth'], probs, steps))
    K = Hh // G
    max_steps = int(steps.ceil().long().max()) + P
    gen = torch.Generator(device='cpu').manual_seed(3)
    noise = torch.rand(G, K, max_steps, generator=gen).clamp(min=0.001, max=0.999).to(dev)
    return (pi.reshape(G, K, P).contiguous(), mn.reshape(G, K, P).contiguous(),
            mx.reshape(G, K, P).contiguous(), noise.contiguous(), pr.reshape(G, K, P).contiguous(),
            stp.reshape(G, K).contiguous(), -1)


def test_intersect_kernel_bit_exact_vs_reference_grid(cuda_dev):
    """Node ids in visiting order and the t values of every hit equal the reference
    extension's, bit for bit."""
    rec = Recorder(OwnGrid(cuda_dev))
    idx, _, _ = intersect_case(rec, cuda_dev)
    assert (idx >= 0).sum() > idx.shape[1]  # plenty of hits
    assert rec.digests == golden()['intersect']


def test_sampling_kernel_bit_exact_vs_reference_grid(cuda_dev):
    """Voxel, mid-point depth and distance of every sample equal the reference extension's,
    bit for bit, on the same intersections (themselves checked against the reference's)."""
    rec = Recorder(OwnGrid(cuda_dev))
    args = sampling_case(rec, cuda_dev)
    g = golden()['sampling']
    assert rec.digests == g['intersect']
    rec.digests = []
    rec.inverse_cdf_sampling(*args)
    assert rec.digests == g['samples']


@pytest.mark.parametrize('need_pose', [True, False])
def test_full_step_vs_oracle(cuda_dev, need_pose):
    from oracle.voxfusion import VoxOracle
    model, rays_o, rays_d, ts, td = scene(cuda_dev, R=300, seed=2)
    dev = cuda_dev
    ora = VoxOracle()
    with torch.no_grad():
        g = torch.Generator().manual_seed(9)
        model.embeddings.copy_(torch.randn(model.embeddings.shape, generator=g) * 0.3)
        ora.embeddings.copy_(model.embeddings.cpu())
        ora.decoder.load_state_dict(model.decoder.state_dict())
    voxels, children, features = model.export_octree()
    ora.set_map(voxels, children, features)
    # noise by hit rank (the reference draws a [G, K, max_steps] tensor)
    gen = torch.Generator().manual_seed(5)
    noise_rank = torch.rand(rays_o.shape[0], model.config.max_samples_per_ray,
                            generator=gen).clamp(0.001, 0.999)

    def noise_fn(shape):
        G, K, ms = shape
        out = torch.full((G * K, ms), 0.5)
        n = min(G * K, noise_rank.shape[0])
        out[:n] = noise_rank[:n, :ms]
        return out.reshape(G, K, ms)
    ro_o = rays_o.clone().requires_grad_(True)
    rd_o = rays_d.clone().requires_grad_(True)
    marched = ora.march(ro_o.detach(), rd_o.detach(), noise_fn)
    out_o, ld_o = ora.render(ro_o, rd_o, ts, td, marched)
    sum(ld_o.values()).backward()
    hits = marched[1]
    rank = torch.cumsum(hits.long(), 0) - 1
    noise = torch.full((rays_o.shape[0], model.config.max_samples_per_ray), 0.5)
    noise[hits] = noise_rank[rank[hits]]
    ro = rays_o.to(dev).requires_grad_(need_pose)
    rd = rays_d.to(dev).requires_grad_(need_pose)
    inp = dict(rays_o=ro, rays_d=rd, target_s=ts.to(dev), target_d=td.to(dev), noise=noise.to(dev))
    out = model(inp)
    ld = model.get_loss_dict(out, inp, True, 0)
    sum(ld.values()).backward()
    torch.cuda.synchronize()
    m = model.last_march
    assert m['overflow'] == 0
    assert torch.equal(out['ray_mask'].cpu(), hits)
    # sample structure: voxel ids exact, depths to a few ulp (true division vs __fdividef)
    smp = marched[2]
    S = smp['sampled_point_voxel_idx'].shape[1]
    assert m['s_max'] == S and m['n_hit_rays'] == int(hits.sum())
    got_idx = m['smp_idx'].cpu()[hits][:, :S]
    assert (got_idx != smp['sampled_point_voxel_idx']).float().mean() < 2e-3
    same = got_idx == smp['sampled_point_voxel_idx']
    dd = (m['smp_depth'].cpu()[hits][:, :S] - smp['sampled_point_depth']).abs()
    assert float(dd[same].max()) < 1e-5
    assert max_abs(out['depth'], out_o['depth']) < 2e-4
    assert max_abs(out['rgb'], out_o['rgb']) < 2e-4
    for k in ld_o:
        a, b = float(ld[k].detach()), float(ld_o[k].detach())
        assert abs(a - b) <= 5e-4 * max(abs(b), 1e-6), (k, a, b)
    assert rel_err(model.embeddings.grad, ora.embeddings.grad) < 5e-3
    sd_o = dict(ora.decoder.named_parameters())
    for n, p in model.decoder.named_parameters():
        assert rel_err(p.grad, sd_o[n].grad) < 5e-3, n
    if need_pose:
        assert rel_err(ro.grad, ro_o.grad) < 5e-3
        assert rel_err(rd.grad, rd_o.grad) < 5e-3


def test_no_hit_returns_none(cuda_dev):
    model, rays_o, rays_d, ts, td = scene(cuda_dev, R=64)
    dev = cuda_dev
    ro = torch.ones(16, 3, device=dev)
    rd = torch.tensor([[0.0, 0.0, 1.0]], device=dev).expand(16, 3).contiguous()
    out = model(dict(rays_o=ro, rays_d=rd, target_s=ts[:16].to(dev), target_d=td[:16].to(dev)))
    assert out is None  # reference: render_rays prints "no hit" and returns None


def _march_through_grid(grid, ora, rays_o, rays_d, noise_fn, dev):
    """VoxOracle.march with BOTH native stages executed by `grid` (svo_intersect +
    inverse_cdf_sampling), glued exactly as voxel_helpers_voxfusion.py:237-255,399-481 glue
    them.  The CPU restatement divides exactly where the reference kernels use __fdividef;
    chained through bits equal to the reference extension's, the oracle sees the reference's
    own bits."""
    from oracle.voxfusion import MAX_DEPTH, ray_intersect

    def gpu_intersect(ro, rd, cen, ch, vs, n_max):
        i, a, b = grid.svo_intersect(ro[None].to(dev).contiguous(), rd[None].to(dev).contiguous(),
                                     cen[None].to(dev).contiguous(), ch[None].to(dev).contiguous(),
                                     vs, n_max)
        return i[0].cpu(), a[0].cpu(), b[0].cpu()
    inter, hits = ray_intersect(rays_o, rays_d, ora.centres, ora.children, ora.voxel_size,
                                intersect_fn=gpu_intersect)
    inter = {k: v[hits] for k, v in inter.items()}
    dists = (inter['max_depth'] - inter['min_depth']).masked_fill(
        inter['intersected_voxel_idx'].eq(-1), 0)
    probs = dists / dists.sum(dim=-1, keepdim=True)
    steps = dists.sum(-1) / ora.step_size
    pts_idx = inter['intersected_voxel_idx']
    G, N, P = 200, pts_idx.size(0), pts_idx.size(1)
    Hh = int(np.ceil(N / G)) * G
    pad = lambda t: torch.cat([t, t[:1].expand(Hh - N, *t.shape[1:])], 0) if Hh > N else t
    pi, mn, mx, pr, stp = map(pad, (pts_idx, inter['min_depth'], inter['max_depth'], probs, steps))
    K = Hh // G
    max_steps = int(steps.ceil().long().max()) + P
    noise = noise_fn((G, K, max_steps))
    d = lambda t: t.to(dev).contiguous()
    r_idx, r_depth, r_dist = grid.inverse_cdf_sampling(
        d(pi.reshape(G, K, P)), d(mn.reshape(G, K, P)), d(mx.reshape(G, K, P)), d(noise),
        d(pr.reshape(G, K, P)), d(stp.reshape(G, K)), -1)
    s_idx = r_idx.reshape(Hh, -1)[:N].cpu()
    s_depth = r_depth.reshape(Hh, -1)[:N].cpu()
    s_dist = r_dist.reshape(Hh, -1)[:N].cpu()
    max_len = int(s_idx.ne(-1).sum(-1).max())
    s_idx, s_depth, s_dist = s_idx[:, :max_len], s_depth[:, :max_len], s_dist[:, :max_len]
    s_dist = s_dist.clamp(min=0.0)
    s_depth = s_depth.masked_fill(s_idx.eq(-1), MAX_DEPTH)
    s_dist = s_dist.masked_fill(s_idx.eq(-1), 0.0)
    samples = {'sampled_point_depth': s_depth, 'sampled_point_distance': s_dist,
               'sampled_point_voxel_idx': s_idx, 'probs': probs, 'steps': steps, 'K': K}
    return inter, hits, samples


def chained_case(dev, R):
    """Model and oracle on the same map, embeddings and decoder, with the noise drawn by hit
    rank, for the chained full-step test."""
    from oracle.voxfusion import VoxOracle
    model, rays_o, rays_d, ts, td = scene(dev, R=R, seed=4)
    ora = VoxOracle()
    with torch.no_grad():
        g = torch.Generator().manual_seed(9)
        model.embeddings.copy_(torch.randn(model.embeddings.shape, generator=g) * 0.3)
        ora.embeddings.copy_(model.embeddings.cpu())
        ora.decoder.load_state_dict(model.decoder.state_dict())
    voxels, children, features = model.export_octree()
    ora.set_map(voxels, children, features)
    gen = torch.Generator().manual_seed(5)
    noise_rank = torch.rand(rays_o.shape[0], model.config.max_samples_per_ray,
                            generator=gen).clamp(0.001, 0.999)

    def noise_fn(shape):
        G, K, ms = shape
        out = torch.full((G * K, ms), 0.5)
        n = min(G * K, noise_rank.shape[0])
        out[:n] = noise_rank[:n, :ms]
        return out.reshape(G, K, ms)
    return model, ora, rays_o, rays_d, ts, td, noise_rank, noise_fn


@pytest.mark.parametrize('R', [300, 5 * 1024])
def test_full_step_vs_oracle_chained_through_reference_grid(cuda_dev, R):
    """Full step (march + sample + decode + composite + loss + backward) with the oracle fed
    intersections / samples bit-identical to the reference extension's own (every one checked
    against its stored digest): sample->voxel ids and depths BIT-EXACT, gradients rel-l2
    <= 5e-4.  R = 5 x 1024 is the default mapping batch (5 keyframes x 1024 rays,
    slam/configs/input_config.py vox-fusion entry)."""
    dev = cuda_dev
    model, ora, rays_o, rays_d, ts, td, noise_rank, noise_fn = chained_case(dev, R)
    grid = Recorder(OwnGrid(dev))
    ro_o = rays_o.clone().requires_grad_(True)
    rd_o = rays_d.clone().requires_grad_(True)
    marched = _march_through_grid(grid, ora, ro_o.detach(), rd_o.detach(), noise_fn, dev)
    assert grid.digests == golden()['chained'][str(R)]
    out_o, ld_o = ora.render(ro_o, rd_o, ts, td, marched)
    sum(ld_o.values()).backward()
    hits = marched[1]
    rank = torch.cumsum(hits.long(), 0) - 1
    noise = torch.full((rays_o.shape[0], model.config.max_samples_per_ray), 0.5)
    noise[hits] = noise_rank[rank[hits]]
    ro = rays_o.to(dev).requires_grad_(True)
    rd = rays_d.to(dev).requires_grad_(True)
    inp = dict(rays_o=ro, rays_d=rd, target_s=ts.to(dev), target_d=td.to(dev), noise=noise.to(dev))
    out = model(inp)
    ld = model.get_loss_dict(out, inp, True, 0)
    sum(ld.values()).backward()
    torch.cuda.synchronize()
    m = model.last_march
    assert m['overflow'] == 0
    assert torch.equal(out['ray_mask'].cpu(), hits)
    smp = marched[2]
    S = smp['sampled_point_voxel_idx'].shape[1]
    assert m['s_max'] == S and m['n_hit_rays'] == int(hits.sum())
    got_idx = m['smp_idx'].cpu()[hits][:, :S]
    assert torch.equal(got_idx, smp['sampled_point_voxel_idx'])               # bit-exact
    valid = got_idx >= 0
    assert torch.equal(m['smp_depth'].cpu()[hits][:, :S][valid],
                       smp['sampled_point_depth'][valid])                     # bit-exact
    assert max_abs(out['depth'], out_o['depth']) < 5e-5
    assert max_abs(out['rgb'], out_o['rgb']) < 5e-5
    for k in ld_o:
        a, b = float(ld[k].detach()), float(ld_o[k].detach())
        assert abs(a - b) <= 1e-4 * max(abs(b), 1e-6), (k, a, b)
    TOL = 5e-4
    assert rel_err(model.embeddings.grad, ora.embeddings.grad) < TOL
    sd_o = dict(ora.decoder.named_parameters())
    for n, p in model.decoder.named_parameters():
        assert rel_err(p.grad, sd_o[n].grad) < TOL, n
    assert rel_err(ro.grad, ro_o.grad) < TOL
    assert rel_err(rd.grad, rd_o.grad) < TOL


def test_device_octree_on_gpu_equals_host_octree(cuda_dev):
    """The map grown on the device (default) == the map grown by the host C++ octree: same
    node count, centres, structure and vertex tables after two frames."""
    from xrdslam_b200.sparse_voxel import SparseVoxelConfig
    from xrdslam_b200.synthetic import make_sequence
    cam, poses, frames = make_sequence(2, width=160, height=120, offset=(OFFSET,) * 3)
    H, W = cam.height, cam.width
    j, i = torch.meshgrid(torch.arange(H, dtype=torch.float32),
                          torch.arange(W, dtype=torch.float32), indexing='ij')
    dirs = torch.stack([(i - cam.cx) / cam.fx, -(j - cam.cy) / cam.fy, -torch.ones_like(i)], -1)
    models = [SparseVoxelConfig(device_octree=flag).setup(camera=cam).to(cuda_dev)
              for flag in (True, False)]
    for (rgb, depth), c2w in zip(frames, poses):
        c2w = torch.from_numpy(c2w)
        d = torch.from_numpy(depth)
        pts = (dirs * d[..., None])[d > 0].reshape(-1, 3)
        pts = (pts @ c2w[:3, :3].T + c2w[:3, 3]).to(cuda_dev)
        for m in models:
            m.insert_points(pts)
    a, b = models[0].map_states, models[1].map_states
    assert models[0]._dev_svo is not None and models[1]._dev_svo is None
    for k in ('voxel_vertex_idx', 'voxel_center_xyz', 'voxel_structure'):
        assert a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k
    for x, y in zip(models[0].export_octree(), models[1].export_octree()):
        assert torch.equal(x, y)
