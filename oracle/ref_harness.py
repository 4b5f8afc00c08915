"""Import the REAL reference classes from /root/reference (build container only).

ORACLE / TEST INFRASTRUCTURE.  Used only by tests/golden/make_golden.py, which runs the
reference's own Python and writes what the tests compare against into tests/golden/; the
tests themselves never import the reference.

The reference does not import cleanly under py3.12 (SURVEY.md section 0.4):
non-arithmetic packages are replaced by MagicMock modules, ``tinycudann`` by the
torch restatement in oracle/tcnn_restated.py and ``pytorch3d.transforms`` by the
three restated functions in oracle/transforms_restated.py.
"""
from __future__ import annotations

import os
import sys
import types
from unittest.mock import MagicMock

REF_ROOT = os.environ.get('XRDSLAM_REFERENCE', '/root/reference')

_STUBS = [
    'diff_gaussian_rasterization', 'faiss', 'grid', 'matplotlib',
    'matplotlib.pyplot', 'open3d', 'pytorch_msssim', 'skimage',
    'skimage.color', 'skimage.measure', 'skimage.filters', 'torchmetrics',
    'torchmetrics.image', 'torchmetrics.image.lpip', 'transforms3d', 'trimesh',
    'cv2'
]


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, 'slam'))


def install():
    """Idempotently put the reference on sys.path with the stubs in place."""
    if not available():
        raise RuntimeError(f'reference not found at {REF_ROOT}')
    if getattr(install, '_done', False):
        return
    for name in _STUBS:
        if name in sys.modules:
            continue
        try:
            __import__(name)
            continue
        except Exception:
            pass
        m = MagicMock()
        m.__path__ = []
        m.__name__ = name
        sys.modules[name] = m
    # tinycudann -> restated torch modules
    from oracle import tcnn_restated
    tc = types.ModuleType('tinycudann')
    tc.Encoding = tcnn_restated.Encoding
    tc.Network = MagicMock()
    sys.modules['tinycudann'] = tc
    # pytorch3d.transforms -> restated
    from oracle import transforms_restated
    p3 = types.ModuleType('pytorch3d')
    p3.__path__ = []
    p3t = types.ModuleType('pytorch3d.transforms')
    for fn in ('matrix_to_quaternion', 'quaternion_to_axis_angle',
               'quaternion_to_matrix'):
        setattr(p3t, fn, getattr(transforms_restated, fn))
    p3.transforms = p3t
    sys.modules.setdefault('pytorch3d', p3)
    sys.modules.setdefault('pytorch3d.transforms', p3t)
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    install._done = True


def ref_joint_encoding(bounding_box, camera=None, **cfg_overrides):
    """Instantiate the reference's JointEncoding (Co-SLAM model) on CPU."""
    install()
    from slam.common.camera import Camera
    from slam.models.joint_encoding import JointEncoding, JointEncodingConfig
    if camera is None:
        camera = Camera(320.0, 320.0, 319.5, 239.5, 640, 480)
    kw = dict(cam_depth_trunc=100.0, tcnn_encoding=True)
    kw.update(cfg_overrides)
    cfg = JointEncodingConfig(**kw)
    return JointEncoding(cfg, camera=camera, bounding_box=bounding_box)


def ref_conv_onet(bounding_box, camera=None, **cfg_overrides):
    """Instantiate the reference's ConvOnet (NICE-SLAM model) on CPU.  The pretrained
    decoder files are Git-LFS pointer stubs (SURVEY 0.5) -> load_pretrain is bypassed and
    the decoders keep their seeded xavier init."""
    install()
    import torch
    from slam.common.camera import Camera
    from slam.models.conv_onet import ConvOnet, ConvOnetConfig
    if camera is None:
        camera = Camera(320.0, 320.0, 319.5, 239.5, 640, 480)
    kw = dict(coarse=False, mapping_frustum_feature_selection=False)
    kw.update(cfg_overrides)
    orig = ConvOnet.load_pretrain
    ConvOnet.load_pretrain = lambda self: None
    try:
        model = ConvOnet(ConvOnetConfig(**kw), camera=camera,
                         bounding_box=torch.as_tensor(bounding_box, dtype=torch.float64).clone())
    finally:
        ConvOnet.load_pretrain = orig
    return model


def copy_nice_ref_to_oracle(ref, ora):
    """Copy decoders + grids of a reference ConvOnet into oracle.nice.NiceOracle."""
    import torch
    with torch.no_grad():
        for name in ('middle', 'fine', 'color'):
            r = getattr(ref.decoder, name + '_decoder')
            o = getattr(ora, name)
            o.B.copy_(r.embedder._B)
            for i in range(5):
                o.fc_c[i].weight.copy_(r.fc_c[i].weight)
                o.fc_c[i].bias.copy_(r.fc_c[i].bias)
                o.pts[i].weight.copy_(r.pts_linears[i].weight)
                o.pts[i].bias.copy_(r.pts_linears[i].bias)
            o.out.weight.copy_(r.output_linear.weight)
            o.out.bias.copy_(r.output_linear.bias)
        for k in ('grid_middle', 'grid_fine', 'grid_color'):
            ora.grids[k].copy_(ref.grid_c[k])
        if getattr(ora, 'coarse', None) is not None:
            r, o = ref.decoder.coarse_decoder, ora.coarse
            for i in range(5):
                o.pts[i].weight.copy_(r.pts_linears[i].weight)
                o.pts[i].bias.copy_(r.pts_linears[i].bias)
            o.out.weight.copy_(r.output_linear.weight)
            o.out.bias.copy_(r.output_linear.bias)
            ora.grids['grid_coarse'].copy_(ref.grid_c['grid_coarse'])


# ---- Point-SLAM: the reference's ConvOnet2 with an exact-kNN stand-in for faiss -----------
class _ExactIndex:
    """Minimal faiss.Index stand-in: exact L2 search (the real IndexIVFFlat(nlist 400,
    nprobe 4) is approximate and un-vendored: parity is defined against exact kNN)."""
    def __init__(self):
        import numpy as np
        self.xb = np.zeros((0, 3), np.float32)
        self.is_trained = False
        self.nprobe = 1

    @property
    def ntotal(self):
        return self.xb.shape[0]

    def train(self, x):
        self.is_trained = True

    def add(self, x):
        import numpy as np
        self.xb = np.concatenate([self.xb, np.asarray(x, np.float32)], 0)

    def search(self, q, k):
        import numpy as np
        import torch
        from oracle.pointslam import exact_knn
        D, I = exact_knn(torch.from_numpy(self.xb), torch.from_numpy(np.asarray(q, np.float32)), k)
        return D.numpy(), I.numpy().astype(np.int64)


def install_faiss_stub():
    import types
    f = types.ModuleType('faiss')
    f.METRIC_L2 = 1
    f.StandardGpuResources = lambda: None
    f.IndexFlatL2 = lambda d: None
    f.IndexIVFFlat = lambda quant, d, nlist, metric: _ExactIndex()
    f.index_cpu_to_gpu = lambda res, dev, index: index
    sys.modules['faiss'] = f


def ref_conv_onet2(**cfg_overrides):
    """The reference's Point-SLAM model (ConvOnet2) on CPU: pretrained-decoder loading
    bypassed (Git-LFS stubs), faiss replaced by the exact stand-in above."""
    install_faiss_stub()
    install()
    import importlib
    import slam.model_components.neural_point_cloud as npc_mod
    importlib.reload(npc_mod)  # bind the stub
    from slam.common.camera import Camera
    import slam.models.conv_onet_pointslam as m
    importlib.reload(m)
    orig = m.ConvOnet2.load_pretrain
    m.ConvOnet2.load_pretrain = lambda self: None
    try:
        model = m.ConvOnet2(m.ConvOnet2Config(**cfg_overrides),
                            camera=Camera(320.0, 320.0, 319.5, 239.5, 640, 480))
    finally:
        m.ConvOnet2.load_pretrain = orig
    return model


# ---- Vox-Fusion: the reference's SparseVoxel python (features, decoder, weights, losses) on
# ---- CPU, fed with precomputed intersections / samples (its CUDA ops are pinned separately
# ---- against oracle/_ref/grid.so on the GPU box)
def ref_sparse_voxel_cpu(map_states, embeddings, marched):
    """-> (model, module): a reference SparseVoxel whose map lives on the CPU and whose
    ray_intersect / ray_sample return `marched` = (intersections dict [R,H], hits [R] bool,
    samples dict [R',S])."""
    install()
    import torch
    import slam.models.sparse_voxel as sv
    from slam.model_components.decoder_voxfusion import Decoder
    cfg = sv.SparseVoxelConfig()
    model = sv.SparseVoxel.__new__(sv.SparseVoxel)
    torch.nn.Module.__init__(model)
    model.config = cfg
    cfg.step_size = cfg.voxel_size * cfg.step_size
    model.embeddings = torch.nn.Parameter(embeddings.clone())
    model.decoder = Decoder(depth=cfg.depth, width=cfg.width, in_dim=cfg.embed_dim,
                            embedder=cfg.embedder)
    ms = dict(map_states)
    ms['voxel_vertex_emb'] = model.embeddings
    model.map_states = ms
    inter, hits, samples = marched

    def fake_intersect(rays_o, rays_d, centres, children, voxel_size, n_max, max_distance):
        return {k: v.unsqueeze(0) for k, v in inter.items()}, hits.unsqueeze(0)

    def fake_sample(intersections, step_size):
        keys = ('sampled_point_depth', 'sampled_point_distance', 'sampled_point_voxel_idx')
        return {k: samples[k].clone() for k in keys}  # what the reference's ray_sample returns
    sv.ray_intersect, sv.ray_sample = fake_intersect, fake_sample
    return model, sv


import contextlib


@contextlib.contextmanager
def cuda_calls_are_noops():
    """The reference hard-codes `.cuda()` / `.to('cuda:N')` in a few helpers
    (voxel_helpers_voxfusion.py:108-110, decoder_nice.py:388-405): on this GPU-less container
    they become identity for the duration of the block."""
    import torch
    orig_cuda, orig_to = torch.Tensor.cuda, torch.Tensor.to

    def to(self, *a, **k):
        # decoder_nice.py:388 builds device = f'cuda:{p.get_device()}' ('cuda:-1' on the host)
        if a and isinstance(a[0], str) and a[0].startswith('cuda'):
            a = a[1:]
            if not a and not k:
                return self
        if isinstance(k.get('device'), str) and k['device'].startswith('cuda'):
            k = {kk: v for kk, v in k.items() if kk != 'device'}
            if not a and not k:
                return self
        return orig_to(self, *a, **k)
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.Tensor.to = to
    try:
        yield
    finally:
        torch.Tensor.cuda, torch.Tensor.to = orig_cuda, orig_to
