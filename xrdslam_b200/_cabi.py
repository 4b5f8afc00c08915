"""ctypes binding of include/xrdslam_b200.h (the C-ABI shared library).

The product path has NO fallback: if the library is missing or cannot be loaded
this module raises at import of the symbol table, and every op raises
``XrdError`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libxrdslam_b200.so')

XRD_MAX_LEVELS = 16
_STATUS = {
    0: 'XRD_OK',
    -1: 'XRD_E_SHAPE',
    -2: 'XRD_E_ARCH',
    -3: 'XRD_E_WORKSPACE',
    -4: 'XRD_E_NOHIT',
    -5: 'XRD_E_CUDA',
    -6: 'XRD_E_NULL',
}
XRD_E_NOHIT = -4


class XrdError(RuntimeError):
    def __init__(self, fn, status, cuda_err=0):
        self.status = status
        super().__init__(
            f'{fn} failed: {_STATUS.get(status, status)}'
            + (f' (cudaError {cuda_err})' if status == -5 else ''))


fp = C.POINTER(C.c_float)
vp = C.c_void_p


class XrdRays(C.Structure):
    _fields_ = [('n_rays', C.c_int), ('rays_o', vp), ('rays_d', vp),
                ('target_s', vp), ('target_d', vp)]


class XrdHashGrid(C.Structure):
    _fields_ = [('n_levels', C.c_int),
                ('scale', C.c_float * XRD_MAX_LEVELS),
                ('resolution', C.c_uint32 * XRD_MAX_LEVELS),
                ('size', C.c_uint32 * XRD_MAX_LEVELS),
                ('offset', C.c_uint32 * XRD_MAX_LEVELS),
                ('hashed', C.c_uint32 * XRD_MAX_LEVELS),
                ('n_entries', C.c_uint32), ('bbox_min', C.c_double * 3),
                ('bbox_max', C.c_double * 3), ('table', vp)]


class XrdCoslamMlp(C.Structure):
    _fields_ = [('w_sdf0', vp), ('w_sdf1', vp), ('w_col0', vp), ('w_col1', vp)]


class XrdCoslamCfg(C.Structure):
    _fields_ = [('n_samples', C.c_int), ('n_sample_d', C.c_int),
                ('n_range_d', C.c_int), ('perturb', C.c_int),
                ('trunc', C.c_float), ('depth_trunc', C.c_float),
                ('w_rgb', C.c_float), ('w_depth', C.c_float),
                ('w_sdf', C.c_float), ('w_fs', C.c_float),
                ('lin_uniform', vp), ('lin_range', vp), ('lin_nodepth', vp),
                ('lin_full', vp), ('seed', C.c_uint64),
                ('rays_per_tile', C.c_int), ('precision', C.c_int),
                ('phase', C.c_int), ('n_rays_global', C.c_int),
                ('counts_global', vp), ('counts_out', vp), ('seed_dev', vp)]


class XrdCoslamOut(C.Structure):
    _fields_ = [('rgb', vp), ('depth', vp), ('disp', vp), ('acc', vp),
                ('depth_var', vp), ('z_vals', vp), ('raw', vp), ('losses', vp)]


class XrdCoslamGrads(C.Structure):
    _fields_ = [('d_table', vp), ('d_w_sdf0', vp), ('d_w_sdf1', vp),
                ('d_w_col0', vp), ('d_w_col1', vp), ('d_rays_o', vp),
                ('d_rays_d', vp), ('loss_scale', C.c_float * 4)]


class XrdNiceDecoder(C.Structure):
    _fields_ = [('B', vp), ('pts_w', vp * 5), ('pts_b', vp * 5), ('fcc_w', vp * 5),
                ('fcc_b', vp * 5), ('out_w', vp), ('out_b', vp), ('c_dim', C.c_int),
                ('n_out', C.c_int)]


class XrdNiceDecoderGrads(C.Structure):
    _fields_ = [('B', vp), ('pts_w', vp * 5), ('pts_b', vp * 5), ('fcc_w', vp * 5),
                ('fcc_b', vp * 5), ('out_w', vp), ('out_b', vp)]


class XrdNiceGrid(C.Structure):
    _fields_ = [('data', vp), ('nx', C.c_int), ('ny', C.c_int), ('nz', C.c_int)]


class XrdNiceCfg(C.Structure):
    _fields_ = [('stage', C.c_int), ('is_mapping', C.c_int), ('n_samples', C.c_int),
                ('n_surface', C.c_int), ('bound_min', C.c_double * 3),
                ('bound_max', C.c_double * 3), ('w_color', C.c_float),
                ('handle_dynamic', C.c_int), ('use_color_in_tracking', C.c_int),
                ('t_uniform', vp), ('t_surface', vp), ('max_depth_global', vp)]


class XrdNiceCoarseDecoder(C.Structure):
    _fields_ = [('pts_w', vp * 5), ('pts_b', vp * 5), ('out_w', vp), ('out_b', vp)]


class XrdNiceCoarseCfg(C.Structure):
    _fields_ = [('n_samples', C.c_int), ('bound_min', C.c_double * 3),
                ('bound_max', C.c_double * 3), ('coarse_bound_min', C.c_double * 3),
                ('coarse_bound_max', C.c_double * 3), ('t_uniform', vp)]


class XrdNiceOut(C.Structure):
    _fields_ = [('rgb', vp), ('depth', vp), ('uncertainty', vp), ('z_vals', vp),
                ('raw', vp), ('losses', vp)]


class XrdNiceGrads(C.Structure):
    _fields_ = [('d_grid', vp * 3), ('d_color', C.POINTER(XrdNiceDecoderGrads)),
                ('d_rays_o', vp), ('d_rays_d', vp)]


class XrdVoxMap(C.Structure):
    _fields_ = [('n_nodes', C.c_int), ('centres', vp), ('children', vp), ('vertex_idx', vp),
                ('embeddings', vp), ('n_embeddings', C.c_int)]


class XrdVoxMarchCfg(C.Structure):
    _fields_ = [('voxel_size', C.c_float), ('step_size', C.c_float), ('max_hits', C.c_int),
                ('max_distance', C.c_float), ('max_samples', C.c_int),
                ('rays_per_block', C.c_int), ('seed', C.c_uint64)]


class XrdVoxMarch(C.Structure):
    _fields_ = [('hit_idx', vp), ('hit_tmin', vp), ('hit_tmax', vp), ('smp_idx', vp),
                ('smp_depth', vp), ('smp_dist', vp), ('smp_count', vp), ('smp_base', vp),
                ('ray_mask', vp), ('stats', vp)]


class XrdVoxDecoder(C.Structure):
    _fields_ = [(n, vp) for n in ('w0', 'b0', 'w1', 'b1', 'ws', 'bs', 'wc0', 'bc0', 'wc1', 'bc1')]


class XrdVoxDecoderGrads(C.Structure):
    _fields_ = [(n, vp) for n in ('w0', 'b0', 'w1', 'b1', 'ws', 'bs', 'wc0', 'bc0', 'wc1', 'bc1')]


class XrdVoxRenderCfg(C.Structure):
    _fields_ = [('voxel_size', C.c_float), ('trunc', C.c_float), ('max_depth', C.c_float),
                ('pad_depth', C.c_float), ('w_rgb', C.c_float), ('w_depth', C.c_float),
                ('w_sdf', C.c_float), ('w_fs', C.c_float), ('n_points', C.c_int),
                ('s_max', C.c_int), ('n_hit_rays', C.c_int)]


class XrdVoxOut(C.Structure):
    _fields_ = [('rgb', vp), ('depth', vp), ('losses', vp)]


class XrdVoxGrads(C.Structure):
    _fields_ = [('d_embeddings', vp), ('d_decoder', C.POINTER(XrdVoxDecoderGrads)),
                ('d_rays_o', vp), ('d_rays_d', vp)]


class XrdMcVolumes(C.Structure):
    _fields_ = [('field', vp), ('n_volumes', C.c_int), ('nx', C.c_int), ('ny', C.c_int),
                ('nz', C.c_int), ('origin', C.c_double * 3), ('spacing', C.c_double * 3),
                ('origins', vp), ('spacings', vp)]


class XrdPointIndex(C.Structure):
    _fields_ = [('pos', vp), ('n_points', C.c_int), ('cell', C.c_float),
                ('table_size', C.c_int), ('cell_start', vp), ('cell_end', vp),
                ('sorted_ids', vp)]


class XrdPointCfg(C.Structure):
    _fields_ = [('stage', C.c_int), ('is_mapping', C.c_int), ('n_surface', C.c_int),
                ('near_end_surface', C.c_float), ('far_end_surface', C.c_float),
                ('near_end', C.c_float), ('sigmoid_coef', C.c_float), ('min_nn_num', C.c_int),
                ('w_color', C.c_float), ('handle_dynamic', C.c_int),
                ('use_color_in_tracking', C.c_int), ('t_surface', vp), ('far', vp),
                ('radius_query', vp), ('rand_feat', vp), ('rand_feat_color', vp)]


class XrdPointFeats(C.Structure):
    _fields_ = [('geo_feats', vp), ('frustum_mask', vp), ('col_feats', vp)]


class XrdPointColorDecoder(C.Structure):
    _fields_ = [('B', vp), ('B_rel', vp), ('nb_w1', vp), ('nb_b1', vp), ('nb_w2', vp),
                ('nb_b2', vp), ('w', vp * 5), ('b', vp * 5), ('wc', vp * 5), ('bc', vp * 5),
                ('wo', vp), ('bo', vp)]


class XrdPointColorDecoderGrads(C.Structure):
    _fields_ = [('B_rel', vp), ('nb_w1', vp), ('nb_b1', vp), ('nb_w2', vp), ('nb_b2', vp),
                ('w', vp * 5), ('b', vp * 5), ('wc', vp * 5), ('bc', vp * 5), ('wo', vp),
                ('bo', vp)]


class XrdPointOut(C.Structure):
    _fields_ = [('rgb', vp), ('depth', vp), ('uncertainty', vp), ('valid_ray_mask', vp),
                ('z_vals', vp), ('losses', vp)]


class XrdPointGrads(C.Structure):
    _fields_ = [('d_geo_feats', vp), ('d_rays_o', vp), ('d_rays_d', vp), ('d_col_feats', vp),
                ('color', C.POINTER(XrdPointColorDecoderGrads))]


_lib = None

# name -> (restype, argtypes); every symbol include/xrdslam_b200.h declares
class XrdAdamTensor(C.Structure):
    _fields_ = [('param', vp), ('grad', vp), ('exp_avg', vp), ('exp_avg_sq', vp),
                ('n', C.c_longlong), ('lr', C.c_float), ('beta1', C.c_float),
                ('beta2', C.c_float), ('eps', C.c_float), ('weight_decay', C.c_float),
                ('bias_correction1', C.c_float), ('bias_correction2', C.c_float),
                ('row_mask', vp), ('row_len', C.c_int), ('dyn', vp)]


class XrdPixelSampleCfg(C.Structure):
    _fields_ = [('n_frames', C.c_int), ('n_per_frame', C.c_int), ('H', C.c_int), ('W', C.c_int),
                ('H0', C.c_int), ('H1', C.c_int), ('W0', C.c_int), ('W1', C.c_int),
                ('fx', C.c_float), ('fy', C.c_float), ('cx', C.c_float), ('cy', C.c_float)]


SYMBOLS = {
    'xrd_sample_pixels': (C.c_int, [C.POINTER(XrdPixelSampleCfg), C.POINTER(vp), C.POINTER(vp), vp,
                                    vp, vp, vp, vp, vp, vp]),
    'xrd_rays_from_poses': (C.c_int, [C.c_int, vp, vp, vp, C.c_int, vp, vp, vp]),
    'xrd_rays_pose_grads': (C.c_int, [C.c_int, vp, vp, C.c_int, vp, vp, vp, vp]),
    'xrd_adam_step': (C.c_int, [C.POINTER(XrdAdamTensor), C.c_int, C.c_int, vp]),
    'xrd_pose_matrices': (C.c_int, [C.c_int, vp, vp, vp, vp]),
    'xrd_pose_matrices_grads': (C.c_int, [C.c_int, vp, vp, vp, vp, vp, vp]),
    'xrd_abi_version': (C.c_int, []),
    'xrd_last_cuda_error': (C.c_int, []),
    'xrd_check_device': (C.c_int, [C.c_int]),
    'xrd_debug_kernel_events': (C.c_int, [vp, vp]),
    'xrd_linspace_f32': (C.c_int, [C.c_float, C.c_float, C.c_int, fp]),
    'xrd_hashgrid_layout':
    (C.c_int, [C.POINTER(XrdHashGrid), C.c_int, C.c_int, C.c_int, C.c_float]),
    'xrd_coslam_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'xrd_coslam_step': (C.c_int, [
        C.POINTER(XrdRays),
        C.POINTER(XrdHashGrid),
        C.POINTER(XrdCoslamMlp),
        C.POINTER(XrdCoslamCfg), vp,
        C.POINTER(XrdCoslamOut),
        C.POINTER(XrdCoslamGrads), vp, C.c_size_t, vp
    ]),
    'xrd_coslam_smoothness_workspace_bytes': (C.c_size_t, [C.c_int]),
    'xrd_coslam_smoothness': (C.c_int, [
        C.POINTER(XrdHashGrid), C.c_int, C.c_double, C.c_double, C.c_float, fp,
        vp, vp, C.c_float, vp, C.c_size_t, vp
    ]),
    'xrd_coslam_smoothness_dev': (C.c_int, [
        C.POINTER(XrdHashGrid), C.c_int, C.c_double, C.c_double, C.c_float, vp,
        vp, vp, C.c_float, vp, C.c_size_t, vp
    ]),
    'xrd_hashgrid_encode':
    (C.c_int, [C.POINTER(XrdHashGrid), vp, C.c_int, vp, vp, vp]),
    'xrd_octree_create': (vp, [C.c_int]),
    'xrd_octree_destroy': (None, [vp]),
    'xrd_octree_num_nodes': (C.c_int, [vp]),
    'xrd_octree_insert': (C.c_int, [vp, vp, C.c_int]),
    'xrd_octree_export': (C.c_int, [vp, vp, vp, vp]),
    'xrd_voxfusion_march': (C.c_int, [C.POINTER(XrdRays), C.POINTER(XrdVoxMap),
                                      C.POINTER(XrdVoxMarchCfg), vp, C.POINTER(XrdVoxMarch), vp]),
    'xrd_voxfusion_intersect_raw': (C.c_int, [C.POINTER(XrdRays), C.POINTER(XrdVoxMap),
                                              C.c_float, C.c_int, vp, vp, vp, vp]),
    'xrd_voxfusion_sample_raw': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp,
                                           vp, vp, vp, vp, vp, vp]),
    'xrd_voxfusion_render_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    'xrd_voxfusion_render': (C.c_int, [
        C.POINTER(XrdRays), C.POINTER(XrdVoxMap), C.POINTER(XrdVoxMarch),
        C.POINTER(XrdVoxMarchCfg), C.POINTER(XrdVoxDecoder), C.POINTER(XrdVoxRenderCfg),
        C.POINTER(XrdVoxOut), C.POINTER(XrdVoxGrads), vp, C.c_size_t, vp]),
    'xrd_voxfusion_query_workspace_bytes': (C.c_size_t, [C.c_int]),
    'xrd_voxfusion_query': (C.c_int, [C.POINTER(XrdVoxMap), C.POINTER(XrdVoxDecoder), C.c_float,
                                      vp, vp, C.c_int, vp, vp, C.c_size_t, vp]),
    'xrd_mc_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    'xrd_mc_count': (C.c_int, [C.POINTER(XrdMcVolumes), C.c_float, vp, vp, C.c_size_t, vp]),
    'xrd_mc_emit': (C.c_int, [C.POINTER(XrdMcVolumes), C.c_float, vp, vp, vp, C.c_size_t, vp]),
    'xrd_pointslam_knn_query': (C.c_int, [C.POINTER(XrdPointIndex), vp, vp, C.c_int, C.c_int,
                                          vp, vp, vp, vp]),
    'xrd_coslam_query': (C.c_int, [C.POINTER(XrdHashGrid), C.POINTER(XrdCoslamMlp), vp, C.c_int,
                                   C.c_int, vp, vp, vp, vp]),
    'xrd_debug_gemm_mode': (C.c_int, [C.c_int]),
    'xrd_debug_gemm_variant': (C.c_int, [C.c_int]),
    'xrd_debug_gemm': (C.c_int, [C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, vp,
                                 C.c_int, vp, C.c_int, vp, C.c_int, vp, C.c_int, vp]),
    'xrd_debug_gemm_ex': (C.c_int, [C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, vp,
                                    C.c_int, vp, C.c_int, vp, C.c_int, vp, C.c_int, vp, C.c_int,
                                    C.c_int, vp]),
    'xrd_debug_dw': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    'xrd_pointslam_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    'xrd_pointslam_step': (C.c_int, [
        C.POINTER(XrdRays), C.POINTER(XrdPointIndex), C.POINTER(XrdPointFeats),
        C.POINTER(XrdNiceDecoder), C.POINTER(XrdPointColorDecoder), C.POINTER(XrdPointCfg),
        C.POINTER(XrdPointOut), C.POINTER(XrdPointGrads), vp, C.c_size_t, vp]),
    'xrd_nice_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    'xrd_pointslam_knn_build_workspace_bytes': (C.c_size_t, [C.c_int]),
    'xrd_pointslam_knn_build': (C.c_int, [vp, C.c_int, C.c_float, C.c_int, vp, vp, vp, vp, C.c_size_t,
                                          vp]),
    'xrd_nice_query_workspace_bytes': (C.c_size_t, [C.c_int]),
    'xrd_nice_query': (C.c_int, [vp, C.c_int, C.POINTER(XrdNiceGrid), C.POINTER(XrdNiceDecoder),
                                 C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, vp, vp,
                                 C.c_size_t, vp]),
    'xrd_nice_coarse_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    'xrd_nice_coarse_step': (C.c_int, [
        C.POINTER(XrdRays), C.POINTER(XrdNiceGrid), C.POINTER(XrdNiceCoarseDecoder),
        C.POINTER(XrdNiceCoarseCfg), C.POINTER(XrdNiceOut), vp, vp, vp, C.c_int, vp, C.c_size_t,
        vp]),
    'xrd_nice_step': (C.c_int, [
        C.POINTER(XrdRays), C.POINTER(XrdNiceGrid), C.POINTER(XrdNiceDecoder),
        C.POINTER(XrdNiceCfg), C.POINTER(XrdNiceOut), C.POINTER(XrdNiceGrads), vp,
        C.c_size_t, vp
    ]),
}


def lib():
    """Load the shared library (once) and type every exported symbol."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f'{LIB_PATH} not found: build it with '
                '`python -m xrdslam_b200.build` (there is no CPU fallback)')
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)  # AttributeError if the .so lacks a symbol
            f.restype = res
            f.argtypes = args
        if L.xrd_abi_version() != 1:
            raise ImportError('xrdslam_b200 ABI version mismatch')
        _lib = L
    return _lib


def check(fn_name, status):
    if status != 0:
        raise XrdError(fn_name, status, lib().xrd_last_cuda_error())


def ptr(t):
    """Device/host pointer of a (contiguous) torch tensor, or None."""
    if t is None:
        return None
    assert t.is_contiguous(), 'C-ABI needs contiguous tensors'
    return t.data_ptr()
