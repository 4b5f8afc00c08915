/*
 * xrdslam_b200 -- C-ABI of the B200-native render-and-optimise hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point is
 * `extern "C"`, takes plain pointers / sizes / POD structs, never allocates,
 * never frees, never synchronises the stream: one call = an asynchronous enqueue
 * of sm_100a kernels on `stream` (a cudaStream_t passed as void*).  All buffers,
 * including the workspace, are owned by the caller (torch on the Python side).
 * Return value: XRD_OK (0) or a negative XrdStatus.  No exceptions, no exit().
 *
 * What each entry point replaces in the reference (paths relative to
 * /root/reference, commit f0366f20):
 *
 *   xrd_coslam_step        slam/models/joint_encoding.py:158-163  get_outputs
 *                          -> render_rays :250-344, run_network :483-507,
 *                          query_color_sdf :463-481 (tcnn HashGrid + OneBlob via
 *                          slam/model_components/encodings_coslam.py:39-75,
 *                          decoders slam/model_components/decoder_coslam.py:139-163),
 *                          sdf2weights :346-374, raw2outputs :376-406,
 *                          get_loss_dict :94-147 (+ utils.py:100-186) and the
 *                          autograd backward of all of it (loss.backward(),
 *                          slam/algorithms/base_algorithm.py:266).
 *   xrd_coslam_smoothness  slam/models/joint_encoding.py:165-197 smoothness
 *                          (forward + gradient w.r.t. the hash table).
 *   xrd_hashgrid_layout    tcnn GridEncodingTemplated ctor (level offsets), the
 *                          config built at encodings_coslam.py:39-53.
 *   xrd_linspace_f32       torch.linspace as used at joint_encoding.py:264-279.
 *
 * (NICE-SLAM / Vox-Fusion / Point-SLAM entry points are declared further down.)
 */
#ifndef XRDSLAM_B200_H_
#define XRDSLAM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XRD_ABI_VERSION 1
#define XRD_MAX_LEVELS 16

typedef enum {
  XRD_OK = 0,
  XRD_E_SHAPE = -1,     /* inconsistent sizes / unsupported configuration   */
  XRD_E_ARCH = -2,      /* device is not sm_100                              */
  XRD_E_WORKSPACE = -3, /* workspace too small                               */
  XRD_E_NOHIT = -4,     /* Vox-Fusion: no ray hit any voxel (reference: None) */
  XRD_E_CUDA = -5,      /* a CUDA runtime call failed (see xrd_last_cuda_error) */
  XRD_E_NULL = -6       /* a required pointer is NULL                        */
} XrdStatus;

int xrd_abi_version(void);
/* cudaError_t of the last failing runtime call on this thread (0 if none). */
int xrd_last_cuda_error(void);
/* 0 if device `dev` is compute capability 10.x, XRD_E_ARCH otherwise. */
int xrd_check_device(int dev);

/* Measurement hook (bench.py roofline): when both events are non-NULL the NEXT
 * dominant-kernel launch made from this thread (k_fused of xrd_coslam_step, the
 * fused render kernels of the other representations) is bracketed by
 * cudaEventRecord(start)/(stop) on the launching stream.  Pass NULL, NULL to
 * clear.  The events are cudaEvent_t handles owned by the caller. */
int xrd_debug_kernel_events(void* start_event, void* stop_event);

/* ---- shared ------------------------------------------------------------ */

/* A batch of rays.  All pointers are DEVICE pointers, fp32, contiguous. */
typedef struct {
  int n_rays;
  const float* rays_o;   /* [R,3] */
  const float* rays_d;   /* [R,3] */
  const float* target_s; /* [R,3] colour target, may be NULL (render only)   */
  const float* target_d; /* [R]   depth target,  may be NULL                 */
} XrdRays;

/* torch.linspace(start, end, steps) for float32 by ATen's scalar formula (host
 * function, writes `steps` floats to host memory `out`).  ATen's vectorised CPU
 * path differs in the last bit for some elements depending on the host's SIMD
 * width; callers that need the reference's exact z samples pass tables made by
 * torch.linspace on the same host (the Python plugin does). */
int xrd_linspace_f32(float start, float end, int steps, float* out);

/* ---- shared front-end / optimiser (SURVEY rows A2, A7, B3; "next" row f1) ---------- */

/* World-frame rays from camera-frame directions and a per-ray pose row:
 *   rays_d[r] = sum_j dirs_cam[r][j] * poses[id][:3, j],  rays_o[r] = poses[id][:3, 3]
 * replaces slam/common/common.py:39-53 (get_rays_from_uv) and the per-ray pose gather of
 * slam/algorithms/coslam.py:208-216.  poses: DEVICE [n_poses,4,4] row-major c2w; pose_ids:
 * DEVICE [R] int64 or NULL (all rays use pose 0); negative ids index from the end (python). */
int xrd_rays_from_poses(int n_rays, const float* dirs_cam, const int64_t* pose_ids,
                        const float* poses, int n_poses, float* rays_o, float* rays_d,
                        void* stream);

/* Backward of the above: d_poses [n_poses,4,4] (zeroed inside, bottom row stays 0)
 *   d_poses[id][:3,:3] += outer(d_rays_d[r], dirs_cam[r]),  d_poses[id][:3,3] += d_rays_o[r]
 * (what torch's index_put(accumulate=True) backward of `poses_all[ids]` computes). */
int xrd_rays_pose_grads(int n_rays, const float* dirs_cam, const int64_t* pose_ids, int n_poses,
                        const float* d_rays_o, const float* d_rays_d, float* d_poses,
                        void* stream);

/* Pixel sampling for a window of frames in one launch: gathers depth / colour of the chosen
 * pixels of device-resident frames and builds the camera-frame directions
 *   dirs = [(i - cx) / fx, -(j - cy) / fy, -1],  i = idx % (W1 - W0) + W0,  j = idx / (W1 - W0) + H0
 * (slam/common/common.py:56-71 select_uv, :109-122 get_sample_uv, :45-47; the reference
 * re-uploads both full images for every frame of every iteration).  indices: DEVICE
 * [n_frames * n_per_frame] int64 into the cropped region (row-major), frame-major; the draw
 * itself (torch.randint, with replacement, Q7) stays with the caller.  depth_imgs / rgb_imgs:
 * HOST arrays of n_frames DEVICE pointers ([H,W] and [H,W,3] fp32).  Outputs are frame-major;
 * pose_ids[q] = frame index (feeds xrd_rays_from_poses); ij: optional [n,2] (column, row). */
typedef struct {
  int n_frames;    /* <= 32 */
  int n_per_frame;
  int H, W;        /* image size */
  int H0, H1, W0, W1; /* sampled region (Hedge / Wedge crop) */
  float fx, fy, cx, cy;
} XrdPixelSampleCfg;

int xrd_sample_pixels(const XrdPixelSampleCfg* cfg, const float* const* depth_imgs,
                      const float* const* rgb_imgs, const int64_t* indices, float* dirs,
                      float* depth, float* rgb, int64_t* pose_ids, int64_t* ij, void* stream);

/* c2w [n,4,4] from axis-angle `rot` [n,3] and translation `trans` [n,3] (all DEVICE):
 * slam/utils/opt_pose.py:51-55,77-95 (OptimizablePose.matrix / Rodrigues). */
int xrd_pose_matrices(int n_poses, const float* rot, const float* trans, float* c2w, void* stream);

/* Backward of the above (what torch autograd computes through opt_pose.py): d_rot / d_trans
 * [n,3] are ACCUMULATED into (Co-SLAM steps its mapping poses every 5th iteration on the summed
 * gradients, SURVEY Q11).  fixed: DEVICE [n] or NULL; rows with fixed != 0 receive nothing
 * (the first frame of the window, coslam.py:181-182 / base_algorithm.py:196-199). */
int xrd_pose_matrices_grads(int n_poses, const float* rot, const float* d_c2w,
                            const uint8_t* fixed, float* d_rot, float* d_trans, void* stream);

/* One tensor of a multi-tensor Adam step (torch.optim.Adam, amsgrad=False); all DEVICE fp32.
 * bias_correction{1,2} = 1 - beta{1,2}^step with step counted from 1 (host, double -> float). */
#define XRD_ADAM_MAX_TENSORS 24
typedef struct {
  float* param; float* grad; float* exp_avg; float* exp_avg_sq;
  long long n;
  float lr, beta1, beta2, eps, weight_decay, bias_correction1, bias_correction2;
  /* optional row mask: element i is updated only if row_mask[i / row_len] != 0.  This is the
   * frustum feature selection of NICE-SLAM (slam/models/conv_onet.py:94-114,187-211: the
   * reference optimises a compacted copy val[mask] and scatters it back into the full grid
   * every iteration); rows = voxels of the channel-last grid, row_len = 32. */
  const uint8_t* row_mask;
  int row_len;
  /* optional DEVICE [3] = {lr, bias_correction1, bias_correction2} overriding the host values:
   * lets a captured CUDA graph replay the step with per-iteration scalars. */
  const float* dyn;
} XrdAdamTensor;

/* tensors: HOST array.  zero_grad != 0 also clears every grad (folds zero_grad_all,
 * slam/engine/optimizers.py:150-162, into the pass).  Replaces optimizer_step_all (:125-148)
 * for device-resident parameter groups. */
int xrd_adam_step(const XrdAdamTensor* tensors, int n_tensors, int zero_grad, void* stream);

/* ---- Co-SLAM ------------------------------------------------------------ */

/* Multi-resolution hash grid in tcnn's parameter layout: one flat fp32 array,
 * level-major, entry-major, feature-minor, 2 features per entry. */
typedef struct {
  int n_levels;                        /* <= XRD_MAX_LEVELS (Co-SLAM: 16)      */
  float scale[XRD_MAX_LEVELS];         /* grid_scale(level)                    */
  uint32_t resolution[XRD_MAX_LEVELS]; /* grid_resolution(scale)               */
  uint32_t size[XRD_MAX_LEVELS];       /* entries in level                     */
  uint32_t offset[XRD_MAX_LEVELS];     /* first entry of level                 */
  uint32_t hashed[XRD_MAX_LEVELS];     /* 1: coherent-prime hash, 0: dense     */
  uint32_t n_entries;                  /* sum(size)                            */
  double bbox_min[3];                  /* scene bound, float64 as the reference */
  double bbox_max[3];
  const float* table;                  /* DEVICE [n_entries*2]                 */
} XrdHashGrid;

/* Fill scale/resolution/size/offset/hashed/n_entries (host function). */
int xrd_hashgrid_layout(XrdHashGrid* g, int n_levels, int log2_hashmap_size,
                        int base_resolution, float per_level_scale);

/* ColorSDFNet_v2 weights, torch nn.Linear layout [out,in], no bias. DEVICE. */
typedef struct {
  const float* w_sdf0; /* [32,80]  in = hash32 ++ oneblob48                  */
  const float* w_sdf1; /* [16,32]  out = sdf ++ geo15                        */
  const float* w_col0; /* [32,63]  in = oneblob48 ++ geo15                   */
  const float* w_col1; /* [3,32]                                             */
} XrdCoslamMlp;

typedef struct {
  int n_samples;      /* S: samples per ray actually marched (43 with depth) */
  int n_sample_d;     /* 32 uniform samples in [near,far]                    */
  int n_range_d;      /* 11 depth-guided samples                             */
  int perturb;        /* stratified jitter on/off                            */
  float trunc;        /* training_trunc * sc_factor (0.1)                    */
  float depth_trunc;  /* cam_depth_trunc (100)                               */
  float w_rgb, w_depth, w_sdf, w_fs; /* loss weights 5, 0.1, 1000, 10        */
  /* DEVICE tables, normally produced with torch.linspace / xrd_linspace_f32: */
  const float* lin_uniform;  /* [n_sample_d]  linspace(near, far)             */
  const float* lin_range;    /* [n_range_d]   linspace(-range_d, range_d)     */
  const float* lin_nodepth;  /* [n_range_d]   linspace(near, far)             */
  const float* lin_full;     /* [n_samples]   used when target_d == NULL      */
  uint64_t seed;             /* Philox seed when noise == NULL                */
  int rays_per_tile;         /* 0 = automatic (grouped kernel for large gradient
                              * batches, tile kernel otherwise); -1 = tile kernel,
                              * -2 = grouped kernel, > 0 = tile kernel, rays/tile */
  int precision;             /* decoder GEMMs on the tensor cores:
                              * 0 = 3xTF32 everywhere (fp32-level accuracy),
                              * 1 = 3xTF32 forward (outputs/losses fp32-level),
                              *     plain TF32 backward (gradients ~1e-3 rel),
                              * 2 = plain TF32 everywhere                       */
  /* data-parallel mapping (loss normalisers are batch-global, SURVEY Q9):       */
  int phase;                 /* 0 = sample+render, 1 = sample only (z_vals and
                              * counts_out), 2 = render only (z_vals given)     */
  int n_rays_global;         /* rays of the all-rank batch; 0 = n_rays          */
  const int* counts_global;  /* DEVICE [3] n_fs, n_sdf, n_valid of the all-rank
                              * batch; NULL = this call's own counts            */
  int* counts_out;           /* DEVICE [4], written in phase 1                  */
  const uint64_t* seed_dev;  /* DEVICE scalar overriding `seed` (read by the kernel:
                              * a captured CUDA graph replays with a fresh seed)  */
} XrdCoslamCfg;

/* Per-ray / per-sample outputs (DEVICE, any may be NULL except losses when
 * grads are requested). */
typedef struct {
  float* rgb;       /* [R,3] */
  float* depth;     /* [R]   */
  float* disp;      /* [R]   */
  float* acc;       /* [R]   */
  float* depth_var; /* [R]   */
  float* z_vals;    /* [R,S] */
  float* raw;       /* [R,S,4] rgb logits ++ sdf */
  float* losses;    /* [4] rgb, depth, sdf, fs -- already multiplied by w_*  */
} XrdCoslamOut;

/* Gradients of (rgb+depth+sdf+fs) loss scaled by loss_scale[4] per term.
 * d_table and d_w_* are ACCUMULATED into (caller zeroes them: mapping-pose Adam
 * uses accum_step, Q11); d_rays_* are overwritten.  The five map gradients are
 * all-or-nothing: all NULL selects the pose-only pass used by tracking (no
 * scatter, no weight-gradient tiles). */
typedef struct {
  float* d_table;  /* [n_entries*2] */
  float* d_w_sdf0; /* [32,80] */
  float* d_w_sdf1; /* [16,32] */
  float* d_w_col0; /* [32,63] */
  float* d_w_col1; /* [3,32]  */
  float* d_rays_o; /* [R,3] or NULL */
  float* d_rays_d; /* [R,3] or NULL */
  float loss_scale[4]; /* upstream d total / d term (normally 1,1,1,1) */
} XrdCoslamGrads;

size_t xrd_coslam_workspace_bytes(int n_rays, int n_samples);

/* One fused forward(+backward) pass.  noise: DEVICE [R,S] uniform(0,1) replacing
 * torch.rand(z_vals.shape) (joint_encoding.py:292) or NULL for in-kernel Philox.
 * grads == NULL -> forward only (render_img). */
int xrd_coslam_step(const XrdRays* rays, const XrdHashGrid* grid,
                    const XrdCoslamMlp* mlp, const XrdCoslamCfg* cfg,
                    const float* noise, XrdCoslamOut* out,
                    XrdCoslamGrads* grads, void* workspace,
                    size_t workspace_bytes, void* stream);

size_t xrd_coslam_smoothness_workspace_bytes(int sample_points);

/* Smoothness / TV regulariser on the hash features (joint_encoding.py:165-197).
 * smooth_rand: HOST [6] = torch.rand(3) ++ torch.rand((1,1,1,3)).  Writes
 * weight*loss to DEVICE loss[0]; if d_table != NULL accumulates
 * grad_scale*weight*dloss/dtable into it. */
/* (xrd_coslam_smoothness_dev: the same with smooth_rand in DEVICE memory, read by the
 * kernels -- for CUDA-graph replay.) */
int xrd_coslam_smoothness(const XrdHashGrid* grid, int sample_points,
                          double voxel_size, double margin, float weight,
                          const float* smooth_rand, float* loss, float* d_table,
                          float grad_scale, void* workspace,
                          size_t workspace_bytes, void* stream);
int xrd_coslam_smoothness_dev(const XrdHashGrid* grid, int sample_points,
                          double voxel_size, double margin, float weight,
                          const float* smooth_rand, float* loss, float* d_table,
                          float grad_scale, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Point queries of the mesher path (slam/models/joint_encoding.py:408-481 query_fn /
 * color_func / query_sdf / query_color_sdf; slam/common/mesher.py:138-263 calls them on
 * marching-cubes lattice points): pts DEVICE [P,3], world coordinates (normalised = 0: the
 * kernel applies (p - bbox_min) / (bbox_max - bbox_min) in float64 like the reference) or
 * already normalised (1).  Any of raw [P,4] (rgb logits ++ sdf), geo [P,15], feat [P,32]
 * (hash features, query_sdf(embed=True)) may be NULL. */
int xrd_coslam_query(const XrdHashGrid* grid, const XrdCoslamMlp* mlp, const float* pts,
                     int n_points, int normalised, float* raw, float* geo, float* feat,
                     void* stream);

/* Hash-grid encoding only (used by the mesher path query_sdf(embed=True) and
 * by the index-parity tests): x DEVICE [P,3] normalised coords ->
 * feat [P,2*n_levels]; idx (optional) [P,n_levels,8] uint32 entry indices. */
int xrd_hashgrid_encode(const XrdHashGrid* grid, const float* x, int n_points,
                        float* feat, uint32_t* idx, void* stream);

/* ---- NICE-SLAM -------------------------------------------------------------
 *
 *   xrd_nice_step   slam/models/conv_onet.py:132-143 get_outputs -> render_batch_ray
 *                   :377-524 (bbox far plane, 32 uniform + 16 surface samples in float64,
 *                   sort), eval_points :339-375, NICE.forward
 *                   slam/model_components/decoder_nice.py:386-414 with the three MLP
 *                   decoders :207-234 (F.grid_sample trilerp :195-205, Gaussian Fourier
 *                   embedding :11-38), raw2outputs_nerf_color
 *                   slam/model_components/utils.py:189-244, get_loss_dict
 *                   conv_onet.py:145-185 (incl. the batch-global median of the tracking
 *                   mask) and autograd's backward.
 *
 * Feature grids are CHANNEL-LAST fp32 [Z][Y][X][32] (the reference holds [1,32,Z,Y,X];
 * one voxel = one 128-byte line here).  Decoder weights keep torch's [out,in] layout. */

typedef struct {
  const float* B;        /* [3][93]   Gaussian Fourier matrix (embedder._B)      */
  const float* pts_w[5]; /* [32][in]  in = 93, 32, 32, 125 (cat[embed, h]), 32     */
  const float* pts_b[5]; /* [32]                                                   */
  const float* fcc_w[5]; /* [32][c_dim]                                            */
  const float* fcc_b[5]; /* [32]                                                   */
  const float* out_w;    /* [n_out][32]                                            */
  const float* out_b;    /* [n_out]                                                */
  int c_dim;             /* 32 (middle, color) or 64 (fine: own grid ++ middle)    */
  int n_out;             /* 1 (occupancy) or 4 (colour decoder)                    */
} XrdNiceDecoder;

typedef struct {          /* same shapes as XrdNiceDecoder, ACCUMULATED into       */
  float* B;
  float* pts_w[5];
  float* pts_b[5];
  float* fcc_w[5];
  float* fcc_b[5];
  float* out_w;
  float* out_b;
} XrdNiceDecoderGrads;

typedef struct {
  const float* data; /* DEVICE [Z][Y][X][32] */
  int nx, ny, nz;
} XrdNiceGrid;

typedef enum { XRD_NICE_MIDDLE = 0, XRD_NICE_FINE = 1, XRD_NICE_COLOR = 2 } XrdNiceStage;

typedef struct {
  int stage;              /* XrdNiceStage                                          */
  int is_mapping;         /* loss form (conv_onet.py:160-185)                      */
  int n_samples;          /* 32 uniform                                            */
  int n_surface;          /* 16 near the surface                                   */
  double bound_min[3];    /* scene bound AFTER load_bound (float64)                */
  double bound_max[3];
  float w_color;          /* tracking 0.5 / mapping 0.2                            */
  int handle_dynamic;     /* tracking: 10 x median mask                            */
  int use_color_in_tracking;
  const float* t_uniform; /* DEVICE [n_samples] torch.linspace(0,1,n_samples)       */
  const float* t_surface; /* DEVICE [n_surface] torch.linspace(0,1,n_surface)       */
  const float* max_depth_global; /* DEVICE scalar: max(target_d) over the all-rank batch
                           * under data-parallel mapping (far clamp and zero-depth
                           * sampling are batch-global, SURVEY Q9); NULL -> computed
                           * from this call's rays                                  */
} XrdNiceCfg;

typedef struct {
  float* rgb;         /* [R,3]                                                     */
  double* depth;      /* [R]   float64 like the reference                          */
  double* uncertainty;/* [R]                                                       */
  double* z_vals;     /* [R,S] optional                                            */
  float* raw;         /* [R,S,4] optional (rgb, occupancy logit)                   */
  float* losses;      /* [2] depth_loss, rgb_loss (rgb 0 when the stage has none)  */
} XrdNiceOut;

typedef struct {
  float* d_grid[3];            /* middle, fine, color: [Z][Y][X][32], ACCUMULATED;
                                * NULL entries are skipped                         */
  XrdNiceDecoderGrads* d_color;/* colour-decoder gradients or NULL (frozen)         */
  float* d_rays_o;             /* [R,3] or NULL                                     */
  float* d_rays_d;             /* [R,3] or NULL                                     */
} XrdNiceGrads;

size_t xrd_nice_workspace_bytes(int n_rays, int n_samples_total, int with_grads);

/* decoders[3] = middle, fine, color; grids[3] = middle, fine, color. */
int xrd_nice_step(const XrdRays* rays, const XrdNiceGrid grids[3],
                  const XrdNiceDecoder decoders[3], const XrdNiceCfg* cfg,
                  XrdNiceOut* out, XrdNiceGrads* grads, void* workspace,
                  size_t workspace_bytes, void* stream);

/* Mesher queries (slam/models/conv_onet.py:213-240 query_fn = NICE.forward(stage 'fine'),
 * color_func = stage 'color'; slam/common/mesher.py:138-167): raw [P,4] = (rgb or 0, occupancy
 * logit middle [+ fine]) at free points DEVICE [P,3] fp32; no out-of-bound masking (the mesher
 * applies its own). */
size_t xrd_nice_query_workspace_bytes(int n_points);
int xrd_nice_query(const float* points, int n_points, const XrdNiceGrid grids[3],
                   const XrdNiceDecoder decoders[3], const double bound_min[3],
                   const double bound_max[3], int stage, float* raw, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Stage 'coarse' (slam/models/conv_onet.py:137-138 target_d = None, :397-402 near = 0.01 /
 * far = bound exit, 32 uniform samples; slam/model_components/decoder_nice.py:237-320
 * MLP_no_xyz, :389-393): its own decoder and grid; the grid is sampled with the scene bound
 * multiplied by model_coarse_bound_enlarge (conv_onet.py:335-337) while the out-of-bound mask
 * and the far plane use the scene bound.  Mapping depth loss only (conv_onet.py:176-181);
 * the decoder is frozen, gradients go to the grid (ACCUMULATED into d_grid) and the rays. */
typedef struct {
  const float* pts_w[5]; /* DEVICE [32,32] x3, [32,64] (input = [feature, hidden]), [32,32] */
  const float* pts_b[5]; /* DEVICE [32]                                                    */
  const float* out_w;    /* DEVICE [1,32]                                                  */
  const float* out_b;    /* DEVICE [1]                                                     */
} XrdNiceCoarseDecoder;

typedef struct {
  int n_samples;               /* 32                                                      */
  double bound_min[3];         /* scene bound after load_bound                            */
  double bound_max[3];
  double coarse_bound_min[3];  /* scene bound * model_coarse_bound_enlarge                */
  double coarse_bound_max[3];
  const float* t_uniform;      /* DEVICE [n_samples] torch.linspace(0,1,n_samples)        */
} XrdNiceCoarseCfg;

size_t xrd_nice_coarse_workspace_bytes(int n_rays, int n_samples, int with_grads);
/* out->losses[0] = depth loss (losses[1] = 0).  with_grads = 0: forward only. */
int xrd_nice_coarse_step(const XrdRays* rays, const XrdNiceGrid* grid,
                         const XrdNiceCoarseDecoder* dec, const XrdNiceCoarseCfg* cfg,
                         XrdNiceOut* out, float* d_grid, float* d_rays_o, float* d_rays_d,
                         int with_grads, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Vox-Fusion -------------------------------------------------------------
 *
 * Map structure (host side, once per mapping call -- SURVEY row f2):
 *   xrd_octree_*   third_party/sparse_octree: Octree::init/insert
 *                  (src/octree.cpp:35-115), get_centres_and_children (:297-346); node ids
 *                  (= embedding rows, SURVEY Q4) follow the reference's creation order.
 * The octree handle is a host object that owns its memory (like svo.Octree). */
typedef struct XrdOctree XrdOctree;
XrdOctree* xrd_octree_create(int grid_dim); /* 256; NULL on failure                 */
void xrd_octree_destroy(XrdOctree* t);
int xrd_octree_num_nodes(const XrdOctree* t);
/* voxels: HOST int32 [n][3] voxel coordinates (floor(p / voxel_size)); returns the node
 * count after the insertion (negative XrdStatus on error). */
int xrd_octree_insert(XrdOctree* t, const int32_t* voxels, int n);
/* HOST outputs sized by xrd_octree_num_nodes: voxels f32 [N][4], children f32 [N][8],
 * features i32 [N][8].  Returns N. */
int xrd_octree_export(const XrdOctree* t, float* voxels, float* children, int32_t* features);

/* Per-iteration path:
 *   xrd_voxfusion_march   slam/model_components/voxel_helpers_voxfusion.py:647-687 ray_intersect
 *                         (third_party/sparse_voxels/src/intersect_gpu.cu:191-270
 *                         svo_intersect_point_kernel + the host-side fill/sort/trim) and
 *                         :690-714 ray_sample (src/sample_gpu.cu:133-239
 *                         inverse_cdf_sampling_kernel incl. its batching quirks).
 *   xrd_voxfusion_render  slam/models/sparse_voxel.py:152-274 render_rays after sampling:
 *                         get_features (voxel_helpers_voxfusion.py:106-123,147-153), Decoder
 *                         (slam/model_components/decoder_voxfusion.py:122-149), sdf2weights
 *                         (:276-304), get_loss_dict (:103-143, utils.py:154-186) + backward.
 * The two calls are separated by ONE host read of `XrdVoxMarch.stats` (the reference syncs at
 * the same place: `hits.sum() == 0` -> None, sparse_voxel.py:179-181): the render workspace is
 * sized by the number of valid sample points. */
typedef struct {
  int n_nodes;
  const float* centres;      /* DEVICE [N][3]  (xyz + side/2) * voxel_size               */
  const int32_t* children;   /* DEVICE [N][9]  8 child ids (-1: none) ++ side            */
  const int32_t* vertex_idx; /* DEVICE [N][8]  corner-leaf ids = embedding rows          */
  const float* embeddings;   /* DEVICE [n_embeddings][16]                                */
  int n_embeddings;
} XrdVoxMap;

typedef struct {
  float voxel_size;   /* 0.2                                                              */
  float step_size;    /* voxel_size * 0.05 = 0.01 m                                       */
  int max_hits;       /* 50 (ray_intersect's max_hits_temp)                               */
  float max_distance; /* 10                                                               */
  int max_samples;    /* capacity per ray of the sample arrays (>= batch max + hits)      */
  int rays_per_block; /* inverse_cdf batching: K = ceil(R' / 200) of the reference
                         wrapper (voxel_helpers_voxfusion.py:411-424); 0 = derive       */
  uint64_t seed;      /* Philox when noise == NULL                                        */
} XrdVoxMarchCfg;

typedef struct {
  /* sorted, trimmed intersections (DEVICE) */
  int32_t* hit_idx;   /* [R][max_hits]                                                    */
  float* hit_tmin;    /* [R][max_hits]                                                    */
  float* hit_tmax;    /* [R][max_hits]                                                    */
  /* samples (DEVICE) */
  int32_t* smp_idx;   /* [R][max_samples]  voxel id or -1                                 */
  float* smp_depth;   /* [R][max_samples]                                                 */
  float* smp_dist;    /* [R][max_samples]                                                 */
  int32_t* smp_count; /* [R]  valid samples of the ray                                    */
  int32_t* smp_base;  /* [R]  first slot of the ray in the compact point list            */
  uint8_t* ray_mask;  /* [R]  ray hit at least one voxel                                  */
  int32_t* stats;     /* DEVICE [8 + 2R]: 0 n_hit_rays, 1 n_points, 2 S_max (batch max
                         samples), 3 P_max (batch max hits), 4 overflow (samples dropped by
                         the cap); [8, 8+R) rank of each ray among the hit rays, [8+R, 8+2R)
                         rank -> ray                                                       */
} XrdVoxMarch;

/* noise: DEVICE [R][max_samples] uniform(0,1) (clamped to [0.001,0.999] inside) or NULL. */
int xrd_voxfusion_march(const XrdRays* rays, const XrdVoxMap* map, const XrdVoxMarchCfg* cfg,
                        const float* noise, XrdVoxMarch* out, void* stream);

/* Parity hooks: the raw kernels with the reference kernels' exact signatures of data.
 * intersect: unsorted DFS-order hits (idx -1 padded), as svo_intersect returns them.
 * sample: explicit probs / steps / noise, compact layout [R][H] -> [R][max_steps]. */
int xrd_voxfusion_intersect_raw(const XrdRays* rays, const XrdVoxMap* map, float voxel_size,
                                int n_max, int32_t* idx, float* tmin, float* tmax, void* stream);
int xrd_voxfusion_sample_raw(int n_rays, int max_hits, int max_steps, int rays_per_block,
                             const int32_t* pts_idx, const float* min_depth,
                             const float* max_depth, const float* noise, const float* probs,
                             const float* steps, int32_t* smp_idx, float* smp_depth,
                             float* smp_dist, void* stream);

typedef struct {            /* torch nn.Linear layouts [out][in] + bias, DEVICE            */
  const float *w0, *b0;     /* pts_linears.0   [128][16]                                   */
  const float *w1, *b1;     /* pts_linears.1   [128][128]                                  */
  const float *ws, *bs;     /* sdf_out         [129][128]  (sdf, feat128)                  */
  const float *wc0, *bc0;   /* color_out.0     [128][144]  in = feat128 ++ emb16           */
  const float *wc1, *bc1;   /* color_out.2     [3][128]                                    */
} XrdVoxDecoder;

typedef struct {            /* same shapes, ACCUMULATED into                               */
  float *w0, *b0, *w1, *b1, *ws, *bs, *wc0, *bc0, *wc1, *bc1;
} XrdVoxDecoderGrads;

typedef struct {
  float voxel_size;
  float trunc;        /* training_trunc * sc_factor (0.05)                                */
  float max_depth;    /* loss: valid depth in (0.01, max_dpeth)                           */
  float pad_depth;    /* MAX_DEPTH = 10 that pads z_vals (voxel_helpers_voxfusion.py:11)   */
  float w_rgb, w_depth, w_sdf, w_fs; /* .5, 1, 5000, 10                                   */
  int n_points;       /* host copy of stats[1]                                            */
  int s_max;          /* host copy of stats[2]                                            */
  int n_hit_rays;     /* host copy of stats[0]                                            */
} XrdVoxRenderCfg;

typedef struct {
  float* rgb;     /* [R,3]  0 for rays without a hit                                      */
  float* depth;   /* [R]                                                                   */
  float* losses;  /* [4] rgb, depth, sdf, fs (weighted)                                    */
} XrdVoxOut;

typedef struct {
  float* d_embeddings;          /* [n_embeddings][16], ACCUMULATED                        */
  XrdVoxDecoderGrads* d_decoder;/* or NULL                                                */
  float* d_rays_o;              /* [R,3] or NULL                                          */
  float* d_rays_d;              /* [R,3] or NULL                                          */
} XrdVoxGrads;

size_t xrd_voxfusion_render_workspace_bytes(int n_rays, int n_points, int with_grads);

/* Point query of the mesher path (slam/model_components/voxel_helpers_voxfusion.py:15-95
 * get_scores / eval_points): trilinear embedding of the voxel's 8 vertex embeddings
 * (get_features :106-153) and the decoder forward (decoder_voxfusion.py:122-140 get_values) at
 * DEVICE points [P,3] fp32, each with its voxel id (DEVICE [P] int32, a row of map->centres /
 * map->vertex_idx).  raw: DEVICE [P,4] = (rgb after the colour head's sigmoid, sdf).  The
 * workspace is forward-only. */
size_t xrd_voxfusion_query_workspace_bytes(int n_points);
int xrd_voxfusion_query(const XrdVoxMap* map, const XrdVoxDecoder* dec, float voxel_size,
                        const float* points, const int32_t* voxel_ids, int n_points, float* raw,
                        void* workspace, size_t workspace_bytes, void* stream);

int xrd_voxfusion_render(const XrdRays* rays, const XrdVoxMap* map, const XrdVoxMarch* march,
                         const XrdVoxMarchCfg* mcfg, const XrdVoxDecoder* dec,
                         const XrdVoxRenderCfg* cfg, XrdVoxOut* out, XrdVoxGrads* grads,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- Marching cubes -----------------------------------------------------------
 *
 *   xrd_mc_count / xrd_mc_emit  the isosurface step of the mesher: skimage.measure.marching_cubes
 *                               on the host in slam/common/mesher.py:203-233 (one 256^3 volume)
 *                               and slam/algorithms/voxfusion.py:253-279 (one call per voxel).
 * A batch of B fp32 volumes [B][nx][ny][nz] (x slowest).  A corner is inside when value < level;
 * a lattice edge whose ends lie on opposite sides gets one vertex (welded inside a volume, never
 * across volumes) at
 *   t = (level - v0) / (v1 - v0)                        fp32, v0 = lower-index end
 *   world_d = origin_d + (i_d + t * e_d) * spacing_d    fp64, stored as fp32.
 * Vertices are ordered by (volume, i, j, k, axis), faces by (volume, cube, table order); the
 * output is bit-identical run to run.  Winding: the right-hand normal of every triangle points
 * toward increasing field values.  Case tables and the ambiguous-face rule:
 * scripts/gen_mc_tables.py.
 *
 * xrd_mc_count writes (V, F) to DEVICE counts[2]; the caller reads them, allocates
 * verts [V,3] fp32 and faces [F,3] int32 and calls xrd_mc_emit with the same volumes, level and
 * the UNTOUCHED workspace (it holds the scans between the two calls). */
typedef struct {
  const float* field;      /* DEVICE [n_volumes][nx][ny][nz]                                   */
  int n_volumes, nx, ny, nz; /* nx, ny, nz >= 2                                               */
  double origin[3];        /* world position of lattice point (0,0,0), shared by all volumes   */
  double spacing[3];       /* lattice step per axis, shared                                    */
  const double* origins;   /* DEVICE [n_volumes][3] per-volume origin, or NULL: origin[]       */
  const double* spacings;  /* DEVICE [n_volumes][3] per-volume spacing, or NULL: spacing[]     */
} XrdMcVolumes;

size_t xrd_mc_workspace_bytes(int n_volumes, int nx, int ny, int nz);
int xrd_mc_count(const XrdMcVolumes* v, float level, int* counts, void* workspace,
                 size_t workspace_bytes, void* stream);
/* verts or faces may be NULL (skipped). */
int xrd_mc_emit(const XrdMcVolumes* v, float level, float* verts, int32_t* faces, void* workspace,
                size_t workspace_bytes, void* stream);

/* ---- Point-SLAM -------------------------------------------------------------
 *
 *   xrd_pointslam_knn_query  slam/model_components/neural_point_cloud.py:223-282
 *                            find_neighbors_faiss.  The reference's index is faiss-gpu
 *                            IndexIVFFlat(nlist 400, nprobe 4) -- approximate, un-vendored;
 *                            this is an EXACT radius-limited 8-NN (ties by lower id) over a
 *                            uniform hash grid, with faiss's sentinels (id -1, D = FLT_MAX).
 *   xrd_pointslam_step       slam/models/conv_onet_pointslam.py:311-461 render_batch_ray
 *                            (5 surface samples), :248-309 eval_points, POINT.forward
 *                            slam/model_components/decoder_pointslam.py:595-655 stage
 *                            'geometry' (MLP_geometry :162-273: inverse-distance kNN feature
 *                            interpolation + 5x32 Fourier MLP) and stage 'color' (adds
 *                            MLP_color :408-542 with the per-neighbour MLP_col_neighbor
 *                            :276-292), raw2outputs_nerf_color2
 *                            slam/model_components/utils.py:247-295, get_loss_dict
 *                            conv_onet_pointslam.py:144-195 and autograd's backward.
 */
typedef struct {
  const float* pos;           /* DEVICE [N][3] neural point positions                      */
  int n_points;
  float cell;                 /* grid cell edge (>= the largest query radius / 2)          */
  int table_size;             /* power of two                                              */
  const int32_t* cell_start;  /* DEVICE [table_size] first slot of the bucket              */
  const int32_t* cell_end;    /* DEVICE [table_size] one past the last slot                */
  const int32_t* sorted_ids;  /* DEVICE [N] point ids ordered by bucket                    */
} XrdPointIndex;

/* bucket of cell (ix,iy,iz): ((ix*73856093) ^ (iy*19349663) ^ (iz*83492791)) & (table-1),
 * uint32 arithmetic, ix = floor(x * (1/cell)).
 * xrd_pointslam_knn_build fills cell_start / cell_end [table_size] and sorted_ids [n_points]
 * (ids ascending inside a bucket) for DEVICE positions [n_points,3] -- what faiss's
 * index.add() does in the reference (slam/model_components/neural_point_cloud.py:48-52,
 * 173-176), on the device with no host round trip. */
size_t xrd_pointslam_knn_build_workspace_bytes(int table_size);
int xrd_pointslam_knn_build(const float* pos, int n_points, float cell, int table_size,
                            int32_t* cell_start, int32_t* cell_end, int32_t* sorted_ids,
                            void* workspace, size_t workspace_bytes, void* stream);
int xrd_pointslam_knn_query(const XrdPointIndex* index, const float* queries, const float* radius,
                            int radius_stride, int n_queries, float* D, int32_t* I,
                            int32_t* neighbor_num, void* stream);

typedef struct {
  int stage;               /* 0 = 'geometry', 1 = 'color'                                   */
  int is_mapping;
  int n_surface;           /* 5                                                             */
  float near_end_surface;  /* 0.98                                                          */
  float far_end_surface;   /* 1.02                                                          */
  float near_end;          /* 0.3                                                           */
  float sigmoid_coef;      /* 0.1                                                           */
  int min_nn_num;          /* 2                                                             */
  float w_color;
  int handle_dynamic;
  int use_color_in_tracking;
  const float* t_surface;  /* DEVICE [n_surface] torch.linspace(0,1,n)                      */
  const float* far;        /* DEVICE scalar min(5*mean(d), max(1.2*d)) (batch-global, Q9)   */
  const float* radius_query; /* DEVICE [R] per-ray dynamic query radius                     */
  const float* rand_feat;  /* DEVICE [32] feature of samples with < min_nn neighbours (Q6)
                              or NULL = zeros                                               */
  const float* rand_feat_color; /* the colour decoder's own draw (decoder_pointslam.py:463) */
} XrdPointCfg;

typedef struct {
  const float* geo_feats;      /* DEVICE [N][32]                                            */
  const uint8_t* frustum_mask; /* DEVICE [N] or NULL (multiplies geo_feats only, row P9)     */
  const float* col_feats;      /* DEVICE [N][32]; stage colour only                         */
} XrdPointFeats;

/* Colour decoder (slam/model_components/decoder_pointslam.py:313-542 MLP_color + :276-292
 * MLP_col_neighbor), all row-major [out][in] like nn.Linear:
 *   per neighbour k: f_k = nb_w2 . softplus100(nb_w1 . [sin, cos(2 pi (x_k - p) B_rel), col_feat_k]) ; c = sum_k w_k f_k
 *   h = softplus100(w[i] . h + b[i]) + (wc[i] . c + bc[i]),  i = 0..4, input cat after i = 2
 *   rgb = sigmoid(wo . h + bo);  first input = [sin, cos](2 pi p B). */
typedef struct {
  const float* B;      /* [3][20] fixed (GaussianFourierFeatureTransform, not learnable)   */
  const float* B_rel;  /* [3][10] learnable                                                */
  const float* nb_w1; const float* nb_b1; /* [128][52], [128]                              */
  const float* nb_w2; const float* nb_b2; /* [32][128], [32]                               */
  const float* w[5];  const float* b[5];  /* [128][40|128|128|168|128], [128]              */
  const float* wc[5]; const float* bc[5]; /* fc_c: [128][32], [128]                        */
  const float* wo;    const float* bo;    /* [3][128], [3]                                 */
} XrdPointColorDecoder;

/* Same shapes; every non-NULL array is ACCUMULATED into. */
typedef struct {
  float* B_rel;
  float* nb_w1; float* nb_b1; float* nb_w2; float* nb_b2;
  float* w[5]; float* b[5]; float* wc[5]; float* bc[5];
  float* wo; float* bo;
} XrdPointColorDecoderGrads;

typedef struct {
  float* rgb;              /* [R,3] (zeros in stage geometry)                               */
  float* depth;            /* [R]                                                           */
  float* uncertainty;      /* [R]                                                           */
  uint8_t* valid_ray_mask; /* [R]                                                           */
  float* z_vals;           /* [R,n_surface] optional                                        */
  float* losses;           /* [2] geo_loss, rgb_loss (already weighted)                     */
} XrdPointOut;

typedef struct {
  float* d_geo_feats;      /* [N][32] ACCUMULATED                                           */
  float* d_rays_o;         /* [R,3] or NULL                                                 */
  float* d_rays_d;
  float* d_col_feats;      /* [N][32] ACCUMULATED; stage colour, or NULL                    */
  XrdPointColorDecoderGrads* color; /* colour-decoder gradients or NULL (decoder fixed)     */
} XrdPointGrads;

/* Measurement / parity hook: arithmetic of the wide-MLP GEMMs (Point-SLAM colour stage and
 * the Vox-Fusion decoder):
 * 0 = fp32 SIMT, 1 = 3xTF32 tensor cores (default, fp32-level accuracy): tcgen05 / TMEM / TMA
 * kernel where the shape qualifies, mma.sync otherwise, 2 = plain TF32 (mma.sync),
 * 3 = 3xTF32 on mma.sync only.  Thread-local, like the error state. */
int xrd_debug_gemm_mode(int mode);
/* bring-up hook of the tcgen05 GEMM (descriptor field variants); 0 = production */
int xrd_debug_gemm_variant(int variant);

/* The wide-MLP GEMM itself (unit tests): C[m][n] = act(sum_k A(m,k) B[k][n] + bias[m]) with
 * A(m,k) = transA ? A[k*lda+m] : A[m*lda+k]; act 0 none, 1 relu, 2 softplus(beta 100),
 * 3 sigmoid; result zeroed where relu_mask[m][n] <= 0; + addend[m][n].  DEVICE pointers. */
int xrd_debug_gemm(int M, int N, int K, const float* A, int lda, int transA, const float* B,
                   int ldb, float* C, int ldc, const float* bias, int act,
                   const float* relu_mask, int ldmask, const float* addend, int ldadd,
                   void* stream);

/* ... plus act_out[m][n] (the masked activation before the addend) and accumulate (C += ). */
int xrd_debug_gemm_ex(int M, int N, int K, const float* A, int lda, int transA, const float* B,
                      int ldb, float* C, int ldc, const float* bias, int act,
                      const float* relu_mask, int ldmask, const float* addend, int ldadd,
                      float* act_out, int ldact, int accumulate, void* stream);

/* The weight-gradient kernel of the per-point MLPs (unit tests): out[j][i] += sum_p B[j][p] A[i][p]
 * over P points (rows of Pp floats), B[j][p] dropped where bit (j & 31) of mask[j / 32][p] is
 * clear (mask may be NULL), bias[j] += sum_p B[j][p] (bias may be NULL).  DEVICE pointers. */
int xrd_debug_dw(int nA, int nB, int P, int Pp, const float* A, const float* B,
                 const uint32_t* mask, float* out, float* bias, void* stream);

size_t xrd_pointslam_workspace_bytes(int n_rays, int n_surface, int stage, int with_grads);

int xrd_pointslam_step(const XrdRays* rays, const XrdPointIndex* index,
                       const XrdPointFeats* feats, const XrdNiceDecoder* geo_decoder,
                       const XrdPointColorDecoder* color_decoder /* NULL in stage geometry */,
                       const XrdPointCfg* cfg, XrdPointOut* out, XrdPointGrads* grads,
                       void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XRDSLAM_B200_H_ */
