// Vox-Fusion render-and-optimise step (sm_100a): in-kernel octree traversal, inverse-CDF
// sampling, embedding trilerp, width-128 decoder, SDF compositing, losses and backward.
//
// Replaces (reference @ f0366f20):
//   third_party/sparse_voxels/src/intersect_gpu.cu:75-140,191-270  RayAABBIntersection,
//       svo_intersect_point_kernel (+ slam/model_components/voxel_helpers_voxfusion.py:233-278,
//       647-687: G-fold tree replication, host-side fill / sort / trim)
//   third_party/sparse_voxels/src/sample_gpu.cu:133-239 inverse_cdf_sampling_kernel
//       (+ voxel_helpers_voxfusion.py:399-481,690-714), including its batching quirks
//   slam/models/sparse_voxel.py:152-304 render_rays / sdf2weights, :103-143 get_loss_dict,
//   voxel_helpers_voxfusion.py:97-166 get_features / trilinear_interp,
//   slam/model_components/decoder_voxfusion.py:122-149 Decoder.get_values, and autograd.
#include <math.h>

#include "common.cuh"
#include "dw.cuh"
#include "gemm_t5.cuh"

namespace xrd {
namespace vox {

constexpr int EMB = 16;
constexpr int W = 128;
constexpr int T = 128;  // threads per CTA of the per-point kernels

// ------------------------------------------------------------ intersect ---
__device__ __forceinline__ float2 ray_aabb(const float o[3], const float d[3], const float c[3],
                                           float half_voxel) {
  // third_party/sparse_voxels/src/intersect_gpu.cu:75-140 (same operations, same order)
  float f_low = 0.f, f_high = 100000.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float inv = __fdividef(1.0f, d[k]);
    float lo = (c[k] - half_voxel - o[k]) * inv;
    float hi = (c[k] + half_voxel - o[k]) * inv;
    if (hi < lo) { const float t = lo; lo = hi; hi = t; }
    if (hi < f_low) return make_float2(-1.0f, -1.0f);
    if (lo > f_high) return make_float2(-1.0f, -1.0f);
    f_low = (lo > f_low) ? lo : f_low;
    f_high = (hi < f_high) ? hi : f_high;
    if (f_low > f_high) return make_float2(-1.0f, -1.0f);
  }
  return make_float2(f_low, f_high);
}

// depth-first traversal from the root (node 0); leaf hits in visiting order, at most n_max
__device__ __forceinline__ int traverse(const float* __restrict__ centres,
                                        const int* __restrict__ children, float voxel_size,
                                        const float o[3], const float d[3], int n_max,
                                        int* hit_idx, float* hit_lo, float* hit_hi) {
  const float half_voxel = voxel_size * 0.5f;
  int stack[256];
  int ptr = 0, cnt = 0;
  stack[0] = 0;
  while (ptr > -1 && cnt < n_max) {
    const int k = stack[ptr];
    const float c[3] = {centres[k * 3], centres[k * 3 + 1], centres[k * 3 + 2]};
    const int side = children[k * 9 + 8];
    const float2 t = ray_aabb(o, d, c, half_voxel * (float)side);
    --ptr;
    if (t.x > -1.0f) {
      if (side == 1) {
        hit_idx[cnt] = k; hit_lo[cnt] = t.x; hit_hi[cnt] = t.y;
        ++cnt;
        continue;
      }
      for (int u = 0; u < 8; ++u) {
        const int ch = children[k * 9 + u];
        if (ch > -1 && ptr < 255) stack[++ptr] = ch;
      }
    }
  }
  return cnt;
}

__global__ void __launch_bounds__(128) k_intersect_raw(int R, const float* rays_o,
                                                       const float* rays_d, const float* centres,
                                                       const int* children, float voxel_size,
                                                       int n_max, int* idx, float* tmin,
                                                       float* tmax) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const float o[3] = {rays_o[r * 3], rays_o[r * 3 + 1], rays_o[r * 3 + 2]};
  const float d[3] = {rays_d[r * 3], rays_d[r * 3 + 1], rays_d[r * 3 + 2]};
  int hi[64]; float lo_[64], hi_[64];
  const int nm = min(n_max, 64);
  const int cnt = traverse(centres, children, voxel_size, o, d, nm, hi, lo_, hi_);
  for (int l = 0; l < n_max; ++l) {
    idx[(size_t)r * n_max + l] = l < cnt ? hi[l] : -1;
    tmin[(size_t)r * n_max + l] = l < cnt ? lo_[l] : 0.f;
    tmax[(size_t)r * n_max + l] = l < cnt ? hi_[l] : 0.f;
  }
}

struct MarchParams {
  int R;
  const float *rays_o, *rays_d, *centres;
  const int* children;
  float voxel_size, step_size, max_distance;
  int max_hits, scap, rays_per_block;
  const float* noise;
  uint64_t seed;
  int *hit_idx; float *hit_tmin, *hit_tmax;
  int *smp_idx; float *smp_depth, *smp_dist;
  int *smp_count, *smp_base;
  unsigned char* ray_mask;
  int* stats;
  int* rank;      // [R] rank of the ray among hit rays
  int* rank2ray;  // [R]
};

// traversal + the host-side post-processing of ray_intersect (fill, sort by t_min, trim)
__global__ void __launch_bounds__(128) k_march_intersect(const MarchParams P) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.R) return;
  const float o[3] = {P.rays_o[r * 3], P.rays_o[r * 3 + 1], P.rays_o[r * 3 + 2]};
  const float d[3] = {P.rays_d[r * 3], P.rays_d[r * 3 + 1], P.rays_d[r * 3 + 2]};
  int id[64]; float lo[64], hi[64];
  const int nm = min(P.max_hits, 64);
  const int cnt = traverse(P.centres, P.children, P.voxel_size, o, d, nm, id, lo, hi);
  // insertion sort by t_min (fillers carry max_distance and stay behind)
  for (int a = 1; a < cnt; ++a) {
    const int ki = id[a]; const float kl = lo[a], kh = hi[a];
    int b = a - 1;
    while (b >= 0 && lo[b] > kl) { id[b + 1] = id[b]; lo[b + 1] = lo[b]; hi[b + 1] = hi[b]; --b; }
    id[b + 1] = ki; lo[b + 1] = kl; hi[b + 1] = kh;
  }
  int n = 0;
  for (int a = 0; a < nm; ++a) {
    const bool ok = a < cnt && !(lo[a] > P.max_distance);  // pts_idx[min_depth > max_distance] = -1
    const size_t q = (size_t)r * P.max_hits + a;
    P.hit_idx[q] = ok ? id[a] : -1;
    P.hit_tmin[q] = ok ? lo[a] : P.max_distance;
    P.hit_tmax[q] = ok ? hi[a] : P.max_distance;
    n += ok;
  }
  P.ray_mask[r] = n > 0;
  if (n > 0) atomicMax(&P.stats[3], n);
}

// rank of every hit ray among the hit rays (the reference compacts rays with ray_mask)
__global__ void __launch_bounds__(1024) k_rank(const MarchParams P) {
  __shared__ int s_part[32];
  __shared__ int s_run;
  if (threadIdx.x == 0) s_run = 0;
  __syncthreads();
  for (int base = 0; base < P.R; base += blockDim.x) {
    const int r = base + threadIdx.x;
    const int f = (r < P.R) ? (int)P.ray_mask[r] : 0;
    int inc = f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, inc, o);
      if ((threadIdx.x & 31) >= o) inc += v;
    }
    if ((threadIdx.x & 31) == 31) s_part[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      int v = threadIdx.x < (blockDim.x >> 5) ? s_part[threadIdx.x] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, o);
        if (threadIdx.x >= o) v += u;
      }
      s_part[threadIdx.x] = v;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int excl = s_run + (warp ? s_part[warp - 1] : 0) + inc - f;
    if (r < P.R) {
      P.rank[r] = f ? excl : -1;
      if (f) P.rank2ray[excl] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_run += s_part[(blockDim.x >> 5) - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) P.stats[0] = s_run;
}

// third_party/sparse_voxels/src/sample_gpu.cu:133-239, one ray.  `row0_idx` is the hit list of
// the first ray of this ray's block in the reference's [G=200, K] batching (quirk: the tail
// loop reads pts_idx[curr_bin] without the ray offset), `j` the ray's index inside its block
// and `K` the rays per block (quirk: the tail loop runs only while K > j*max_hits + curr_bin).
__device__ __forceinline__ int inverse_cdf_ray(const int* pts_idx, const float* min_depth,
                                               const float* max_depth, const float* probs,
                                               float steps, const float* noise,
                                               uint64_t seed, uint64_t noise_base, int max_hits,
                                               int max_steps, int j, int K, const int* row0_idx,
                                               int* s_idx, float* s_depth, float* s_dist,
                                               int* overflow) {
  const int H = j * max_hits;
  int curr_bin = 0, s = 0;
  float curr_min_depth = min_depth[0], curr_max_depth = max_depth[0];
  float curr_min_cdf = 0.f, curr_max_cdf = probs[0];
  const float step_size = (float)(1.0 / (double)steps);
  float z_low = curr_min_depth;
  const int total_steps = (int)ceilf(steps);
  bool done = false;
  auto put = [&](int id, float dist, float depth) {
    if (s < max_steps) { s_idx[s] = id; s_dist[s] = dist; s_depth[s] = depth; }
    else if (overflow) atomicAdd(overflow, 1);
    ++s;
  };
  for (int curr_step = 0; curr_step < total_steps; ++curr_step) {
    float u01;
    if (noise) u01 = noise[curr_step < max_steps ? curr_step : max_steps - 1];
    else { float q[4]; philox4(seed, noise_base + curr_step, q); u01 = q[0]; }
    u01 = fminf(fmaxf(u01, 0.001f), 0.999f);
    const float curr_cdf = ((float)curr_step + u01) * step_size;
    while (curr_cdf > curr_max_cdf) {
      put(pts_idx[curr_bin], curr_max_depth - z_low, (float)((double)(curr_max_depth + z_low) * .5));
      ++curr_bin;
      if (curr_bin >= max_hits || pts_idx[curr_bin] == -1) { done = true; break; }
      curr_min_depth = min_depth[curr_bin];
      curr_max_depth = max_depth[curr_bin];
      curr_min_cdf = curr_max_cdf;
      curr_max_cdf = curr_max_cdf + probs[curr_bin];
      z_low = curr_min_depth;
    }
    if (done) break;
    const float u = (curr_cdf - curr_min_cdf) / (curr_max_cdf - curr_min_cdf);
    const float z = curr_min_depth + u * (curr_max_depth - curr_min_depth);
    put(pts_idx[curr_bin], z - z_low, (float)((double)(z + z_low) * .5));
    z_low = z;
  }
  // "if there are bins still remained": `~done` is always true; K > H + curr_bin binds
  while ((z_low < curr_max_depth) && (K > (H + curr_bin))) {
    put(pts_idx[curr_bin], curr_max_depth - z_low, (float)((double)(curr_max_depth + z_low) * .5));
    ++curr_bin;
    if (curr_bin >= max_hits || row0_idx[curr_bin] == -1) break;
    curr_min_depth = min_depth[curr_bin];
    curr_max_depth = max_depth[curr_bin];
    z_low = curr_min_depth;
  }
  return s;
}

__global__ void __launch_bounds__(128) k_sample_raw(int R, int max_hits, int max_steps, int K,
                                                    const int* pts_idx, const float* min_depth,
                                                    const float* max_depth, const float* noise,
                                                    const float* probs, const float* steps,
                                                    int* s_idx, float* s_depth, float* s_dist) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const int j = r % K, r0 = r - j;
  for (int q = 0; q < max_steps; ++q) {
    s_idx[(size_t)r * max_steps + q] = -1;
    s_depth[(size_t)r * max_steps + q] = 0.f;
    s_dist[(size_t)r * max_steps + q] = 0.f;
  }
  inverse_cdf_ray(pts_idx + (size_t)r * max_hits, min_depth + (size_t)r * max_hits,
                  max_depth + (size_t)r * max_hits, probs + (size_t)r * max_hits, steps[r],
                  noise + (size_t)r * max_steps, 0, 0, max_hits, max_steps, j, K,
                  pts_idx + (size_t)r0 * max_hits, s_idx + (size_t)r * max_steps,
                  s_depth + (size_t)r * max_steps, s_dist + (size_t)r * max_steps, nullptr);
}

__global__ void __launch_bounds__(128) k_march_sample(const MarchParams P) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.R) return;
  const int mh = P.max_hits;
  int cnt = 0;
  if (P.ray_mask[r]) {
    const int Pm = P.stats[3];   // batch max hits = width of the reference's trimmed arrays
    const int Rh = P.stats[0];
    const int K = P.rays_per_block > 0 ? P.rays_per_block : (Rh + 199) / 200;
    const int n = P.rank[r], j = n % K;
    const int r0 = P.rank2ray[n - j];
    const int* id = P.hit_idx + (size_t)r * mh;
    const float* lo = P.hit_tmin + (size_t)r * mh;
    const float* hi = P.hit_tmax + (size_t)r * mh;
    // ray_sample: dists, probs = dists / sum, steps = sum / step_size (fp32)
    float probs[64];
    float sum = 0.f;
    for (int a = 0; a < Pm; ++a) { probs[a] = (id[a] != -1) ? hi[a] - lo[a] : 0.f; sum += probs[a]; }
    for (int a = 0; a < Pm; ++a) probs[a] = probs[a] / sum;
    const float steps = sum / P.step_size;
    cnt = inverse_cdf_ray(id, lo, hi, probs, steps,
                          P.noise ? P.noise + (size_t)r * P.scap : nullptr, P.seed,
                          (uint64_t)r * P.scap, Pm, P.scap, j, K, P.hit_idx + (size_t)r0 * mh,
                          P.smp_idx + (size_t)r * P.scap, P.smp_depth + (size_t)r * P.scap,
                          P.smp_dist + (size_t)r * P.scap, &P.stats[4]);
    cnt = min(cnt, P.scap);
    // the tail loop can append one entry of an exhausted hit list (idx -1): the reference masks
    // it afterwards (sampled_depth.masked_fill_(idx == -1, MAX_DEPTH), sample_mask = idx != -1)
    while (cnt > 0 && P.smp_idx[(size_t)r * P.scap + cnt - 1] == -1) {
      P.smp_depth[(size_t)r * P.scap + cnt - 1] = P.max_distance;
      P.smp_dist[(size_t)r * P.scap + cnt - 1] = 0.f;
      --cnt;
    }
    for (int q = 0; q < cnt; ++q)  // sampled_dists.clamp(min=0)
      P.smp_dist[(size_t)r * P.scap + q] = fmaxf(P.smp_dist[(size_t)r * P.scap + q], 0.f);
  }
  P.smp_count[r] = cnt;
  P.smp_base[r] = cnt ? atomicAdd(&P.stats[1], cnt) : 0;
  if (cnt) atomicMax(&P.stats[2], cnt);
}

// ----------------------------------------------------------- per point ---
struct PointParams {
  int P, Pp, R;
  const int *pt_ray, *pt_k;
  const float *rays_o, *rays_d;
  const float* smp_depth; const int* smp_idx; int scap;
  const float* centres; const int* vertex_idx; const float* emb;
  float voxel_size;
  XrdVoxDecoder dec;
  float* acts;        // rows of Pp: x16 | h1 128 | h2 128 | feat 128 | c1 128
  float* sdf; float* rgb;  // [P], [3][P]
  // backward
  const float* d_sdf; const float* d_rgb;  // [P], [3][P]
  float* grads;       // rows of Pp: do 4 | dprec1 128 | dso 129 (dsdf, dfeat) | dpre2 128 | dpre1 128
  float* d_emb;
  float* dp;          // [3][P]
  int need_dp;
  // query mode: sample points given directly (pt_ray / pt_k unused)
  const float* pts; const int* pts_vox;
};
// activation rows: h1 | h2 | feat | x   (feat and x adjacent: the colour net's 144-wide input
// cat[feat, x] is one GEMM operand) | c1
__host__ __device__ inline int ra_h1() { return 0; }
__host__ __device__ inline int ra_h2() { return W; }
__host__ __device__ inline int ra_feat() { return 2 * W; }
__host__ __device__ inline int ra_x() { return 3 * W; }
__host__ __device__ inline int ra_c1() { return 3 * W + EMB; }
__host__ __device__ inline int ra_rows() { return EMB + 4 * W; }
// gradient rows: do 4 | dc1 128 | dso 129 (dsdf, dfeat) | dxc 16 (right after dfeat: the
// 144-row output of wc0^T dc1) | d2 128 | d1 128 | dx 16
__host__ __device__ inline int rg_do() { return 0; }
__host__ __device__ inline int rg_dc1() { return 4; }
__host__ __device__ inline int rg_dso() { return 4 + W; }        // row 0 = dsdf, 1..128 = dfeat
__host__ __device__ inline int rg_dxc() { return 4 + W + 129; }
__host__ __device__ inline int rg_d2() { return 4 + W + 129 + EMB; }
__host__ __device__ inline int rg_d1() { return 4 + 2 * W + 129 + EMB; }
__host__ __device__ inline int rg_dx() { return 4 + 3 * W + 129 + EMB; }
__host__ __device__ inline int rg_rows() { return 4 + 3 * W + 129 + 2 * EMB; }

struct Corner {
  int vid[8];
  float w[8];
  float p[3];
};
// p = (xyz - centre) / voxel_size + 0.5 and the 8 trilinear weights of voxel `vox`
__device__ __forceinline__ void corners_at(const PointParams& P, const float xyz[3], int vox,
                                           Corner& c) {
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    c.p[d] = __fadd_rn(__fdiv_rn(__fsub_rn(xyz[d], P.centres[vox * 3 + d]), P.voxel_size), 0.5f);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    c.vid[i] = P.vertex_idx[vox * 8 + i];
    const int qx = i >> 2, qy = (i >> 1) & 1, qz = i & 1;  // offset_points: x slowest
    const float wx = qx ? c.p[0] : 1.f - c.p[0];
    const float wy = qy ? c.p[1] : 1.f - c.p[1];
    const float wz = qz ? c.p[2] : 1.f - c.p[2];
    c.w[i] = wx * wy * wz;
  }
}
__device__ __forceinline__ void corners(const PointParams& P, int r, int k, float xyz[3], Corner& c) {
  const float depth = P.smp_depth[(size_t)r * P.scap + k];
#pragma unroll
  for (int d = 0; d < 3; ++d)
    xyz[d] = __fadd_rn(P.rays_o[r * 3 + d], __fmul_rn(P.rays_d[r * 3 + d], depth));
  corners_at(P, xyz, P.smp_idx[(size_t)r * P.scap + k], c);
}

// ---- GEMM decoder path: gather / head / scatter kernels around gemm.cuh -------------------
// x = trilinear embedding of the sample point -> activation rows ra_x
__global__ void __launch_bounds__(T) k_vox_gather(const PointParams P) {
  const int p = blockIdx.x * T + threadIdx.x;
  if (p >= P.P) return;
  float xyz[3];
  Corner c;
  if (P.pts) {  // free query points (xrd_voxfusion_query)
#pragma unroll
    for (int d = 0; d < 3; ++d) xyz[d] = P.pts[(size_t)p * 3 + d];
    corners_at(P, xyz, P.pts_vox[p], c);
  } else {
    corners(P, P.pt_ray[p], P.pt_k[p], xyz, c);
  }
  float x[EMB];
#pragma unroll
  for (int q = 0; q < EMB; ++q) x[q] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4* e = reinterpret_cast<const float4*>(P.emb + (size_t)c.vid[i] * EMB);
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4) {
      const float4 v = __ldg(&e[q4]);
      x[4 * q4 + 0] = fmaf(c.w[i], v.x, x[4 * q4 + 0]);
      x[4 * q4 + 1] = fmaf(c.w[i], v.y, x[4 * q4 + 1]);
      x[4 * q4 + 2] = fmaf(c.w[i], v.z, x[4 * q4 + 2]);
      x[4 * q4 + 3] = fmaf(c.w[i], v.w, x[4 * q4 + 3]);
    }
  }
#pragma unroll
  for (int q = 0; q < EMB; ++q) P.acts[(size_t)(ra_x() + q) * P.Pp + p] = x[q];
}

// d(colour logits) = d_rgb * c (1 - c) -> rows rg_do (+ a zero 4th row); dsdf -> row rg_dso
__global__ void __launch_bounds__(256) k_vox_dout(const PointParams P) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P.P) return;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    const float c = P.rgb[(size_t)q * P.P + p];
    P.grads[(size_t)(rg_do() + q) * P.Pp + p] = P.d_rgb[(size_t)q * P.P + p] * c * (1.f - c);
  }
  P.grads[(size_t)(rg_do() + 3) * P.Pp + p] = 0.f;
  P.grads[(size_t)rg_dso() * P.Pp + p] = P.d_sdf[p];
}

// dx (rows rg_dx) -> embedding scatter + d loss / d xyz
__global__ void __launch_bounds__(T) k_vox_scatter(const PointParams P) {
  const int p = blockIdx.x * T + threadIdx.x;
  if (p >= P.P) return;
  float dx[EMB];
#pragma unroll
  for (int q = 0; q < EMB; ++q) dx[q] = P.grads[(size_t)(rg_dx() + q) * P.Pp + p];
  float xyz[3];
  Corner c;
  corners(P, P.pt_ray[p], P.pt_k[p], xyz, c);
  float gp[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const size_t off = (size_t)c.vid[i] * EMB;
    if (P.d_emb)
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4)
        red_add_v4(P.d_emb + off + 4 * q4, c.w[i] * dx[4 * q4], c.w[i] * dx[4 * q4 + 1],
                   c.w[i] * dx[4 * q4 + 2], c.w[i] * dx[4 * q4 + 3]);
    if (P.need_dp) {
      float s = 0.f;
      const float4* e = reinterpret_cast<const float4*>(P.emb + off);
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        const float4 v = __ldg(&e[q4]);
        s += v.x * dx[4 * q4] + v.y * dx[4 * q4 + 1] + v.z * dx[4 * q4 + 2] + v.w * dx[4 * q4 + 3];
      }
      const int qx = i >> 2, qy = (i >> 1) & 1, qz = i & 1;
      const float wx = qx ? c.p[0] : 1.f - c.p[0], wy = qy ? c.p[1] : 1.f - c.p[1],
                  wz = qz ? c.p[2] : 1.f - c.p[2];
      gp[0] += (qx ? 1.f : -1.f) * wy * wz * s;
      gp[1] += (qy ? 1.f : -1.f) * wx * wz * s;
      gp[2] += (qz ? 1.f : -1.f) * wx * wy * s;
    }
  }
  if (P.need_dp)
#pragma unroll
    for (int d = 0; d < 3; ++d) P.dp[(size_t)d * P.P + p] = gp[d] / P.voxel_size;
}

__global__ void __launch_bounds__(128) k_points(int R, const int* count, const int* base,
                                                int* pt_ray, int* pt_k) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const int c = count[r], b = base[r];
  for (int k = 0; k < c; ++k) { pt_ray[b + k] = r; pt_k[b + k] = k; }
}

// ------------------------------------------------------------ per ray ---
struct RayParams {
  int R, scap, S, Rh, P;   // S = batch max samples, Rh = hit rays
  const float *target_s, *target_d;
  const unsigned char* ray_mask;
  const int *count, *base;
  const float* smp_depth;
  const float *sdf, *rgb;   // per point
  float trunc, max_depth, pad_depth, w_rgb, w_depth, w_sdf, w_fs;
  int* counts;              // n_fs, n_sdf, n_valid
  double* loss_acc;         // rgb, depth, sdf, fs
  float *o_rgb, *o_depth;
  float *d_sdf, *d_rgb;
  int bwd;
};

// batch-global sample counts (get_masks, utils.py:100-132) incl. the padded tail (Q3)
__global__ void __launch_bounds__(128) k_counts(const RayParams P) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  int nfs = 0, nsdf = 0, nvalid = 0;
  if (r < P.R && P.ray_mask[r]) {
    const float td = P.target_d[r];
    const int cnt = P.count[r];
    for (int k = 0; k < P.S; ++k) {
      const float z = k < cnt ? P.smp_depth[(size_t)r * P.scap + k] : P.pad_depth;
      const bool front = z < __fsub_rn(td, P.trunc), back = z > __fadd_rn(td, P.trunc);
      nfs += front;
      nsdf += (!front && !back && td > 0.f);
    }
    nvalid = (td > 0.01f) && (td < P.max_depth);
  }
  nfs = warp_sum_i(nfs); nsdf = warp_sum_i(nsdf); nvalid = warp_sum_i(nvalid);
  if ((threadIdx.x & 31) == 0) {
    if (nfs) atomicAdd(&P.counts[0], nfs);
    if (nsdf) atomicAdd(&P.counts[1], nsdf);
    if (nvalid) atomicAdd(&P.counts[2], nvalid);
  }
}

// warp per ray: sdf2weights (sparse_voxel.py:276-304) incl. the padded tail, outputs, losses
__global__ void __launch_bounds__(128) k_composite(const RayParams P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + warp;
  if (r >= P.R) return;
  if (!P.ray_mask[r]) {
    if (lane == 0) { P.o_depth[r] = 0.f; P.o_rgb[r * 3] = P.o_rgb[r * 3 + 1] = P.o_rgb[r * 3 + 2] = 0.f; }
    return;
  }
  const int cnt = P.count[r], base = P.base[r], S = P.S;
  const float tr = P.trunc;
  const float* zr = P.smp_depth + (size_t)r * P.scap;
  auto sdf_at = [&](int k) { return k < cnt ? P.sdf[base + k] : 1.0f; };  // masked_scatter_ones
  auto z_at = [&](int k) { return k < cnt ? zr[k] : P.pad_depth; };
  int first = 0x7fffffff;
  for (int k = lane; k < S - 1; k += 32)
    if (sdf_at(k + 1) * sdf_at(k) < 0.f) first = min(first, k);
  first = warp_min_i(first);
  if (first == 0x7fffffff) first = 0;
  const float zlim = z_at(first) + tr;
  float usum = 0.f;
  for (int k = lane; k < cnt; k += 32) {
    const float s = P.sdf[base + k];
    const float a = sigmoidf_acc(s / tr) * sigmoidf_acc((-s) / tr);
    usum += (zr[k] < zlim) ? a : 0.f;
  }
  usum = warp_sum(usum);
  const float Wn = usum + 1e-8f;
  float o_r = 0.f, o_g = 0.f, o_b = 0.f, o_d = 0.f;
  for (int k = lane; k < cnt; k += 32) {
    const float s = P.sdf[base + k];
    const float a = sigmoidf_acc(s / tr) * sigmoidf_acc((-s) / tr);
    const float w = ((zr[k] < zlim) ? a : 0.f) / Wn;
    o_r = fmaf(w, P.rgb[base + k], o_r);
    o_g = fmaf(w, P.rgb[(size_t)P.P + base + k], o_g);
    o_b = fmaf(w, P.rgb[2 * (size_t)P.P + base + k], o_b);
    o_d = fmaf(w, zr[k], o_d);
  }
  o_r = warp_sum(o_r); o_g = warp_sum(o_g); o_b = warp_sum(o_b); o_d = warp_sum(o_d);
  if (lane == 0) { P.o_depth[r] = o_d; P.o_rgb[r * 3] = o_r; P.o_rgb[r * 3 + 1] = o_g; P.o_rgb[r * 3 + 2] = o_b; }
  if (!P.bwd) return;
  const float td = P.target_d[r];
  const float tgt[3] = {P.target_s[r * 3], P.target_s[r * 3 + 1], P.target_s[r * 3 + 2]};
  const bool valid = (td > 0.01f) && (td < P.max_depth);
  const float n_fs = (float)P.counts[0], n_sdf = (float)P.counts[1];
  const float n = (float)(P.counts[0] + P.counts[1]);
  const float fs_w = 1.0f - n_fs / n, sdf_w = 1.0f - n_sdf / n;
  const float RS = (float)P.Rh * (float)S;
  // d total / d rgb, d depth (l1 means over Rh*3 and over the valid rays)
  const float e3[3] = {o_r - tgt[0], o_g - tgt[1], o_b - tgt[2]};
  float g3[3];
#pragma unroll
  for (int c = 0; c < 3; ++c)
    g3[c] = valid ? P.w_rgb * ((e3[c] > 0.f) ? 1.f : ((e3[c] < 0.f) ? -1.f : 0.f)) / (3.f * (float)P.Rh) : 0.f;
  const float ed = o_d - td;
  const float g_d = valid ? P.w_depth * ((ed > 0.f) ? 1.f : ((ed < 0.f) ? -1.f : 0.f)) / (float)P.counts[2] : 0.f;
  if (lane == 0) {
    if (valid) {
      atomicAdd(&P.loss_acc[0], (double)(fabsf(e3[0]) + fabsf(e3[1]) + fabsf(e3[2])));
      atomicAdd(&P.loss_acc[1], (double)fabsf(ed));
    }
  }
  float qw = 0.f;
  for (int k = lane; k < cnt; k += 32) {
    const float s = P.sdf[base + k];
    const float a = sigmoidf_acc(s / tr) * sigmoidf_acc((-s) / tr);
    const float w = ((zr[k] < zlim) ? a : 0.f) / Wn;
    const float q_ = g3[0] * P.rgb[base + k] + g3[1] * P.rgb[(size_t)P.P + base + k] +
                     g3[2] * P.rgb[2 * (size_t)P.P + base + k] + g_d * zr[k];
    qw = fmaf(q_, w, qw);
  }
  qw = warp_sum(qw);
  const float c_fs = P.w_fs * fs_w * 2.0f / RS, c_sdf = P.w_sdf * sdf_w * 2.0f / RS;
  float a_fs = 0.f, a_sdf = 0.f;
  for (int k = lane; k < S; k += 32) {
    const float z = z_at(k), s = sdf_at(k);
    const bool front = z < __fsub_rn(td, tr), back = z > __fadd_rn(td, tr);
    float ds = 0.f;
    if (front) { ds += c_fs * (s - 1.f); a_fs += (s - 1.f) * (s - 1.f); }
    if (!front && !back && td > 0.f) {
      const float e = (z + s * tr) - td;
      ds += c_sdf * e * tr;
      a_sdf += e * e;
    }
    if (k < cnt) {
      const float sg = sigmoidf_acc(s / tr);
      const float a = sg * sigmoidf_acc((-s) / tr);
      const bool m = z < zlim;
      const float w = (m ? a : 0.f) / Wn;
      const float cr = P.rgb[base + k], cg = P.rgb[(size_t)P.P + base + k],
                  cb = P.rgb[2 * (size_t)P.P + base + k];
      const float q_ = g3[0] * cr + g3[1] * cg + g3[2] * cb + g_d * z;
      if (m) ds += (q_ - qw) / Wn * a * (1.f - 2.f * sg) / tr;
      P.d_sdf[base + k] = ds;
      P.d_rgb[base + k] = g3[0] * w;
      P.d_rgb[(size_t)P.P + base + k] = g3[1] * w;
      P.d_rgb[2 * (size_t)P.P + base + k] = g3[2] * w;
    }
  }
  a_fs = warp_sum(a_fs); a_sdf = warp_sum(a_sdf);
  if (lane == 0) {
    if (a_sdf != 0.f) atomicAdd(&P.loss_acc[2], (double)a_sdf);
    if (a_fs != 0.f) atomicAdd(&P.loss_acc[3], (double)a_fs);
  }
}

__global__ void k_finalize(const double* acc, const int* counts, int Rh, int S, float w_rgb,
                           float w_depth, float w_sdf, float w_fs, float* losses) {
  if (threadIdx.x || blockIdx.x) return;
  const float n_fs = (float)counts[0], n_sdf = (float)counts[1];
  const float n = (float)(counts[0] + counts[1]);
  const float fs_w = 1.0f - n_fs / n, sdf_w = 1.0f - n_sdf / n;
  const double RS = (double)Rh * (double)S;
  losses[0] = (float)(acc[0] / (3.0 * Rh)) * w_rgb;
  losses[1] = (float)(acc[1] / (double)counts[2]) * w_depth;
  losses[2] = (float)(acc[2] / RS) * sdf_w * w_sdf;
  losses[3] = (float)(acc[3] / RS) * fs_w * w_fs;
}

__global__ void __launch_bounds__(128) k_rayreduce(int R, int scap, int P, const int* count,
                                                   const int* base, const float* smp_depth,
                                                   const float* dp, float* d_o, float* d_d) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + warp;
  if (r >= R) return;
  float a[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const int cnt = count[r], b = base[r];
  for (int k = lane; k < cnt; k += 32) {
    const float z = smp_depth[(size_t)r * scap + k];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const float g = dp[(size_t)d * P + b + k];
      a[d] += g;
      a[3 + d] += g * z;
    }
  }
#pragma unroll
  for (int d = 0; d < 6; ++d) a[d] = warp_sum(a[d]);
  if (lane == 0)
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if (d_o) d_o[r * 3 + d] = a[d];
      if (d_d) d_d[r * 3 + d] = a[3 + d];
    }
}

}  // namespace vox
}  // namespace xrd

using namespace xrd;
using namespace xrd::vox;

extern "C" int xrd_voxfusion_intersect_raw(const XrdRays* rays, const XrdVoxMap* map,
                                           float voxel_size, int n_max, int32_t* idx, float* tmin,
                                           float* tmax, void* stream) {
  if (!rays || !map || !idx || !tmin || !tmax) return XRD_E_NULL;
  if (n_max < 1 || n_max > 64) return XRD_E_SHAPE;
  if (rays->n_rays <= 0) return XRD_OK;
  k_intersect_raw<<<(rays->n_rays + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      rays->n_rays, rays->rays_o, rays->rays_d, map->centres, map->children, voxel_size, n_max,
      idx, tmin, tmax);
  XRD_LAUNCH_CHECK();
  return XRD_OK;
}

extern "C" int xrd_voxfusion_sample_raw(int n_rays, int max_hits, int max_steps,
                                        int rays_per_block, const int32_t* pts_idx,
                                        const float* min_depth, const float* max_depth,
                                        const float* noise, const float* probs, const float* steps,
                                        int32_t* smp_idx, float* smp_depth, float* smp_dist,
                                        void* stream) {
  if (!pts_idx || !min_depth || !max_depth || !noise || !probs || !steps || !smp_idx ||
      !smp_depth || !smp_dist)
    return XRD_E_NULL;
  if (n_rays <= 0) return XRD_OK;
  if (rays_per_block < 1) return XRD_E_SHAPE;
  k_sample_raw<<<(n_rays + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      n_rays, max_hits, max_steps, rays_per_block, pts_idx, min_depth, max_depth, noise, probs,
      steps, smp_idx, smp_depth, smp_dist);
  XRD_LAUNCH_CHECK();
  return XRD_OK;
}

extern "C" int xrd_voxfusion_march(const XrdRays* rays, const XrdVoxMap* map,
                                   const XrdVoxMarchCfg* cfg, const float* noise, XrdVoxMarch* out,
                                   void* stream_) {
  if (!rays || !map || !cfg || !out) return XRD_E_NULL;
  if (!rays->rays_o || !rays->rays_d || !map->centres || !map->children) return XRD_E_NULL;
  if (!out->hit_idx || !out->hit_tmin || !out->hit_tmax || !out->smp_idx || !out->smp_depth ||
      !out->smp_dist || !out->smp_count || !out->smp_base || !out->ray_mask || !out->stats)
    return XRD_E_NULL;
  if (cfg->max_hits < 1 || cfg->max_hits > 64 || cfg->max_samples < 8) return XRD_E_SHAPE;
  const int R = rays->n_rays;
  if (R <= 0) return XRD_OK;
  cudaStream_t stream = (cudaStream_t)stream_;
  MarchParams P;
  P.R = R; P.rays_o = rays->rays_o; P.rays_d = rays->rays_d; P.centres = map->centres;
  P.children = map->children; P.voxel_size = cfg->voxel_size; P.step_size = cfg->step_size;
  P.max_distance = cfg->max_distance; P.max_hits = cfg->max_hits; P.scap = cfg->max_samples;
  P.rays_per_block = cfg->rays_per_block; P.noise = noise; P.seed = cfg->seed;
  P.hit_idx = out->hit_idx; P.hit_tmin = out->hit_tmin; P.hit_tmax = out->hit_tmax;
  P.smp_idx = out->smp_idx; P.smp_depth = out->smp_depth; P.smp_dist = out->smp_dist;
  P.smp_count = out->smp_count; P.smp_base = out->smp_base; P.ray_mask = out->ray_mask;
  P.stats = out->stats;
  // rank / rank2ray live behind the 8 stats ints: callers allocate stats as [8 + 2R]
  P.rank = out->stats + 8; P.rank2ray = out->stats + 8 + R;
  XRD_CUDA_TRY(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int), stream));
  k_march_intersect<<<(R + 127) / 128, 128, 0, stream>>>(P);
  XRD_LAUNCH_CHECK();
  k_rank<<<1, 1024, 0, stream>>>(P);
  XRD_LAUNCH_CHECK();
  k_march_sample<<<(R + 127) / 128, 128, 0, stream>>>(P);
  XRD_LAUNCH_CHECK();
  return XRD_OK;
}

namespace {
struct VWs {
  size_t hdr, pt_ray, pt_k, sdf, rgb, d_sdf, d_rgb, dp, acts, grads, total;
};
VWs vws(int R, int Pn, int with_grads) {
  VWs L;
  const size_t P = (size_t)(Pn > 0 ? Pn : 1), Pp = align_up(P, 64);
  size_t q = 0;
  auto take = [&](size_t b) { size_t o = q; q += align_up(b, 256); return o; };
  L.hdr = take(256);
  L.pt_ray = take(P * 4); L.pt_k = take(P * 4);
  L.sdf = take(P * 4); L.rgb = take(3 * P * 4);
  L.d_sdf = L.d_rgb = L.dp = L.grads = 0;
  L.acts = take((size_t)ra_rows() * Pp * 4);  // the GEMM decoder path keeps activations in HBM
  if (with_grads) {
    L.d_sdf = take(P * 4); L.d_rgb = take(3 * P * 4); L.dp = take(3 * P * 4);
    L.grads = take((size_t)rg_rows() * Pp * 4);
  }
  (void)R;
  L.total = q;
  return L;
}
}  // namespace

#define XRD_GEMM(...)                                         \
  do {                                                        \
    GemmArgs g_ = __VA_ARGS__;                                \
    XRD_CUDA_TRY(launch_gemm(g_, stream));                    \
  } while (0)

// Embedding gather + decoder (decoder_voxfusion.py:122-149) as GEMMs over [feature][point] rows:
// Q.sdf [P] and Q.rgb [3][P] (after the colour head's sigmoid); activations stay in Q.acts.
static int vox_forward(const PointParams& Q, const XrdVoxDecoder* dec, cudaStream_t stream) {
  const int Pn = Q.P, Pp = Q.Pp;
  auto ar = [&](int row) { return Q.acts + (size_t)row * Pp; };
  k_vox_gather<<<(Pn + T - 1) / T, T, 0, stream>>>(Q);
  XRD_LAUNCH_CHECK();
  XRD_GEMM({W, Pn, EMB, dec->w0, EMB, 0, ar(ra_x()), Pp, ar(ra_h1()), Pp, dec->b0, ACT_RELU});
  XRD_GEMM({W, Pn, W, dec->w1, W, 0, ar(ra_h1()), Pp, ar(ra_h2()), Pp, dec->b1, ACT_RELU});
  // sdf_out: torch row 0 = sdf, rows 1..128 = feat
  XRD_GEMM({W, Pn, W, dec->ws + W, W, 0, ar(ra_h2()), Pp, ar(ra_feat()), Pp, dec->bs + 1, ACT_NONE});
  XRD_GEMM({1, Pn, W, dec->ws, W, 0, ar(ra_h2()), Pp, Q.sdf, Pn, dec->bs, ACT_NONE});
  // colour: relu(wc0 [feat, x] + bc0) -> sigmoid(wc1 . + bc1)
  XRD_GEMM({W, Pn, W + EMB, dec->wc0, W + EMB, 0, ar(ra_feat()), Pp, ar(ra_c1()), Pp, dec->bc0, ACT_RELU});
  XRD_GEMM({3, Pn, W, dec->wc1, W, 0, ar(ra_c1()), Pp, Q.rgb, Pn, dec->bc1, ACT_SIGMOID});
  return XRD_OK;
}

__global__ void __launch_bounds__(256) k_vox_pack_raw(int P, const float* rgb, const float* sdf,
                                                      float* raw) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  raw[(size_t)p * 4 + 0] = rgb[p];
  raw[(size_t)p * 4 + 1] = rgb[(size_t)P + p];
  raw[(size_t)p * 4 + 2] = rgb[(size_t)2 * P + p];
  raw[(size_t)p * 4 + 3] = sdf[p];
}

extern "C" size_t xrd_voxfusion_query_workspace_bytes(int n_points) {
  return vws(0, n_points, 0).total;
}

extern "C" int xrd_voxfusion_query(const XrdVoxMap* map, const XrdVoxDecoder* dec, float voxel_size,
                                   const float* points, const int32_t* voxel_ids, int n_points,
                                   float* raw, void* workspace, size_t workspace_bytes,
                                   void* stream_) {
  if (!map || !dec || !workspace) return XRD_E_NULL;
  if (n_points < 0) return XRD_E_SHAPE;
  if (n_points == 0) return XRD_OK;
  if (!points || !voxel_ids || !raw || !map->centres || !map->vertex_idx || !map->embeddings)
    return XRD_E_NULL;
  const VWs L = vws(0, n_points, 0);
  if (workspace_bytes < L.total) return XRD_E_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  char* ws = reinterpret_cast<char*>(workspace);
  PointParams Q{};
  Q.P = n_points; Q.Pp = (int)align_up((size_t)n_points, 64);
  Q.pts = points; Q.pts_vox = voxel_ids;
  Q.centres = map->centres; Q.vertex_idx = map->vertex_idx; Q.emb = map->embeddings;
  Q.voxel_size = voxel_size; Q.dec = *dec;
  Q.acts = reinterpret_cast<float*>(ws + L.acts);
  Q.sdf = reinterpret_cast<float*>(ws + L.sdf); Q.rgb = reinterpret_cast<float*>(ws + L.rgb);
  const int st = vox_forward(Q, dec, stream);
  if (st != XRD_OK) return st;
  k_vox_pack_raw<<<(n_points + 255) / 256, 256, 0, stream>>>(n_points, Q.rgb, Q.sdf, raw);
  XRD_LAUNCH_CHECK();
  return XRD_OK;
}

extern "C" size_t xrd_voxfusion_render_workspace_bytes(int n_rays, int n_points, int with_grads) {
  return vws(n_rays, n_points, with_grads).total;
}

extern "C" int xrd_voxfusion_render(const XrdRays* rays, const XrdVoxMap* map,
                                    const XrdVoxMarch* march, const XrdVoxMarchCfg* mcfg,
                                    const XrdVoxDecoder* dec, const XrdVoxRenderCfg* cfg,
                                    XrdVoxOut* out, XrdVoxGrads* grads, void* workspace,
                                    size_t workspace_bytes, void* stream_) {
  if (!rays || !map || !march || !mcfg || !dec || !cfg || !out || !workspace) return XRD_E_NULL;
  if (!out->rgb || !out->depth) return XRD_E_NULL;
  if (!map->vertex_idx || !map->embeddings) return XRD_E_NULL;
  if (grads && (!rays->target_s || !rays->target_d || !out->losses)) return XRD_E_NULL;
  const int R = rays->n_rays, Pn = cfg->n_points;
  if (R <= 0) return XRD_OK;
  if (cfg->n_hit_rays <= 0 || Pn <= 0) return XRD_E_NOHIT;  // reference: render_rays -> None
  const VWs L = vws(R, Pn, grads != nullptr);
  if (workspace_bytes < L.total) return XRD_E_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  char* ws = reinterpret_cast<char*>(workspace);
  const int Pp = (int)align_up((size_t)Pn, 64);
  int* counts = reinterpret_cast<int*>(ws + L.hdr);
  double* loss_acc = reinterpret_cast<double*>(ws + L.hdr + 64);
  int* pt_ray = reinterpret_cast<int*>(ws + L.pt_ray);
  int* pt_k = reinterpret_cast<int*>(ws + L.pt_k);
  XRD_CUDA_TRY(cudaMemsetAsync(ws + L.hdr, 0, 256, stream));
  k_points<<<(R + 127) / 128, 128, 0, stream>>>(R, march->smp_count, march->smp_base, pt_ray, pt_k);
  XRD_LAUNCH_CHECK();
  PointParams Q;
  Q.P = Pn; Q.Pp = Pp; Q.R = R; Q.pt_ray = pt_ray; Q.pt_k = pt_k;
  Q.rays_o = rays->rays_o; Q.rays_d = rays->rays_d;
  Q.smp_depth = march->smp_depth; Q.smp_idx = march->smp_idx; Q.scap = mcfg->max_samples;
  Q.centres = map->centres; Q.vertex_idx = map->vertex_idx; Q.emb = map->embeddings;
  Q.voxel_size = cfg->voxel_size; Q.dec = *dec;
  Q.acts = reinterpret_cast<float*>(ws + L.acts);
  Q.sdf = reinterpret_cast<float*>(ws + L.sdf); Q.rgb = reinterpret_cast<float*>(ws + L.rgb);
  Q.d_sdf = nullptr; Q.d_rgb = nullptr; Q.grads = nullptr; Q.d_emb = nullptr; Q.dp = nullptr;
  Q.need_dp = 0;
  Q.pts = nullptr; Q.pts_vox = nullptr;
  auto ar = [&](int row) { return Q.acts + (size_t)row * Pp; };
  {
  // timed bracket = the forward decoder chain: gather + 6 GEMM launches (bench.py's roofline)
  KernelTimer kt(stream);
  const int st = vox_forward(Q, dec, stream);
  if (st != XRD_OK) return st;
  }

  RayParams Y;
  Y.R = R; Y.scap = mcfg->max_samples; Y.S = cfg->s_max; Y.Rh = cfg->n_hit_rays; Y.P = Pn;
  Y.target_s = rays->target_s; Y.target_d = rays->target_d; Y.ray_mask = march->ray_mask;
  Y.count = march->smp_count; Y.base = march->smp_base; Y.smp_depth = march->smp_depth;
  Y.sdf = Q.sdf; Y.rgb = Q.rgb; Y.trunc = cfg->trunc; Y.max_depth = cfg->max_depth;
  Y.pad_depth = cfg->pad_depth; Y.w_rgb = cfg->w_rgb; Y.w_depth = cfg->w_depth;
  Y.w_sdf = cfg->w_sdf; Y.w_fs = cfg->w_fs; Y.counts = counts; Y.loss_acc = loss_acc;
  Y.o_rgb = out->rgb; Y.o_depth = out->depth; Y.d_sdf = nullptr; Y.d_rgb = nullptr; Y.bwd = 0;
  if (grads) {
    k_counts<<<(R + 127) / 128, 128, 0, stream>>>(Y);
    XRD_LAUNCH_CHECK();
    Y.d_sdf = reinterpret_cast<float*>(ws + L.d_sdf);
    Y.d_rgb = reinterpret_cast<float*>(ws + L.d_rgb);
    Y.bwd = 1;
  }
  k_composite<<<(R + 3) / 4, 128, 0, stream>>>(Y);
  XRD_LAUNCH_CHECK();
  if (!grads) return XRD_OK;
  k_finalize<<<1, 32, 0, stream>>>(loss_acc, counts, cfg->n_hit_rays, cfg->s_max, cfg->w_rgb,
                                   cfg->w_depth, cfg->w_sdf, cfg->w_fs, out->losses);
  XRD_LAUNCH_CHECK();

  Q.d_sdf = Y.d_sdf; Q.d_rgb = Y.d_rgb;
  Q.grads = reinterpret_cast<float*>(ws + L.grads);
  Q.d_emb = grads->d_embeddings;
  Q.dp = reinterpret_cast<float*>(ws + L.dp);
  Q.need_dp = (grads->d_rays_o || grads->d_rays_d) ? 1 : 0;
  auto gr_ = [&](int row) { return Q.grads + (size_t)row * Pp; };
  k_vox_dout<<<(Pn + 255) / 256, 256, 0, stream>>>(Q);
  XRD_LAUNCH_CHECK();
  {
    GemmArgs g{};  // dc1 = relu'(c1) * (wc1^T do)
    g.M = W; g.N = Pn; g.K = 3; g.A = dec->wc1; g.lda = W; g.transA = 1; g.B = gr_(rg_do()); g.ldb = Pp;
    g.C = gr_(rg_dc1()); g.ldc = Pp; g.relu_mask = ar(ra_c1()); g.ldmask = Pp;
    XRD_CUDA_TRY(launch_gemm(g, stream));
    // d[feat, x] = wc0^T dc1  (144 rows: dfeat | dxc)
    g = GemmArgs{};
    g.M = W + EMB; g.N = Pn; g.K = W; g.A = dec->wc0; g.lda = W + EMB; g.transA = 1;
    g.B = gr_(rg_dc1()); g.ldb = Pp; g.C = gr_(rg_dso() + 1); g.ldc = Pp;
    XRD_CUDA_TRY(launch_gemm(g, stream));
    // d2 = relu'(h2) * (ws^T [dsdf, dfeat])
    g = GemmArgs{};
    g.M = W; g.N = Pn; g.K = W + 1; g.A = dec->ws; g.lda = W; g.transA = 1; g.B = gr_(rg_dso());
    g.ldb = Pp; g.C = gr_(rg_d2()); g.ldc = Pp; g.relu_mask = ar(ra_h2()); g.ldmask = Pp;
    XRD_CUDA_TRY(launch_gemm(g, stream));
    // d1 = relu'(h1) * (w1^T d2)
    g = GemmArgs{};
    g.M = W; g.N = Pn; g.K = W; g.A = dec->w1; g.lda = W; g.transA = 1; g.B = gr_(rg_d2()); g.ldb = Pp;
    g.C = gr_(rg_d1()); g.ldc = Pp; g.relu_mask = ar(ra_h1()); g.ldmask = Pp;
    XRD_CUDA_TRY(launch_gemm(g, stream));
    // dx = w0^T d1 + dxc
    g = GemmArgs{};
    g.M = EMB; g.N = Pn; g.K = W; g.A = dec->w0; g.lda = EMB; g.transA = 1; g.B = gr_(rg_d1()); g.ldb = Pp;
    g.C = gr_(rg_dx()); g.ldc = Pp; g.addend = gr_(rg_dxc()); g.ldadd = Pp;
    XRD_CUDA_TRY(launch_gemm(g, stream));
  }
  k_vox_scatter<<<(Pn + T - 1) / T, T, 0, stream>>>(Q);
  XRD_LAUNCH_CHECK();

  if (grads->d_decoder) {
    const XrdVoxDecoderGrads* G = grads->d_decoder;
    const float* A = Q.acts;
    const float* Gd = Q.grads;
    DwParams D;
    D.n_jobs = 0; D.P = Pn; D.Pp = Pp; D.chunk = 512;
    auto ar = [&](int row) { return A + (size_t)row * Pp; };
    auto gr = [&](int row) { return Gd + (size_t)row * Pp; };
    auto add = [&](const float* a, int nA, const float* b, int nB, float* o, int sj, int si, float* bias) {
      if (!o) return;
      DwJob& J = D.jobs[D.n_jobs++];
      J.A = a; J.nA = nA; J.B = b; J.nB = nB; J.mask = nullptr; J.out = o; J.sj = sj; J.si = si; J.bias = bias;
    };
    for (int c = 0; c < W; c += 32) {
      add(ar(ra_x()), EMB, gr(rg_d1() + c), 32, G->w0 ? G->w0 + (size_t)c * EMB : nullptr, EMB, 1, G->b0 ? G->b0 + c : nullptr);
      add(ar(ra_h1()), W, gr(rg_d2() + c), 32, G->w1 ? G->w1 + (size_t)c * W : nullptr, W, 1, G->b1 ? G->b1 + c : nullptr);
      add(ar(ra_h2()), W, gr(rg_dso() + c), 32, G->ws ? G->ws + (size_t)c * W : nullptr, W, 1, G->bs ? G->bs + c : nullptr);
      add(ar(ra_feat()), W, gr(rg_dc1() + c), 32, G->wc0 ? G->wc0 + (size_t)c * (W + EMB) : nullptr, W + EMB, 1, G->bc0 ? G->bc0 + c : nullptr);
      add(ar(ra_x()), EMB, gr(rg_dc1() + c), 32, G->wc0 ? G->wc0 + (size_t)c * (W + EMB) + W : nullptr, W + EMB, 1, nullptr);
    }
    add(ar(ra_h2()), W, gr(rg_dso() + W), 1, G->ws ? G->ws + (size_t)W * W : nullptr, W, 1, G->bs ? G->bs + W : nullptr);
    add(ar(ra_c1()), W, gr(rg_do()), 3, G->wc1, W, 1, G->bc1);
    if (D.n_jobs > DW_MAX_JOBS) return XRD_E_SHAPE;
    XRD_CUDA_TRY(launch_dw(D, stream));
  }
  if (Q.need_dp) {
    k_rayreduce<<<(R + 3) / 4, 128, 0, stream>>>(R, mcfg->max_samples, Pn, march->smp_count,
                                                 march->smp_base, march->smp_depth, Q.dp,
                                                 grads->d_rays_o, grads->d_rays_d);
    XRD_LAUNCH_CHECK();
  }
  return XRD_OK;
}


// Direct entry to the wide-MLP GEMM (gemm.cuh / gemm_t5.cuh) for the unit tests:
//   C[m][n] = act( sum_k A(m,k) B[k][n] + bias[m] ), optional relu mask / addend, under the
//   calling thread's xrd_debug_gemm_mode.  All pointers DEVICE.
extern "C" int xrd_debug_gemm(int M, int N, int K, const float* A, int lda, int transA, const float* B,
                              int ldb, float* C, int ldc, const float* bias, int act,
                              const float* relu_mask, int ldmask, const float* addend, int ldadd,
                              void* stream) {
  if (!A || !B || !C) return XRD_E_NULL;
  if (M <= 0 || N <= 0 || K <= 0) return XRD_E_SHAPE;
  xrd::GemmArgs g{};
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.transA = transA; g.B = B; g.ldb = ldb;
  g.C = C; g.ldc = ldc; g.bias = bias; g.act = act; g.relu_mask = relu_mask; g.ldmask = ldmask;
  g.addend = addend; g.ldadd = ldadd;
  XRD_CUDA_TRY(xrd::launch_gemm(g, (cudaStream_t)stream));
  return XRD_OK;
}

// ... with the remaining epilogue options: act_out[m][n] receives the masked activation before
// the addend, accumulate != 0 adds the result to C.
extern "C" int xrd_debug_gemm_ex(int M, int N, int K, const float* A, int lda, int transA, const float* B,
                                 int ldb, float* C, int ldc, const float* bias, int act,
                                 const float* relu_mask, int ldmask, const float* addend, int ldadd,
                                 float* act_out, int ldact, int accumulate, void* stream) {
  if (!A || !B || !C) return XRD_E_NULL;
  if (M <= 0 || N <= 0 || K <= 0) return XRD_E_SHAPE;
  xrd::GemmArgs g{};
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.transA = transA; g.B = B; g.ldb = ldb;
  g.C = C; g.ldc = ldc; g.bias = bias; g.act = act; g.relu_mask = relu_mask; g.ldmask = ldmask;
  g.addend = addend; g.ldadd = ldadd; g.act_out = act_out; g.ldact = ldact; g.accumulate = accumulate;
  XRD_CUDA_TRY(xrd::launch_gemm(g, (cudaStream_t)stream));
  return XRD_OK;
}

// Direct entry to the weight-gradient kernels (dw.cuh) for the unit tests:
//   out[j][i] += sum_p B[j][p] (where bit (j & 31) of mask[j / 32][p] is set) * A[i][p],
//   bias[j] += sum_p B[j][p] (masked)
// A [nA][Pp], B [nB][Pp] rows of P valid points; the rows of B are cut into 32-row jobs exactly
// as the model kernels do, under the calling thread's xrd_debug_gemm_mode.  DEVICE pointers.
extern "C" int xrd_debug_dw(int nA, int nB, int P, int Pp, const float* A, const float* B,
                            const uint32_t* mask, float* out, float* bias, void* stream) {
  if (!A || !B || !out) return XRD_E_NULL;
  if (nA <= 0 || nB <= 0 || P <= 0 || Pp < P) return XRD_E_SHAPE;
  xrd::DwParams D;
  D.n_jobs = 0; D.P = P; D.Pp = Pp; D.chunk = 512;
  for (int c = 0; c < nB; c += 32) {
    if (D.n_jobs >= xrd::DW_MAX_JOBS) return XRD_E_SHAPE;
    xrd::DwJob& J = D.jobs[D.n_jobs++];
    J.A = A; J.nA = nA; J.B = B + (size_t)c * Pp; J.nB = nB - c < 32 ? nB - c : 32;
    J.mask = mask ? mask + (size_t)(c / 32) * P : nullptr;
    J.out = out + (size_t)c * nA; J.sj = nA; J.si = 1;
    J.bias = bias ? bias + c : nullptr;
  }
  XRD_CUDA_TRY(xrd::launch_dw(D, (cudaStream_t)stream));
  return XRD_OK;
}
