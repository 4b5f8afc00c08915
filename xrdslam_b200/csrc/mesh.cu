// Marching cubes over a batch of scalar volumes (the mesher's isosurface step).
//
// Replaces skimage.measure.marching_cubes on the host (slam/common/mesher.py:203-233, one call
// on the whole 256^3 field; slam/algorithms/voxfusion.py:253-279, one call per voxel).
// Two phases, both on the caller's stream:
//   count: per cube the case index and its triangle count, per lattice point the crossing
//          flags of its +x/+y/+z edges; exclusive scans over both; totals (V, F) to the device.
//   emit:  one vertex per crossing edge (welded inside a volume), ordered by
//          (volume, i, j, k, axis); faces ordered by (volume, cube, table order).
// Every output position comes from a scan, so the result does not depend on the schedule.
// Case tables: mc_tables.cuh (scripts/gen_mc_tables.py); oracle: oracle/marching_cubes.py.
#include "common.cuh"
#include "mc_tables.cuh"

namespace xrd {
namespace {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

struct Vol {
  const float* field;
  int B, nx, ny, nz;
  long long npt;   // points per volume
  long long ncube; // cubes per volume
};

__device__ __forceinline__ bool inside(float v, float level) { return v < level; }

// ---- count -------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mc_edge_flags(Vol V, float level, uint8_t* flags,
                                                       int* vcount) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= V.npt * V.B) return;
  const long long q = p % V.npt;
  const int k = (int)(q % V.nz), j = (int)((q / V.nz) % V.ny), i = (int)(q / ((long long)V.nz * V.ny));
  const float v0 = V.field[p];
  const bool s0 = inside(v0, level);
  int f = 0;
  if (i + 1 < V.nx && inside(V.field[p + (long long)V.ny * V.nz], level) != s0) f |= 1;
  if (j + 1 < V.ny && inside(V.field[p + V.nz], level) != s0) f |= 2;
  if (k + 1 < V.nz && inside(V.field[p + 1], level) != s0) f |= 4;
  flags[p] = (uint8_t)f;
  vcount[p] = __popc(f);
}

__device__ __forceinline__ void cube_origin(const Vol& V, long long c, long long& p0, int& i, int& j,
                                            int& k, int& b) {
  const int cz = V.nz - 1, cy = V.ny - 1;
  b = (int)(c / V.ncube);
  const long long q = c % V.ncube;
  k = (int)(q % cz);
  j = (int)((q / cz) % cy);
  i = (int)(q / ((long long)cz * cy));
  p0 = (long long)b * V.npt + ((long long)i * V.ny + j) * V.nz + k;
}

__device__ __forceinline__ int cube_case(const Vol& V, long long p0, float level) {
  const long long sx = (long long)V.ny * V.nz, sy = V.nz;
  int cs = 0;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const long long a = p0 + (n & 1) * sx + ((n >> 1) & 1) * sy + ((n >> 2) & 1);
    if (inside(V.field[a], level)) cs |= 1 << n;
  }
  return cs;
}

__global__ void __launch_bounds__(256) k_mc_cube_count(Vol V, float level, int* tcount) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= V.ncube * V.B) return;
  long long p0;
  int i, j, k, b;
  cube_origin(V, c, p0, i, j, k, b);
  tcount[c] = mc::c_tri_count[cube_case(V, p0, level)];
}

// ---- exclusive scan (3 passes, integer: deterministic) --------------------------------
__device__ __forceinline__ int block_exclusive_scan(int v, int* sh, int& total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = lane < (int)(blockDim.x >> 5) ? sh[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    sh[lane] = s;  // inclusive warp prefix
  }
  __syncthreads();
  total = sh[(blockDim.x >> 5) - 1];
  const int excl = x - v + (w ? sh[w - 1] : 0);
  __syncthreads();
  return excl;
}

// tile-local exclusive scan in place; tile total -> sums[blockIdx.x]
__global__ void __launch_bounds__(kScanThreads) k_scan_tiles(int* data, long long n, int* sums) {
  __shared__ int sh[32];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  int v[kScanItems], s = 0;
#pragma unroll
  for (int q = 0; q < kScanItems; ++q) {
    v[q] = base + q < n ? data[base + q] : 0;
    s += v[q];
  }
  int total;
  int run = block_exclusive_scan(s, sh, total);
#pragma unroll
  for (int q = 0; q < kScanItems; ++q) {
    if (base + q < n) data[base + q] = run;
    run += v[q];
  }
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// exclusive scan of the tile totals in place (one block), grand total -> *total_out
__global__ void __launch_bounds__(1024) k_scan_sums(int* sums, int n, int* total_out) {
  __shared__ int sh[32];
  int carry = 0;
  for (int b = 0; b < n; b += blockDim.x) {
    const int idx = b + threadIdx.x;
    const int v = idx < n ? sums[idx] : 0;
    int total;
    const int e = block_exclusive_scan(v, sh, total);
    if (idx < n) sums[idx] = carry + e;
    carry += total;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_add(int* data, long long n, const int* sums) {
  const int add = sums[blockIdx.x];
  const long long base = (long long)blockIdx.x * kScanTile;
  for (int q = threadIdx.x; q < kScanTile; q += kScanThreads)
    if (base + q < n) data[base + q] += add;
}

int scan_exclusive(int* data, long long n, int* sums, int* total, cudaStream_t s) {
  const int tiles = (int)((n + kScanTile - 1) / kScanTile);
  k_scan_tiles<<<tiles, kScanThreads, 0, s>>>(data, n, sums);
  XRD_LAUNCH_CHECK();
  k_scan_sums<<<1, 1024, 0, s>>>(sums, tiles, total);
  XRD_LAUNCH_CHECK();
  k_scan_add<<<tiles, kScanThreads, 0, s>>>(data, n, sums);
  XRD_LAUNCH_CHECK();
  return XRD_OK;
}

// ---- emit ----------------------------------------------------------------------------------
// t = (level - v0) / (v1 - v0) in fp32 (v0 at the lower-index end);
// world_d = origin_d + (i_d + t * e_d) * spacing_d in fp64, stored as fp32.
__global__ void __launch_bounds__(256) k_mc_emit_verts(Vol V, float level, const uint8_t* flags,
                                                       const int* voff, const double* origins,
                                                       const double* spacings, double3 origin,
                                                       double3 spacing, float* verts) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= V.npt * V.B) return;
  const int f = flags[p];
  if (!f) return;
  const int b = (int)(p / V.npt);
  const long long q = p % V.npt;
  const int idx[3] = {(int)(q / ((long long)V.nz * V.ny)), (int)((q / V.nz) % V.ny), (int)(q % V.nz)};
  double org[3] = {origin.x, origin.y, origin.z}, sp[3] = {spacing.x, spacing.y, spacing.z};
  if (origins)
    for (int d = 0; d < 3; ++d) org[d] = origins[(size_t)b * 3 + d];
  if (spacings)
    for (int d = 0; d < 3; ++d) sp[d] = spacings[(size_t)b * 3 + d];
  const long long stride[3] = {(long long)V.ny * V.nz, V.nz, 1};
  const float v0 = V.field[p];
  int o = voff[p];
  for (int a = 0; a < 3; ++a) {
    if (!(f >> a & 1)) continue;
    const float v1 = V.field[p + stride[a]];
    const float t = __fdiv_rn(__fsub_rn(level, v0), __fsub_rn(v1, v0));
    for (int d = 0; d < 3; ++d) {
      const double id = d == a ? __dadd_rn((double)idx[d], (double)t) : (double)idx[d];
      verts[(size_t)o * 3 + d] = (float)__dadd_rn(org[d], __dmul_rn(id, sp[d]));
    }
    ++o;
  }
}

__global__ void __launch_bounds__(256) k_mc_emit_faces(Vol V, float level, const uint8_t* flags,
                                                       const int* voff, const int* toff,
                                                       int32_t* faces) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= V.ncube * V.B) return;
  long long p0;
  int i, j, k, b;
  cube_origin(V, c, p0, i, j, k, b);
  const int cs = cube_case(V, p0, level);
  const int nt = mc::c_tri_count[cs];
  if (!nt) return;
  const long long sx = (long long)V.ny * V.nz, sy = V.nz;
  const int base = toff[c];
  for (int t = 0; t < 3 * nt; ++t) {
    const int e = mc::c_tri_table[cs][t];
    const int a = e >> 2, b0 = e & 1, b1 = (e >> 1) & 1;
    const int dx = a == 0 ? 0 : b0, dy = a == 1 ? 0 : (a == 0 ? b0 : b1), dz = a == 2 ? 0 : b1;
    const long long p = p0 + dx * sx + dy * sy + dz;
    faces[(size_t)base * 3 + t] = voff[p] + __popc(flags[p] & ((1 << a) - 1));
  }
}

struct McWs {
  size_t flags, voff, toff, vsums, tsums, total;
};

McWs mc_ws(long long npt, long long ncube) {
  McWs L;
  size_t q = 0;
  auto take = [&](size_t b) { size_t o = q; q += align_up(b, 256); return o; };
  L.flags = take((size_t)npt);
  L.voff = take((size_t)npt * 4);
  L.toff = take((size_t)(ncube > 0 ? ncube : 1) * 4);
  L.vsums = take((size_t)((npt + kScanTile - 1) / kScanTile + 1) * 4);
  L.tsums = take((size_t)((ncube + kScanTile - 1) / kScanTile + 1) * 4);
  L.total = q;
  return L;
}

// validates the shape; fills Vol
int mc_check(const XrdMcVolumes* v, Vol& V) {
  if (!v || !v->field) return XRD_E_NULL;
  if (v->n_volumes < 0 || v->nx < 2 || v->ny < 2 || v->nz < 2) return XRD_E_SHAPE;
  V.field = v->field;
  V.B = v->n_volumes; V.nx = v->nx; V.ny = v->ny; V.nz = v->nz;
  V.npt = (long long)v->nx * v->ny * v->nz;
  V.ncube = (long long)(v->nx - 1) * (v->ny - 1) * (v->nz - 1);
  // vertex and face ids are int32: at most 3 vertices per point, XRD_MC_MAX_TRIS per cube
  if (3 * V.npt * V.B > 0x7fffffffLL || XRD_MC_MAX_TRIS * V.ncube * V.B > 0x7fffffffLL)
    return XRD_E_SHAPE;
  return XRD_OK;
}

}  // namespace
}  // namespace xrd

using namespace xrd;

extern "C" size_t xrd_mc_workspace_bytes(int n_volumes, int nx, int ny, int nz) {
  if (n_volumes < 0 || nx < 2 || ny < 2 || nz < 2) return 0;
  const long long B = n_volumes;
  return mc_ws(B * nx * ny * nz, B * (nx - 1) * (ny - 1) * (nz - 1)).total;
}

extern "C" int xrd_mc_count(const XrdMcVolumes* v, float level, int* counts, void* ws_,
                            size_t ws_bytes, void* stream_) {
  Vol V;
  const int st = mc_check(v, V);
  if (st != XRD_OK) return st;
  if (!counts || !ws_) return XRD_E_NULL;
  const long long npt = V.npt * V.B, ncube = V.ncube * V.B;
  const McWs L = mc_ws(npt, ncube);
  if (ws_bytes < L.total) return XRD_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  if (npt == 0) {
    XRD_CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int), s));
    return XRD_OK;
  }
  char* ws = reinterpret_cast<char*>(ws_);
  uint8_t* flags = reinterpret_cast<uint8_t*>(ws + L.flags);
  int* voff = reinterpret_cast<int*>(ws + L.voff);
  int* toff = reinterpret_cast<int*>(ws + L.toff);
  k_mc_edge_flags<<<(unsigned)((npt + 255) / 256), 256, 0, s>>>(V, level, flags, voff);
  XRD_LAUNCH_CHECK();
  k_mc_cube_count<<<(unsigned)((ncube + 255) / 256), 256, 0, s>>>(V, level, toff);
  XRD_LAUNCH_CHECK();
  int r = scan_exclusive(voff, npt, reinterpret_cast<int*>(ws + L.vsums), counts + 0, s);
  if (r != XRD_OK) return r;
  return scan_exclusive(toff, ncube, reinterpret_cast<int*>(ws + L.tsums), counts + 1, s);
}

extern "C" int xrd_mc_emit(const XrdMcVolumes* v, float level, float* verts, int32_t* faces,
                           void* ws_, size_t ws_bytes, void* stream_) {
  Vol V;
  const int st = mc_check(v, V);
  if (st != XRD_OK) return st;
  if (!ws_) return XRD_E_NULL;
  const long long npt = V.npt * V.B, ncube = V.ncube * V.B;
  const McWs L = mc_ws(npt, ncube);
  if (ws_bytes < L.total) return XRD_E_WORKSPACE;
  if (npt == 0) return XRD_OK;
  cudaStream_t s = (cudaStream_t)stream_;
  char* ws = reinterpret_cast<char*>(ws_);
  const uint8_t* flags = reinterpret_cast<const uint8_t*>(ws + L.flags);
  const int* voff = reinterpret_cast<const int*>(ws + L.voff);
  const int* toff = reinterpret_cast<const int*>(ws + L.toff);
  if (verts) {
    k_mc_emit_verts<<<(unsigned)((npt + 255) / 256), 256, 0, s>>>(
        V, level, flags, voff, v->origins, v->spacings,
        make_double3(v->origin[0], v->origin[1], v->origin[2]),
        make_double3(v->spacing[0], v->spacing[1], v->spacing[2]), verts);
    XRD_LAUNCH_CHECK();
  }
  if (faces) {
    k_mc_emit_faces<<<(unsigned)((ncube + 255) / 256), 256, 0, s>>>(V, level, flags, voff, toff,
                                                                     faces);
    XRD_LAUNCH_CHECK();
  }
  return XRD_OK;
}
