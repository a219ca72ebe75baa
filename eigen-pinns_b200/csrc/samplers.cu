// Farthest-point and voxel down-sampling, fp64, bit-exact w.r.t. the numpy reference
// (src/samplers.py:97-143 and :9-94).
//
// Exactness rules shared by both kernels: d = sqrt((dx*dx + dy*dy) + dz*dz) with explicit
// round-to-nearest intrinsics (no FMA contraction), running minimum, and the FIRST index wins
// every arg-max / arg-min tie (symmetric meshes are full of exact ties).
//
// FPS: one persistent cooperative kernel runs all n_samples-1 dependent iterations.  Each CTA
// (one per SM, 1024 threads) keeps its slice of the point set and of the running-minimum array in
// shared memory (32 B per point, up to 7168 points per SM, 1.06 M points on 148 SMs), so an
// iteration touches no HBM at all: local update + arg-max, one 24-byte record per CTA, one grid
// barrier, and every CTA redundantly reduces the <= 148 records.  Larger clouds fall back to the
// same kernel reading coordinates / distances from global memory (L2 for a few million points;
// 40 N bytes per iteration of HBM traffic beyond that).
#include <cooperative_groups.h>
#include "ep_common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kFpsThreads = 1024;
constexpr int kFpsSmemPoints = 7168;                 // 7168 * 32 B = 224 KB
constexpr int kMaxFpsBlocks = 1024;

struct FpsRecord { double d; long long i; double x, y, z; };   // 40 bytes

__device__ __forceinline__ double dist3(double px, double py, double pz, double qx, double qy, double qz) {
  const double dx = __dsub_rn(px, qx), dy = __dsub_rn(py, qy), dz = __dsub_rn(pz, qz);
  const double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  return __dsqrt_rn(s);
}

__device__ __forceinline__ bool better(double d1, long long i1, double d2, long long i2) {
  return d1 > d2 || (d1 == d2 && i1 < i2);
}

// arg-max over the block with first-index ties; result valid in every thread
__device__ void block_argmax(double& d, long long& i, double* sh_d, long long* sh_i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, d, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (better(od, oi, d, i)) { d = od; i = oi; }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) { sh_d[warp] = d; sh_i[warp] = i; }
  __syncthreads();
  const int n_warps = blockDim.x >> 5;
  double bd = sh_d[0];
  long long bi = sh_i[0];
  for (int w = 1; w < n_warps; ++w)
    if (better(sh_d[w], sh_i[w], bd, bi)) { bd = sh_d[w]; bi = sh_i[w]; }
  d = bd; i = bi;
}

template <bool ONCHIP>
__global__ void __launch_bounds__(kFpsThreads, 1)
fps_kernel(long long N, const double* __restrict__ pts, int n_samples, long long start, long long per_block,
           double* __restrict__ gdist, long long* __restrict__ out, FpsRecord* __restrict__ records) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double sh_d[32];
  __shared__ long long sh_i[32];
  __shared__ FpsRecord sh_last;
  cg::grid_group grid = cg::this_grid();
  double* xs = reinterpret_cast<double*>(smem_raw);
  double* ys = xs + (ONCHIP ? per_block : 0);
  double* zs = ys + (ONCHIP ? per_block : 0);
  double* ds = zs + (ONCHIP ? per_block : 0);
  const long long base = (long long)blockIdx.x * per_block;
  const long long cnt = max(0LL, min(per_block, N - base));
  const int tid = threadIdx.x;

  if (ONCHIP) {
    for (long long l = tid; l < cnt; l += blockDim.x) {
      const double* p = pts + (base + l) * 3;
      xs[l] = p[0]; ys[l] = p[1]; zs[l] = p[2];
      ds[l] = __longlong_as_double(0x7ff0000000000000LL);
    }
  } else {
    for (long long l = tid; l < cnt; l += blockDim.x) gdist[base + l] = __longlong_as_double(0x7ff0000000000000LL);
  }
  if (tid == 0) {
    sh_last.i = start;
    sh_last.x = pts[start * 3 + 0]; sh_last.y = pts[start * 3 + 1]; sh_last.z = pts[start * 3 + 2];
    if (blockIdx.x == 0) out[0] = start;
  }
  __syncthreads();

  for (int s = 1; s < n_samples; ++s) {
    const double qx = sh_last.x, qy = sh_last.y, qz = sh_last.z;
    double best_d = -1.0;
    long long best_i = 0x7fffffffffffffffLL;
    for (long long l = tid; l < cnt; l += blockDim.x) {
      double px, py, pz, old;
      if (ONCHIP) { px = xs[l]; py = ys[l]; pz = zs[l]; old = ds[l]; }
      else {
        const double* p = pts + (base + l) * 3;
        px = p[0]; py = p[1]; pz = p[2]; old = gdist[base + l];
      }
      const double d = dist3(px, py, pz, qx, qy, qz);
      const double nd = (d < old) ? d : old;                  // np.minimum
      if (ONCHIP) ds[l] = nd; else gdist[base + l] = nd;
      if (nd > best_d) { best_d = nd; best_i = base + l; }     // ascending l: first index kept
    }
    block_argmax(best_d, best_i, sh_d, sh_i);
    FpsRecord* rec = records + (size_t)(s & 1) * gridDim.x;
    if (tid == 0) {
      FpsRecord r;
      r.d = best_d; r.i = best_i;
      if (best_i < N) {
        if (ONCHIP) { const long long l = best_i - base; r.x = xs[l]; r.y = ys[l]; r.z = zs[l]; }
        else { r.x = pts[best_i * 3]; r.y = pts[best_i * 3 + 1]; r.z = pts[best_i * 3 + 2]; }
      } else { r.x = r.y = r.z = 0.0; }
      rec[blockIdx.x] = r;
    }
    grid.sync();
    // every CTA reduces the per-CTA records (<= kMaxFpsBlocks of them)
    double rd = -1.0;
    long long ri = 0x7fffffffffffffffLL;
    int slot = -1;
    for (int b = tid; b < (int)gridDim.x; b += blockDim.x) {
      const double od = rec[b].d;
      const long long oi = rec[b].i;
      if (better(od, oi, rd, ri)) { rd = od; ri = oi; slot = b; }
    }
    const long long mine = ri;
    block_argmax(rd, ri, sh_d, sh_i);
    if (slot >= 0 && mine == ri) {            // exactly one thread holds the winning record
      sh_last = rec[slot];
      if (blockIdx.x == 0) out[s] = ri;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ bounds
__global__ void __launch_bounds__(256)
bounds_partial_kernel(long long N, const double* __restrict__ pts, double* __restrict__ parts) {
  __shared__ double sh[6][8];
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double v = pts[i * 3 + a];
      lo[a] = fmin(lo[a], v); hi[a] = fmax(hi[a], v);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
    }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int a = 0; a < 3; ++a) { sh[a][warp] = lo[a]; sh[3 + a][warp] = hi[a]; }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = sh[threadIdx.x][0];
    for (int w = 1; w < 8; ++w) v = threadIdx.x < 3 ? fmin(v, sh[threadIdx.x][w]) : fmax(v, sh[threadIdx.x][w]);
    parts[(size_t)blockIdx.x * 6 + threadIdx.x] = v;
  }
}

constexpr int kBoundsBlocks = 128;
__device__ double g_bounds_parts[kBoundsBlocks * 6];

__global__ void bounds_final_kernel(int n_parts, double* __restrict__ lo_hi) {
  const int a = threadIdx.x;
  if (a < 6) {
    double v = g_bounds_parts[a];
    for (int b = 1; b < n_parts; ++b)
      v = a < 3 ? fmin(v, g_bounds_parts[b * 6 + a]) : fmax(v, g_bounds_parts[b * 6 + a]);
    lo_hi[a] = v;
  }
}

// ------------------------------------------------------------------ voxel
constexpr unsigned long long kEmptyU64 = 0xffffffffffffffffULL;
constexpr int kScanBlock = 1024;

__global__ void __launch_bounds__(256)
voxel_init_kernel(long long n_vox, unsigned long long* __restrict__ tab_d, unsigned long long* __restrict__ tab_i) {
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < n_vox; v += (long long)gridDim.x * blockDim.x) {
    tab_d[v] = kEmptyU64; tab_i[v] = kEmptyU64;
  }
}

__global__ void __launch_bounds__(256)
voxel_assign_kernel(long long N, const double* __restrict__ pts, double lx, double ly, double lz, double voxel,
                    long long dx, long long dy, long long dz, long long* __restrict__ vid,
                    unsigned long long* __restrict__ dcode, unsigned long long* __restrict__ tab_d) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
    const double px = pts[i * 3], py = pts[i * 3 + 1], pz = pts[i * 3 + 2];
    long long cx = (long long)__ddiv_rn(__dsub_rn(px, lx), voxel);       // .astype(int): truncation
    long long cy = (long long)__ddiv_rn(__dsub_rn(py, ly), voxel);
    long long cz = (long long)__ddiv_rn(__dsub_rn(pz, lz), voxel);
    cx = min(max(cx, 0LL), dx - 1); cy = min(max(cy, 0LL), dy - 1); cz = min(max(cz, 0LL), dz - 1);
    const long long v = cx * dy * dz + cy * dz + cz;
    const double ccx = __dadd_rn(lx, __dmul_rn((double)cx + 0.5, voxel));
    const double ccy = __dadd_rn(ly, __dmul_rn((double)cy + 0.5, voxel));
    const double ccz = __dadd_rn(lz, __dmul_rn((double)cz + 0.5, voxel));
    const double d = dist3(px, py, pz, ccx, ccy, ccz);
    const unsigned long long code = (unsigned long long)__double_as_longlong(d);   // d >= 0: order preserving
    vid[i] = v;
    dcode[i] = code;
    atomicMin(tab_d + v, code);
  }
}

// Small grids (the coarse levels of a hierarchy: a few hundred to a few thousand voxels for 10^6 points) make the global
// atomicMin above the whole cost - a Gaussian cloud puts most points into a few dozen voxels.  Here every warp first
// reduces the lanes that fall into the same voxel (match_any + two 32-bit min reductions = exact 64-bit min), the block
// keeps a table of minima in shared memory, and only the occupied entries go to global memory: blocks x occupied
// voxels global atomics instead of one per point.  Same minima, so the picks are unchanged.
constexpr int kVoxelSmemMax = 4096;                       // voxels (32 KB of shared memory)
__global__ void __launch_bounds__(256)
voxel_assign_small_kernel(long long N, const double* __restrict__ pts, double lx, double ly, double lz, double voxel,
                          long long dx, long long dy, long long dz, long long* __restrict__ vid,
                          unsigned long long* __restrict__ dcode, unsigned long long* __restrict__ tab_d, int n_vox) {
  extern __shared__ unsigned long long s_tab[];
  for (int v = threadIdx.x; v < n_vox; v += blockDim.x) s_tab[v] = kEmptyU64;
  __syncthreads();
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n_iter = (N + stride - 1) / stride;      // all lanes iterate together (the reductions need the mask)
  for (long long it = 0; it < n_iter; ++it) {
    const long long i = first + it * stride;
    const bool live = i < N;
    long long v = -1;
    unsigned long long code = kEmptyU64;
    if (live) {
      const double px = pts[i * 3], py = pts[i * 3 + 1], pz = pts[i * 3 + 2];
      long long cx = (long long)__ddiv_rn(__dsub_rn(px, lx), voxel);
      long long cy = (long long)__ddiv_rn(__dsub_rn(py, ly), voxel);
      long long cz = (long long)__ddiv_rn(__dsub_rn(pz, lz), voxel);
      cx = min(max(cx, 0LL), dx - 1); cy = min(max(cy, 0LL), dy - 1); cz = min(max(cz, 0LL), dz - 1);
      v = cx * dy * dz + cy * dz + cz;
      const double ccx = __dadd_rn(lx, __dmul_rn((double)cx + 0.5, voxel));
      const double ccy = __dadd_rn(ly, __dmul_rn((double)cy + 0.5, voxel));
      const double ccz = __dadd_rn(lz, __dmul_rn((double)cz + 0.5, voxel));
      code = (unsigned long long)__double_as_longlong(dist3(px, py, pz, ccx, ccy, ccz));
      vid[i] = v;
      dcode[i] = code;
    }
    const unsigned group = __match_any_sync(0xffffffffu, (int)v);           // lanes of this warp in the same voxel
    const unsigned hi = (unsigned)(code >> 32), lo = (unsigned)code;
    const unsigned m_hi = __reduce_min_sync(group, hi);
    const unsigned m_lo = __reduce_min_sync(group, hi == m_hi ? lo : 0xffffffffu);
    if (live && (threadIdx.x & 31) == (unsigned)(__ffs(group) - 1))
      atomicMin(&s_tab[v], ((unsigned long long)m_hi << 32) | m_lo);
  }
  __syncthreads();
  for (int v = threadIdx.x; v < n_vox; v += blockDim.x) {
    const unsigned long long m = s_tab[v];
    if (m != kEmptyU64) atomicMin(tab_d + v, m);
  }
}

__global__ void __launch_bounds__(256)
voxel_pick_kernel(long long N, const long long* __restrict__ vid, const unsigned long long* __restrict__ dcode,
                  const unsigned long long* __restrict__ tab_d, unsigned long long* __restrict__ tab_i) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
    const long long v = vid[i];
    if (dcode[i] == tab_d[v]) atomicMin(tab_i + v, (unsigned long long)i);          // first index on ties
  }
}

__global__ void __launch_bounds__(kScanBlock)
voxel_count_kernel(long long n_vox, const unsigned long long* __restrict__ tab_i, long long* __restrict__ counts) {
  const long long v = (long long)blockIdx.x * kScanBlock + threadIdx.x;
  const int occ = (v < n_vox) && (tab_i[v] != kEmptyU64);
  const int c = __syncthreads_count(occ);
  if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

// exclusive scan of counts[0..nb) in place (single CTA), total -> *out_count
__global__ void __launch_bounds__(1024)
voxel_scan_kernel(long long nb, long long* __restrict__ counts, long long* __restrict__ out_count) {
  __shared__ long long sh[1024];
  const int tid = threadIdx.x;
  const long long per = (nb + 1023) / 1024;
  const long long b0 = tid * per, b1 = min(nb, b0 + per);
  long long s = 0;
  for (long long b = b0; b < b1; ++b) s += counts[b];
  sh[tid] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    long long t = (tid >= o) ? sh[tid - o] : 0;
    __syncthreads();
    sh[tid] += t;
    __syncthreads();
  }
  long long run = sh[tid] - s;                 // exclusive prefix of this thread's chunk
  for (long long b = b0; b < b1; ++b) { const long long c = counts[b]; counts[b] = run; run += c; }
  if (tid == 1023) *out_count = sh[1023];
}

__global__ void __launch_bounds__(kScanBlock)
voxel_scatter_kernel(long long n_vox, const unsigned long long* __restrict__ tab_i,
                     const long long* __restrict__ offsets, long long* __restrict__ out_idx, long long max_out) {
  __shared__ int warp_cnt[kScanBlock / 32];
  const long long v = (long long)blockIdx.x * kScanBlock + threadIdx.x;
  const unsigned long long pick = (v < n_vox) ? tab_i[v] : kEmptyU64;
  const bool occ = pick != kEmptyU64;
  const unsigned ballot = __ballot_sync(0xffffffffu, occ);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) warp_cnt[warp] = __popc(ballot);
  __syncthreads();
  int before = 0;
  for (int w = 0; w < warp; ++w) before += warp_cnt[w];
  if (occ) {
    const long long pos = offsets[blockIdx.x] + before + __popc(ballot & ((1u << lane) - 1u));
    if (pos < max_out) out_idx[pos] = (long long)pick;
  }
}

int stream_grid(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = (long long)ep::sm_count() * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

struct FpsPlan { bool onchip; int grid; long long per_block; size_t smem; };

int plan_fps(long long N, FpsPlan* p) {
  static int coop_blocks_onchip = -1, coop_blocks_global = -1;
  const size_t smem_full = (size_t)kFpsSmemPoints * 32;
  if (coop_blocks_onchip < 0) {
    int dev = 0, coop = 0;
    EP_CUDA_CHECK(cudaGetDevice(&dev));
    EP_CUDA_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) { ep::set_error("device does not support cooperative launch"); return EP_ERR_UNSUPPORTED; }
    EP_CUDA_CHECK(cudaFuncSetAttribute(fps_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_full));
    int per_sm = 0;
    EP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fps_kernel<true>, kFpsThreads, smem_full));
    coop_blocks_onchip = per_sm * ep::sm_count();
    EP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fps_kernel<false>, kFpsThreads, 0));
    coop_blocks_global = per_sm * ep::sm_count();
    if (coop_blocks_global > kMaxFpsBlocks) coop_blocks_global = kMaxFpsBlocks;
  }
  const long long onchip_cap = (long long)coop_blocks_onchip * kFpsSmemPoints;
  if (coop_blocks_onchip > 0 && N <= onchip_cap) {
    p->onchip = true;
    long long g = ep::ceil_div64(N, kFpsThreads);             // at least one point per thread before adding CTAs
    if (g > coop_blocks_onchip) g = coop_blocks_onchip;
    if (g < 1) g = 1;
    p->grid = (int)g;
    p->per_block = ep::ceil_div64(N, g);
    p->smem = (size_t)p->per_block * 32;
  } else {
    if (coop_blocks_global <= 0) { ep::set_error("fps: no co-resident CTAs available"); return EP_ERR_UNSUPPORTED; }
    p->onchip = false;
    p->grid = coop_blocks_global;
    p->per_block = ep::ceil_div64(N, p->grid);
    p->smem = 0;
  }
  return EP_OK;
}

}  // namespace

extern "C" {

size_t ep_fps_workspace_bytes(int64_t n_points) {
  if (n_points <= 0) return 0;
  return sizeof(FpsRecord) * 2 * kMaxFpsBlocks + sizeof(double) * (size_t)n_points;
}

int ep_fps_f64(int64_t n_points, const double* pts, int n_samples, int64_t start, int64_t* out_order,
               void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n_points > 0 && n_samples > 0, "bad size");
  EP_REQUIRE(n_samples <= n_points, "n_samples > n_points");
  EP_REQUIRE(start >= 0 && start < n_points, "start out of range");
  EP_REQUIRE(pts && out_order && workspace, "null pointer");
  if (workspace_bytes < ep_fps_workspace_bytes(n_points)) {
    ep::set_error("ep_fps_f64: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  FpsPlan plan;
  int rc = plan_fps(n_points, &plan);
  if (rc != EP_OK) return rc;
  FpsRecord* records = static_cast<FpsRecord*>(workspace);
  double* gdist = reinterpret_cast<double*>(records + 2 * kMaxFpsBlocks);
  long long N = n_points, st = start, per_block = plan.per_block;
  long long* out = reinterpret_cast<long long*>(out_order);
  void* args[] = {&N, (void*)&pts, &n_samples, &st, &per_block, &gdist, &out, &records};
  if (plan.onchip) {
    EP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)fps_kernel<true>, dim3(plan.grid), dim3(kFpsThreads), args,
                                              plan.smem, ep::as_stream(stream)));
  } else {
    EP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)fps_kernel<false>, dim3(plan.grid), dim3(kFpsThreads), args,
                                              0, ep::as_stream(stream)));
  }
  return EP_OK;
}

int ep_fps_f64_host(int64_t n_points, const double* pts_host, int n_samples, int64_t start,
                    int64_t* out_order_host) {
  EP_REQUIRE(n_points > 0 && n_samples > 0 && pts_host && out_order_host, "bad argument");
  double* d_pts = nullptr;
  int64_t* d_out = nullptr;
  void* d_ws = nullptr;
  const size_t ws = ep_fps_workspace_bytes(n_points);
  int rc = EP_OK;
  cudaError_t e;
  if ((e = cudaMalloc(&d_pts, sizeof(double) * 3 * (size_t)n_points)) != cudaSuccess ||
      (e = cudaMalloc(&d_out, sizeof(int64_t) * (size_t)n_samples)) != cudaSuccess ||
      (e = cudaMalloc(&d_ws, ws)) != cudaSuccess) {
    rc = ep::cuda_fail(e, "cudaMalloc");
  }
  if (rc == EP_OK && (e = cudaMemcpy(d_pts, pts_host, sizeof(double) * 3 * (size_t)n_points, cudaMemcpyHostToDevice)) != cudaSuccess)
    rc = ep::cuda_fail(e, "cudaMemcpy H2D");
  if (rc == EP_OK) rc = ep_fps_f64(n_points, d_pts, n_samples, start, d_out, d_ws, ws, nullptr);
  if (rc == EP_OK && (e = cudaMemcpy(out_order_host, d_out, sizeof(int64_t) * (size_t)n_samples, cudaMemcpyDeviceToHost)) != cudaSuccess)
    rc = ep::cuda_fail(e, "cudaMemcpy D2H");
  cudaFree(d_pts); cudaFree(d_out); cudaFree(d_ws);
  return rc;
}

int ep_bounds_f64(int64_t n_points, const double* pts, double* lo_hi, ep_stream_t stream) {
  EP_REQUIRE(n_points > 0 && pts && lo_hi, "bad argument");
  cudaStream_t st = ep::as_stream(stream);
  double* parts = nullptr;
  EP_CUDA_CHECK(cudaGetSymbolAddress(reinterpret_cast<void**>(&parts), g_bounds_parts));
  int grid = (int)ep::ceil_div64(n_points, 256);
  if (grid > kBoundsBlocks) grid = kBoundsBlocks;
  bounds_partial_kernel<<<grid, 256, 0, st>>>(n_points, pts, parts);
  EP_LAUNCH_CHECK("bounds_partial_kernel");
  bounds_final_kernel<<<1, 32, 0, st>>>(grid, lo_hi);
  EP_LAUNCH_CHECK("bounds_final_kernel");
  return EP_OK;
}

size_t ep_voxel_workspace_bytes(int64_t n_points, int64_t n_voxels) {
  if (n_points <= 0 || n_voxels <= 0) return 0;
  const size_t nb = (size_t)ep::ceil_div64(n_voxels, kScanBlock);
  return 8 * (2 * (size_t)n_voxels + 2 * (size_t)n_points + nb + 1);
}

int ep_voxel_select_f64(int64_t n_points, const double* pts, const double* lo, double voxel, const int64_t* dims,
                        int64_t* out_idx, int64_t max_out, int64_t* out_count, void* workspace,
                        size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n_points > 0 && pts && lo && dims && out_idx && out_count && workspace, "bad argument");
  EP_REQUIRE(voxel > 0.0 && dims[0] > 0 && dims[1] > 0 && dims[2] > 0, "bad voxel grid");
  const long long n_vox = dims[0] * dims[1] * dims[2];
  EP_REQUIRE(n_vox > 0 && n_vox < (1LL << 40), "voxel grid too large");
  if (workspace_bytes < ep_voxel_workspace_bytes(n_points, n_vox)) {
    ep::set_error("ep_voxel_select_f64: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  cudaStream_t st = ep::as_stream(stream);
  unsigned long long* tab_d = static_cast<unsigned long long*>(workspace);
  unsigned long long* tab_i = tab_d + n_vox;
  long long* vid = reinterpret_cast<long long*>(tab_i + n_vox);
  unsigned long long* dcode = reinterpret_cast<unsigned long long*>(vid + n_points);
  long long* counts = reinterpret_cast<long long*>(dcode + n_points);
  const long long nb = ep::ceil_div64(n_vox, kScanBlock);
  EP_REQUIRE(nb < 0x7fffffffLL, "voxel grid too large");
  voxel_init_kernel<<<stream_grid(n_vox, 256), 256, 0, st>>>(n_vox, tab_d, tab_i);
  EP_LAUNCH_CHECK("voxel_init_kernel");
  if (n_vox <= kVoxelSmemMax) {
    int grid = 2 * ep::sm_count();
    const long long need = ep::ceil_div64(n_points, 256);
    if (need < grid) grid = (int)need;
    voxel_assign_small_kernel<<<grid, 256, sizeof(unsigned long long) * (size_t)n_vox, st>>>(
        n_points, pts, lo[0], lo[1], lo[2], voxel, dims[0], dims[1], dims[2], vid, dcode, tab_d, (int)n_vox);
    EP_LAUNCH_CHECK("voxel_assign_small_kernel");
  } else {
    voxel_assign_kernel<<<stream_grid(n_points, 256), 256, 0, st>>>(n_points, pts, lo[0], lo[1], lo[2], voxel, dims[0],
                                                                   dims[1], dims[2], vid, dcode, tab_d);
    EP_LAUNCH_CHECK("voxel_assign_kernel");
  }
  voxel_pick_kernel<<<stream_grid(n_points, 256), 256, 0, st>>>(n_points, vid, dcode, tab_d, tab_i);
  EP_LAUNCH_CHECK("voxel_pick_kernel");
  voxel_count_kernel<<<(unsigned)nb, kScanBlock, 0, st>>>(n_vox, tab_i, counts);
  EP_LAUNCH_CHECK("voxel_count_kernel");
  voxel_scan_kernel<<<1, 1024, 0, st>>>(nb, counts, reinterpret_cast<long long*>(out_count));
  EP_LAUNCH_CHECK("voxel_scan_kernel");
  voxel_scatter_kernel<<<(unsigned)nb, kScanBlock, 0, st>>>(n_vox, tab_i, counts, reinterpret_cast<long long*>(out_idx),
                                                           max_out);
  EP_LAUNCH_CHECK("voxel_scatter_kernel");
  return EP_OK;
}

int ep_voxel_select_f64_host(int64_t n_points, const double* pts_host, const double* lo, double voxel,
                             const int64_t* dims, int64_t* out_idx_host, int64_t max_out, int64_t* out_count_host) {
  EP_REQUIRE(n_points > 0 && pts_host && lo && dims && out_idx_host && out_count_host && max_out > 0, "bad argument");
  const long long n_vox = dims[0] * dims[1] * dims[2];
  const size_t ws = ep_voxel_workspace_bytes(n_points, n_vox);
  double* d_pts = nullptr;
  int64_t* d_out = nullptr;
  int64_t* d_cnt = nullptr;
  void* d_ws = nullptr;
  int rc = EP_OK;
  cudaError_t e;
  if ((e = cudaMalloc(&d_pts, sizeof(double) * 3 * (size_t)n_points)) != cudaSuccess ||
      (e = cudaMalloc(&d_out, sizeof(int64_t) * (size_t)max_out)) != cudaSuccess ||
      (e = cudaMalloc(&d_cnt, sizeof(int64_t))) != cudaSuccess || (e = cudaMalloc(&d_ws, ws)) != cudaSuccess) {
    rc = ep::cuda_fail(e, "cudaMalloc");
  }
  if (rc == EP_OK && (e = cudaMemcpy(d_pts, pts_host, sizeof(double) * 3 * (size_t)n_points, cudaMemcpyHostToDevice)) != cudaSuccess)
    rc = ep::cuda_fail(e, "cudaMemcpy H2D");
  if (rc == EP_OK) rc = ep_voxel_select_f64(n_points, d_pts, lo, voxel, dims, d_out, max_out, d_cnt, d_ws, ws, nullptr);
  if (rc == EP_OK && (e = cudaMemcpy(out_count_host, d_cnt, sizeof(int64_t), cudaMemcpyDeviceToHost)) != cudaSuccess)
    rc = ep::cuda_fail(e, "cudaMemcpy D2H count");
  if (rc == EP_OK) {
    const int64_t m = *out_count_host < max_out ? *out_count_host : max_out;
    if (m > 0 && (e = cudaMemcpy(out_idx_host, d_out, sizeof(int64_t) * (size_t)m, cudaMemcpyDeviceToHost)) != cudaSuccess)
      rc = ep::cuda_fail(e, "cudaMemcpy D2H idx");
  }
  cudaFree(d_pts); cudaFree(d_out); cudaFree(d_cnt); cudaFree(d_ws);
  return rc;
}

}  // extern "C"
