// Learnable per-mode scales of the AdaptiveCorrector and the smoothness term on the correction
// (delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4, `train_gnn`: corr = net(h) * mode_scales,
// loss += w * sum(corr * (L corr)) / (n k)).
//
//   forward   U_pred = U_base + sigma * (c o s)                          (c: raw MLP output, s: k scales)
//   backward  g = dL/dcorr left by the eigen-loss backward (sigma already applied), w2 = 2 w / (n_global k)
//             dc_ij = s_j g_ij + w2 s_j^2 (K c)_ij                          (written over g)
//             ds_j  = sum_i c_ij g_ij + w2 s_j P_j,  P_j = sum_i c_ij (K c)_ij
//             L_sc  = w / (n_global k) sum_j s_j^2 P_j                     (K (c o s) = (K c) o s, K symmetric)
//
// Both kernels walk the rows with a fixed (row lane, column unit) assignment per thread, so every thread keeps its
// columns' scales in registers and the backward accumulates its column sums without shuffles.  A column unit is a
// float4 when k % 4 == 0 and every row start is 16-byte aligned, else one float.  The backward's column sums are fp64
// (products of two fp32 values are exact in fp64), written per CTA and reduced by one CTA in a fixed order: the result
// does not depend on timing.  Kept in its own translation unit so that the other kernels' code is untouched.
#include "ep_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kBwdMaxBlocks = 1024;             // fixed cap: the workspace size depends on k only
constexpr int kReduceThreads = 1024;

struct Layout {
  int units;       // column units per row (k / 4 or k)
  int rows;        // rows per CTA pass (kThreads / units)
};

inline Layout layout_for(int k, bool vec) {
  Layout L;
  L.units = vec ? k / 4 : k;
  L.rows = kThreads / L.units;
  return L;
}

template <int V>
struct Vec;
template <>
struct Vec<4> {
  using T = float4;
  __device__ static float get(const T& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
  __device__ static void set(T& v, int i, float x) {
    if (i == 0) v.x = x; else if (i == 1) v.y = x; else if (i == 2) v.z = x; else v.w = x;
  }
};
template <>
struct Vec<1> {
  using T = float;
  __device__ static float get(const T& v, int) { return v; }
  __device__ static void set(T& v, int, float x) { v = x; }
};

// U_pred = U_base + sigma * (c o s), rounded as ep_axpy_out_f32 rounds (product, then sum; no FMA)
template <int V>
__global__ void __launch_bounds__(kThreads)
mode_scale_fwd_kernel(int n, int k, int units, int rows, const float* __restrict__ c, int ldc,
                      const float* __restrict__ U_base, int ldb, const float* __restrict__ s, float sigma,
                      const float* __restrict__ sigma_dev, float* __restrict__ U_pred, int ldu) {
  using T = typename Vec<V>::T;
  const int u = threadIdx.x % units, lane = threadIdx.x / units;
  if (lane >= rows) return;
  const float sg = sigma_dev ? *sigma_dev : sigma;
  float sj[V];
#pragma unroll
  for (int v = 0; v < V; ++v) sj[v] = s ? s[u * V + v] : 1.0f;
  const int col = u * V;
  for (long long r = (long long)blockIdx.x * rows + lane; r < n; r += (long long)gridDim.x * rows) {
    const T cv = *reinterpret_cast<const T*>(c + r * ldc + col);
    const T bv = *reinterpret_cast<const T*>(U_base + r * ldb + col);
    T o;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const float cs = s ? __fmul_rn(Vec<V>::get(cv, v), sj[v]) : Vec<V>::get(cv, v);
      Vec<V>::set(o, v, __fadd_rn(Vec<V>::get(bv, v), __fmul_rn(sg, cs)));
    }
    *reinterpret_cast<T*>(U_pred + r * ldu + col) = o;
  }
}

// Phase 1 of the backward: dc over g in place, per-CTA fp64 column sums of c g and c Kc.
// parts layout: [2k][gridDim.x], entry (j, b) = sum c g of column j in CTA b, entry (k + j, b) = sum c Kc.
template <int V>
__global__ void __launch_bounds__(kThreads)
mode_scale_bwd_kernel(int n, int k, int units, int rows, const float* __restrict__ c, int ldc,
                      const float* __restrict__ Kc, int ldkc, const float* __restrict__ s, float w2,
                      float* __restrict__ g, int ldd, double* __restrict__ parts) {
  using T = typename Vec<V>::T;
  __shared__ double sh[2 * kThreads * V];       // [lane][unit][V] for c g, then for c Kc
  const int u = threadIdx.x % units, lane = threadIdx.x / units;
  const bool active = lane < rows;
  const int col = u * V;
  float sj[V], aj[V];
  double scg[V], sck[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
    sj[v] = (active && s) ? s[col + v] : 1.0f;
    aj[v] = w2 * sj[v] * sj[v];
    scg[v] = 0.0;
    sck[v] = 0.0;
  }
  const bool rewrite = (s != nullptr) || (Kc != nullptr);
  if (active) {
    for (long long r = (long long)blockIdx.x * rows + lane; r < n; r += (long long)gridDim.x * rows) {
      const T cv = *reinterpret_cast<const T*>(c + r * ldc + col);
      T gv = *reinterpret_cast<const T*>(g + r * ldd + col);
      T kv;
      if (Kc) kv = *reinterpret_cast<const T*>(Kc + r * ldkc + col);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float cx = Vec<V>::get(cv, v), gx = Vec<V>::get(gv, v);
        scg[v] += (double)cx * (double)gx;
        float d = sj[v] * gx;
        if (Kc) {
          const float kx = Vec<V>::get(kv, v);
          sck[v] += (double)cx * (double)kx;
          d = fmaf(aj[v], kx, d);
        }
        Vec<V>::set(gv, v, d);
      }
      if (rewrite) *reinterpret_cast<T*>(g + r * ldd + col) = gv;
    }
  }
  // CTA reduction in a fixed order: column j = col + v sums its row lanes 0, 1, ..., rows - 1
  const int width = units * V;                   // == k
  if (active) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      sh[lane * width + col + v] = scg[v];
      sh[kThreads * V + lane * width + col + v] = sck[v];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * k; e += kThreads) {
    const int half = e >= k, j = e - half * k;
    const double* base = sh + half * kThreads * V;
    double t = 0.0;
    for (int l = 0; l < rows; ++l) t += base[l * width + j];
    parts[(size_t)e * gridDim.x + blockIdx.x] = t;
  }
}

// Phase 2: one CTA.  Warp q reduces the pairs e = q, q + 32, ...: lane l sums CTAs l, l + 32, ... in order, then a
// fixed shuffle tree.  Then ds (written or accumulated into grad_s) and L_sc into loss_acc[8] and [5].
__global__ void __launch_bounds__(kReduceThreads)
mode_scale_reduce_kernel(int nblocks, int k, const double* __restrict__ parts, const float* __restrict__ s,
                         double w, double n_global, int has_kc, float* __restrict__ grad_s, int accumulate,
                         double* __restrict__ loss_acc) {
  __shared__ double tot[2 * 256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int e = warp; e < 2 * k; e += kReduceThreads / 32) {
    double t = 0.0;
    for (int b = lane; b < nblocks; b += 32) t += parts[(size_t)e * nblocks + b];
    t = ep::warp_sum(t);
    if (lane == 0) tot[e] = t;
  }
  __syncthreads();
  const double w2 = 2.0 * w / (n_global * (double)k);
  if (grad_s != nullptr) {
    for (int j = threadIdx.x; j < k; j += kReduceThreads) {
      const double sj = (double)s[j];
      double ds = tot[j];
      if (has_kc) ds += w2 * sj * tot[k + j];
      grad_s[j] = accumulate ? grad_s[j] + (float)ds : (float)ds;
    }
  }
  if (threadIdx.x == 0 && has_kc && loss_acc != nullptr) {
    double L = 0.0;
    for (int j = 0; j < k; ++j) {
      const double sj = s ? (double)s[j] : 1.0;
      L += sj * sj * tot[k + j];
    }
    L *= w / (n_global * (double)k);
    loss_acc[8] += L;
    loss_acc[5] += L;
  }
}

bool rows_vec4(int k, const void* p, int ld) { return k % 4 == 0 && ld % 4 == 0 && ep::aligned16(p); }

int grid_for(int n, int rows, int cap) {
  long long g = ((long long)n + rows - 1) / rows;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" {

int ep_mode_scale_fwd_f32(int n, int k, const float* c, int ldc, const float* U_base, int ldb, const float* s,
                          float sigma, const float* sigma_dev, float* U_pred, int ldu, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0, "bad size");
  EP_REQUIRE(k <= 256, "k > 256 not supported");
  if (n == 0) return EP_OK;
  EP_REQUIRE(c && U_base && U_pred, "null pointer");
  EP_REQUIRE(ldc >= k && ldb >= k && ldu >= k, "leading dimension < k");
  cudaStream_t st = ep::as_stream(stream);
  const bool vec = rows_vec4(k, c, ldc) && rows_vec4(k, U_base, ldb) && rows_vec4(k, U_pred, ldu);
  const Layout L = layout_for(k, vec);
  const int grid = grid_for(n, L.rows, ep::sm_count() * 8);
  if (vec)
    mode_scale_fwd_kernel<4><<<grid, kThreads, 0, st>>>(n, k, L.units, L.rows, c, ldc, U_base, ldb, s, sigma, sigma_dev,
                                                        U_pred, ldu);
  else
    mode_scale_fwd_kernel<1><<<grid, kThreads, 0, st>>>(n, k, L.units, L.rows, c, ldc, U_base, ldb, s, sigma, sigma_dev,
                                                        U_pred, ldu);
  EP_LAUNCH_CHECK("mode_scale_fwd_kernel");
  return EP_OK;
}

size_t ep_mode_scale_bwd_workspace_bytes(int k) {
  if (k <= 0 || k > 256) return 0;
  return sizeof(double) * 2 * (size_t)k * kBwdMaxBlocks;
}

int ep_mode_scale_bwd_f32(int n, int k, double n_global, const float* c, int ldc, const float* Kc, int ldkc,
                          const float* s, float w_smooth_corr, float* dcorr, int ldd, float* grad_s, int accumulate,
                          double* loss_acc, void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0, "bad size");
  EP_REQUIRE(k <= 256, "k > 256 not supported");
  EP_REQUIRE(n_global > 0, "n_global must be positive");
  EP_REQUIRE(workspace, "null workspace");
  EP_REQUIRE(s || !grad_s, "grad_s needs the scales s");
  EP_REQUIRE(n == 0 || (c && dcorr), "null pointer");
  EP_REQUIRE(ldc >= k && ldd >= k && (!Kc || ldkc >= k), "leading dimension < k");
  if (workspace_bytes < ep_mode_scale_bwd_workspace_bytes(k)) {
    ep::set_error("ep_mode_scale_bwd_f32: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  cudaStream_t st = ep::as_stream(stream);
  const bool vec = rows_vec4(k, c, ldc) && rows_vec4(k, dcorr, ldd) && (!Kc || rows_vec4(k, Kc, ldkc));
  const Layout L = layout_for(k, vec);
  // one wave of resident CTAs (64 registers for the float4 form: 4 per SM), never more than the workspace holds
  static int resident[2] = {0, 0};
  int& per_sm = resident[vec ? 1 : 0];
  if (per_sm == 0) {
    EP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        &per_sm, vec ? mode_scale_bwd_kernel<4> : mode_scale_bwd_kernel<1>, kThreads, 0));
    if (per_sm < 1) per_sm = 1;
  }
  const int cap = per_sm * ep::sm_count() < kBwdMaxBlocks ? per_sm * ep::sm_count() : kBwdMaxBlocks;
  const int grid = n > 0 ? grid_for(n, L.rows, cap) : 0;
  const float w2 = (float)(2.0 * (double)w_smooth_corr / (n_global * (double)k));
  double* parts = static_cast<double*>(workspace);
  if (grid > 0) {
    if (vec)
      mode_scale_bwd_kernel<4><<<grid, kThreads, 0, st>>>(n, k, L.units, L.rows, c, ldc, Kc, ldkc, s, w2, dcorr, ldd,
                                                          parts);
    else
      mode_scale_bwd_kernel<1><<<grid, kThreads, 0, st>>>(n, k, L.units, L.rows, c, ldc, Kc, ldkc, s, w2, dcorr, ldd,
                                                          parts);
    EP_LAUNCH_CHECK("mode_scale_bwd_kernel");
  }
  mode_scale_reduce_kernel<<<1, kReduceThreads, 0, st>>>(grid, k, parts, s, (double)w_smooth_corr, n_global,
                                                         Kc != nullptr, grad_s, accumulate, loss_acc);
  EP_LAUNCH_CHECK("mode_scale_reduce_kernel");
  return EP_OK;
}

}  // extern "C"
