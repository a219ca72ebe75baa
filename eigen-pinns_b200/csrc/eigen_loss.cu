// Eigen-loss kernels: Rayleigh quotient, residual, Gram / orthonormality (forward partials,
// finalisation, analytic backward).  Reference arithmetic: src/multigrid_model.py:291-348.
//
// Data layout: U, KU, MU are row-major n x k fp32 in HBM (the partials kernel also takes fp64 for the notebook
// variants).  The four column sums behind the Rayleigh
// quotient and the one-pass residual expansion sum(KU^2) - 2 lam sum(KU MU) + lam^2 sum(MU^2) are
// accumulated in fp64 from the first product on (exact products, ~1e-16 relative sums), so the
// expansion stays accurate near convergence where the residual is a tiny difference of large terms.
// The Gram matrix is accumulated in fp32 for at most four 32-row tiles and then folded into fp64.
// Algorithmic traffic of the partials kernel: 12 n k bytes read, flops 2 n k^2 + 8 n k.
#include "ep_common.cuh"
#include "eigen_coef.cuh"

namespace {

constexpr int kPartialThreads = 256;
__device__ __forceinline__ bool ep_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__host__ __device__ inline int partials_len(int k) { return k * k + 5 * k; }   // G | num | sKK | sKM | sMM | colsum(MU)

// rows per tile of the partials kernel: the three R x KP tiles take at most 24 KB of static shared memory
// (fp32: R = 32, 16 at KP = 128; fp64: R = 32, 32, 16, 8 for KP = 16 ... 128)
template <typename T>
__host__ __device__ constexpr int partial_rows(int kp) {
  return 8192 / (kp * (int)sizeof(T)) < 32 ? 8192 / (kp * (int)sizeof(T)) : 32;
}

// 16-byte vector of the partials kernel's input type (global loads and shared-memory reads)
template <typename T> struct Vec16;
template <> struct Vec16<float> {
  using type = float4;
  static constexpr int N = 4;
  __device__ static float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ static float4 make(const float (&t)[4]) { return make_float4(t[0], t[1], t[2], t[3]); }
  __device__ static void split(float4 v, float* t) { t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w; }
};
template <> struct Vec16<double> {
  using type = double2;
  static constexpr int N = 2;
  __device__ static double2 zero() { return make_double2(0.0, 0.0); }
  __device__ static double2 make(const double (&t)[2]) { return make_double2(t[0], t[1]); }
  __device__ static void split(double2 v, double* t) { t[0] = v.x; t[1] = v.y; }
};

inline int partial_blocks(int n, int rows_per_tile) {
  int tiles = ep::ceil_div(n, rows_per_tile);
  int cap = ep::sm_count() * 4;
  int g = tiles < cap ? tiles : cap;
  return g < 1 ? 1 : g;
}

// Gram / column-sum partials.  KP = padded column count; each thread owns a TG x TG block of the Gram
// matrix, (KP/TG)^2 threads form a sub-group and the 256 / (KP/TG)^2 sub-groups take alternate rows of the
// tile, so every FMA group costs two 16-byte shared-memory reads (TG = 4: 16 FMA per 2 LDS.128).
// T = double (the notebook variants) accumulates the Gram matrix straight in fp64: there is no fp32 stage to fold.
template <typename T, int KP, int TG>
__global__ void __launch_bounds__(kPartialThreads)
eigen_partials_kernel(int n, int k, const T* __restrict__ U, int ldu, const T* __restrict__ KU,
                      const T* __restrict__ MU, int ld, double* __restrict__ block_out) {
  constexpr int TPD = KP / TG;
  constexpr int NT = TPD * TPD;
  constexpr int NSG = kPartialThreads / NT;
  constexpr int R = partial_rows<T>(KP);
  constexpr int CPL = (KP + 31) / 32;
  constexpr bool kFold = sizeof(T) == 4;          // fp32 input: fp32 Gram tiles folded into fp64
  constexpr int FLUSH = 4;                       // fold fp32 -> fp64 every FLUSH tiles
  static_assert(NT * NSG == kPartialThreads && NSG >= 1, "bad tiling");
  __shared__ __align__(16) T Us[R][KP];
  __shared__ __align__(16) T KUs[R][KP];
  __shared__ __align__(16) T MUs[R][KP];
  using V = typename Vec16<T>::type;
  constexpr int VW = Vec16<T>::N;
  __shared__ double red[(NSG > 1) ? KP * KP : 8 * KP];

  const int tid = threadIdx.x;
  const int sg = tid / NT, tin = tid % NT;
  const int ty = tin / TPD, tx = tin % TPD;
  const int warp = tid >> 5, lane = tid & 31;

  double g64[TG][TG];
  float g32[TG][TG];
  double c64[5][CPL];
#pragma unroll
  for (int i = 0; i < TG; ++i)
#pragma unroll
    for (int j = 0; j < TG; ++j) { g64[i][j] = 0.0; g32[i][j] = 0.f; }
#pragma unroll
  for (int q = 0; q < 5; ++q)
#pragma unroll
    for (int c = 0; c < CPL; ++c) c64[q][c] = 0.0;

  const int n_tiles = (n + R - 1) / R;
  int since_flush = 0;
  // Register-staged double buffering: the next tile's global loads are in flight while this tile is reduced.
  constexpr int VPT = (R * KP / VW + kPartialThreads - 1) / kPartialThreads;     // 16-byte vectors per thread per array
  const bool vec_ok = (k % VW == 0) && (ldu % VW == 0) && (ld % VW == 0) && ep_aligned16(U) && ep_aligned16(KU) && ep_aligned16(MU);
  V pu[VPT], pk[VPT], pm[VPT];
  auto prefetch = [&](int tile) {
    const int row0 = tile * R;
#pragma unroll
    for (int v = 0; v < VPT; ++v) {
      const int e4 = tid + v * kPartialThreads;          // vector index inside the R x KP tile
      const int r = e4 / (KP / VW), c = (e4 - r * (KP / VW)) * VW;
      const int row = row0 + r;
      V zu = Vec16<T>::zero(), zk = zu, zm = zu;
      if (r < R && row < n && c < k) {
        if (vec_ok) {
          zu = __ldg(reinterpret_cast<const V*>(U + (size_t)row * ldu + c));
          zk = __ldg(reinterpret_cast<const V*>(KU + (size_t)row * ld + c));
          zm = __ldg(reinterpret_cast<const V*>(MU + (size_t)row * ld + c));
        } else {
          T tu[VW], tk[VW], tm[VW];
#pragma unroll
          for (int j = 0; j < VW; ++j) {
            const bool ok = (c + j) < k;
            tu[j] = ok ? __ldg(U + (size_t)row * ldu + c + j) : T(0);
            tk[j] = ok ? __ldg(KU + (size_t)row * ld + c + j) : T(0);
            tm[j] = ok ? __ldg(MU + (size_t)row * ld + c + j) : T(0);
          }
          zu = Vec16<T>::make(tu);
          zk = Vec16<T>::make(tk);
          zm = Vec16<T>::make(tm);
        }
      }
      pu[v] = zu; pk[v] = zk; pm[v] = zm;
    }
  };
  if ((int)blockIdx.x < n_tiles) prefetch(blockIdx.x);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    __syncthreads();
#pragma unroll
    for (int v = 0; v < VPT; ++v) {
      const int e4 = tid + v * kPartialThreads;
      const int r = e4 / (KP / VW), c = (e4 - r * (KP / VW)) * VW;
      if (r < R) {
        *reinterpret_cast<V*>(&Us[r][c]) = pu[v];
        *reinterpret_cast<V*>(&KUs[r][c]) = pk[v];
        *reinterpret_cast<V*>(&MUs[r][c]) = pm[v];
      }
    }
    __syncthreads();
    if (tile + (int)gridDim.x < n_tiles) prefetch(tile + gridDim.x);
#pragma unroll 2
    for (int r = sg; r < R; r += NSG) {
      T a[TG], b[TG];
#pragma unroll
      for (int i = 0; i < TG; i += VW) {
        Vec16<T>::split(*reinterpret_cast<const V*>(&Us[r][ty * TG + i]), a + i);
        Vec16<T>::split(*reinterpret_cast<const V*>(&MUs[r][tx * TG + i]), b + i);
      }
#pragma unroll
      for (int i = 0; i < TG; ++i)
#pragma unroll
        for (int j = 0; j < TG; ++j) {
          if constexpr (kFold) g32[i][j] = fmaf(a[i], b[j], g32[i][j]);
          else                 g64[i][j] = fma(a[i], b[j], g64[i][j]);
        }
    }
    if (kFold && ++since_flush == FLUSH) {
      since_flush = 0;
#pragma unroll
      for (int i = 0; i < TG; ++i)
#pragma unroll
        for (int j = 0; j < TG; ++j) { g64[i][j] += (double)g32[i][j]; g32[i][j] = 0.f; }
    }
    // column sums: warp w owns rows w, w+8, ...; lane owns columns lane, lane+32, ...
#pragma unroll
    for (int cc = 0; cc < CPL; ++cc) {
      const int c = lane + 32 * cc;
      if (c < KP) {
        // fp64 from the first product on: products of two fp32 values are exact in fp64, so the one-pass
        // expansion sKK - 2 lam sKM + lam^2 sMM keeps ~9 digits even when the residual is 1e-4 of |KU|
        // (near convergence); B200 issues DFMA at half the FFMA rate and this loop is 4 DFMA per 12 bytes.
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0;
        for (int r = warp; r < R; r += kPartialThreads / 32) {
          const double u = (double)Us[r][c], ku = (double)KUs[r][c], mu = (double)MUs[r][c];
          s0 = fma(u, ku, s0);
          s1 = fma(ku, ku, s1);
          s2 = fma(ku, mu, s2);
          s3 = fma(mu, mu, s3);
          s4 += mu;                                  // 1^T M U  (zero-mean term of the notebook variants)
        }
        c64[0][cc] += s0; c64[1][cc] += s1;
        c64[2][cc] += s2; c64[3][cc] += s3; c64[4][cc] += s4;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < TG; ++i)
#pragma unroll
    for (int j = 0; j < TG; ++j)
      if (kFold) g64[i][j] += (double)g32[i][j];

  double* out = block_out + (size_t)blockIdx.x * partials_len(k);
  if (NSG > 1) {                                  // combine the row sub-groups in a fixed order
    for (int s2 = 0; s2 < NSG; ++s2) {
      __syncthreads();
      if (sg == s2) {
#pragma unroll
        for (int i = 0; i < TG; ++i)
#pragma unroll
          for (int j = 0; j < TG; ++j) {
            const int idx = (ty * TG + i) * KP + tx * TG + j;
            red[idx] = (s2 == 0) ? g64[i][j] : red[idx] + g64[i][j];
          }
      }
    }
    __syncthreads();
    for (int e = tid; e < KP * KP; e += kPartialThreads) {
      const int a_ = e / KP, b_ = e - a_ * KP;
      if (a_ < k && b_ < k) out[a_ * k + b_] = red[e];
    }
  } else {
#pragma unroll
    for (int i = 0; i < TG; ++i)
#pragma unroll
      for (int j = 0; j < TG; ++j) {
        const int a_ = ty * TG + i, b_ = tx * TG + j;
        if (a_ < k && b_ < k) out[a_ * k + b_] = g64[i][j];
      }
  }
  for (int q = 0; q < 5; ++q) {
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < CPL; ++cc) {
      const int c = lane + 32 * cc;
      if (c < KP) red[warp * KP + c] = c64[q][cc];
    }
    __syncthreads();
    if (tid < k) {
      double s = 0.0;
      for (int w = 0; w < kPartialThreads / 32; ++w) s += red[w * KP + tid];
      out[k * k + q * k + tid] = s;
    }
  }
}

// sum of the per-block partials: one warp per output, lanes stride over the blocks, fixed shuffle tree
__global__ void __launch_bounds__(256)
reduce_partials_kernel(int n_blocks, int len, const double* __restrict__ block_out, double* __restrict__ out) {
  const int e = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (e >= len) return;
  double s = 0.0;
  for (int b = lane; b < n_blocks; b += 32) s += block_out[(size_t)b * len + e];
  s = ep::warp_sum(s);
  if (lane == 0) out[e] = s;
}

__device__ double block_sum_256(double v, double* scratch) {
  v = ep::warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < 8; ++w) s += scratch[w];
  return s;
}

__global__ void __launch_bounds__(256)
eigen_finalize_kernel(int k, double n_global, const double* __restrict__ P, float w_res, float w_orth,
                      int flags, const float* __restrict__ lam_target, float w_trace, float w_order,
                      float w_eigen, float w_mean, float w_smooth, const float* __restrict__ lam_bar_extra,
                      float* __restrict__ lam_out, float* __restrict__ coef, double* __restrict__ loss_acc) {
  __shared__ double s_lam[128];
  __shared__ double scratch[8];
  const int tid = threadIdx.x;
  const bool level0 = (flags & EP_FINALIZE_EIGENVALUE_TERMS) != 0;
  const double* G = P;
  const double* num = P + (size_t)k * k;
  const double* sKK = num + k;
  const double* sKM = sKK + k;
  const double* sMM = sKM + k;
  const double* sMU = sMM + k;                    // column sums of M U
  double res_j = 0.0, lam_j = 0.0, den_j = 1.0;
  if (tid < k) {
    den_j = G[(size_t)tid * k + tid] + 1e-12;
    lam_j = num[tid] / den_j;
    s_lam[tid] = lam_j;
    res_j = sKK[tid] - 2.0 * lam_j * sKM[tid] + lam_j * lam_j * sMM[tid];
    if (res_j < 0.0) res_j = 0.0;
  }
  const double res_sum = block_sum_256(res_j, scratch);
  double orth = 0.0;
  for (int e = tid; e < k * k; e += 256) {
    const int a = e / k, b = e - a * k;
    const double d = G[e] - (a == b ? 1.0 : 0.0);
    orth += d * d;
  }
  const double orth_sum = block_sum_256(orth, scratch);
  const double L_res = res_sum / (n_global * (double)k);
  const double L_orth = orth_sum / (double)k;
  // eigenvalue terms on this level's lambda (reference uses level 0 only)
  double tr = 0.0, ordr = 0.0, eig = 0.0, extra_bar = 0.0;
  if (level0 && tid < k) {
    tr = lam_j / (double)k;
    extra_bar += (double)w_trace / (double)k;
    if (tid + 1 < k) {                       // pair (tid, tid+1): relu(lam_tid - lam_{tid+1})
      const double d = s_lam[tid] - s_lam[tid + 1];
      if (d > 0.0) { ordr += d; extra_bar += (double)w_order; }
    }
    if (tid > 0) {                           // pair (tid-1, tid) contributes -w_order to this lam
      const double d = s_lam[tid - 1] - s_lam[tid];
      if (d > 0.0) extra_bar -= (double)w_order;
    }
    if (lam_target != nullptr) {
      const double d = lam_j - (double)lam_target[tid];
      eig = d * d / (double)k;
      extra_bar += (double)w_eigen * 2.0 * d / (double)k;
    }
  }
  // notebook variants (SURVEY 8a-bis), both zero-weighted in src/:
  //   zero-mean   mean_{j>=1} (1^T M u_j)^2                       (multigrid_gnn_farthest_point_sampling.ipynb cell 0)
  //   smoothness  sum_j u_j^T K u_j / (n k) = sum_j num_j/(n k)    (multigrid_gnn_refine_fixed.ipynb cell 4, U_pred part)
  double mean_j = 0.0, smooth_j = 0.0;
  if (tid < k) {
    if (tid >= 1 && k > 1) mean_j = sMU[tid] * sMU[tid] / (double)(k - 1);
    smooth_j = num[tid] / (n_global * (double)k);
  }
  const double mean_sum = block_sum_256(mean_j, scratch);
  const double smooth_sum = block_sum_256(smooth_j, scratch);
  const double tr_sum = block_sum_256(tr, scratch);
  const double ord_sum = block_sum_256(ordr, scratch);
  const double eig_sum = block_sum_256(eig, scratch);
  const double c_res = 2.0 * (double)w_res / (n_global * (double)k);
  const ep::Coef<float> cf(coef, k);
  double den_bar_j = 0.0;
  if (tid < k) {
    double lam_bar = -c_res * (sKM[tid] - lam_j * sMM[tid]) + extra_bar;
    if (lam_bar_extra != nullptr) lam_bar += (double)lam_bar_extra[tid];
    const double num_bar = lam_bar / den_j + (double)w_smooth / (n_global * (double)k);
    den_bar_j = -lam_bar * lam_j / den_j;
    cf.lam[tid] = (float)lam_j;
    cf.num_bar[tid] = (float)num_bar;
    cf.den_bar[tid] = (float)den_bar_j;
    if (lam_out) lam_out[tid] = (float)lam_j;
    // dL/d(MU)_ij of the zero-mean term is the same for every row i: g_j = 2 w_mean (1^T M u_j) / (k - 1)
    cf.g_mean[tid] = (tid >= 1 && k > 1) ? (float)(2.0 * (double)w_mean * sMU[tid] / (double)(k - 1)) : 0.f;
  }
  __syncthreads();
  const double go = 2.0 * (double)w_orth / (double)k;
  for (int e = tid; e < k * k; e += 256) {
    const int a = e / k, b = e - a * k;
    cf.G_bar[e] = (float)(go * (G[e] - (a == b ? 1.0 : 0.0)));   // den_bar is applied separately (coef)
  }
  if (tid == 0) {
    *cf.c_res = (float)c_res;
    const double t0 = (double)w_res * L_res, t1 = (double)w_orth * L_orth;
    const double t2 = (double)w_trace * tr_sum, t3 = (double)w_order * ord_sum, t4 = (double)w_eigen * eig_sum;
    const double t7 = (double)w_mean * mean_sum, t8 = (double)w_smooth * smooth_sum;
    const double tot = t0 + t1 + t2 + t3 + t4 + t7 + t8;
    if (flags & EP_FINALIZE_OVERWRITE) {      // first level of a step: no separate zero-fill launch
      loss_acc[0] = t0; loss_acc[1] = t1; loss_acc[2] = t2; loss_acc[3] = t3; loss_acc[4] = t4;
      loss_acc[5] = tot; loss_acc[6] = 0.0; loss_acc[7] = t7; loss_acc[8] = t8;
    } else {
      loss_acc[0] += t0; loss_acc[1] += t1; loss_acc[2] += t2; loss_acc[3] += t3; loss_acc[4] += t4;
      loss_acc[5] += tot; loss_acc[7] += t7; loss_acc[8] += t8;
    }
  }
}

// Backward preparation.  Tile = R rows x KP columns, 4 x 4 outputs per thread.
//   KU_bar = R_bar + a U;   MU_bar = -lam R_bar + U Gp;   D = a KU + MU Gp^T
//   with R_bar = c (KU - lam MU),  Gp = G_bar + diag(den_bar).
template <int KP>
__global__ void __launch_bounds__(256)
eigen_bwd_prepare_kernel(int n, int k, const float* __restrict__ U, int ldu, const float* __restrict__ KU,
                         const float* __restrict__ MU, int ld, const float* __restrict__ coef,
                         float* __restrict__ KU_bar, float* __restrict__ MU_bar, float* __restrict__ D) {
  constexpr int R = 4096 / KP;
  constexpr int GP = KP + 4;                    // pitch of the two Gram copies (float4 aligned)
  constexpr int TP = KP + 1;                    // pitch of the row tiles (conflict-free scalar reads)
  extern __shared__ __align__(16) float smem[];
  float* Gs = smem;                             // Gs[m][j]  = Gp[m][j]
  float* GTs = Gs + KP * GP;                    // GTs[m][j] = Gp[j][m]
  float* Us = GTs + KP * GP;                    // R x TP
  float* MUs = Us + R * TP;                     // R x TP
  float* s_lam = MUs + R * TP;                  // KP
  float* s_a = s_lam + KP;                      // KP   (num_bar)
  const int tid = threadIdx.x;
  const ep::Coef<const float> cf(coef, k);
  const float c_res = *cf.c_res;
  for (int e = tid; e < KP * KP; e += 256) {
    const int a = e / KP, b = e - a * KP;
    float g = 0.f;
    if (a < k && b < k) {
      g = cf.G_bar[a * k + b];
      if (a == b) g += cf.den_bar[a];
    }
    Gs[a * GP + b] = g;
    GTs[b * GP + a] = g;
  }
  for (int e = tid; e < KP; e += 256) {
    s_lam[e] = e < k ? cf.lam[e] : 0.f;
    s_a[e] = e < k ? cf.num_bar[e] : 0.f;
  }
  constexpr int CG = KP / 4;                    // column groups
  const int tc = tid % CG, tr = tid / CG;       // tr in [0, R/4)
  const int n_tiles = (n + R - 1) / R;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * R;
    __syncthreads();
    for (int e = tid; e < R * KP; e += 256) {
      const int r = e / KP, c = e - r * KP;
      const int row = row0 + r;
      const bool ok = (row < n) && (c < k);
      Us[r * TP + c] = ok ? __ldg(U + (size_t)row * ldu + c) : 0.f;
      MUs[r * TP + c] = ok ? __ldg(MU + (size_t)row * ld + c) : 0.f;
    }
    __syncthreads();
    float acc1[4][4], acc2[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { acc1[i][j] = 0.f; acc2[i][j] = 0.f; }
#pragma unroll 4
    for (int m = 0; m < KP; ++m) {
      const float4 g = *reinterpret_cast<const float4*>(Gs + m * GP + 4 * tc);
      const float4 gt = *reinterpret_cast<const float4*>(GTs + m * GP + 4 * tc);
      float u[4], mu[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { u[i] = Us[(4 * tr + i) * TP + m]; mu[i] = MUs[(4 * tr + i) * TP + m]; }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc1[i][0] = fmaf(u[i], g.x, acc1[i][0]); acc1[i][1] = fmaf(u[i], g.y, acc1[i][1]);
        acc1[i][2] = fmaf(u[i], g.z, acc1[i][2]); acc1[i][3] = fmaf(u[i], g.w, acc1[i][3]);
        acc2[i][0] = fmaf(mu[i], gt.x, acc2[i][0]); acc2[i][1] = fmaf(mu[i], gt.y, acc2[i][1]);
        acc2[i][2] = fmaf(mu[i], gt.z, acc2[i][2]); acc2[i][3] = fmaf(mu[i], gt.w, acc2[i][3]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = 4 * tr + i, row = row0 + r;
      if (row >= n) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 4 * tc + j;
        if (c >= k) continue;
        const float ku = __ldg(KU + (size_t)row * ld + c);
        const float mu = MUs[r * TP + c], u = Us[r * TP + c];
        const float lam = s_lam[c], a = s_a[c];
        const float rbar = c_res * (ku - lam * mu);
        KU_bar[(size_t)row * ld + c] = rbar + a * u;
        MU_bar[(size_t)row * ld + c] = acc1[i][j] - lam * rbar + cf.g_mean[c];
        D[(size_t)row * ld + c] = fmaf(a, ku, acc2[i][j]);
      }
    }
  }
}

// Fused backward for SYMMETRIC K, M (FEM and tufted Laplacians):
//   dU_i = s [ c sum_j (K_ij - lam M_ij) (KU_j - lam MU_j) + 2 a KU_i + MU_i S ],  S = Gp + Gp^T
// (uses K (U diag a) = KU diag a and M (U Gp) = MU Gp, so neither KU_bar / MU_bar / D nor a second
// k x k product is materialised).  One gather pass over the CSR pattern: reads the pattern, KU, MU once,
// writes dU once -> 12 nnz + 4 (n+1) + 12 n k bytes, like the forward dual SpMM.
// Thread layout as in the SpMM: LPR lanes per row, 4 columns per lane; the k x k product takes the row's
// MU values from the other lanes with shuffles and S from shared memory.
// KVT = k / 4 when instantiated for a fixed width (fully unrolled product), 0 = generic;  GRAM_IN_OUT: dU already holds
// out_scale * MU_i S (tensor-core kernel), the k x k product is compiled out and the gathered terms are added to it
template <int KVT, bool GRAM_IN_OUT>
__global__ void __launch_bounds__(256)
eigen_bwd_fused_sym_kernel(int row0, int n, int k, int lpr_shift, const int32_t* __restrict__ rowptr,
                           const int32_t* __restrict__ col, const float* __restrict__ valK,
                           const float* __restrict__ valM, const float* __restrict__ KU,
                           const float* __restrict__ MU, int ld, const float* __restrict__ coef, float out_scale_v,
                           const float* __restrict__ out_scale_dev, float* __restrict__ dU, int ldo) {
  const float out_scale = out_scale_dev ? __ldg(out_scale_dev) : out_scale_v;
  extern __shared__ __align__(16) float fsm[];
  float* S = fsm;                 // k x k
  float* s_lam = S + k * k;       // k
  float* s_a2 = s_lam + k;        // k
  const ep::Coef<const float> cf(coef, k);
  const float c_res = *cf.c_res;
  for (int e = threadIdx.x; e < k * k; e += blockDim.x) S[e] = ep::coef_sym_entry(cf, k, e);
  for (int e = threadIdx.x; e < k; e += blockDim.x) { s_lam[e] = cf.lam[e]; s_a2[e] = 2.f * cf.num_bar[e]; }
  __syncthreads();

  const int lpr = 1 << lpr_shift;
  const int kv = KVT > 0 ? KVT : (k >> 2);
  const int lane_r = threadIdx.x & (lpr - 1);
  const bool active = lane_r < kv;
  const int cofs = active ? 4 * lane_r : 0;
  const float4 lam4 = *reinterpret_cast<const float4*>(s_lam + cofs);
  const float4 a24 = *reinterpret_cast<const float4*>(s_a2 + cofs);
  const float4 gm4 = make_float4(__ldg(cf.g_mean + cofs), __ldg(cf.g_mean + cofs + 1), __ldg(cf.g_mean + cofs + 2),
                                 __ldg(cf.g_mean + cofs + 3));
  const long long groups_per_grid = ((long long)gridDim.x * blockDim.x) >> lpr_shift;
  for (long long ri = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> lpr_shift;
       ri < (long long)((n + groups_per_grid - 1) / groups_per_grid) * groups_per_grid; ri += groups_per_grid) {
    const bool valid = ri < n;
    const long long row = row0 + ri;               // output rows [row0, row0 + n)
    const int start = valid ? __ldg(rowptr + row) : 0;
    const int end = valid ? __ldg(rowptr + row + 1) : 0;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float m_rowsum = 0.f;                           // (M 1)_i : the zero-mean term's dL/dU_i = (M 1)_i g
    if (active) {
      for (int j = start; j < end; j += 4) {
        int c[4]; float kk[4], mm[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool ok = (j + u) < end;
          c[u] = ok ? __ldg(col + j + u) : -1;
          kk[u] = ok ? __ldg(valK + j + u) : 0.f;
          mm[u] = ok ? __ldg(valM + j + u) : 0.f;
          m_rowsum += mm[u];
        }
        float4 ku[4], mu[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (c[u] >= 0) {
            ku[u] = __ldg(reinterpret_cast<const float4*>(KU + (size_t)c[u] * ld + cofs));
            mu[u] = __ldg(reinterpret_cast<const float4*>(MU + (size_t)c[u] * ld + cofs));
          } else { ku[u] = make_float4(0.f, 0.f, 0.f, 0.f); mu[u] = ku[u]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc.x = fmaf(kk[u] - lam4.x * mm[u], ku[u].x - lam4.x * mu[u].x, acc.x);
          acc.y = fmaf(kk[u] - lam4.y * mm[u], ku[u].y - lam4.y * mu[u].y, acc.y);
          acc.z = fmaf(kk[u] - lam4.z * mm[u], ku[u].z - lam4.z * mu[u].z, acc.z);
          acc.w = fmaf(kk[u] - lam4.w * mm[u], ku[u].w - lam4.w * mu[u].w, acc.w);
        }
      }
    }
    acc.x = fmaf(acc.x, c_res, m_rowsum * gm4.x); acc.y = fmaf(acc.y, c_res, m_rowsum * gm4.y);
    acc.z = fmaf(acc.z, c_res, m_rowsum * gm4.z); acc.w = fmaf(acc.w, c_res, m_rowsum * gm4.w);
    float4 mu_i = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active && valid) {
      const float4 ku_i = __ldg(reinterpret_cast<const float4*>(KU + (size_t)row * ld + cofs));
      mu_i = __ldg(reinterpret_cast<const float4*>(MU + (size_t)row * ld + cofs));
      acc.x = fmaf(a24.x, ku_i.x, acc.x); acc.y = fmaf(a24.y, ku_i.y, acc.y);
      acc.z = fmaf(a24.z, ku_i.z, acc.z); acc.w = fmaf(a24.w, ku_i.w, acc.w);
    }
    // acc += MU_i S : lane L of the row group holds MU_i[4L .. 4L+3]
    if constexpr (!GRAM_IN_OUT) {
#pragma unroll
    for (int L = 0; L < kv; ++L) {
      const float m0 = __shfl_sync(0xffffffffu, mu_i.x, L, lpr);
      const float m1 = __shfl_sync(0xffffffffu, mu_i.y, L, lpr);
      const float m2 = __shfl_sync(0xffffffffu, mu_i.z, L, lpr);
      const float m3 = __shfl_sync(0xffffffffu, mu_i.w, L, lpr);
      const float* Sr = S + (size_t)(4 * L) * k + cofs;
      const float4 s0 = *reinterpret_cast<const float4*>(Sr);
      const float4 s1 = *reinterpret_cast<const float4*>(Sr + k);
      const float4 s2 = *reinterpret_cast<const float4*>(Sr + 2 * k);
      const float4 s3 = *reinterpret_cast<const float4*>(Sr + 3 * k);
      acc.x = fmaf(m0, s0.x, acc.x); acc.y = fmaf(m0, s0.y, acc.y); acc.z = fmaf(m0, s0.z, acc.z); acc.w = fmaf(m0, s0.w, acc.w);
      acc.x = fmaf(m1, s1.x, acc.x); acc.y = fmaf(m1, s1.y, acc.y); acc.z = fmaf(m1, s1.z, acc.z); acc.w = fmaf(m1, s1.w, acc.w);
      acc.x = fmaf(m2, s2.x, acc.x); acc.y = fmaf(m2, s2.y, acc.y); acc.z = fmaf(m2, s2.z, acc.z); acc.w = fmaf(m2, s2.w, acc.w);
      acc.x = fmaf(m3, s3.x, acc.x); acc.y = fmaf(m3, s3.y, acc.y); acc.z = fmaf(m3, s3.z, acc.z); acc.w = fmaf(m3, s3.w, acc.w);
    }
    }
    if (active && valid) {
      float4* dst = reinterpret_cast<float4*>(dU + (size_t)row * ldo + cofs);
      if (GRAM_IN_OUT) {
        const float4 t = *dst;
        acc.x = fmaf(acc.x, out_scale, t.x); acc.y = fmaf(acc.y, out_scale, t.y);
        acc.z = fmaf(acc.z, out_scale, t.z); acc.w = fmaf(acc.w, out_scale, t.w);
      } else {
        acc.x *= out_scale; acc.y *= out_scale; acc.z *= out_scale; acc.w *= out_scale;
      }
      *dst = acc;
    }
  }
}

template <int KP>
int launch_bwd_prepare(int n, int k, const float* U, int ldu, const float* KU, const float* MU, int ld,
                       const float* coef, float* KU_bar, float* MU_bar, float* D, cudaStream_t st) {
  constexpr int R = 4096 / KP;
  const size_t smem = sizeof(float) * (2 * KP * (KP + 4) + 2 * R * (KP + 1) + 2 * KP);
  static bool configured = false;
  if (!configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(eigen_bwd_prepare_kernel<KP>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int grid = partial_blocks(n, R);
  eigen_bwd_prepare_kernel<KP><<<grid, 256, smem, st>>>(n, k, U, ldu, KU, MU, ld, coef, KU_bar, MU_bar, D);
  EP_LAUNCH_CHECK("eigen_bwd_prepare_kernel");
  return EP_OK;
}

__global__ void __launch_bounds__(256)
scale_columns_kernel(long long n, int k, const float* __restrict__ U, int ldu, const double* __restrict__ G,
                     int ldg, double eps, float* __restrict__ out, int ldo) {
  const long long total = n * k;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / k;
    const int c = (int)(i - r * k);
    const float nrm = (float)sqrt(G[(size_t)c * ldg + c] + eps);
    out[r * ldo + c] = U[r * ldu + c] / nrm;
  }
}

__global__ void __launch_bounds__(256)
axpy_out_kernel(size_t n, float alpha, const float* __restrict__ alpha_dev, const float* __restrict__ a,
                const float* __restrict__ b, float* __restrict__ out) {
  const float al = alpha_dev ? *alpha_dev : alpha;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __fadd_rn(a[i], __fmul_rn(al, b[i]));     // corr = scale*raw (rounded), U = base + corr
}

// loss_acc[slot] += w * sum_j v[j] and loss_acc[5] (total) likewise: device-side bookkeeping of terms that are
// assembled from existing kernels (projection term), so a captured CUDA graph needs no host arithmetic
__global__ void loss_add_sum_kernel(int len, const double* __restrict__ v, double w, int slot, double* __restrict__ loss_acc) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int j = 0; j < len; ++j) s += v[j];
    loss_acc[slot] += w * s;
    loss_acc[5] += w * s;
  }
}

int stream_grid(size_t total) {
  size_t g = (total + 255) / 256;
  const size_t cap = (size_t)ep::sm_count() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" {

size_t ep_eigen_partials_len(int k) { return k > 0 ? (size_t)partials_len(k) : 0; }

size_t ep_eigen_partials_workspace_bytes(int k) {
  if (k <= 0) return 0;
  return sizeof(double) * (size_t)partials_len(k) * (size_t)(ep::sm_count() * 4);
}

size_t ep_eigen_coef_len(int k) { return k > 0 ? (size_t)ep::coef_len(k) : 0; }

int ep_eigen_partials_f32(int n, int k, const float* U, int ldu, const float* KU, const float* MU, int ld,
                          double* out, void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0, "bad size");
  EP_REQUIRE(k <= 128, "k > 128 not instantiated");
  EP_REQUIRE(out && workspace && (n == 0 || (U && KU && MU)), "null pointer");
  EP_REQUIRE(ldu >= k && ld >= k, "leading dimension < k");
  cudaStream_t st = ep::as_stream(stream);
  const int len = partials_len(k);
  const int rows = k > 64 ? 16 : 32;
  const int grid = partial_blocks(n, rows);
  if (workspace_bytes < sizeof(double) * (size_t)len * grid) {
    ep::set_error("ep_eigen_partials_f32: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  double* blocks = static_cast<double*>(workspace);
  if (k <= 16)      eigen_partials_kernel<float, 16, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else if (k <= 32) eigen_partials_kernel<float, 32, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else if (k <= 64) eigen_partials_kernel<float, 64, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else              eigen_partials_kernel<float, 128, 8><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  EP_LAUNCH_CHECK("eigen_partials_kernel");
  reduce_partials_kernel<<<ep::ceil_div(len, 8), 256, 0, st>>>(grid, len, blocks, out);
  EP_LAUNCH_CHECK("reduce_partials_kernel");
  return EP_OK;
}

int ep_eigen_partials_f64(int n, int k, const double* U, int ldu, const double* KU, const double* MU, int ld,
                          double* out, void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0, "bad size");
  EP_REQUIRE(k <= 128, "k > 128 not instantiated");
  EP_REQUIRE(out && workspace && (n == 0 || (U && KU && MU)), "null pointer");
  EP_REQUIRE(ldu >= k && ld >= k, "leading dimension < k");
  cudaStream_t st = ep::as_stream(stream);
  const int len = partials_len(k);
  const int rows = partial_rows<double>(k <= 16 ? 16 : k <= 32 ? 32 : k <= 64 ? 64 : 128);
  const int grid = partial_blocks(n, rows);           // <= 4 blocks per SM, as in fp32: same workspace size
  if (workspace_bytes < sizeof(double) * (size_t)len * grid) {
    ep::set_error("ep_eigen_partials_f64: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  double* blocks = static_cast<double*>(workspace);
  if (k <= 16)      eigen_partials_kernel<double, 16, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else if (k <= 32) eigen_partials_kernel<double, 32, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else if (k <= 64) eigen_partials_kernel<double, 64, 4><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  else              eigen_partials_kernel<double, 128, 8><<<grid, kPartialThreads, 0, st>>>(n, k, U, ldu, KU, MU, ld, blocks);
  EP_LAUNCH_CHECK("eigen_partials_kernel<double>");
  reduce_partials_kernel<<<ep::ceil_div(len, 8), 256, 0, st>>>(grid, len, blocks, out);
  EP_LAUNCH_CHECK("reduce_partials_kernel");
  return EP_OK;
}

int ep_eigen_finalize_f32(int k, double n_global, const double* partials, float w_res, float w_orth,
                          int flags, const float* lam_target, float w_trace, float w_order, float w_eigen,
                          float w_mean, float w_smooth, const float* lam_bar_extra, float* lam_out, float* coef,
                          double* loss_acc, ep_stream_t stream) {
  EP_REQUIRE(k > 0 && k <= 128, "k out of range");
  EP_REQUIRE(n_global > 0, "n_global must be positive");
  EP_REQUIRE(partials && coef && loss_acc, "null pointer");
  eigen_finalize_kernel<<<1, 256, 0, ep::as_stream(stream)>>>(k, n_global, partials, w_res, w_orth, flags,
                                                               lam_target, w_trace, w_order, w_eigen, w_mean,
                                                               w_smooth, lam_bar_extra, lam_out, coef, loss_acc);
  EP_LAUNCH_CHECK("eigen_finalize_kernel");
  return EP_OK;
}

int ep_loss_add_sum_f64(int len, const double* values, double weight, int slot, double* loss_acc, ep_stream_t stream) {
  EP_REQUIRE(len > 0 && values && loss_acc && slot >= 0 && slot < 9 && slot != 5, "bad argument");
  loss_add_sum_kernel<<<1, 32, 0, ep::as_stream(stream)>>>(len, values, weight, slot, loss_acc);
  EP_LAUNCH_CHECK("loss_add_sum_kernel");
  return EP_OK;
}

int ep_eigen_bwd_prepare_f32(int n, int k, const float* U, int ldu, const float* KU, const float* MU, int ld,
                             const float* coef, float* KU_bar, float* MU_bar, float* D, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0 && k <= 128, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(U && KU && MU && coef && KU_bar && MU_bar && D, "null pointer");
  EP_REQUIRE(ldu >= k && ld >= k, "leading dimension < k");
  cudaStream_t st = ep::as_stream(stream);
  if (k <= 16) return launch_bwd_prepare<16>(n, k, U, ldu, KU, MU, ld, coef, KU_bar, MU_bar, D, st);
  if (k <= 32) return launch_bwd_prepare<32>(n, k, U, ldu, KU, MU, ld, coef, KU_bar, MU_bar, D, st);
  if (k <= 64) return launch_bwd_prepare<64>(n, k, U, ldu, KU, MU, ld, coef, KU_bar, MU_bar, D, st);
  return launch_bwd_prepare<128>(n, k, U, ldu, KU, MU, ld, coef, KU_bar, MU_bar, D, st);
}

int ep_eigen_bwd_fused_sym_rows_f32(int row0, int n, int k, const int32_t* rowptr, const int32_t* col,
                                    const float* valK, const float* valM, const float* KU, const float* MU, int ld,
                                    const float* coef, float out_scale, const float* out_scale_dev, float* dU, int ldo,
                                    ep_stream_t stream) {
  return ep_eigen_bwd_gather_sym_rows_f32(row0, n, k, rowptr, col, valK, valM, KU, MU, ld, coef, out_scale, out_scale_dev,
                                          dU, ldo, 0, stream);
}

int ep_eigen_bwd_gather_sym_rows_f32(int row0, int n, int k, const int32_t* rowptr, const int32_t* col,
                                     const float* valK, const float* valM, const float* KU, const float* MU, int ld,
                                     const float* coef, float out_scale, const float* out_scale_dev, float* dU, int ldo,
                                     int gram_in_out, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0 && row0 >= 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(rowptr && col && valK && valM && KU && MU && coef && dU, "null pointer");
  if (k % 4 != 0 || k > 128 || ld % 4 != 0 || ldo % 4 != 0 || !ep::aligned16(KU) || !ep::aligned16(MU) ||
      !ep::aligned16(dU)) {
    ep::set_error("ep_eigen_bwd_fused_sym_rows_f32: needs k %% 4 == 0, k <= 128 and 16-byte aligned rows");
    return EP_ERR_UNSUPPORTED;
  }
  const int kv = k / 4;
  int lpr_shift = 0;
  while ((1 << lpr_shift) < kv) ++lpr_shift;
  const size_t smem = sizeof(float) * ((size_t)k * k + 2 * k);
  static size_t configured = 0;
  if (smem > 48 * 1024 && smem > configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(eigen_bwd_fused_sym_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EP_CUDA_CHECK(cudaFuncSetAttribute(eigen_bwd_fused_sym_kernel<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EP_CUDA_CHECK(cudaFuncSetAttribute(eigen_bwd_fused_sym_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const long long threads = (long long)n << lpr_shift;
  long long grid = (threads + 255) / 256;
  const long long cap = (long long)ep::sm_count() * 8;
  if (grid > cap) grid = cap;
  cudaStream_t st = ep::as_stream(stream);
#define EP_FUSED_LAUNCH(KVT, G) eigen_bwd_fused_sym_kernel<KVT, G><<<(unsigned)grid, 256, smem, st>>>( \
      row0, n, k, lpr_shift, rowptr, col, valK, valM, KU, MU, ld, coef, out_scale, out_scale_dev, dU, ldo)
  if (gram_in_out) {
    switch (kv) {
      case 4: EP_FUSED_LAUNCH(4, true); break;
      case 8: EP_FUSED_LAUNCH(8, true); break;
      case 16: EP_FUSED_LAUNCH(16, true); break;
      default: EP_FUSED_LAUNCH(0, true); break;
    }
  } else {
    switch (kv) {
      case 4: EP_FUSED_LAUNCH(4, false); break;
      case 8: EP_FUSED_LAUNCH(8, false); break;
      case 16: EP_FUSED_LAUNCH(16, false); break;
      case 32: EP_FUSED_LAUNCH(32, false); break;
      default: EP_FUSED_LAUNCH(0, false); break;
    }
  }
#undef EP_FUSED_LAUNCH
  EP_LAUNCH_CHECK("eigen_bwd_fused_sym_kernel");
  return EP_OK;
}

int ep_scale_columns_rsqrt_f32(int n, int k, const float* U, int ldu, const double* G, int ldg, double eps,
                               float* out, int ldo, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && k > 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(U && G && out, "null pointer");
  scale_columns_kernel<<<stream_grid((size_t)n * k), 256, 0, ep::as_stream(stream)>>>(n, k, U, ldu, G, ldg, eps,
                                                                                      out, ldo);
  EP_LAUNCH_CHECK("scale_columns_kernel");
  return EP_OK;
}

int ep_axpy_out_f32(size_t n, float alpha, const float* alpha_dev, const float* a, const float* b, float* out,
                    ep_stream_t stream) {
  if (n == 0) return EP_OK;
  EP_REQUIRE(a && b && out, "null pointer");
  axpy_out_kernel<<<stream_grid(n), 256, 0, ep::as_stream(stream)>>>(n, alpha, alpha_dev, a, b, out);
  EP_LAUNCH_CHECK("axpy_out_kernel");
  return EP_OK;
}

}  // extern "C"
