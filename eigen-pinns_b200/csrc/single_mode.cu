// One eigenfunction at a time with a learnable eigenvalue and deflation against the earlier modes
// (delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1: EigenfunctionNN, compute_eigenvalue_loss,
// compute_normalization_loss, compute_orthogonality_loss), as the pieces of an autograd-free training step:
//
//   loss      r = L u - lambda M u,  lambda = |w|,  Q = [M u_0 | ... | M u_{P-1}] (constant, n x P row-major)
//             eig = mean(r^2), norm = (u^T M u - 1)^2, ortho = sum_p (u^T Q_p)^2, total = eig + norm + w_o ortho
//   backward  dL/du = L gL + M gM + D  with gL = (2/n) r, gM = -(2/n) lambda r, D = 4 (u^T M u - 1) M u + Q c,
//             c_p = 2 w_o u^T Q_p  (L, M symmetric; the sum is ep_spmm2_sum_csr_*), dL/dlambda = -(2/n) sum r o M u
//   folding   layer(h (+) lambda) = h W[:, :d]^T + (b + lambda W[:, d]): the forward writes W_eff, b_eff for the plain
//             layer kernels, the backward maps dW_eff, db_eff back to dW, db and dw (sign(w), 0 at w = 0 as torch)
//
// Sums are fp64 (the fp32 inputs are widened first), written per CTA and reduced by one CTA in a fixed order, so the
// results do not depend on timing and the launches can be captured in a CUDA graph.  Also the fp64 twins of the
// clip + Adam optimiser entries (csrc/optim.cu), so that an fp64 network updates in one launch.  Kept in its own
// translation unit so that the other kernels' code is untouched.
#include "ep_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 1024;                // fixed cap: the workspace size depends on P only
constexpr int kMaxPrev = 64;                    // P_max
constexpr int kMaxLayers = 8;

// per-CTA partials: entry e of CTA b at parts[e * gridDim.x + b]; e = 0 sum r^2, 1 u^T M u, 2 sum r o M u, 3 + p u^T Q_p
template <typename T>
__global__ void __launch_bounds__(kThreads)
single_mode_fwd_kernel(int n, int P, const T* __restrict__ u, const T* __restrict__ Lu, const T* __restrict__ Mu,
                       const T* __restrict__ Q, int ldq, const T* __restrict__ w, double* __restrict__ parts) {
  __shared__ double sh[kThreads];
  __shared__ double warp_tot[3][kThreads / 32];
  const double lam = (double)fabs(w[0]);
  double srr = 0.0, sum = 0.0, srm = 0.0;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    const double l = (double)Lu[i], m = (double)Mu[i];
    const double r = __dsub_rn(l, __dmul_rn(lam, m));
    srr += r * r;
    sum += (double)u[i] * m;
    srm += r * m;
  }
  srr = ep::warp_sum(srr);
  sum = ep::warp_sum(sum);
  srm = ep::warp_sum(srm);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    warp_tot[0][warp] = srr;
    warp_tot[1][warp] = sum;
    warp_tot[2][warp] = srm;
  }
  // u^T Q: thread (row lane, column p), rows = kThreads / P rows per CTA pass
  double sq = 0.0;
  const int rows = P > 0 ? kThreads / P : 0;
  const int p = P > 0 ? threadIdx.x % P : 0, rl = P > 0 ? threadIdx.x / P : 0;
  const bool active = P > 0 && rl < rows;
  if (active)
    for (long long i = (long long)blockIdx.x * rows + rl; i < n; i += (long long)gridDim.x * rows)
      sq += (double)u[i] * (double)Q[i * ldq + p];
  sh[threadIdx.x] = sq;
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int q = 0; q < kThreads / 32; ++q) t += warp_tot[threadIdx.x][q];
    parts[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = t;
  }
  for (int e = threadIdx.x; e < P; e += kThreads) {
    double t = 0.0;
    for (int l = 0; l < rows; ++l) t += sh[l * P + e];
    parts[(size_t)(3 + e) * gridDim.x + blockIdx.x] = t;
  }
}

// One CTA: warp q reduces the entries e = q, q + 32, ...: lane l sums CTAs l, l + 32, ... in order, then a fixed shuffle
// tree.  Thread 0 then forms the loss terms and the backward coefficients.
__global__ void __launch_bounds__(1024)
single_mode_reduce_kernel(int nblocks, int n, int P, const double* __restrict__ parts, double ortho_weight,
                          double* __restrict__ loss, double* __restrict__ coef) {
  __shared__ double tot[3 + kMaxPrev];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int e = warp; e < 3 + P; e += blockDim.x / 32) {
    double t = 0.0;
    for (int b = lane; b < nblocks; b += 32) t += parts[(size_t)e * nblocks + b];
    t = ep::warp_sum(t);
    if (lane == 0) tot[e] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double two_n = 2.0 / (double)n;
    const double eig = tot[0] / (double)n;
    const double dn = tot[1] - 1.0;
    double ortho = 0.0;
    for (int p = 0; p < P; ++p) {
      ortho += tot[3 + p] * tot[3 + p];
      coef[3 + p] = 2.0 * ortho_weight * tot[3 + p];
    }
    const double norm = dn * dn;
    loss[0] = eig + norm + ortho_weight * ortho;
    loss[1] = eig;
    loss[2] = norm;
    loss[3] = ortho;
    coef[0] = two_n;
    coef[1] = 4.0 * dn;
    coef[2] = -two_n * tot[2];
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
single_mode_bwd_kernel(int n, int P, const T* __restrict__ Lu, const T* __restrict__ Mu, const T* __restrict__ Q,
                       int ldq, const T* __restrict__ w, const double* __restrict__ coef, T* __restrict__ gL,
                       T* __restrict__ gM, T* __restrict__ D) {
  __shared__ double c[3 + kMaxPrev];
  for (int e = threadIdx.x; e < 3 + P; e += kThreads) c[e] = coef[e];
  __syncthreads();
  const double lam = (double)fabs(w[0]);
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    const double m = (double)Mu[i];
    const double r = __dsub_rn((double)Lu[i], __dmul_rn(lam, m));
    const double g = c[0] * r;
    gL[i] = (T)g;
    gM[i] = (T)(-lam * g);
    double d = c[1] * m;
    for (int p = 0; p < P; ++p) d += c[3 + p] * (double)Q[i * ldq + p];
    D[i] = (T)d;
  }
}

// Flat layouts of the folding kernels (per layer l with input width d_l and output width o_l, in layer order):
//   params / grad  [W_l (o_l x (d_l + 1)) | b_l (o_l)] ... then w      eff / grad_eff  [W_eff,l (o_l x d_l) | b_eff,l] ...
struct FoldLayout {
  int layers;
  int in[kMaxLayers], out[kMaxLayers];
  long long p_off[kMaxLayers + 1], e_off[kMaxLayers + 1];   // [layers] = end of the layer blocks (p_off: offset of w)
};

__device__ __forceinline__ int layer_of(const FoldLayout& F, const long long* off, long long idx) {
  int l = 0;
  while (l + 1 < F.layers && idx >= off[l + 1]) ++l;
  return l;
}

__device__ __forceinline__ float mul_add_rn(float a, float b, float c) { return __fadd_rn(c, __fmul_rn(a, b)); }
__device__ __forceinline__ double mul_add_rn(double a, double b, double c) { return __dadd_rn(c, __dmul_rn(a, b)); }

template <typename T>
__global__ void __launch_bounds__(kThreads)
fold_fwd_kernel(FoldLayout F, const T* __restrict__ params, T* __restrict__ eff) {
  const T lam = fabs(params[F.p_off[F.layers]]);
  for (long long idx = (long long)blockIdx.x * kThreads + threadIdx.x; idx < F.e_off[F.layers];
       idx += (long long)gridDim.x * kThreads) {
    const int l = layer_of(F, F.e_off, idx);
    const int d = F.in[l], o = F.out[l];
    const long long loc = idx - F.e_off[l];
    const T* W = params + F.p_off[l];
    if (loc < (long long)o * d) {
      const long long j = loc / d, col = loc - j * d;
      eff[idx] = W[j * (d + 1) + col];
    } else {
      const long long j = loc - (long long)o * d;
      eff[idx] = mul_add_rn(lam, W[j * (d + 1) + d], W[(long long)o * (d + 1) + j]);     // b + lambda W[:, d]
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
fold_bwd_kernel(FoldLayout F, const T* __restrict__ params, const T* __restrict__ grad_eff,
                const double* __restrict__ dloss_dlam, T* __restrict__ grad) {
  const T w = params[F.p_off[F.layers]];
  const T lam = fabs(w);
  for (long long idx = (long long)blockIdx.x * kThreads + threadIdx.x; idx < F.p_off[F.layers];
       idx += (long long)gridDim.x * kThreads) {
    const int l = layer_of(F, F.p_off, idx);
    const int d = F.in[l], o = F.out[l];
    const long long loc = idx - F.p_off[l];
    const T* db_eff = grad_eff + F.e_off[l] + (long long)o * d;
    if (loc < (long long)o * (d + 1)) {
      const long long j = loc / (d + 1), col = loc - j * (d + 1);
      grad[idx] = col < d ? grad_eff[F.e_off[l] + j * d + col] : lam * db_eff[j];
    } else {
      grad[idx] = db_eff[loc - (long long)o * (d + 1)];
    }
  }
  if (blockIdx.x != 0) return;
  // dw = sign(w) (dL/dlambda + sum_l db_eff,l^T W_l[:, d_l]): thread t sums the pairs t, t + kThreads, ... of the
  // concatenated (l, j) sequence, then a fixed tree
  __shared__ double warp_tot[kThreads / 32];
  double s = 0.0;
  long long base = 0;
  for (int l = 0; l < F.layers; ++l) {
    const int d = F.in[l], o = F.out[l];
    const T* W = params + F.p_off[l];
    const T* db_eff = grad_eff + F.e_off[l] + (long long)o * d;
    for (long long j = ((threadIdx.x - base) % kThreads + kThreads) % kThreads; j < o; j += kThreads)
      s += (double)db_eff[j] * (double)W[j * (d + 1) + d];
    base += o;
  }
  s = ep::warp_sum(s);
  if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = dloss_dlam ? *dloss_dlam : 0.0;
    for (int q = 0; q < kThreads / 32; ++q) t += warp_tot[q];
    const double sgn = w > T(0) ? 1.0 : (w < T(0) ? -1.0 : 0.0);
    grad[F.p_off[F.layers]] = (T)(sgn * t);
  }
}

__global__ void __launch_bounds__(256)
sqnorm_partial_f64_kernel(size_t n, const double* __restrict__ g, double* __restrict__ parts) {
  __shared__ double sh[8];
  double s = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    s += g[i] * g[i];
  s = ep::warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int q = 0; q < 8; ++q) t += sh[q];
    parts[blockIdx.x] = t;
  }
}

constexpr int kNormBlocks = 64;
__device__ double g_norm_parts_f64[kNormBlocks];

__global__ void sqnorm_final_f64_kernel(int n_parts, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < n_parts; ++i) t += g_norm_parts_f64[i];
    *out = t;
  }
}

// torch.optim.Adam's update in double, as adam_clip_kernel of csrc/optim.cu does it in float
__global__ void __launch_bounds__(256)
adam_clip_f64_kernel(size_t n, double* __restrict__ p, const double* __restrict__ g, double* __restrict__ m,
                     double* __restrict__ v, double lr, const double* __restrict__ hyper_dev, double beta1,
                     double beta2, double eps, double wd, int step_v, double max_norm,
                     const double* __restrict__ sq_norm) {
  double coef = 1.0;
  if (sq_norm != nullptr && max_norm > 0.0) coef = fmin(max_norm / (sqrt(*sq_norm) + 1e-6), 1.0);
  const double lr_now = hyper_dev ? hyper_dev[0] : lr;
  const int t = hyper_dev ? (int)hyper_dev[1] : step_v;
  const double step_size = lr_now / (1.0 - pow(beta1, (double)t));
  const double bc2s = sqrt(1.0 - pow(beta2, (double)t));
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const double pi = p[i];
    double gi = g[i] * coef;
    gi = fma(wd, pi, gi);
    const double mi = m[i] + (gi - m[i]) * (1.0 - beta1);
    const double vi = fma(1.0 - beta2, gi * gi, v[i] * beta2);
    const double denom = sqrt(vi) / bc2s + eps;
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - step_size * (mi / denom);
  }
}

int grid_for(long long work, int cap) {
  long long g = (work + kThreads - 1) / kThreads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

int fwd_grid(int n) {
  const int cap = 2 * ep::sm_count() < kMaxBlocks ? 2 * ep::sm_count() : kMaxBlocks;
  return grid_for(n, cap);
}

int check_sizes(const char* fn, int n, int P, int ldq, const void* Q) {
  if (n < 1 || P < 0) {
    ep::set_error("%s: n must be >= 1 and P >= 0", fn);
    return EP_ERR_INVALID;
  }
  if (P > kMaxPrev) {
    ep::set_error("%s: P = %d earlier modes > %d not supported", fn, P, kMaxPrev);
    return EP_ERR_UNSUPPORTED;
  }
  if (P > 0 && (!Q || ldq < P)) {
    ep::set_error("%s: Q is NULL or ldq < P", fn);
    return EP_ERR_INVALID;
  }
  return EP_OK;
}

template <typename T>
int single_mode_fwd(const char* fn, int n, int P, const T* u, const T* Lu, const T* Mu, const T* Q, int ldq,
                    const T* w, double ortho_weight, double* loss, double* coef, void* workspace,
                    size_t workspace_bytes, ep_stream_t stream) {
  if (int rc = check_sizes(fn, n, P, ldq, Q)) return rc;
  if (!(u && Lu && Mu && w && loss && coef && workspace)) {
    ep::set_error("%s: null pointer", fn);
    return EP_ERR_INVALID;
  }
  if (workspace_bytes < ep_single_mode_workspace_bytes(P)) {
    ep::set_error("%s: workspace too small", fn);
    return EP_ERR_WORKSPACE;
  }
  cudaStream_t st = ep::as_stream(stream);
  const int grid = fwd_grid(n);
  double* parts = static_cast<double*>(workspace);
  single_mode_fwd_kernel<T><<<grid, kThreads, 0, st>>>(n, P, u, Lu, Mu, Q, ldq, w, parts);
  EP_LAUNCH_CHECK("single_mode_fwd_kernel");
  single_mode_reduce_kernel<<<1, 1024, 0, st>>>(grid, n, P, parts, ortho_weight, loss, coef);
  EP_LAUNCH_CHECK("single_mode_reduce_kernel");
  return EP_OK;
}

template <typename T>
int single_mode_bwd(const char* fn, int n, int P, const T* Lu, const T* Mu, const T* Q, int ldq, const T* w,
                    const double* coef, T* gL, T* gM, T* D, ep_stream_t stream) {
  if (int rc = check_sizes(fn, n, P, ldq, Q)) return rc;
  if (!(Lu && Mu && w && coef && gL && gM && D)) {
    ep::set_error("%s: null pointer", fn);
    return EP_ERR_INVALID;
  }
  single_mode_bwd_kernel<T><<<grid_for(n, ep::sm_count() * 8), kThreads, 0, ep::as_stream(stream)>>>(
      n, P, Lu, Mu, Q, ldq, w, coef, gL, gM, D);
  EP_LAUNCH_CHECK("single_mode_bwd_kernel");
  return EP_OK;
}

int fold_layout(const char* fn, int n_layers, const int* dims, FoldLayout* F) {
  if (n_layers < 1 || n_layers > kMaxLayers || !dims) {
    ep::set_error("%s: need 1 to %d layers and their widths", fn, kMaxLayers);
    return EP_ERR_INVALID;
  }
  F->layers = n_layers;
  F->p_off[0] = F->e_off[0] = 0;
  for (int l = 0; l < n_layers; ++l) {
    if (dims[l] < 1 || dims[l + 1] < 1) {
      ep::set_error("%s: layer widths must be positive", fn);
      return EP_ERR_INVALID;
    }
    F->in[l] = dims[l];
    F->out[l] = dims[l + 1];
    F->p_off[l + 1] = F->p_off[l] + (long long)dims[l + 1] * (dims[l] + 2);
    F->e_off[l + 1] = F->e_off[l] + (long long)dims[l + 1] * (dims[l] + 1);
  }
  return EP_OK;
}

template <typename T>
int fold_fwd(const char* fn, int n_layers, const int* dims, const T* params, T* eff, ep_stream_t stream) {
  FoldLayout F;
  if (int rc = fold_layout(fn, n_layers, dims, &F)) return rc;
  if (!(params && eff)) {
    ep::set_error("%s: null pointer", fn);
    return EP_ERR_INVALID;
  }
  fold_fwd_kernel<T><<<grid_for(F.e_off[n_layers], ep::sm_count() * 2), kThreads, 0, ep::as_stream(stream)>>>(
      F, params, eff);
  EP_LAUNCH_CHECK("fold_fwd_kernel");
  return EP_OK;
}

template <typename T>
int fold_bwd(const char* fn, int n_layers, const int* dims, const T* params, const T* grad_eff,
             const double* dloss_dlam, T* grad, ep_stream_t stream) {
  FoldLayout F;
  if (int rc = fold_layout(fn, n_layers, dims, &F)) return rc;
  if (!(params && grad_eff && grad)) {
    ep::set_error("%s: null pointer", fn);
    return EP_ERR_INVALID;
  }
  fold_bwd_kernel<T><<<grid_for(F.p_off[n_layers], ep::sm_count() * 2), kThreads, 0, ep::as_stream(stream)>>>(
      F, params, grad_eff, dloss_dlam, grad);
  EP_LAUNCH_CHECK("fold_bwd_kernel");
  return EP_OK;
}

}  // namespace

extern "C" {

size_t ep_single_mode_workspace_bytes(int P) {
  if (P < 0 || P > kMaxPrev) return 0;
  return sizeof(double) * (size_t)(3 + P) * kMaxBlocks;
}

int ep_single_mode_max_prev(void) { return kMaxPrev; }

int ep_single_mode_fwd_f32(int n, int P, const float* u, const float* Lu, const float* Mu, const float* Q, int ldq,
                           const float* w, double ortho_weight, double* loss, double* coef, void* workspace,
                           size_t workspace_bytes, ep_stream_t stream) {
  return single_mode_fwd(__func__, n, P, u, Lu, Mu, Q, ldq, w, ortho_weight, loss, coef, workspace, workspace_bytes,
                         stream);
}

int ep_single_mode_fwd_f64(int n, int P, const double* u, const double* Lu, const double* Mu, const double* Q,
                           int ldq, const double* w, double ortho_weight, double* loss, double* coef, void* workspace,
                           size_t workspace_bytes, ep_stream_t stream) {
  return single_mode_fwd(__func__, n, P, u, Lu, Mu, Q, ldq, w, ortho_weight, loss, coef, workspace, workspace_bytes,
                         stream);
}

int ep_single_mode_bwd_f32(int n, int P, const float* Lu, const float* Mu, const float* Q, int ldq, const float* w,
                           const double* coef, float* gL, float* gM, float* D, ep_stream_t stream) {
  return single_mode_bwd(__func__, n, P, Lu, Mu, Q, ldq, w, coef, gL, gM, D, stream);
}

int ep_single_mode_bwd_f64(int n, int P, const double* Lu, const double* Mu, const double* Q, int ldq,
                           const double* w, const double* coef, double* gL, double* gM, double* D,
                           ep_stream_t stream) {
  return single_mode_bwd(__func__, n, P, Lu, Mu, Q, ldq, w, coef, gL, gM, D, stream);
}

int ep_single_mode_fold_fwd_f32(int n_layers, const int* dims, const float* params, float* eff, ep_stream_t stream) {
  return fold_fwd(__func__, n_layers, dims, params, eff, stream);
}

int ep_single_mode_fold_fwd_f64(int n_layers, const int* dims, const double* params, double* eff,
                                ep_stream_t stream) {
  return fold_fwd(__func__, n_layers, dims, params, eff, stream);
}

int ep_single_mode_fold_bwd_f32(int n_layers, const int* dims, const float* params, const float* grad_eff,
                                const double* dloss_dlam, float* grad, ep_stream_t stream) {
  return fold_bwd(__func__, n_layers, dims, params, grad_eff, dloss_dlam, grad, stream);
}

int ep_single_mode_fold_bwd_f64(int n_layers, const int* dims, const double* params, const double* grad_eff,
                                const double* dloss_dlam, double* grad, ep_stream_t stream) {
  return fold_bwd(__func__, n_layers, dims, params, grad_eff, dloss_dlam, grad, stream);
}

int ep_grad_sqnorm_f64(size_t n, const double* g, double* sq_out, ep_stream_t stream) {
  EP_REQUIRE(sq_out && (n == 0 || g), "null pointer");
  cudaStream_t st = ep::as_stream(stream);
  double* parts = nullptr;
  EP_CUDA_CHECK(cudaGetSymbolAddress(reinterpret_cast<void**>(&parts), g_norm_parts_f64));
  sqnorm_partial_f64_kernel<<<kNormBlocks, 256, 0, st>>>(n, g, parts);
  EP_LAUNCH_CHECK("sqnorm_partial_f64_kernel");
  sqnorm_final_f64_kernel<<<1, 32, 0, st>>>(kNormBlocks, sq_out);
  EP_LAUNCH_CHECK("sqnorm_final_f64_kernel");
  return EP_OK;
}

int ep_adam_clip_step_f64(size_t n, double* p, const double* g, double* m, double* v, double lr,
                          const double* hyper_dev, double beta1, double beta2, double eps, double weight_decay,
                          int step, double max_norm, const double* sq_norm, ep_stream_t stream) {
  if (n == 0) return EP_OK;
  EP_REQUIRE(p && g && m && v, "null pointer");
  EP_REQUIRE(step >= 1 || hyper_dev, "step counts from 1");
  size_t grid = (n + 255) / 256;
  const size_t cap = (size_t)ep::sm_count() * 8;
  if (grid > cap) grid = cap;
  adam_clip_f64_kernel<<<(unsigned)grid, 256, 0, ep::as_stream(stream)>>>(n, p, g, m, v, lr, hyper_dev, beta1, beta2,
                                                                         eps, weight_decay, step >= 1 ? step : 1,
                                                                         max_norm, sq_norm);
  EP_LAUNCH_CHECK("adam_clip_f64_kernel");
  return EP_OK;
}

}  // extern "C"
