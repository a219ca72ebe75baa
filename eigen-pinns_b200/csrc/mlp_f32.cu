// Corrector MLP, fp32 SIMT path ("parity mode").  Reference: src/corrector_model.py:12-21,31
// (nn.Sequential of Linear / ReLU) and the autograd backward behind multigrid_model.py:258.
//
// One tiled GEMM kernel (64 x 64 x 16 tile, 256 threads, 4 x 4 outputs per thread) serves the
// three products of a Linear layer; the operand strides say which one it is:
//   forward  Y  = X W^T (+ b, ReLU)      A = X  (k contiguous)   B(k,j) = W[j,k] (k contiguous)
//   dX       dX = dY W  (* [X > 0])      A = dY (k contiguous)   B(k,j) = W[k,j] (j contiguous)
//   dW       dW = dY^T X                 A(i,k) = dY[k,i] (i contiguous)  B = X (j contiguous)
// dW reduces over all vertices, so it is split along K over blockIdx.z into a workspace and
// summed in a fixed order (deterministic); db is a two-stage column sum.
// This path exists for fp32 parity with the reference CPU arithmetic; the throughput path is the
// bf16 tcgen05 kernel in mlp_tc.cu.  The same kernels instantiated for double (plain DFMA, same tiling)
// serve the fp64 dense layers of the notebook variants (variants.py).
#include "ep_common.cuh"
#include <type_traits>
#include "dropout.cuh"

namespace {

constexpr int BM = 64, BN = 64, BK = 16, PITCH = 68;

__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float relu_t(float v) { return fmaxf(v, 0.f); }
__device__ __forceinline__ double relu_t(double v) { return fmax(v, 0.0); }

// four consecutive shared-memory values: one LDS.128 in fp32, two in fp64 (PITCH * 8 B keeps them 16-byte aligned)
__device__ __forceinline__ void lds4(const float* p, float* v) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void lds4(const double* p, double* v) {
  const double2 t0 = *reinterpret_cast<const double2*>(p);
  const double2 t1 = *reinterpret_cast<const double2*>(p + 2);
  v[0] = t0.x; v[1] = t0.y; v[2] = t1.x; v[3] = t1.y;
}

template <typename T, bool A_KC, bool B_KC>
__global__ void __launch_bounds__(256)
gemm_kernel(int M, int N, int K, const T* __restrict__ A, long long sa_i, long long sa_k,
            const T* __restrict__ B, long long sb_k, long long sb_j, T* __restrict__ C, int ldc,
            long long c_split_stride, const T* __restrict__ bias, int relu,
            const T* __restrict__ mask, int ldm, int k_chunk) {
  __shared__ __align__(16) T As[BK][PITCH];
  __shared__ __align__(16) T Bs[BK][PITCH];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int i0 = blockIdx.y * BM, j0 = blockIdx.x * BN;
  const int k_begin = blockIdx.z * k_chunk;
  const int k_end = min(K, k_begin + k_chunk);
  T acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = T(0);

  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + 256 * q;
      int ai, ak, bk, bj;
      if (A_KC) { ai = e >> 4; ak = e & 15; } else { ak = e >> 6; ai = e & 63; }
      if (B_KC) { bj = e >> 4; bk = e & 15; } else { bk = e >> 6; bj = e & 63; }
      const int gi = i0 + ai, gk = k0 + ak;
      As[ak][ai] = (gi < M && gk < k_end) ? __ldg(A + gi * sa_i + gk * sa_k) : T(0);
      const int gj = j0 + bj, gk2 = k0 + bk;
      Bs[bk][bj] = (gj < N && gk2 < k_end) ? __ldg(B + gk2 * sb_k + gj * sb_j) : T(0);
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      T av[4], bv[4];
      lds4(&As[kk][ty * 4], av);
      lds4(&Bs[kk][tx * 4], bv);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma_t(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  T* Cz = C + (long long)blockIdx.z * c_split_stride;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = i0 + ty * 4 + i;
    if (gi >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gj = j0 + tx * 4 + j;
      if (gj >= N) continue;
      T v = acc[i][j];
      if (bias) v += __ldg(bias + gj);
      if (relu) v = relu_t(v);
      if (mask) v = (__ldg(mask + (size_t)gi * ldm + gj) > T(0)) ? v : T(0);
      Cz[(size_t)gi * ldc + gj] = v;
    }
  }
}

// gemm_kernel<float> (no split-K) for a hidden layer followed by dropout, kept apart so that gemm_kernel's code does not
// change.  DROP_FWD (forward, A = X, B = W^T): y = keep ? relu(z) * s : 0 with the keep mask of dropout.cuh.
// DROP_BWD (dX): dX = (dY W) * [X > 0] * s - X is the stored, dropped activation, so its sign pattern already carries
// the keep mask.
enum Drop { DROP_FWD = 1, DROP_BWD = 2 };

template <bool A_KC, bool B_KC, int DROP>
__global__ void __launch_bounds__(256)
gemm_dropout_kernel(int M, int N, int K, const float* __restrict__ A, long long sa_i, long long sa_k,
                    const float* __restrict__ B, long long sb_k, long long sb_j, float* __restrict__ C, int ldc,
                    const float* __restrict__ bias, const float* __restrict__ mask, int ldm, const dropout::Params dp) {
  using T = float;
  __shared__ __align__(16) T As[BK][PITCH];
  __shared__ __align__(16) T Bs[BK][PITCH];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int i0 = blockIdx.y * BM, j0 = blockIdx.x * BN;
  T acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = T(0);

  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + 256 * q;
      int ai, ak, bk, bj;
      if (A_KC) { ai = e >> 4; ak = e & 15; } else { ak = e >> 6; ai = e & 63; }
      if (B_KC) { bj = e >> 4; bk = e & 15; } else { bk = e >> 6; bj = e & 63; }
      const int gi = i0 + ai, gk = k0 + ak;
      As[ak][ai] = (gi < M && gk < K) ? __ldg(A + gi * sa_i + gk * sa_k) : T(0);
      const int gj = j0 + bj, gk2 = k0 + bk;
      Bs[bk][bj] = (gj < N && gk2 < K) ? __ldg(B + gk2 * sb_k + gj * sb_j) : T(0);
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      T av[4], bv[4];
      lds4(&As[kk][ty * 4], av);
      lds4(&Bs[kk][tx * 4], bv);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma_t(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int step = DROP == DROP_FWD ? dropout::step_of(dp) : 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = i0 + ty * 4 + i;
    if (gi >= M) continue;
    uint32_t keep = 0;                 // the thread's four columns lie in one 8-column chunk: one Philox call per row
    if (DROP == DROP_FWD)
      keep = dropout::keep_byte(dp.seed, step, dp.layer, dp.row0 + gi, (j0 + tx * 4) >> 3, dp.thr) >> ((tx & 1) * 4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gj = j0 + tx * 4 + j;
      if (gj >= N) continue;
      T v = acc[i][j];
      if (DROP == DROP_FWD) {
        if (bias) v += __ldg(bias + gj);
        v = ((keep >> j) & 1u) ? relu_t(v) * dp.s : T(0);
      } else {
        v = (__ldg(mask + (size_t)gi * ldm + gj) > T(0)) ? v * dp.s : T(0);
      }
      C[(size_t)gi * ldc + gj] = v;
    }
  }
}

// Activation epilogues of the notebook networks (variants.py), ep_linear_act_{fwd,bwd}_*.  Accurate libm math (expf / exp,
// sinf / sin, cosf / cos, tanhf / tanh), no fast-math intrinsics.
enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_SILU = 2, ACT_SIN = 3, ACT_TANH = 4 };

__device__ __forceinline__ float exp_t(float v) { return expf(v); }
__device__ __forceinline__ double exp_t(double v) { return exp(v); }
__device__ __forceinline__ float sin_t(float v) { return sinf(v); }
__device__ __forceinline__ double sin_t(double v) { return sin(v); }
__device__ __forceinline__ float cos_t(float v) { return cosf(v); }
__device__ __forceinline__ double cos_t(double v) { return cos(v); }
__device__ __forceinline__ float tanh_t(float v) { return tanhf(v); }
__device__ __forceinline__ double tanh_t(double v) { return tanh(v); }

template <int ACT, typename T>
__device__ __forceinline__ T act_fwd(T z) {
  if (ACT == ACT_RELU) return relu_t(z);
  if (ACT == ACT_SILU) return z / (T(1) + exp_t(-z));
  if (ACT == ACT_SIN) return sin_t(z);
  if (ACT == ACT_TANH) return tanh_t(z);
  return z;
}

// act'(z) from what the backward reads: z for SiLU (s (1 + z (1 - s)), s = sigmoid z) and sin (cos z); the activation
// x = tanh z itself for tanh (1 - x^2)
template <int ACT, typename T>
__device__ __forceinline__ T act_grad(T v) {
  if (ACT == ACT_SILU) {
    const T s = T(1) / (T(1) + exp_t(-v));
    return s * (T(1) + v * (T(1) - s));
  }
  if (ACT == ACT_SIN) return cos_t(v);
  return T(1) - v * v;
}

// The tile and main loop of gemm_kernel<T, true, !DX> (no split-K), kept apart so that gemm_kernel's code does not
// change, with an activation epilogue:
//   forward (DX = false, A = X, B = W^T):  z = X W^T + b, Z = z if Z != NULL, C = act(z)   (ACT: any Act)
//   dX      (DX = true,  A = dY, B = W):   C = (dY W) * act'(aux), aux = Z of the layer that produced X (SiLU, sin) or
//                                          X itself (tanh)
// Three CTAs per SM (at most 85 registers): left to its default, ptxas gives the fp32 sin dX form 64 registers and
// spills one of them in the main loop.
template <typename T, int ACT, bool DX>
__global__ void __launch_bounds__(256, 3)
gemm_act_kernel(int M, int N, int K, const T* __restrict__ A, long long sa_i, long long sa_k, const T* __restrict__ B,
                long long sb_k, long long sb_j, T* __restrict__ C, int ldc, const T* __restrict__ bias,
                const T* __restrict__ aux, int ld_aux, T* __restrict__ Z, int ldz) {
  constexpr bool A_KC = true, B_KC = !DX;
  __shared__ __align__(16) T As[BK][PITCH];
  __shared__ __align__(16) T Bs[BK][PITCH];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int i0 = blockIdx.y * BM, j0 = blockIdx.x * BN;
  T acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = T(0);

  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + 256 * q;
      int ai, ak, bk, bj;
      if (A_KC) { ai = e >> 4; ak = e & 15; } else { ak = e >> 6; ai = e & 63; }
      if (B_KC) { bj = e >> 4; bk = e & 15; } else { bk = e >> 6; bj = e & 63; }
      const int gi = i0 + ai, gk = k0 + ak;
      As[ak][ai] = (gi < M && gk < K) ? __ldg(A + gi * sa_i + gk * sa_k) : T(0);
      const int gj = j0 + bj, gk2 = k0 + bk;
      Bs[bk][bj] = (gj < N && gk2 < K) ? __ldg(B + gk2 * sb_k + gj * sb_j) : T(0);
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      T av[4], bv[4];
      lds4(&As[kk][ty * 4], av);
      lds4(&Bs[kk][tx * 4], bv);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma_t(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = i0 + ty * 4 + i;
    if (gi >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gj = j0 + tx * 4 + j;
      if (gj >= N) continue;
      T v = acc[i][j];
      if (DX) {
        v *= act_grad<ACT>(__ldg(aux + (size_t)gi * ld_aux + gj));
      } else {
        if (bias) v += __ldg(bias + gj);
        if (Z) Z[(size_t)gi * ldz + gj] = v;
        v = act_fwd<ACT>(v);
      }
      C[(size_t)gi * ldc + gj] = v;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
sum_splits_kernel(int n_split, size_t len, const T* __restrict__ parts, T* __restrict__ out) {
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= len) return;
  T s = T(0);
  for (int z = 0; z < n_split; ++z) s += parts[(size_t)z * len + e];
  out[e] = s;
}

// partial column sums: block b sums rows [b*rows_per_block, ...) of dY into parts[b][:]
template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(int n, int cols, const T* __restrict__ dY, int ld, int rows_per_block,
                      T* __restrict__ parts) {
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(n, r0 + rows_per_block);
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    T s = T(0);
    for (int r = r0; r < r1; ++r) s += __ldg(dY + (size_t)r * ld + c);
    parts[(size_t)blockIdx.x * cols + c] = s;
  }
}

struct BwdPlan { int n_split; int k_chunk; int cs_blocks; int cs_rows; };

BwdPlan plan_bwd(int n, int in, int out) {
  BwdPlan p;
  const int tiles = ep::ceil_div(out, BM) * ep::ceil_div(in, BN);
  int want = ep::ceil_div(ep::sm_count() * 4, tiles);
  int max_split = ep::ceil_div(n, 4 * BK);
  if (want > max_split) want = max_split;
  if (want < 1) want = 1;
  p.k_chunk = ep::ceil_div(ep::ceil_div(n, want), BK) * BK;
  p.n_split = ep::ceil_div(n, p.k_chunk);
  if (p.n_split < 1) p.n_split = 1;
  p.cs_rows = 256;
  p.cs_blocks = ep::ceil_div(n, p.cs_rows);
  if (p.cs_blocks > ep::sm_count() * 8) {
    p.cs_blocks = ep::sm_count() * 8;
    p.cs_rows = ep::ceil_div(n, p.cs_blocks);
    p.cs_blocks = ep::ceil_div(n, p.cs_rows);
  }
  if (p.cs_blocks < 1) p.cs_blocks = 1;
  return p;
}

template <typename T>
int linear_fwd(int n, int in, int out, const T* X, int ldx, const T* W, const T* b, T* Y, int ldy, int act,
               cudaStream_t st) {
  dim3 grid(ep::ceil_div(out, BN), ep::ceil_div(n, BM), 1);
  if (grid.y > 65535) {                       // fold: process in row slabs
    const int slab = 65535 * BM;
    for (int r0 = 0; r0 < n; r0 += slab) {
      const int rows = (n - r0) < slab ? (n - r0) : slab;
      int rc = linear_fwd(rows, in, out, X + (size_t)r0 * ldx, ldx, W, b, Y + (size_t)r0 * ldy, ldy, act, st);
      if (rc != EP_OK) return rc;
    }
    return EP_OK;
  }
  gemm_kernel<T, true, true><<<grid, 256, 0, st>>>(
      n, out, in, X, ldx, 1, W, 1, in, Y, ldy, 0, b, act == 1, nullptr, 0, in);
  EP_LAUNCH_CHECK("gemm_kernel<fwd>");
  return EP_OK;
}

// drop_s > 0: X is the output of a hidden layer with dropout, dX = (dY W) * [X > 0] * drop_s (fp32 only)
template <typename T>
int linear_bwd(int n, int in, int out, const T* X, int ldx, const T* W, const T* dY, int lddy, T* dX, int lddx,
               int relu_mask, T* dW, T* db, void* workspace, cudaStream_t st, float drop_s = 0.f) {
  BwdPlan p = plan_bwd(n, in, out);
  T* parts = static_cast<T*>(workspace);
  T* cs_parts = parts + (size_t)p.n_split * in * out;
  // dW[o, i] = sum_r dY[r, o] X[r, i]
  {
    dim3 grid(ep::ceil_div(in, BN), ep::ceil_div(out, BM), p.n_split);
    gemm_kernel<T, false, false><<<grid, 256, 0, st>>>(out, in, n, dY, 1, lddy, X, ldx, 1, parts, in,
                                                      (long long)in * out, nullptr, 0, nullptr, 0, p.k_chunk);
    EP_LAUNCH_CHECK("gemm_kernel<dW>");
    const size_t len = (size_t)in * out;
    sum_splits_kernel<<<(unsigned)((len + 255) / 256), 256, 0, st>>>(p.n_split, len, parts, dW);
    EP_LAUNCH_CHECK("sum_splits_kernel<dW>");
  }
  // db[o] = sum_r dY[r, o]
  {
    colsum_partial_kernel<<<p.cs_blocks, 256, 0, st>>>(n, out, dY, lddy, p.cs_rows, cs_parts);
    EP_LAUNCH_CHECK("colsum_partial_kernel");
    sum_splits_kernel<<<ep::ceil_div(out, 256), 256, 0, st>>>(p.cs_blocks, (size_t)out, cs_parts, db);
    EP_LAUNCH_CHECK("sum_splits_kernel<db>");
  }
  // dX = (dY W) * [X > 0]
  if (dX) {
    const int slab = 65535 * BM;
    for (int r0 = 0; r0 < n; r0 += slab) {
      const int rows = (n - r0) < slab ? (n - r0) : slab;
      dim3 grid(ep::ceil_div(in, BN), ep::ceil_div(rows, BM), 1);
      if constexpr (std::is_same<T, float>::value) {
        if (drop_s > 0.f) {
          dropout::Params d{};
          d.s = drop_s;
          gemm_dropout_kernel<true, false, DROP_BWD><<<grid, 256, 0, st>>>(
              rows, in, out, dY + (size_t)r0 * lddy, lddy, 1, W, in, 1, dX + (size_t)r0 * lddx, lddx, nullptr,
              X + (size_t)r0 * ldx, ldx, d);
          EP_LAUNCH_CHECK("gemm_dropout_kernel<dX>");
          continue;
        }
      }
      gemm_kernel<T, true, false><<<grid, 256, 0, st>>>(
          rows, in, out, dY + (size_t)r0 * lddy, lddy, 1, W, in, 1, dX + (size_t)r0 * lddx, lddx, 0, nullptr, 0,
          relu_mask ? X + (size_t)r0 * ldx : nullptr, ldx, out);
      EP_LAUNCH_CHECK("gemm_kernel<dX>");
    }
  }
  return EP_OK;
}

// forward of a hidden layer followed by dropout: Y = keep ? relu(X W^T + b) * s : 0
int linear_fwd_dropout(int n, int in, int out, const float* X, int ldx, const float* W, const float* b, float* Y, int ldy,
                       dropout::Params dp, cudaStream_t st) {
  const int slab = 65535 * BM;
  for (int r0 = 0; r0 < n; r0 += slab) {
    const int rows = (n - r0) < slab ? (n - r0) : slab;
    dim3 grid(ep::ceil_div(out, BN), ep::ceil_div(rows, BM), 1);
    dropout::Params d = dp;
    d.row0 += r0;
    gemm_dropout_kernel<true, true, DROP_FWD><<<grid, 256, 0, st>>>(
        rows, out, in, X + (size_t)r0 * ldx, ldx, 1, W, 1, in, Y + (size_t)r0 * ldy, ldy, b, nullptr, 0, d);
    EP_LAUNCH_CHECK("gemm_dropout_kernel<fwd>");
  }
  return EP_OK;
}

size_t bwd_workspace_bytes(int n, int in, int out, size_t elem) {
  if (n <= 0 || in <= 0 || out <= 0) return 0;
  BwdPlan p = plan_bwd(n, in, out);
  return elem * ((size_t)p.n_split * in * out + (size_t)p.cs_blocks * out);
}

// Y = act(X W^T + b), Z = X W^T + b (if Z != NULL); row slabs of 65535 tiles as in linear_fwd
template <typename T, int ACT>
int linear_act_fwd(int n, int in, int out, const T* X, int ldx, const T* W, const T* b, T* Y, int ldy, T* Z, int ldz,
                   cudaStream_t st) {
  const int slab = 65535 * BM;
  for (int r0 = 0; r0 < n; r0 += slab) {
    const int rows = (n - r0) < slab ? (n - r0) : slab;
    dim3 grid(ep::ceil_div(out, BN), ep::ceil_div(rows, BM), 1);
    gemm_act_kernel<T, ACT, false><<<grid, 256, 0, st>>>(
        rows, out, in, X + (size_t)r0 * ldx, ldx, 1, W, 1, in, Y + (size_t)r0 * ldy, ldy, b, nullptr, 0,
        Z ? Z + (size_t)r0 * ldz : nullptr, ldz);
    EP_LAUNCH_CHECK("gemm_act_kernel<fwd>");
  }
  return EP_OK;
}

// dX = (dY W) * act'(aux)
template <typename T, int ACT>
int linear_act_dx(int n, int in, int out, const T* aux, int ld_aux, const T* W, const T* dY, int lddy, T* dX, int lddx,
                  cudaStream_t st) {
  const int slab = 65535 * BM;
  for (int r0 = 0; r0 < n; r0 += slab) {
    const int rows = (n - r0) < slab ? (n - r0) : slab;
    dim3 grid(ep::ceil_div(in, BN), ep::ceil_div(rows, BM), 1);
    gemm_act_kernel<T, ACT, true><<<grid, 256, 0, st>>>(
        rows, in, out, dY + (size_t)r0 * lddy, lddy, 1, W, in, 1, dX + (size_t)r0 * lddx, lddx, nullptr,
        aux + (size_t)r0 * ld_aux, ld_aux, nullptr, 0);
    EP_LAUNCH_CHECK("gemm_act_kernel<dX>");
  }
  return EP_OK;
}

// EP_REQUIRE with the entry point's name in the message
#define ACT_REQUIRE(cond, msg)                                                  \
  do {                                                                          \
    if (!(cond)) { ep::set_error("%s: %s", name, msg); return EP_ERR_INVALID; } \
  } while (0)

template <typename T>
int act_fwd_entry(const char* name, int n, int in, int out, const T* X, int ldx, const T* W, const T* b, T* Y, int ldy, T* Z, int ldz,
                  int act, ep_stream_t stream) {
  ACT_REQUIRE(n >= 0 && in > 0 && out > 0, "bad size");
  ACT_REQUIRE(act >= ACT_NONE && act <= ACT_TANH, "unknown activation (0 none, 1 ReLU, 2 SiLU, 3 sin, 4 tanh)");
  if (n == 0) return EP_OK;
  ACT_REQUIRE(X && W && Y, "null pointer");
  ACT_REQUIRE(ldx >= in && ldy >= out && (!Z || ldz >= out), "leading dimension too small");
  ACT_REQUIRE(ep::ceil_div(n, BM) <= 65535 * 1024, "n too large");
  cudaStream_t st = ep::as_stream(stream);
  switch (act) {
    case ACT_NONE: return linear_act_fwd<T, ACT_NONE>(n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, st);
    case ACT_RELU: return linear_act_fwd<T, ACT_RELU>(n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, st);
    case ACT_SILU: return linear_act_fwd<T, ACT_SILU>(n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, st);
    case ACT_SIN: return linear_act_fwd<T, ACT_SIN>(n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, st);
    default: return linear_act_fwd<T, ACT_TANH>(n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, st);
  }
}

// act_x 0 / 1: dX through linear_bwd's gemm_kernel (no mask / [X > 0]); 2 - 4: dW, db there, dX by gemm_act_kernel
template <typename T>
int act_bwd_entry(const char* name, int n, int in, int out, const T* X, int ldx, const T* Zx, int ldzx, int act_x, const T* W,
                  const T* dY, int lddy, T* dX, int lddx, T* dW, T* db, void* workspace, size_t workspace_bytes,
                  ep_stream_t stream) {
  ACT_REQUIRE(n > 0 && in > 0 && out > 0, "bad size");
  ACT_REQUIRE(act_x >= ACT_NONE && act_x <= ACT_TANH, "unknown activation (0 none, 1 ReLU, 2 SiLU, 3 sin, 4 tanh)");
  ACT_REQUIRE(X && W && dY && dW && db && workspace, "null pointer");
  const bool needs_z = dX && (act_x == ACT_SILU || act_x == ACT_SIN);
  ACT_REQUIRE(!needs_z || Zx, "Zx is NULL but the activation of X (SiLU or sin) needs its pre-activation");
  ACT_REQUIRE(ldx >= in && lddy >= out && (!dX || lddx >= in) && (!needs_z || ldzx >= in),
             "leading dimension too small");
  if (workspace_bytes < bwd_workspace_bytes(n, in, out, sizeof(T))) {
    ep::set_error("%s: workspace too small", name);
    return EP_ERR_WORKSPACE;
  }
  cudaStream_t st = ep::as_stream(stream);
  const bool plain_dx = act_x <= ACT_RELU;
  int rc = linear_bwd(n, in, out, X, ldx, W, dY, lddy, plain_dx ? dX : nullptr, lddx, act_x == ACT_RELU, dW, db,
                      workspace, st);
  if (rc != EP_OK || plain_dx || !dX) return rc;
  switch (act_x) {
    case ACT_SILU: return linear_act_dx<T, ACT_SILU>(n, in, out, Zx, ldzx, W, dY, lddy, dX, lddx, st);
    case ACT_SIN: return linear_act_dx<T, ACT_SIN>(n, in, out, Zx, ldzx, W, dY, lddy, dX, lddx, st);
    default: return linear_act_dx<T, ACT_TANH>(n, in, out, X, ldx, W, dY, lddy, dX, lddx, st);
  }
}

#undef ACT_REQUIRE

}  // namespace

extern "C" {

int ep_linear_fwd_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b,
                      float* Y, int ldy, int act, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && in > 0 && out > 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(X && W && Y, "null pointer");
  EP_REQUIRE(ldx >= in && ldy >= out, "leading dimension too small");
  EP_REQUIRE(ep::ceil_div(n, BM) <= 65535 * 1024, "n too large");
  return linear_fwd(n, in, out, X, ldx, W, b, Y, ldy, act, ep::as_stream(stream));
}

int ep_linear_fwd_f64(int n, int in, int out, const double* X, int ldx, const double* W, const double* b,
                      double* Y, int ldy, int act, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && in > 0 && out > 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(X && W && Y, "null pointer");
  EP_REQUIRE(ldx >= in && ldy >= out, "leading dimension too small");
  EP_REQUIRE(ep::ceil_div(n, BM) <= 65535 * 1024, "n too large");
  return linear_fwd(n, in, out, X, ldx, W, b, Y, ldy, act, ep::as_stream(stream));
}

size_t ep_linear_bwd_workspace_bytes(int n, int in, int out) { return bwd_workspace_bytes(n, in, out, sizeof(float)); }

size_t ep_linear_bwd_workspace_bytes_f64(int n, int in, int out) {
  return bwd_workspace_bytes(n, in, out, sizeof(double));
}

int ep_linear_bwd_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* dY,
                      int lddy, float* dX, int lddx, int relu_mask, float* dW, float* db, void* workspace,
                      size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && in > 0 && out > 0, "bad size");
  EP_REQUIRE(X && W && dY && dW && db && workspace, "null pointer");
  EP_REQUIRE(ldx >= in && lddy >= out && (!dX || lddx >= in), "leading dimension too small");
  if (workspace_bytes < ep_linear_bwd_workspace_bytes(n, in, out)) {
    ep::set_error("ep_linear_bwd_f32: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  return linear_bwd(n, in, out, X, ldx, W, dY, lddy, dX, lddx, relu_mask, dW, db, workspace, ep::as_stream(stream));
}

int ep_linear_fwd_dropout_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b,
                              float* Y, int ldy, float p, unsigned long long seed, int step, const int* step_dev,
                              int layer, long long row0, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && in > 0 && out > 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(X && W && Y, "null pointer");
  EP_REQUIRE(ldx >= in && ldy >= out, "leading dimension too small");
  EP_REQUIRE(ep::ceil_div(n, BM) <= 65535 * 1024, "n too large");
  dropout::Params dp{};
  if (int rc = dropout::host_params("ep_linear_fwd_dropout_f32", p, &dp.thr, &dp.s)) return rc;
  dp.seed = seed; dp.row0 = row0; dp.step_dev = step_dev; dp.step = step; dp.layer = layer;
  return linear_fwd_dropout(n, in, out, X, ldx, W, b, Y, ldy, dp, ep::as_stream(stream));
}

int ep_linear_bwd_dropout_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* dY,
                              int lddy, float* dX, int lddx, float p, float* dW, float* db, void* workspace,
                              size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && in > 0 && out > 0, "bad size");
  EP_REQUIRE(X && W && dY && dX && dW && db && workspace, "null pointer");
  EP_REQUIRE(ldx >= in && lddy >= out && lddx >= in, "leading dimension too small");
  if (workspace_bytes < ep_linear_bwd_workspace_bytes(n, in, out)) {
    ep::set_error("ep_linear_bwd_dropout_f32: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  uint32_t thr;
  float s;
  if (int rc = dropout::host_params("ep_linear_bwd_dropout_f32", p, &thr, &s)) return rc;
  return linear_bwd(n, in, out, X, ldx, W, dY, lddy, dX, lddx, 1, dW, db, workspace, ep::as_stream(stream), s);
}

int ep_linear_bwd_f64(int n, int in, int out, const double* X, int ldx, const double* W, const double* dY,
                      int lddy, double* dX, int lddx, int relu_mask, double* dW, double* db, void* workspace,
                      size_t workspace_bytes, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && in > 0 && out > 0, "bad size");
  EP_REQUIRE(X && W && dY && dW && db && workspace, "null pointer");
  EP_REQUIRE(ldx >= in && lddy >= out && (!dX || lddx >= in), "leading dimension too small");
  if (workspace_bytes < ep_linear_bwd_workspace_bytes_f64(n, in, out)) {
    ep::set_error("ep_linear_bwd_f64: workspace too small");
    return EP_ERR_WORKSPACE;
  }
  return linear_bwd(n, in, out, X, ldx, W, dY, lddy, dX, lddx, relu_mask, dW, db, workspace, ep::as_stream(stream));
}

int ep_linear_act_fwd_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b, float* Y,
                          int ldy, float* Z, int ldz, int act, ep_stream_t stream) {
  return act_fwd_entry("ep_linear_act_fwd_f32", n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, act, stream);
}

int ep_linear_act_fwd_f64(int n, int in, int out, const double* X, int ldx, const double* W, const double* b, double* Y,
                          int ldy, double* Z, int ldz, int act, ep_stream_t stream) {
  return act_fwd_entry("ep_linear_act_fwd_f64", n, in, out, X, ldx, W, b, Y, ldy, Z, ldz, act, stream);
}

int ep_linear_act_bwd_f32(int n, int in, int out, const float* X, int ldx, const float* Zx, int ldzx, int act_x,
                          const float* W, const float* dY, int lddy, float* dX, int lddx, float* dW, float* db,
                          void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  return act_bwd_entry("ep_linear_act_bwd_f32", n, in, out, X, ldx, Zx, ldzx, act_x, W, dY, lddy, dX, lddx, dW, db,
                       workspace, workspace_bytes, stream);
}

int ep_linear_act_bwd_f64(int n, int in, int out, const double* X, int ldx, const double* Zx, int ldzx, int act_x,
                          const double* W, const double* dY, int lddy, double* dX, int lddx, double* dW, double* db,
                          void* workspace, size_t workspace_bytes, ep_stream_t stream) {
  return act_bwd_entry("ep_linear_act_bwd_f64", n, in, out, X, ldx, Zx, ldzx, act_x, W, dY, lddy, dX, lddx, dW, db,
                       workspace, workspace_bytes, stream);
}

}  // extern "C"
