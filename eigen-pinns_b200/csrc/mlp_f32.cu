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

template <typename T>
int linear_bwd(int n, int in, int out, const T* X, int ldx, const T* W, const T* dY, int lddy, T* dX, int lddx,
               int relu_mask, T* dW, T* db, void* workspace, cudaStream_t st) {
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
      gemm_kernel<T, true, false><<<grid, 256, 0, st>>>(
          rows, in, out, dY + (size_t)r0 * lddy, lddy, 1, W, in, 1, dX + (size_t)r0 * lddx, lddx, 0, nullptr, 0,
          relu_mask ? X + (size_t)r0 * ldx : nullptr, ldx, out);
      EP_LAUNCH_CHECK("gemm_kernel<dX>");
    }
  }
  return EP_OK;
}

size_t bwd_workspace_bytes(int n, int in, int out, size_t elem) {
  if (n <= 0 || in <= 0 || out <= 0) return 0;
  BwdPlan p = plan_bwd(n, in, out);
  return elem * ((size_t)p.n_split * in * out + (size_t)p.cs_blocks * out);
}

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

}  // extern "C"
