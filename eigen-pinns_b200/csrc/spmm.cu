// CSR SpMM family for the stiffness / mass operators (HBM-bound gather kernels).
//
// Layout: A is CSR (int32 rowptr/col, fp32 or fp64 val), X / Y are row-major n x k of the same
// scalar type.  A "row group" of LPR lanes owns one output row; every lane owns V consecutive
// columns (V = 4 floats or 2 doubles when k, the leading dimensions and the base pointers allow
// 16-byte accesses), so one gathered row of X is read with LPR coalesced 16-byte loads (k = 32
// fp32 -> 8 lanes x 16 B = one 128-byte line; fp64 -> 16 lanes x 16 B = two lines).  With ~7 non-zeros per FEM row the non-zero loop is unrolled by 4 so that four
// gathers are in flight per lane before the first FMA.
//
// Algorithmic traffic (SURVEY 8d): single  8 nnz + 4 (n+1) + 8 n k   bytes
//                                  dual   12 nnz + 4 (n+1) + 12 n k  (both products)
//                                  sum    12 nnz + 4 (n+1) + 16 n k  (+4 n k when D given)
// fp64 (the notebook variants): 8-byte values and rows, e.g. dual 20 nnz + 4 (n+1) + 24 n k.
#include "ep_common.cuh"

namespace {

int g_spmm_waves = 4;      // persistent grid = this many full-machine waves (measured best on B200; tunable: ep_tune_set)

template <typename S, int V> struct VecT;
template <> struct VecT<float, 1> { using type = float; };
template <> struct VecT<float, 2> { using type = float2; };
template <> struct VecT<float, 4> { using type = float4; };
template <> struct VecT<double, 1> { using type = double; };
template <> struct VecT<double, 2> { using type = double2; };

template <typename T> __device__ __forceinline__ T vzero();
template <> __device__ __forceinline__ float vzero<float>() { return 0.f; }
template <> __device__ __forceinline__ float2 vzero<float2>() { return make_float2(0.f, 0.f); }
template <> __device__ __forceinline__ float4 vzero<float4>() { return make_float4(0.f, 0.f, 0.f, 0.f); }
template <> __device__ __forceinline__ double vzero<double>() { return 0.0; }
template <> __device__ __forceinline__ double2 vzero<double2>() { return make_double2(0.0, 0.0); }

__device__ __forceinline__ void vfma(float a, float x, float& acc) { acc = fmaf(a, x, acc); }
__device__ __forceinline__ void vfma(float a, float2 x, float2& acc) {
  acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y);
}
__device__ __forceinline__ void vfma(float a, float4 x, float4& acc) {
  acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y);
  acc.z = fmaf(a, x.z, acc.z); acc.w = fmaf(a, x.w, acc.w);
}
__device__ __forceinline__ void vfma(double a, double x, double& acc) { acc = fma(a, x, acc); }
__device__ __forceinline__ void vfma(double a, double2 x, double2& acc) {
  acc.x = fma(a, x.x, acc.x); acc.y = fma(a, x.y, acc.y);
}
__device__ __forceinline__ float vadd(float a, float b) { return a + b; }
__device__ __forceinline__ float2 vadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float4 vadd(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ double vadd(double a, double b) { return a + b; }
__device__ __forceinline__ double2 vadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float vscale(float a, float s) { return a * s; }
__device__ __forceinline__ float2 vscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
__device__ __forceinline__ float4 vscale(float4 a, float s) {
  return make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
}
__device__ __forceinline__ double vscale(double a, double s) { return a * s; }
__device__ __forceinline__ double2 vscale(double2 a, double s) { return make_double2(a.x * s, a.y * s); }

// MODE 0: YA = A XA            MODE 1: YA = A XA, YB = B XA
// MODE 2: YA = s (A XA + B XB + D)
template <typename S, int V, int MODE>
__global__ void __launch_bounds__(256)
spmm_kernel(int n_rows, int kv, int lpr_shift, const int32_t* __restrict__ rowptr,
            const int32_t* __restrict__ col, const S* __restrict__ valA,
            const S* __restrict__ valB, const S* __restrict__ XA,
            const S* __restrict__ XB, int ldx, const S* __restrict__ D, int ldd,
            S out_scale, const S* __restrict__ out_scale_dev, S* __restrict__ YA,
            S* __restrict__ YB, int ldy) {
  using T = typename VecT<S, V>::type;
  const int lpr = 1 << lpr_shift;
  const int lane = (int)(threadIdx.x & (lpr - 1));
  const long long groups_per_grid = ((long long)gridDim.x * blockDim.x) >> lpr_shift;
  // persistent row loop: the grid is sized to fill the machine once, every row group walks rows with a stride
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> lpr_shift; row < n_rows;
       row += groups_per_grid) {
    const int start = __ldg(rowptr + row);
    const int end = __ldg(rowptr + row + 1);
    for (int cv = lane; cv < kv; cv += lpr) {
      T accA = vzero<T>();
      T accB = vzero<T>();
      const S* xa = XA + (size_t)cv * V;
      const S* xb = (MODE == 2) ? XB + (size_t)cv * V : nullptr;
      for (int j = start; j < end; j += 4) {
        int c[4];
        S a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool ok = (j + u) < end;
          c[u] = ok ? __ldg(col + j + u) : -1;
          a[u] = ok ? __ldg(valA + j + u) : S(0);
          b[u] = (MODE != 0 && ok) ? __ldg(valB + j + u) : S(0);
        }
        T x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          x[u] = (c[u] >= 0) ? __ldg(reinterpret_cast<const T*>(xa + (size_t)c[u] * ldx)) : vzero<T>();
          if (MODE == 2)
            y[u] = (c[u] >= 0) ? __ldg(reinterpret_cast<const T*>(xb + (size_t)c[u] * ldx)) : vzero<T>();
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (c[u] >= 0) {
            vfma(a[u], x[u], accA);
            if (MODE == 1) vfma(b[u], x[u], accB);
            if (MODE == 2) vfma(b[u], y[u], accA);
          }
        }
      }
      if (MODE == 2) {
        if (D != nullptr)
          accA = vadd(accA, __ldg(reinterpret_cast<const T*>(D + (size_t)row * ldd + (size_t)cv * V)));
        accA = vscale(accA, out_scale_dev ? __ldg(out_scale_dev) : out_scale);
      }
      *reinterpret_cast<T*>(YA + (size_t)row * ldy + (size_t)cv * V) = accA;
      if (MODE == 1) *reinterpret_cast<T*>(YB + (size_t)row * ldy + (size_t)cv * V) = accB;
    }
  }
}

template <typename S, int MODE>
int launch_spmm(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const S* valA,
                const S* valB, const S* XA, const S* XB, int ldx, const S* D, int ldd,
                S out_scale, const S* out_scale_dev, S* YA, S* YB, int ldy, cudaStream_t st) {
  if (n_rows == 0 || k == 0) return EP_OK;
  int V = 1;
  auto ok_for = [&](int v) {
    if (k % v || ldx % v || ldy % v) return false;
    if (D && ldd % v) return false;
    const size_t mask = (size_t)v * sizeof(S) - 1;
    const void* ptrs[] = {XA, XB, D, YA, YB};
    for (const void* p : ptrs)
      if (p && (reinterpret_cast<uintptr_t>(p) & mask)) return false;
    return true;
  };
  if (sizeof(S) == 4 && ok_for(4)) V = 4; else if (ok_for(2)) V = 2;     // widest access: 16 bytes
  const int kv = k / V;
  int lpr_shift = 0;
  while ((1 << lpr_shift) < kv && lpr_shift < 5) ++lpr_shift;
  const long long threads = (long long)n_rows << lpr_shift;
  const int block = 256;
  long long grid = (threads + block - 1) / block;
  const long long cap = (long long)ep::sm_count() * 8 * g_spmm_waves;      // 8 CTAs of 256 threads fill one SM
  if (grid > cap) grid = cap;
#define EP_SPMM_LAUNCH(VV)                                                                      \
  spmm_kernel<S, VV, MODE><<<(unsigned)grid, block, 0, st>>>(n_rows, kv, lpr_shift, rowptr, col,   \
      valA, valB, XA, XB, ldx, D, ldd, out_scale, out_scale_dev, YA, YB, ldy)
  if (V == 1) EP_SPMM_LAUNCH(1);
  else if (V == 2) EP_SPMM_LAUNCH(2);
  else if constexpr (sizeof(S) == 4) EP_SPMM_LAUNCH(4);
#undef EP_SPMM_LAUNCH
  EP_LAUNCH_CHECK("spmm_kernel");
  return EP_OK;
}

// H[i, :d] = x[i, :];  H[i, d:2d] = mean over CSR neighbours of x (edge order), deg clamped to >= 1
__global__ void __launch_bounds__(256)
neighbor_mean_concat_kernel(int n, int d, const int32_t* __restrict__ rowptr,
                            const int32_t* __restrict__ col, const float* __restrict__ x, int ldx,
                            float* __restrict__ H, int ldh) {
  const int warps_per_block = blockDim.x >> 5;
  const int row = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const int start = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  const float deg = fmaxf((float)(end - start), 1.0f);
  for (int c = lane; c < d; c += 32) {
    float acc = 0.f;
    for (int j = start; j < end; ++j) acc += __ldg(x + (size_t)__ldg(col + j) * ldx + c);
    H[(size_t)row * ldh + c] = __ldg(x + (size_t)row * ldx + c);
    H[(size_t)row * ldh + d + c] = acc / deg;
  }
}

__global__ void __launch_bounds__(256)
copy2d_kernel(long long rows, int cols, const float* __restrict__ src, int lds, float* __restrict__ dst, int ldd) {
  const long long total = rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i - r * cols);
    dst[r * ldd + c] = src[r * lds + c];
  }
}

template <bool ADD>
__global__ void __launch_bounds__(256)
rows_indexed_kernel(int n_idx, int k, const int32_t* __restrict__ idx, const float* __restrict__ src,
                    int lds, float* __restrict__ dst, int ldd) {
  const long long total = (long long)n_idx * k;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / k);
    const int c = (int)(i - (long long)r * k);
    if (ADD) dst[(size_t)__ldg(idx + r) * ldd + c] += src[(size_t)r * lds + c];       // scatter-add
    else     dst[(size_t)r * ldd + c] = src[(size_t)__ldg(idx + r) * lds + c];        // gather
  }
}

int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = (long long)ep::sm_count() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" {

int ep_tune_set(int key, int value) {
  if (key == 1 && value >= 1 && value <= 64) { g_spmm_waves = value; return EP_OK; }
  if (key == 3 || key == 4) { ep::set_tune_flag(key, value); return EP_OK; }
  ep::set_error("ep_tune_set: unknown key or bad value");
  return EP_ERR_INVALID;
}

int ep_spmm_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const float* val,
                    const float* X, int ldx, float* Y, int ldy, ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && val && X && Y)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k, "leading dimension < k");
  return launch_spmm<float, 0>(n_rows, k, rowptr, col, val, nullptr, X, nullptr, ldx, nullptr, 0, 1.f, nullptr, Y,
                               nullptr, ldy, ep::as_stream(stream));
}

int ep_spmm_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const double* val,
                    const double* X, int ldx, double* Y, int ldy, ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && val && X && Y)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k, "leading dimension < k");
  return launch_spmm<double, 0>(n_rows, k, rowptr, col, val, nullptr, X, nullptr, ldx, nullptr, 0, 1.0, nullptr, Y,
                                nullptr, ldy, ep::as_stream(stream));
}

int ep_spmm2_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const float* valA,
                     const float* valB, const float* X, int ldx, float* YA, float* YB, int ldy,
                     ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && valA && valB && X && YA && YB)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k, "leading dimension < k");
  return launch_spmm<float, 1>(n_rows, k, rowptr, col, valA, valB, X, nullptr, ldx, nullptr, 0, 1.f, nullptr, YA, YB,
                               ldy, ep::as_stream(stream));
}

int ep_spmm2_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const double* valA,
                     const double* valB, const double* X, int ldx, double* YA, double* YB, int ldy,
                     ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && valA && valB && X && YA && YB)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k, "leading dimension < k");
  return launch_spmm<double, 1>(n_rows, k, rowptr, col, valA, valB, X, nullptr, ldx, nullptr, 0, 1.0, nullptr, YA, YB,
                                ldy, ep::as_stream(stream));
}

int ep_spmm2_sum_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                         const float* valA, const float* valB, const float* XA, const float* XB,
                         int ldx, const float* D, int ldd, float out_scale, const float* out_scale_dev, float* Y,
                         int ldy, ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && valA && valB && XA && XB && Y)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k && (!D || ldd >= k), "leading dimension < k");
  return launch_spmm<float, 2>(n_rows, k, rowptr, col, valA, valB, XA, XB, ldx, D, ldd, out_scale, out_scale_dev, Y,
                               nullptr, ldy, ep::as_stream(stream));
}

int ep_spmm2_sum_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                         const double* valA, const double* valB, const double* XA, const double* XB,
                         int ldx, const double* D, int ldd, double out_scale, const double* out_scale_dev, double* Y,
                         int ldy, ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
  EP_REQUIRE(rowptr && (n_rows == 0 || (col && valA && valB && XA && XB && Y)), "null pointer");
  EP_REQUIRE(ldx >= k && ldy >= k && (!D || ldd >= k), "leading dimension < k");
  return launch_spmm<double, 2>(n_rows, k, rowptr, col, valA, valB, XA, XB, ldx, D, ldd, out_scale, out_scale_dev, Y,
                                nullptr, ldy, ep::as_stream(stream));
}

int ep_neighbor_mean_concat_f32(int n, int d, const int32_t* rowptr, const int32_t* col,
                                const float* x, int ldx, float* H, int ldh, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && d >= 0, "negative size");
  if (n == 0 || d == 0) return EP_OK;
  EP_REQUIRE(rowptr && col && x && H, "null pointer");
  EP_REQUIRE(ldx >= d && ldh >= 2 * d, "leading dimension too small");
  const int block = 256, wpb = block / 32;
  neighbor_mean_concat_kernel<<<ep::ceil_div(n, wpb), block, 0, ep::as_stream(stream)>>>(
      n, d, rowptr, col, x, ldx, H, ldh);
  EP_LAUNCH_CHECK("neighbor_mean_concat_kernel");
  return EP_OK;
}

int ep_spmm_concat_f32(int n, int d, const int32_t* rowptr, const int32_t* col, const float* val,
                       const float* x, int ldx, float* H, int ldh, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && d >= 0, "negative size");
  if (n == 0 || d == 0) return EP_OK;
  EP_REQUIRE(rowptr && col && val && x && H, "null pointer");
  EP_REQUIRE(ldx >= d && ldh >= 2 * d, "leading dimension too small");
  cudaStream_t st = ep::as_stream(stream);
  copy2d_kernel<<<grid_for((long long)n * d, 256), 256, 0, st>>>(n, d, x, ldx, H, ldh);
  EP_LAUNCH_CHECK("copy2d_kernel");
  return launch_spmm<float, 0>(n, d, rowptr, col, val, nullptr, x, nullptr, ldx, nullptr, 0, 1.f, nullptr, H + d,
                        nullptr, ldh, st);
}

int ep_gather_rows_f32(int n_idx, int k, const int32_t* idx, const float* src, int lds, float* dst,
                       int ldd, ep_stream_t stream) {
  EP_REQUIRE(n_idx >= 0 && k >= 0, "negative size");
  if (n_idx == 0 || k == 0) return EP_OK;
  EP_REQUIRE(idx && src && dst, "null pointer");
  rows_indexed_kernel<false><<<grid_for((long long)n_idx * k, 256), 256, 0, ep::as_stream(stream)>>>(
      n_idx, k, idx, src, lds, dst, ldd);
  EP_LAUNCH_CHECK("gather_rows");
  return EP_OK;
}

int ep_scatter_add_rows_f32(int n_idx, int k, const int32_t* idx, const float* src, int lds, float* dst,
                            int ldd, ep_stream_t stream) {
  EP_REQUIRE(n_idx >= 0 && k >= 0, "negative size");
  if (n_idx == 0 || k == 0) return EP_OK;
  EP_REQUIRE(idx && src && dst, "null pointer");
  rows_indexed_kernel<true><<<grid_for((long long)n_idx * k, 256), 256, 0, ep::as_stream(stream)>>>(
      n_idx, k, idx, src, lds, dst, ldd);
  EP_LAUNCH_CHECK("scatter_add_rows");
  return EP_OK;
}

}  // extern "C"
