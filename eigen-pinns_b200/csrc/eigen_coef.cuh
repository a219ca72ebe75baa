// The coefficient vector of the eigen-loss backward: eigen_finalize_kernel writes it, the backward kernels of
// eigen_loss.cu and small_gemm_tc.cu read it (layout documented at ep_eigen_finalize_f32, include/eigenpinns_b200.h):
//   [c_res | lam (k) | num_bar (k) | den_bar (k) | G_bar (k x k, row-major) | g_mean (k)]   fp32
#pragma once

namespace ep {

__host__ __device__ constexpr int coef_len(int k) { return 1 + 4 * k + k * k; }

// The blocks of one coefficient vector; T = float for the writer, const float for the readers.
template <typename T>
struct Coef {
  T* c_res;
  T* lam;
  T* num_bar;
  T* den_bar;
  T* G_bar;
  T* g_mean;
  __device__ __forceinline__ Coef(T* coef, int k)
      : c_res(coef), lam(coef + 1), num_bar(lam + k), den_bar(num_bar + k), G_bar(den_bar + k), g_mean(G_bar + k * k) {}
};

// Entry e = m * k + j of the symmetric k x k factor of the dense backward term MU_i S:
//   S = Gp + Gp^T = G_bar + G_bar^T + 2 diag(den_bar),   Gp = G_bar + diag(den_bar)
__device__ __forceinline__ float coef_sym_entry(const Coef<const float>& c, int k, int e) {
  const int m = e / k, j = e - m * k;
  float v = c.G_bar[e] + c.G_bar[j * k + m];
  if (m == j) v += 2.f * c.den_bar[m];
  return v;
}

}  // namespace ep
