// T = out_scale * X S on the tensor cores at fp32 accuracy: the k x k product of the eigen-loss backward.
//   X : n x k fp32 rows (M U of the level), S = Gp + Gp^T (k x k, symmetric), Gp = G_bar + diag(den_bar)
// dL/dU contains the dense term  MU_i S  per vertex (SURVEY Appendix A: U G_bar and MU G_bar^T folded for symmetric
// operators).  In the one-pass SIMT backward this product was 2 k^2 flops per vertex done with shuffles and
// shared-memory reads: instruction-issue bound, 53 % of that kernel's time at k = 32 and 75 % at k = 64 (round-1
// ncu).  It is a plain [n x k] . [k x k] contraction, so it runs here as tcgen05.mma kind::tf32 with the 3-pass
// split that keeps fp32 accuracy:
//     x = hi + lo,  hi = x with the 13 low mantissa bits cleared (exactly a TF32 number),  lo = x - hi (exact)
//     X S ~= X_hi S_hi + X_lo S_hi + X_hi S_lo        (dropped: lo * lo ~ 2^-22 relative)
// accumulated in fp32 in TMEM.  One 128-vertex tile per CTA iteration: rows are loaded from HBM coalesced, split and
// written to shared memory in the canonical no-swizzle K-major layout (8 rows x 16 B core matrices, the same layout
// mlp_tc.cu uses with 2-byte elements), 3 k/8 MMAs, accumulator drained row-per-thread.  HBM-bound: 8 n k bytes.
// Built for k = 64 only: at k = 32 the SIMT product of the one-pass backward hides behind its gather (B200, 1 M
// vertices: 0.45 ms for the one-pass kernel against 0.54 ms for this kernel + the gather pass).
#include "tc_common.cuh"
#include "eigen_coef.cuh"

namespace {

using namespace tc;

constexpr int SG_THREADS = 256;

// kind::tf32 instruction descriptor: tf32 x tf32 -> fp32, both operands K-major
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

// K = number of columns of X = order of S; one CTA handles tiles blockIdx.x, + gridDim.x, ...
template <int K>
__global__ void __launch_bounds__(SG_THREADS)
rows_times_sym_tf32x3_kernel(int row0, int n, const float* __restrict__ X, int ldx, const float* __restrict__ coef,
                             float out_scale_v, const float* __restrict__ out_scale_dev, float* __restrict__ T, int ldt) {
  static_assert(K == 64, "the drain reads 32 accumulator columns per half");
  constexpr int KC = K / 4;                          // 16-byte chunks (4 fp32) along K
  constexpr uint32_t A_BYTES = TILE_M * K * 4;
  constexpr uint32_t B_BYTES = K * K * 4;
  constexpr uint32_t TM_COLS = K;                    // power of two >= 32
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* A_hi = smem;
  uint8_t* A_lo = A_hi + A_BYTES;
  uint8_t* B_hi = A_lo + A_BYTES;
  uint8_t* B_lo = B_hi + B_BYTES;
  uint64_t* done = reinterpret_cast<uint64_t*>(B_lo + B_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float out_scale = out_scale_dev ? __ldg(out_scale_dev) : out_scale_v;
  if (threadIdx.x == 0) { mbar_init(done, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(tmem_slot, TM_COLS);
  // S = Gp + Gp^T from the finalize coefficients; B[n][kk] = S[kk][n] = S[n][kk], K-major, chunk-major in shared memory
  const ep::Coef<const float> cf(coef, K);
  for (int e = threadIdx.x; e < K * K; e += SG_THREADS) {
    const int nn = e / K, kk = e - nn * K;
    const float v = ep::coef_sym_entry(cf, K, e);
    const float hi = tf32_hi(v);
    const uint32_t off = (uint32_t)(kk >> 2) * (K * 16) + (uint32_t)nn * 16 + (uint32_t)(kk & 3) * 4;
    *reinterpret_cast<float*>(B_hi + off) = hi;
    *reinterpret_cast<float*>(B_lo + off) = v - hi;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc_tf32(TILE_M, K);
  const int n_tiles = (n + TILE_M - 1) / TILE_M;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    // ---- load + split: a warp iteration covers 8 rows x 4 chunks (64 contiguous bytes per row; the eight lanes of a
    //      quarter warp write 128 contiguous bytes of one chunk column -> conflict-free 16-byte shared stores)
    constexpr int BLOCKS = (TILE_M / 8) * (KC / 4);
    for (int b = warp; b < BLOCKS; b += SG_THREADS / 32) {
      const int rg = b / (KC / 4), cg = b - rg * (KC / 4);
      const int r = rg * 8 + (lane & 7), c = cg * 4 + (lane >> 3);
      const long long row = (long long)tile * TILE_M + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < n) v = __ldg(reinterpret_cast<const float4*>(X + (size_t)(row0 + row) * ldx + c * 4));
      const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
      const float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
      const uint32_t off = (uint32_t)c * CHUNK_BYTES + (uint32_t)r * 16;
      *reinterpret_cast<float4*>(A_hi + off) = hi;
      *reinterpret_cast<float4*>(A_lo + off) = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();                                  // operands written; every warp has drained the previous accumulator
    if (threadIdx.x == 0) {
      tc_fence_after();
      const uint32_t a_hi = smem_u32(A_hi), a_lo = smem_u32(A_lo), b_hi = smem_u32(B_hi), b_lo = smem_u32(B_lo);
#pragma unroll
      for (int j = 0; j < K / 8; ++j) {                // K = 8 per MMA = two 16-byte chunks
        const uint32_t ao = (uint32_t)(2 * j) * CHUNK_BYTES, bo = (uint32_t)(2 * j) * (K * 16);
        umma_tf32(tmem_base, make_desc(a_hi + ao, CHUNK_BYTES, 128), make_desc(b_hi + bo, K * 16, 128), idesc, j != 0);
        umma_tf32(tmem_base, make_desc(a_lo + ao, CHUNK_BYTES, 128), make_desc(b_hi + bo, K * 16, 128), idesc, 1u);
        umma_tf32(tmem_base, make_desc(a_hi + ao, CHUNK_BYTES, 128), make_desc(b_lo + bo, K * 16, 128), idesc, 1u);
      }
      umma_commit(done);
    }
    mbar_wait(done, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- drain: thread = one vertex row (TMEM lane quadrant = warp % 4), warps 4..7 take the upper half of the columns
    {
      const int q = warp & 3, half = warp >> 2;
      const long long row = (long long)tile * TILE_M + q * 32 + lane;
      constexpr int CPH = K / 2;                       // columns per half
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * CPH);
      float* dst = T + (size_t)(row0 + row) * ldt + half * CPH;
      uint32_t v[32];
      tmem_ld32(t_addr, v);
      if (row < n) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          reinterpret_cast<float4*>(dst)[j] = make_float4(out_scale * __uint_as_float(v[4 * j]), out_scale * __uint_as_float(v[4 * j + 1]),
                                                          out_scale * __uint_as_float(v[4 * j + 2]), out_scale * __uint_as_float(v[4 * j + 3]));
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, TM_COLS); }
}

template <int K>
int launch_rows_times_sym(int row0, int n, const float* X, int ldx, const float* coef, float scale, const float* scale_dev,
                          float* T, int ldt, cudaStream_t st) {
  const size_t smem = 2 * (size_t)TILE_M * K * 4 + 2 * (size_t)K * K * 4 + 8 + 16 + 128;
  static bool configured = false;
  if (!configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(rows_times_sym_tf32x3_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int n_tiles = (n + TILE_M - 1) / TILE_M;
  int grid = ep::sm_count() * 2;                                  // resident CTAs per SM (shared memory / TMEM columns)
  if (grid > n_tiles) grid = n_tiles;
  rows_times_sym_tf32x3_kernel<K><<<grid, SG_THREADS, smem, st>>>(row0, n, X, ldx, coef, scale, scale_dev, T, ldt);
  EP_LAUNCH_CHECK("rows_times_sym_tf32x3_kernel");
  return EP_OK;
}

}  // namespace

extern "C" {

int ep_eigen_bwd_gram_term_tf32x3(int row0, int n_rows, int k, const float* MU, int ld, const float* coef, float out_scale,
                                  const float* out_scale_dev, float* dU, int ldo, ep_stream_t stream) {
  EP_REQUIRE(n_rows >= 0 && row0 >= 0 && k > 0, "bad size");
  if (n_rows == 0) return EP_OK;
  EP_REQUIRE(MU && coef && dU, "null pointer");
  if (k != 64 || ld % 4 != 0 || ldo % 4 != 0 || !ep::aligned16(MU) || !ep::aligned16(dU)) {
    ep::set_error("ep_eigen_bwd_gram_term_tf32x3: k must be 64 and rows 16-byte aligned");
    return EP_ERR_UNSUPPORTED;
  }
  return launch_rows_times_sym<64>(row0, n_rows, MU, ld, coef, out_scale, out_scale_dev, dU, ldo, ep::as_stream(stream));
}

}  // extern "C"
