// tcgen05 / TMEM / mbarrier / bulk-copy helpers shared by the tensor-core kernels (sm_100a inline PTX).
#pragma once
#include <cuda_bf16.h>
#include "ep_common.cuh"
#include "dropout.cuh"

namespace tc {

constexpr int TILE_M = 128;
constexpr int CHUNK_BYTES = TILE_M * 16;          // one 8-feature chunk of a tile: 2048 B
constexpr int STAGE_CHUNKS = 4;                   // K = 32 per ring stage
constexpr int STAGE_BYTES = STAGE_CHUNKS * CHUNK_BYTES;   // 8 KB
constexpr int N_STAGES = 8;
constexpr int LINEAR_THREADS = 192;
constexpr uint32_t TMEM_COLS = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 26); ++spin)
    if (mbar_try_wait(bar, parity)) return;
  printf("eigenpinns_b200: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
  __trap();
}
// for the one thread whose reaction time is on the critical path (the MMA issuer): poll with test_wait - try_wait
// parks the thread in hardware and wakes it late when the shared-memory pipe is busy (~250 clk per wait measured)
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 28); ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return;
  }
  printf("eigenpinns_b200: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
  __trap();
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {       // non-blocking
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor, SWIZZLE_NONE, Blackwell version field = 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// kind::f16 instruction descriptor: bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
// max(x, 0) and round-to-nearest bf16 of two values in ONE instruction (upper half = hi, lower half = lo)
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// ---- ReLU bit mask ------------------------------------------------------------------------------------------
// One 32-bit word per (vertex row, block of 32 features).  Inside a block the features are stored as 16 packed
// bf16x2 words w_0..w_15 (w_i = features 2i | 2i+1); bit i of the mask word = "feature 2i is > 0", bit 16 + i =
// "feature 2i+1 is > 0", where > 0 refers to the STORED (ReLU'd, bf16) activation.  This order costs three integer
// instructions per PAIR to build (the halves of a ReLU'd word have a clear sign bit, so adding 0x7FFF to each half
// carries into bit 15 / 31 exactly when the half is non-zero) and four per pair to apply to a packed gradient word.
__device__ __forceinline__ uint32_t relu_mask_apply(uint32_t w, uint32_t mask_word, int i) {
  return w & (((mask_word >> i) & 0x00010001u) * 0xFFFFu);
}
// tcgen05.ld without the wait, and a wait that carries the destination registers as operands so that no use of
// them can be scheduled above it: lets the load of the next 32 columns fly while the current ones are processed.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
      : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
        "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
        "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
        "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
      :: "memory");
}
// One 32-column block of a hidden-layer epilogue: v = fp32 accumulators of one vertex row.
//   forward : w_i = bf16x2(relu(v + bias)), returns the ReLU mask word
//   dX      : w_i = bf16x2(v) & mask
__device__ __forceinline__ uint32_t epi_block_fwd(const uint32_t (&v)[32], const float4 (&b)[8], uint32_t (&w)[16]) {
#pragma unroll
  for (int g4 = 0; g4 < 8; ++g4) {
    w[2 * g4] = pack_relu_bf16x2(__uint_as_float(v[4 * g4]) + b[g4].x, __uint_as_float(v[4 * g4 + 1]) + b[g4].y);
    w[2 * g4 + 1] = pack_relu_bf16x2(__uint_as_float(v[4 * g4 + 2]) + b[g4].z, __uint_as_float(v[4 * g4 + 3]) + b[g4].w);
  }
  uint32_t acc[4] = {0u, 0u, 0u, 0u};             // four independent chains instead of one 16-deep dependency chain
#pragma unroll
  for (int i = 0; i < 16; ++i)                    // bit i <- lo half of w_i non-zero, bit 16 + i <- hi half
    acc[i & 3] |= ((w[i] + 0x7FFF7FFFu) >> (15 - i)) & (0x00010001u << i);
  return (acc[0] | acc[1]) | (acc[2] | acc[3]);
}
// the same with the bias read from shared memory where it is used (keeps 32 registers free for a second accumulator block)
__device__ __forceinline__ uint32_t epi_block_fwd_sb(const uint32_t (&v)[32], const float* bias_smem, uint32_t (&w)[16]) {
#pragma unroll
  for (int g4 = 0; g4 < 8; ++g4) {
    const float4 b = *reinterpret_cast<const float4*>(bias_smem + 4 * g4);
    w[2 * g4] = pack_relu_bf16x2(__uint_as_float(v[4 * g4]) + b.x, __uint_as_float(v[4 * g4 + 1]) + b.y);
    w[2 * g4 + 1] = pack_relu_bf16x2(__uint_as_float(v[4 * g4 + 2]) + b.z, __uint_as_float(v[4 * g4 + 3]) + b.w);
  }
  uint32_t acc[4] = {0u, 0u, 0u, 0u};
#pragma unroll
  for (int i = 0; i < 16; ++i)
    acc[i & 3] |= ((w[i] + 0x7FFF7FFFu) >> (15 - i)) & (0x00010001u << i);
  return (acc[0] | acc[1]) | (acc[2] | acc[3]);
}
__device__ __forceinline__ void epi_block_dx(const uint32_t (&v)[32], uint32_t mask_word, uint32_t (&w)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i)
    w[i] = relu_mask_apply(pack_bf16x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), mask_word, i);
}

// ---- dropout forms (dropout.cuh) ------------------------------------------------------------------------------
// Keep bits of a 32-column block (bit j = feature 8 * chunk0 + j kept): four Philox calls, chunks chunk0 .. chunk0 + 3.
__device__ __forceinline__ uint32_t keep_block32(unsigned long long seed, int step, int layer, long long row, int chunk0,
                                                 uint32_t thr) {
  uint32_t k = 0;
#pragma unroll
  for (int g = 0; g < 4; ++g) k |= dropout::keep_byte(seed, step, layer, row, chunk0 + g, thr) << (8 * g);
  return k;
}
// z = v + bias, scaled by s where kept and zeroed where dropped, then ReLU + bf16 as in epi_block_fwd; the ReLU mask is
// built from the packed value, so it is "kept and z > 0" and the backward needs nothing else to know the dropped units
__device__ __forceinline__ float drop_scale(float z, uint32_t keep, int j, float s) { return ((keep >> j) & 1u) ? z * s : 0.f; }
__device__ __forceinline__ uint32_t epi_mask_bits(const uint32_t (&w)[16]) {
  uint32_t acc[4] = {0u, 0u, 0u, 0u};
#pragma unroll
  for (int i = 0; i < 16; ++i)
    acc[i & 3] |= ((w[i] + 0x7FFF7FFFu) >> (15 - i)) & (0x00010001u << i);
  return (acc[0] | acc[1]) | (acc[2] | acc[3]);
}
__device__ __forceinline__ uint32_t epi_block_fwd_drop(const uint32_t (&v)[32], const float4 (&b)[8], uint32_t keep,
                                                       float s, uint32_t (&w)[16]) {
#pragma unroll
  for (int g4 = 0; g4 < 8; ++g4) {
    const int j = 4 * g4;
    w[2 * g4] = pack_relu_bf16x2(drop_scale(__uint_as_float(v[j]) + b[g4].x, keep, j, s),
                                 drop_scale(__uint_as_float(v[j + 1]) + b[g4].y, keep, j + 1, s));
    w[2 * g4 + 1] = pack_relu_bf16x2(drop_scale(__uint_as_float(v[j + 2]) + b[g4].z, keep, j + 2, s),
                                     drop_scale(__uint_as_float(v[j + 3]) + b[g4].w, keep, j + 3, s));
  }
  return epi_mask_bits(w);
}
__device__ __forceinline__ uint32_t epi_block_fwd_drop_sb(const uint32_t (&v)[32], const float* bias_smem, uint32_t keep,
                                                          float s, uint32_t (&w)[16]) {
#pragma unroll
  for (int g4 = 0; g4 < 8; ++g4) {
    const float4 b = *reinterpret_cast<const float4*>(bias_smem + 4 * g4);
    const int j = 4 * g4;
    w[2 * g4] = pack_relu_bf16x2(drop_scale(__uint_as_float(v[j]) + b.x, keep, j, s),
                                 drop_scale(__uint_as_float(v[j + 1]) + b.y, keep, j + 1, s));
    w[2 * g4 + 1] = pack_relu_bf16x2(drop_scale(__uint_as_float(v[j + 2]) + b.z, keep, j + 2, s),
                                     drop_scale(__uint_as_float(v[j + 3]) + b.w, keep, j + 3, s));
  }
  return epi_mask_bits(w);
}
// dX of a layer whose input had dropout: w_i = bf16x2(v * s) & mask (multiplied in fp32, rounded once)
__device__ __forceinline__ void epi_block_dx_scaled(const uint32_t (&v)[32], uint32_t mask_word, float s, uint32_t (&w)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i)
    w[i] = relu_mask_apply(pack_bf16x2(__uint_as_float(v[2 * i]) * s, __uint_as_float(v[2 * i + 1]) * s), mask_word, i);
}

}  // namespace tc
