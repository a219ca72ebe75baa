// Corrector MLP on the 5th-generation tensor cores (bf16 operands, fp32 accumulation in TMEM).
// Reference arithmetic: src/corrector_model.py:12-21,31 and the autograd backward of
// src/multigrid_model.py:258 (here analytic, layer by layer).
//
// ---- packed activation layout -------------------------------------------------------------------
// Activations (and their gradients) live in HBM as bf16 in 128-vertex tiles of "core-matrix-major"
// order:   packed[tile][c][r][8]   c = feature / 8 (16-byte chunk), r = vertex in tile (0..127),
// so one tile of a 256-wide layer is 64 KB contiguous.  This is exactly the tcgen05 canonical
// NO-SWIZZLE shared-memory layout, both ways round:
//   * as a K-major operand  (rows = vertices, K = features):  8 x 16 B core matrices, SBO = 128 B
//     between 8-vertex groups, LBO = 2048 B between feature chunks           -> forward, dX GEMMs
//   * as an MN-major operand (MN = features, K = vertices):   LBO(K-group) = 128 B, SBO(MN chunk)
//     = 2048 B                                                               -> dW = dZ^T H GEMM
// Hence a tile goes HBM -> SMEM with plain 1-D TMA bulk copies (cp.async.bulk, no tensor map), the
// epilogue's 16-byte stores of thread r / chunk c are perfectly coalesced (consecutive threads ->
// consecutive 16 B), and no transposition is ever materialised.
// Weights are re-packed (fp32 -> bf16) once per step into [K/8][N][8] (K-major B operand), both W
// and W^T.
//
// ---- kernels ------------------------------------------------------------------------------------
//  tc_linear_kernel   C = A W^T with W resident in SMEM for the whole (persistent) CTA, A tiles
//                     streamed through an 8-stage TMA ring, two TMEM accumulators so the epilogue of
//                     tile i overlaps the MMAs of tile i+1.  Epilogues: bias+ReLU -> packed bf16 |
//                     ReLU-mask -> packed bf16 (dX) | bias -> fp32 rows + U_pred = U_base + s*corr.
//  tc_dw_kernel       dW = X^T Y accumulated in TMEM over all tiles of the CTA (256 x 256 fp32 = all
//                     512 TMEM columns), both operands MN-major; the otherwise idle warps sum the
//                     columns of dZ from SMEM for db.  Per-CTA partials are reduced in fixed order.
// Warp roles: warp 0 = TMA producer (one lane), warp 1 = TMEM allocator + MMA issuer (one lane),
// warps 2..5 = epilogue (TMEM lane quadrant = warp % 4).
//
// Every layer is HBM-bound in this form (AI = 128 flop/B at width 256 vs. a ridge of ~250);
// DESIGN.md derives the byte counts the roofline numbers use.
#include "tc_common.cuh"

namespace tc {

enum LinearMode { MODE_HIDDEN = 0, MODE_DX = 1, MODE_FINAL = 2 };
// DROP (tc_linear_dropout_kernel): MODE_HIDDEN applies the dropout of dropout.cuh before the bf16 pack, MODE_DX scales
// the masked gradient by s (its mask was built from the dropped activation).

struct LinearArgs {
  const uint8_t* A;          // packed input tiles, KC chunks each
  const uint8_t* B;          // packed weights [KC][N][8] bf16
  int n_tiles, KC, N;
  const float* bias; int n_bias;   // bias[0..n_bias) (columns beyond are padding) or NULL
  int relu;
  uint8_t* out_packed;       // MODE_HIDDEN / MODE_DX: [tile][N/8][128][8]
  uint32_t* mask_out;        // MODE_HIDDEN: ReLU bit mask [row][N/32] (bit j of word w: activation 32w+j > 0), may be NULL
  const uint32_t* mask_in;   // MODE_DX: the bit mask written by the forward pass of the previous layer
  float* corr; int ldc;      // MODE_FINAL: fp32 rows
  const float* U_base; float* U_pred; int ldu; float scale; const float* scale_dev;
  int n_rows, n_out;
};

template <int MODE, bool DROP>
__device__ __forceinline__ void tc_linear_body(const LinearArgs& a, const dropout::Params& dp) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int KC = a.KC, N = a.N;
  uint8_t* Bs = smem;                                           // KC * N * 16 bytes
  uint8_t* As = Bs + (size_t)KC * N * 16;                       // N_STAGES * STAGE_BYTES
  uint64_t* bars = reinterpret_cast<uint64_t*>(As + N_STAGES * STAGE_BYTES);
  uint64_t* full = bars;                 // [N_STAGES]
  uint64_t* empty = bars + N_STAGES;     // [N_STAGES]
  uint64_t* tfull = bars + 2 * N_STAGES; // [2]
  uint64_t* tempty = tfull + 2;          // [2]
  uint64_t* bready = tempty + 2;         // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bready + 1);
  float* bias_s = reinterpret_cast<float*>(tmem_slot + 2);      // N floats
  float* stage_f = bias_s + N;                                  // MODE_FINAL only: 4 x 32 x 33 floats

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < N_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(&tfull[0], 1); mbar_init(&tfull[1], 1);
    mbar_init(&tempty[0], 128); mbar_init(&tempty[1], 128);
    mbar_init(bready, 1);
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < N; i += blockDim.x) bias_s[i] = (a.bias && i < a.n_bias) ? a.bias[i] : 0.f;
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int k_stages = KC / STAGE_CHUNKS;

  if (warp == 0) {
    if (lane == 0) {
      // resident weights: one barrier, copies of <= 64 KB
      const uint32_t b_bytes = (uint32_t)KC * N * 16;
      mbar_expect_tx(bready, b_bytes);
      for (uint32_t off = 0; off < b_bytes; off += 65536u) {
        const uint32_t len = min(65536u, b_bytes - off);
        bulk_g2s(Bs + off, a.B + off, len, bready);
      }
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const uint8_t* src = a.A + (size_t)tile * KC * CHUNK_BYTES;
        for (int ks = 0; ks < k_stages; ++ks) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], STAGE_BYTES);
          bulk_g2s(As + stage * STAGE_BYTES, src + (size_t)ks * STAGE_BYTES, STAGE_BYTES, &full[stage]);
          if (++stage == N_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(TILE_M, N, false, false);
      mbar_wait(bready, 0);
      tc_fence_after();
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      const uint32_t b_lbo = (uint32_t)N * 16;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_addr = tmem_base + (uint32_t)acc * 256u;
        for (int ks = 0; ks < k_stages; ++ks) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(As + stage * STAGE_BYTES);
#pragma unroll
          for (int j = 0; j < STAGE_CHUNKS / 2; ++j) {
            const uint64_t adesc = make_desc(a_base + j * 2 * CHUNK_BYTES, CHUNK_BYTES, 128);
            const uint64_t bdesc = make_desc(smem_u32(Bs) + (uint32_t)(ks * STAGE_CHUNKS + j * 2) * b_lbo, b_lbo, 128);
            umma_bf16(d_addr, adesc, bdesc, idesc, (ks | j) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (++stage == N_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // epilogue: thread = one vertex row of the tile; TMEM lane quadrant = warp % 4
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int ncb = N / 32;                              // 32-column blocks (<= 8)
    int acc = 0; uint32_t acc_phase = 0;
    const float scale = (MODE == MODE_FINAL && a.scale_dev) ? *a.scale_dev : a.scale;
    const int drop_step = (DROP && MODE == MODE_HIDDEN) ? dropout::step_of(dp) : 0;
    float* stg = stage_f + (size_t)q * 32 * 33;           // MODE_FINAL: per-warp 32 x 33 transpose buffer
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      const long long row = (long long)tile * TILE_M + r;
      uint32_t mw[8];
      if (MODE == MODE_DX) {                              // ReLU mask of this row, fetched before the MMAs finish
#pragma unroll
        for (int w = 0; w < 8; ++w) mw[w] = (w < ncb) ? __ldg(a.mask_in + (size_t)row * ncb + w) : 0u;
      }
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * 256u;
      const size_t tile_off = (size_t)tile * (N / 8) * CHUNK_BYTES + (size_t)r * 16;
      const int cb_end = (MODE == MODE_FINAL) ? ncb : 8;     // FINAL: runtime bound, not unrolled (register budget)
#pragma unroll
      for (int cb = 0; cb < cb_end; ++cb) {
        if (cb < ncb) {
          float ub[32];
          if (MODE == MODE_FINAL) {
            // U_base rows of this warp's 32 x 32 block, fetched (coalesced, all in flight) before the accumulator is read
            const int col = cb * 32 + lane;
            const long long row0 = (long long)tile * TILE_M + q * 32;
#pragma unroll
            for (int rr = 0; rr < 32; ++rr)
              ub[rr] = (a.U_base && col < a.n_out && row0 + rr < a.n_rows)
                           ? __ldg(a.U_base + (size_t)(row0 + rr) * a.ldu + col) : 0.f;
          }
          uint32_t v[32];
          tmem_ld32(t_addr + cb * 32, v);
          if (MODE == MODE_FINAL) {
            // transpose through shared memory so that every store instruction writes 128 contiguous bytes
#pragma unroll
            for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = __uint_as_float(v[j]) + bias_s[cb * 32 + j];
            __syncwarp();
            const int col = cb * 32 + lane;
            const long long row0 = (long long)tile * TILE_M + q * 32;
            if (col < a.n_out) {
#pragma unroll
              for (int rr = 0; rr < 32; ++rr) {
                const long long grow = row0 + rr;
                if (grow < a.n_rows) {
                  const float c = stg[rr * 33 + lane];
                  a.corr[(size_t)grow * a.ldc + col] = c;
                  if (a.U_pred) a.U_pred[(size_t)grow * a.ldu + col] = __fadd_rn(ub[rr], __fmul_rn(scale, c));
                }
              }
            }
            __syncwarp();
          } else {
            uint32_t w[16];
            uint32_t bits = 0;
            if (MODE == MODE_HIDDEN) {
              float4 b4[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) b4[j] = *reinterpret_cast<const float4*>(bias_s + cb * 32 + 4 * j);
              if constexpr (DROP) {
                const uint32_t keep = keep_block32(dp.seed, drop_step, dp.layer, dp.row0 + row, cb * 4, dp.thr);
                bits = epi_block_fwd_drop(v, b4, keep, dp.s, w);
              } else {
                bits = epi_block_fwd(v, b4, w);
              }
            }
            else if constexpr (DROP) epi_block_dx_scaled(v, mw[cb], dp.s, w);
            else epi_block_dx(v, mw[cb], w);
#pragma unroll
            for (int g = 0; g < 4; ++g)                       // 4 chunks of 8 columns
              *reinterpret_cast<uint4*>(a.out_packed + tile_off + (size_t)(cb * 4 + g) * CHUNK_BYTES) =
                  make_uint4(w[4 * g], w[4 * g + 1], w[4 * g + 2], w[4 * g + 3]);
            if (MODE == MODE_HIDDEN && a.mask_out) a.mask_out[(size_t)row * ncb + cb] = bits;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

template <int MODE>
__global__ void __launch_bounds__(LINEAR_THREADS, 1) tc_linear_kernel(LinearArgs a) {
  tc_linear_body<MODE, false>(a, dropout::Params{});
}

// MODE_HIDDEN / MODE_DX of a hidden layer followed by dropout
template <int MODE>
__global__ void __launch_bounds__(LINEAR_THREADS, 1) tc_linear_dropout_kernel(LinearArgs a, const dropout::Params dp) {
  tc_linear_body<MODE, true>(a, dp);
}

// ------------------------------------------------------------------------------------------- layer chain
// tc_chain2_kernel: ALL layers of the corrector MLP forward in one launch (corrector_model.py:31),
//   x0 -> relu(. W0^T + b0) -> ... -> . W_{L-1}^T + b_{L-1},
// run by CLUSTERS OF TWO CTAs with tcgen05.mma.cta_group::2.
// The activation tile never leaves the SM between layers: the epilogue of layer l writes bf16 straight into the
// shared-memory slot that is the A operand of layer l+1 (same packed K-major layout, in place) and, because the
// backward pass needs it, streams the same 16-byte chunks to HBM (write-only traffic; nothing is read back).
// Weights do not fit one SM (0.72 MB for 82->256x6->32), so they stream from L2 through a ring of K = 32 slabs.
// Why CTA pairs: a single CTA that holds two tiles cannot overlap the MMAs of one tile with the drain of another, since
// both TMEM accumulators and all shared memory that the weights leave belong to the tile pair in flight.  A CTA pair
// changes the budget:
//   * one MMA covers M = 256 rows, 128 from each CTA's operand tile, and the hardware takes HALF of the B operand from
//     each CTA's shared memory: a CTA stores only its N/2 output columns of every weight slab (8 KB instead of 16 KB per
//     K = 32), so a ring of 80 KB holds a whole layer (64 KB) and each CTA streams every layer ONCE per two tiles;
//   * a CTA therefore works on two tiles of its own in ping-pong ("slots" P and Q, one 64 KB operand tile and one
//     256-column accumulator each): while the pair's tensor cores run layer l of slot Q, all eight epilogue warps of
//     each CTA drain layer l of slot P and write the operand of layer l + 1 - and vice versa.  Both slots use the same
//     ring slots of layer l (P is their first reader, Q releases them).
// Barriers (rank 0 = leader, issues every MMA; counts in brackets: leader / peer):
//   wempty[s]     [1/1]      tcgen05.commit.cta_group::2 ... multicast: the pair's MMAs that read ring slot s have retired
//   landed[l & 1] [4/3]      all weight slabs of one layer are in this CTA's ring: one arrive.expect_tx per producer
//                            warp with the bytes of its slabs, complete_tx by every slab copy; leader: + one remote
//                            arrive by the peer
//   in_full[u]    [2/1]      input tile of slot u has landed; leader: + one remote arrive by the peer
//   acc_full[u]   [1/1]      commit multicast: all MMAs of one layer of slot u have retired -> epilogues of both CTAs
//   act_ready[u]  [512/-]    every epilogue thread of BOTH CTAs has drained its part of the accumulator and written +
//                            fenced its part of the next operand (the peer's threads arrive remotely)
// The peer forwards `landed` and `in_full` with one thread (warp 1, otherwise idle there).  Learned the hard
// way (clock64 traces, tools/prof_chain.py): (1) a remote arrive with .release.cluster semantics from the 256 epilogue
// threads costs ~2000 clk per step - it waits for the thread's outstanding HBM stores; the default semantics do not, and
// the operand tile is fenced into the async proxy before the arrive anyway; (2) every mbarrier try_wait in the
// MMA-issuing thread costs ~250 clk while the tensor pipe saturates shared memory, so a wait per weight slab (16 per
// layer) starves the tensor pipe (360 instead of 130 clk per MMA) - hence one barrier per LAYER and merged counts: the
// MMA thread waits for at most three barriers per (layer, slot) step and then issues 16 MMAs back to back.
// Weight slabs come from the second, "pair" copy of the packed weights ([K/32][half][4][N/2][8], see pack_weight_kernel):
// a CTA's half of a slab is one contiguous bulk copy; three warps take turns issuing them (a thread sustains one
// cp.async.bulk round per ~635 clk whatever its size, tools/micro/bulk_bw.cu).
// Work: cluster c takes units c, c + n_clusters, ...; unit = tiles (2 unit, 2 unit + 1), one per CTA.
// Algorithmic HBM bytes per vertex (82->256x6->32): read 2*96, write 6*(2*256 + 32) + 2*4*32 -> 3.7 KB, against
// 6.9 KB for the layer-by-layer kernels (every hidden activation is read back once).
// Measured (B200, 998,562 rows, 82->256x6->32): 0.99 ms against 1.08 ms for a single-CTA chain over the same tile pairs,
// bit-identical outputs.  Per 256-wide layer and CTA (two tiles): ~7800 clk against 10100; the tensor pipe is busy 34 %
// of the time (ncu, profiles/r02_ncu_chain2_summary.csv).  What bounds it now is the drain: 2600-3500 clk per
// 128 x 256 tile whether 8 or 16 warps do it, with or without the TMEM load of the next block in flight - the L1 /
// shared-memory data pipe carries 1400 wavefronts per tile for the epilogue (64 KB st.shared + 64 KB st.global + bias
// reads) plus 1024 for the MMA operands of the other slot (69 % busy over the kernel).
constexpr int CH_MAX_LAYERS = 8;
constexpr int CH_ACT_BYTES = 65536;           // one 128 x 256 bf16 tile

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

struct ChainLayer {
  const uint8_t* B;        // packed weights [KC][N][8] bf16, followed by their "pair" copy
  const float* bias;       // bias[0..n_bias) or NULL
  uint8_t* out_packed;     // [tile][N/8][128][8] or NULL (not stored)
  uint32_t* mask;          // ReLU bit mask written, or NULL (not stored)
  int KC, N, n_bias, pad_;
};
struct ChainArgs {
  const uint8_t* A0;       // packed input tiles, L[0].KC chunks each
  int n_tiles, n_layers;
  ChainLayer L[CH_MAX_LAYERS];
  float* corr; int ldc;    // last layer: fp32 rows (corr may be NULL)
  const float* U_base; float* U_pred; int ldu; float scale; const float* scale_dev;
  int n_rows, n_out, relu;
  unsigned long long* trace;   // optional timing trace of CTA 0 (clock64 stamps), experiments only
};
// dropout after the ReLU of every hidden layer l (tc_chain2_dropout_kernel); layer index = l, thr[l] = 0 keeps all
struct ChainDropout {
  unsigned long long seed;
  long long row0;
  const int* step_dev;
  int step, pad_;
  uint32_t thr[CH_MAX_LAYERS];
  float s[CH_MAX_LAYERS];
};

constexpr int C2_PRODUCERS = 3;               // weight-issuing warps: 0, 10, 11
constexpr int C2_THREADS = 384;               // + warp 1: MMA issuer (leader) / forwarder (peer), warps 2..9: epilogue.
                                              // Twelve warps = three per scheduler = up to 168 registers; a 13th caps at 128.
constexpr int C2_STAGES = 10;
constexpr int C2_SLOT_BYTES = 8192;           // K = 32 rows x 128 columns (this CTA's half of a 256-wide slab)
constexpr int C2_N_BARRIERS = C2_STAGES + 8;

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(const void* smem_ptr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(smem_ptr)), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z) : "memory");
}
__device__ __forceinline__ void umma2_commit_pair(uint64_t* bar) {     // arrives at this offset in BOTH CTAs
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot_in_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}

#define CHAIN2_DROPOUT 0
#include "chain2_kernel.cuh"
#undef CHAIN2_DROPOUT
// the chain with dropout after every hidden ReLU (ChainDropout): a separate kernel, so that the epilogue of the one
// above - the forward's limiter - carries no dropout code
#define CHAIN2_DROPOUT 1
#include "chain2_kernel.cuh"
#undef CHAIN2_DROPOUT

// ------------------------------------------------------------------------------------------- dW
constexpr int DW_THREADS = 192;
constexpr int DW_XSTAGES = 3;          // half tiles of X: 16 chunks = 32 KB
constexpr int DW_YSTAGES = 2;          // whole Y tiles: NCy chunks
constexpr int XHALF_CHUNKS = 16;
constexpr int XHALF_BYTES = XHALF_CHUNKS * CHUNK_BYTES;

struct DwArgs {
  const uint8_t* X;   // packed, Mdim features (128 or 256)
  const uint8_t* Y;   // packed, Ndim features (multiple of 32, <= 256)
  int n_tiles, Mdim, Ndim;
  int db_from_y;      // 0: column sums of X, 1: column sums of Y
  float* partial;     // [grid][Mdim * Ndim]
  float* db_partial;  // [grid][256]
};

__global__ void __launch_bounds__(DW_THREADS, 1) tc_dw_kernel(DwArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int NCy = a.Ndim / 8;
  const int y_bytes = NCy * CHUNK_BYTES;
  const int m_halves = a.Mdim / 128;
  uint8_t* Xs = smem;                                         // DW_XSTAGES * XHALF_BYTES
  uint8_t* Ys = Xs + DW_XSTAGES * XHALF_BYTES;                // DW_YSTAGES * y_bytes
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ys + (size_t)DW_YSTAGES * y_bytes);
  uint64_t* xfull = bars;                         // [3]
  uint64_t* xempty = bars + DW_XSTAGES;           // [3]
  uint64_t* yfull = xempty + DW_XSTAGES;          // [2]
  uint64_t* yempty = yfull + DW_YSTAGES;          // [2]
  uint64_t* done = yempty + DW_YSTAGES;           // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < DW_XSTAGES; ++s) { mbar_init(&xfull[s], 1); mbar_init(&xempty[s], a.db_from_y ? 1 : 129); }
    for (int s = 0; s < DW_YSTAGES; ++s) { mbar_init(&yfull[s], 1); mbar_init(&yempty[s], a.db_from_y ? 129 : 1); }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int xs = 0, ys = 0; uint32_t xph = 0, yph = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        mbar_wait(&yempty[ys], yph ^ 1);
        mbar_expect_tx(&yfull[ys], (uint32_t)y_bytes);
        bulk_g2s(Ys + (size_t)ys * y_bytes, a.Y + (size_t)tile * y_bytes, (uint32_t)y_bytes, &yfull[ys]);
        if (++ys == DW_YSTAGES) { ys = 0; yph ^= 1; }
        for (int mh = 0; mh < m_halves; ++mh) {
          mbar_wait(&xempty[xs], xph ^ 1);
          mbar_expect_tx(&xfull[xs], XHALF_BYTES);
          bulk_g2s(Xs + xs * XHALF_BYTES, a.X + ((size_t)tile * m_halves + mh) * XHALF_BYTES, XHALF_BYTES, &xfull[xs]);
          if (++xs == DW_XSTAGES) { xs = 0; xph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(128, a.Ndim, true, true);
      int xs = 0, ys = 0; uint32_t xph = 0, yph = 0;
      bool first = true;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        mbar_wait(&yfull[ys], yph);
        tc_fence_after();
        const uint32_t y_base = smem_u32(Ys + (size_t)ys * y_bytes);
        for (int mh = 0; mh < m_halves; ++mh) {
          mbar_wait(&xfull[xs], xph);
          tc_fence_after();
          const uint32_t x_base = smem_u32(Xs + xs * XHALF_BYTES);
#pragma unroll
          for (int s = 0; s < TILE_M / 16; ++s) {              // 16 vertices (two 8-row K groups) per MMA
            const uint64_t adesc = make_desc(x_base + s * 256, 128, CHUNK_BYTES);
            const uint64_t bdesc = make_desc(y_base + s * 256, 128, CHUNK_BYTES);
            umma_bf16(tmem_base + (uint32_t)mh * 256u, adesc, bdesc, idesc, (!first || s > 0) ? 1u : 0u);
          }
          umma_commit(&xempty[xs]);
          if (++xs == DW_XSTAGES) { xs = 0; xph ^= 1; }
        }
        umma_commit(&yempty[ys]);
        if (++ys == DW_YSTAGES) { ys = 0; yph ^= 1; }
        first = false;
      }
      umma_commit(done);
    }
  } else {
    // ---- db: column sums of the dZ operand straight from shared memory (conflict-free 16 B reads)
    const int we = warp - 2;                     // 0..3
    float acc[2][4][8];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[h][c][j] = 0.f;
    int xs = 0, ys = 0; uint32_t xph = 0, yph = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      if (a.db_from_y) {
        mbar_wait(&yfull[ys], yph);
        const uint8_t* yb = Ys + (size_t)ys * y_bytes;
#pragma unroll
        for (int slot = 0; slot < 8; ++slot) {          // chunk = we + 4 * slot (NCy <= 32)
          const int c = we + 4 * slot;
          if (c < NCy) {
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
              const uint4 w = *reinterpret_cast<const uint4*>(yb + (size_t)c * CHUNK_BYTES + (rr * 32 + lane) * 16);
              const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (int j = 0; j < 8; ++j)
                acc[slot >> 2][slot & 3][j] += __uint_as_float(((ww[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) << 16);
            }
          }
        }
        mbar_arrive(&yempty[ys]);
        if (++ys == DW_YSTAGES) { ys = 0; yph ^= 1; }
      } else {
        for (int mh = 0; mh < m_halves; ++mh) {
          mbar_wait(&xfull[xs], xph);
          const uint8_t* xb = Xs + xs * XHALF_BYTES;
#pragma unroll
          for (int cl = 0; cl < 4; ++cl) {
            const int c = we * 4 + cl;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
              const uint4 w = *reinterpret_cast<const uint4*>(xb + (size_t)c * CHUNK_BYTES + (rr * 32 + lane) * 16);
              const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float val = __uint_as_float(((ww[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) << 16);
                if (mh == 0) acc[0][cl][j] += val; else acc[1][cl][j] += val;
              }
            }
          }
          mbar_arrive(&xempty[xs]);
          if (++xs == DW_XSTAGES) { xs = 0; xph ^= 1; }
        }
      }
    }
    float* dbp = a.db_partial + (size_t)blockIdx.x * 256;
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float s = ep::warp_sum(acc[h][c][j]);
          if (lane == 0) {
            // feature index of this accumulator
            const int feat = a.db_from_y ? ((we + 4 * (h * 4 + c)) * 8 + j) : (h * 128 + (we * 4 + c) * 8 + j);
            if (feat < 256) dbp[feat] = s;
          }
        }
    // ---- final: TMEM -> per-CTA fp32 partial
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3;
    float* part = a.partial + (size_t)blockIdx.x * a.Mdim * a.Ndim;
    for (int mh = 0; mh < m_halves; ++mh) {
      const int m = mh * 128 + q * 32 + lane;
      for (int cb = 0; cb < a.Ndim / 32; ++cb) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)mh * 256u + cb * 32, v);
        float4* dst = reinterpret_cast<float4*>(part + (size_t)m * a.Ndim + cb * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                               __uint_as_float(v[4 * j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// out[o][i] = sum_cta partial[cta][m][n], (m, n) = (o, i) or (i, o) when transposed.  64 outputs per block,
// four thread groups split the CTA partials and are combined in a fixed order (deterministic).
__global__ void __launch_bounds__(256)
dw_reduce_kernel(int n_cta, int Mdim, int Ndim, const float* __restrict__ partial, int out_rows, int out_cols,
                 int transposed, float* __restrict__ dW, const float* __restrict__ db_partial, int db_len,
                 float* __restrict__ db) {
  __shared__ float sh[4][64];
  const int total = out_rows * out_cols;
  const int el = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int e = blockIdx.x * 64 + el;
  float s = 0.f;
  if (e < total) {
    const int o = e / out_cols, i = e - o * out_cols;
    const size_t idx = transposed ? (size_t)i * Ndim + o : (size_t)o * Ndim + i;
    const size_t stride = (size_t)Mdim * Ndim;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int c = g;
    for (; c + 12 < n_cta; c += 16) {
      s0 += partial[(size_t)c * stride + idx];
      s1 += partial[(size_t)(c + 4) * stride + idx];
      s2 += partial[(size_t)(c + 8) * stride + idx];
      s3 += partial[(size_t)(c + 12) * stride + idx];
    }
    for (; c < n_cta; c += 4) s0 += partial[(size_t)c * stride + idx];
    s = (s0 + s1) + (s2 + s3);
  }
  sh[g][el] = s;
  __syncthreads();
  if (g == 0 && e < total) dW[e] = (sh[0][el] + sh[1][el]) + (sh[2][el] + sh[3][el]);
  if (blockIdx.x == 0) {
    for (int f = threadIdx.x; f < db_len; f += blockDim.x) {
      float t = 0.f;
      for (int c = 0; c < n_cta; ++c) t += db_partial[(size_t)c * 256 + f];
      db[f] = t;
    }
  }
}

// ------------------------------------------------------------------------------------------- packing
// fp32 rows [n x d] -> packed bf16 tiles [tile][dp/8][128][8], zero padded (rows >= n, cols >= d)
__global__ void __launch_bounds__(256)
pack_rows_kernel(int n, int d, int dp, const float* __restrict__ X, int ldx, uint8_t* __restrict__ out, int n_tiles) {
  // item = one 16-byte chunk.  A warp covers 8 rows x 4 chunks: reads are 128 contiguous bytes per row,
  // writes 128 contiguous bytes per chunk column (8 rows x 16 B).
  const int nc = dp / 8, ncg = nc / 4;                                // dp is a multiple of 32
  const long long total = (long long)n_tiles * nc * TILE_M;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < total;
       it += (long long)gridDim.x * blockDim.x) {
    const int lane = (int)(it & 31);
    const long long w = it >> 5;
    const int rg = (int)(w & 15);
    const long long w2 = w >> 4;
    const int cg = (int)(w2 % ncg);
    const long long tile = w2 / ncg;
    const int r = rg * 8 + (lane >> 2);
    const int c = cg * 4 + (lane & 3);
    const long long row = tile * TILE_M + r;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = c * 8 + j;
      f[j] = (row < n && col < d) ? __ldg(X + (size_t)row * ldx + col) : 0.f;
    }
    uint4 o;
    o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
    o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(out + (((size_t)tile * nc + c) * TILE_M + r) * 16) = o;
  }
}

// W fp32 [out x in] -> Wp [inp/8][outp][8] (B operand of the forward GEMM) and WTp [outp/8][inp][8] (dX GEMM), each
// followed by a second copy in the layout of the CTA-pair chain kernel: [K/32 slabs][half of N][4 chunks][N/2][8], so that
// the N/2 columns one CTA of a pair needs of a K = 32 slab are contiguous (K = in, N = out for Wp; K = out, N = in for WTp).
constexpr int W_REPLICAS = 2;
__global__ void __launch_bounds__(256)
pack_weight_kernel(int out, int in, int outp, int inp, const float* __restrict__ W, __nv_bfloat16* __restrict__ Wp,
                   __nv_bfloat16* __restrict__ WTp, bool pair_copy) {
  const int total = outp * inp;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int o = e / inp, i = e - o * inp;
    const float w = (o < out && i < in) ? __ldg(W + (size_t)o * in + i) : 0.f;
    const __nv_bfloat16 b = __float2bfloat16_rn(w);
    Wp[(size_t)(i >> 3) * outp * 8 + (size_t)o * 8 + (i & 7)] = b;
    if (WTp) WTp[(size_t)(o >> 3) * inp * 8 + (size_t)i * 8 + (o & 7)] = b;
    if (pair_copy) {
      {
        const int kc = i >> 3, nh = outp >> 1, half = o >= nh ? 1 : 0;
        Wp[(size_t)total + ((size_t)(((kc >> 2) * 2 + half) * 4 + (kc & 3)) * nh + (o - half * nh)) * 8 + (i & 7)] = b;
      }
      if (WTp) {
        const int kc = o >> 3, nh = inp >> 1, half = i >= nh ? 1 : 0;
        WTp[(size_t)total + ((size_t)(((kc >> 2) * 2 + half) * 4 + (kc & 3)) * nh + (i - half * nh)) * 8 + (o & 7)] = b;
      }
    }
  }
}

inline int pad_to(int v, int m) { return (v + m - 1) / m * m; }
inline int n_tiles_for(int n) { return (n + TILE_M - 1) / TILE_M; }

}  // namespace tc

using namespace tc;

namespace {

template <int MODE>
int launch_linear(const LinearArgs& a, cudaStream_t st, int max_ctas = 0, const dropout::Params* dp = nullptr) {
  const size_t smem = (size_t)a.KC * a.N * 16 + (size_t)N_STAGES * STAGE_BYTES + 8 * (2 * N_STAGES + 5) + 16 +
                      sizeof(float) * a.N + (MODE == MODE_FINAL ? sizeof(float) * 4 * 32 * 33 : 0) + 128;
  int grid = ep::sm_count();
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  if (grid > a.n_tiles) grid = a.n_tiles;
  if constexpr (MODE != MODE_FINAL) {
    if (dp) {
      static size_t configured_drop = 0;
      if (smem > configured_drop) {
        EP_CUDA_CHECK(cudaFuncSetAttribute(tc_linear_dropout_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem));
        configured_drop = smem;
      }
      tc_linear_dropout_kernel<MODE><<<grid, LINEAR_THREADS, smem, st>>>(a, *dp);
      EP_LAUNCH_CHECK("tc_linear_dropout_kernel");
      return EP_OK;
    }
  }
  static size_t configured = 0;
  if (smem > configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(tc_linear_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  tc_linear_kernel<MODE><<<grid, LINEAR_THREADS, smem, st>>>(a);
  EP_LAUNCH_CHECK("tc_linear_kernel");
  return EP_OK;
}

bool dims_ok(int kp, int np) { return kp % 32 == 0 && np % 32 == 0 && kp >= 32 && np >= 32 && kp <= 256 && np <= 256; }

int launch_chain(const ChainArgs& a, cudaStream_t st, const ChainDropout* dp = nullptr) {
  // one cluster of two CTAs per unit of two tiles, at most one CTA per SM
  const size_t smem = 2 * (size_t)CH_ACT_BYTES + (size_t)C2_STAGES * C2_SLOT_BYTES + sizeof(float) * CH_MAX_LAYERS * 256 +
                      8 * C2_N_BARRIERS + 16 + 128;
  const int n_pairs = (a.n_tiles + 1) / 2;
  int clusters = ep::sm_count() / 2;
  if (clusters > n_pairs) clusters = n_pairs;
  ChainArgs b = a;
  if (dp) {
    static bool configured_drop = false;
    if (!configured_drop) {
      EP_CUDA_CHECK(cudaFuncSetAttribute(tc_chain2_dropout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      configured_drop = true;
    }
    tc_chain2_dropout_kernel<<<2 * clusters, C2_THREADS, smem, st>>>(b, *dp);
    EP_LAUNCH_CHECK("tc_chain2_dropout_kernel");
    return EP_OK;
  }
  static bool configured = false;
  if (!configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(tc_chain2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  b.trace = reinterpret_cast<unsigned long long*>(((uintptr_t)(uint32_t)ep::tune_flag(4) << 32) | (uint32_t)ep::tune_flag(3));
  tc_chain2_kernel<<<2 * clusters, C2_THREADS, smem, st>>>(b);
  EP_LAUNCH_CHECK("tc_chain2_kernel");
  return EP_OK;
}

int chain_dims_ok(const char* who, int n_layers, const int* dims_padded) {
  if (n_layers < 1 || n_layers > CH_MAX_LAYERS || !dims_padded) {
    ep::set_error("%s: 1 <= n_layers <= %d", who, CH_MAX_LAYERS);
    return EP_ERR_UNSUPPORTED;
  }
  for (int l = 0; l <= n_layers; ++l)
    if (dims_padded[l] % 32 != 0 || dims_padded[l] < 32 || dims_padded[l] > 256) {
      ep::set_error("%s: padded widths must be multiples of 32 in [32, 256]", who);
      return EP_ERR_UNSUPPORTED;
    }
  return EP_OK;
}

}  // namespace

extern "C" {

int ep_tc_pad_features(int d, int wide) { return wide ? pad_to(d, 128) : pad_to(d, 32); }

size_t ep_tc_packed_rows_bytes(int n, int d_padded) {
  if (n <= 0 || d_padded <= 0) return 0;
  return (size_t)n_tiles_for(n) * TILE_M * d_padded * 2;
}

size_t ep_tc_packed_weight_bytes(int out_padded, int in_padded) { return (size_t)W_REPLICAS * out_padded * in_padded * 2; }

size_t ep_tc_relu_mask_bytes(int n, int d_padded) {
  if (n <= 0 || d_padded <= 0) return 0;
  return (size_t)n_tiles_for(n) * TILE_M * (d_padded / 32) * 4;
}

int ep_tc_pack_rows_bf16(int n, int d, int d_padded, const float* X, int ldx, void* packed, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && d > 0 && d_padded >= d && d_padded % 32 == 0, "bad size (d_padded must be a multiple of 32)");
  EP_REQUIRE(X && packed && ldx >= d, "bad argument");
  const int nt = n_tiles_for(n);
  const long long total = (long long)nt * (d_padded / 8) * TILE_M;
  long long grid = (total + 255) / 256;
  if (grid > (long long)ep::sm_count() * 16) grid = (long long)ep::sm_count() * 16;
  pack_rows_kernel<<<(unsigned)grid, 256, 0, ep::as_stream(stream)>>>(n, d, d_padded, X, ldx, static_cast<uint8_t*>(packed), nt);
  EP_LAUNCH_CHECK("pack_rows_kernel");
  return EP_OK;
}

int ep_tc_pack_weight_bf16(int out, int in, int out_padded, int in_padded, const float* W, void* Wp, void* WTp,
                           ep_stream_t stream) {
  EP_REQUIRE(out > 0 && in > 0 && out_padded >= out && in_padded >= in, "bad size");
  EP_REQUIRE(out_padded % 8 == 0 && in_padded % 8 == 0 && W && Wp, "bad argument");
  const int total = out_padded * in_padded;
  pack_weight_kernel<<<ep::ceil_div(total, 256), 256, 0, ep::as_stream(stream)>>>(
      out, in, out_padded, in_padded, W, static_cast<__nv_bfloat16*>(Wp), static_cast<__nv_bfloat16*>(WTp),
      out_padded % 32 == 0 && in_padded % 32 == 0);
  EP_LAUNCH_CHECK("pack_weight_kernel");
  return EP_OK;
}

int ep_tc_linear_fwd_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed, const void* Wp,
                          const float* bias, int relu, void* out_packed, void* relu_mask_out, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && A_packed && Wp && out_packed, "bad argument");
  if (!relu) { ep::set_error("ep_tc_linear_fwd_bf16: hidden layers are Linear + ReLU (relu must be 1)"); return EP_ERR_UNSUPPORTED; }
  if (!dims_ok(in_padded, out_padded)) { ep::set_error("ep_tc_linear_fwd_bf16: padded dims must be multiples of 32 in [32, 256]"); return EP_ERR_UNSUPPORTED; }
  LinearArgs a{};
  a.A = static_cast<const uint8_t*>(A_packed); a.B = static_cast<const uint8_t*>(Wp);
  a.n_tiles = n_tiles_for(n); a.KC = in_padded / 8; a.N = out_padded; a.bias = bias; a.n_bias = out; a.relu = relu;
  a.out_packed = static_cast<uint8_t*>(out_packed); a.mask_out = static_cast<uint32_t*>(relu_mask_out);
  a.n_rows = n; a.n_out = out_padded;
  return launch_linear<MODE_HIDDEN>(a, ep::as_stream(stream));
}

int ep_tc_linear_final_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed, const void* Wp,
                            const float* bias, float* corr, int ldc, const float* U_base, float scale,
                            const float* scale_dev, float* U_pred, int ldu, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && A_packed && Wp && corr && out > 0 && out <= out_padded && ldc >= out, "bad argument");
  EP_REQUIRE((U_base == nullptr) == (U_pred == nullptr) && (!U_pred || ldu >= out), "U_base / U_pred mismatch");
  if (!dims_ok(in_padded, out_padded)) { ep::set_error("ep_tc_linear_final_bf16: unsupported dims"); return EP_ERR_UNSUPPORTED; }
  LinearArgs a{};
  a.A = static_cast<const uint8_t*>(A_packed); a.B = static_cast<const uint8_t*>(Wp);
  a.n_tiles = n_tiles_for(n); a.KC = in_padded / 8; a.N = out_padded; a.bias = bias; a.n_bias = out;
  a.corr = corr; a.ldc = ldc; a.U_base = U_base; a.U_pred = U_pred; a.ldu = ldu; a.scale = scale; a.scale_dev = scale_dev;
  a.n_rows = n; a.n_out = out;
  return launch_linear<MODE_FINAL>(a, ep::as_stream(stream));
}

int ep_tc_linear_fwd_dropout_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed, const void* Wp,
                                  const float* bias, void* out_packed, void* relu_mask_out, float p,
                                  unsigned long long seed, int step, const int* step_dev, int layer, long long row0,
                                  ep_stream_t stream) {
  EP_REQUIRE(n > 0 && A_packed && Wp && out_packed, "bad argument");
  if (!dims_ok(in_padded, out_padded)) { ep::set_error("ep_tc_linear_fwd_dropout_bf16: padded dims must be multiples of 32 in [32, 256]"); return EP_ERR_UNSUPPORTED; }
  dropout::Params dp{};
  if (int rc = dropout::host_params("ep_tc_linear_fwd_dropout_bf16", p, &dp.thr, &dp.s)) return rc;
  dp.seed = seed; dp.row0 = row0; dp.step_dev = step_dev; dp.step = step; dp.layer = layer;
  LinearArgs a{};
  a.A = static_cast<const uint8_t*>(A_packed); a.B = static_cast<const uint8_t*>(Wp);
  a.n_tiles = n_tiles_for(n); a.KC = in_padded / 8; a.N = out_padded; a.bias = bias; a.n_bias = out; a.relu = 1;
  a.out_packed = static_cast<uint8_t*>(out_packed); a.mask_out = static_cast<uint32_t*>(relu_mask_out);
  a.n_rows = n; a.n_out = out_padded;
  return launch_linear<MODE_HIDDEN>(a, ep::as_stream(stream), 0, &dp);
}

int ep_tc_linear_dx_dropout_bf16(int n, int out_padded, int in_padded, const void* dZ_packed, const void* WTp,
                                 const void* relu_mask, void* dZprev_packed, float p, int max_ctas, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && dZ_packed && WTp && relu_mask && dZprev_packed, "bad argument");
  if (!dims_ok(out_padded, in_padded)) { ep::set_error("ep_tc_linear_dx_dropout_bf16: unsupported dims"); return EP_ERR_UNSUPPORTED; }
  dropout::Params dp{};
  if (int rc = dropout::host_params("ep_tc_linear_dx_dropout_bf16", p, &dp.thr, &dp.s)) return rc;
  LinearArgs a{};
  a.A = static_cast<const uint8_t*>(dZ_packed); a.B = static_cast<const uint8_t*>(WTp);
  a.n_tiles = n_tiles_for(n); a.KC = out_padded / 8; a.N = in_padded;
  a.out_packed = static_cast<uint8_t*>(dZprev_packed); a.mask_in = static_cast<const uint32_t*>(relu_mask);
  a.n_rows = n; a.n_out = in_padded;
  return launch_linear<MODE_DX>(a, ep::as_stream(stream), max_ctas, &dp);
}

int ep_tc_linear_dx_bf16(int n, int out_padded, int in_padded, const void* dZ_packed, const void* WTp,
                         const void* relu_mask, void* dZprev_packed, int max_ctas, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && dZ_packed && WTp && relu_mask && dZprev_packed, "bad argument");
  if (!dims_ok(out_padded, in_padded)) { ep::set_error("ep_tc_linear_dx_bf16: unsupported dims"); return EP_ERR_UNSUPPORTED; }
  LinearArgs a{};
  a.A = static_cast<const uint8_t*>(dZ_packed); a.B = static_cast<const uint8_t*>(WTp);
  a.n_tiles = n_tiles_for(n); a.KC = out_padded / 8; a.N = in_padded;
  a.out_packed = static_cast<uint8_t*>(dZprev_packed); a.mask_in = static_cast<const uint32_t*>(relu_mask);
  a.n_rows = n; a.n_out = in_padded;
  return launch_linear<MODE_DX>(a, ep::as_stream(stream), max_ctas);
}

}  // extern "C"

namespace {

int chain_fwd(const char* who, int n, int n_layers, const int* dims_padded, const int* dims_out, const void* A0_packed,
              const void* const* Wp, const float* const* bias, void* const* act_out, void* const* relu_mask_out,
              float* corr, int ldc, const float* U_base, float scale, const float* scale_dev, float* U_pred, int ldu,
              const ChainDropout* dp, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && A0_packed && Wp && bias && dims_out, "bad argument");
  EP_REQUIRE(n_layers >= 2, "the forward chain needs at least one hidden layer");
  if (int rc = chain_dims_ok(who, n_layers, dims_padded)) return rc;
  const int k = dims_out[n_layers - 1];
  EP_REQUIRE(k > 0 && k <= dims_padded[n_layers], "bad output width");
  EP_REQUIRE((U_base == nullptr) == (U_pred == nullptr) && (!U_pred || ldu >= k) && (!corr || ldc >= k),
             "U_base / U_pred / corr mismatch");
  EP_REQUIRE(corr || U_pred, "nothing to write");
  ChainArgs a{};
  a.A0 = static_cast<const uint8_t*>(A0_packed);
  a.n_tiles = n_tiles_for(n); a.n_layers = n_layers;
  for (int l = 0; l < n_layers; ++l) {
    EP_REQUIRE(Wp[l], "null weight pointer");
    a.L[l].B = static_cast<const uint8_t*>(Wp[l]);
    a.L[l].bias = bias[l];
    a.L[l].KC = dims_padded[l] / 8; a.L[l].N = dims_padded[l + 1]; a.L[l].n_bias = dims_out[l];
    const bool hidden = l + 1 < n_layers;
    a.L[l].out_packed = (hidden && act_out) ? static_cast<uint8_t*>(act_out[l]) : nullptr;
    a.L[l].mask = (hidden && relu_mask_out) ? static_cast<uint32_t*>(relu_mask_out[l]) : nullptr;
  }
  a.corr = corr; a.ldc = ldc; a.U_base = U_base; a.U_pred = U_pred; a.ldu = ldu; a.scale = scale; a.scale_dev = scale_dev;
  a.n_rows = n; a.n_out = k; a.relu = 1;
  return launch_chain(a, ep::as_stream(stream), dp);
}

}  // namespace

extern "C" {

int ep_tc_chain_fwd_bf16(int n, int n_layers, const int* dims_padded, const int* dims_out, const void* A0_packed,
                         const void* const* Wp, const float* const* bias, void* const* act_out,
                         void* const* relu_mask_out, float* corr, int ldc, const float* U_base, float scale,
                         const float* scale_dev, float* U_pred, int ldu, ep_stream_t stream) {
  return chain_fwd("ep_tc_chain_fwd_bf16", n, n_layers, dims_padded, dims_out, A0_packed, Wp, bias, act_out,
                   relu_mask_out, corr, ldc, U_base, scale, scale_dev, U_pred, ldu, nullptr, stream);
}

int ep_tc_chain_fwd_dropout_bf16(int n, int n_layers, const int* dims_padded, const int* dims_out, const void* A0_packed,
                                 const void* const* Wp, const float* const* bias, void* const* act_out,
                                 void* const* relu_mask_out, float* corr, int ldc, const float* U_base, float scale,
                                 const float* scale_dev, float* U_pred, int ldu, const float* p_layers, float p,
                                 unsigned long long seed, int step, const int* step_dev, long long row0,
                                 ep_stream_t stream) {
  ChainDropout dp{};
  dp.seed = seed; dp.row0 = row0; dp.step_dev = step_dev; dp.step = step;
  EP_REQUIRE(n_layers >= 2 && n_layers <= CH_MAX_LAYERS, "1 <= hidden layers < 8");
  for (int l = 0; l + 1 < n_layers; ++l)
    if (int rc = dropout::host_params("ep_tc_chain_fwd_dropout_bf16", p_layers ? p_layers[l] : p, &dp.thr[l], &dp.s[l]))
      return rc;
  return chain_fwd("ep_tc_chain_fwd_dropout_bf16", n, n_layers, dims_padded, dims_out, A0_packed, Wp, bias, act_out,
                   relu_mask_out, corr, ldc, U_base, scale, scale_dev, U_pred, ldu, &dp, stream);
}

size_t ep_tc_dw_workspace_bytes(void) { return sizeof(float) * (size_t)ep::sm_count() * (256 * 256 + 256); }

int ep_tc_linear_dw_bf16(int n, int out, int in, int out_padded, int in_padded, const void* dZ_packed,
                         const void* act_packed, float* dW, float* db, void* workspace, size_t workspace_bytes,
                         int max_ctas, ep_stream_t stream) {
  EP_REQUIRE(n > 0 && dZ_packed && act_packed && dW && db && workspace, "bad argument");
  EP_REQUIRE(out <= out_padded && in <= in_padded, "bad padding");
  if (workspace_bytes < ep_tc_dw_workspace_bytes()) { ep::set_error("ep_tc_linear_dw_bf16: workspace too small"); return EP_ERR_WORKSPACE; }
  DwArgs a{};
  int transposed;
  if (out_padded % 128 == 0 && out_padded <= 256 && in_padded % 32 == 0 && in_padded <= 256) {
    a.X = static_cast<const uint8_t*>(dZ_packed); a.Y = static_cast<const uint8_t*>(act_packed);
    a.Mdim = out_padded; a.Ndim = in_padded; a.db_from_y = 0; transposed = 0;
  } else if (in_padded % 128 == 0 && in_padded <= 256 && out_padded % 32 == 0 && out_padded <= 256) {
    a.X = static_cast<const uint8_t*>(act_packed); a.Y = static_cast<const uint8_t*>(dZ_packed);
    a.Mdim = in_padded; a.Ndim = out_padded; a.db_from_y = 1; transposed = 1;
  } else {
    ep::set_error("ep_tc_linear_dw_bf16: one padded dimension must be 128 or 256, the other a multiple of 32 <= 256");
    return EP_ERR_UNSUPPORTED;
  }
  a.n_tiles = n_tiles_for(n);
  int grid = ep::sm_count();
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  if (grid > a.n_tiles) grid = a.n_tiles;
  a.partial = static_cast<float*>(workspace);
  a.db_partial = a.partial + (size_t)ep::sm_count() * 256 * 256;
  const size_t smem = (size_t)DW_XSTAGES * XHALF_BYTES + (size_t)DW_YSTAGES * (a.Ndim / 8) * CHUNK_BYTES +
                      8 * (2 * DW_XSTAGES + 2 * DW_YSTAGES + 1) + 16 + 128;
  static size_t configured = 0;
  if (smem > configured) {
    EP_CUDA_CHECK(cudaFuncSetAttribute(tc_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  cudaStream_t st = ep::as_stream(stream);
  tc_dw_kernel<<<grid, DW_THREADS, smem, st>>>(a);
  EP_LAUNCH_CHECK("tc_dw_kernel");
  const int total = out * in;
  dw_reduce_kernel<<<ep::ceil_div(total, 64), 256, 0, st>>>(
      grid, a.Mdim, a.Ndim, a.partial, out, in, transposed, dW, a.db_partial, out, db);
  EP_LAUNCH_CHECK("dw_reduce_kernel");
  return EP_OK;
}

}  // extern "C"
