// tc_chain2_kernel (CHAIN2_DROPOUT 0) and tc_chain2_dropout_kernel (CHAIN2_DROPOUT 1): mlp_tc.cu includes this body
// twice, inside namespace tc after the chain's helpers.  The dropout lines are preprocessor blocks rather than a
// template parameter so that the compiler sees tc_chain2_kernel token for token as it was before dropout existed: the
// kernel runs twelve warps under a 168-register cap, and even an inlined body function changes its register allocation.
// See the notes above tc_chain2_kernel in mlp_tc.cu for the design.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(C2_THREADS, 1)
#if CHAIN2_DROPOUT
tc_chain2_dropout_kernel(const __grid_constant__ ChainArgs a, const __grid_constant__ ChainDropout dp) {
#else
tc_chain2_kernel(const __grid_constant__ ChainArgs a) {
#endif
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* act0 = smem;                                   // operand tile of slot P
  uint8_t* act1 = smem + CH_ACT_BYTES;                    // operand tile of slot Q
  uint8_t* ring = smem + 2 * CH_ACT_BYTES;
  float* bias_s = reinterpret_cast<float*>(ring + C2_STAGES * C2_SLOT_BYTES);          // [CH_MAX_LAYERS][256]
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + CH_MAX_LAYERS * 256);
  uint64_t* wempty = bars;                         // [C2_STAGES]
  uint64_t* landed = wempty + C2_STAGES;           // [2]
  uint64_t* in_full = landed + 2;                  // [2]
  uint64_t* acc_full = in_full + 2;                // [2]
  uint64_t* act_ready = acc_full + 2;              // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + C2_N_BARRIERS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = a.n_layers;
  const int rank = (int)cluster_ctarank();
  const bool leader = rank == 0;
  if (threadIdx.x == 0) {
    for (int s = 0; s < C2_STAGES; ++s) mbar_init(&wempty[s], 1);
    for (int u = 0; u < 2; ++u) {
      mbar_init(&landed[u], C2_PRODUCERS + (leader ? 1 : 0));
      mbar_init(&in_full[u], leader ? 2 : 1);
      mbar_init(&acc_full[u], 1);
      mbar_init(&act_ready[u], 512);
    }
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < L * 256; i += blockDim.x) {
    const int l = i >> 8, c = i & 255;
    bias_s[i] = (a.L[l].bias && c < a.L[l].n_bias) ? a.L[l].bias[c] : 0.f;
  }
  if (warp == 1) tmem_alloc2(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                 // both CTAs' barriers and TMEM exist before anything crosses over
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_units = (a.n_tiles + 1) >> 1;
  const int n_clusters = (int)gridDim.x >> 1;
  const int cluster_id = (int)blockIdx.x >> 1;
  const int my_units = cluster_id < n_units ? (n_units - cluster_id + n_clusters - 1) / n_clusters : 0;
  auto unit_of = [&](int j) { return cluster_id + j * n_clusters; };
  const uint32_t in_bytes = (uint32_t)a.L[0].KC * CHUNK_BYTES;

  if (warp == 0 || warp >= 10) {
    // ---- weights: this CTA's N/2 output columns of every K = 32 slab, each layer once per unit pair; the slabs of the
    //      whole sequence are dealt round-robin to the C2_PRODUCERS issuing warps
    if (lane == 0) {
      const int me = warp == 0 ? 0 : warp - 9;
      uint32_t gs = 0;                               // slab counter over the whole sequence
      uint32_t lc = 0;                               // layer counter over the whole sequence
      for (int j = 0; j < my_units; j += 2) {
        for (int l = 0; l < L; ++l, ++lc) {
          const int N = a.L[l].N;
          const uint32_t half_bytes = (uint32_t)(N >> 1) * 64u;          // 4 chunks x N/2 columns x 16 B
          const int n_slabs = a.L[l].KC >> 2;
          const uint8_t* src = a.L[l].B + (size_t)a.L[l].KC * N * 16 + (size_t)rank * half_bytes;    // the "pair" copy
          // Every producer announces the bytes of ITS slabs of this layer with one arrive.expect_tx (so the transaction
          // count never goes negative) - after the barrier's previous phase (layer lc - 2) is complete.
          {
            int mine = 0;
            for (int s = 0; s < n_slabs; ++s) mine += ((gs + s) % C2_PRODUCERS) == (uint32_t)me ? 1 : 0;
            if (lc >= 2) mbar_wait(&landed[lc & 1], ((lc - 2) >> 1) & 1);
            if (mine) mbar_expect_tx(&landed[lc & 1], (uint32_t)mine * half_bytes);
            else mbar_arrive(&landed[lc & 1]);
          }
          for (int s = 0; s < n_slabs; ++s, ++gs) {
            if ((int)(gs % C2_PRODUCERS) != me) continue;
            const uint32_t stage = gs % C2_STAGES, phase = (gs / C2_STAGES) & 1;
            mbar_wait(&wempty[stage], phase ^ 1);
            bulk_g2s(ring + stage * C2_SLOT_BYTES, src + (size_t)s * 2 * half_bytes, half_bytes, &landed[lc & 1]);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && !leader) {
      // ---- peer: tell the leader when a layer's weights / the input tile of a slot have landed here (or that there is
      //      no tile); the two event streams interleave, so poll both
      const uint32_t remote_w[2] = {map_to_cta(&landed[0], 0), map_to_cta(&landed[1], 0)};
      const uint32_t remote_i[2] = {map_to_cta(&in_full[0], 0), map_to_cta(&in_full[1], 0)};
      const uint32_t n_layers_total = (uint32_t)((my_units + 1) >> 1) * (uint32_t)L;
      uint32_t lc = 0, nu[2] = {0, 0};
      int j = 0;
      for (uint32_t spin = 0; lc < n_layers_total || j < my_units; ++spin) {
        if (lc < n_layers_total && mbar_test(&landed[lc & 1], (lc >> 1) & 1)) { mbar_arrive_remote(remote_w[lc & 1]); ++lc; spin = 0; }
        if (j < my_units) {
          const int u = j & 1;
          if (2 * unit_of(j) + rank >= a.n_tiles || mbar_test(&in_full[u], nu[u] & 1)) {
            mbar_arrive_remote(remote_i[u]); ++nu[u]; ++j; spin = 0;
          }
        }
        if (spin > (1u << 28)) { printf("eigenpinns_b200: forwarder timed out (block %d)\n", blockIdx.x); __trap(); }
      }
    } else if (lane == 0) {
      // ---- leader: every MMA of the pair
      uint32_t stage = 0;
      uint32_t lc = 0;
      uint32_t gl[2] = {0, 0};                       // layers completed per slot
      uint32_t nu[2] = {0, 0};                       // units started per slot
      const uint32_t abase[2] = {smem_u32(act0), smem_u32(act1)};
      for (int j = 0; j < my_units; j += 2) {
        const bool has_q = (j + 1) < my_units;
        for (int l = 0; l < L; ++l, ++lc) {
          const int N = a.L[l].N;
          const uint32_t idesc = make_idesc(256, N, false, false);
          const uint32_t b_lbo = (uint32_t)(N >> 1) * 16;
          const int n_slabs = a.L[l].KC >> 2;
          for (int u = 0; u < (has_q ? 2 : 1); ++u) {
            if (l == 0) mbar_wait_spin(&in_full[u], nu[u] & 1);
            if (u == 0) mbar_wait_spin(&landed[lc & 1], (lc >> 1) & 1);
            if (gl[u] > 0) mbar_wait_spin(&act_ready[u], (gl[u] - 1) & 1);
            tc_fence_after();
            const uint32_t tg = gl[0] + gl[1];
            if (a.trace && blockIdx.x == 0 && tg < 64) a.trace[tg * 8 + 0] = clock64();      // operands ready
            const bool releases = (u == 1) || !has_q;       // last reader of the layer's slots
            for (int s = 0; s < n_slabs; ++s) {
              uint32_t slot = stage + s;
              if (slot >= C2_STAGES) slot -= C2_STAGES;
              const uint32_t b_base = smem_u32(ring + slot * C2_SLOT_BYTES);
#pragma unroll
              for (int jj = 0; jj < 2; ++jj) {
                const uint64_t bdesc = make_desc(b_base + (uint32_t)(jj * 2) * b_lbo, b_lbo, 128);
                const uint64_t adesc = make_desc(abase[u] + (uint32_t)(s * 4 + jj * 2) * CHUNK_BYTES, CHUNK_BYTES, 128);
                umma2_bf16(tmem_base + (uint32_t)u * 256u, adesc, bdesc, idesc, (s | jj) != 0 ? 1u : 0u);
              }
              if (releases) umma2_commit_pair(&wempty[slot]);
            }
            umma2_commit_pair(&acc_full[u]);
            if (a.trace && blockIdx.x == 0 && tg < 64) a.trace[tg * 8 + 1] = clock64();      // all MMAs issued
            ++gl[u];
          }
          stage += n_slabs;
          if (stage >= C2_STAGES) stage -= C2_STAGES;
        }
        ++nu[0]; ++nu[1];
      }
    }
  } else {
    // ---- epilogue: 8 warps on ONE tile (slot u of the current step); TMEM lane quadrant q, column half hf
    const int q = warp & 3;
    const int hf = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const bool elected = (warp == 2 && lane == 0);
    const uint32_t ready_remote[2] = {map_to_cta(&act_ready[0], 0), map_to_cta(&act_ready[1], 0)};
    auto issue_input = [&](int j) {                    // input tile of this CTA for its j-th unit -> slot j & 1
      const int u = j & 1;
      const int tile = 2 * unit_of(j) + rank;
      if (tile < a.n_tiles) {
        mbar_expect_tx(&in_full[u], in_bytes);
        bulk_g2s(u ? act1 : act0, a.A0 + (size_t)tile * in_bytes, in_bytes, &in_full[u]);
      }
    };
    if (elected) { if (my_units > 0) issue_input(0); if (my_units > 1) issue_input(1); }
    const float scale = a.scale_dev ? *a.scale_dev : a.scale;
#if CHAIN2_DROPOUT
    const int drop_step = dp.step_dev ? *dp.step_dev : dp.step;
#endif
    const bool vec_out = ((a.ldc | a.ldu | a.n_out) & 3) == 0 &&
                         ((reinterpret_cast<uintptr_t>(a.corr) | reinterpret_cast<uintptr_t>(a.U_base) |
                           reinterpret_cast<uintptr_t>(a.U_pred)) & 15u) == 0;
    uint32_t gl[2] = {0, 0};
    for (int j = 0; j < my_units; j += 2) {
      const bool has_q = (j + 1) < my_units;
      for (int l = 0; l < L; ++l) {
        const int N = a.L[l].N, ncb = N >> 5;
        const int my_cb = min(4, ncb - 4 * hf);           // 32-column blocks of this warp (<= 0: none)
        uint8_t* const out_packed = a.L[l].out_packed;
        uint32_t* const mask_ptr = a.L[l].mask;
        const float* bl = bias_s + l * 256 + hf * 128;
        const bool last = (l == L - 1);
        for (int u = 0; u < (has_q ? 2 : 1); ++u) {
          const int tile = 2 * unit_of(j + u) + rank;
          const bool valid = tile < a.n_tiles;
          const bool work = valid && my_cb > 0;
          const long long row = (long long)tile * TILE_M + r;
          uint8_t* act = u ? act1 : act0;
          const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)u * 256u + (uint32_t)hf * 128u;
          float4 ub[8];
          const bool final_rows = last && work && row < a.n_rows;
          if (final_rows && vec_out && a.U_pred) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              const int col = hf * 128 + 4 * jj;
              ub[jj] = col < a.n_out ? __ldg(reinterpret_cast<const float4*>(a.U_base + (size_t)row * a.ldu + col))
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
          mbar_wait(&acc_full[u], gl[u] & 1);
          tc_fence_after();
          const uint32_t tg = gl[0] + gl[1];
          if (a.trace && blockIdx.x == 0 && tg < 64 && threadIdx.x == 64) a.trace[tg * 8 + 2] = clock64();   // accumulator ready
          if (last && elected && (j + u + 2) < my_units) issue_input(j + u + 2);     // slot u's operand tile is free
          if (work) {
            if (last) {
              const bool in_rows = row < a.n_rows;
              for (int cb = 0; cb < my_cb; ++cb) {
                const int col0 = hf * 128 + cb * 32;
                if (cb > 0 && vec_out && in_rows && a.U_pred) {
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) {
                    const int col = col0 + 4 * jj;
                    ub[jj] = col < a.n_out ? __ldg(reinterpret_cast<const float4*>(a.U_base + (size_t)row * a.ldu + col))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
                }
                uint32_t v[32];
                tmem_ld32(t_addr + cb * 32, v);
                if (in_rows) {
                  if (vec_out) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                      const int col = col0 + 4 * jj;
                      if (col < a.n_out) {
                        const float4 bj = *reinterpret_cast<const float4*>(bl + cb * 32 + 4 * jj);
                        float4 c;
                        c.x = __uint_as_float(v[4 * jj]) + bj.x;     c.y = __uint_as_float(v[4 * jj + 1]) + bj.y;
                        c.z = __uint_as_float(v[4 * jj + 2]) + bj.z; c.w = __uint_as_float(v[4 * jj + 3]) + bj.w;
                        if (a.corr) *reinterpret_cast<float4*>(a.corr + (size_t)row * a.ldc + col) = c;
                        if (a.U_pred) {
                          float4 uu;
                          uu.x = __fadd_rn(ub[jj].x, __fmul_rn(scale, c.x)); uu.y = __fadd_rn(ub[jj].y, __fmul_rn(scale, c.y));
                          uu.z = __fadd_rn(ub[jj].z, __fmul_rn(scale, c.z)); uu.w = __fadd_rn(ub[jj].w, __fmul_rn(scale, c.w));
                          *reinterpret_cast<float4*>(a.U_pred + (size_t)row * a.ldu + col) = uu;
                        }
                      }
                    }
                  } else {
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                      const int col = col0 + jj;
                      if (col < a.n_out) {
                        const float c = __uint_as_float(v[jj]) + bl[cb * 32 + jj];
                        if (a.corr) a.corr[(size_t)row * a.ldc + col] = c;
                        if (a.U_pred)
                          a.U_pred[(size_t)row * a.ldu + col] =
                              __fadd_rn(__ldg(a.U_base + (size_t)row * a.ldu + col), __fmul_rn(scale, c));
                      }
                    }
                  }
                }
              }
            } else {
              const size_t tile_off = (size_t)tile * (N >> 3) * CHUNK_BYTES + (size_t)r * 16;
              const bool to_smem = !last;
              uint32_t bits[4];
              uint32_t va[32], vb[32];                     // two accumulator blocks: the load of block cb + 1 flies
              tmem_ld32_issue(t_addr, va);                 // while block cb is converted and stored
#pragma unroll
              for (int cb = 0; cb < 4; ++cb) {
                if (cb < my_cb) {
                  uint32_t (&v)[32] = (cb & 1) ? vb : va;
                  tmem_ld32_wait(v);
                  if (cb + 1 < my_cb) tmem_ld32_issue(t_addr + (cb + 1) * 32, (cb & 1) ? va : vb);
                  uint32_t w[16];
#if CHAIN2_DROPOUT
                  const uint32_t keep = keep_block32(dp.seed, drop_step, l, dp.row0 + row, (hf * 4 + cb) * 4, dp.thr[l]);
                  bits[cb] = epi_block_fwd_drop_sb(v, bl + cb * 32, keep, dp.s[l], w);
#else
                  bits[cb] = epi_block_fwd_sb(v, bl + cb * 32, w);
#endif
#pragma unroll
                  for (int g4 = 0; g4 < 4; ++g4) {
                    const uint4 o = make_uint4(w[4 * g4], w[4 * g4 + 1], w[4 * g4 + 2], w[4 * g4 + 3]);
                    const size_t c_off = (size_t)((hf * 4 + cb) * 4 + g4) * CHUNK_BYTES;
                    if (to_smem) *reinterpret_cast<uint4*>(act + c_off + (size_t)r * 16) = o;
                    if (out_packed) *reinterpret_cast<uint4*>(out_packed + tile_off + c_off) = o;
                  }
                } else {
                  bits[cb] = 0u;
                }
              }
              if (mask_ptr) {
                uint32_t* mrow = mask_ptr + (size_t)row * ncb + 4 * hf;
                if (my_cb == 4) {
                  *reinterpret_cast<uint4*>(mrow) = make_uint4(bits[0], bits[1], bits[2], bits[3]);
                } else {
#pragma unroll
                  for (int cb = 0; cb < 4; ++cb) if (cb < my_cb) mrow[cb] = bits[cb];
                }
              }
            }
          }
          if (a.trace && blockIdx.x == 0 && tg < 64 && threadIdx.x == 64) a.trace[tg * 8 + 3] = clock64();   // drained
          if (!last) fence_proxy_async_smem();           // generic-proxy writes -> visible to the tensor core of this SM
          tc_fence_before();
          mbar_arrive_remote(ready_remote[u]);         // the leader's barrier, whichever CTA this is
          if (a.trace && blockIdx.x == 0 && tg < 64 && threadIdx.x == 64) a.trace[tg * 8 + 4] = clock64();   // arrived
          ++gl[u];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                 // neither CTA leaves (or frees TMEM) while the other may still signal it
  if (warp == 1) { tc_fence_after(); tmem_dealloc2(tmem_base, TMEM_COLS); }
}
