// Counter-based dropout masks of the corrector's hidden layers (the nn.Dropout after every hidden ReLU of
// src/corrector_model.py::_build_net), shared by the fp32 and the tcgen05 kernels so that both modes drop the same units.
//
// The keep decision of hidden layer `layer`, vertex row `row` (row of the MLP input) and output feature `col` is a pure
// function of (seed, step, layer, row, col): it is regenerated wherever it is needed and never stored.
//   Philox4x32-10 (Salmon et al., SC'11):  key = seed (lo, hi),  counter = (row, col / 8, layer, step)
//   one call = four 32-bit words = eight 16-bit lanes, one per feature of the 8-column chunk col / 8:
//     feature 8c + 2j <- low half of word j,  8c + 2j + 1 <- high half of word j
//   keep  <=>  lane >= thr,  thr = round(p * 65536) in [0, 65536),  kept units are scaled by s = 1 / (1 - thr / 65536)
// so P(keep) = 1 - p_q with p_q = thr / 65536 (|p_q - p| <= 2^-17) and E[y] = relu(z) exactly.  These masks are not
// torch's RNG stream: a dropout run matches the reference in distribution only.  oracle/dropout_port.py is the numpy
// port (bit-identical).
#pragma once
#include <stdint.h>

namespace dropout {

// Everything a kernel needs to regenerate / apply the masks of one layer (or, in the chain, of every layer).
struct Params {
  unsigned long long seed;
  long long row0;            // added to the row index (vertex offset of a shard; 0 on one GPU)
  const int* step_dev;       // overrides step when not NULL (the Adam step t of a captured graph)
  int step;
  int layer;
  uint32_t thr;              // round(p * 65536); 0 keeps everything
  float s;                   // 1 / (1 - thr / 65536)
};

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Keep bits of one 8-feature chunk: bit f (0..7) = feature 8 * chunk + f is kept.
__host__ __device__ __forceinline__ uint32_t keep_byte(unsigned long long seed, int step, int layer, long long row,
                                                       int chunk, uint32_t thr) {
  uint32_t w[4];
  philox4x32_10((uint32_t)row, (uint32_t)chunk, (uint32_t)layer, (uint32_t)step, (uint32_t)seed,
                (uint32_t)(seed >> 32), w);
  uint32_t bits = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    bits |= ((w[j] & 0xFFFFu) >= thr ? 1u : 0u) << (2 * j);
    bits |= ((w[j] >> 16) >= thr ? 1u : 0u) << (2 * j + 1);
  }
  return bits;
}

// thr and s of a drop probability p; EP_ERR_INVALID (and the library's error string) unless 0 <= p and thr < 65536
int host_params(const char* who, float p, uint32_t* thr, float* s);

__device__ __forceinline__ int step_of(const Params& d) { return d.step_dev ? *d.step_dev : d.step; }

}  // namespace dropout
