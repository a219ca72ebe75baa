// Dropout keep masks on their own: the probability -> (threshold, scale) conversion every dropout entry point uses, and
// ep_dropout_keep_mask_u8, which writes the mask of one layer for tests and for hosts that apply it elsewhere.
#include <math.h>
#include "ep_common.cuh"
#include "dropout.cuh"

namespace dropout {

int host_params(const char* who, float p, uint32_t* thr, float* s) {
  const double t = nearbyint((double)p * 65536.0);
  if (!(p >= 0.f) || !(t < 65536.0)) {
    ep::set_error("%s: dropout probability %g must lie in [0, 1) (and round to fewer than 65536 / 65536)", who, (double)p);
    return EP_ERR_INVALID;
  }
  *thr = (uint32_t)t;
  *s = 1.f / (1.f - (float)*thr / 65536.f);
  return EP_OK;
}

}  // namespace dropout

namespace {

// one thread per (row, 8-feature chunk)
__global__ void __launch_bounds__(256)
keep_mask_kernel(long long n, int width, dropout::Params dp, uint8_t* __restrict__ out) {
  const int n_chunks = (width + 7) >> 3;
  const int step = dropout::step_of(dp);
  const long long total = n * n_chunks;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < total;
       it += (long long)gridDim.x * blockDim.x) {
    const long long r = it / n_chunks;
    const int c = (int)(it - r * n_chunks);
    const uint32_t bits = dropout::keep_byte(dp.seed, step, dp.layer, dp.row0 + r, c, dp.thr);
    for (int f = 0; f < 8 && 8 * c + f < width; ++f) out[r * width + 8 * c + f] = (uint8_t)((bits >> f) & 1u);
  }
}

}  // namespace

extern "C" {

int ep_dropout_keep_mask_u8(long long n, int width, float p, unsigned long long seed, int step, const int* step_dev,
                            int layer, long long row0, unsigned char* keep, ep_stream_t stream) {
  EP_REQUIRE(n >= 0 && width > 0, "bad size");
  if (n == 0) return EP_OK;
  EP_REQUIRE(keep, "null pointer");
  dropout::Params dp{};
  if (int rc = dropout::host_params("ep_dropout_keep_mask_u8", p, &dp.thr, &dp.s)) return rc;
  dp.seed = seed; dp.row0 = row0; dp.step_dev = step_dev; dp.step = step; dp.layer = layer;
  const long long total = n * ((width + 7) / 8);
  long long grid = (total + 255) / 256;
  if (grid > (long long)ep::sm_count() * 16) grid = (long long)ep::sm_count() * 16;
  keep_mask_kernel<<<(unsigned)grid, 256, 0, ep::as_stream(stream)>>>(n, width, dp, keep);
  EP_LAUNCH_CHECK("keep_mask_kernel");
  return EP_OK;
}

}  // extern "C"
