// perceptual.cuh — helpers shared by the perceptual-metric kernels (lpips.cu, dists.cu): the grid of the grid-stride
// element kernels, the storage-precision predicates and the warp sums of the two-pass heads.
#pragma once

#include "common.cuh"

namespace b200dn {
namespace perceptual {

constexpr int LP_THREADS = 256;

inline int lp_grid(int64_t work_items) {
  const int sms = device_sm_count();
  if (sms <= 0) return -1;
  int64_t g = cdiv64(work_items, LP_THREADS);
  const int64_t cap = static_cast<int64_t>(sms) * 16;
  if (g > cap) g = cap;
  return static_cast<int>(g < 1 ? 1 : g);
}

inline bool bf16_prec(int prec) {
  return prec == B200DN_PREC_BF16 || prec == B200DN_PREC_BF16X2 || prec == B200DN_PREC_BF16X3;
}
inline bool two_planes(int prec) { return prec == B200DN_PREC_BF16X2 || prec == B200DN_PREC_BF16X3; }

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace perceptual
}  // namespace b200dn
