// The arithmetic of median / MAD normalisation (riser/preprocess.py:108-147, riser/retrain/preprocess.py:8-44), kept
// once for every kernel that has to reproduce it bit for bit: the int16 and float32 normalisers of preprocess.cu,
// normalise_f32.cu and normalise_long.cu, and the float32 window statistics of polya_f32.cu.
#pragma once

#include "common.cuh"

namespace riser {

constexpr double kOutlierLimit = 3.5;       // riser/preprocess.py:6
constexpr double kScalingFactor = 1.4826;   // riser/preprocess.py:7

// riser/preprocess.py:141-147 (retrain/preprocess.py:18-33 with the caller's limit)
template <class V>
__device__ __forceinline__ V clip_outlier(V v, V lim) {
  return v > lim ? lim : (v < -lim ? -lim : v);
}

// Order-preserving uint32 image of a float32 and its inverse: radix selection over the keys orders the floats.
__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}

// Block-wide exclusive prefix sum of v; warp_sums holds one word per warp of the block.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_sums) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += n;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  uint32_t base = 0;
  for (uint32_t w = 0; w < warp; ++w) base += warp_sums[w];
  __syncthreads();
  return base + inc - v;
}

// np.median's last step on float32 data: the mean of the middle value (odd count) or of the two middle values a, b
// (even count) as np.mean forms it, a float32 sum that starts from the identity +0, divided by the count --
// float32((a + b + 0) / 2), or a + 0.  The +0 shows only for -0.0: the median of [-1, -0., -0., 1] is +0.0.
__device__ __forceinline__ float np_median_f32(float a, float b, bool odd) {
  return odd ? __fadd_rn(a, 0.f) : __fmul_rn(__fadd_rn(__fadd_rn(a, b), 0.f), 0.5f);
}

// (x - median) / (1.4826 MAD) of int16 samples in float64, as k / D with k = 2x - 2 median (an exact small integer)
// and D = 2 denom (exact): with y = RN(1/D), q0 = RN(k y), e = k - q0 D (exact in one FMA), RN(q0 + e y) is the
// correctly rounded quotient (Markstein's final division step), i.e. bit-identical to the reference's float64 divide
// at 3 FP64 ops instead of a full DDIV.
struct Quot16 {
  double D, y;
  __device__ __forceinline__ explicit Quot16(double denom) {
    D = __dmul_rn(2.0, denom);
    y = __ddiv_rn(1.0, D);
  }
  __device__ __forceinline__ double operator()(int k) const {
    // (double) k without an I2F: 2^52 + 2^31 + k has k ^ 0x80000000 in its low word; one exact DADD removes the offset
    const double kd = __dadd_rn(__hiloint2double(0x43300000, k ^ static_cast<int>(0x80000000u)), -4503601774854144.0);
    const double q0 = __dmul_rn(kd, y);
    return __fma_rn(__fma_rn(-q0, D, kd), y, q0);
  }
};

// (a + b) / 2 in the reference's operation order, not contracted to an FMA
__device__ __forceinline__ double half_sum(double a, double b) { return __dmul_rn(__dadd_rn(a, b), 0.5); }
__device__ __forceinline__ float half_sum(float a, float b) { return __fmul_rn(__fadd_rn(a, b), 0.5f); }

// Normalise samples first, first + stride, ... < end of an n-sample window: o[i] = norm(i), the sample's quotient in
// the arithmetic type V (double with the limit 3.5 for int16 samples, float with the caller's limit for float32).
// A run of consecutive outliers (|quotient| > lim, a set fixed by the raw quotients) is rewritten by the thread that
// owns its first element, sequentially as the reference loops (riser/preprocess.py:130-138): arr[j-1] is already
// updated, arr[j+1] is still raw, and the end points of the window copy their single neighbour unclipped.  A run
// may continue past `end`.
template <class V, class Norm>
__device__ __forceinline__ void normalise_span(Norm norm, V lim, int64_t first, int64_t end, int64_t n, int stride,
                                               float* __restrict__ o) {
  for (int64_t i = first; i < end; i += stride) {
    const V v = norm(i);
    if (!(fabs(v) > lim)) {
      o[i] = static_cast<float>(v);
      continue;
    }
    if (i > 0 && fabs(norm(i - 1)) > lim) continue;         // the run's first element walks it
    V prev = (i > 0) ? norm(i - 1) : V(0);
    int64_t j = i;
    V right = (j + 1 < n) ? norm(j + 1) : v;
    for (;;) {
      V nv;
      if (j == 0) nv = right;
      else if (j == n - 1) nv = prev;
      else nv = clip_outlier(half_sum(prev, right), lim);
      o[j] = static_cast<float>(nv);
      prev = nv;
      if (j + 1 >= n || !(fabs(right) > lim)) break;
      ++j;
      right = (j + 1 < n) ? norm(j + 1) : V(0);
    }
  }
}

}  // namespace riser
