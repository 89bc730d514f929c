// poly(A) end detection on float32 (calibrated, pA) signal: riser/preprocess.py:42-79 as numpy evaluates it for
// float32 input, where every window statistic stays float32:
//   median   the two middle order statistics a, b of the window: float32(float32(a + b) / 2)
//   MAD      the same rule on float32(|x - median|)
//   mean     np.add.reduce's pairwise sum in float32, divided by the count in float32
//   rolling  np.mean(signal[i - 1000 : i]): its own 1000-element pairwise tree (not the two window sums)
//   change   (mean - rolling) / rolling * 100 in float32, compared with > 20; MAD compared with <= 20 / > 20
// Order statistics are exact on the order-preserving uint32 image of the floats (warp-wide bit descent).  Every
// add / multiply / divide is an explicit round-to-nearest intrinsic so that nvcc cannot contract to FMA.
// One CTA per read, one warp per 500-sample window, the warp's next window fetched while the current one is worked
// on; the two-state scan over the windows is that of polya_kernel (preprocess.cu).
#include "normalise.cuh"

#include <algorithm>
#include <utility>

namespace riser {
namespace {

constexpr int kRes = 500;                   // _TRIM_RESOLUTION, riser/preprocess.py:10
constexpr int kPerLane = (kRes + 31) / 32;  // 16 samples per lane
constexpr int kQuads = kRes / 4;            // 125 float4 per window
constexpr int kMaxWindows = 512;            // as polya_kernel
constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kPwBlock = 128;               // numpy's PW_BLOCKSIZE

// ---------------------------------------------------------------- numpy's pairwise float32 sum, unrolled at compile
// time: a range of n > 128 elements splits at n2 = n/2 - (n/2) % 8; a leaf of <= 128 (>= 8) elements sums into 8
// interleaved accumulators r[j] += a[i + j], combines them as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and adds the
// n % 8 trailing elements one by one.
constexpr int pw_split(int n) { return n / 2 - (n / 2) % 8; }
constexpr int pw_leaves(int n) { return n <= kPwBlock ? 1 : pw_leaves(pw_split(n)) + pw_leaves(n - pw_split(n)); }
constexpr int pw_min_leaf(int n) {
  return n <= kPwBlock ? n : std::min(pw_min_leaf(pw_split(n)), pw_min_leaf(n - pw_split(n)));
}
// start and length of the k-th leaf of a tree over [s, s + n)
constexpr int pw_leaf_start(int n, int k, int s = 0) {
  return n <= kPwBlock ? s
                       : (k < pw_leaves(pw_split(n)) ? pw_leaf_start(pw_split(n), k, s)
                                                     : pw_leaf_start(n - pw_split(n), k - pw_leaves(pw_split(n)),
                                                                     s + pw_split(n)));
}
constexpr int pw_leaf_len(int n, int k) {
  return n <= kPwBlock ? n
                       : (k < pw_leaves(pw_split(n)) ? pw_leaf_len(pw_split(n), k)
                                                     : pw_leaf_len(n - pw_split(n), k - pw_leaves(pw_split(n))));
}
static_assert(pw_leaves(500) == 5 && pw_leaf_start(500, 3) == 368 && pw_leaf_len(500, 4) == 68, "numpy tree, n=500");
static_assert(pw_leaves(1000) == 8 && pw_leaf_start(1000, 4) == 496 && pw_leaf_len(1000, 7) == 128,
              "numpy tree, n=1000");

// combine the leaf sums in the tree's order
template <int N, int K0 = 0>
__device__ __forceinline__ float pw_combine(const float (&leaf)[64]) {
  if constexpr (N <= kPwBlock) {
    return leaf[K0];
  } else {
    constexpr int n2 = pw_split(N);
    return __fadd_rn(pw_combine<n2, K0>(leaf), pw_combine<N - n2, K0 + pw_leaves(n2)>(leaf));
  }
}

// leaf K of the tree over x[0:N], built by lane group K % 4 (lane j of the group holds accumulator j); every lane
// of the warp receives the leaf's sum
template <int N, int K>
__device__ __forceinline__ float pw_leaf(const float* __restrict__ x, int lane) {
  constexpr int s = pw_leaf_start(N, K), len = pw_leaf_len(N, K), body = len - len % 8;
  const bool mine = (lane >> 3) == K % 4;
  const int j = lane & 7;
  float r = 0.f;
  if (mine) {
    r = __ldg(x + s + j);
#pragma unroll
    for (int i = 8; i < body; i += 8) r = __fadd_rn(r, __ldg(x + s + i + j));
  }
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));      // ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7))
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 2));
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 4));
  if (mine) {
#pragma unroll
    for (int i = body; i < len; ++i) r = __fadd_rn(r, __ldg(x + s + i));
  }
  return __shfl_sync(0xffffffffu, r, (K % 4) * 8);
}

template <int N, int... K>
__device__ __forceinline__ float np_sum_f32_impl(const float* __restrict__ x, int lane,
                                                 std::integer_sequence<int, K...>) {
  const float leaf[64] = {pw_leaf<N, K>(x, lane)...};
  return __fadd_rn(pw_combine<N>(leaf), 0.f);
}

// np.add.reduce(x[0:N]) of float32 x, computed by the whole warp (every lane returns it).  The reduction starts
// from the identity 0 as numpy's does (which only shows for an all -0.0 range: the sum is +0.0).
template <int N>
__device__ __forceinline__ float np_sum_f32(const float* __restrict__ x, int lane) {
  static_assert(pw_min_leaf(N) >= 8, "leaves below 8 elements take numpy's short loop, not handled");
  static_assert(pw_leaves(N) <= 64, "leaf list");
  return np_sum_f32_impl<N>(x, lane, std::make_integer_sequence<int, pw_leaves(N)>{});
}

__device__ __forceinline__ int bits_of(uint32_t v) { return 32 - __clz(v); }

// numpy's median of the warp's 500 keys (padding lanes hold 0xffffffff): the two middle keys (ranks 249, 250) found
// by bit descent on key - kmin, one warp-wide count per bit
__device__ __forceinline__ void warp_mid_keys(const uint32_t (&key)[kPerLane], uint32_t& k1, uint32_t& k2) {
  uint32_t kmin = 0xffffffffu, kmax = 0u;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    kmin = min(kmin, key[j]);
    if (key[j] != 0xffffffffu) kmax = max(kmax, key[j]);
  }
  kmin = __reduce_min_sync(0xffffffffu, kmin);
  kmax = __reduce_max_sync(0xffffffffu, kmax);
  const int nbits = bits_of(kmax - kmin);
  constexpr uint32_t k = kRes / 2 - 1;
  uint32_t prefix = 0;
  for (int bit = nbits - 1; bit >= 0; --bit) {
    const uint32_t t = prefix | (1u << bit);
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) cnt += (key[j] != 0xffffffffu && key[j] - kmin < t) ? 1 : 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (k >= static_cast<uint32_t>(cnt)) prefix = t;
  }
  const uint32_t v1 = prefix + kmin;
  int le = 0;
  uint32_t next = 0xffffffffu;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    le += key[j] <= v1 ? 1 : 0;                  // (padding keys are 0xffffffff: never <= a real v1 below it)
    if (key[j] > v1) next = min(next, key[j]);
  }
  le = __reduce_add_sync(0xffffffffu, le);
  next = __reduce_min_sync(0xffffffffu, next);
  k1 = v1;
  k2 = (le > kRes / 2) ? v1 : next;
}

__global__ void __launch_bounds__(kThreads)
polya_f32_kernel(const float* __restrict__ sig, const int64_t* __restrict__ off, const int32_t* __restrict__ nsamp,
                 int B, int32_t* __restrict__ polya_end, int32_t* __restrict__ polya_start, float* __restrict__ stats,
                 int max_windows) {
  __shared__ uint8_t w_flag[kMaxWindows];       // bit 0: the window may start poly(A); bit 1: its MAD > 20
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int n = nsamp[b];
    const float* g = sig + off[b];
    const int nw = min(n / kRes, kMaxWindows);
    // 16-byte loads when the read is 16-byte aligned (a window is 2,000 bytes); which lane holds which sample is
    // irrelevant to the order statistics
    const bool al16 = (reinterpret_cast<uintptr_t>(g) & 15) == 0;
    float4 raw[kPerLane / 4];
    auto fetch = [&](int w) {
      const float4* wp4 = reinterpret_cast<const float4*>(g + w * kRes);
#pragma unroll
      for (int j = 0; j < kPerLane / 4; ++j) {
        const int idx = j * 32 + lane;
        raw[j] = (idx < kQuads) ? __ldg(wp4 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    if (al16 && warp < nw) fetch(warp);
    for (int w = warp; w < nw; w += kWarps) {
      const float* wp = g + w * kRes;
      float v[kPerLane];
      bool ok[kPerLane];
      if (al16) {
#pragma unroll
        for (int j = 0; j < kPerLane / 4; ++j) {
          v[4 * j] = raw[j].x;
          v[4 * j + 1] = raw[j].y;
          v[4 * j + 2] = raw[j].z;
          v[4 * j + 3] = raw[j].w;
          ok[4 * j] = ok[4 * j + 1] = ok[4 * j + 2] = ok[4 * j + 3] = (j * 32 + lane) < kQuads;
        }
        if (w + kWarps < nw) fetch(w + kWarps);
      } else {
#pragma unroll
        for (int j = 0; j < kPerLane; ++j) {
          const int idx = j * 32 + lane;
          ok[j] = idx < kRes;
          v[j] = ok[j] ? __ldg(wp + idx) : 0.f;
        }
      }
      uint32_t key[kPerLane], k1, k2;
#pragma unroll
      for (int j = 0; j < kPerLane; ++j) key[j] = ok[j] ? f2key(v[j]) : 0xffffffffu;
      warp_mid_keys(key, k1, k2);
      const float med = np_median_f32(key2f(k1), key2f(k2), kRes % 2);
      // |x - median| >= 0: the float's bit pattern is already order-preserving
#pragma unroll
      for (int j = 0; j < kPerLane; ++j) key[j] = ok[j] ? __float_as_uint(fabsf(__fsub_rn(v[j], med))) : 0xffffffffu;
      warp_mid_keys(key, k1, k2);
      const float mad = np_median_f32(__uint_as_float(k1), __uint_as_float(k2), kRes % 2);
      const float mean = __fdiv_rn(np_sum_f32<kRes>(wp, lane), static_cast<float>(kRes));
      float rolling = mean;
      if (w > 2) rolling = __fdiv_rn(np_sum_f32<2 * kRes>(wp - 2 * kRes, lane), static_cast<float>(2 * kRes));
      if (lane == 0) {
        const float change = __fmul_rn(__fdiv_rn(__fsub_rn(mean, rolling), rolling), 100.f);
        const bool cs = w > 0 && change > 20.f && mad <= 20.f;
        const bool ce = mad > 20.f;
        w_flag[w] = static_cast<uint8_t>((cs ? 1 : 0) | (ce ? 2 : 0));
        if (stats && w < max_windows) {
          float* st = stats + (static_cast<int64_t>(b) * max_windows + w) * 4;
          st[0] = med;
          st[1] = mad;
          st[2] = mean;
          st[3] = rolling;
        }
      }
    }
    __syncthreads();
    if (warp == 0) {
      // riser/preprocess.py:45-72, the ballot scan of polya_kernel: start = first window > 0 with change > 20 and
      // MAD <= 20; end = first window after it with MAD > 20; 0 doubles as "unset" like Python truthiness
      int pstart = 0, pend = 0;
      for (int w0 = 0; w0 < nw && pend == 0; w0 += 32) {
        const int w = w0 + lane;
        const int f = (w < nw) ? w_flag[w] : 0;
        const uint32_t ms = __ballot_sync(0xffffffffu, f & 1);
        uint32_t me = __ballot_sync(0xffffffffu, f & 2);
        if (pstart == 0 && ms) pstart = (w0 + __ffs(ms) - 1) * kRes;
        if (pstart != 0) {
          const int ws = pstart / kRes - w0;            // start window relative to this chunk (< 0: earlier chunk)
          if (ws > 0) me &= ~((1u << ws) - 1u);
          if (me) pend = (w0 + __ffs(me) - 1) * kRes;
        }
      }
      if (lane == 0) {
        polya_end[b] = pend ? pend : -1;
        if (polya_start) polya_start[b] = pstart ? pstart : -1;
      }
    }
    __syncthreads();
  }
}

}  // namespace
}  // namespace riser

using namespace riser;

extern "C" int riser_polya_end_f32(const float* sig, const int64_t* off, const int32_t* n, int B, int32_t* polya_end,
                                   int32_t* polya_start, float* stats, int max_windows, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_polya_end_f32: B < 0");
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(sig && off && n && polya_end, "riser_polya_end_f32: null pointer");
  RISER_REQUIRE(!stats || max_windows > 0, "riser_polya_end_f32: stats given but max_windows <= 0");
  int per_sm = 0, dev = 0, sms = 148;
  RISER_CUDA_TRY(cudaGetDevice(&dev));
  RISER_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  RISER_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, polya_f32_kernel, kThreads, 0));
  const int grid = std::min(B, sms * std::max(per_sm, 1));
  polya_f32_kernel<<<grid, kThreads, 0, as_stream(stream)>>>(sig, off, n, B, polya_end, polya_start, stats,
                                                             max_windows);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
