// float32 variant of the normalisation kernel for the training-data preparation path
// (riser/retrain/preprocess.py:8-44, SURVEY.md 8f-4): the input is the pA-scaled signal
// (float32, `read.get_raw_data(scale=True)`), and numpy keeps every step in float32 --
// median (mean of the two middle values in float32), MAD, (x - median) / (1.4826f * mad),
// outlier smoothing with a caller-supplied limit, no MAD == 0 guard (IEEE inf / nan as numpy).
// Exact order statistics come from a 3-pass (11 + 11 + 10 bit) block-wide radix select over
// the order-preserving integer image of the floats.  Data-prep path: written for exactness,
// not for the HBM roofline.
#include "normalise.cuh"

#include <algorithm>

namespace riser {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kBins = 2048;
constexpr int kPerThread = kBins / kThreads;
constexpr int kMaxLenF32 = 49152;

struct Scratch {
  uint32_t hist[kBins];
  uint32_t warp_sums[kWarps];
  uint32_t res[3];       // bin, keys before the bin, keys in the bin
  uint32_t red[kWarps];
};

// key of rank k (0-based) among key(0..n-1); *count_le = number of keys <= that key
template <class KeyFn>
__device__ uint32_t radix_select(KeyFn key, int n, uint32_t k, Scratch& s, uint32_t* count_le) {
  const int tid = threadIdx.x;
  uint32_t prefix = 0, mask = 0, below = 0;
  const int shifts[3] = {21, 10, 0};
  const int bits[3] = {11, 11, 10};
  for (int pass = 0; pass < 3; ++pass) {
    const int shift = shifts[pass];
    const uint32_t bmask = (1u << bits[pass]) - 1u;
    for (int i = tid; i < kBins; i += kThreads) s.hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
      const uint32_t kx = key(i);
      if ((kx & mask) == prefix) atomicAdd(&s.hist[(kx >> shift) & bmask], 1u);
    }
    __syncthreads();
    uint32_t c[kPerThread], local = 0;
#pragma unroll
    for (int j = 0; j < kPerThread; ++j) {
      c[j] = s.hist[tid * kPerThread + j];
      local += c[j];
    }
    const uint32_t ex = block_exclusive_scan(local, s.warp_sums);
    if (k >= ex && k < ex + local) {
      uint32_t run = ex;
#pragma unroll
      for (int j = 0; j < kPerThread; ++j) {
        if (k >= run && k < run + c[j]) {
          s.res[0] = tid * kPerThread + j;
          s.res[1] = run;
          s.res[2] = c[j];
        }
        run += c[j];
      }
    }
    __syncthreads();
    const uint32_t bin = s.res[0], before = s.res[1], inbin = s.res[2];
    __syncthreads();
    prefix |= bin << shift;
    mask |= bmask << shift;
    below += before;
    k -= before;
    if (pass == 2) *count_le = below + inbin;
  }
  return prefix;
}

// the two middle order statistics (ranks k1 <= k2)
template <class KeyFn>
__device__ void select_middle(KeyFn key, int n, uint32_t k1, uint32_t k2, Scratch& s, uint32_t& v1, uint32_t& v2) {
  uint32_t le = 0;
  v1 = radix_select(key, n, k1, s, &le);
  v2 = v1;
  if (k2 != k1 && le <= k2) {      // rank k2 is the smallest key above v1
    uint32_t m = 0xffffffffu;
    for (int i = threadIdx.x; i < n; i += kThreads) {
      const uint32_t kx = key(i);
      if (kx > v1) m = min(m, kx);
    }
    m = __reduce_min_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = s.red[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) m = min(m, s.red[w]);
    __syncthreads();
    v2 = m;
  }
}

__global__ void __launch_bounds__(kThreads)
normalise_f32_kernel(const float* __restrict__ sig, const int64_t* __restrict__ off, const int32_t* __restrict__ len,
                     int B, float lim, float* __restrict__ out, int64_t ld_out, int zero_if_mad0,
                     float* __restrict__ med_mad) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Scratch& s = *reinterpret_cast<Scratch*>(smem_raw);
  float* x = reinterpret_cast<float*>(smem_raw + ((sizeof(Scratch) + 15) & ~size_t(15)));
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int n = len[b];
    if (n <= 0) continue;
    const float* g = sig + off[b];
    float* o = out + static_cast<int64_t>(b) * ld_out;
    for (int i = tid; i < n; i += kThreads) x[i] = g[i];
    __syncthreads();
    const uint32_t k1 = static_cast<uint32_t>((n - 1) >> 1), k2 = static_cast<uint32_t>(n >> 1);
    uint32_t a1, a2;
    select_middle([&](int i) { return f2key(x[i]); }, n, k1, k2, s, a1, a2);
    const float med = np_median_f32(key2f(a1), key2f(a2), k1 == k2);
    select_middle([&](int i) { return __float_as_uint(fabsf(__fsub_rn(x[i], med))); }, n, k1, k2, s, a1, a2);
    const float mad = np_median_f32(__uint_as_float(a1), __uint_as_float(a2), k1 == k2);
    if (med_mad && tid == 0) {
      med_mad[2 * b] = med;
      med_mad[2 * b + 1] = mad;
    }
    if (zero_if_mad0 && mad == 0.f) {          // the live path's guard (riser/preprocess.py:122-124)
      for (int i = tid; i < n; i += kThreads) o[i] = 0.f;
      __syncthreads();
      continue;
    }
    const float denom = __fmul_rn(static_cast<float>(kScalingFactor), mad);       // retrain/preprocess.py:44
    normalise_span([&](int64_t i) { return __fdiv_rn(__fsub_rn(x[i], med), denom); }, lim, tid, n, n, kThreads, o);
    __syncthreads();
  }
}

}  // namespace
}  // namespace riser

extern "C" int riser_normalise_f32_max_len(void) { return riser::kMaxLenF32; }

namespace riser {
namespace {
int launch_f32(const char* who, const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
               float outlier_lim, int zero_if_mad0, float* out, int64_t ld_out, float* med_mad, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "%s: B < 0", who);
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(sig && off && len && out, "%s: null pointer", who);
  RISER_REQUIRE(max_len > 0 && max_len <= kMaxLenF32 && ld_out >= max_len,
                "%s: max_len %d outside (0, %d] or ld_out too small", who, max_len, kMaxLenF32);
  const size_t smem = ((sizeof(Scratch) + 15) & ~size_t(15)) + 4 * static_cast<size_t>(max_len);
  RISER_CUDA_TRY(cudaFuncSetAttribute(normalise_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
  int per_sm = 1, dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, normalise_f32_kernel, kThreads, smem);
  const int grid = std::min(B, sms * std::max(1, per_sm));
  normalise_f32_kernel<<<grid, kThreads, smem, as_stream(stream)>>>(sig, off, len, B, outlier_lim, out, ld_out,
                                                                    zero_if_mad0, med_mad);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
}  // namespace
}  // namespace riser

extern "C" int riser_normalise_f32(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                                   float outlier_lim, float* out, int64_t ld_out, riser_stream_t stream) {
  return riser::launch_f32("riser_normalise_f32", sig, off, len, B, max_len, outlier_lim, 0, out, ld_out, nullptr, stream);
}

extern "C" int riser_normalise_f32_live(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                                        float* out, int64_t ld_out, float* med_mad, riser_stream_t stream) {
  return riser::launch_f32("riser_normalise_f32_live", sig, off, len, B, max_len, 3.5f, 1, out, ld_out, med_mad, stream);
}
