// Normalisation of windows of any length (up to INT32_MAX samples) for sm_100a:
//   riser_normalise_long      -- int16 windows, the arithmetic of riser_normalise (riser/preprocess.py:108-147)
//   riser_normalise_f32_long  -- float32 windows, the arithmetic of riser_normalise_f32 / riser_normalise_f32_live
//                                (riser/retrain/preprocess.py:8-44; riser/preprocess.py:108-147 on float32 input)
// The kernels of preprocess.cu and normalise_f32.cu stage a whole window in one CTA's shared memory, which bounds the
// window (98,304 int16 / 49,152 float32 samples).  Here the window stays in global memory and is worked on by many
// CTAs at once, a work item being one kChunk-sample chunk of one read:
//   median, MAD  exact multi-pass radix select over order-preserving integer keys.  Each pass: the CTAs histogram
//                their chunks' keys that match the prefix found so far into a per-read 2048-bin histogram in the
//                caller's workspace; one CTA per read then locates the bin of rank (n - 1) / 2 and narrows the prefix.
//                The last pass also keeps the smallest key ABOVE the prefix, so the second middle value of an even
//                count (the smallest key above the first) needs no extra pass.
//                int16: median keys x + 32768 (16 bits: 11 + 5), MAD keys |2x - 2 median| (17 bits: 11 + 6) ->
//                {2 median, 4 MAD} exactly as riser_normalise reports them.  float32: the order-preserving image of
//                the float (11 + 11 + 10 bits) for the median, the bits of |x - median| for the MAD.
//   normalise    every sample's quotient, in the operation order of the shared-memory kernels; an outlier run
//                (the set |v| > limit is fixed up front) is walked sequentially by the thread that owns its first
//                element -- runs cross chunk boundaries freely since everything is in global memory.
// No host synchronisation, no allocation, and for a given (B, max_len) a fixed launch sequence (CUDA-graph capturable).
#include "common.cuh"

#include <algorithm>

namespace riser {
namespace {

constexpr int kLThreads = 256;
constexpr int kLWarps = kLThreads / 32;
constexpr int kLBins = 2048;
constexpr int kLBinsPerThread = kLBins / kLThreads;
constexpr int kChunk = 16384;               // samples per work item
constexpr int kBlocksPerSm = 8;             // persistent grid: 8 x 256 threads fill an SM

constexpr double kOutlierLimit = 3.5;       // riser/preprocess.py:6
constexpr double kScalingFactor = 1.4826;   // riser/preprocess.py:7

// Per-read selection state in the workspace, after the B histograms.
struct LongState {
  uint32_t prefix, mask;    // key bits fixed so far
  uint32_t k, below;        // rank still sought inside the prefix; keys below the prefix
  uint32_t min_above;       // last pass: smallest key whose fixed bits exceed the prefix
  int32_t med2, mad4;       // int16 results
  float med, mad;           // float32 results
  uint32_t pad[7];
};
static_assert(sizeof(LongState) == 64, "64-byte state per read");

struct PassSpec {
  int shift, bits;
};

__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}

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

__device__ __forceinline__ int window_len(const int32_t* len, int b, int max_len) { return min(len[b], max_len); }

// Key of a sample for the median (stage 0) or the MAD (stage 1) select.
template <int STAGE>
__device__ __forceinline__ uint32_t sel_key(int16_t x, const LongState& s) {
  if (STAGE == 0) return static_cast<uint32_t>(static_cast<int>(x) + 32768);
  return static_cast<uint32_t>(abs(2 * static_cast<int>(x) - s.med2));
}
template <int STAGE>
__device__ __forceinline__ uint32_t sel_key(float x, const LongState& s) {
  if (STAGE == 0) return f2key(x);
  return __float_as_uint(fabsf(__fsub_rn(x, s.med)));
}

__global__ void __launch_bounds__(kLThreads)
long_init_kernel(const int32_t* __restrict__ len, int B, int max_len, uint32_t* __restrict__ hist,
                 LongState* __restrict__ st) {
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    uint4* h = reinterpret_cast<uint4*>(hist + static_cast<size_t>(b) * kLBins);
    for (int i = threadIdx.x; i < kLBins / 4; i += kLThreads) h[i] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) {
      const int n = window_len(len, b, max_len);
      LongState s = {};
      s.k = n > 0 ? static_cast<uint32_t>((n - 1) >> 1) : 0u;
      s.min_above = 0xffffffffu;
      st[b] = s;
    }
  }
}

// One radix pass: every chunk's keys whose fixed bits equal the read's prefix are counted in bin (key >> shift) of
// the read's global histogram; in the last pass the keys above the prefix give the read's min_above.
template <class T, int STAGE>
__global__ void __launch_bounds__(kLThreads)
long_hist_kernel(const T* __restrict__ sig, const int64_t* __restrict__ off, const int32_t* __restrict__ start,
                 const int32_t* __restrict__ len, int B, int max_len, int n_chunks, uint32_t* __restrict__ hist,
                 LongState* __restrict__ st, PassSpec pass, int last) {
  __shared__ __align__(16) uint32_t h[kLBins];
  __shared__ uint32_t cta_min;
  const int tid = threadIdx.x;
  const int64_t items = static_cast<int64_t>(B) * n_chunks;
  const uint32_t bmask = (1u << pass.bits) - 1u;
  for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
    const int b = static_cast<int>(it / n_chunks);
    const int64_t i0 = (it - static_cast<int64_t>(b) * n_chunks) * kChunk;
    const int n = window_len(len, b, max_len);
    if (i0 >= n) continue;                     // block-uniform
    const int64_t i1 = std::min(static_cast<int64_t>(n), i0 + kChunk);
    const T* g = sig + off[b] + (start ? start[b] : 0);
    const LongState s = st[b];
    for (int i = tid; i < kLBins / 4; i += kLThreads) reinterpret_cast<uint4*>(h)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) cta_min = 0xffffffffu;
    __syncthreads();
    uint32_t my_min = 0xffffffffu;
    for (int64_t i = i0 + tid; i < i1; i += kLThreads) {
      const uint32_t kx = sel_key<STAGE>(g[i], s);
      const uint32_t fixed = kx & s.mask;
      if (fixed == s.prefix) atomicAdd(&h[(kx >> pass.shift) & bmask], 1u);
      else if (last && fixed > s.prefix) my_min = min(my_min, kx);
    }
    if (last) {
      my_min = __reduce_min_sync(0xffffffffu, my_min);
      if ((tid & 31) == 0 && my_min != 0xffffffffu) atomicMin(&cta_min, my_min);
    }
    __syncthreads();
    uint32_t* gh = hist + static_cast<size_t>(b) * kLBins;
    for (int i = tid; i <= static_cast<int>(bmask); i += kLThreads) {
      const uint32_t v = h[i];
      if (v) atomicAdd(&gh[i], v);
    }
    if (last && tid == 0 && cta_min != 0xffffffffu) atomicMin(&st[b].min_above, cta_min);
    __syncthreads();                           // h and cta_min are reused by the CTA's next item
  }
}

// One CTA per read: locate the bin of rank s.k in the read's histogram (clearing it for the next pass) and narrow the
// prefix.  After the last pass of a select: the two middle order statistics -> the median (stage 0, and the state is
// reset for the MAD select) or the MAD (stage 1), combined as the shared-memory kernels combine them.
template <bool F32>
__global__ void __launch_bounds__(kLThreads)
long_narrow_kernel(const int32_t* __restrict__ len, int B, int max_len, uint32_t* __restrict__ hist,
                   LongState* __restrict__ st, PassSpec pass, int last, int stage) {
  __shared__ uint32_t warp_sums[kLWarps];
  __shared__ uint32_t res[3];
  __shared__ uint32_t red[kLWarps];
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int n = window_len(len, b, max_len);
    if (n <= 0) continue;                      // block-uniform
    const LongState s = st[b];
    uint4* gh = reinterpret_cast<uint4*>(hist + static_cast<size_t>(b) * kLBins) + 2 * tid;
    const uint4 lo = gh[0], hi = gh[1];
    gh[0] = gh[1] = make_uint4(0u, 0u, 0u, 0u);
    const uint32_t c[kLBinsPerThread] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    uint32_t local = 0;
#pragma unroll
    for (int j = 0; j < kLBinsPerThread; ++j) local += c[j];
    const uint32_t ex = block_exclusive_scan(local, warp_sums);
    if (s.k >= ex && s.k < ex + local) {
      uint32_t run = ex;
#pragma unroll
      for (int j = 0; j < kLBinsPerThread; ++j) {
        if (s.k >= run && s.k < run + c[j]) {
          res[0] = tid * kLBinsPerThread + j;
          res[1] = run;
          res[2] = c[j];
        }
        run += c[j];
      }
    }
    __syncthreads();
    const uint32_t bin = res[0], before = res[1], inbin = res[2];
    const uint32_t prefix = s.prefix | (bin << pass.shift);
    if (!last) {
      if (tid == 0) {
        st[b].prefix = prefix;
        st[b].mask = s.mask | (((1u << pass.bits) - 1u) << pass.shift);
        st[b].k = s.k - before;
        st[b].below = s.below + before;
      }
      __syncthreads();
      continue;
    }
    const uint32_t k1 = static_cast<uint32_t>((n - 1) >> 1), k2 = static_cast<uint32_t>(n >> 1);
    const uint32_t v1 = prefix;
    uint32_t v2 = v1;
    if (k2 != k1 && s.below + before + inbin <= k2) {      // rank k2 is the smallest key above v1
      uint32_t nb = 0xffffffffu;
#pragma unroll
      for (int j = kLBinsPerThread - 1; j >= 0; --j) {
        const uint32_t bj = tid * kLBinsPerThread + j;
        if (bj > bin && c[j]) nb = bj;
      }
      nb = __reduce_min_sync(0xffffffffu, nb);
      if ((tid & 31) == 0) red[tid >> 5] = nb;
      __syncthreads();
#pragma unroll
      for (int w = 0; w < kLWarps; ++w) nb = min(nb, red[w]);
      v2 = (nb != 0xffffffffu) ? (s.prefix | (nb << pass.shift)) : s.min_above;
    }
    if (tid == 0) {
      LongState& o = st[b];
      if (stage == 0) {
        if (F32) o.med = (k1 == k2) ? key2f(v1) : __fmul_rn(__fadd_rn(key2f(v1), key2f(v2)), 0.5f);   // numpy: float32 mean of the pair
        else o.med2 = static_cast<int>(v1) + static_cast<int>(v2) - 65536;
        o.prefix = o.mask = o.below = 0;
        o.k = k1;
        o.min_above = 0xffffffffu;
      } else {
        if (F32) o.mad = (k1 == k2) ? __uint_as_float(v1)
                                    : __fmul_rn(__fadd_rn(__uint_as_float(v1), __uint_as_float(v2)), 0.5f);
        else o.mad4 = static_cast<int32_t>(v1 + v2);
      }
    }
    __syncthreads();
  }
}

// (x - median) / (1.4826 MAD) in float64 as k / D with k = 2x - 2 median (an exact small integer) and D = 2 * denom
// (exact): y = RN(1/D), q0 = RN(k y), e = k - q0 D (exact in one FMA), RN(q0 + e y) is the correctly rounded quotient
// (Markstein's final division step) -- the reference's float64 divide, as normalise_kernel computes it.
struct Quot16 {
  double D, y;
  int med2;
  __device__ __forceinline__ double operator()(int x) const {
    const double k = static_cast<double>(2 * x - med2);
    const double q0 = __dmul_rn(k, y);
    return __fma_rn(__fma_rn(-q0, D, k), y, q0);
  }
};

__device__ __forceinline__ double clip_outlier(double v) {   // riser/preprocess.py:141-147
  if (v > kOutlierLimit) return kOutlierLimit;
  if (v < -kOutlierLimit) return -kOutlierLimit;
  return v;
}

__global__ void __launch_bounds__(kLThreads)
long_norm_i16_kernel(const int16_t* __restrict__ sig, const int64_t* __restrict__ off,
                     const int32_t* __restrict__ start, const int32_t* __restrict__ len, int B, int max_len,
                     int n_chunks, const LongState* __restrict__ st, float* __restrict__ out, int64_t ld_out,
                     int32_t* __restrict__ med2_mad4) {
  const int tid = threadIdx.x;
  const int64_t items = static_cast<int64_t>(B) * n_chunks;
  for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
    const int b = static_cast<int>(it / n_chunks);
    const int64_t i0 = (it - static_cast<int64_t>(b) * n_chunks) * kChunk;
    const int64_t n = window_len(len, b, max_len);
    if (i0 >= n) continue;
    const int64_t i1 = std::min(n, i0 + kChunk);
    const int16_t* g = sig + off[b] + (start ? start[b] : 0);
    float* o = out + static_cast<int64_t>(b) * ld_out;
    const int med2 = st[b].med2, mad4 = st[b].mad4;
    if (med2_mad4 && i0 == 0 && tid == 0) {
      med2_mad4[2 * b] = med2;
      med2_mad4[2 * b + 1] = mad4;
    }
    if (mad4 == 0) {                          // riser/preprocess.py:123-124
      for (int64_t i = i0 + tid; i < i1; i += kLThreads) o[i] = 0.f;
      continue;
    }
    const double denom = __dmul_rn(kScalingFactor, static_cast<double>(mad4) * 0.25);
    const double D = __dmul_rn(2.0, denom);
    const Quot16 q{D, __ddiv_rn(1.0, D), med2};
    for (int64_t i = i0 + tid; i < i1; i += kLThreads) {
      const double v = q(g[i]);
      if (!(fabs(v) > kOutlierLimit)) {
        o[i] = static_cast<float>(v);
        continue;
      }
      if (i > 0 && fabs(q(g[i - 1])) > kOutlierLimit) continue;     // the run's first element walks it
      // riser/preprocess.py:130-138: arr[j-1] is already updated, arr[j+1] still raw; the end points of the array
      // copy their single neighbour and are not clipped
      double prev = (i > 0) ? q(g[i - 1]) : 0.0;
      int64_t j = i;
      double right = (j + 1 < n) ? q(g[j + 1]) : v;
      for (;;) {
        double nv;
        if (j == 0) nv = right;
        else if (j == n - 1) nv = prev;
        else nv = clip_outlier(__dmul_rn(__dadd_rn(prev, right), 0.5));
        o[j] = static_cast<float>(nv);
        prev = nv;
        if (j + 1 >= n || !(fabs(right) > kOutlierLimit)) break;
        ++j;
        right = (j + 1 < n) ? q(g[j + 1]) : 0.0;
      }
    }
  }
}

__global__ void __launch_bounds__(kLThreads)
long_norm_f32_kernel(const float* __restrict__ sig, const int64_t* __restrict__ off, const int32_t* __restrict__ len,
                     int B, int max_len, int n_chunks, const LongState* __restrict__ st, float lim, int zero_if_mad0,
                     float* __restrict__ out, int64_t ld_out, float* __restrict__ med_mad) {
  const int tid = threadIdx.x;
  const int64_t items = static_cast<int64_t>(B) * n_chunks;
  auto clip = [&](float v) { return v > lim ? lim : (v < -lim ? -lim : v); };
  for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
    const int b = static_cast<int>(it / n_chunks);
    const int64_t i0 = (it - static_cast<int64_t>(b) * n_chunks) * kChunk;
    const int64_t n = window_len(len, b, max_len);
    if (i0 >= n) continue;
    const int64_t i1 = std::min(n, i0 + kChunk);
    const float* g = sig + off[b];
    float* o = out + static_cast<int64_t>(b) * ld_out;
    const float med = st[b].med, mad = st[b].mad;
    if (med_mad && i0 == 0 && tid == 0) {
      med_mad[2 * b] = med;
      med_mad[2 * b + 1] = mad;
    }
    if (zero_if_mad0 && mad == 0.f) {         // the live path's guard (riser/preprocess.py:122-124)
      for (int64_t i = i0 + tid; i < i1; i += kLThreads) o[i] = 0.f;
      continue;
    }
    const float denom = __fmul_rn(1.4826f, mad);        // retrain/preprocess.py:44
    auto norm = [&](int64_t i) { return __fdiv_rn(__fsub_rn(g[i], med), denom); };
    for (int64_t i = i0 + tid; i < i1; i += kLThreads) {
      const float v = norm(i);
      if (!(fabsf(v) > lim)) {
        o[i] = v;
        continue;
      }
      if (i > 0 && fabsf(norm(i - 1)) > lim) continue;  // the run's first element walks it
      float prev = (i > 0) ? norm(i - 1) : 0.f;         // retrain/preprocess.py:18-33, sequential
      int64_t j = i;
      float right = (j + 1 < n) ? norm(j + 1) : v;
      for (;;) {
        float nv;
        if (j == 0) nv = right;
        else if (j == n - 1) nv = prev;
        else nv = clip(__fmul_rn(__fadd_rn(prev, right), 0.5f));
        o[j] = nv;
        prev = nv;
        if (j + 1 >= n || !(fabsf(right) > lim)) break;
        ++j;
        right = (j + 1 < n) ? norm(j + 1) : 0.f;
      }
    }
  }
}

int long_sm_count() {
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int& c = sms[dev & 63];
  if (c == 0 && cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) c = 148;
  return c;
}

size_t long_workspace_bytes(int B) {
  return B > 0 ? static_cast<size_t>(B) * (kLBins * sizeof(uint32_t) + sizeof(LongState)) : 0;
}

// The launch sequence shared by both entry points: init, then per select (median, MAD) and radix pass one histogram
// and one narrow launch; the caller launches the elementwise kernel on the returned state.
template <class T>
int launch_select(const char* who, const T* sig, const int64_t* off, const int32_t* start, const int32_t* len, int B,
                  int max_len, int64_t ld_out, const void* out, void* workspace, size_t workspace_bytes,
                  cudaStream_t stream, int& grid_items, int& n_chunks, LongState*& st) {
  RISER_REQUIRE(sig && off && len && out && workspace, "%s: null pointer", who);
  RISER_REQUIRE(max_len > 0 && ld_out >= max_len, "%s: max_len %d <= 0 or ld_out %lld < max_len", who, max_len,
                static_cast<long long>(ld_out));
  RISER_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "%s: workspace must be 16-byte aligned", who);
  if (workspace_bytes < long_workspace_bytes(B))
    return fail(RISER_ENOMEM, "%s: workspace of %zu bytes, %zu needed", who, workspace_bytes, long_workspace_bytes(B));
  uint32_t* hist = static_cast<uint32_t*>(workspace);
  st = reinterpret_cast<LongState*>(hist + static_cast<size_t>(B) * kLBins);
  n_chunks = (max_len + kChunk - 1) / kChunk;
  const int64_t slots = static_cast<int64_t>(long_sm_count()) * kBlocksPerSm;
  grid_items = static_cast<int>(std::min(static_cast<int64_t>(B) * n_chunks, slots));
  const int grid_reads = static_cast<int>(std::min(static_cast<int64_t>(B), slots));
  constexpr bool kF32 = sizeof(T) == 4;
  static const PassSpec kPasses16[2][2] = {{{5, 11}, {0, 5}}, {{6, 11}, {0, 6}}};
  static const PassSpec kPasses32[2][3] = {{{21, 11}, {10, 11}, {0, 10}}, {{21, 11}, {10, 11}, {0, 10}}};
  const int n_pass = kF32 ? 3 : 2;
  long_init_kernel<<<grid_reads, kLThreads, 0, stream>>>(len, B, max_len, hist, st);
  for (int stage = 0; stage < 2; ++stage) {
    for (int p = 0; p < n_pass; ++p) {
      const PassSpec ps = kF32 ? kPasses32[stage][p] : kPasses16[stage][p];
      const int last = p == n_pass - 1;
      auto hk = stage == 0 ? long_hist_kernel<T, 0> : long_hist_kernel<T, 1>;
      hk<<<grid_items, kLThreads, 0, stream>>>(sig, off, start, len, B, max_len, n_chunks, hist, st, ps, last);
      long_narrow_kernel<kF32><<<grid_reads, kLThreads, 0, stream>>>(len, B, max_len, hist, st, ps, last, stage);
    }
  }
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

}  // namespace
}  // namespace riser

using namespace riser;

extern "C" size_t riser_normalise_long_workspace_bytes(int B, int max_len) {
  (void)max_len;
  return long_workspace_bytes(B);
}

extern "C" int riser_normalise_long(const int16_t* sig, const int64_t* off, const int32_t* start, const int32_t* len,
                                    int B, int max_len, float* out, int64_t ld_out, int32_t* med2_mad4,
                                    void* workspace, size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_normalise_long: B < 0");
  if (B == 0) return RISER_OK;
  int grid = 0, n_chunks = 0;
  LongState* st = nullptr;
  const int rc = launch_select("riser_normalise_long", sig, off, start, len, B, max_len, ld_out, out, workspace,
                               workspace_bytes, as_stream(stream), grid, n_chunks, st);
  if (rc != RISER_OK) return rc;
  long_norm_i16_kernel<<<grid, kLThreads, 0, as_stream(stream)>>>(sig, off, start, len, B, max_len, n_chunks, st, out,
                                                                  ld_out, med2_mad4);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_normalise_f32_long(const float* sig, const int64_t* off, const int32_t* len, int B, int max_len,
                                        float outlier_lim, int zero_if_mad0, float* out, int64_t ld_out,
                                        float* med_mad, void* workspace, size_t workspace_bytes,
                                        riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_normalise_f32_long: B < 0");
  if (B == 0) return RISER_OK;
  int grid = 0, n_chunks = 0;
  LongState* st = nullptr;
  const int rc = launch_select("riser_normalise_f32_long", sig, off, static_cast<const int32_t*>(nullptr), len, B,
                               max_len, ld_out, out, workspace, workspace_bytes, as_stream(stream), grid, n_chunks, st);
  if (rc != RISER_OK) return rc;
  long_norm_f32_kernel<<<grid, kLThreads, 0, as_stream(stream)>>>(sig, off, len, B, max_len, n_chunks, st,
                                                                  outlier_lim, zero_if_mad0 ? 1 : 0, out, ld_out,
                                                                  med_mad);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
