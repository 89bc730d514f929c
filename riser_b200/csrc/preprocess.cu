// Preprocessing kernels of the RISER hot path for sm_100a:
//   riser_normalise  -- fused median / MAD / normalise / outlier smoothing over ragged
//                       int16 windows (riser/preprocess.py:108-147)
//   riser_polya_end  -- 500-sample window statistics + the 2-state poly(A) scan
//                       (riser/preprocess.py:42-79)
// Both are HBM-bound byte/integer work: one CTA per read, the window staged once in
// shared memory with 16-byte coalesced loads, exact integer selection (histogram radix
// select for whole windows, warp-shuffle bit-descent select for 500-sample windows),
// float64 arithmetic in the reference's operation order, fp32 results written with
// 16-byte stores.
#include "common.cuh"

#include <algorithm>
#include <stdlib.h>
#include <type_traits>

namespace riser {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kBins = 2048;             // first-pass histogram bins
constexpr int kBinsPerThread = kBins / kThreads;
constexpr int kSubBins = 128;           // refinement pass (shift <= 7)
constexpr int kMaxLen = 98304;          // samples staged in smem (192 KB)
constexpr int kMaxRuns = 512;           // outlier-run start indices collected per read (more: rescan path)

constexpr int kDefaultF64 = 1;          // samples per group of four on the float64 pipe (0 / 1 / 4: 0.1106 / 0.1085 / 0.1085 ms)

constexpr double kOutlierLimit = 3.5;   // riser/preprocess.py:6
constexpr double kScalingFactor = 1.4826;  // riser/preprocess.py:7

struct SelectScratch {
  uint64_t bar;         // bulk-copy completion of the staging buffer
  alignas(16) uint32_t hist[kBins];
  uint32_t sub[kSubBins];
  uint32_t warp_sums[kWarps];
  uint32_t res[4];      // bin1, before1, bin2, before2
  uint32_t refined;
  uint32_t n_runs;
  int32_t red[2 * kWarps];
  int32_t runs[kMaxRuns];
};

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_sums) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t n = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += n;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  uint32_t base = 0;
  for (uint32_t w = 0; w < warp; ++w) base += warp_sums[w];
  __syncthreads();
  return base + inc - v;
}

// A window of n samples staged in shared memory at the 16-byte phase it has in global memory:
// sample i is stage[a + i], 0 <= a < 8.  for_each() hands every sample of the window to f, one
// 16-byte chunk (8 samples) per thread and step; the two edge chunks are masked.
struct StagedWindow {
  const int16_t* stage;
  int a, n;
  __device__ __forceinline__ int operator[](int i) const { return stage[a + i]; }
  template <class F>
  __device__ __forceinline__ void full_chunk(int c, F& f) const {      // all 8 samples of chunk c lie in the window
    const uint4 v = reinterpret_cast<const uint4*>(stage)[c];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      f(static_cast<int>(static_cast<int16_t>(w[j] & 0xffffu)));
      f(static_cast<int>(w[j]) >> 16);
    }
  }
  // Chunk order: warp w owns the contiguous full chunks [w R, (w + 1) R); lane l walks l S .. l S + S - 1 of them with
  // S odd, so the 16-byte loads of a warp stay bank-conflict free while its lanes work on samples ~8 S apart --
  // neighbouring samples of a squiggle sit on the same current level, and 32 lanes hitting the same few histogram
  // bins serialise the shared-memory atomics.  The (< 64) chunks left over per warp are taken lane by lane.  The
  // (< 8) samples before the first and after the last full chunk are taken one per thread by threads 0..15, so the
  // chunk loop carries no edge tests.
  template <class F>
  __device__ __forceinline__ void for_each(F f) const {
    const int end = a + n;
    const int c_first = (a + 7) >> 3, c_last = end >> 3;        // full chunks: [c_first, c_last) (may be empty)
    const int head_end = min(end, 8 * c_first);                 // head samples: positions [a, head_end)
    const int tail_start = max(8 * c_last, head_end);           // tail samples: positions [tail_start, end)
    const int tid = threadIdx.x;
    if (tid < 16) {
      const int pos = (tid < 8) ? a + tid : tail_start + tid - 8;
      if (pos < ((tid < 8) ? head_end : end)) f(static_cast<int>(stage[pos]));
    }
    const int lane = tid & 31, warp = tid >> 5;
    const int n_full = max(c_last - c_first, 0);
    const int R = (n_full + kWarps - 1) / kWarps;
    const int c0 = c_first + warp * R, c1 = min(c0 + R, c_first + n_full);
    int S = (c1 - c0) >> 5;
    S = (S > 0) ? ((S - 1) | 1) : 0;          // largest odd number <= (c1 - c0) / 32
    for (int i = 0; i < S; ++i) full_chunk(c0 + lane * S + i, f);
    for (int c = c0 + 32 * S + lane; c < c1; c += 32) full_chunk(c, f);
  }
};

// Exact order statistics k1 <= k2 (0-based) of the keys key(sample) over the window, all <= maxkey.
// Pass A: histogram of key >> shift with shift chosen so that it fits kBins; block scan
// locates the bins holding the two ranks.  Pass B (only when shift > 0): histogram of the
// low bits inside the located bin.  Block-uniform control flow; all threads get r1, r2.
template <class KeyFn>
__device__ int select_two(KeyFn key, const StagedWindow& win, uint32_t maxkey, uint32_t k1, uint32_t k2,
                          SelectScratch& s, uint32_t& r1, uint32_t& r2, bool keep_prefix = false, int rot = -1) {
  // rot >= 0: the histogram of the keys is already in s.hist, CIRCULAR -- key u sits in bin (u + rot) & (kBins - 1)
  // (the fused min / max + histogram pass of the normalise kernel bins by `sample & (kBins - 1)` before it knows the
  // minimum; maxkey < kBins then) -- and published by a block barrier; the prefix is written back in the same order.
  const int tid = threadIdx.x;
  int shift = 0;
  while ((maxkey >> shift) >= static_cast<uint32_t>(kBins)) ++shift;
  const bool prebuilt = rot >= 0;
  if (!prebuilt) {
    rot = 0;
    for (int i = tid; i < kBins / 4; i += kThreads) reinterpret_cast<uint4*>(s.hist)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    if (shift == 0) {       // (every real squiggle window: no shift instruction per sample)
      win.for_each([&](int e) { atomicAdd(&s.hist[key(e)], 1u); });
    } else {
      win.for_each([&](int e) { atomicAdd(&s.hist[key(e) >> shift], 1u); });
    }
    __syncthreads();
  }
  // Thread t owns the aligned block of 8 bins (t + rot / 8) mod 256, i.e. the keys 8 t - rot % 8 .. + 7: contiguous in key
  // order, read and written back with 16-byte accesses.  (The rot % 8 bins thread 0 holds "before key 0" are the top
  // keys wrapped around: the caller only passes rot when maxkey < kBins - 8, so they are empty.)
  static_assert(kBinsPerThread == 8, "two uint4 per thread");
  const int phys = ((tid + (rot >> 3)) & (kThreads - 1)) * kBinsPerThread;
  const int key0 = tid * kBinsPerThread - (rot & 7);
  uint32_t c[kBinsPerThread];
  uint32_t local = 0;
  {
    const uint4 lo = *reinterpret_cast<const uint4*>(&s.hist[phys]), hi = *reinterpret_cast<const uint4*>(&s.hist[phys + 4]);
    c[0] = lo.x; c[1] = lo.y; c[2] = lo.z; c[3] = lo.w; c[4] = hi.x; c[5] = hi.y; c[6] = hi.z; c[7] = hi.w;
  }
#pragma unroll
  for (int j = 0; j < kBinsPerThread; ++j) local += c[j];
  const uint32_t ex = block_exclusive_scan(local, s.warp_sums);
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const uint32_t k = which ? k2 : k1;
    if (k >= ex && k < ex + local) {
      uint32_t run = ex;
#pragma unroll
      for (int j = 0; j < kBinsPerThread; ++j) {
        if (k >= run && k < run + c[j]) {
          s.res[2 * which] = static_cast<uint32_t>(key0 + j);
          s.res[2 * which + 1] = run;
        }
        run += c[j];
      }
    }
  }
  __syncthreads();
  const uint32_t bin1 = s.res[0], before1 = s.res[1], bin2 = s.res[2], before2 = s.res[3];
  if (shift == 0) {
    r1 = bin1;
    r2 = bin2;
    if (keep_prefix) {   // hist[j] <- number of keys <= j (used to get the MAD without a second pass)
      uint32_t run = ex;
#pragma unroll
      for (int j = 0; j < kBinsPerThread; ++j) {
        run += c[j];
        c[j] = run;
      }
      *reinterpret_cast<uint4*>(&s.hist[phys]) = make_uint4(c[0], c[1], c[2], c[3]);
      *reinterpret_cast<uint4*>(&s.hist[phys + 4]) = make_uint4(c[4], c[5], c[6], c[7]);
    }
    __syncthreads();
    return 0;
  }
  const uint32_t mask = (1u << shift) - 1u;
#pragma unroll 1
  for (int which = 0; which < 2; ++which) {
    const uint32_t bin = which ? bin2 : bin1;
    const uint32_t kk = which ? (k2 - before2) : (k1 - before1);
    __syncthreads();
    for (int i = tid; i < kSubBins; i += kThreads) s.sub[i] = 0;
    __syncthreads();
    win.for_each([&](int e) {
      const uint32_t kx = key(e);
      if ((kx >> shift) == bin) atomicAdd(&s.sub[kx & mask], 1u);
    });
    __syncthreads();
    if (tid == 0) {
      uint32_t run = 0, found = 0;
      for (uint32_t j = 0; j <= mask; ++j) {
        if (kk >= run && kk < run + s.sub[j]) found = j;
        run += s.sub[j];
      }
      s.refined = (bin << shift) | found;
    }
    __syncthreads();
    if (which) r2 = s.refined; else r1 = s.refined;
  }
  __syncthreads();
  return shift;
}

__device__ __forceinline__ double clip_outlier(double v) {
  // riser/preprocess.py:141-147
  if (v > kOutlierLimit) return kOutlierLimit;
  if (v < -kOutlierLimit) return -kOutlierLimit;
  return v;
}

// Kernel structure (one CTA per read, persistent over reads b = blockIdx.x, + gridDim.x, ...):
//   stage    one 1-D bulk copy (cp.async.bulk, mbarrier complete_tx) of the 16-byte blocks that hold the
//            window; the CTA's NEXT read is prefetched into L2 while the current one is processed, so its
//            copy is an L2 hit
//   min/max  packed 16-bit min / max over the staged chunks
//   median   histogram radix select (select_two); MAD from the same histogram by a warp-wide
//            32-ary search on the distance (or a second select when the range needed a shift)
//   normalise + smooth: every sample gets the exact quotient; the starts of outlier runs are collected
//            in shared memory and walked afterwards, one run per thread, so a rare outlier no longer
//            stalls its whole warp in a divergent slow path
__global__ void __launch_bounds__(kThreads, 5)
normalise_kernel(const int16_t* __restrict__ sig, const int64_t* __restrict__ off,
                 const int32_t* __restrict__ start, const int32_t* __restrict__ len, int B,
                 float* __restrict__ out, int64_t ld_out, int32_t* __restrict__ med2_mad4,
                 int max_len) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  SelectScratch& s = *reinterpret_cast<SelectScratch*>(smem_raw);
  int16_t* stage = reinterpret_cast<int16_t*>(smem_raw + ((sizeof(SelectScratch) + 127) & ~size_t(127)));
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    mbar_init(&s.bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  // thread 0: bulk copy of a window of nr samples at gr (whole 16-byte blocks) into the staging buffer
  auto issue = [&](int nr, const int16_t* gr) {
    if (nr <= 0) return;
    const int ar = static_cast<int>((reinterpret_cast<uintptr_t>(gr) >> 1) & 7);
    const uint32_t bytes = static_cast<uint32_t>(((ar + nr + 7) >> 3) << 4);
    mbar_arrive_expect_tx(&s.bar, bytes);
    bulk_load_1d(stage, gr - ar, bytes, &s.bar);
  };
  // the NEXT read's blocks are pulled into L2 while this one is processed, so that its copy at the top of the
  // next iteration is an L2 hit and the HBM reads spread over the compute phases
  auto prefetch = [&](int nr, const int16_t* gr) {
    if (nr <= 0) return;
    const int ar = static_cast<int>((reinterpret_cast<uintptr_t>(gr) >> 1) & 7);
    bulk_prefetch_l2(gr - ar, static_cast<uint32_t>(((ar + nr + 7) >> 3) << 4));
  };
  // window length / position of the read being processed and of the CTA's next one (loaded an iteration ahead,
  // so that no global-load latency sits between the end of a read and the copy of the next)
  auto meta = [&](int r, int& nr, const int16_t*& gr) {
    nr = 0;
    gr = sig;
    if (r < B) {
      nr = min(len[r], max_len);      // memory safety: a window longer than the caller's max_len is cut to it
      gr = sig + off[r] + (start ? start[r] : 0);
    }
  };
  int n_cur, n_nxt;
  const int16_t *g_cur, *g_nxt;
  meta(blockIdx.x, n_cur, g_cur);
  uint32_t phase = 0;                  // parity the next wait on bar uses

  for (int b = blockIdx.x; b < B; b += gridDim.x, n_cur = n_nxt, g_cur = g_nxt) {
    if (tid == 0) issue(n_cur, g_cur);
    meta(b + gridDim.x, n_nxt, g_nxt);
    if (tid == 0) prefetch(n_nxt, g_nxt);
    const int n = n_cur;
    if (n <= 0) continue;                 // block-uniform; nothing was issued for this read
    const int16_t* g = g_cur;
    float* o = out + static_cast<int64_t>(b) * ld_out;
    const int a = static_cast<int>((reinterpret_cast<uintptr_t>(g) >> 1) & 7);
    const StagedWindow x{stage, a, n};     // x[i] == g[i]
    // (the value histogram of the fused pass below is cleared while the read's copy is in flight)
    for (int i = tid; i < kBins / 4; i += kThreads) reinterpret_cast<uint4*>(s.hist)[i] = make_uint4(0u, 0u, 0u, 0u);
    mbar_wait(&s.bar, phase);
    phase ^= 1u;
    __syncthreads();

    // ---- min / max of the window AND its value histogram in one pass over the staged chunks: a sample is counted in
    //      bin `x & (kBins - 1)` -- circular, so the minimum need not be known yet; if the range turns out to fit the
    //      bins (every real squiggle) the bins of the values vmin .. vmax are distinct and bin u of the usual
    //      histogram is (u + vmin) & (kBins - 1); otherwise the select below rebuilds a shifted histogram.
    //      (The bins were cleared before the copy wait; the barrier above orders that against these atomics.)
    int vmin = 32767, vmax = -32768;
    {
      uint32_t mn2 = 0x7fff7fffu, mx2 = 0x80008000u;
      const uint32_t hist_addr = smem_u32(s.hist);
      auto count4 = [&](uint32_t four_x) {      // four_x = 4 * sample (any upper bits): bin byte offset = four_x & 4 (kBins - 1)
        asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hist_addr + (four_x & (4u * (kBins - 1)))) : "memory");
      };
      auto one = [&](int e) {
        vmin = min(vmin, e);
        vmax = max(vmax, e);
        count4(static_cast<uint32_t>(e) << 2);
      };
      auto full = [&](int c) {
        const uint4 v = reinterpret_cast<const uint4*>(stage)[c];
        mn2 = __vimin3_s16x2(mn2, v.x, v.y);
        mn2 = __vimin3_s16x2(mn2, v.z, v.w);
        mx2 = __vimax3_s16x2(mx2, v.x, v.y);
        mx2 = __vimax3_s16x2(mx2, v.z, v.w);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          count4(w[j] << 2);                    // lower half: bits 2 .. 12 of (w << 2) are 4 * (x & 2047)
          count4(w[j] >> 14);                   // upper half
        }
      };
      // the chunk order of StagedWindow::for_each (lane-decorrelated, edge samples one per thread)
      const int end = a + n;
      const int c_first = (a + 7) >> 3, c_last = end >> 3;
      const int head_end = min(end, 8 * c_first), tail_start = max(8 * c_last, head_end);
      if (tid < 16) {
        const int pos = (tid < 8) ? a + tid : tail_start + tid - 8;
        if (pos < ((tid < 8) ? head_end : end)) one(static_cast<int>(stage[pos]));
      }
      const int n_full = max(c_last - c_first, 0);
      const int R = (n_full + kWarps - 1) / kWarps;
      const int c0 = c_first + warp * R, c1 = min(c0 + R, c_first + n_full);
      int S = (c1 - c0) >> 5;
      S = (S > 0) ? ((S - 1) | 1) : 0;
      for (int i = 0; i < S; ++i) full(c0 + lane * S + i);
      for (int c = c0 + 32 * S + lane; c < c1; c += 32) full(c);
      vmin = min(vmin, min(static_cast<int>(static_cast<int16_t>(mn2 & 0xffffu)), static_cast<int>(static_cast<int16_t>(mn2 >> 16))));
      vmax = max(vmax, max(static_cast<int>(static_cast<int16_t>(mx2 & 0xffffu)), static_cast<int>(static_cast<int16_t>(mx2 >> 16))));
    }
    vmin = __reduce_min_sync(0xffffffffu, vmin);
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    if (lane == 0) {
      s.red[warp] = vmin;
      s.red[kWarps + warp] = vmax;
    }
    __syncthreads();          // (also publishes the histogram)
    vmin = s.red[0];
    vmax = s.red[kWarps];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) {
      vmin = min(vmin, s.red[w]);
      vmax = max(vmax, s.red[kWarps + w]);
    }

    // ---- median: mean of the two middle order statistics -> med2 = 2 * median (exact)
    const uint32_t k1 = static_cast<uint32_t>((n - 1) >> 1), k2 = static_cast<uint32_t>(n >> 1);
    uint32_t r1, r2;
    const int range = vmax - vmin;
    const int rot = (range < kBins - 8) ? (vmin & (kBins - 1)) : -1;      // circular histogram usable as it stands?
    const int rot_eff = max(rot, 0);      // bin of key u in the histogram the select leaves behind (shift 0): (u + rot_eff) & (kBins - 1)
    const int shift_used = select_two([&](int e) { return static_cast<uint32_t>(e - vmin); }, x,
                                      static_cast<uint32_t>(range), k1, k2, s, r1, r2, true, rot);
    const int med2 = 2 * vmin + static_cast<int>(r1 + r2);

    // ---- MAD on keys d = |2x - med2| = 2|x - median| -> mad4 = 4 * MAD (exact)
    const uint32_t dmax = static_cast<uint32_t>(max(abs(2 * vmin - med2), abs(2 * vmax - med2)));
    uint32_t mad4;
    if (shift_used == 0) {
      // The value histogram already holds the whole distribution: with P[u] = #{x - vmin <= u}
      // and m = med2 - 2*vmin, #{|2x - med2| <= d} = P[floor((m+d)/2)] - P[ceil((m-d)/2) - 1];
      // the two middle order statistics of d are found by a 32-ary search on d (warps 0 and 1,
      // one probe per lane and round: 3 rounds for an 11-bit distance).
      if (warp < 2) {
        const int m = static_cast<int>(r1 + r2);
        const uint32_t want = (warp ? k2 : k1) + 1;
        int lo_d = 0, hi_d = static_cast<int>(dmax);      // invariant: count(hi_d) >= want
        while (lo_d < hi_d) {
          const int step = (hi_d - lo_d + 32) >> 5;       // ceil(span / 32)
          const int d = min(lo_d + (lane + 1) * step - 1, hi_d);
          const int hi_u = min((m + d) >> 1, range);
          const int lo_u = (m - d + 1) >> 1;              // ceil((m - d) / 2), may be <= 0
          const uint32_t cnt = s.hist[(hi_u + rot_eff) & (kBins - 1)] - (lo_u > 0 ? s.hist[(lo_u - 1 + rot_eff) & (kBins - 1)] : 0u);
          const uint32_t okm = __ballot_sync(0xffffffffu, cnt >= want);   // lane 31 probes hi_d: never empty
          const int f = __ffs(okm) - 1;
          hi_d = min(lo_d + (f + 1) * step - 1, hi_d);
          lo_d = lo_d + f * step;
        }
        if (lane == 0) s.res[warp] = static_cast<uint32_t>(lo_d);
      }
      __syncthreads();
      mad4 = s.res[0] + s.res[1];
    } else {
      select_two([&](int e) { return static_cast<uint32_t>(abs(2 * e - med2)); }, x, dmax, k1, k2,
                 s, r1, r2);
      mad4 = r1 + r2;
    }
    if (med2_mad4 && tid == 0) {
      med2_mad4[2 * b] = med2;
      med2_mad4[2 * b + 1] = static_cast<int32_t>(mad4);
    }

    const int n_groups = (n + 3) >> 2;
    if (mad4 == 0) {   // riser/preprocess.py:123-124
      for (int gidx = tid; gidx < n_groups; gidx += kThreads) {
        const int i0 = 4 * gidx;
        if (i0 + 4 <= n) {
          *reinterpret_cast<float4*>(o + i0) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
          for (int i = i0; i < n; ++i) o[i] = 0.f;
        }
      }
    } else {
      const double denom = __dmul_rn(kScalingFactor, static_cast<double>(mad4) * 0.25);
      // (x - median) / denom == k / D with k = 2x - 2*median (an exact small integer) and D = 2 * denom
      // (exact).  With y = RN(1/D), q0 = RN(k*y), e = k - q0*D (exact in one FMA), RN(q0 + e*y) is the
      // correctly rounded quotient (Markstein's final division step), i.e. bit-identical to the reference's
      // float64 divide at 3 FP64 ops instead of a full DDIV.
      const double Dd = __dmul_rn(2.0, denom);
      const double yrcp = __ddiv_rn(1.0, Dd);
      auto quot = [&](int ki) {
        // (double) ki without an I2F: 2^52 + 2^31 + ki has ki ^ 0x80000000 in its low word; one exact DADD removes the offset
        const double k = __dadd_rn(__hiloint2double(0x43300000, ki ^ static_cast<int>(0x80000000u)), -4503601774854144.0);
        const double q0 = __dmul_rn(k, yrcp);
        const double e = __fma_rn(-q0, Dd, k);
        return __fma_rn(e, yrcp, q0);
      };
      // A window holds at most range + 1 distinct values (~1,000 for a squiggle against 4,096-16,000 samples),
      // and the float64 pipe is what bounds this kernel: when the value range fits the histogram, the fp32 result
      // of every VALUE is tabulated once (in the histogram's storage, free after the MAD search) and the per-sample
      // work becomes one shared-memory look-up.
      const bool use_lut = (shift_used == 0);
      float* lut = reinterpret_cast<float*>(s.hist);
      if (use_lut)
        for (int u = tid; u <= range; u += kThreads)      // (circular by VALUE: the entry of sample value v sits at v & (kBins - 1))
          lut[(vmin + u) & (kBins - 1)] = static_cast<float>(quot(2 * (vmin + u) - med2));

      // ---- outlier threshold in the integer key domain: |z| > 3.5  <=>  d > dthr, where
      //      z = fl((d/2) / denom) is monotone in d.  Found once per read with exact divides: the lanes of
      //      warp 0 test the 32 candidates around 7 * denom at once (serial search as a fallback).
      if (warp == 0) {
        auto zval = [&](int d) { return __ddiv_rn(static_cast<double>(d) * 0.5, denom); };
        const int base = static_cast<int>(__dmul_rn(7.0, denom));
        const int d = base - 8 + lane;
        const uint32_t okm = __ballot_sync(0xffffffffu, d < 0 || zval(d) <= kOutlierLimit);
        if (lane == 0) {
          const int cnt = __popc(okm);
          int d0;
          if (cnt > 0 && cnt < 32 && okm == ((1u << cnt) - 1u)) {
            d0 = base - 9 + cnt;
          } else {
            d0 = base;
            while (zval(d0 + 1) <= kOutlierLimit) ++d0;
            while (d0 > 0 && zval(d0) > kOutlierLimit) --d0;
          }
          s.refined = static_cast<uint32_t>(max(d0, 0));
          s.n_runs = 0;
        }
      }
      __syncthreads();
      const uint32_t dthr = s.refined;
      auto flagged = [&](int i) { return static_cast<uint32_t>(abs(2 * x[i] - med2)) > dthr; };
      // riser/preprocess.py:130-138 for the run of consecutive outliers that starts at i: arr[j-1] is
      // already updated, arr[j+1] is still raw; the end points of the array are not clipped.
      // The recurrence is sequential, and a float64 op has a long dependent latency: per step only ONE fma
      // (prev / 2 + raw / 2, the same rounding as (prev + raw) / 2) and the clip stay on the chain; the raw
      // neighbour's quotient and the "is the next sample an outlier" test are computed a step ahead.
      auto walk = [&](int i) {
        double prev = (i > 0) ? quot(2 * x[i - 1] - med2) : 0.0;
        double rh_next = 0.5 * quot(2 * x[min(i + 1, n - 1)] - med2);        // raw value of sample j + 1, halved
        for (int j = i;; ++j) {
          const double rh = rh_next;
          const bool more = (j + 1 < n) && flagged(j + 1);
          if (more) rh_next = 0.5 * quot(2 * x[min(j + 2, n - 1)] - med2);
          double nv;
          if (j == 0) {
            nv = 2.0 * rh;                       // arr[0] = arr[1] (raw)
          } else if (j == n - 1) {
            nv = prev;                           // arr[n-1] = arr[n-2] (already updated)
          } else {
            nv = clip_outlier(__fma_rn(prev, 0.5, rh));
          }
          o[j] = static_cast<float>(nv);
          prev = nv;
          if (!more) break;
        }
      };

      // ---- normalise: 4 samples per thread and step, 16-byte stores; outlier-run starts are pushed to s.runs.
      //      The window's phase inside its 8-byte staging words (sh = a & 3, block-uniform) selects one of four
      //      specialised loops: at most two shared loads and two funnel shifts per group, running pointers, no
      //      per-group address arithmetic (the loop is issue-bound: 87 -> ~30 instructions per group).
      const int sh = a & 3;
      // |2x - med2| > dthr  <=>  x > x_hi or x < x_lo (clamped to int16: beyond the type nothing can exceed);
      // tested for the group's four samples at once on the packed 16-bit halves
      const int x_hi = min(32767, (med2 + static_cast<int>(dthr)) >> 1);            // floor
      const int x_lo = max(-32768, (med2 - static_cast<int>(dthr) + 1) >> 1);       // ceil
      const uint32_t hi2 = (static_cast<uint32_t>(x_hi) & 0xffffu) * 0x10001u;
      const uint32_t lo2 = (static_cast<uint32_t>(x_lo) & 0xffffu) * 0x10001u;
      // Outlier bookkeeping stays out of the hot loop: a thread only notes WHICH of its groups held an outlier (one
      // bit per step) and looks at those groups again afterwards, pushing the starts of outlier runs to s.runs.
      auto note_runs = [&](uint32_t mask, int step0) {
        while (mask) {
          const int it_ = __ffs(mask) - 1;
          mask &= mask - 1;
          const int i0 = 4 * (tid + (step0 + it_) * kThreads);
          const int cnt = min(4, n - i0);
          bool fprev = (i0 > 0) && flagged(i0 - 1);
          for (int e = 0; e < cnt; ++e) {
            const bool fe = flagged(i0 + e);
            if (fe && !fprev) {
              const uint32_t pos = atomicAdd(&s.n_runs, 1u);
              if (pos < static_cast<uint32_t>(kMaxRuns)) s.runs[pos] = i0 + e;
            }
            fprev = fe;
          }
        }
      };
      const int n_full = n >> 2;                       // groups of four whole samples
      auto group_loop = [&](auto sh_const, auto nf_const, auto value_of, auto value_of_x4, auto f64_x4) {
        constexpr int SH = decltype(sh_const)::value;
        constexpr int NF = decltype(nf_const)::value;
        // group g = samples 4g .. 4g + 3 = 16-bit halves SH .. SH + 3 of the staging words wbase[2g ..]
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(stage + (a & ~3)) + 2 * tid;
        float4* op = reinterpret_cast<float4*>(o) + tid;
        for (int g0 = 0; g0 < n_full; g0 += 32 * kThreads) {       // 32 steps (32,768 samples) per mask word
          uint32_t gmask = 0, bit = 1;
          const int g1 = min(n_full, g0 + 32 * kThreads);
#pragma unroll 2
          for (int g = g0 + tid; g < g1; g += kThreads, wp += 2 * kThreads, op += kThreads, bit <<= 1) {
            uint32_t p0, p1;
            if (SH == 0) {
              const uint2 v = *reinterpret_cast<const uint2*>(wp);
              p0 = v.x;
              p1 = v.y;
            } else if (SH == 1) {
              const uint2 v = *reinterpret_cast<const uint2*>(wp);
              const uint32_t c = wp[2];
              p0 = __funnelshift_r(v.x, v.y, 16);
              p1 = __funnelshift_r(v.y, c, 16);
            } else if (SH == 2) {
              p0 = wp[1];
              p1 = wp[2];
            } else {
              const uint32_t c = wp[1];
              const uint2 v = *reinterpret_cast<const uint2*>(wp + 2);
              p0 = __funnelshift_r(c, v.x, 16);
              p1 = __funnelshift_r(v.x, v.y, 16);
            }
            float4 v;      // value_of_x4(p): the value of a sample given 4 * sample; NF of the four on the float64 pipe
            v.x = (NF >= 4) ? f64_x4(static_cast<int>(p0 << 16) >> 14) : value_of_x4(static_cast<int>(p0 << 16) >> 14);
            v.y = (NF >= 2) ? f64_x4(static_cast<int>(p0 & 0xffff0000u) >> 14) : value_of_x4(static_cast<int>(p0 & 0xffff0000u) >> 14);
            v.z = (NF >= 3) ? f64_x4(static_cast<int>(p1 << 16) >> 14) : value_of_x4(static_cast<int>(p1 << 16) >> 14);
            v.w = (NF >= 1) ? f64_x4(static_cast<int>(p1 & 0xffff0000u) >> 14) : value_of_x4(static_cast<int>(p1 & 0xffff0000u) >> 14);
            *op = v;
            // some sample of this group is an outlier
            if (__vimax3_s16x2(p0, p1, hi2) != hi2 || __vimin3_s16x2(p0, p1, lo2) != lo2) gmask |= bit;
          }
          if (gmask) note_runs(gmask, g0 / kThreads);
        }
        // the (< 4) samples after the last whole group: one thread, sample by sample
        if (tid == (n_full & (kThreads - 1)) && (n & 3)) {
          uint32_t m = 0;
          for (int i = 4 * n_full; i < n; ++i) {
            o[i] = value_of(x[i]);
            m |= flagged(i) ? 1u : 0u;
          }
          if (m) note_runs(1u, n_full / kThreads);
        }
      };
      auto f64_value = [&](int xv) { return static_cast<float>(quot(2 * xv - med2)); };
      auto f64_x4 = [&](int x4) { return static_cast<float>(quot((x4 >> 1) - med2)); };
      auto dispatch = [&](auto nf_const, auto value_of, auto value_of_x4) {
        if (sh == 0) group_loop(std::integral_constant<int, 0>{}, nf_const, value_of, value_of_x4, f64_x4);
        else if (sh == 1) group_loop(std::integral_constant<int, 1>{}, nf_const, value_of, value_of_x4, f64_x4);
        else if (sh == 2) group_loop(std::integral_constant<int, 2>{}, nf_const, value_of, value_of_x4, f64_x4);
        else group_loop(std::integral_constant<int, 3>{}, nf_const, value_of, value_of_x4, f64_x4);
      };
      if (use_lut) {
        const uint32_t lut_addr = smem_u32(lut);      // shared-space byte address; entry of value v at 4 (v & (kBins - 1))
        auto lut_value = [&](int xv) { return lut[xv & (kBins - 1)]; };
        auto lut_x4 = [&](int x4) {
          float f;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f) : "r"(lut_addr + (static_cast<uint32_t>(x4) & (4u * (kBins - 1)))));
          return f;
        };
        // kDefaultF64 of every group of four samples take their quotient from the float64 pipe rather than the table
        // (same results: the table's bank conflicts load the LSU pipe, which then bounds the kernel)
        dispatch(std::integral_constant<int, kDefaultF64>{}, lut_value, lut_x4);
      } else {
        dispatch(std::integral_constant<int, 4>{}, f64_value, f64_x4);
      }
      __syncthreads();   // every sample has its plain quotient; the runs overwrite theirs
      const uint32_t n_runs = s.n_runs;
      if (n_runs <= static_cast<uint32_t>(kMaxRuns)) {
        for (uint32_t r = tid; r < n_runs; r += kThreads) walk(s.runs[r]);
      } else {             // list overflowed: find the run starts again
        for (int i = tid; i < n; i += kThreads)
          if (flagged(i) && !(i > 0 && flagged(i - 1))) walk(i);
      }
    }
    __syncthreads();   // stage / scratch are reused by the next read
  }
}

// ------------------------------------------------------------------------------------
// poly(A) end detection.  One CTA per read; one warp per 500-sample window.

constexpr int kRes = 500;               // _TRIM_RESOLUTION, riser/preprocess.py:10
constexpr int kPerLane = (kRes + 31) / 32;   // 16
constexpr int kMaxWindows = 512;        // windows per read (256,000 samples; the live path stops near 18,500)
constexpr int kPolyaThreads = 128;      // 4 warps per read: an 18,000-sample prefix has 36 windows, 9 per warp
constexpr int kPolyaWarps = kPolyaThreads / 32;
constexpr int kWinBins = 1024;          // value range a window's shared-memory histogram covers
constexpr int kWinHist = 33 * 32 + 32;  // per-warp histogram storage: 32 lanes x (odd) segment of up to 33 bins

// rank-k (0-based) key among this warp's keys (all < 2^nbits; padding lanes hold 0xffffffff): binary search
// on the value, one warp-wide count #{key < T} per bit (REDUX) -- the "warp-shuffle selection" of the north
// star.  nbits comes from the window's own range, so a 500-sample window costs ~10 steps, not 16.
__device__ __forceinline__ uint32_t warp_select(const uint32_t (&key)[kPerLane], int nbits, uint32_t k) {
  uint32_t prefix = 0;
  for (int bit = nbits - 1; bit >= 0; --bit) {
    const uint32_t t = prefix | (1u << bit);
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) cnt += (key[j] < t) ? 1 : 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (k >= static_cast<uint32_t>(cnt)) prefix = t;      // rank k lies at or above t
  }
  return prefix;
}

// the two middle order statistics (ranks 249 and 250 of 500) -> their sum
__device__ __forceinline__ uint32_t warp_mid_sum(const uint32_t (&key)[kPerLane], int nbits) {
  const uint32_t v1 = warp_select(key, nbits, kRes / 2 - 1);
  int le = 0;
  uint32_t next = 0xffffffffu;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    le += key[j] <= v1 ? 1 : 0;
    if (key[j] > v1) next = min(next, key[j]);      // (padding keys are 0xffffffff: never the minimum of 500 real keys)
  }
  le = __reduce_add_sync(0xffffffffu, le);
  next = __reduce_min_sync(0xffffffffu, next);
  const uint32_t v2 = (le > kRes / 2) ? v1 : next;
  return v1 + v2;
}

__device__ __forceinline__ int bits_of(uint32_t v) { return 32 - __clz(v); }

// Median and MAD of one 500-sample window from a per-warp shared-memory histogram of x - vmin (range < kWinBins,
// which covers every real squiggle window; wider windows take the bit-descent path below): ~3x fewer instructions
// than two 10..11-step bit-descents.  h becomes the inclusive prefix P[u] = #{x - vmin <= u}; the two middle order
// statistics are found by warp-wide searches on P, and those of |2x - 2 median| from the same P (as in the
// normalise kernel): #{|2(x - vmin) - m| <= d} = P[floor((m + d) / 2)] - P[ceil((m - d) / 2) - 1].
__device__ __forceinline__ void warp_hist_stats(const int (&v)[kPerLane], const bool (&ok)[kPerLane], int vmin, int range,
                                                uint32_t* h, int& med2, uint32_t& mad4) {
  const int lane = threadIdx.x & 31;
  const int nb = range + 1;
  int seg = (nb + 31) >> 5;                 // bins per lane; odd, so the lanes' segments start in distinct banks
  seg |= 1;
  const int n_clear = (32 * seg + 3) >> 2;  // 16-byte words to clear
  for (int i = lane; i < n_clear; i += 32) reinterpret_cast<uint4*>(h)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncwarp();
#pragma unroll
  for (int j = 0; j < kPerLane; ++j)
    if (ok[j]) atomicAdd(&h[v[j] - vmin], 1u);
  __syncwarp();
  // in-place inclusive prefix: lane sums its segment, warp scan of the sums, second sweep writes
  uint32_t* mine = h + lane * seg;
  uint32_t tot = 0;
  for (int i = 0; i < seg; ++i) tot += mine[i];
  uint32_t inc = tot;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += u;
  }
  uint32_t run = inc - tot;
  for (int i = 0; i < seg; ++i) {
    run += mine[i];
    mine[i] = run;
  }
  __syncwarp();
  // smallest u with P[u] >= want, for want = 250 (lanes 0-15) and 251 (lanes 16-31): 16-ary search
  const int half = lane >> 4, sub = lane & 15;
  const uint32_t want = static_cast<uint32_t>(kRes / 2 + half);
  const uint32_t hmask = half ? 0xffff0000u : 0x0000ffffu;
  int lo = 0, hi = range;                   // invariant: P[hi] >= want (P[range] = 500)
  while (__any_sync(0xffffffffu, lo < hi)) {   // the two half-warp searches run in lock-step; a finished one idles
    const int step = (hi - lo + 16) >> 4;   // ceil(span / 16)
    const int u = min(lo + (sub + 1) * step - 1, hi);
    const uint32_t okm = __ballot_sync(0xffffffffu, h[u] >= want) & hmask;
    const int f = (__ffs(okm) - 1) & 15;    // sub-lane 15 probes hi: never empty
    hi = min(lo + (f + 1) * step - 1, hi);
    lo = lo + f * step;
  }
  const int u1 = __shfl_sync(0xffffffffu, lo, 0), u2 = __shfl_sync(0xffffffffu, lo, 16);
  const int m = u1 + u2;
  med2 = 2 * vmin + m;
  // the same search on the distance d = |2(x - vmin) - m|
  lo = 0;
  hi = max(m, 2 * range - m);               // count(hi) = 500
  while (__any_sync(0xffffffffu, lo < hi)) {   // the two half-warp searches run in lock-step; a finished one idles
    const int step = (hi - lo + 16) >> 4;
    const int d = min(lo + (sub + 1) * step - 1, hi);
    const int hi_u = min((m + d) >> 1, range);
    const int lo_u = (m - d + 1) >> 1;      // ceil((m - d) / 2), may be <= 0
    const uint32_t cnt = h[hi_u] - (lo_u > 0 ? h[lo_u - 1] : 0u);
    const uint32_t okm = __ballot_sync(0xffffffffu, cnt >= want) & hmask;
    const int f = (__ffs(okm) - 1) & 15;
    hi = min(lo + (f + 1) * step - 1, hi);
    lo = lo + f * step;
  }
  mad4 = static_cast<uint32_t>(__shfl_sync(0xffffffffu, lo, 0) + __shfl_sync(0xffffffffu, lo, 16));
  __syncwarp();                             // h is cleared again for the warp's next window
}

// Product path of the poly(A) scan (no per-window statistics requested): riser/preprocess.py:45-72 only needs a
// window's SUM and whether its MAD exceeds 20, so the exact MAD search and the prefix array are skipped.  The window
// stays in its packed 16-bit words (8 per lane, word j * 32 + lane of the window's 250); sum, minimum and maximum
// come from packed SIMD instructions; the histogram is read by ROWS of 32 bins (one bin per lane): the row holding
// the two middle order statistics is found by adding row totals, the bins inside it by one warp scan.  With
// d = |2 x - 2 median| and c = #{d <= 40} (three rows at most), 4 MAD = d_(249) + d_(250) > 80 iff c <= 249,
// <= 80 iff c >= 251; c == 250 (the two statistics straddle 40) is decided from the largest d <= 40 and the smallest
// d > 40 found in the histogram.  Returns false when the window's range does not fit the histogram (the caller's
// exact bit-descent path then handles it).
__device__ __forceinline__ bool warp_window_fast(const uint32_t (&raw)[kPerLane / 2], uint32_t* h, int& sum_out,
                                                 bool& mad_gt20) {
  const int lane = threadIdx.x & 31;
  const bool last_ok = (7 * 32 + lane) < kRes / 2;            // word 7 exists for lanes 0..25 only
  const uint32_t r7 = last_ok ? raw[7] : raw[0];              // (a copy of a valid word leaves min / max unchanged)
  int sum = 0;
#pragma unroll
  for (int j = 0; j < 7; ++j) sum = __dp2a_lo(static_cast<int>(raw[j]), 0x0101, sum);
  if (last_ok) sum = __dp2a_lo(static_cast<int>(raw[7]), 0x0101, sum);
  uint32_t mn2 = __vimin3_s16x2(raw[0], raw[1], raw[2]), mx2 = __vimax3_s16x2(raw[0], raw[1], raw[2]);
  mn2 = __vimin3_s16x2(mn2, raw[3], raw[4]);
  mx2 = __vimax3_s16x2(mx2, raw[3], raw[4]);
  mn2 = __vimin3_s16x2(mn2, raw[5], raw[6]);
  mx2 = __vimax3_s16x2(mx2, raw[5], raw[6]);
  mn2 = __vimin3_s16x2(mn2, r7, r7);
  mx2 = __vimax3_s16x2(mx2, r7, r7);
  int vmin = min(static_cast<int>(static_cast<int16_t>(mn2 & 0xffffu)), static_cast<int>(mn2) >> 16);
  int vmax = max(static_cast<int>(static_cast<int16_t>(mx2 & 0xffffu)), static_cast<int>(mx2) >> 16);
  sum = __reduce_add_sync(0xffffffffu, sum);
  vmin = __reduce_min_sync(0xffffffffu, vmin);
  vmax = __reduce_max_sync(0xffffffffu, vmax);
  const int range = vmax - vmin;
  if (range >= kWinBins) return false;
  sum_out = sum;
  for (int i = lane; i < ((range + 4) >> 2); i += 32) reinterpret_cast<uint4*>(h)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncwarp();
  const uint32_t h_addr = smem_u32(h) - 4u * static_cast<uint32_t>(vmin);
  auto count = [&](uint32_t word) {       // both halves of a packed word: bin address = h + 4 (x - vmin)
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(h_addr + static_cast<uint32_t>(static_cast<int>(word << 16) >> 14)) : "memory");
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(h_addr + static_cast<uint32_t>(static_cast<int>(word & 0xffff0000u) >> 14)) : "memory");
  };
#pragma unroll
  for (int j = 0; j < 7; ++j) count(raw[j]);
  if (last_ok) count(raw[7]);
  __syncwarp();
  // ---- the two middle order statistics (0-based ranks 249, 250) as bin indices u1 <= u2
  const int n_rows = (range + 32) >> 5;
  uint32_t before = 0, c = 0;
  int row = 0;
  for (;; row += 2) {                      // warp-uniform; ends at the latest in the last row (total = 500)
    // two rows per step: their totals (<= 500 each) travel through one warp reduction as 16-bit halves
    const int b = 32 * row + lane;
    const uint32_t c0 = (b <= range) ? h[b] : 0u, c1 = (b + 32 <= range) ? h[b + 32] : 0u;
    const uint32_t tot = __reduce_add_sync(0xffffffffu, c0 | (c1 << 16));
    c = c0;
    if (before + (tot & 0xffffu) >= static_cast<uint32_t>(kRes / 2) || row + 1 >= n_rows) break;
    before += tot & 0xffffu;
    c = c1;
    if (before + (tot >> 16) >= static_cast<uint32_t>(kRes / 2) || row + 2 >= n_rows) {
      ++row;
      break;
    }
    before += tot >> 16;
  }
  uint32_t inc = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += u;
  }
  inc += before;
  const uint32_t m1 = __ballot_sync(0xffffffffu, inc >= static_cast<uint32_t>(kRes / 2));
  const uint32_t m2 = __ballot_sync(0xffffffffu, inc >= static_cast<uint32_t>(kRes / 2 + 1));
  const int u1 = 32 * row + __ffs(m1) - 1;
  int u2;
  if (m2) {
    u2 = 32 * row + __ffs(m2) - 1;
  } else {                                 // rank 250 is the first occupied bin of a later row
    u2 = range;
    for (int r = row + 1; r < n_rows; ++r) {
      const int b = 32 * r + lane;
      const uint32_t occ = __ballot_sync(0xffffffffu, b <= range && h[b] != 0u);
      if (occ) {
        u2 = 32 * r + __ffs(occ) - 1;
        break;
      }
    }
  }
  const int m = u1 + u2;                   // 2 median = 2 vmin + m
  // ---- c40 = #{u : |2 u - m| <= 40}; the largest such d and the smallest d above 40 for the straddling case
  const int lo_u = max(0, (m - 40 + 1) >> 1), hi_u = min(range, (m + 40) >> 1);
  uint32_t c40 = 0;
  for (int r = lo_u >> 5; r <= (hi_u >> 5); ++r) {
    const int b = 32 * r + lane;
    if (b >= lo_u && b <= hi_u) c40 += h[b];
  }
  c40 = __reduce_add_sync(0xffffffffu, c40);
  if (c40 != static_cast<uint32_t>(kRes / 2)) {
    mad_gt20 = c40 < static_cast<uint32_t>(kRes / 2);
  } else {
    int d1 = 0, d2 = 0x7fffffff;           // d1: ranks 0..249 all lie at d <= 40; d2: rank 250 is the smallest d > 40
    for (int r = 0; r < n_rows; ++r) {
      const int b = 32 * r + lane;
      if (b <= range && h[b] != 0u) {
        const int d = abs(2 * b - m);
        if (d <= 40) d1 = max(d1, d); else d2 = min(d2, d);
      }
    }
    d1 = __reduce_max_sync(0xffffffffu, d1);
    d2 = __reduce_min_sync(0xffffffffu, d2);
    mad_gt20 = d1 + d2 > 80;
  }
  __syncwarp();                            // h is cleared again for the warp's next window
  return true;
}

__global__ void __launch_bounds__(kPolyaThreads)
polya_kernel(const int16_t* __restrict__ sig, const int64_t* __restrict__ off,
             const int32_t* __restrict__ nsamp, int B, int32_t* __restrict__ polya_end,
             int32_t* __restrict__ polya_start, int32_t* __restrict__ stats, int max_windows) {
  __shared__ int32_t w_sum[kMaxWindows];
  __shared__ int32_t w_mad4[kMaxWindows];
  __shared__ __align__(16) uint32_t w_hist[kPolyaWarps][kWinHist];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int n = nsamp[b];
    const int16_t* g = sig + off[b];
    const int nw = min(n / kRes, kMaxWindows);
    // 4-byte loads when the read is 4-byte aligned (a window is 1,000 bytes): a lane takes sample pairs -- which lane
    // holds which sample is irrelevant to the statistics -- and the NEXT window of this warp is fetched while the
    // current one is worked on
    const bool al4 = (reinterpret_cast<uintptr_t>(g) & 3) == 0;
    uint32_t raw[kPerLane / 2];
    auto fetch = [&](int w) {
      const uint32_t* wp2 = reinterpret_cast<const uint32_t*>(g + w * kRes);
#pragma unroll
      for (int j = 0; j < kPerLane / 2; ++j) {
        const int idx = j * 32 + lane;
        raw[j] = (idx < kRes / 2) ? __ldg(wp2 + idx) : 0u;
      }
    };
    if (al4 && warp < nw) fetch(warp);
    for (int w = warp; w < nw; w += kPolyaWarps) {
      const int16_t* wp = g + w * kRes;
      int v[kPerLane];
      int sum = 0, vmin = 32767, vmax = -32768;
      bool ok[kPerLane];
      if (al4) {
        uint32_t cur[kPerLane / 2];
#pragma unroll
        for (int j = 0; j < kPerLane / 2; ++j) cur[j] = raw[j];
        if (w + kPolyaWarps < nw) fetch(w + kPolyaWarps);
        if (!stats) {
          int fsum;
          bool gt;
          if (warp_window_fast(cur, w_hist[warp], fsum, gt)) {
            if (lane == 0) {
              w_sum[w] = fsum;
              w_mad4[w] = gt ? 84 : 80;      // (the scan below only asks whether mad4 / 4 exceeds 20)
            }
            continue;
          }
        }
#pragma unroll
        for (int j = 0; j < kPerLane / 2; ++j) {
          ok[2 * j] = ok[2 * j + 1] = (j * 32 + lane) < kRes / 2;
          v[2 * j] = static_cast<int16_t>(cur[j] & 0xffffu);
          v[2 * j + 1] = static_cast<int16_t>(cur[j] >> 16);
        }
      } else {
#pragma unroll
        for (int j = 0; j < kPerLane; ++j) {
          const int idx = j * 32 + lane;
          ok[j] = idx < kRes;
          v[j] = ok[j] ? static_cast<int>(wp[idx]) : 0;
        }
      }
#pragma unroll
      for (int j = 0; j < kPerLane; ++j) {
        sum += v[j];
        vmin = min(vmin, ok[j] ? v[j] : 32767);
        vmax = max(vmax, ok[j] ? v[j] : -32768);
      }
      sum = __reduce_add_sync(0xffffffffu, sum);
      vmin = __reduce_min_sync(0xffffffffu, vmin);
      vmax = __reduce_max_sync(0xffffffffu, vmax);
      if (vmax - vmin < kWinBins) {
        int med2h;
        uint32_t mad4h;
        warp_hist_stats(v, ok, vmin, vmax - vmin, w_hist[warp], med2h, mad4h);
        if (lane == 0) {
          w_sum[w] = sum;
          w_mad4[w] = static_cast<int32_t>(mad4h);
          if (stats && w < max_windows) {
            int32_t* st = stats + (static_cast<int64_t>(b) * max_windows + w) * 3;
            st[0] = sum;
            st[1] = med2h;
            st[2] = static_cast<int32_t>(mad4h);
          }
        }
        continue;
      }
      // median on keys x - min (as many bits as the window's range needs)
      uint32_t key[kPerLane];
#pragma unroll
      for (int j = 0; j < kPerLane; ++j)
        key[j] = ok[j] ? static_cast<uint32_t>(v[j] - vmin) : 0xffffffffu;
      const int med2 = 2 * vmin + static_cast<int>(warp_mid_sum(key, bits_of(static_cast<uint32_t>(vmax - vmin))));   // 2 * median
      // MAD on keys |2x - 2 median|
      const uint32_t dmax = static_cast<uint32_t>(max(abs(2 * vmin - med2), abs(2 * vmax - med2)));
#pragma unroll
      for (int j = 0; j < kPerLane; ++j)
        key[j] = ok[j] ? static_cast<uint32_t>(abs(2 * v[j] - med2)) : 0xffffffffu;
      const uint32_t mad4 = warp_mid_sum(key, bits_of(dmax));                         // 4 * MAD
      if (lane == 0) {
        w_sum[w] = sum;
        w_mad4[w] = static_cast<int32_t>(mad4);
        if (stats && w < max_windows) {
          int32_t* st = stats + (static_cast<int64_t>(b) * max_windows + w) * 3;
          st[0] = sum;
          st[1] = med2;
          st[2] = static_cast<int32_t>(mad4);
        }
      }
    }
    __syncthreads();
    if (warp == 0) {
      // riser/preprocess.py:45-72.  0 doubles as "unset" exactly like Python truthiness.  The per-window tests
      // (three float64 divides each) are independent, so the lanes evaluate 32 windows at a time and the two-state
      // scan runs on the ballots: start = first window > 0 with mean_change > 20 and mad <= 20; end = first window
      // after it with mad > 20.
      int pstart = 0, pend = 0;
      for (int w0 = 0; w0 < nw && pend == 0; w0 += 32) {
        const int w = w0 + lane;
        bool cs = false, ce = false;
        if (w < nw) {
          const double mean = __ddiv_rn(static_cast<double>(w_sum[w]), static_cast<double>(kRes));
          double rolling = mean;
          if (w > 2)
            rolling = __ddiv_rn(static_cast<double>(w_sum[w - 2] + w_sum[w - 1]),
                                static_cast<double>(2 * kRes));
          const double change = __dmul_rn(__ddiv_rn(__dsub_rn(mean, rolling), rolling), 100.0);
          const double mad = static_cast<double>(w_mad4[w]) * 0.25;
          cs = w > 0 && change > 20.0 && mad <= 20.0;
          ce = mad > 20.0;
        }
        const uint32_t ms = __ballot_sync(0xffffffffu, cs);
        uint32_t me = __ballot_sync(0xffffffffu, ce);
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

// riser/control.py:36-60 length gating
__global__ void select_window_kernel(const int32_t* __restrict__ n, const int32_t* __restrict__ cached,
                                     const int32_t* __restrict__ detected, int B, int min_len, int max_len,
                                     int fixed_trim, int32_t* __restrict__ start, int32_t* __restrict__ len) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int nb = n[b];
  int end = cached ? cached[b] : -1;
  if (end < 0 && detected) end = detected[b];
  int st = 0, ln = 0;
  if (end > 0) {                               // Python truthiness: 0 / None = not found
    const int avail = nb - (end + 1);
    if (avail >= min_len) {
      st = end + 1;
      ln = min(avail, max_len);
    }
  } else if (nb > fixed_trim + max_len) {      // preprocess.py:84-85 (strict)
    st = fixed_trim;
    ln = max_len;
  }
  start[b] = st;
  len[b] = ln;
}

int g_sm_count = 0;
int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      g_sm_count = 148;
  }
  return g_sm_count;
}

}  // namespace
}  // namespace riser

using namespace riser;

extern "C" int riser_version(void) { return 100; }
extern "C" const char* riser_last_error(void) { return err_buf(); }

extern "C" int riser_device_info(int device, int* sm, int* major, int* minor) {
  RISER_REQUIRE(sm && major && minor, "riser_device_info: null output pointer");
  RISER_CUDA_TRY(cudaDeviceGetAttribute(sm, cudaDevAttrMultiProcessorCount, device));
  RISER_CUDA_TRY(cudaDeviceGetAttribute(major, cudaDevAttrComputeCapabilityMajor, device));
  RISER_CUDA_TRY(cudaDeviceGetAttribute(minor, cudaDevAttrComputeCapabilityMinor, device));
  return RISER_OK;
}

extern "C" int riser_normalise_max_len(void) { return kMaxLen; }

extern "C" int riser_normalise(const int16_t* sig, const int64_t* off, const int32_t* start,
                               const int32_t* len, int B, int max_len, float* out, int64_t ld_out,
                               int32_t* med2_mad4, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_normalise: B < 0");
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(sig && off && len && out, "riser_normalise: null pointer");
  RISER_REQUIRE(max_len > 0 && max_len <= kMaxLen, "riser_normalise: max_len %d outside (0, %d]",
                max_len, kMaxLen);
  RISER_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ld_out & 3) == 0 && ld_out >= max_len,
                "riser_normalise: out must be 16-byte aligned, ld_out a multiple of 4 and >= max_len");
  // staging buffer of whole 16-byte blocks: window + up to 7 samples of phase + tail block, 128-byte pitch
  const int buf_samples = (max_len + 16 + 63) & ~63;
  const size_t scratch = (sizeof(SelectScratch) + 127) & ~size_t(127);
  // One staging buffer + L2 prefetch of the next read: a second buffer (the next read's copy in flight during this
  // read's work) costs a resident CTA per SM and measured slower.
  const size_t smem = scratch + 2 * static_cast<size_t>(buf_samples);
  static size_t configured[64] = {0};   // per device
  int dev = 0;
  RISER_CUDA_TRY(cudaGetDevice(&dev));
  if (smem > configured[dev & 63]) {
    RISER_CUDA_TRY(cudaFuncSetAttribute(normalise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    configured[dev & 63] = smem;
  }
  int per_sm = 0;
  RISER_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, normalise_kernel, kThreads, smem));
  if (per_sm < 1) per_sm = 1;
  const int grid = std::min(B, sm_count() * per_sm);
  normalise_kernel<<<grid, kThreads, smem, as_stream(stream)>>>(sig, off, start, len, B, out, ld_out,
                                                               med2_mad4, max_len);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_select_window(const int32_t* n, const int32_t* cached_end, const int32_t* detected_end,
                                   int B, int min_len, int max_len, int fixed_trim, int32_t* start,
                                   int32_t* len, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_select_window: B < 0");
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(n && start && len, "riser_select_window: null pointer");
  select_window_kernel<<<(B + 255) / 256, 256, 0, as_stream(stream)>>>(n, cached_end, detected_end, B, min_len,
                                                                     max_len, fixed_trim, start, len);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_polya_end(const int16_t* sig, const int64_t* off, const int32_t* n, int B,
                               int32_t* polya_end, int32_t* polya_start, int32_t* stats, int max_windows,
                               riser_stream_t stream) {
  RISER_REQUIRE(B >= 0, "riser_polya_end: B < 0");
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(sig && off && n && polya_end, "riser_polya_end: null pointer");
  RISER_REQUIRE(!stats || max_windows > 0, "riser_polya_end: stats given but max_windows <= 0");
  int per_sm = 0;
  RISER_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, polya_kernel, kPolyaThreads, 0));
  const int grid = std::min(B, sm_count() * std::max(per_sm, 1));
  polya_kernel<<<grid, kPolyaThreads, 0, as_stream(stream)>>>(sig, off, n, B, polya_end, polya_start, stats, max_windows);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
