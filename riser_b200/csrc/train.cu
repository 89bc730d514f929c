// Backward pass of the ConvNet (riser/nets/cnn.py:8-65) for training on the GPU (riser_b200/training.py).
//
// The forward pass and the input gradients (dgrad) reuse the channel-last fp32 ops of csrc/resnet.cu
// (riser_conv1d_cl with the tap-flipped, transposed weight; riser_maxpool1d_pad_cl; riser_len_chain).  This file
// holds what they do not cover:
//   * riser_conv1d_wgrad_cl: weight and bias gradients of a stride-1 'same' Conv1d.  The GEMM
//       dW_j[co][ci] = sum over rows r of dZ[r][co] X[r + j - pad][ci]
//     reduces over the rows of the whole batch, so it runs on tcgen05 with the rows as the K dimension: a CTA owns a
//     128-output-channel x N-input-channel tile for every tap (K accumulators side by side in TMEM) and one of S
//     row splits.  The operands are converted in the kernel from fp32 to bf16 hi + lo planes (a = hi + lo exact to
//     ~2^-17 relative; bf16 keeps fp32's exponent range, so gradients need no scaling) and the three products
//     hi*hi + hi*lo + lo*hi accumulate in fp32.  The bias gradient is one more input channel that is 1 on every
//     valid row: the centre tap's accumulator column for it is sum_r dZ[r][co].  Each split writes its partial
//     sums to the workspace and a second launch adds them in split order: no float atomics, the same bits on every
//     run.
//   riser_conv1d_wgrad_ex is the same kernel for any stride and padding (the ResNet's strided, padded convolutions,
//   csrc/train_resnet.cu): the B operand of tap j for output row t is x[t * stride + j - pad] and the ones channel is
//   1 on every valid output row, so the bias gradient does not depend on the taps that read the padding.
//   * riser_relu_pool_bwd_cl: the gradient through ReLU and MaxPool1d(2, 2), the ResNet stem's MaxPool1d(2, 2,
//     padding 1), or ReLU alone;
//   * riser_gap_linear_ce_bwd: AdaptiveAvgPool1d(1) + Linear + CrossEntropyLoss (mean), forward and backward.
#include "common.cuh"

#include <cuda_bf16.h>

#include <algorithm>

namespace riser {
namespace {

constexpr int kWgThreads = 256;
constexpr int kWgRows = 32;            // rows (K elements) per stage: one 64-byte bf16 row of a SWIZZLE_64B tile
constexpr int kWgM = 128;              // output channels per CTA (MMA M)
constexpr int kWgTargetCtas = 148;     // split factor: tiles x splits ~ one wave of a B200 (a constant, so that the
                                       // summation order, hence the result, is the same on every device)
constexpr uint32_t kWgAPlane = kWgM * 64;   // bytes of one A plane (128 rows x 64 B)

struct WgArgs {
  const float* dz;       // [B][L_pad][Cout]
  const float* x;        // [B][Lin_pad][Cin]
  const int32_t* len;    // [B] output lengths
  const int32_t* len_in; // [B] input lengths
  float* part;           // [S][K][Cin + 1][Cout]
  int B, L_pad, Cin, Cout, K, pad;
  int Lin_pad, stride;
  int n;                 // MMA N (input channels per CTA, multiple of 16)
  int S;
  int64_t rows;          // B * L_pad (output rows)
  int64_t chunks;        // ceil(rows / kWgRows)
  uint32_t stage_bytes, tmem_cols;
};

__device__ __forceinline__ uint32_t sw64(int r, int byte) {    // SWIZZLE_64B: 16-byte chunk c of row r at c ^ ((r >> 1) & 3)
  return static_cast<uint32_t>(r * 64 + ((((byte >> 4) ^ (r >> 1)) & 3) << 4) + (byte & 15));
}

__device__ __forceinline__ uint64_t wg_desc(uint32_t addr) {    // K-major SWIZZLE_64B, 8-row atoms of 512 B
  constexpr uint64_t kHi = (static_cast<uint64_t>(1) << 16) | (static_cast<uint64_t>(512 >> 4) << 32) |
                           (static_cast<uint64_t>(1) << 46) | (static_cast<uint64_t>(4) << 61);
  return kHi | static_cast<uint64_t>(addr >> 4);
}

// kind::f16 instruction descriptor with bf16 A and B (format code 1), fp32 D, both K-major
__host__ __device__ inline uint32_t idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// 8 fp32 values -> bf16 hi (16 bytes) and bf16 lo = bf16(v - hi)
__device__ __forceinline__ void split8_bf16(const float (&v)[8], uint4& hi, uint4& lo) {
  __nv_bfloat162 h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    h[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    const float2 back = __bfloat1622float2(h[j]);
    l[j] = __floats2bfloat162_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
  }
  hi = *reinterpret_cast<const uint4*>(h);
  lo = *reinterpret_cast<const uint4*>(l);
}

__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_tc_kernel(const WgArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  __shared__ uint64_t mma_done[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int co0 = blockIdx.x * kWgM, ci0 = blockIdx.y * a.n, s = blockIdx.z;
  const int Cin1 = a.Cin + 1;                       // + the ones channel of the bias gradient
  const uint32_t b_plane = static_cast<uint32_t>(a.n) * 64u;
  if (tid == 0) {
    mbar_init(&mma_done[0], 1);
    mbar_init(&mma_done[1], 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(&tmem_slot, a.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t idesc = idesc_bf16(kWgM, a.n);
  const int a_units = kWgM * 4, b_units = a.n * 4;  // (channel, 8-row group) units of a stage

  int it = 0;                                       // stages issued by this CTA
  for (int64_t q = s; q < a.chunks; q += a.S) {
    const int64_t r0 = q * kWgRows;
    // skip a chunk with no valid row (the same decision in every warp: a ballot over the chunk's 32 rows)
    bool v_row = false;
    {
      const int64_t r = r0 + lane;
      if (r < a.rows) {
        const int b = static_cast<int>(r / a.L_pad), t = static_cast<int>(r - static_cast<int64_t>(b) * a.L_pad);
        v_row = t < __ldg(a.len + b);
      }
    }
    if (__ballot_sync(0xffffffffu, v_row) == 0u) continue;
    const int slot = it & 1;
    if (it >= 2) mbar_wait(&mma_done[slot], static_cast<uint32_t>((it >> 1) - 1) & 1u);   // its previous MMAs are done
    unsigned char* st = base + slot * a.stage_bytes;
    // A = dZ^T: row c = output channel co0 + c, K = the chunk's rows; rows t >= len read as 0
    for (int u = tid; u < a_units + a.K * b_units; u += kWgThreads) {
      int c, g, j = -1;
      if (u < a_units) {
        c = u % kWgM; g = u / kWgM;
      } else {
        const int ub = u - a_units;
        j = ub / b_units;
        const int rem = ub - j * b_units;
        c = rem % a.n; g = rem / a.n;
      }
      float v[8];
      int64_t r = r0 + 8 * g;
      int b = static_cast<int>(r / a.L_pad), t = static_cast<int>(r - static_cast<int64_t>(b) * a.L_pad);
      if (j < 0) {
        const int co = co0 + c;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float val = 0.f;
          if (r < a.rows && co < a.Cout && t < __ldg(a.len + b))
            val = __ldg(a.dz + r * a.Cout + co);
          v[e] = val;
          ++r;
          if (++t == a.L_pad) { t = 0; ++b; }
        }
        uint4 hi, lo;
        split8_bf16(v, hi, lo);
        *reinterpret_cast<uint4*>(st + sw64(c, 16 * g)) = hi;
        *reinterpret_cast<uint4*>(st + kWgAPlane + sw64(c, 16 * g)) = lo;
      } else {
        // B_j = X at t * stride + j - pad: row c = input channel ci0 + c (ci == Cin: 1 on valid output rows), K = the
        // chunk's output rows
        const int ci = ci0 + c, sh = j - a.pad;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float val = 0.f;
          if (r < a.rows && ci <= a.Cin) {
            if (ci == a.Cin) {
              if (t < __ldg(a.len + b)) val = 1.f;
            } else {
              const int ts = t * a.stride + sh;
              if (ts >= 0 && ts < __ldg(a.len_in + b))
                val = __ldg(a.x + (static_cast<int64_t>(b) * a.Lin_pad + ts) * a.Cin + ci);
            }
          }
          v[e] = val;
          ++r;
          if (++t == a.L_pad) { t = 0; ++b; }
        }
        uint4 hi, lo;
        split8_bf16(v, hi, lo);
        unsigned char* bt = st + 2 * kWgAPlane + static_cast<uint32_t>(j) * 2u * b_plane;
        *reinterpret_cast<uint4*>(bt + sw64(c, 16 * g)) = hi;
        *reinterpret_cast<uint4*>(bt + b_plane + sw64(c, 16 * g)) = lo;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t sa = smem_u32(st);
      for (int j = 0; j < a.K; ++j) {
        const uint32_t sb = sa + 2 * kWgAPlane + static_cast<uint32_t>(j) * 2u * b_plane;
        const uint32_t d = tmem_base + static_cast<uint32_t>(j * a.n);
#pragma unroll
        for (int k = 0; k < 2; ++k) {              // two K = 16 steps of 32 bytes in the 64-byte row
          const uint64_t ah = wg_desc(sa) + 2 * k, al = wg_desc(sa + kWgAPlane) + 2 * k;
          const uint64_t bh = wg_desc(sb) + 2 * k, bl = wg_desc(sb + b_plane) + 2 * k;
          umma_f16(d, ah, bh, idesc, (it == 0 && k == 0) ? 0u : 1u);
          umma_f16(d, ah, bl, idesc, 1u);
          umma_f16(d, al, bh, idesc, 1u);
        }
      }
      umma_commit(&mma_done[slot]);
    }
    ++it;
  }
  if (it > 0) mbar_wait(&mma_done[(it - 1) & 1], static_cast<uint32_t>((it - 1) >> 1) & 1u);
  tc_fence_after();

  // epilogue: accumulator row = output channel, column j * n + c = (tap j, input channel ci0 + c)
  const int quad = warp & 3, half = warp >> 2;
  const int co = co0 + 32 * quad + lane;
  const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(32 * quad) << 16);
  for (int c16 = 16 * half; c16 < a.K * a.n; c16 += 32) {
    uint32_t v[16];
    tmem_ld_32x16(t_lane + c16, v);
    tmem_ld_wait();
    const int j = c16 / a.n, cn = c16 - j * a.n;
    if (co >= a.Cout) continue;
    float* dst = a.part + ((static_cast<int64_t>(s) * a.K + j) * Cin1) * a.Cout + co;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int ci = ci0 + cn + e;
      if (ci < Cin1) dst[static_cast<int64_t>(ci) * a.Cout] = it > 0 ? __uint_as_float(v[e]) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, a.tmem_cols);
  }
}

// dW[co][ci][j] = sum over splits s (in order) of part[s][j][ci][co]; db[co] the same over the ones channel of tap
// (K - 1) / 2 (the ones channel is the same in every tap); no db when db is NULL
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ dw, float* __restrict__ db, int S, int K,
                    int pad, int Cin, int Cout) {
  const int64_t n_w = static_cast<int64_t>(Cout) * Cin * K;
  const int64_t plane = static_cast<int64_t>(Cin + 1) * Cout;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < n_w + (db ? Cout : 0);
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int co, ci, j;
    if (idx < n_w) {
      co = static_cast<int>(idx / (static_cast<int64_t>(Cin) * K));
      const int rem = static_cast<int>(idx - static_cast<int64_t>(co) * Cin * K);
      ci = rem / K;
      j = rem - ci * K;
    } else {
      co = static_cast<int>(idx - n_w);
      ci = Cin;
      j = pad;
    }
    const float* p = part + (static_cast<int64_t>(j) * (Cin + 1) + ci) * Cout + co;
    float acc = 0.f;
    for (int s = 0; s < S; ++s) acc += p[static_cast<int64_t>(s) * K * plane];
    if (idx < n_w) dw[idx] = acc; else db[co] = acc;
  }
}

struct WgPlan {
  int n, n_tiles, m_tiles, S;
  int64_t chunks;
  uint32_t stage_bytes, tmem_cols;
};

// Tile and split of a shape: N = the input channels (+ the ones channel) spread evenly over as few tiles as the
// 512 TMEM columns allow for K accumulators (K <= 32); S splits of the output rows so that the tiles fill about one
// wave.
bool wg_plan(int B, int L_pad, int Cin, int Cout, int K, WgPlan& p) {
  if (B <= 0 || L_pad <= 0 || Cin <= 0 || Cout <= 0 || K <= 0) return false;
  const int n_max = std::min(256, (512 / K) / 16 * 16);
  if (n_max < 16) return false;
  const int cin1 = Cin + 1;
  p.n_tiles = (cin1 + n_max - 1) / n_max;
  p.n = ((cin1 + p.n_tiles - 1) / p.n_tiles + 15) / 16 * 16;
  p.m_tiles = (Cout + kWgM - 1) / kWgM;
  p.chunks = (static_cast<int64_t>(B) * L_pad + kWgRows - 1) / kWgRows;
  const int tiles = p.n_tiles * p.m_tiles;
  p.S = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(kWgTargetCtas / tiles, p.chunks)));
  p.stage_bytes = 2 * kWgAPlane + static_cast<uint32_t>(K) * 2u * static_cast<uint32_t>(p.n) * 64u;
  p.tmem_cols = 32;
  while (p.tmem_cols < static_cast<uint32_t>(K * p.n)) p.tmem_cols <<= 1;
  return true;
}

int grid_for(int64_t total) { return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, 148 * 16))); }

// ------------------------------------------------------------------ ReLU + MaxPool1d(2, 2) backward
// dz[b][t][c] = (t < len and t < 2 (len / 2) and t is the first maximum of its pair ? dp[b][t / 2][c] : 0) * (y > 0)
// (pool = 1); the same for the windows (t - 1, t) of MaxPool1d(2, 2, padding 1) (pool = 2); dz = (t < len ?
// dp[b][t][c] : 0) * (y > 0) (pool = 0)
__global__ void __launch_bounds__(256)
relu_pool_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dp, const int32_t* __restrict__ len,
                     float* __restrict__ dz, int B, int L_pad, int Lp_pad, int C, int pool) {
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const int64_t bt = idx / C;
    const int t = static_cast<int>(bt % L_pad);
    const int b = static_cast<int>(bt / L_pad);
    const int n = len[b];
    float g = 0.f;
    const float yv = (t < n) ? y[idx] : 0.f;
    if (pool == 2) {
      // MaxPool1d(2, 2, padding 1): window p is (in[2p - 1], in[2p]); t is the second of window t / 2 (t even) or the
      // first of window (t + 1) / 2 (t odd).  The padding is never chosen: a window with one row inside the read
      // takes that row.
      if (t < n) {
        const int p = (t + 1) >> 1, i0 = 2 * p - 1, i1 = 2 * p;
        bool second;
        if (i0 < 0) {
          second = true;
        } else if (i1 >= n) {
          second = false;
        } else {
          const float* yb = y + (static_cast<int64_t>(b) * L_pad) * C + c;
          const float y0 = yb[static_cast<int64_t>(i0) * C], y1 = yb[static_cast<int64_t>(i1) * C];
          second = y1 > y0 || y1 != y1;
        }
        if ((t == i1) == second) g = dp[(static_cast<int64_t>(b) * Lp_pad + p) * C + c];
      }
    } else if (pool) {
      if (t < (n / 2) * 2) {
        const int t0 = t & ~1;
        const float* yb = y + (static_cast<int64_t>(b) * L_pad) * C + c;
        const float y0 = yb[static_cast<int64_t>(t0) * C], y1 = yb[static_cast<int64_t>(t0 + 1) * C];
        // torch's max_pool1d takes the second only when it is larger or NaN: a tie goes to the first
        const bool first = !(y1 > y0 || y1 != y1);
        if ((t == t0) == first) g = dp[(static_cast<int64_t>(b) * Lp_pad + t / 2) * C + c];
      }
    } else if (t < n) {
      g = dp[idx];
    }
    dz[idx] = yv > 0.f ? g : 0.f;
  }
}

// ------------------------------------------------------------------ head: GAP + Linear + cross entropy
// One CTA per read, in float64: feat = mean of the valid rows, z = W feat + bias, loss = logsumexp(z) - z[y],
// dlogits = (softmax(z) - onehot(y)) / B_total (B_total = B, or a data-parallel replica's global batch), dh = (W^T dlogits)
// / len on the valid rows, 0 on the others.  A read with len 0 or a label outside [0, n_classes) gets a NaN loss and no
// gradient.
constexpr int kHeadMaxClasses = 32;
__global__ void __launch_bounds__(256)
head_ce_kernel(const float* __restrict__ h, const int32_t* __restrict__ len, const float* __restrict__ fc_w,
               const float* __restrict__ fc_b, const int64_t* __restrict__ labels, int B_total, int L_pad, int C,
               int n_classes, float* __restrict__ loss, float* __restrict__ logits, float* __restrict__ dlogits,
               float* __restrict__ feat, float* __restrict__ dh) {
  extern __shared__ double fs[];                    // [C] features, then [C] activation gradient
  __shared__ double z[kHeadMaxClasses], dz[kHeadMaxClasses];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = len[b];
  const int64_t y = labels[b];
  const bool ok = L > 0 && y >= 0 && y < n_classes;
  const float* hb = h + static_cast<int64_t>(b) * L_pad * C;
  for (int c = tid; c < C; c += blockDim.x) {
    double s = 0.0;
    for (int t = 0; t < L; ++t) s += static_cast<double>(hb[static_cast<int64_t>(t) * C + c]);
    fs[c] = L > 0 ? s / L : 0.0;
    feat[static_cast<int64_t>(b) * C + c] = static_cast<float>(fs[c]);
  }
  __syncthreads();
  for (int k = warp; k < n_classes; k += blockDim.x / 32) {
    double acc = 0.0;
    for (int c = lane; c < C; c += 32) acc += fs[c] * static_cast<double>(fc_w[static_cast<int64_t>(k) * C + c]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) z[k] = acc + fc_b[k];
  }
  __syncthreads();
  if (tid == 0) {
    double m = z[0];
    for (int k = 1; k < n_classes; ++k) m = fmax(m, z[k]);
    double se = 0.0;
    for (int k = 0; k < n_classes; ++k) se += exp(z[k] - m);
    const double lse = m + log(se);
    loss[b] = ok ? static_cast<float>(lse - z[y]) : nanf("");
    for (int k = 0; k < n_classes; ++k) {
      dz[k] = ok ? (exp(z[k] - lse) - (k == y ? 1.0 : 0.0)) / B_total : 0.0;
      logits[static_cast<int64_t>(b) * n_classes + k] = static_cast<float>(z[k]);
      dlogits[static_cast<int64_t>(b) * n_classes + k] = static_cast<float>(dz[k]);
    }
  }
  __syncthreads();
  double* gs = fs + C;
  for (int c = tid; c < C; c += blockDim.x) {
    double g = 0.0;
    for (int k = 0; k < n_classes; ++k) g += static_cast<double>(fc_w[static_cast<int64_t>(k) * C + c]) * dz[k];
    gs[c] = L > 0 ? g / L : 0.0;
  }
  __syncthreads();
  float* dhb = dh + static_cast<int64_t>(b) * L_pad * C;
  for (int64_t i = tid; i < static_cast<int64_t>(L_pad) * C; i += blockDim.x) {
    const int t = static_cast<int>(i / C), c = static_cast<int>(i - static_cast<int64_t>(t) * C);
    dhb[i] = t < L ? static_cast<float>(gs[c]) : 0.f;
  }
}

// dfc_w[k][c] = sum_b dlogits[b][k] feat[b][c], dfc_b[k] = sum_b dlogits[b][k] (b in order, float64), and the loss
// summed over the reads / B_total
__global__ void __launch_bounds__(256)
head_reduce_kernel(const float* __restrict__ loss, const float* __restrict__ dlogits, const float* __restrict__ feat,
                   int B, int B_total, int C, int n_classes, float* __restrict__ loss_mean, float* __restrict__ dfc_w,
                   float* __restrict__ dfc_b) {
  const int64_t n_w = static_cast<int64_t>(n_classes) * C;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx <= n_w + n_classes;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    double acc = 0.0;
    if (idx < n_w) {
      const int k = static_cast<int>(idx / C), c = static_cast<int>(idx - static_cast<int64_t>(k) * C);
      for (int b = 0; b < B; ++b)
        acc += static_cast<double>(dlogits[static_cast<int64_t>(b) * n_classes + k]) *
               static_cast<double>(feat[static_cast<int64_t>(b) * C + c]);
      dfc_w[idx] = static_cast<float>(acc);
    } else if (idx < n_w + n_classes) {
      const int k = static_cast<int>(idx - n_w);
      for (int b = 0; b < B; ++b) acc += static_cast<double>(dlogits[static_cast<int64_t>(b) * n_classes + k]);
      dfc_b[k] = static_cast<float>(acc);
    } else {
      for (int b = 0; b < B; ++b) acc += static_cast<double>(loss[b]);
      *loss_mean = static_cast<float>(acc / B_total);
    }
  }
}

}  // namespace
}  // namespace riser

using namespace riser;

namespace {

int wgrad_launch(const char* who, const float* dz, const float* x, const int32_t* len_out, const int32_t* len_in, int B,
                 int Lout_pad, int Lin_pad, int Cin, int Cout, int K, int stride, int pad, float* dw, float* db,
                 void* workspace, size_t workspace_bytes, riser_stream_t stream) {
  WgPlan p;
  RISER_REQUIRE(wg_plan(B, Lout_pad, Cin, Cout, K, p),
                "%s: unsupported shape (B %d, L_pad %d, Cin %d, Cout %d, K %d)", who, B, Lout_pad, Cin, Cout, K);
  RISER_REQUIRE(p.chunks < (static_cast<int64_t>(1) << 31), "%s: too many rows", who);
  const size_t need = static_cast<size_t>(p.S) * K * (Cin + 1) * static_cast<size_t>(Cout) * sizeof(float);
  if (workspace_bytes < need) return fail(RISER_ENOMEM, "%s: workspace %zu bytes < %zu", who, workspace_bytes, need);
  WgArgs a;
  a.dz = dz; a.x = x; a.len = len_out; a.len_in = len_in; a.part = static_cast<float*>(workspace);
  a.B = B; a.L_pad = Lout_pad; a.Cin = Cin; a.Cout = Cout; a.K = K; a.pad = pad;
  a.Lin_pad = Lin_pad; a.stride = stride;
  a.n = p.n; a.S = p.S; a.rows = static_cast<int64_t>(B) * Lout_pad; a.chunks = p.chunks;
  a.stage_bytes = p.stage_bytes; a.tmem_cols = p.tmem_cols;
  // CTAs that share an SM must fit their TMEM allocations in its 512 columns (an allocation that cannot be served
  // waits for a resident CTA to exit): ask for enough shared memory that no more are co-scheduled
  const size_t by_tmem = 512 / p.tmem_cols;
  const size_t smem = std::max<size_t>(1024 + 2 * static_cast<size_t>(p.stage_bytes), 227 * 1024 / (by_tmem + 1) + 1024);
  int dev = 0, max_smem = 0;
  RISER_CUDA_TRY(cudaGetDevice(&dev));
  RISER_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  RISER_REQUIRE(smem <= static_cast<size_t>(max_smem), "%s: %zu bytes of shared memory", who, smem);
  RISER_CUDA_TRY(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  wgrad_tc_kernel<<<dim3(p.m_tiles, p.n_tiles, p.S), kWgThreads, smem, as_stream(stream)>>>(a);
  RISER_CUDA_TRY(cudaGetLastError());
  const int64_t total = static_cast<int64_t>(Cout) * Cin * K + (db ? Cout : 0);
  wgrad_reduce_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(a.part, dw, db, p.S, K, (K - 1) / 2, Cin, Cout);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

}  // namespace

extern "C" size_t riser_conv1d_wgrad_ex_workspace_bytes(int B, int Lout_pad, int Cin, int Cout, int K) {
  WgPlan p;
  if (!wg_plan(B, Lout_pad, Cin, Cout, K, p)) return 0;
  return static_cast<size_t>(p.S) * K * (Cin + 1) * static_cast<size_t>(Cout) * sizeof(float);
}

extern "C" size_t riser_conv1d_wgrad_workspace_bytes(int B, int L_pad, int Cin, int Cout, int K) {
  return (K & 1) ? riser_conv1d_wgrad_ex_workspace_bytes(B, L_pad, Cin, Cout, K) : 0;
}

extern "C" int riser_conv1d_wgrad_cl(const float* dz, const float* x, const int32_t* len, int B, int L_pad, int Cin,
                                     int Cout, int K, float* dw, float* db, void* workspace, size_t workspace_bytes,
                                     riser_stream_t stream) {
  RISER_REQUIRE(dz && x && len && dw && db && workspace, "riser_conv1d_wgrad_cl: null pointer");
  RISER_REQUIRE((K & 1) == 1, "riser_conv1d_wgrad_cl: unsupported shape (K %d: odd K <= 31)", K);
  return wgrad_launch("riser_conv1d_wgrad_cl", dz, x, len, len, B, L_pad, L_pad, Cin, Cout, K, 1, (K - 1) / 2, dw, db,
                      workspace, workspace_bytes, stream);
}

extern "C" int riser_conv1d_wgrad_ex(const float* dz, const float* x, const int32_t* len_out, const int32_t* len_in,
                                     int B, int Lout_pad, int Lin_pad, int Cin, int Cout, int K, int stride, int pad,
                                     float* dw, float* db, void* workspace, size_t workspace_bytes,
                                     riser_stream_t stream) {
  RISER_REQUIRE(dz && x && len_out && len_in && dw && workspace, "riser_conv1d_wgrad_ex: null pointer");
  RISER_REQUIRE(Lin_pad > 0 && stride > 0 && pad >= 0 && K <= 32, "riser_conv1d_wgrad_ex: bad shape (Lin_pad %d, "
                "stride %d, pad %d, K %d <= 32)", Lin_pad, stride, pad, K);
  return wgrad_launch("riser_conv1d_wgrad_ex", dz, x, len_out, len_in, B, Lout_pad, Lin_pad, Cin, Cout, K, stride, pad,
                      dw, db, workspace, workspace_bytes, stream);
}

extern "C" int riser_relu_pool_bwd_cl(const float* y, const float* dp, const int32_t* len, float* dz, int B, int L_pad,
                                      int Lp_pad, int C, int pool, riser_stream_t stream) {
  RISER_REQUIRE(y && dp && len && dz, "riser_relu_pool_bwd_cl: null pointer");
  RISER_REQUIRE(pool >= 0 && pool <= 2, "riser_relu_pool_bwd_cl: pool %d (0, 1 or 2)", pool);
  RISER_REQUIRE(B >= 0 && L_pad > 0 && C > 0 &&
                    (pool == 2 ? Lp_pad >= L_pad / 2 + 1 : pool ? Lp_pad >= L_pad / 2 : Lp_pad == L_pad),
                "riser_relu_pool_bwd_cl: bad shape");
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  if (total == 0) return RISER_OK;
  relu_pool_bwd_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(y, dp, len, dz, B, L_pad, Lp_pad, C, pool);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_gap_linear_ce_bwd_ex(const float* h, const int32_t* len, const float* fc_w, const float* fc_b,
                                          const int64_t* labels, int B, int B_total, int L_pad, int C, int n_classes,
                                          float* loss, float* loss_mean, float* logits, float* dlogits, float* feat,
                                          float* dfc_w, float* dfc_b, float* dh, riser_stream_t stream) {
  RISER_REQUIRE(h && len && fc_w && fc_b && labels && loss && loss_mean && logits && dlogits && feat && dfc_w && dfc_b &&
                    dh, "riser_gap_linear_ce_bwd: null pointer");
  RISER_REQUIRE(B > 0 && B_total >= B && L_pad > 0 && C > 0 && n_classes >= 1 && n_classes <= kHeadMaxClasses,
                "riser_gap_linear_ce_bwd: bad shape (B %d <= B_total %d, n_classes %d <= %d)", B, B_total, n_classes,
                kHeadMaxClasses);
  const size_t smem = 2 * sizeof(double) * static_cast<size_t>(C);
  RISER_REQUIRE(smem <= 200 * 1024, "riser_gap_linear_ce_bwd: %d channels", C);
  if (smem > 48 * 1024)
    RISER_CUDA_TRY(cudaFuncSetAttribute(head_ce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  head_ce_kernel<<<B, 256, smem, as_stream(stream)>>>(h, len, fc_w, fc_b, labels, B_total, L_pad, C, n_classes, loss,
                                                      logits, dlogits, feat, dh);
  RISER_CUDA_TRY(cudaGetLastError());
  const int64_t total = static_cast<int64_t>(n_classes) * C + n_classes + 1;
  head_reduce_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(loss, dlogits, feat, B, B_total, C, n_classes,
                                                                     loss_mean, dfc_w, dfc_b);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_gap_linear_ce_bwd(const float* h, const int32_t* len, const float* fc_w, const float* fc_b,
                                       const int64_t* labels, int B, int L_pad, int C, int n_classes, float* loss,
                                       float* loss_mean, float* logits, float* dlogits, float* feat, float* dfc_w,
                                       float* dfc_b, float* dh, riser_stream_t stream) {
  return riser_gap_linear_ce_bwd_ex(h, len, fc_w, fc_b, labels, B, B, L_pad, C, n_classes, loss, loss_mean, logits,
                                    dlogits, feat, dfc_w, dfc_b, dh, stream);
}
