// ResNet variant on the tensor pipe (riser/nets/resnet.py:26-70; SURVEY.md 8 rows a12 / f-2).
//
// One kernel, two modes:
//   * single conv   Conv1d(k in {1, 3}, stride in {1, 2}, 'same'-style padding (k - 1) / 2) with the eval-mode
//                   BatchNorm folded into weights + bias on the host, optional residual tile added in the
//                   epilogue, optional ReLU.  (conv_block of resnet.py:26-37; the 1x1 / 3x3 / 1x1 convs of
//                   BottleneckBlock, resnet.py:60-70, and blocks whose weights do not fit shared memory fused.)
//   * fused BasicBlock (resnet.py:50-57 with ResidualBlock.forward, resnet.py:39-47):
//                   out = ReLU( conv2(ReLU(conv1_s(x))) + shortcut(x) ),  shortcut = identity or Conv1d(1, stride s)+BN.
//                   The intermediate activation never leaves the SM: conv1's accumulators are drained by a
//                   mid-epilogue (bias, ReLU, length mask, fp16 hi + lo split) straight into conv2's A operand in
//                   shared memory; the 1x1 shortcut convolution accumulates into conv2's accumulator (it is
//                   linear), an identity shortcut is added in fp32 in the final epilogue.
//
// Implicit GEMM on tcgen05: M = 128 consecutive output positions of ONE read, N = output channels (padded to 16),
// K = taps x input channels.  Operands are fp16 hi + lo planes (three passes hi*hi + lo*hi + hi*lo, fp32
// accumulation in TMEM: fp32-class results, the 1e-3 probability bar with room) in the K-major SWIZZLE_64B
// layout (32-channel K blocks, 64-byte rows).  The taps of a stride-1 convolution are row-shifted views of one
// staged tile (descriptor start address + tap * 64 bytes); a stride-2 convolution reads an even-row tile E and an
// odd-row tile O:  y[m] = w0 O[m-1] + w1 E[m] + w2 O[m].  Activations in HBM stay fp32 channel-last
// [B][L][Cp] (Cp = channels padded to 8) with per-read valid lengths, as in csrc/resnet.cu, so the stem, the
// stem max-pool and the head kernels are shared with the CUDA-core path.
//
// A CTA is eight warps working through the phases of an item together (convert input -> MMA -> mid-epilogue -> MMA ->
// epilogue); overlap comes from several CTAs per SM and from the input of the NEXT item, which one elected thread
// pulls into a raw fp32 staging ring with a 1-D bulk copy (the rows an item needs are contiguous in memory) while the
// current item is worked on.  An identity shortcut is read back from that staging buffer.  Weights are copied into
// shared memory once per CTA (persistent over items) from a host-packed image that already has the operand layout.
//
// Passes (precision mode P, include/riser_b200.h RISER_PREC_*): with a = a_hi + a_lo and W = W_hi + W_lo,
//   F16_X3  a_hi W_hi + a_lo W_hi + a_hi W_lo (the default of riser_res_tc).  When 2 N <= 256 the two terms that
//           share a_hi are ONE instruction -- B = [W_hi; W_lo] stacked, N doubled, the W_lo half landing in its own
//           accumulator columns, added by the epilogue -- so a tap and K step cost two MMAs instead of three (these
//           narrow MMAs are paced by their A-operand fetch, not by N).
//   F16_W2  a_hi W_hi + a_hi W_lo: one stacked MMA per tap and K step when 2 N <= 256, else two.
//   F16     a_hi W_hi.
//   F16_F8  a_hi W_hi (kind::f16) + one e4m3 row per K block against the e4m3 weight row (kind::f8f6f4, K = 32 per
//           instruction, two per K block): [e4m3(a 2^-3) x32 | e4m3((a - a_hi) 2^9) x32] . [e4m3(W_lo 2^3) x32 |
//           e4m3(W 2^-9) x32], the two correction terms of X3 with 3 mantissa bits each (csrc/convnet.cu's F16_F8).
// A tiles: hi fp16, plus (X3) the lo fp16 tile or (F8) the e4m3 tile in its place -- an e4m3 row of a 32-channel K
// block is 64 bytes like an fp16 row, so it keeps the SWIZZLE_64B layout and the same descriptors; F16 and W2 have
// no second A tile and need less shared memory.
#include "common.cuh"

#include <algorithm>

namespace riser {
namespace {

constexpr int kRtThreads = 256;      // two warps per TMEM lane quadrant: they split the 16-column chunks of the epilogues
constexpr uint32_t kRtTile = 136 * 64;      // one staged tile: up to 130 rows (+ slack) of 64 bytes = 32 fp16 channels

struct ResTcArgs {
  const float* in;          // [B][Lin_pad][cin_p] fp32
  const int32_t* len_in;    // [B]
  const int32_t* len_out;   // [B] valid output rows (after the stride; conv2 keeps the length)
  float* out;               // [B][Lout_pad][cout_p]
  const float* residual;    // identity shortcut / residual operand [B][Lout_pad][cout_p], or nullptr
  const uint4* w1;          // packed image: [tap][kb1][plane (1 for F16, else 2)][n1 rows][64 B]
  const uint4* w2;          // fused: [3][kb2][plane][n2][64 B]; nullptr = single conv mode
  const uint4* wsc;         // fused, shortcut conv: [1][kb1][plane][n2][64 B]; nullptr = none
  const float* bias1;       // [n1]
  const float* bias2;       // [n2] (conv2 bias + shortcut-conv bias)
  float inv_scale1, inv_scale2;
  int B, Lin_pad, Lout_pad;
  int cin_p, cmid_p, cout_p;     // channel counts padded to 8 (cmid_p: conv1's output in fused mode)
  int n1, n2;                    // MMA N of conv1 / conv2 (multiples of 16)
  int kb1, kb2;                  // 32-channel K blocks of conv1 / conv2
  int taps, stride;              // conv1: taps in {1, 3}, stride in {1, 2}
  int relu;                      // single conv mode: ReLU in the epilogue
  int tile_rows;                 // output rows per item: 128 (single) or 126 (fused)
  int tiles_per_read, n_items;
  // floor(2^40 / tiles_per_read) + 1: item / tiles_per_read = (item * magic) >> 40, exact while
  // item * tiles_per_read < 2^40 (n_items < 2^20 and tiles_per_read <= n_items); tiles_per_read = 1 included
  uint64_t tiles_magic;
  int d2_col;                    // TMEM column of conv2's accumulator
  int tmem_cols;                 // columns allocated (power of two >= 32)
  int cat1, cat2;                // conv1 / conv2: [W_hi; W_lo] stacked (accumulator = 2 n columns; W2 and X3 only)
  int raw_stages;                // raw fp32 input staging buffers (1 or 2)
  int raw_rows;                  // input rows an item stages
  uint32_t raw_bytes;            // bytes of one staging buffer
  int n_mma1, n_mma2;            // MMAs of conv1 / conv2 (+ shortcut conv): sizes of the replay lists
};

struct RtSmem {
  uint64_t bar;
  uint64_t raw_full[2];
  uint64_t w_full;
  uint32_t tmem_base;
};

// One MMA of an item: the operand descriptors never change from item to item (same shared-memory tiles), so the
// issuing thread builds the list once and replays it -- two 16-byte loads and the instruction per MMA instead of
// the loop nest with its descriptor arithmetic (a single thread issues them all: its instruction count is what
// paces these short MMAs).
struct alignas(16) RtMma {
  uint64_t da, db;
  uint32_t idesc, d_col, acc, f8;      // f8: kind::f8f6f4 (the e4m3 pass of F16_F8), else kind::f16
};

constexpr int kPrecF16 = RISER_PREC_F16, kPrecW2 = RISER_PREC_F16_W2, kPrecX3 = RISER_PREC_F16_X3,
              kPrecF8 = RISER_PREC_F16_F8;
// A operand tiles per K block (hi, + lo or the e4m3 row) and weight planes per (tap, K block) of a mode
__host__ __device__ constexpr int a_planes(int p) { return (p == kPrecX3 || p == kPrecF8) ? 2 : 1; }
__host__ __device__ constexpr int w_planes(int p) { return p == kPrecF16 ? 1 : 2; }
// the accumulator of a conv holds [a W_hi | a W_lo] side by side (the stacked B operand)
__host__ __device__ constexpr bool cat_of(int p, int n) { return (p == kPrecX3 || p == kPrecW2) && 2 * n <= 256; }

// F16_F8 row scales, the powers of two of riser_b200/model.py F8_A_SHIFT / F8_LO_SHIFT (as csrc/convnet.cu):
// a8 = e4m3(a 2^-3) pairs with the W_lo 2^3 weight row, lo8 = e4m3((a - a_hi) 2^9) with the W 2^-9 row.
// e4m3(a 2^-3) saturates at |a| = 3584.
constexpr float kRtF8AScale = 1.f / 8.f;
constexpr float kRtF8LoScale = 512.f;

// fp32 x 8 -> fp16 hi (8 halfs = one 16-byte chunk) and lo = fp16(v - hi)
__device__ __forceinline__ void split8(const float (&v)[8], uint4& hi, uint4& lo) {
  __half2 h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    h[j] = __hmin2(__hmax2(__floats2half2_rn(v[2 * j], v[2 * j + 1]), __floats2half2_rn(-65504.f, -65504.f)),
                   __floats2half2_rn(65504.f, 65504.f));
    const float2 back = __half22float2(h[j]);
    l[j] = __floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
  }
  hi = *reinterpret_cast<const uint4*>(h);
  lo = *reinterpret_cast<const uint4*>(l);
}

// fp32 x 8 -> fp16 hi only (F16, W2)
__device__ __forceinline__ uint4 half8(const float (&v)[8]) {
  __half2 h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    h[j] = __hmin2(__hmax2(__floats2half2_rn(v[2 * j], v[2 * j + 1]), __floats2half2_rn(-65504.f, -65504.f)),
                   __floats2half2_rn(65504.f, 65504.f));
  return *reinterpret_cast<const uint4*>(h);
}

// fp32 x 8 -> fp16 hi, a8 = e4m3(v 2^-3) and lo8 = e4m3((v - hi) 2^9) (8 bytes each; F16_F8)
__device__ __forceinline__ void split8_f8(const float (&v)[8], uint4& hi, uint2& a8, uint2& lo8) {
  hi = half8(v);
  const __half2* h = reinterpret_cast<const __half2*>(&hi);
  uint32_t pa[2], pl[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint32_t wa[2], wl[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int c = 4 * j + 2 * e;
      const float2 back = __half22float2(h[c / 2]);
      wa[e] = __nv_cvt_float2_to_fp8x2(make_float2(v[c] * kRtF8AScale, v[c + 1] * kRtF8AScale), __NV_SATFINITE,
                                       __NV_E4M3);
      wl[e] = __nv_cvt_float2_to_fp8x2(make_float2((v[c] - back.x) * kRtF8LoScale, (v[c + 1] - back.y) * kRtF8LoScale),
                                       __NV_SATFINITE, __NV_E4M3);
    }
    pa[j] = wa[0] | (wa[1] << 16);
    pl[j] = wl[0] | (wl[1] << 16);
  }
  a8 = make_uint2(pa[0], pa[1]);
  lo8 = make_uint2(pl[0], pl[1]);
}

// Byte offset of (row r, byte) in a SWIZZLE_64B tile: 16-byte chunk c of a row lands at c ^ ((r >> 1) & 3)
__device__ __forceinline__ uint32_t sw64(int r, int byte) {
  return static_cast<uint32_t>(r * 64 + ((((byte >> 4) ^ (r >> 1)) & 3) << 4) + (byte & 15));
}

// The operand tiles of 8 channels (group g, K block g >> 2) of row r in the mode's format: hi at `hi_tile`, and the
// lo fp16 (X3) or the a8 / lo8 bytes (F8) at the same place in the tile `lo_off` bytes further
template <int P>
__device__ __forceinline__ void store_act8(unsigned char* hi_tile, uint32_t lo_off, int g, int r, const float (&v)[8]) {
  unsigned char* t = hi_tile + (g >> 2) * kRtTile;
  if (P == kPrecX3) {
    uint4 hi, lo;
    split8(v, hi, lo);
    *reinterpret_cast<uint4*>(t + sw64(r, 16 * (g & 3))) = hi;
    *reinterpret_cast<uint4*>(t + lo_off + sw64(r, 16 * (g & 3))) = lo;
  } else if (P == kPrecF8) {
    uint4 hi;
    uint2 a8, lo8;
    split8_f8(v, hi, a8, lo8);
    *reinterpret_cast<uint4*>(t + sw64(r, 16 * (g & 3))) = hi;
    *reinterpret_cast<uint2*>(t + lo_off + sw64(r, 8 * (g & 3))) = a8;          // e4m3 row bytes [0, 32): a8
    *reinterpret_cast<uint2*>(t + lo_off + sw64(r, 32 + 8 * (g & 3))) = lo8;    // bytes [32, 64): lo8
  } else {
    *reinterpret_cast<uint4*>(t + sw64(r, 16 * (g & 3))) = half8(v);
  }
}

__device__ __forceinline__ uint64_t rt_desc(uint32_t addr) {      // K-major SWIZZLE_64B, 8-row atoms of 512 B
  constexpr uint64_t kHi = (static_cast<uint64_t>(1) << 16) | (static_cast<uint64_t>(512 >> 4) << 32) |
                           (static_cast<uint64_t>(1) << 46) | (static_cast<uint64_t>(4) << 61);
  return kHi | static_cast<uint64_t>(addr >> 4);
}

// weight image: [tap][K block][plane][n rows][64 B] -- for a (tap, K block) the hi rows are followed by the lo rows
// (W2, X3: the stacked operand [W_hi; W_lo] is one contiguous 2n-row tile) or the e4m3 rows (F8); F16 has hi only
template <int P>
__device__ __forceinline__ uint32_t w_tile(uint32_t base, int tap, int kb, int n_kb, int n) {
  return base + static_cast<uint32_t>((tap * n_kb + kb) * w_planes(P) * n * 64);
}

// The MMAs of one term  D += A(view) * W(tap)  over the K blocks, appended to a replay list.  X3: a_hi x [W_hi; W_lo] +
// a_lo x W_hi (cat), or the three products one by one; W2: a_hi x [W_hi; W_lo] (cat) or its two products; F16:
// a_hi x W_hi; F8: a_hi x W_hi per K step, then the two e4m3 steps of the K block.  a_hi / a_lo: shared-memory
// addresses of the hi / second A tiles of K block 0 (consecutive K blocks kRtTile apart), already shifted to the
// view's first row.
template <int P>
__device__ __forceinline__ int list_term(RtMma* list, int n_list, uint32_t d_col, uint32_t a_hi, uint32_t a_lo,
                                         uint32_t w_base, int tap, int n_kb, int k_ch, int n, bool cat,
                                         uint32_t idesc_n, uint32_t idesc_2n) {
  for (int kb = 0; kb < n_kb; ++kb) {
    const int nk = min(2, (k_ch - 32 * kb + 15) >> 4);
    const uint32_t wt = w_tile<P>(w_base, tap, kb, n_kb, n);
    for (int k = 0; k < nk; ++k) {
      const uint64_t ah = rt_desc(a_hi + kb * kRtTile) + 2 * k, al = rt_desc(a_lo + kb * kRtTile) + 2 * k;
      const uint64_t wh = rt_desc(wt) + 2 * k, wl = rt_desc(wt + n * 64) + 2 * k;
      const uint32_t acc = n_list ? 1u : 0u;
      if (P == kPrecX3) {
        if (cat) {
          list[n_list++] = RtMma{ah, wh, idesc_2n, d_col, acc, 0u};   // columns [0, n): a_hi W_hi, [n, 2n): a_hi W_lo
          list[n_list++] = RtMma{al, wh, idesc_n, d_col, 1u, 0u};     // columns [0, n) += a_lo W_hi
        } else {
          list[n_list++] = RtMma{ah, wh, idesc_n, d_col, acc, 0u};
          list[n_list++] = RtMma{al, wh, idesc_n, d_col, 1u, 0u};
          list[n_list++] = RtMma{ah, wl, idesc_n, d_col, 1u, 0u};
        }
      } else if (P == kPrecW2) {
        if (cat) {
          list[n_list++] = RtMma{ah, wh, idesc_2n, d_col, acc, 0u};
        } else {
          list[n_list++] = RtMma{ah, wh, idesc_n, d_col, acc, 0u};
          list[n_list++] = RtMma{ah, wl, idesc_n, d_col, 1u, 0u};
        }
      } else {
        list[n_list++] = RtMma{ah, wh, idesc_n, d_col, acc, 0u};
      }
    }
    if (P == kPrecF8) {       // [a8 | lo8] x [W_lo 2^3 | W 2^-9]: 64 e4m3 per row = two K = 32 steps of 32 bytes
      const uint64_t a8 = rt_desc(a_lo + kb * kRtTile), w8 = rt_desc(wt + n * 64);
      for (int k = 0; k < 2; ++k) list[n_list++] = RtMma{a8 + 2 * k, w8 + 2 * k, idesc_n, d_col, 1u, 1u};
    }
  }
  return n_list;
}

// One thread replays the list: measured 1.009 ms against 1.045 ms for the same MMAs issued from a warp-uniform loop
// nest (512 x 12,048, basic).
template <int P>
__device__ __forceinline__ void replay(const RtMma* list, int n, uint32_t tmem_base) {
#pragma unroll 4
  for (int i = 0; i < n; ++i) {
    const RtMma e = list[i];
    if (P == kPrecF8 && e.f8)
      umma_f8(tmem_base + e.d_col, e.da, e.db, e.idesc, e.acc);
    else
      umma_f16(tmem_base + e.d_col, e.da, e.db, e.idesc, e.acc);
  }
}

template <int P>
__global__ void __launch_bounds__(kRtThreads)
res_tc_kernel(const ResTcArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const bool fused = a.w2 != nullptr;
  const int parts = a.stride == 2 ? 2 : 1;                       // staged input tiles per plane: X, or E and O
  constexpr uint32_t kWp = w_planes(P), kAp = a_planes(P);
  const uint32_t w1_bytes = kWp * a.taps * a.kb1 * a.n1 * 64u;
  const uint32_t w2_bytes = fused ? kWp * 3 * a.kb2 * a.n2 * 64u : 0u;
  const uint32_t wsc_bytes = a.wsc ? kWp * a.kb1 * a.n2 * 64u : 0u;
  const uint32_t a1_bytes = kAp * parts * a.kb1 * kRtTile;
  const uint32_t a2_bytes = fused ? kAp * a.kb2 * kRtTile : 0u;
  unsigned char* w1s = base;
  unsigned char* w2s = w1s + w1_bytes;
  unsigned char* wscs = w2s + w2_bytes;
  unsigned char* a1s = wscs + ((wsc_bytes + 511u) & ~511u);      // (images are multiples of 1024 B; keep 512-byte atoms aligned)
  unsigned char* a2s = a1s + a1_bytes;
  unsigned char* raws = a2s + a2_bytes;                          // raw fp32 input rows, raw_stages buffers
  float* bias1s = reinterpret_cast<float*>(raws + a.raw_stages * a.raw_bytes);
  float* bias2s = bias1s + a.n1;
  RtMma* list1 = reinterpret_cast<RtMma*>(bias2s + (fused ? a.n2 : 0));
  RtMma* list2 = list1 + a.n_mma1;
  RtSmem& s = *reinterpret_cast<RtSmem*>(list2 + a.n_mma2);

  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  if (tid == 0) {
    mbar_init(&s.bar, 1);
    mbar_init(&s.raw_full[0], 1);
    mbar_init(&s.raw_full[1], 1);
    mbar_init(&s.w_full, 1);
    fence_mbar_init();
    // weights (already in the operand layout): bulk copies, waited for before the first MMA
    mbar_arrive_expect_tx(&s.w_full, w1_bytes + w2_bytes + wsc_bytes);
    bulk_load_1d(w1s, a.w1, w1_bytes, &s.w_full);
    if (w2_bytes) bulk_load_1d(w2s, a.w2, w2_bytes, &s.w_full);
    if (wsc_bytes) bulk_load_1d(wscs, a.wsc, wsc_bytes, &s.w_full);
  }
  if (warp == 0) {
    tmem_alloc(&s.tmem_base, a.tmem_cols);
    tmem_relinquish();
  }
  // biases once per CTA; operand tiles zeroed once: channels beyond cin_p / cmid_p inside the last K block are never
  // written afterwards and must not hold NaN patterns
  for (uint32_t i = tid; i < (a1_bytes + a2_bytes) / 16; i += kRtThreads)
    reinterpret_cast<uint4*>(a1s)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < a.n1; i += kRtThreads) bias1s[i] = a.bias1[i];
  if (fused)
    for (int i = tid; i < a.n2; i += kRtThreads) bias2s[i] = a.bias2[i];
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  const uint32_t idesc1 = umma_idesc_f16(128, a.n1), idesc1c = umma_idesc_f16(128, 2 * a.n1);
  const uint32_t idesc2 = umma_idesc_f16(128, a.n2), idesc2c = umma_idesc_f16(128, 2 * a.n2);
  const uint32_t w1_addr = smem_u32(w1s), w2_addr = smem_u32(w2s), wsc_addr = smem_u32(wscs);
  const uint32_t a1_addr = smem_u32(a1s), a2_addr = smem_u32(a2s);
  const uint32_t a1_lo = parts * a.kb1 * kRtTile, a2_lo = a.kb2 * kRtTile;     // hi -> lo / e4m3 tile offsets (X3, F8)
  const int groups = a.cin_p >> 3;                               // 8-channel groups per input row
  const int pad = (a.taps - 1) >> 1;
  const int row_bytes = a.cin_p * 4;
  const int step_g = kRtThreads % groups, step_r = kRtThreads / groups;
  uint32_t phase = 0;
  if (tid == 0) {
    // conv1: D1[128 x n1] = sum over taps / K of A1(view) * W1
    int n = 0;
    for (int tap = 0; tap < a.taps; ++tap) {
      int part = 0, shift = tap;
      if (a.stride == 2) {
        if (a.taps == 1 || tap == 1) { part = 0; shift = 0; }           // E[m]  (w1 E[m])
        else { part = 1; shift = (tap == 2) ? 1 : 0; }                  // w0 O[m-1], w2 O[m]
      }
      const uint32_t av = a1_addr + part * a.kb1 * kRtTile + shift * 64;
      n = list_term<P>(list1, n, 0u, av, av + a1_lo, w1_addr, tap, a.kb1, a.cin_p, a.n1, a.cat1 != 0, idesc1, idesc1c);
    }
    if (fused) {
      // conv2 (+ 1x1 shortcut conv): D2[i] = sum_t W2_t A2[i + t]  (+ Wsc x[s (p0 + i)])
      n = 0;
      for (int tap = 0; tap < 3; ++tap) {
        const uint32_t av = a2_addr + tap * 64;
        n = list_term<P>(list2, n, a.d2_col, av, av + a2_lo, w2_addr, tap, a.kb2, a.cmid_p, a.n2, a.cat2 != 0, idesc2, idesc2c);
      }
      if (a.wsc) {
        // x[s (p0 + i)]: stride 1 -> X row i + 1 + pad; stride 2 -> E row i + 1
        const uint32_t av = a1_addr + ((a.stride == 2) ? 1 : 1 + pad) * 64;
        n = list_term<P>(list2, n, a.d2_col, av, av + a1_lo, wsc_addr, 0, a.kb1, a.cin_p, a.n2, a.cat2 != 0, idesc2, idesc2c);
      }
    }
    mbar_wait(&s.w_full, 0);                                     // the weight images have landed
  }
  __syncwarp();

  // item -> (read, first output row); an item whose rows all lie beyond its read's valid length is skipped
  auto decode = [&](int item, int& b, int& p0) {
    b = static_cast<int>((static_cast<uint64_t>(item) * a.tiles_magic) >> 40);     // item / tiles_per_read
    p0 = (item - b * a.tiles_per_read) * a.tile_rows;
  };
  auto next_active = [&](int item) {
    for (; item < a.n_items; item += gridDim.x) {
      int b, p0;
      decode(item, b, p0);
      if (p0 < __ldg(a.len_out + b)) break;
    }
    return item;
  };
  // first input position an item stages (raw row 0): stride 1: q0 - pad; stride 2: 2 q0 - 1   (q0 = first conv1 row)
  auto first_pos = [&](int p0) {
    const int q0 = fused ? p0 - 1 : p0;
    return a.stride == 2 ? 2 * q0 - 1 : q0 - pad;
  };
  // one elected thread: bulk copy of the valid part of an item's input rows (contiguous in memory) into a staging buffer
  auto prefetch = [&](int item, int slot) {
    int b, p0;
    decode(item, b, p0);
    const int lo = first_pos(p0), n_in = __ldg(a.len_in + b);
    const int lo_c = max(lo, 0), hi_c = min(lo + a.raw_rows, n_in);
    const uint32_t bytes = hi_c > lo_c ? static_cast<uint32_t>(hi_c - lo_c) * row_bytes : 0u;
    mbar_arrive_expect_tx(&s.raw_full[slot], bytes);
    if (bytes)
      bulk_load_1d(raws + slot * a.raw_bytes + static_cast<uint32_t>(lo_c - lo) * row_bytes,
                   a.in + (static_cast<int64_t>(b) * a.Lin_pad + lo_c) * a.cin_p, bytes, &s.raw_full[slot]);
  };

  int item = next_active(blockIdx.x);
  if (tid == 0 && item < a.n_items) prefetch(item, 0);
  for (int k = 0; item < a.n_items; ++k) {
    const int slot = (a.raw_stages == 2) ? (k & 1) : 0;
    const int nxt = next_active(item + gridDim.x);
    int b, p0;
    decode(item, b, p0);
    const int n_out = __ldg(a.len_out + b), n_in = __ldg(a.len_in + b);
    const int q0 = fused ? p0 - 1 : p0;                           // first row conv1 computes (fused: one halo row each side)
    const int pos0 = first_pos(p0);
    // two staging buffers: the next item's rows start to arrive now, while this item is worked on
    if (a.raw_stages == 2 && tid == 0 && nxt < a.n_items) prefetch(nxt, slot ^ 1);

    // ---------------- convert: raw fp32 rows -> the mode's A tiles (swizzled K-major)
    // stride 1: X row r = x[q0 - pad + r];  stride 2: E row r = x[2 (q0 + r)], O row r = x[2 (q0 - 1 + r) + 1]
    mbar_wait(&s.raw_full[slot], (a.raw_stages == 2) ? ((k >> 1) & 1) : (k & 1));
    const float* raw = reinterpret_cast<const float*>(raws + slot * a.raw_bytes);
    // unit u = (raw row rr, 8-channel group g), u = rr * groups + g; a thread's units are kRtThreads apart
    int g = tid % groups, rr = tid / groups;                      // raw row = input position pos0 + rr
    for (; rr < a.raw_rows; g += step_g, rr += step_r) {
      if (g >= groups) {
        g -= groups;
        ++rr;
        if (rr >= a.raw_rows) break;
      }
      const int pos = pos0 + rr;
      int part = 0, r = rr;
      if (a.stride == 2) {
        part = (rr & 1) ^ 1;                                      // pos0 is odd: raw rows alternate O, E, O, ...
        r = rr >> 1;
      }
      float v[8];
      if (pos >= 0 && pos < n_in) {
        const float4* src = reinterpret_cast<const float4*>(raw + rr * a.cin_p + 8 * g);
        const float4 v0 = src[0], v1 = src[1];
        v[0] = v0.x; v[1] = v0.y; v[2] = v0.z; v[3] = v0.w;
        v[4] = v1.x; v[5] = v1.y; v[6] = v1.z; v[7] = v1.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = 0.f;
      }
      store_act8<P>(a1s + part * a.kb1 * kRtTile, a1_lo, g, r, v);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    // one staging buffer: it is free again unless the epilogue reads the identity shortcut from it
    const bool res_from_raw = fused && a.residual && a.stride == 1 && !a.wsc;
    if (a.raw_stages == 1 && !res_from_raw && tid == 0 && nxt < a.n_items) prefetch(nxt, 0);

    // ---------------- conv1: D1[128 x n1] = sum over taps / K of A1(view) * W1
    if (tid == 0) {
      tc_fence_after();
      replay<P>(list1, a.n_mma1, tmem_base);
      umma_commit(&s.bar);
    }
    mbar_wait(&s.bar, phase);
    phase ^= 1;
    tc_fence_after();

    const int quad = warp & 3, half = warp >> 2;                   // TMEM lane quadrant; which chunks of it this warp takes
    const int row = 32 * quad + lane;                              // this thread's accumulator row (TMEM lane)
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(32 * quad) << 16);
    if (fused) {
      // ---------------- mid-epilogue: bias + ReLU + length mask -> conv2's A operand in the mode's format (row j =
      // mid row q0 + j)
      const int m = q0 + row;
      const bool live = (m >= 0 && m < n_out);
      for (int c16 = 16 * half; c16 < a.n1; c16 += 32) {
        uint32_t v[16], w[16];
        tmem_ld_32x16(t_lane + c16, v);
        if (a.cat1) tmem_ld_32x16(t_lane + a.n1 + c16, w);
        tmem_ld_wait();
#pragma unroll
        for (int h8 = 0; h8 < 2; ++h8) {
          const int c = c16 + 8 * h8;
          if (c >= a.cmid_p) continue;
          float r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float acc = __uint_as_float(v[8 * h8 + j]);
            if (a.cat1) acc += __uint_as_float(w[8 * h8 + j]);
            r[j] = live ? fmaxf(fmaf(acc, a.inv_scale1, bias1s[c + j]), 0.f) : 0.f;
          }
          store_act8<P>(a2s, a2_lo, c >> 3, row, r);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      __syncthreads();

      // ---------------- conv2 (+ 1x1 shortcut conv): D2[i] = sum_t W2_t A2[i + t]  (+ Wsc x[s (p0 + i)])
      if (tid == 0) {
        tc_fence_after();
        replay<P>(list2, a.n_mma2, tmem_base);
        umma_commit(&s.bar);
      }
      mbar_wait(&s.bar, phase);
      phase ^= 1;
      tc_fence_after();
    }

    // ---------------- epilogue: bias (+ residual) (+ ReLU) -> fp32 rows of the output
    {
      const int p = p0 + row;
      const bool ok = row < a.tile_rows && p < n_out;
      const int n = fused ? a.n2 : a.n1;
      const bool cat = fused ? (a.cat2 != 0) : (a.cat1 != 0);
      const float* bs = fused ? bias2s : bias1s;
      const float inv = fused ? a.inv_scale2 : a.inv_scale1;
      const bool do_relu = fused || a.relu;
      const uint32_t t_acc = t_lane + (fused ? a.d2_col : 0);
      float* orow = a.out + (static_cast<int64_t>(b) * a.Lout_pad + p) * a.cout_p;
      // residual row: from the staged input (identity shortcut of a fused stride-1 block: x[p0 + row] is raw row row + 2)
      // or from memory (single conv mode: the block's shortcut branch)
      const float* rrow = nullptr;
      if (a.residual)
        rrow = res_from_raw ? raw + (row + 1 + pad) * a.cin_p
                            : a.residual + (static_cast<int64_t>(b) * a.Lout_pad + p) * a.cout_p;
      for (int c16 = 16 * half; c16 < n; c16 += 32) {
        uint32_t v[16], w[16];
        tmem_ld_32x16(t_acc + c16, v);
        if (cat) tmem_ld_32x16(t_acc + n + c16, w);
        tmem_ld_wait();
        if (!ok) continue;
#pragma unroll
        for (int h8 = 0; h8 < 2; ++h8) {
          const int c = c16 + 8 * h8;
          if (c >= a.cout_p) continue;
          float r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float acc = __uint_as_float(v[8 * h8 + j]);
            if (cat) acc += __uint_as_float(w[8 * h8 + j]);
            r[j] = fmaf(acc, inv, bs[c + j]);
          }
          if (rrow) {
            const float4 r0 = *reinterpret_cast<const float4*>(rrow + c);
            const float4 r1 = *reinterpret_cast<const float4*>(rrow + c + 4);
            r[0] += r0.x; r[1] += r0.y; r[2] += r0.z; r[3] += r0.w;
            r[4] += r1.x; r[5] += r1.y; r[6] += r1.z; r[7] += r1.w;
          }
          if (do_relu) {
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = fmaxf(r[j], 0.f);
          }
          st_global_256(orow + c, make_uint4(__float_as_uint(r[0]), __float_as_uint(r[1]), __float_as_uint(r[2]), __float_as_uint(r[3])),
                        make_uint4(__float_as_uint(r[4]), __float_as_uint(r[5]), __float_as_uint(r[6]), __float_as_uint(r[7])));
        }
      }
    }
    // accumulators, operand tiles and (one staging buffer) the raw rows are free once every warp is past its loads
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (a.raw_stages == 1 && res_from_raw && tid == 0 && nxt < a.n_items) prefetch(nxt, 0);
    item = nxt;
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, a.tmem_cols);
  }
}

int pow2_at_least(int x) {
  int p = 32;
  while (p < x) p <<= 1;
  return p;
}

}  // namespace
}  // namespace riser

using namespace riser;

// Shared memory the kernel needs for a shape (0 = the shape is not supported: too wide for one MMA / TMEM budget).
namespace riser {
namespace {
int raw_rows_of(int taps, int stride) { return stride == 2 ? 258 : 128 + (taps - 1); }
// MMAs of `taps` terms over k_ch channels in mode p (list_term): per fp16 K step X3 two stacked / three, W2 one stacked /
// two, F16 one, F8 one; F8 adds two e4m3 steps per K block
int mma_count(int taps, int k_ch, int n, int p) {
  int steps = 0;
  const int kb = (k_ch + 31) / 32;
  for (int b = 0; b < kb; ++b) steps += std::min(2, (k_ch - 32 * b + 15) >> 4);
  const bool cat = cat_of(p, n);
  const int per = p == kPrecX3 ? (cat ? 2 : 3) : p == kPrecW2 ? (cat ? 1 : 2) : 1;
  return taps * (steps * per + (p == kPrecF8 ? 2 * kb : 0));
}
int acc_cols(int n, int p) { return ((cat_of(p, n) ? 2 * n : n) + 31) / 32 * 32; }
bool prec_ok(int p) { return p == kPrecF16 || p == kPrecW2 || p == kPrecX3 || p == kPrecF8; }
size_t raw_bytes_of(int cin_p, int taps, int stride) {
  return (static_cast<size_t>(raw_rows_of(taps, stride)) * cin_p * 4 + 127) & ~size_t(127);
}
}  // namespace
}  // namespace riser

// Shared memory the kernel needs for a shape with ONE raw staging buffer (0 = the shape or the mode is not supported).
// Modes without a second A tile (F16, W2) or without a weight lo plane (F16) need less.
extern "C" size_t riser_res_tc_smem_ex(int cin_p, int cmid_p, int n1, int n2, int taps, int stride, int fused,
                                       int shortcut_conv, int precision) {
  if (!prec_ok(precision)) return 0;
  if (cin_p <= 0 || (cin_p & 7) || n1 <= 0 || (n1 & 15) || n1 > 256 || (taps != 1 && taps != 3) ||
      (stride != 1 && stride != 2))
    return 0;
  if (fused && (cmid_p <= 0 || (cmid_p & 7) || n2 <= 0 || (n2 & 15) || n2 > 256 || taps != 3)) return 0;
  const int kb1 = (cin_p + 31) / 32, kb2 = fused ? (cmid_p + 31) / 32 : 0;
  const int parts = stride == 2 ? 2 : 1;
  const size_t wp = w_planes(precision), ap = a_planes(precision);
  size_t bytes = 1024 + wp * taps * kb1 * n1 * 64u + ap * parts * kb1 * kRtTile + raw_bytes_of(cin_p, taps, stride) +
                 sizeof(float) * n1 + sizeof(RtSmem) + 64 +
                 sizeof(RtMma) * (mma_count(taps, cin_p, n1, precision) +
                                  (fused ? mma_count(3, cmid_p, n2, precision) +
                                               (shortcut_conv ? mma_count(1, cin_p, n2, precision) : 0) : 0));
  if (fused) {
    bytes += wp * 3 * kb2 * n2 * 64u + ap * kb2 * kRtTile + sizeof(float) * n2;
    if (shortcut_conv) bytes += ((wp * kb1 * n2 * 64u) + 511u) & ~size_t(511);
    if (acc_cols(n1, precision) + acc_cols(n2, precision) > 512) return 0;
  }
  return bytes;
}

extern "C" size_t riser_res_tc_smem(int cin_p, int cmid_p, int n1, int n2, int taps, int stride, int fused,
                                    int shortcut_conv) {
  return riser_res_tc_smem_ex(cin_p, cmid_p, n1, n2, taps, stride, fused, shortcut_conv, RISER_PREC_F16_X3);
}

// Replaces one conv_block (+ optional residual) or one whole BasicBlock of riser/nets/resnet.py on the tensor
// pipe in the given precision mode; see the header for the argument conventions.
extern "C" int riser_res_tc_ex(const float* in, const int32_t* len_in, const int32_t* len_out, float* out,
                               const float* residual, const void* w1, const void* w2, const void* wsc,
                               const float* bias1, const float* bias2, float inv_scale1, float inv_scale2, int B,
                               int Lin_pad, int Lout_pad, int cin_p, int cmid_p, int cout_p, int n1, int n2, int taps,
                               int stride, int relu, riser_stream_t stream, int precision) {
  RISER_REQUIRE(prec_ok(precision), "riser_res_tc: unknown precision mode %d", precision);
  RISER_REQUIRE(in && len_in && len_out && out && w1 && bias1, "riser_res_tc: null pointer");
  RISER_REQUIRE(B > 0 && Lin_pad > 0 && Lout_pad > 0, "riser_res_tc: bad shape");
  const int fused = w2 != nullptr;
  RISER_REQUIRE(!fused || bias2, "riser_res_tc: fused mode needs bias2");
  RISER_REQUIRE(fused || !wsc, "riser_res_tc: a shortcut convolution needs the fused mode");
  RISER_REQUIRE(cout_p > 0 && (cout_p & 7) == 0 && cout_p <= (fused ? n2 : n1), "riser_res_tc: cout_p %d", cout_p);
  RISER_REQUIRE(((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) |
                  reinterpret_cast<uintptr_t>(residual)) & 31) == 0,
                "riser_res_tc: activation buffers must be 32-byte aligned");
  const size_t smem = riser_res_tc_smem_ex(cin_p, cmid_p, n1, n2, taps, stride, fused, wsc != nullptr, precision);
  RISER_REQUIRE(smem > 0, "riser_res_tc: unsupported shape (cin_p %d, n1 %d, n2 %d, taps %d, stride %d)", cin_p, n1,
                n2, taps, stride);
  int dev = 0, sms = 148, max_smem = 0;
  RISER_CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  RISER_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  RISER_REQUIRE(smem <= static_cast<size_t>(max_smem), "riser_res_tc: needs %zu bytes of shared memory (> %d)", smem,
                max_smem);
  ResTcArgs a;
  a.in = in; a.len_in = len_in; a.len_out = len_out; a.out = out; a.residual = residual;
  a.w1 = static_cast<const uint4*>(w1); a.w2 = static_cast<const uint4*>(w2); a.wsc = static_cast<const uint4*>(wsc);
  a.bias1 = bias1; a.bias2 = bias2; a.inv_scale1 = inv_scale1; a.inv_scale2 = inv_scale2;
  a.B = B; a.Lin_pad = Lin_pad; a.Lout_pad = Lout_pad;
  a.cin_p = cin_p; a.cmid_p = cmid_p; a.cout_p = cout_p; a.n1 = n1; a.n2 = fused ? n2 : 0;
  a.kb1 = (cin_p + 31) / 32; a.kb2 = fused ? (cmid_p + 31) / 32 : 0;
  a.taps = taps; a.stride = stride; a.relu = relu;
  a.tile_rows = fused ? 126 : 128;
  a.tiles_per_read = (Lout_pad + a.tile_rows - 1) / a.tile_rows;
  a.n_items = B * a.tiles_per_read;
  RISER_REQUIRE(a.n_items < (1 << 20), "riser_res_tc: %d work items (B x tiles per read) exceed 2^20", a.n_items);
  a.tiles_magic = (1ull << 40) / static_cast<uint64_t>(a.tiles_per_read) + 1ull;
  a.cat1 = cat_of(precision, n1) ? 1 : 0;
  a.cat2 = (fused && cat_of(precision, n2)) ? 1 : 0;
  a.d2_col = acc_cols(n1, precision);
  a.tmem_cols = pow2_at_least(a.d2_col + (fused ? acc_cols(n2, precision) : 0));
  a.n_mma1 = mma_count(taps, cin_p, n1, precision);
  a.n_mma2 = fused ? mma_count(3, cmid_p, n2, precision) + (wsc ? mma_count(1, cin_p, n2, precision) : 0) : 0;
  a.raw_rows = raw_rows_of(taps, stride);
  a.raw_bytes = static_cast<uint32_t>(raw_bytes_of(cin_p, taps, stride));
  // CTAs per SM: as many as shared memory allows, but their TMEM allocations must fit the 512 columns of an SM
  // (an allocation that cannot be served would wait for a resident CTA to exit); the dynamic shared-memory
  // request is raised where needed so that the hardware never co-schedules more
  const int by_tmem = 512 / a.tmem_cols;
  int ctas = std::max(1, std::min<int>(by_tmem, static_cast<int>((227 * 1024) / (smem + 1024))));
  ctas = std::min(ctas, 8);
  // a second staging buffer (the next item's rows arrive during the whole current item) when it costs no resident CTA
  a.raw_stages = (smem + a.raw_bytes <= static_cast<size_t>(max_smem) &&
                  static_cast<int>((227 * 1024) / (smem + a.raw_bytes + 1024)) >= ctas) ? 2 : 1;
  size_t request = smem + (a.raw_stages == 2 ? a.raw_bytes : 0);
  const size_t floor_for_cap = static_cast<size_t>(227 * 1024) / (ctas + 1) + 1;      // > 1/(ctas+1) of the SM's shared memory
  if (request < floor_for_cap) request = std::min<size_t>(floor_for_cap, max_smem);
  void (*kernel)(const ResTcArgs) = precision == kPrecF16 ? res_tc_kernel<kPrecF16>
                                    : precision == kPrecW2  ? res_tc_kernel<kPrecW2>
                                    : precision == kPrecF8  ? res_tc_kernel<kPrecF8>
                                                            : res_tc_kernel<kPrecX3>;
  RISER_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
  const int grid = std::min(a.n_items, sms * ctas);
  kernel<<<grid, kRtThreads, request, as_stream(stream)>>>(a);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_res_tc(const float* in, const int32_t* len_in, const int32_t* len_out, float* out,
                            const float* residual, const void* w1, const void* w2, const void* wsc,
                            const float* bias1, const float* bias2, float inv_scale1, float inv_scale2, int B,
                            int Lin_pad, int Lout_pad, int cin_p, int cmid_p, int cout_p, int n1, int n2, int taps,
                            int stride, int relu, riser_stream_t stream) {
  return riser_res_tc_ex(in, len_in, len_out, out, residual, w1, w2, wsc, bias1, bias2, inv_scale1, inv_scale2, B,
                         Lin_pad, Lout_pad, cin_p, cmid_p, cout_p, n1, n2, taps, stride, relu, stream,
                         RISER_PREC_F16_X3);
}
