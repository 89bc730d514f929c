// Network forward of the RISER hot path for sm_100a (riser/nets/cnn.py ConvNet as
// configured by riser/model/*.yaml, run by riser/model.py:22-28):
//
//   layer 0      Conv1d(1->C0,k3,same)+ReLU+MaxPool(2,2)   CUDA cores (K = 3, bandwidth bound)
//   layers 1..   Conv1d(Cin->Cout,k3,same)+ReLU+MaxPool    implicit GEMM on tcgen05 tensor
//                cores: M = flattened (read, position) rows, N = Cout, K = 3 taps x Cin.
//                Operands are fp16 tiles staged by TMA (SWIZZLE_128B), accumulators fp32 in
//                TMEM (double buffered), and bias + ReLU + max-pool + ragged-length mask are
//                a fused epilogue that writes the next layer's channel-last input.
//   head         masked global average pool / Linear(C,2) / softmax          CUDA cores
//   decide       control.py:75-82 decision codes
//
// Activation layout: layer i's input is act_i[B * Lp_i][Cp_i] fp16, channel-last, where
// read b owns rows [b*Lp_i, (b+1)*Lp_i), Lp_i even and > the longest valid length, and
// every row at or beyond a read's valid length is ZERO.  Because each read is followed by
// at least one zero row, the 'same' padding of the 3-tap convolution is obtained for free
// by loading the flat row range shifted by -1 / 0 / +1 (TMA zero-fills outside the buffer),
// and M tiles are plain 128-row slices of the flat buffer, independent of read boundaries.
#include "common.cuh"

#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

namespace riser {
namespace {

constexpr int kMaxLayers = 16;
constexpr int kBlockM = 128;          // rows per tile (UMMA M)
constexpr int kBlockK = 64;           // fp16 elements per K block = 128 bytes = one swizzle row
constexpr int kMaxNTile = 256;        // UMMA N limit
constexpr int kTmemCols = 512;        // two accumulator buffers of up to 256 columns
constexpr int kMinLen = 4096;         // riser/preprocess.py:8

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// N tile (multiple of 16, <= 256) that pads Cout the least; ties -> the larger tile.
int pick_n_tile(int cout) {
  const int c16 = round_up(cout, 16);
  if (c16 <= kMaxNTile) return c16;
  int best = 128, best_pad = round_up(cout, 128);
  for (int nt = 128; nt <= kMaxNTile; nt += 16) {
    const int p = round_up(cout, nt);
    if (p < best_pad || (p == best_pad && nt > best)) {
      best = nt;
      best_pad = p;
    }
  }
  return best;
}

struct LayerPack {
  int cin = 0, cout = 0, cin_p = 0, cout_p = 0, n_tile = 0, n_tiles = 0;
  __half* w = nullptr;    // [passes][3][cout_p][cin_p] fp16 (layers >= 1)
  uint8_t* w8 = nullptr;  // F16_F8 mode: [3][cout_p][2*cin_p] e4m3 = [W_lo * 2^3 | W * 2^-9] (correction pass)
  __half* wkc = nullptr;  // layer 1, F16_X3 terms concatenated along K: [3][cout_p][64] = [W_hi | W_hi | W_lo | 0] (fused01 MODE 4)
  float* w0 = nullptr;    // layer 0 only: fp32 [cout][3]
  float* bias = nullptr;  // fp32 [cout_p], zero padded
  int passes = 1;           // fp16 weight planes of this layer (hi [, lo])
  int f8 = 0;               // this layer's input rows are [hi | a8 | lo8] and its corrections run as one e4m3 pass
  float w_inv_scale = 1.f;  // weights are stored multiplied by a power of two (keeps the fp16 lo
                            // plane out of the subnormal range); the epilogue undoes it exactly
};

}  // namespace
}  // namespace riser

struct riser_model {
  int n_layers = 0;
  int precision = 0;
  int passes = 1;       // weight planes
  int act_planes = 1;   // activation planes (F16_F8: 2 = [hi fp16 | a8 e4m3 | lo8 e4m3], same bytes as hi + lo)
  int f8 = 0;           // RISER_PREC_F16_F8: layers >= f8_from take the e4m3 correction pass, earlier ones
                        // (epilogue-bound, not tensor-bound) keep the hi + lo fp16 planes of F16_X3
  int f8_from = 0;
  int device = 0;
  int sm_count = 148;
  riser::LayerPack layer[riser::kMaxLayers];
  float* fc_w = nullptr;   // [2][c_last]
  float* fc_b = nullptr;   // [2]
  int c_last = 0;
};

namespace riser {
namespace {

struct ConvArgs {
  const float* bias;
  const int32_t* len0;
  void* out;
  const uint8_t* flags;   // per M super-tile: 0 = every row pair lies beyond its read's valid length + 1 -> skip
  int rows_in, Lp_in, Lp_out, shift;
  int cin_p, cout_p, n_tile, n_tiles, k_blocks;
  int n_supers;           // M super-tiles of the batch (x n_tiles work items)
  int ms;                 // 128-row M sub-tiles per work item (they share every weight tile)
  int planes;             // activation planes read (1, or 2 = hi + lo)
  int wplanes;            // weight planes (1, or 2 = hi + lo)
  int out_planes, out_fp32;
  int a_stages, b_stages, acc_stages, resident;
  int epi_sets;           // epilogue warp sets (each = 4 warps covering the TMEM lane quadrants)
  int dual;               // conv_tc_kernel, MS == 2: one MMA-issuing thread PER SUB-TILE (warp 1 and the last warp)
  uint32_t nt_magic;      // conv_pair_kernel: floor(2^32 / n_tiles) + 1 -- item / n_tiles = umulhi(item, nt_magic) (items < 2^24); 0 = divide
  int acc_cols;           // TMEM columns per accumulator slot (n_tile rounded up to 32)
  int half_lp;            // Lp_in / 2
  int a_tx_bytes;         // bytes TMA delivers per A tile (box rows x row bytes)
  int k32;                // 1 = 32-channel K blocks: 64-byte rows, SWIZZLE_64B (else 64 / 128 B / SWIZZLE_128B)
  int kb16;               // K blocks of the fp16 pass (== k_blocks unless f8: then k_blocks - kb16 e4m3 blocks follow)
  int f8;                 // 1 = RISER_PREC_F16_F8: input rows are [hi fp16 | a8 | lo8], see riser_model_create
  int out_f8;             // output rows in that format
  int out_eo;             // output rows in the even / odd plane layout of conv_eo_kernel (else flat [B * Lp_out])
  int n_pairs_out, half_lp_out;
  // fused01_kernel (layers 0 + 1): layer 0 is computed in-kernel from the normalised signal
  const float* x;
  long long ld_x;
  const float* w0;        // layer-0 weights [cout0][3], bias [cout0]
  const float* b0;
  int cout0;
  unsigned long long pair_magic;   // floor(2^40 / half_lp) + 1: pair index -> read index
  uint32_t idesc;
  float w_inv_scale;
  int n_last;                // conv_pair_kernel: width of the LAST N tile (<= n_tile; the others are n_tile wide)
  uint32_t idesc_last;
};

// conv_eo2_kernel (two even / odd layers in one launch; see the kernel)
struct Eo2Args {
  const float* bias1;
  const float* bias2;
  const int32_t* len0;
  void* out;
  int B, n_seg;                 // items = B * n_seg (segment fastest)
  int half_lp_in;               // pairs per read in the first layer's input planes
  int Lp_out, half_lp_out, n_pairs_out, out_eo, out_f8, out_planes, cout_p2;
  int shift1, shift2;           // valid rows: len0 >> shift1 (intermediate), len0 >> shift2 (output)
  int cin_p1, n1, n2;           // first layer's padded input channels; N tiles (= padded Cout) of the two layers
  int kb1, kb2;                 // 32-channel K blocks
  int acc1, acc2;               // TMEM columns per accumulator: [even n | odd n] rounded to 32
  uint32_t idesc1_n, idesc1_2n, idesc2_n, idesc2_2n;
  float inv_scale1, inv_scale2;
};

typedef void (*ConvKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap,
                             const ConvArgs);
typedef void (*EoKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const ConvArgs);
typedef void (*PairKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap,
                             const CUtensorMap, const ConvArgs);
typedef void (*FusedKernelFn)(const CUtensorMap, const CUtensorMap, const ConvArgs);
typedef void (*Eo2KernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const Eo2Args);

// Which kernel runs a conv layer: the codes of riser_plan_layer_kernel (include/riser_b200.h)
enum LayerKind { kTcKernel = 0, kEoKernel = 1, kPairKernel = 2, kFused01Kernel = 3, kEo2Kernel = 5 };

struct ActivityLayer {
  int Lp_in, rows_in, rows_per_super, shift, n_supers, flag_off;
};
struct ActivityArgs {
  ActivityLayer layer[kMaxLayers];
  int n_layers, total;
};

struct LayerPlan {
  CUtensorMap tm_a, tm_b, tm_a8, tm_b8;   // (EO layers: tm_a = E plane, tm_a8 = O plane)
  CUtensorMap tm_bl, tm_b8l;              // conv_pair_kernel: weight maps whose box is half of the LAST N tile
  int eo = 0;                             // input in the even / odd plane layout -> conv_eo_kernel
  int fused_prev = 0;                     // computed inside the previous layer's launch: its input buffer is never written
  int kind = kTcKernel;                   // kEo2Kernel: this layer and the next one run as ONE conv_eo2_kernel launch
  int kc = 0;                             // kFused01Kernel: the K-concatenated operand (fused01_kernel<4>)
  union {                                 // the kernel of `kind` (unset when fused_prev)
    ConvKernelFn tc;
    EoKernelFn eo;
    PairKernelFn pair;
    FusedKernelFn fused01;
    Eo2KernelFn eo2;
  } fn = {nullptr};
  int grid = 0, block = 0;                // launch configuration of fn
  size_t smem = 0;
  ConvArgs args;                          // everything but len0, x, ld_x, which each forward fills in
  Eo2Args eo2;                            // kEo2Kernel: arguments of the two-layer launch (but len0)
  int rows_per_super = 0;   // flat input rows one work item covers (ms * 128; 510 for the fused layers 0+1)
};

}  // namespace
}  // namespace riser

struct riser_plan {
  const riser_model* model = nullptr;
  int B = 0, max_len = 0;
  int fuse_l0 = 0;                      // 1 = layers 0 + 1 run as one fused01_kernel launch
  uint8_t* flags = nullptr;             // tile activity flags (plan-owned), see tile_activity_kernel
  riser::ActivityArgs activity;
  int Lp[riser::kMaxLayers + 1];
  size_t act_off[riser::kMaxLayers + 1];
  char* ws = nullptr;
  riser::LayerPlan layer[riser::kMaxLayers];
};

namespace riser {
namespace {

// F16_F8 activation format: besides the fp16 value h = fp16(r), a row carries a8 = e4m3(r * 2^-3) (the operand of
// the W_lo * 2^3 correction) and lo8 = e4m3((r - h) * 2^9) (the operand of the W * 2^-9 correction).  The 2^-3
// (model.py F8_A_SHIFT) keeps a8 below e4m3's 448 for |r| < 3584 (unshifted it saturated above 448); lo8 stays exact
// in range to |r| = 2048.  A larger shift would push a8 of small activations into e4m3's subnormals (DESIGN.md 2).
constexpr float kF8AScale = 1.f / 8.f;
constexpr float kF8LoScale = 512.f;
template <int N>
__device__ __forceinline__ void store_f8_planes(const float (&r)[N], const __half2 (&h)[N / 2], uint8_t* a8,
                                                int lo_stride) {
  uint32_t pa[N / 4], pl[N / 4];
#pragma unroll
  for (int j = 0; j < N / 4; ++j) {
    uint32_t wa[2], wl[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int c = 4 * j + 2 * e;
      const float2 back = __half22float2(h[c / 2]);
      wa[e] = __nv_cvt_float2_to_fp8x2(make_float2(r[c] * kF8AScale, r[c + 1] * kF8AScale), __NV_SATFINITE,
                                       __NV_E4M3);
      wl[e] = __nv_cvt_float2_to_fp8x2(make_float2((r[c] - back.x) * kF8LoScale, (r[c + 1] - back.y) * kF8LoScale),
                                       __NV_SATFINITE, __NV_E4M3);
    }
    pa[j] = wa[0] | (wa[1] << 16);
    pl[j] = wl[0] | (wl[1] << 16);
  }
  if (N == 8) {
    *reinterpret_cast<uint2*>(a8) = make_uint2(pa[0], pa[1]);
    *reinterpret_cast<uint2*>(a8 + lo_stride) = make_uint2(pl[0], pl[1]);
  } else {
#pragma unroll
    for (int j = 0; j < N / 16; ++j) {
      *reinterpret_cast<uint4*>(a8 + 16 * j) = make_uint4(pa[4 * j], pa[4 * j + 1], pa[4 * j + 2], pa[4 * j + 3]);
      *reinterpret_cast<uint4*>(a8 + lo_stride + 16 * j) =
          make_uint4(pl[4 * j], pl[4 * j + 1], pl[4 * j + 2], pl[4 * j + 3]);
    }
  }
}

// ------------------------------------------------------------------------------------
// layer 0: x fp32 [B, ld_x] -> act_1 [B*Lp1][cout_p] fp16.  One thread per (output row,
// 8-channel group): consecutive lanes write consecutive 16-byte chunks (coalesced).
__global__ void __launch_bounds__(256)
layer0_kernel(const float* __restrict__ x, int64_t ld_x, const int32_t* __restrict__ len0,
              const float* __restrict__ w, const float* __restrict__ bias, __half* __restrict__ out,
              int B, int Lp1, int cout, int cout_p, int planes, int f8) {
  __shared__ float sw[64 * 3];
  __shared__ float sb[64];
  for (int i = threadIdx.x; i < cout_p * 3; i += blockDim.x) sw[i] = (i < cout * 3) ? w[i] : 0.f;
  for (int i = threadIdx.x; i < cout_p; i += blockDim.x) sb[i] = (i < cout) ? bias[i] : 0.f;
  __syncthreads();
  const uint32_t groups = cout_p >> 3;
  const uint32_t total = static_cast<uint32_t>(B) * Lp1 * groups;
  for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const uint32_t r = idx / groups;
    const int c8 = static_cast<int>(idx - r * groups);
    const int b = static_cast<int>(r / static_cast<uint32_t>(Lp1));
    const int tp = static_cast<int>(r - static_cast<uint32_t>(b) * Lp1);
    const int L = len0[b];
    uint4* o = reinterpret_cast<uint4*>(out + static_cast<int64_t>(r) * cout_p * planes) + c8;
    uint8_t* o8 = reinterpret_cast<uint8_t*>(out) + static_cast<int64_t>(r) * cout_p * 4 + 2 * cout_p + c8 * 8;
    if (tp >= (L >> 1)) {
      *o = make_uint4(0, 0, 0, 0);
      if (f8) {
        *reinterpret_cast<uint2*>(o8) = make_uint2(0, 0);
        *reinterpret_cast<uint2*>(o8 + cout_p) = make_uint2(0, 0);
      } else if (planes == 2) {
        o[groups] = make_uint4(0, 0, 0, 0);
      }
      continue;
    }
    const float* xr = x + static_cast<int64_t>(b) * ld_x;
    const int t = 2 * tp;
    const float xm1 = (t > 0) ? xr[t - 1] : 0.f;
    const float2 x01 = *reinterpret_cast<const float2*>(xr + t);
    const float x2 = (t + 2 < L) ? xr[t + 2] : 0.f;
    __half2 h[4], hl[4];
    float vv[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = c8 * 8 + 2 * j + e;
        const float w0 = sw[c * 3], w1 = sw[c * 3 + 1], w2 = sw[c * 3 + 2], bb = sb[c];
        const float y0 = fmaf(w2, x01.y, fmaf(w1, x01.x, fmaf(w0, xm1, bb)));
        const float y1 = fmaf(w2, x2, fmaf(w1, x01.y, fmaf(w0, x01.x, bb)));
        v[e] = fminf(fmaxf(fmaxf(y0, y1), 0.f), 65504.f);
      }
      h[j] = __floats2half2_rn(v[0], v[1]);
      const float2 back = __half22float2(h[j]);
      hl[j] = __floats2half2_rn(v[0] - back.x, v[1] - back.y);
      vv[2 * j] = v[0];
      vv[2 * j + 1] = v[1];
    }
    *o = *reinterpret_cast<uint4*>(h);
    if (f8) store_f8_planes<8>(vv, h, o8, cout_p);
    else if (planes == 2) o[groups] = *reinterpret_cast<uint4*>(hl);
  }
}

// ------------------------------------------------------------------------------------
// tcgen05 implicit-GEMM convolution with fused bias + ReLU + MaxPool(2,2) + length mask.
//
// Work item = (M super-tile of `ms` x 128 flat rows, N tile).  Per 64-channel K block the
// producer loads, for every sub-tile and activation plane, ONE 130-row A tile (the 128 rows
// plus a halo row on each side); the three taps read it through descriptors whose start
// address is shifted by 0 / 1 / 2 rows (the 128-byte swizzle is a function of the absolute
// shared-memory address, so a row shift keeps TMA's and the MMA's views consistent).
// Weight tiles are either resident in shared memory for the whole kernel (one N tile and
// all taps fit: the early layers) or streamed through their own ring, each loaded tile
// being used by every sub-tile and plane before it is released.
// Roles: warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2..9 = two epilogue
// sets (each covers the four TMEM lane quadrants; the sets split the 16-column chunks).
constexpr int kMaxAStages = 8, kMaxBStages = 8, kMaxAccStages = 4;
constexpr int kMaxEpiSets = 4;             // up to four sets (warps 2..17)

struct ConvSmem {
  uint64_t a_full[kMaxAStages], a_empty[kMaxAStages];
  uint64_t b_full[kMaxBStages], b_empty[kMaxBStages];
  uint64_t w_full;
  uint64_t tmem_full[kMaxAccStages];
  uint64_t tmem_full_ms[kMaxAccStages][4];   // conv_tc_kernel: "accumulator complete" per stage AND sub-tile
  uint64_t tmem_empty[kMaxAccStages][4];     // per accumulator stage AND sub-tile: released as soon as drained
  uint32_t tmem_base;
  alignas(16) float bias[2][kMaxNTile];
  float4 w0q[32];        // unused; its bytes still count in the plans' shared-memory budgets
};

// fp32 pair -> fp16 pair, saturated to the fp16 range (inf -> 65504) in the half2 domain
__device__ __forceinline__ __half2 sat_half2(float a, float b) {
  return __hmin2(__floats2half2_rn(a, b), __floats2half2_rn(65504.f, 65504.f));
}
// Epilogue for one chunk of 16 accumulator columns held one row per lane.  Rows (lanes) 2j
// and 2j+1 are the two positions of one max-pool pair; the even lane finishes and stores
// columns 0..7 of the chunk, the odd lane columns 8..15.
__device__ __forceinline__ void epilogue_chunk16(const uint32_t (&v)[16], const float* bias_s, int col0,
                                                 bool odd, bool valid, bool writable, void* out_row,
                                                 bool out_fp32, int lo_plane_off, float inv_scale,
                                                 uint8_t* f8_row = nullptr, int f8_stride = 0) {
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float mine = __uint_as_float(odd ? v[j + 8] : v[j]);
    const float send = __uint_as_float(odd ? v[j] : v[j + 8]);
    r[j] = fmaxf(mine, __shfl_xor_sync(0xffffffffu, send, 1));     // max-pool the row pair
  }
  if (!writable) return;
  const int c = col0 + (odd ? 8 : 0);
  if (valid) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias_s + c);
    const float4 b1 = *reinterpret_cast<const float4*>(bias_s + c + 4);
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = fmaxf(fmaf(r[j], inv_scale, bb[j]), 0.f);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = 0.f;
  }
  if (out_fp32) {
    float4* o = reinterpret_cast<float4*>(static_cast<float*>(out_row) + c);
    o[0] = make_float4(r[0], r[1], r[2], r[3]);
    o[1] = make_float4(r[4], r[5], r[6], r[7]);
  } else {
    __half* oh = static_cast<__half*>(out_row) + c;
    __half2 h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = sat_half2(r[2 * j], r[2 * j + 1]);
    *reinterpret_cast<uint4*>(oh) = *reinterpret_cast<const uint4*>(h);
    if (lo_plane_off) {   // residual plane: a = hi + lo, hi = fp16(a), lo = fp16(a - hi)
      __half2 l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 back = __half22float2(h[j]);
        l[j] = __floats2half2_rn(r[2 * j] - back.x, r[2 * j + 1] - back.y);
      }
      *reinterpret_cast<uint4*>(oh + lo_plane_off) = *reinterpret_cast<const uint4*>(l);
    }
    if (f8_row) store_f8_planes<8>(r, h, f8_row + c, f8_stride);
  }
}

// Epilogue for 16 output channels of ONE pooled row held by this lane: ve / vo are the accumulators of the
// even and the odd conv position (same TMEM lane).  max-pool, scale + bias, ReLU, then fp16 hi (+ lo plane,
// or the e4m3 pair of F16_F8) straight into the next layer's row.
__device__ __forceinline__ void epilogue_row16(const uint32_t (&ve)[16], const uint32_t (&vo)[16], const float* bias16,
                                               bool valid, float inv_scale, __half* ohi, int lo_off, uint8_t* f8,
                                               int f8_stride) {
  float r[16];
  if (valid) {
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4) {
      const float4 bb = *reinterpret_cast<const float4*>(bias16 + c4 * 4);
      const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = c4 * 4 + e;
        r[c] = fmaxf(fmaf(fmaxf(__uint_as_float(ve[c]), __uint_as_float(vo[c])), inv_scale, bv[e]), 0.f);
      }
    }
  } else {
#pragma unroll
    for (int c = 0; c < 16; ++c) r[c] = 0.f;
  }
  __half2 hv[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) hv[c] = sat_half2(r[2 * c], r[2 * c + 1]);
  st_global_256(ohi, *reinterpret_cast<const uint4*>(hv), *reinterpret_cast<const uint4*>(hv + 4));
  if (lo_off) {
    __half2 lv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float2 back = __half22float2(hv[c]);
      lv[c] = __floats2half2_rn(r[2 * c] - back.x, r[2 * c + 1] - back.y);
    }
    st_global_256(ohi + lo_off, *reinterpret_cast<const uint4*>(lv), *reinterpret_cast<const uint4*>(lv + 4));
  }
  if (f8) store_f8_planes<16>(r, hv, f8, f8_stride);
}

// Descriptor for a K-major swizzled tile at shared address `addr` (< 256 KB): rows of 128 bytes
// with SWIZZLE_128B (8-row atoms of 1024 B, layout type 2), or -- K32 -- rows of 64 bytes with
// SWIZZLE_64B (8-row atoms of 512 B, layout type 4).
template <bool K32>
__device__ __forceinline__ uint64_t sw_desc(uint32_t addr) {
  constexpr uint64_t kHi = (static_cast<uint64_t>(1) << 16) |
                           (static_cast<uint64_t>((K32 ? 512 : 1024) >> 4) << 32) |
                           (static_cast<uint64_t>(1) << 46) | (static_cast<uint64_t>(K32 ? 4 : 2) << 61);
  return kHi | static_cast<uint64_t>(addr >> 4);
}

// Work items are numbered with the N tile fastest; a CTA visits item, item + grid, ...
// Decoding is kept incremental (no division in the single-thread roles' loops).
struct ItemCursor {
  int super, n, step_super, step_n, n_tiles;
  __device__ __forceinline__ ItemCursor(int first, int grid, int n_tiles_) : n_tiles(n_tiles_) {
    super = first / n_tiles_;
    n = first % n_tiles_;
    step_super = grid / n_tiles_;
    step_n = grid % n_tiles_;
  }
  __device__ __forceinline__ void next() {
    super += step_super;
    n += step_n;
    if (n >= n_tiles) {
      n -= n_tiles;
      ++super;
    }
  }
  __device__ __forceinline__ int peek_super() const {   // super-tile of the following item
    return super + step_super + ((n + step_n >= n_tiles) ? 1 : 0);
  }
};

// Activity flag of the current item, with the next item's flag loaded one iteration ahead so
// that the single-thread roles never wait on it.
struct ItemFlags {
  const uint8_t* flags;
  uint32_t next_flag;
  __device__ __forceinline__ ItemFlags(const uint8_t* f, int first_super, bool any) : flags(f), next_flag(1) {
    if (flags && any) next_flag = __ldg(flags + first_super);
  }
  __device__ __forceinline__ bool take(const ItemCursor& cur, bool has_next) {
    const uint32_t now = next_flag;
    if (flags && has_next) next_flag = __ldg(flags + cur.peek_super());
    return now != 0;
  }
};

template <int MS, int PLANES, int WPLANES, bool RESIDENT, bool K32 = false, bool F8 = false>
__global__ void __launch_bounds__(96 + 128 * kMaxEpiSets, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
               const __grid_constant__ CUtensorMap tm_a8, const __grid_constant__ CUtensorMap tm_b8,
               const ConvArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  // 1024-byte alignment by OFFSET (not by casting through an integer): keeps the pointer in the
  // shared address space, so the compiler emits LDS/STS instead of generic LD/ST
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr int kATiles = MS * PLANES;                       // A tiles per K block
  constexpr int kRowBytes = K32 ? 64 : 128;                  // bytes per operand row (one K block)
  constexpr int kKElems = kRowBytes / 2;                     // fp16 elements per K block
  constexpr uint32_t kATile = 136 * kRowBytes;               // smem stride of one haloed A tile
  constexpr uint32_t kAGroupBytes = kATiles * kATile;
  const uint32_t b_bytes = a.n_tile * kRowBytes;
  unsigned char* a_ring = base;
  unsigned char* b_region = base + static_cast<size_t>(a.a_stages) * kAGroupBytes;
  const size_t b_region_bytes = RESIDENT ? static_cast<size_t>(WPLANES) * 3 * a.k_blocks * b_bytes
                                         : static_cast<size_t>(a.b_stages) * b_bytes;
  ConvSmem& s = *reinterpret_cast<ConvSmem*>(b_region + b_region_bytes);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const int n_items = a.n_supers * a.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    if (F8) {
      tma_prefetch_desc(&tm_a8);
      tma_prefetch_desc(&tm_b8);
    }
    const uint32_t n_issuers = a.dual ? 2 : 1;     // every issuer commits to the operand "empty" barriers
    for (int i = 0; i < a.a_stages; ++i) {
      mbar_init(&s.a_full[i], 1);
      mbar_init(&s.a_empty[i], n_issuers);
    }
    for (int i = 0; i < a.b_stages; ++i) {
      mbar_init(&s.b_full[i], 1);
      mbar_init(&s.b_empty[i], n_issuers);
    }
    mbar_init(&s.w_full, 1);
    for (int i = 0; i < a.acc_stages; ++i) {
      mbar_init(&s.tmem_full[i], 1);
      for (int ms = 0; ms < MS; ++ms) {
        mbar_init(&s.tmem_full_ms[i][ms], 1);
        mbar_init(&s.tmem_empty[i][ms], 4 * a.epi_sets);
      }
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&s.tmem_base, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      if (RESIDENT) {
        mbar_arrive_expect_tx(&s.w_full, static_cast<uint32_t>(b_region_bytes));
        for (int wp = 0; wp < WPLANES; ++wp)
          for (int tap = 0; tap < 3; ++tap)
            for (int kb = 0; kb < a.k_blocks; ++kb) {
              unsigned char* dst = b_region + static_cast<size_t>((wp * 3 + tap) * a.k_blocks + kb) * b_bytes;
              if (F8 && kb >= a.kb16)
                tma_load_2d(dst, &tm_b8, &s.w_full, (kb - a.kb16) * kRowBytes, tap * a.cout_p);
              else
                tma_load_2d(dst, &tm_b, &s.w_full, kb * kKElems, (wp * 3 + tap) * a.cout_p);
            }
      }
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      const uint32_t a_tx = kATiles * a.a_tx_bytes;
      ItemCursor cur(blockIdx.x, gridDim.x, a.n_tiles);
      ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
        if (!fl.take(cur, item + gridDim.x < n_items)) continue;
        const int m0 = cur.super * (MS * kBlockM) - 1;
        const int n0 = cur.n * a.n_tile;
        for (int kb = 0; kb < a.k_blocks; ++kb) {
          mbar_wait(&s.a_empty[sa], pa ^ 1);
          mbar_arrive_expect_tx(&s.a_full[sa], a_tx);
          unsigned char* dst = a_ring + static_cast<size_t>(sa) * kAGroupBytes;
#pragma unroll
          for (int ms = 0; ms < MS; ++ms)
#pragma unroll
            for (int ap = 0; ap < PLANES; ++ap) {
              if (F8 && kb >= a.kb16)   // e4m3 part of the row: bytes [2*cin_p, 4*cin_p)
                tma_load_2d(dst + (ms * PLANES + ap) * kATile, &tm_a8, &s.a_full[sa],
                            2 * a.cin_p + (kb - a.kb16) * kRowBytes, m0 + ms * kBlockM);
              else
                tma_load_2d(dst + (ms * PLANES + ap) * kATile, &tm_a, &s.a_full[sa],
                            ap * a.cin_p + kb * kKElems, m0 + ms * kBlockM);
            }
          if (++sa == a.a_stages) {
            sa = 0;
            pa ^= 1;
          }
          if (!RESIDENT) {
#pragma unroll
            for (int tap = 0; tap < 3; ++tap)
#pragma unroll
              for (int wp = 0; wp < WPLANES; ++wp) {
                mbar_wait(&s.b_empty[sb], pb ^ 1);
                mbar_arrive_expect_tx(&s.b_full[sb], b_bytes);
                if (F8 && kb >= a.kb16)
                  tma_load_2d(b_region + static_cast<size_t>(sb) * b_bytes, &tm_b8, &s.b_full[sb],
                              (kb - a.kb16) * kRowBytes, tap * a.cout_p + n0);
                else
                  tma_load_2d(b_region + static_cast<size_t>(sb) * b_bytes, &tm_b, &s.b_full[sb], kb * kKElems,
                              (wp * 3 + tap) * a.cout_p + n0);
                if (++sb == a.b_stages) {
                  sb = 0;
                  pb ^= 1;
                }
              }
          }
        }
      }
    }
  } else if (warp == 1 || (a.dual && warp == 2 + 4 * a.epi_sets)) {
    // ===================== MMA issuer(s) =====================
    // One thread issues every MMA of an item -- or, `dual` (MS == 2), one thread per sub-tile: the two walk the same
    // operand stages on their own (both commit to the "empty" barriers), so the thread whose accumulator is still
    // being drained falls a few weight tiles behind while the other keeps the tensor pipe busy -- with a single
    // accumulator stage (N > 128) both sub-tiles of an item used to finish together and the pipe idled for the
    // whole drain (profiles/README.md, round 2: 22 % of the issuing thread's time in layer 6) -- and the
    // instruction stream between two MMAs (~16 SASS instructions on one thread) is shared by two threads.
    const int ms_lo = a.dual ? (warp == 1 ? 0 : 1) : 0;
    const int ms_hi = a.dual ? ms_lo + 1 : MS;
    // the whole warp runs the loop (uniform registers); only the elected lane executes the MMAs / commits
    const uint32_t leader = elect_one() ? 1u : 0u;
    if (RESIDENT) {
      mbar_wait(&s.w_full, 0);
      tc_fence_after();
    }
    int sa = 0, sb = 0, stage = 0;
    uint32_t pa = 0, pb = 0, acc_phase = 0;
    const uint32_t a_ring_addr = smem_u32(a_ring), b_region_addr = smem_u32(b_region);
    const int nk_last = (a.cin_p - (a.kb16 - 1) * kKElems) / 16;
    const int nk_last8 = F8 ? (2 * a.cin_p - (a.k_blocks - a.kb16 - 1) * kRowBytes) / 32 : 0;
    const uint32_t acc_stride = MS * a.acc_cols;
    ItemCursor cur(blockIdx.x, gridDim.x, a.n_tiles);
    ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
      if (!fl.take(cur, item + gridDim.x < n_items)) continue;
      const uint32_t d_base = tmem_base + stage * acc_stride;
      for (int kb = 0; kb < a.k_blocks; ++kb) {
        const bool is8 = F8 && kb >= a.kb16;     // e4m3 correction blocks follow the fp16 blocks
        const int nk = is8 ? ((kb == a.k_blocks - 1) ? nk_last8 : (kKElems / 16))
                           : ((kb == a.kb16 - 1) ? nk_last : (kKElems / 16));
        mbar_wait(&s.a_full[sa], pa);
        tc_fence_after();
        const uint32_t a_addr = a_ring_addr + sa * kAGroupBytes;
#pragma unroll
        for (int tap = 0; tap < 3; ++tap) {
#pragma unroll
          for (int wp = 0; wp < WPLANES; ++wp) {
            uint32_t b_addr;
            if (RESIDENT) {
              b_addr = b_region_addr + ((wp * 3 + tap) * a.k_blocks + kb) * b_bytes;
            } else {
              mbar_wait(&s.b_full[sb], pb);
              tc_fence_after();
              b_addr = b_region_addr + sb * b_bytes;
            }
            const uint64_t db = sw_desc<K32>(b_addr);
#pragma unroll
            for (int ms = 0; ms < MS; ++ms) {
              if (ms < ms_lo || ms >= ms_hi) continue;      // (the other issuer's sub-tile)
              if (kb == 0 && tap == 0 && wp == 0) {   // first touch of this accumulator: wait until drained
                mbar_wait(&s.tmem_empty[stage][ms], acc_phase ^ 1);
                tc_fence_after();
              }
#pragma unroll
              for (int ap = 0; ap < (wp == 0 ? PLANES : 1); ++ap) {   // W_lo only meets the hi plane
                const uint64_t da = sw_desc<K32>(a_addr + (ms * PLANES + ap) * kATile + tap * kRowBytes);
                if (leader) {      // one elected lane issues; the K steps of a view in one go
#pragma unroll
                  for (int k = 0; k < kKElems / 16; ++k)
                    if (k < nk) {
                      if (is8)
                        umma_f8(d_base + ms * a.acc_cols, da + 2 * k, db + 2 * k, a.idesc, 1);
                      else
                        umma_f16(d_base + ms * a.acc_cols, da + 2 * k, db + 2 * k, a.idesc,
                                 (kb | tap | wp | ap | k) != 0);
                    }
                }
              }
            }
            if (!RESIDENT) {
              umma_commit_p(leader, &s.b_empty[sb]);
              if (++sb == a.b_stages) {
                sb = 0;
                pb ^= 1;
              }
            }
          }
        }
        umma_commit_p(leader, &s.a_empty[sa]);
        if (++sa == a.a_stages) {
          sa = 0;
          pa ^= 1;
        }
      }
#pragma unroll
      for (int ms = 0; ms < MS; ++ms)
        if (ms >= ms_lo && ms < ms_hi) umma_commit_p(leader, &s.tmem_full_ms[stage][ms]);
      if (++stage == a.acc_stages) {
        stage = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp < 2 + 4 * a.epi_sets) {
    // ===================== epilogue: warps 2..9 = two sets x four lane quadrants =====================
    const int q = warp & 3;
    const int eset = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;        // 0 .. 128 * epi_sets - 1
    const int epi_threads = 128 * a.epi_sets;
    const bool odd = lane & 1;
    const int row_elems = a.cout_p * a.out_planes;
    const int lo_off = (a.out_planes == 2 && !a.out_f8) ? a.cout_p : 0;
    const int n_chunks = a.n_tile >> 4;
    const bool single_n = (a.n_tiles == 1);
    if (single_n) {
      for (int i = et; i < a.n_tile; i += epi_threads) s.bias[0][i] = a.bias[i];
      asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
    }
    int stage = 0, it = -1;
    uint32_t acc_phase = 0;
    ItemCursor cur(blockIdx.x, gridDim.x, a.n_tiles);
    ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
      if (!fl.take(cur, item + gridDim.x < n_items)) continue;
      ++it;
      const int m0 = cur.super * (MS * kBlockM);
      const int n0 = cur.n * a.n_tile;
      const float* bias_s = s.bias[0];
      if (!single_n) {
        bias_s = s.bias[it & 1];
        for (int i = et; i < a.n_tile; i += epi_threads) s.bias[it & 1][i] = a.bias[n0 + i];
        asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
      }
      // row bookkeeping for every sub-tile (before the accumulator wait, to overlap the loads)
      bool valid[MS], writable[MS];
      int64_t out_row[MS];
#pragma unroll
      for (int ms = 0; ms < MS; ++ms) {
        valid[ms] = writable[ms] = false;
        out_row[ms] = 0;
        const int r_even = (m0 + ms * kBlockM + 32 * q + lane) & ~1;
        if (r_even < a.rows_in) {
          const uint32_t pidx = static_cast<uint32_t>(r_even) >> 1;
          const int b = static_cast<int>((static_cast<unsigned long long>(pidx) * a.pair_magic) >> 40);
          const int tp = static_cast<int>(pidx) - b * a.half_lp;
          valid[ms] = tp < (__ldg(a.len0 + b) >> a.shift);
          writable[ms] = tp < a.Lp_out;
          out_row[ms] = a.out_eo ? static_cast<int64_t>(tp & 1) * a.n_pairs_out + static_cast<int64_t>(b) * a.half_lp_out + (tp >> 1)
                                 : static_cast<int64_t>(b) * a.Lp_out + tp;
        }
      }
      // work units = (sub-tile, 16-column chunk), dealt round-robin to the epilogue sets
      int u = eset;
#pragma unroll
      for (int ms = 0; ms < MS; ++ms) {
        mbar_wait(&s.tmem_full_ms[stage][ms], acc_phase);      // this sub-tile's accumulator is complete
        tc_fence_after();
        void* orow = a.out_fp32
                         ? static_cast<void*>(static_cast<float*>(a.out) + out_row[ms] * row_elems + n0)
                         : static_cast<void*>(static_cast<__half*>(a.out) + out_row[ms] * row_elems + n0);
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) +
                                (stage * MS + ms) * a.acc_cols;
        for (; u < (ms + 1) * n_chunks; u += a.epi_sets) {
          const int c = u - ms * n_chunks;
          uint32_t v[16];
          tmem_ld_32x16(t_addr + c * 16, v);
          tmem_ld_wait();
          uint8_t* f8_row = nullptr;
          if (a.out_f8)
            f8_row = static_cast<uint8_t*>(a.out) + out_row[ms] * row_elems * 2 + 2 * a.cout_p + n0;
          epilogue_chunk16(v, bias_s, c * 16, odd, valid[ms], writable[ms], orow, a.out_fp32, lo_off,
                           a.w_inv_scale, f8_row, a.cout_p);
        }
        // this sub-tile's accumulator is drained: the MMA warp may start the next item on it
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s.tmem_empty[stage][ms]);
      }
      if (++stage == a.acc_stages) {
        stage = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <int MS, bool RESIDENT, bool K32>
ConvKernelFn pick_conv_planes(int planes, int wplanes) {
  if (planes == 1 && wplanes == 1) return conv_tc_kernel<MS, 1, 1, RESIDENT, K32>;
  if (planes == 1 && wplanes == 2) return conv_tc_kernel<MS, 1, 2, RESIDENT, K32>;
  return conv_tc_kernel<MS, 2, 2, RESIDENT, K32>;
}
template <bool K32>
ConvKernelFn pick_conv_k(int ms, int planes, int wplanes, int resident) {
  if (resident) {
    if (ms == 4) return pick_conv_planes<4, true, K32>(planes, wplanes);
    if (ms == 2) return pick_conv_planes<2, true, K32>(planes, wplanes);
    return pick_conv_planes<1, true, K32>(planes, wplanes);
  }
  if (ms == 4) return pick_conv_planes<4, false, K32>(planes, wplanes);
  if (ms == 2) return pick_conv_planes<2, false, K32>(planes, wplanes);
  return pick_conv_planes<1, false, K32>(planes, wplanes);
}
// F16_F8 mode: one activation / weight plane per K block, the e4m3 correction blocks after the fp16 ones
template <bool K32>
ConvKernelFn pick_conv_f8(int ms, int resident) {
  if (resident) {
    if (ms == 4) return conv_tc_kernel<4, 1, 1, true, K32, true>;
    if (ms == 2) return conv_tc_kernel<2, 1, 1, true, K32, true>;
    return conv_tc_kernel<1, 1, 1, true, K32, true>;
  }
  if (ms == 4) return conv_tc_kernel<4, 1, 1, false, K32, true>;
  if (ms == 2) return conv_tc_kernel<2, 1, 1, false, K32, true>;
  return conv_tc_kernel<1, 1, 1, false, K32, true>;
}
ConvKernelFn pick_conv_kernel(int ms, int planes, int wplanes, int resident, int k32, int f8) {
  if (f8) return k32 ? pick_conv_f8<true>(ms, resident) : pick_conv_f8<false>(ms, resident);
  return k32 ? pick_conv_k<true>(ms, planes, wplanes, resident) : pick_conv_k<false>(ms, planes, wplanes, resident);
}

// ------------------------------------------------------------------------------------
// Layers 0 + 1 in one launch, BOTH on the tensor pipe (the default; RISER_FUSE_L0=0 runs layer0_kernel instead).
//
// Layer 0 (Conv1d(1->C0,k3,same)+ReLU+MaxPool, nets/cnn.py:55-64) is a GEMM with K = 16:
// row p of its A operand is the signal window x[2p-1 .. 2p+2] split into fp16 hi and lo
// parts plus a constant-one column, and its B operand holds, for the conv position 2p
// (columns 0..23) and 2p+1 (columns 24..47), the taps as fp16 hi + lo and the bias:
//     k:  0..3  x_hi  * w_hi      4..7  x_lo * w_hi      8..11  x_hi * w_lo      12,13  1 * (b_hi, b_lo)
// (everything but the 2^-22 x_lo*w_lo term of the fp32 product).  The two positions of a
// max-pool pair therefore sit in ONE accumulator row (TMEM lane): pooling is an in-lane max.
//
// The same trick is applied to layer 1: its input rows are kept in shared memory as an
// "E" tile (even rows 2j) and an "O" tile (odd rows 2j+1), so that the conv at position 2j
//     w0*O[j-1] + w1*E[j] + w2*O[j]          and at 2j+1      w0*E[j] + w1*O[j] + w2*E[j+1]
// are row-shifted views of the two tiles accumulated into two column ranges of the same lane.
//
// Work item = 255 pooled layer-1 outputs (pair indices u0 .. u0+254; E rows 0..255 = E[u0+i],
// O rows 0..255 = O[u0+i-1]).  Roles (24 warps):
//   warp 0        producer: bulk copies (TMA) of the item's signal segment into a 4-stage ring
//   warps 2..7    cvt1: signal (shared memory) -> layer-0 A rows in shared memory
//   warp 1        MMA issuer (layer 0 of item k+1 is issued before layer 1 of item k)
//   warps 8..15   mid-epilogue: layer-0 accumulators -> max, ReLU, fp16 hi (+ lo) -> layer-1 A tiles
//   warps 16..23  epilogue: layer-1 accumulators -> max, bias, ReLU, mask -> act_2 in HBM
constexpr int kF2Pairs = 255;
// cvt1 warps: 257 rows in two passes (two warps were ~100 % busy; with four the issuer still waited on a0_full:
// 4 -> 6 -> 9 warps 1.04 / 1.01 / 1.00 ms on one box)
constexpr int kF2CvtWarps = 6;
constexpr int kF2Threads = 576 + 32 * kF2CvtWarps;     // producer + issuer + cvt1 + 8 mid-epilogue + 8 epilogue warps
constexpr uint32_t kF2A1Tile = 264 * 64;   // 256 rows + the slack row the shifted taps of row 255 touch
constexpr uint32_t kF2A0Tile = 256 * 64;   // per row: [E window (K=16) | O window (K=16)]
constexpr int kF2N0 = 48;
constexpr int kF2D0Col = 256;              // TMEM: layer-1 accumulators [0,256), layer-0 at 256 + 48*k
constexpr int kF2CvtThreads = 32 * kF2CvtWarps;
constexpr int kF2XStages = 4;
constexpr int kF2MaxLocalItems = 2048;   // work items per CTA whose activity flags fit the shared-memory copy
constexpr uint32_t kF2XStage = 260 * 16;     // pairs i = -2 .. 256 (4 samples each) + pad

struct F2Smem {
  uint64_t w_full;
  uint64_t x_full[kF2XStages], x_empty[kF2XStages];
  uint64_t a0_full[2], a0_empty[2];
  uint64_t d0_full[2], d0_empty[2];          // halves: 0 = E sub-tiles, 1 = O sub-tiles
  uint64_t a1_full[2], a1_empty[2];
  uint64_t d1_full[2], d1_empty[2][2];
  uint32_t tmem_base;
  alignas(16) float bias[32];
  uint8_t my_flags[kF2MaxLocalItems];     // activity flags of this CTA's items (item = blockIdx.x + i * gridDim.x)
};

// Active work items of this CTA in order.  The flags of the CTA's own items are staged in shared memory once
// (a global load per item would sit on the critical path of the single-thread roles).
struct F2Iter {
  const uint8_t* local;      // shared-memory copy, or nullptr = every item is active
  int i, item, n_items, step;
  __device__ __forceinline__ F2Iter(const uint8_t* l, int n) : local(l), i(0), item(blockIdx.x), n_items(n), step(gridDim.x) {}
  __device__ __forceinline__ int take() {
    while (item < n_items) {
      const int cur = item;
      const bool f = local ? (local[i] != 0) : true;
      item += step;
      ++i;
      if (f) return cur;
    }
    return -1;
  }
};

__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }

// MODE: 0 = F16, 1 = F16_W2 (weights hi + lo), 2 = F16_X3 (weights and activations hi + lo),
// 3 = F16_F8 (fp16 pass + e4m3 correction pass: second tile of a stage / second weight set are bytes),
// 4 = F16_X3 with the three terms CONCATENATED ALONG K ("KC"; layer 0 with <= 20 output channels): a layer-1 operand
//     row is [a_hi (20 ch) | a_lo (20) | a_hi (20) | 0 (4)] = 64 channels = one 128-byte SWIZZLE_128B row, the weight
//     row [W_hi | W_hi | W_lo | 0], so a tap costs 4 K steps instead of 3 x 2 (the 32-channel blocks of the plane
//     layout are 37 % zero padding); and E[j] x [w1; w0], O[j] x [w2; w1] feed both conv positions at once (N = 64).
//     The launch is bound by the tensor cores' operand reads from shared memory (81 % of that pipe's peak in the
//     plane layout, where an item was 76 MMAs of >= 45.5 cycles): 36 MMAs per item here.
template <int MODE>
__global__ void __launch_bounds__(kF2Threads, 1)
fused01_kernel(const __grid_constant__ CUtensorMap tm_b, const __grid_constant__ CUtensorMap tm_b8, const ConvArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr bool F8 = (MODE == 3);
  constexpr bool KC = (MODE == 4);
  constexpr int PLANES = (MODE >= 2) ? 2 : 1;
  constexpr int WPLANES = (MODE == 1 || MODE == 2) ? 2 : 1;
  constexpr uint32_t kW1Bytes = KC ? 3 * 32 * 128 : (F8 ? 2 : WPLANES) * 3 * 32 * 64;
  constexpr uint32_t kB0Bytes = kF2N0 * 64;
  constexpr uint32_t kA1Stage = PLANES * 2 * kF2A1Tile;
  unsigned char* w1 = base;
  unsigned char* b0 = w1 + kW1Bytes;
  unsigned char* a0_ring = b0 + kB0Bytes;                 // 2 stages
  unsigned char* a1_ring = a0_ring + 2 * kF2A0Tile;       // 2 stages x [plane][E, O]
  unsigned char* x_ring = a1_ring + 2 * kA1Stage;         // signal segments, kF2XStages stages
  F2Smem& s = *reinterpret_cast<F2Smem*>(x_ring + kF2XStages * kF2XStage);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const int n_items = a.n_supers;
  const int n_pairs = a.rows_in >> 1;
  const uint8_t* flags_l = a.flags ? s.my_flags : nullptr;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_b);
    mbar_init(&s.w_full, 1);
    for (int i = 0; i < kF2XStages; ++i) {
      mbar_init(&s.x_full[i], 1);
      mbar_init(&s.x_empty[i], kF2CvtThreads / 32);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.a0_full[i], kF2CvtThreads / 32);
      mbar_init(&s.a0_empty[i], 1);
      mbar_init(&s.d0_full[i], 1);
      mbar_init(&s.d0_empty[i], 4);
      mbar_init(&s.a1_full[i], 8);
      mbar_init(&s.a1_empty[i], 1);
      mbar_init(&s.d1_full[i], 1);
      mbar_init(&s.d1_empty[i][0], 4);
      mbar_init(&s.d1_empty[i][1], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&s.tmem_base, kTmemCols);
    tmem_relinquish();
  }
  // zero both operand rings once: padded channels / unused K columns are never written again
  for (uint32_t i = threadIdx.x; i < (2 * kF2A0Tile + 2 * kA1Stage + kF2XStages * kF2XStage) / 16; i += kF2Threads)
    reinterpret_cast<uint4*>(a0_ring)[i] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x < 32) s.bias[threadIdx.x] = a.bias[threadIdx.x];
  if (a.flags)
    for (int i = threadIdx.x, it = blockIdx.x + threadIdx.x * gridDim.x; it < n_items; i += kF2Threads, it += kF2Threads * gridDim.x)
      s.my_flags[i] = a.flags[it];
  if (threadIdx.x < kF2N0) {
    // layer-0 B operand, row n: channel n % 24 at conv position 2p + n / 24 (SWIZZLE_64B rows)
    const int n = threadIdx.x, c = n % 24, odd = n / 24;
    float w[3] = {0.f, 0.f, 0.f}, bb = 0.f;
    if (c < a.cout0) {
      w[0] = a.w0[c * 3];
      w[1] = a.w0[c * 3 + 1];
      w[2] = a.w0[c * 3 + 2];
      bb = a.b0[c];
    }
    __half kh[4], kl[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) kh[k] = kl[k] = __float2half_rn(0.f);
#pragma unroll
    for (int tap = 0; tap < 3; ++tap) {
      const __half h = __float2half_rn(w[tap]);
      kh[tap + odd] = h;
      kl[tap + odd] = __float2half_rn(w[tap] - __half2float(h));
    }
    const __half bh = __float2half_rn(bb), bl = __float2half_rn(bb - __half2float(bh));
    __half c0[8] = {kh[0], kh[1], kh[2], kh[3], kh[0], kh[1], kh[2], kh[3]};
    __half c1[8] = {kl[0], kl[1], kl[2], kl[3], bh, bl, __float2half_rn(0.f), __float2half_rn(0.f)};
    const int sw = (n >> 1) & 3;
    *reinterpret_cast<uint4*>(b0 + n * 64 + ((0 ^ sw) << 4)) = *reinterpret_cast<const uint4*>(c0);
    *reinterpret_cast<uint4*>(b0 + n * 64 + ((1 ^ sw) << 4)) = *reinterpret_cast<const uint4*>(c1);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    // ===================== producer: weights once, then the signal segment of every item =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(&s.w_full, kW1Bytes);
      // taps are stored in REVERSE order (slot 2 - tap): [w2; w1] and [w1; w0] are then contiguous 64-row B
      // operands, so one N = 64 MMA feeds the even and the odd conv position from the same A rows
      if (KC) {      // tm_b = the K-concatenated layer-1 weights [tap][32 rows][64 channels], 4 KB per tap
        for (int tap = 0; tap < 3; ++tap) tma_load_2d(w1 + (2 - tap) * 4096, &tm_b, &s.w_full, 0, tap * a.cout_p);
      } else {
        for (int wp = 0; wp < WPLANES; ++wp)
          for (int tap = 0; tap < 3; ++tap)
            tma_load_2d(w1 + (wp * 3 + 2 - tap) * 2048, &tm_b, &s.w_full, 0, (wp * 3 + tap) * a.cout_p);
      }
      if (F8)
        for (int tap = 0; tap < 3; ++tap)
          tma_load_2d(w1 + (3 + 2 - tap) * 2048, &tm_b8, &s.w_full, 0, tap * a.cout_p);
      // Stage slot of pair i (i = -2 .. 256) is 16*(i+2): its four samples x[4t .. 4t+3].  An item spans at
      // most two reads (a read has more pairs than an item); pairs with 4t >= ld_x are not loaded (they lie
      // beyond every valid length and are masked by cvt1).
      const int t_max = static_cast<int>(a.ld_x >> 2);        // pairs per read that exist in x
      F2Iter iter(flags_l, n_items);
      int k = 0;
      for (int item = iter.take(); item >= 0; item = iter.take(), ++k) {
        const int st = k % kF2XStages;
        mbar_wait(&s.x_empty[st], ((k / kF2XStages) & 1) ^ 1);
        unsigned char* dst = x_ring + st * kF2XStage;
        long long u_lo = static_cast<long long>(item) * kF2Pairs - 2;
        long long u_hi = u_lo + 258;                            // inclusive
        const int i_lo = (u_lo < 0) ? static_cast<int>(-u_lo) - 2 : -2;
        if (u_lo < 0) u_lo = 0;
        if (u_hi > n_pairs - 1) u_hi = n_pairs - 1;
        uint32_t bytes[2] = {0, 0};
        const float* src[2] = {nullptr, nullptr};
        int slot[2] = {0, 0};
        if (u_hi >= u_lo) {
          const int b = static_cast<int>((static_cast<unsigned long long>(static_cast<uint32_t>(u_lo)) * a.pair_magic) >> 40);
          const int t0 = static_cast<int>(u_lo) - b * a.half_lp;
          const int n_total = static_cast<int>(u_hi - u_lo) + 1;
          const int n_first = min(n_total, a.half_lp - t0);     // pairs that belong to read b
          const int n1 = max(0, min(n_first, t_max - t0));
          src[0] = a.x + static_cast<long long>(b) * a.ld_x + 4 * t0;
          slot[0] = i_lo + 2;
          bytes[0] = 16u * n1;
          const int n2 = max(0, min(n_total - n_first, t_max));
          src[1] = a.x + static_cast<long long>(b + 1) * a.ld_x;
          slot[1] = i_lo + 2 + n_first;
          bytes[1] = 16u * n2;
        }
        mbar_arrive_expect_tx(&s.x_full[st], bytes[0] + bytes[1]);
        if (bytes[0]) bulk_load_1d(dst + 16 * slot[0], src[0], bytes[0], &s.x_full[st]);
        if (bytes[1]) bulk_load_1d(dst + 16 * slot[1], src[1], bytes[1], &s.x_full[st]);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // (the whole warp runs the loop so that the descriptor arithmetic stays in uniform registers; the elected lane issues)
    const bool leader = elect_one();
    mbar_wait(&s.w_full, 0);
    tc_fence_after();
    const uint32_t w1_addr = smem_u32(w1), b0_addr = smem_u32(b0);
    const uint32_t a0_addr = smem_u32(a0_ring), a1_addr = smem_u32(a1_ring);
    const uint32_t idesc0 = umma_idesc_f16(kBlockM, kF2N0);
    const uint32_t idesc64 = umma_idesc_f16(kBlockM, 64);
    const uint64_t db0 = sw_desc<true>(b0_addr);
    F2Iter iter(flags_l, n_items);
    int k0 = 0;                       // items whose layer 0 has been issued
    auto issue_layer0 = [&]() {
      const int st = k0 & 1;
      mbar_wait(&s.a0_full[st], (k0 >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        mbar_wait(&s.d0_empty[h], (k0 & 1) ^ 1);
        tc_fence_after();
        if (leader) {
#pragma unroll
          for (int sub = 0; sub < 2; ++sub)
            umma_f16(tmem_base + kF2D0Col + (h * 2 + sub) * kF2N0,
                     sw_desc<true>(a0_addr + st * kF2A0Tile + sub * 128 * 64) + 2 * h, db0, idesc0, 0);
        }
        umma_commit_p(leader, &s.d0_full[h]);
      }
      umma_commit_p(leader, &s.a0_empty[st]);
      ++k0;
    };
    int cur = iter.take();
    if (cur >= 0) issue_layer0();
    int k1 = 0;                       // items whose layer 1 has been issued
    while (cur >= 0) {
      const int nxt = iter.take();
      if (nxt >= 0) issue_layer0();
      const int st = k1 & 1;
      mbar_wait(&s.a1_full[st], (k1 >> 1) & 1);
      tc_fence_after();
      const uint32_t a1s = a1_addr + st * kA1Stage;
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        mbar_wait(&s.d1_empty[st][sub], ((k1 >> 1) & 1) ^ 1);
        tc_fence_after();
      }
      // even position 2j: w0*O[j-1] + w1*E[j] + w2*O[j];  odd position 2j+1: w0*E[j] + w1*O[j] + w2*E[j+1]
      // (tile rows: E[j] = E row j, O[j] = O row j + 1; weight slot of tap t = 2 - t).
      // Consecutive MMAs go to DIFFERENT accumulators (sub-tile x parity, round-robin): back-to-back
      // MMAs into the same TMEM tile serialise on the accumulator (~80 cycles each at N = 32).
      auto issue_group = [&](uint32_t a_tiles, uint32_t w_set, bool f8, bool first) {
        if (!leader) return;
#pragma unroll
        for (int tap = 0; tap < 3; ++tap) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const uint64_t db = sw_desc<true>(w_set + (2 - tap) * 2048) + 2 * k;
#pragma unroll
            for (int sub = 0; sub < 2; ++sub) {
#pragma unroll
              for (int pe = 0; pe < 2; ++pe) {
                const int par = (pe == 0) ? ((tap == 1) ? 0 : 1) : ((tap == 1) ? 1 : 0);
                const int shift = (pe == 0) ? ((tap == 2) ? 1 : 0) : ((tap == 0) ? 0 : 1);
                const uint64_t da = sw_desc<true>(a_tiles + par * kF2A1Tile + (sub * 128 + shift) * 64) + 2 * k;
                const uint32_t d = tmem_base + st * 128 + (2 * sub + pe) * 32;
                if (f8) umma_f8(d, da, db, a.idesc, 1);
                else umma_f16(d, da, db, a.idesc, !(first && tap == 0 && k == 0));
              }
            }
          }
        }
      };
      if (KC) {
        // one 64-channel K block per tap set: 4 K steps x 4 MMAs per sub-tile (E tile at a1s, O tile behind it;
        // rows of 128 bytes; weight slots [w2; w1; w0] of 4 KB)
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t w21 = sw_desc<false>(w1_addr) + 2 * k;
            const uint64_t w10 = sw_desc<false>(w1_addr + 4096) + 2 * k;
            const uint64_t w0 = sw_desc<false>(w1_addr + 8192) + 2 * k;
#pragma unroll
            for (int sub = 0; sub < 2; ++sub) {
              const uint32_t e_rows = a1s + sub * 128 * 128, o_rows = e_rows + 2 * kF2A1Tile;
              const uint32_t d_even = tmem_base + st * 128 + 2 * sub * 32, d_odd = d_even + 32;
              umma_f16(d_even, sw_desc<false>(e_rows) + 2 * k, w10, idesc64, k != 0);      // E[j]   -> (even | odd)
              umma_f16(d_even, sw_desc<false>(o_rows + 128) + 2 * k, w21, idesc64, 1);     // O[j]   -> (even | odd)
              umma_f16(d_even, sw_desc<false>(o_rows) + 2 * k, w0, a.idesc, 1);            // O[j-1] -> even
              umma_f16(d_odd, sw_desc<false>(e_rows + 128) + 2 * k, w21, a.idesc, 1);      // E[j+1] x w2 -> odd
            }
          }
        }
      } else {
#pragma unroll
      for (int wp = 0; wp < WPLANES; ++wp)
#pragma unroll
        for (int ap = 0; ap < ((wp == 0 && !F8) ? PLANES : 1); ++ap)
          issue_group(a1s + ap * 2 * kF2A1Tile, w1_addr + wp * 3 * 2048, false, wp == 0 && ap == 0);
      }
      if (F8)   // correction pass: [a8 | lo8] x [W_lo * 2^3 | W * 2^-9], 64 e4m3 per row = 2 k-steps
        issue_group(a1s + 2 * kF2A1Tile, w1_addr + 3 * 2048, true, false);
      umma_commit_p(leader, &s.a1_empty[st]);
      umma_commit_p(leader, &s.d1_full[st]);
      ++k1;
      cur = nxt;
    }
  } else if (warp < 2 + kF2CvtThreads / 32) {
    // ===================== cvt1: signal -> layer-0 A rows =====================
    const int ct = (warp - 2) * 32 + lane;      // 0..kF2CvtThreads-1
    const __half2 one2 = __floats2half2_rn(1.f, 1.f);
    F2Iter iter(flags_l, n_items);
    int k = 0;
    for (int item = iter.take(); item >= 0; item = iter.take(), ++k) {
      const int st = k & 1;
      const int xst = k % kF2XStages;
      mbar_wait(&s.x_full[xst], (k / kF2XStages) & 1);
      mbar_wait(&s.a0_empty[st], ((k >> 1) & 1) ^ 1);
      unsigned char* tile = a0_ring + st * kF2A0Tile;
      const float* xs = reinterpret_cast<const float*>(x_ring + xst * kF2XStage) + 8;   // xs[4*i + e]
      const long long u0 = static_cast<long long>(item) * kF2Pairs;
      for (int i = ct - 1; i <= 255; i += kF2CvtThreads) {
        const long long u = u0 + i;
        const bool inb = (u >= 0 && u < n_pairs);
        const uint32_t uu = inb ? static_cast<uint32_t>(u) : 0u;
        const int b = static_cast<int>((static_cast<unsigned long long>(uu) * a.pair_magic) >> 40);
        const int t4 = 4 * (static_cast<int>(uu) - b * a.half_lp);
        const int L = inb ? __ldg(a.len0 + b) : 0;
        const float4 x03 = *reinterpret_cast<const float4*>(xs + 4 * i);
        const float2 x01 = make_float2(x03.x, x03.y), x23 = make_float2(x03.z, x03.w);
        float xm1 = (t4 > 0) ? xs[4 * i - 1] : 0.f;
        float x4 = xs[4 * i + 4];
        const int half_len = L >> 1;
        const bool e_ok = (t4 >> 1) < half_len;          // row p = 2t is a valid pooled layer-0 row
        const bool o_ok = (t4 >> 1) + 1 < half_len;      // row p = 2t + 1
        float x2 = (t4 + 2 < L) ? x23.x : 0.f;           // 'same' padding at the end of the read
        if (t4 + 4 >= L) x4 = 0.f;
        // fp16 range guard (|x| > 65504 only for pathological reads; the old path saturated too)
        auto clampf = [](float v) { return fminf(fmaxf(v, -65504.f), 65504.f); };
        const float v[6] = {clampf(xm1), clampf(x01.x), clampf(x01.y), clampf(x2), clampf(x23.y), clampf(x4)};
        __half2 hi[3], lo[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          hi[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
          const float2 back = __half22float2(hi[j]);
          lo[j] = __floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
        }
        // windows: E = v[0..3]; O = v[2..5]
        if (i >= 0) {
          unsigned char* row = tile + i * 64;
          const int sw = (i >> 1) & 3;
          uint4 c0 = make_uint4(0, 0, 0, 0), c1 = make_uint4(0, 0, 0, 0);
          if (e_ok) {
            c0 = make_uint4(h2_bits(hi[0]), h2_bits(hi[1]), h2_bits(lo[0]), h2_bits(lo[1]));
            c1 = make_uint4(h2_bits(hi[0]), h2_bits(hi[1]), h2_bits(one2), 0u);
          }
          *reinterpret_cast<uint4*>(row + ((0 ^ sw) << 4)) = c0;
          *reinterpret_cast<uint4*>(row + ((1 ^ sw) << 4)) = c1;
        }
        if (i + 1 <= 255) {
          unsigned char* row = tile + (i + 1) * 64;
          const int sw = ((i + 1) >> 1) & 3;
          uint4 c2 = make_uint4(0, 0, 0, 0), c3 = make_uint4(0, 0, 0, 0);
          if (o_ok) {
            c2 = make_uint4(h2_bits(hi[1]), h2_bits(hi[2]), h2_bits(lo[1]), h2_bits(lo[2]));
            c3 = make_uint4(h2_bits(hi[1]), h2_bits(hi[2]), h2_bits(one2), 0u);
          }
          *reinterpret_cast<uint4*>(row + ((2 ^ sw) << 4)) = c2;
          *reinterpret_cast<uint4*>(row + ((3 ^ sw) << 4)) = c3;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&s.x_empty[xst]);
        mbar_arrive(&s.a0_full[st]);
      }
    }
  } else if (warp < 10 + kF2CvtThreads / 32) {
    // ===================== mid-epilogue: layer-0 accumulators -> layer-1 A tiles =====================
    const int q = warp & 3;
    const int h = (warp - 2 - kF2CvtThreads / 32) >> 2;       // 0: E sub-tiles, 1: O sub-tiles
    F2Iter iter(flags_l, n_items);
    int k = 0;
    for (int item = iter.take(); item >= 0; item = iter.take(), ++k) {
      const int st = k & 1;
      mbar_wait(&s.a1_empty[st], ((k >> 1) & 1) ^ 1);
      mbar_wait(&s.d0_full[h], k & 1);
      tc_fence_after();
      unsigned char* tile_hi = a1_ring + st * kA1Stage + h * kF2A1Tile;
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + kF2D0Col + (h * 2 + sub) * kF2N0;
        uint32_t e0[16], e1[8], o0[16], o1[8];
        tmem_ld_32x16(taddr, e0);
        tmem_ld_32x16(taddr + 24, o0);
        if (a.cout0 > 20) {        // TMEM reads are 64 B/clk per SM: do not fetch the zero columns
          tmem_ld_32x8(taddr + 16, e1);
          tmem_ld_32x8(taddr + 40, o1);
        } else {
#pragma unroll
          for (int j = 4; j < 8; ++j) e1[j] = o1[j] = 0u;
          tmem_ld_32x4(taddr + 16, e1);
          tmem_ld_32x4(taddr + 40, o1);
        }
        tmem_ld_wait();
        if (sub == 1) {          // both sub-tiles are in registers: layer 0 of the next item may overwrite them
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&s.d0_empty[h]);
        }
        const int row = sub * 128 + 32 * q + lane;
        unsigned char* rp = tile_hi + row * 64;
        const int sw = (row >> 1) & 3;
        float v[24];
#pragma unroll
        for (int c = 0; c < 24; ++c) {
          const float ev = __uint_as_float(c < 16 ? e0[c & 15] : e1[c & 7]);
          const float ov = __uint_as_float(c < 16 ? o0[c & 15] : o1[c & 7]);
          v[c] = fmaxf(fmaxf(ev, ov), 0.f);
        }
        __half2 hv[12];
#pragma unroll
        for (int j = 0; j < 12; ++j) hv[j] = sat_half2(v[2 * j], v[2 * j + 1]);
        if (KC) {
          // 128-byte row [hi ch 0..19 | lo ch 0..19 | hi ch 0..19 | 0]: 32 words = hv[0..9], lv[0..9], hv[0..9], 0, 0
          uint32_t w[32];
#pragma unroll
          for (int j = 0; j < 10; ++j) {
            const float2 back = __half22float2(hv[j]);
            w[j] = w[20 + j] = h2_bits(hv[j]);
            w[10 + j] = h2_bits(__floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y));
          }
          w[30] = w[31] = 0u;
          unsigned char* rk = a1_ring + st * kA1Stage + h * 2 * kF2A1Tile + row * 128;
          const int swk = row & 7;                        // SWIZZLE_128B: 16-byte chunk c at c ^ (row & 7)
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8)
            *reinterpret_cast<uint4*>(rk + ((c8 ^ swk) << 4)) = make_uint4(w[4 * c8], w[4 * c8 + 1], w[4 * c8 + 2], w[4 * c8 + 3]);
        } else {
#pragma unroll
          for (int c8 = 0; c8 < 3; ++c8)
            *reinterpret_cast<uint4*>(rp + ((c8 ^ sw) << 4)) = *reinterpret_cast<const uint4*>(hv + 4 * c8);
        }
        if (PLANES == 2 && !F8 && !KC) {
          __half2 lv[12];
#pragma unroll
          for (int j = 0; j < 12; ++j) {
            const float2 back = __half22float2(hv[j]);
            lv[j] = __floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
          }
#pragma unroll
          for (int c8 = 0; c8 < 3; ++c8)
            *reinterpret_cast<uint4*>(rp + 2 * kF2A1Tile + ((c8 ^ sw) << 4)) = *reinterpret_cast<const uint4*>(lv + 4 * c8);
        }
        if (F8) {   // byte row: [a8 ch 0..31 | lo8 ch 0..31], channels 24..31 are zero
          uint32_t pa[6], pl[6];
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            uint32_t wa[2], wl[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = 4 * j + 2 * e;
              const float2 back = __half22float2(hv[c / 2]);
              wa[e] = __nv_cvt_float2_to_fp8x2(make_float2(v[c] * kF8AScale, v[c + 1] * kF8AScale), __NV_SATFINITE,
                                               __NV_E4M3);
              wl[e] = __nv_cvt_float2_to_fp8x2(
                  make_float2((v[c] - back.x) * kF8LoScale, (v[c + 1] - back.y) * kF8LoScale), __NV_SATFINITE, __NV_E4M3);
            }
            pa[j] = wa[0] | (wa[1] << 16);
            pl[j] = wl[0] | (wl[1] << 16);
          }
          unsigned char* rp8 = rp + 2 * kF2A1Tile;
          *reinterpret_cast<uint4*>(rp8 + ((0 ^ sw) << 4)) = make_uint4(pa[0], pa[1], pa[2], pa[3]);
          *reinterpret_cast<uint4*>(rp8 + ((1 ^ sw) << 4)) = make_uint4(pa[4], pa[5], 0u, 0u);
          *reinterpret_cast<uint4*>(rp8 + ((2 ^ sw) << 4)) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
          *reinterpret_cast<uint4*>(rp8 + ((3 ^ sw) << 4)) = make_uint4(pl[4], pl[5], 0u, 0u);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.a1_full[st]);
    }
  } else {
    // ===================== epilogue: layer-1 accumulators -> act_2 =====================
    const int q = warp & 3;
    const int sub = (warp - 10 - kF2CvtThreads / 32) >> 2;
    const int row_elems = a.cout_p * a.out_planes;
    const int lo_off = (a.out_planes == 2 && !a.out_f8) ? a.cout_p : 0;
    const float inv_scale = a.w_inv_scale;
    F2Iter iter(flags_l, n_items);
    int k = 0;
    for (int item = iter.take(); item >= 0; item = iter.take(), ++k) {
      const int st = k & 1;
      const int j = sub * 128 + 32 * q + lane;
      const long long u = static_cast<long long>(item) * kF2Pairs + j;
      const bool ok = (j < kF2Pairs) && (u < n_pairs);
      const uint32_t uu = ok ? static_cast<uint32_t>(u) : 0u;
      const int b = static_cast<int>((static_cast<unsigned long long>(uu) * a.pair_magic) >> 40);
      const int tp = static_cast<int>(uu) - b * a.half_lp;
      const bool valid = ok && tp < (__ldg(a.len0 + b) >> a.shift);
      const bool writable = ok && tp < a.Lp_out;
      const int64_t out_row = a.out_eo ? static_cast<int64_t>(tp & 1) * a.n_pairs_out + static_cast<int64_t>(b) * a.half_lp_out + (tp >> 1)
                                       : static_cast<int64_t>(b) * a.Lp_out + tp;
      __half* orow = static_cast<__half*>(a.out) + out_row * row_elems;
      mbar_wait(&s.d1_full[st], (k >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + st * 128 + 2 * sub * 32;
      // m[c] = max of the two conv positions of a pool pair (accumulator units); bias, ReLU, mask, fp16 hi + lo, stores
      auto finish = [&](int c16, const float (&m)[16]) {
        if (!writable) return;
        float r[16];
        if (valid) {
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 bb = *reinterpret_cast<const float4*>(&s.bias[c16 * 16 + c4 * 4]);
            const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = c4 * 4 + e;
              r[c] = fmaxf(fmaf(m[c], inv_scale, bv[e]), 0.f);
            }
          }
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) r[c] = 0.f;
        }
        __half2 hv[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) hv[c] = sat_half2(r[2 * c], r[2 * c + 1]);
        st_global_256(orow + c16 * 16, *reinterpret_cast<const uint4*>(hv), *reinterpret_cast<const uint4*>(hv + 4));
        if (lo_off) {
          __half2 lv[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float2 back = __half22float2(hv[c]);
            lv[c] = __floats2half2_rn(r[2 * c] - back.x, r[2 * c + 1] - back.y);
          }
          st_global_256(orow + lo_off + c16 * 16, *reinterpret_cast<const uint4*>(lv),
                        *reinterpret_cast<const uint4*>(lv + 4));
        }
        if (a.out_f8)
          store_f8_planes<16>(r, hv, reinterpret_cast<uint8_t*>(orow) + 2 * a.cout_p + c16 * 16, a.cout_p);
      };
      // The second half's accumulator columns are loaded while the first half is finished, and the accumulator is
      // handed back to the MMA warp as soon as they have arrived -- before, not after, the second half's arithmetic and
      // stores (the MMA warp was waiting on d1_empty).
      float m0[16];
      {
        uint32_t ve[16], vo[16];
        tmem_ld_32x16(taddr, ve);
        tmem_ld_32x16(taddr + 32, vo);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) m0[j] = fmaxf(__uint_as_float(ve[j]), __uint_as_float(vo[j]));
      }
      uint32_t ve1[16], vo1[16];
      tmem_ld_32x16(taddr + 16, ve1);
      tmem_ld_32x16(taddr + 32 + 16, vo1);
      finish(0, m0);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.d1_empty[st][sub]);
#pragma unroll
      for (int j = 0; j < 16; ++j) m0[j] = fmaxf(__uint_as_float(ve1[j]), __uint_as_float(vo1[j]));
      finish(1, m0);
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

FusedKernelFn pick_fused01(int mode) {
  if (mode == 0) return fused01_kernel<0>;
  if (mode == 1) return fused01_kernel<1>;
  if (mode == 2) return fused01_kernel<2>;
  if (mode == 4) return fused01_kernel<4>;
  return fused01_kernel<3>;
}
size_t fused01_smem(int planes, int wplanes) {
  return 1024 + static_cast<size_t>(wplanes) * 3 * 32 * 64 + kF2N0 * 64 + 2 * kF2A0Tile +
         2 * static_cast<size_t>(planes) * 2 * kF2A1Tile + kF2XStages * kF2XStage + sizeof(F2Smem) + 64;
}

// ------------------------------------------------------------------------------------
// Narrow layers with the even / odd row layout ("EO", layers 2..4 of the shipped network).
//
// For N <= 128 a tcgen05.mma is paced by its A-operand fetch from shared memory (~64 cycles per
// M = 128, K = 16 instruction whatever N is) and the epilogue by instruction issue, so what counts
// is the NUMBER of MMAs and of epilogue instructions per output.  With the input stored as an
// E plane (rows 2j of every read, flat pair index u = b * half_lp + j) followed by an O plane
// (rows 2j + 1), the conv at position 2j is  w0*O[j-1] + w1*E[j] + w2*O[j]  and at 2j + 1
// w0*E[j] + w1*O[j] + w2*E[j+1]; grouped by A rows
//     E[j]   x [w1; w0] -> (even | odd)        O[j]   x [w2; w1] -> (even | odd)       (N = 2n)
//     O[j-1] x  w0      ->  even                E[j+1] x  w2      ->  odd               (N = n)
// i.e. 4 MMAs instead of 6 per K step, the two positions of a max-pool pair land in the same TMEM
// lane (pooling = in-lane max, no shuffles), and a lane owns a whole output row.  Tiles are flat
// slices of the pair index; the rows that separate reads are zero as in the flat layout (O[-1] of a
// read is the previous read's last odd row, which lies beyond every valid length).
// Weights are resident ([plane][K block][tap slot 2 - tap][n_tile rows x 64 B]); 32-channel K blocks.
constexpr uint32_t kEoTile = 136 * 64;      // 128 rows + 1 halo row (+ 7: TMA box of 136 rows), 64-byte rows

template <int MS, int PLANES, int WPLANES>
__global__ void __launch_bounds__(64 + 128 * kMaxEpiSets, 1)
conv_eo_kernel(const __grid_constant__ CUtensorMap tm_e, const __grid_constant__ CUtensorMap tm_o,
               const __grid_constant__ CUtensorMap tm_b, const ConvArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr uint32_t kGroup = MS * PLANES * 2 * kEoTile;           // A tiles of one K block: [sub][plane][E, O]
  const uint32_t b_bytes = a.n_tile * 64;
  unsigned char* a_ring = base;
  unsigned char* b_region = base + static_cast<size_t>(a.a_stages) * kGroup;
  const size_t b_region_bytes = static_cast<size_t>(WPLANES) * a.k_blocks * 3 * b_bytes;
  ConvSmem& s = *reinterpret_cast<ConvSmem*>(b_region + b_region_bytes);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const int n_items = a.n_supers;
  const int acc2 = a.acc_cols;                 // TMEM columns of one sub-tile: [even n | odd n], rounded to 32

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_e);
    tma_prefetch_desc(&tm_o);
    tma_prefetch_desc(&tm_b);
    for (int i = 0; i < a.a_stages; ++i) {
      mbar_init(&s.a_full[i], 1);
      mbar_init(&s.a_empty[i], 1);
    }
    mbar_init(&s.w_full, 1);
    for (int i = 0; i < a.acc_stages; ++i) {
      mbar_init(&s.tmem_full[i], 1);
      for (int ms = 0; ms < MS; ++ms) mbar_init(&s.tmem_empty[i][ms], 4 * a.epi_sets);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&s.tmem_base, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(&s.w_full, static_cast<uint32_t>(b_region_bytes));
      for (int wp = 0; wp < WPLANES; ++wp)
        for (int kb = 0; kb < a.k_blocks; ++kb)
          for (int tap = 0; tap < 3; ++tap)
            tma_load_2d(b_region + static_cast<size_t>((wp * a.k_blocks + kb) * 3 + 2 - tap) * b_bytes, &tm_b,
                        &s.w_full, kb * 32, (wp * 3 + tap) * a.cout_p);
      int sa = 0;
      uint32_t pa = 0;
      ItemCursor cur(blockIdx.x, gridDim.x, 1);
      ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
        if (!fl.take(cur, item + gridDim.x < n_items)) continue;
        const int u0 = cur.super * (MS * kBlockM);
        for (int kb = 0; kb < a.k_blocks; ++kb) {
          mbar_wait(&s.a_empty[sa], pa ^ 1);
          mbar_arrive_expect_tx(&s.a_full[sa], MS * PLANES * 2 * kEoTile);
          unsigned char* dst = a_ring + static_cast<size_t>(sa) * kGroup;
#pragma unroll
          for (int ms = 0; ms < MS; ++ms)
#pragma unroll
            for (int ap = 0; ap < PLANES; ++ap) {
              unsigned char* t = dst + (ms * PLANES + ap) * 2 * kEoTile;
              const int apc = ap * a.cin_p;
              tma_load_2d(t, &tm_e, &s.a_full[sa], apc + kb * 32, u0 + ms * kBlockM);              // E[j ..]
              tma_load_2d(t + kEoTile, &tm_o, &s.a_full[sa], apc + kb * 32, u0 + ms * kBlockM - 1);  // O[j-1 ..]
            }
          if (++sa == a.a_stages) {
            sa = 0;
            pa ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // (the whole warp runs the loop so that the descriptor arithmetic stays in uniform registers; the elected lane issues)
    const bool leader = elect_one();
    mbar_wait(&s.w_full, 0);
    tc_fence_after();
    int sa = 0, stage = 0;
    uint32_t pa = 0, acc_phase = 0;
    const uint32_t a_ring_addr = smem_u32(a_ring), b_region_addr = smem_u32(b_region);
    const int nk_last = (a.cin_p - (a.k_blocks - 1) * 32) / 16;
    const uint32_t idesc1 = a.idesc;                                  // N = n_tile
    const uint32_t idesc2 = umma_idesc_f16(kBlockM, 2 * a.n_tile);    // N = 2 n_tile: (even | odd)
    ItemCursor cur(blockIdx.x, gridDim.x, 1);
    ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
      if (!fl.take(cur, item + gridDim.x < n_items)) continue;
      const uint32_t d_base = tmem_base + stage * (MS * acc2);
      for (int kb = 0; kb < a.k_blocks; ++kb) {
        const int nk = (kb == a.k_blocks - 1) ? nk_last : 2;
        mbar_wait(&s.a_full[sa], pa);
        tc_fence_after();
        const uint32_t a_addr = a_ring_addr + sa * kGroup;
#pragma unroll
        for (int wp = 0; wp < WPLANES; ++wp) {
          const uint32_t w_set = b_region_addr + ((wp * a.k_blocks + kb) * 3) * b_bytes;   // slots: w2, w1, w0
#pragma unroll
          for (int ms = 0; ms < MS; ++ms) {
            if (kb == 0 && wp == 0) {      // first touch of this accumulator: wait until drained
              mbar_wait(&s.tmem_empty[stage][ms], acc_phase ^ 1);
              tc_fence_after();
            }
            const uint32_t d_even = d_base + ms * acc2, d_odd = d_even + a.n_tile;
#pragma unroll
            for (int ap = 0; ap < (wp == 0 ? PLANES : 1); ++ap) {      // W_lo only meets the hi plane
              const uint32_t e_rows = a_addr + (ms * PLANES + ap) * 2 * kEoTile, o_rows = e_rows + kEoTile;
              if (leader) {
#pragma unroll
                for (int k = 0; k < 2; ++k)
                  if (k < nk) {
                    const uint64_t w21 = sw_desc<true>(w_set) + 2 * k;
                    const uint64_t w10 = sw_desc<true>(w_set + b_bytes) + 2 * k;
                    const uint64_t w0 = sw_desc<true>(w_set + 2 * b_bytes) + 2 * k;
                    umma_f16(d_even, sw_desc<true>(e_rows) + 2 * k, w10, idesc2, (kb | wp | ap | k) != 0);   // E[j]
                    umma_f16(d_even, sw_desc<true>(o_rows + 64) + 2 * k, w21, idesc2, 1);                    // O[j]
                    umma_f16(d_even, sw_desc<true>(o_rows) + 2 * k, w0, idesc1, 1);                          // O[j-1]
                    umma_f16(d_odd, sw_desc<true>(e_rows + 64) + 2 * k, w21, idesc1, 1);                     // E[j+1] x w2
                  }
              }
            }
          }
        }
        umma_commit_p(leader, &s.a_empty[sa]);
        if (++sa == a.a_stages) {
          sa = 0;
          pa ^= 1;
        }
      }
      umma_commit_p(leader, &s.tmem_full[stage]);
      if (++stage == a.acc_stages) {
        stage = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp < 2 + 4 * a.epi_sets) {
    // ===================== epilogue: one output row per lane =====================
    const int q = warp & 3;
    const int eset = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;
    const int epi_threads = 128 * a.epi_sets;
    const int row_elems = a.cout_p * a.out_planes;
    const int lo_off = (a.out_planes == 2 && !a.out_f8) ? a.cout_p : 0;
    const int n_chunks = a.n_tile >> 4;
    const int n_pairs = a.rows_in >> 1;
    for (int i = et; i < a.n_tile; i += epi_threads) s.bias[0][i] = a.bias[i];
    asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
    int stage = 0;
    uint32_t acc_phase = 0;
    ItemCursor cur(blockIdx.x, gridDim.x, 1);
    ItemFlags fl(a.flags, cur.super, blockIdx.x < n_items);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, cur.next()) {
      if (!fl.take(cur, item + gridDim.x < n_items)) continue;
      const int u0 = cur.super * (MS * kBlockM);
      bool valid[MS], writable[MS];
      int64_t out_row[MS];
#pragma unroll
      for (int ms = 0; ms < MS; ++ms) {
        valid[ms] = writable[ms] = false;
        out_row[ms] = 0;
        const int u = u0 + ms * kBlockM + 32 * q + lane;
        if (u < n_pairs) {
          const int b = static_cast<int>((static_cast<unsigned long long>(static_cast<uint32_t>(u)) * a.pair_magic) >> 40);
          const int tp = u - b * a.half_lp;
          valid[ms] = tp < (__ldg(a.len0 + b) >> a.shift);
          writable[ms] = tp < a.Lp_out;
          out_row[ms] = a.out_eo ? static_cast<int64_t>(tp & 1) * a.n_pairs_out + static_cast<int64_t>(b) * a.half_lp_out + (tp >> 1)
                                 : static_cast<int64_t>(b) * a.Lp_out + tp;
        }
      }
      mbar_wait(&s.tmem_full[stage], acc_phase);
      tc_fence_after();
      int uw = eset;       // work units = (sub-tile, 16-column chunk), dealt round-robin to the epilogue sets
#pragma unroll
      for (int ms = 0; ms < MS; ++ms) {
        __half* orow = static_cast<__half*>(a.out) + out_row[ms] * row_elems;
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + (stage * MS + ms) * acc2;
        for (; uw < (ms + 1) * n_chunks; uw += a.epi_sets) {
          const int c = uw - ms * n_chunks;
          uint32_t ve[16], vo[16];
          tmem_ld_32x16(t_addr + c * 16, ve);
          tmem_ld_32x16(t_addr + a.n_tile + c * 16, vo);
          tmem_ld_wait();
          if (writable[ms])
            epilogue_row16(ve, vo, s.bias[0] + c * 16, valid[ms], a.w_inv_scale, orow + c * 16, lo_off,
                           a.out_f8 ? reinterpret_cast<uint8_t*>(orow) + 2 * a.cout_p + c * 16 : nullptr, a.cout_p);
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s.tmem_empty[stage][ms]);
      }
      if (++stage == a.acc_stages) {
        stage = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

EoKernelFn pick_conv_eo(int ms, int planes, int wplanes) {
  if (ms == 2) {
    if (planes == 1 && wplanes == 1) return conv_eo_kernel<2, 1, 1>;
    if (planes == 1 && wplanes == 2) return conv_eo_kernel<2, 1, 2>;
    return conv_eo_kernel<2, 2, 2>;
  }
  if (planes == 1 && wplanes == 1) return conv_eo_kernel<1, 1, 1>;
  if (planes == 1 && wplanes == 2) return conv_eo_kernel<1, 1, 2>;
  return conv_eo_kernel<1, 2, 2>;
}

// ------------------------------------------------------------------------------------
// Two narrow layers in ONE launch ("EO2", layers 2 + 3 of the shipped network): the activation between them never
// exists in HBM (3.1 GB of the 16 GB the conv stack moved per 4096 x 16,000 forward, and the two layers it sat
// between were HBM-bound: 5.7 and 4.9 TB/s).  Both layers keep the even / odd row scheme of conv_eo_kernel.
//
// Work item = (read b, segment s): 127 rows j = 127 s + l of the SECOND layer's pooled output.  They need the
// first layer's output rows 2j - 1 .. 2j + 2, i.e. r in [254 s - 1, 254 s + 255): exactly two 128-lane tiles of the
// first layer (A: r = c + l with c = 254 s - 1, B: c + 128), whose inputs the producer takes from the E / O planes
// in HBM by TMA at any offset (rows before the read's start or beyond its end feed lanes that are masked to zero,
// which is also what gives the convolution its 'same' padding).  A mid-epilogue drains the first layer's
// accumulators (max-pool in-lane, bias, ReLU, length mask, fp16 hi + lo split) into the SECOND layer's operand
// tiles in shared memory -- row r goes to the E tile (even r, index r / 2 - 127 s) or the O tile (odd r, index
// (r - 1) / 2 - 127 s + 1), in the SWIZZLE_64B K-major layout a TMA load would have produced -- and the second layer
// runs 127 valid lanes (lane 127 reads the slack row 128 of both tiles and is discarded).  Halo recomputed: 2 of
// 256 first-layer rows per item.
//
// Roles (18 warps): warp 0 TMA producer (weights of both layers once, then a 2-stage ring of first-layer input
// tiles), warp 1 MMA issuer, warps 2-5 / 6-9 mid-epilogue of tile A / tile B, warps 10-17 final epilogue (two
// sets splitting the 16-column chunks).  Issue order: ..., first layer of item k + 1 (two tiles), second layer of
// item k, ...: the mid-epilogue of item k + 1 runs while the tensor pipe works on the second layer of item k and
// the first layer of item k + 2, the one copy of the intermediate tiles being handed back by the commit behind the
// second layer's MMAs.  TMEM: three first-layer accumulator slots (a tile waits there for the intermediate
// tiles to come free) + one second-layer accumulator.
constexpr int kE2Threads = 576;
constexpr int kE2Rows = 127;              // second-layer output rows per item
constexpr int kE2MaxLocalItems = 4096;    // work items per CTA whose activity flags fit the shared-memory copy

struct Eo2Smem {
  uint64_t w_full;
  uint64_t in_full[2], in_empty[2];
  uint64_t acc1_full[3], acc1_empty[3];
  uint64_t a3_full, a3_empty;
  uint64_t acc2_full, acc2_empty;
  uint32_t tmem_base;
  alignas(16) float bias1[128];
  alignas(16) float bias2[128];
  uint8_t my_flags[kE2MaxLocalItems];   // activity of this CTA's items (item = blockIdx.x + i * gridDim.x)
};

// Active items of this CTA in order (flags staged in shared memory once: no global load in the single-thread roles).
struct Eo2Iter {
  const uint8_t* local;
  int i, item, n_items, step;
  __device__ __forceinline__ Eo2Iter(const uint8_t* l, int n) : local(l), i(0), item(blockIdx.x), n_items(n), step(gridDim.x) {}
  __device__ __forceinline__ int take() {
    while (item < n_items) {
      const int cur = item;
      const bool f = local ? (local[i] != 0) : true;
      item += step;
      ++i;
      if (f) return cur;
    }
    return -1;
  }
};

__global__ void __launch_bounds__(kE2Threads, 1)
conv_eo2_kernel(const __grid_constant__ CUtensorMap tm_e, const __grid_constant__ CUtensorMap tm_o,
                const __grid_constant__ CUtensorMap tm_b1, const __grid_constant__ CUtensorMap tm_b2, const Eo2Args a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const uint32_t b1_bytes = a.n1 * 64, b2_bytes = a.n2 * 64;
  const uint32_t w1_bytes = 2u * a.kb1 * 3 * b1_bytes, w2_bytes = 2u * a.kb2 * 3 * b2_bytes;
  const uint32_t in_stage = a.kb1 * 4 * kEoTile;            // [kb][plane][E, O]
  const uint32_t a3_bytes = a.kb2 * 4 * kEoTile;
  unsigned char* w1 = base;
  unsigned char* w2 = w1 + w1_bytes;
  unsigned char* in_ring = w2 + w2_bytes;
  unsigned char* a3 = in_ring + 2 * in_stage;
  Eo2Smem& s = *reinterpret_cast<Eo2Smem*>(a3 + a3_bytes);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const int n_items = a.B * a.n_seg;
  const bool use_flags = (n_items + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x) <= kE2MaxLocalItems;
  const uint8_t* flags_l = use_flags ? s.my_flags : nullptr;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_e);
    tma_prefetch_desc(&tm_o);
    tma_prefetch_desc(&tm_b1);
    tma_prefetch_desc(&tm_b2);
    mbar_init(&s.w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.in_full[i], 1);
      mbar_init(&s.in_empty[i], 1);
    }
    for (int i = 0; i < 3; ++i) {
      mbar_init(&s.acc1_full[i], 1);
      mbar_init(&s.acc1_empty[i], 4);
    }
    mbar_init(&s.a3_full, 8);
    mbar_init(&s.a3_empty, 1);
    mbar_init(&s.acc2_full, 1);
    mbar_init(&s.acc2_empty, 8);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&s.tmem_base, kTmemCols);
    tmem_relinquish();
  }
  // intermediate tiles: the slack rows (128..135) and the padded channels of the last K block are never written again
  for (uint32_t i = threadIdx.x; i < a3_bytes / 16; i += kE2Threads) reinterpret_cast<uint4*>(a3)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 128; i += kE2Threads) {
    s.bias1[i] = (i < a.n1) ? a.bias1[i] : 0.f;
    s.bias2[i] = (i < a.n2) ? a.bias2[i] : 0.f;
  }
  if (use_flags)
    for (int i = threadIdx.x, it = blockIdx.x + threadIdx.x * gridDim.x; it < n_items; i += kE2Threads, it += kE2Threads * gridDim.x) {
      const int b = it / a.n_seg, sg = it - b * a.n_seg;
      s.my_flags[i] = (kE2Rows * sg <= (__ldg(a.len0 + b) >> a.shift2)) ? 1 : 0;    // "<=": the zero row that ends the read
    }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(&s.w_full, w1_bytes + w2_bytes);
      // taps in REVERSE order (slot 2 - tap): [w2; w1] and [w1; w0] are contiguous B operands (see conv_eo_kernel)
      for (int wp = 0; wp < 2; ++wp)
        for (int kb = 0; kb < a.kb1; ++kb)
          for (int tap = 0; tap < 3; ++tap)
            tma_load_2d(w1 + static_cast<size_t>((wp * a.kb1 + kb) * 3 + 2 - tap) * b1_bytes, &tm_b1, &s.w_full, kb * 32,
                        (wp * 3 + tap) * a.n1);
      for (int wp = 0; wp < 2; ++wp)
        for (int kb = 0; kb < a.kb2; ++kb)
          for (int tap = 0; tap < 3; ++tap)
            tma_load_2d(w2 + static_cast<size_t>((wp * a.kb2 + kb) * 3 + 2 - tap) * b2_bytes, &tm_b2, &s.w_full, kb * 32,
                        (wp * 3 + tap) * a.n2);
      Eo2Iter iter(flags_l, n_items);
      uint32_t q = 0;                       // first-layer tiles loaded so far
      for (int item = iter.take(); item >= 0; item = iter.take()) {
        const int b = item / a.n_seg, sg = item - b * a.n_seg;
        const int c0 = 2 * kE2Rows * sg - 1;
#pragma unroll 1
        for (int t = 0; t < 2; ++t, ++q) {
          const uint32_t st = q & 1;
          mbar_wait(&s.in_empty[st], ((q >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(&s.in_full[st], in_stage);
          unsigned char* dst = in_ring + st * in_stage;
          const int u = b * a.half_lp_in + c0 + kBlockM * t;        // pair index of lane 0's E row
          for (int kb = 0; kb < a.kb1; ++kb)
#pragma unroll
            for (int ap = 0; ap < 2; ++ap) {
              unsigned char* tl = dst + static_cast<size_t>((kb * 2 + ap) * 2) * kEoTile;
              tma_load_2d(tl, &tm_e, &s.in_full[st], ap * a.cin_p1 + kb * 32, u);                 // E[c ..]
              tma_load_2d(tl + kEoTile, &tm_o, &s.in_full[st], ap * a.cin_p1 + kb * 32, u - 1);   // O[c - 1 ..]
            }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // (the whole warp runs the loop -- uniform registers -- and the elected lane issues)
    const bool leader = elect_one();
    mbar_wait(&s.w_full, 0);
    tc_fence_after();
    const uint32_t w1_addr = smem_u32(w1), w2_addr = smem_u32(w2), in_addr = smem_u32(in_ring), a3_addr = smem_u32(a3);
    const int nk_last1 = (a.cin_p1 - (a.kb1 - 1) * 32) / 16, nk_last2 = (a.n1 - (a.kb2 - 1) * 32) / 16;
    // One even / odd tile: E[j] x [w1; w0] and O[j] x [w2; w1] feed both conv positions (N = 2n), O[j-1] x w0 the
    // even and E[j+1] x w2 the odd one (N = n); hi x W_hi, lo x W_hi, hi x W_lo (W_lo only meets the hi plane).
    auto issue_tile = [&](uint32_t tiles, uint32_t w_addr, uint32_t b_bytes, int kbs, int nk_last, uint32_t d_even,
                          uint32_t n, uint32_t idesc_n, uint32_t idesc_2n) {
      const uint32_t d_odd = d_even + n;
      for (int kb = 0; kb < kbs; ++kb) {
        const int nk = (kb == kbs - 1) ? nk_last : 2;
#pragma unroll
        for (int wp = 0; wp < 2; ++wp) {
          const uint32_t w_set = w_addr + ((wp * kbs + kb) * 3) * b_bytes;      // slots: w2, w1, w0
#pragma unroll
          for (int ap = 0; ap < (wp == 0 ? 2 : 1); ++ap) {
            const uint32_t e_rows = tiles + ((kb * 2 + ap) * 2) * kEoTile, o_rows = e_rows + kEoTile;
            if (leader) {
#pragma unroll
              for (int k = 0; k < 2; ++k)
                if (k < nk) {
                  const uint64_t w21 = sw_desc<true>(w_set) + 2 * k;
                  const uint64_t w10 = sw_desc<true>(w_set + b_bytes) + 2 * k;
                  const uint64_t w0 = sw_desc<true>(w_set + 2 * b_bytes) + 2 * k;
                  umma_f16(d_even, sw_desc<true>(e_rows) + 2 * k, w10, idesc_2n, (kb | wp | ap | k) != 0);   // E[j]
                  umma_f16(d_even, sw_desc<true>(o_rows + 64) + 2 * k, w21, idesc_2n, 1);                    // O[j]
                  umma_f16(d_even, sw_desc<true>(o_rows) + 2 * k, w0, idesc_n, 1);                           // O[j-1]
                  umma_f16(d_odd, sw_desc<true>(e_rows + 64) + 2 * k, w21, idesc_n, 1);                      // E[j+1] x w2
                }
            }
          }
        }
      }
    };
    uint32_t q = 0;                       // first-layer tiles issued so far
    auto issue_first = [&]() {            // both first-layer tiles of one item
#pragma unroll 1
      for (int t = 0; t < 2; ++t, ++q) {
        const uint32_t st = q & 1, slot = q % 3;
        mbar_wait(&s.in_full[st], (q >> 1) & 1);
        tc_fence_after();
        mbar_wait(&s.acc1_empty[slot], ((q / 3) & 1) ^ 1);
        tc_fence_after();
        issue_tile(in_addr + st * in_stage, w1_addr, b1_bytes, a.kb1, nk_last1, tmem_base + slot * a.acc1, a.n1,
                   a.idesc1_n, a.idesc1_2n);
        umma_commit_p(leader, &s.in_empty[st]);
        umma_commit_p(leader, &s.acc1_full[slot]);
      }
    };
    Eo2Iter iter(flags_l, n_items);
    int cur = iter.take();
    if (cur >= 0) issue_first();
    uint32_t k = 0;                       // items whose second layer has been issued
    while (cur >= 0) {
      const int nxt = iter.take();
      if (nxt >= 0) issue_first();
      mbar_wait(&s.a3_full, k & 1);
      tc_fence_after();
      mbar_wait(&s.acc2_empty, (k & 1) ^ 1);
      tc_fence_after();
      issue_tile(a3_addr, w2_addr, b2_bytes, a.kb2, nk_last2, tmem_base + 3 * a.acc1, a.n2, a.idesc2_n, a.idesc2_2n);
      umma_commit_p(leader, &s.a3_empty);
      umma_commit_p(leader, &s.acc2_full);
      ++k;
      cur = nxt;
    }
  } else if (warp < 10) {
    // ===================== mid-epilogue: first-layer accumulators -> second-layer operand tiles =====================
    const int q4 = warp & 3;
    const int t = (warp - 2) >> 2;                    // 0: tile A, 1: tile B
    const int lrow = 32 * q4 + lane;
    const float inv_scale = a.inv_scale1;
    const int n_chunks = a.n1 >> 4;
    Eo2Iter iter(flags_l, n_items);
    uint32_t k = 0;
    int item = iter.take();
    int len_item = (item >= 0) ? __ldg(a.len0 + item / a.n_seg) : 0;
    for (; item >= 0; ++k) {
      const int nxt = iter.take();                                      // the next item's length is loaded a whole
      const int len_nxt = (nxt >= 0) ? __ldg(a.len0 + nxt / a.n_seg) : 0;   // item ahead (off the critical path)
      const int b = item / a.n_seg, sg = item - b * a.n_seg;
      const int r = 2 * kE2Rows * sg - 1 + kBlockM * t + lrow;          // row of the intermediate activation
      const bool valid = (r >= 0) && (r < (len_item >> a.shift1));
      // destination: even r -> E tile row r / 2 - 127 s, odd r -> O tile row (r - 1) / 2 - 127 s + 1
      const int eo = r & 1;
      const int idx = ((r - eo) >> 1) - kE2Rows * sg + eo;
      const int sw = (idx >> 1) & 3;
      unsigned char* row0 = a3 + static_cast<size_t>(eo) * kEoTile + idx * 64;
      const uint32_t qq = 2 * k + t, slot = qq % 3;
      mbar_wait(&s.acc1_full[slot], (qq / 3) & 1);
      tc_fence_after();
      mbar_wait(&s.a3_empty, (k & 1) ^ 1);          // the second layer of the previous item has read the tiles
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(32 * q4) << 16) + slot * a.acc1;
      for (int c = 0; c < n_chunks; ++c) {
        uint32_t ve[16], vo[16];
        tmem_ld_32x16(taddr + c * 16, ve);
        tmem_ld_32x16(taddr + a.n1 + c * 16, vo);
        tmem_ld_wait();
        if (c == n_chunks - 1) {          // accumulator in registers: the first layer of a later item may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&s.acc1_empty[slot]);
        }
        float v[16];
        if (valid) {
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 bb = *reinterpret_cast<const float4*>(&s.bias1[c * 16 + c4 * 4]);
            const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = c4 * 4 + e;
              v[j] = fmaxf(fmaf(fmaxf(__uint_as_float(ve[j]), __uint_as_float(vo[j])), inv_scale, bv[e]), 0.f);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
        }
        __half2 hv[8], lv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          hv[j] = sat_half2(v[2 * j], v[2 * j + 1]);
          const float2 back = __half22float2(hv[j]);
          lv[j] = __floats2half2_rn(v[2 * j] - back.x, v[2 * j + 1] - back.y);
        }
        // channels 16c .. 16c+15 = K block c / 2, 16-byte chunks 2 (c & 1), 2 (c & 1) + 1; planes: hi, lo
        unsigned char* rp = row0 + static_cast<size_t>((c >> 1) * 4) * kEoTile;
        const int ch = 2 * (c & 1);
        *reinterpret_cast<uint4*>(rp + (((ch) ^ sw) << 4)) = *reinterpret_cast<const uint4*>(hv);
        *reinterpret_cast<uint4*>(rp + (((ch + 1) ^ sw) << 4)) = *reinterpret_cast<const uint4*>(hv + 4);
        *reinterpret_cast<uint4*>(rp + 2 * kEoTile + (((ch) ^ sw) << 4)) = *reinterpret_cast<const uint4*>(lv);
        *reinterpret_cast<uint4*>(rp + 2 * kEoTile + (((ch + 1) ^ sw) << 4)) = *reinterpret_cast<const uint4*>(lv + 4);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic writes -> visible to the MMA
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.a3_full);
      item = nxt;
      len_item = len_nxt;
    }
  } else {
    // ===================== epilogue: second-layer accumulators -> HBM, one output row per lane =====================
    const int q4 = warp & 3;
    const int eset = (warp - 10) >> 2;
    const int lrow = 32 * q4 + lane;
    const int row_elems = a.cout_p2 * a.out_planes;
    const int lo_off = (a.out_planes == 2 && !a.out_f8) ? a.cout_p2 : 0;
    const int n_chunks = a.n2 >> 4;
    Eo2Iter iter(flags_l, n_items);
    uint32_t k = 0;
    int item = iter.take();
    int len_item = (item >= 0) ? __ldg(a.len0 + item / a.n_seg) : 0;
    for (; item >= 0; ++k) {
      const int nxt = iter.take();
      const int len_nxt = (nxt >= 0) ? __ldg(a.len0 + nxt / a.n_seg) : 0;
      const int b = item / a.n_seg, sg = item - b * a.n_seg;
      const int j = kE2Rows * sg + lrow;
      const bool writable = (lrow < kE2Rows) && (j < a.Lp_out);
      const bool valid = writable && (j < (len_item >> a.shift2));
      const int64_t out_row = a.out_eo ? static_cast<int64_t>(j & 1) * a.n_pairs_out + static_cast<int64_t>(b) * a.half_lp_out + (j >> 1)
                                       : static_cast<int64_t>(b) * a.Lp_out + j;
      __half* orow = static_cast<__half*>(a.out) + out_row * row_elems;
      mbar_wait(&s.acc2_full, k & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(32 * q4) << 16) + 3 * a.acc1;
      for (int c = eset; c < n_chunks; c += 2) {
        uint32_t ve[16], vo[16];
        tmem_ld_32x16(taddr + c * 16, ve);
        tmem_ld_32x16(taddr + a.n2 + c * 16, vo);
        tmem_ld_wait();
        if (writable)
          epilogue_row16(ve, vo, s.bias2 + c * 16, valid, a.inv_scale2, orow + c * 16, lo_off,
                         a.out_f8 ? reinterpret_cast<uint8_t*>(orow) + 2 * a.cout_p2 + c * 16 : nullptr, a.cout_p2);
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.acc2_empty);
      item = nxt;
      len_item = len_nxt;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

size_t conv_eo2_smem(int n1, int n2, int kb1, int kb2) {
  return 1024 + 2ull * kb1 * 3 * n1 * 64 + 2ull * kb2 * 3 * n2 * 64 + 2ull * kb1 * 4 * kEoTile + 1ull * kb2 * 4 * kEoTile +
         sizeof(Eo2Smem) + 64;
}

// ------------------------------------------------------------------------------------
// Wide layers on CTA pairs (cta_group::2, clusters of two CTAs; F16_F8 layers with streamed weights).
//
// One M = 256 MMA spans both SMs of a pair: each CTA stages 128 rows of A (its half of a 256-row
// sub-tile) and HALF of the N rows of every weight tile, so the weight bytes streamed from L2 and the
// shared-memory operand bytes read per MAC are halved per SM -- which is what bounds the e4m3 pass
// of these layers (a one-CTA e4m3 MMA at N = 192 needs 213 B/clk of operands).  The leader CTA's
// thread issues the MMAs; TMA loads of both CTAs complete on the leader's "full" barriers
// (cp.async.bulk.tensor ... cta_group::2 with the peer bit cleared), tcgen05.commit multicasts the
// "empty" / "accumulator full" arrivals to both CTAs, and the peer's epilogue warps release the
// accumulators on the leader's barrier (mapa + remote arrive).
// Work item of a pair = (256 flat rows, N tile); both CTAs walk the same item list.
__global__ void __launch_bounds__(64 + 128 * kMaxEpiSets, 1)
conv_pair_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const __grid_constant__ CUtensorMap tm_a8, const __grid_constant__ CUtensorMap tm_b8,
                 const __grid_constant__ CUtensorMap tm_bl, const __grid_constant__ CUtensorMap tm_b8l,
                 const ConvArgs a) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr uint32_t kATile = 136 * 128;
  const uint32_t b_bytes = (a.n_tile / 2) * 128;           // this CTA's half of a (full-width) weight tile
  unsigned char* a_ring = base;
  unsigned char* b_region = base + static_cast<size_t>(a.a_stages) * kATile;
  // (`resident`: one N tile whose halves fit -- every CTA keeps ITS half of all taps and K blocks for the whole kernel,
  //  [tap][K block][n_tile / 2 rows x 128 B], and nothing but activations is streamed: layer 5)
  const size_t b_region_bytes = a.resident ? static_cast<size_t>(3) * a.k_blocks * b_bytes : static_cast<size_t>(a.b_stages) * b_bytes;
  ConvSmem& s = *reinterpret_cast<ConvSmem*>(b_region + b_region_bytes);

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = (rank == 0);
  const int pair = blockIdx.x >> 1, n_pairs_grid = gridDim.x >> 1;
  const int n_items = a.n_supers * a.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    tma_prefetch_desc(&tm_a8);
    tma_prefetch_desc(&tm_b8);
    tma_prefetch_desc(&tm_bl);
    tma_prefetch_desc(&tm_b8l);
    for (int i = 0; i < a.a_stages; ++i) {
      mbar_init(&s.a_full[i], 1);
      mbar_init(&s.a_empty[i], 1);
    }
    for (int i = 0; i < a.b_stages; ++i) {
      mbar_init(&s.b_full[i], 1);
      mbar_init(&s.b_empty[i], 1);
    }
    mbar_init(&s.w_full, 1);
    for (int i = 0; i < a.acc_stages; ++i) {
      mbar_init(&s.tmem_full[i], 1);
      mbar_init(&s.tmem_empty[i][0], 2 * 4 * a.epi_sets);   // both CTAs' warps
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_pair(&s.tmem_base, kTmemCols);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  // item -> (M super-tile, N tile), N fastest; the pair visits item = pair, pair + n_pairs_grid, ...
  // (the N tile is rotated by the super-tile index: the grid stride may be a multiple of n_tiles, and the last tile
  //  is narrower than the others -- every pair then still gets its share of both widths)
  // (division by the run-time n_tiles through a multiply: the roles that walk the item list -- the MMA-issuing warp
  //  among them -- did two divisions and two remainders, ~120 instructions, per item)
  auto div_nt = [&](int x) {
    if (a.n_tiles == 1) return x;
    return a.nt_magic ? static_cast<int>(__umulhi(static_cast<uint32_t>(x), a.nt_magic)) : x / a.n_tiles;
  };
  auto item_n = [&](int item) {
    const int q = div_nt(item), t = item - q * a.n_tiles + q;          // item % n_tiles + item / n_tiles
    return t - div_nt(t) * a.n_tiles;
  };
  // Activity flag of item, item + stride, ...: the NEXT item's flag is loaded while the current item is worked on
  // (a global load per item otherwise sits on the critical path of the single-thread roles).
  struct PairFlags {
    const uint8_t* flags;
    int n_tiles, stride, n_items;
    uint32_t next;
    uint32_t magic;
    __device__ __forceinline__ uint32_t load(int item) const {
      const int q = (n_tiles == 1) ? item : magic ? static_cast<int>(__umulhi(static_cast<uint32_t>(item), magic)) : item / n_tiles;
      return (flags && item < n_items) ? __ldg(flags + q) : 1u;
    }
    __device__ __forceinline__ PairFlags(const uint8_t* f, int nt, int first, int stride_, int n, uint32_t mg = 0)
        : flags(f), n_tiles(nt), stride(stride_), n_items(n), magic(mg) { next = load(first); }
    __device__ __forceinline__ bool take(int item) {      // call once per item, in order
      const uint32_t now = next;
      next = load(item + stride);
      return now != 0;
    }
  };

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      if (a.resident) {      // both CTAs' halves complete on the leader's barrier (the issuer lives there)
        if (leader) mbar_arrive_expect_tx(&s.w_full, 2u * static_cast<uint32_t>(b_region_bytes));
        const int n0 = static_cast<int>(rank) * (a.n_tile / 2);
        for (int tap = 0; tap < 3; ++tap)
          for (int kb = 0; kb < a.k_blocks; ++kb) {
            unsigned char* dst = b_region + static_cast<size_t>(tap * a.k_blocks + kb) * b_bytes;
            if (kb >= a.kb16) tma_load_2d_pair(dst, &tm_b8, &s.w_full, (kb - a.kb16) * 128, tap * a.cout_p + n0);
            else tma_load_2d_pair(dst, &tm_b, &s.w_full, kb * 64, tap * a.cout_p + n0);
          }
      }
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      PairFlags fl(a.flags, a.n_tiles, pair, n_pairs_grid, n_items, a.nt_magic);
      for (int item = pair; item < n_items; item += n_pairs_grid) {
        if (!fl.take(item)) continue;
        const int m0 = div_nt(item) * 256 + static_cast<int>(rank) * kBlockM - 1;
        const int n_idx = item_n(item);
        const bool last_n = (n_idx == a.n_tiles - 1);
        const int n_half = (last_n ? a.n_last : a.n_tile) / 2;       // weight rows this CTA stages per tile
        const int n0 = n_idx * a.n_tile + static_cast<int>(rank) * n_half;
        const uint32_t b_tx = static_cast<uint32_t>(n_half) * 128;
        const CUtensorMap* tb = last_n ? &tm_bl : &tm_b;
        const CUtensorMap* tb8 = last_n ? &tm_b8l : &tm_b8;
        for (int kb = 0; kb < a.k_blocks; ++kb) {
          const bool is8 = kb >= a.kb16;
          mbar_wait(&s.a_empty[sa], pa ^ 1);
          if (leader) mbar_arrive_expect_tx(&s.a_full[sa], 2 * kATile);
          unsigned char* dst = a_ring + static_cast<size_t>(sa) * kATile;
          if (is8)
            tma_load_2d_pair(dst, &tm_a8, &s.a_full[sa], 2 * a.cin_p + (kb - a.kb16) * 128, m0);
          else
            tma_load_2d_pair(dst, &tm_a, &s.a_full[sa], kb * 64, m0);
          if (++sa == a.a_stages) {
            sa = 0;
            pa ^= 1;
          }
#pragma unroll
          for (int tap = 0; tap < 3; ++tap) {
            if (a.resident) break;
            mbar_wait(&s.b_empty[sb], pb ^ 1);
            if (leader) mbar_arrive_expect_tx(&s.b_full[sb], 2 * b_tx);
            if (is8)
              tma_load_2d_pair(b_region + static_cast<size_t>(sb) * b_bytes, tb8, &s.b_full[sb], (kb - a.kb16) * 128,
                               tap * a.cout_p + n0);
            else
              tma_load_2d_pair(b_region + static_cast<size_t>(sb) * b_bytes, tb, &s.b_full[sb], kb * 64,
                               tap * a.cout_p + n0);
            if (++sb == a.b_stages) {
              sb = 0;
              pb ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    // (The whole warp runs the loop -- uniform registers, see umma_f16_p -- and the elected lane issues.)
    if (leader) {
      const uint32_t lead = elect_one() ? 1u : 0u;
      int sa = 0, sb = 0, stage = 0;
      uint32_t pa = 0, pb = 0, acc_phase = 0;
      const uint32_t a_ring_addr = smem_u32(a_ring), b_region_addr = smem_u32(b_region);
      const int nk_last = (a.cin_p - (a.kb16 - 1) * 64) / 16;
      const int nk_last8 = (2 * a.cin_p - (a.k_blocks - a.kb16 - 1) * 128) / 32;
      if (a.resident) {
        mbar_wait(&s.w_full, 0);
        tc_fence_after();
      }
      PairFlags fl(a.flags, a.n_tiles, pair, n_pairs_grid, n_items, a.nt_magic);
      for (int item = pair; item < n_items; item += n_pairs_grid) {
        if (!fl.take(item)) continue;
        const uint32_t d = tmem_base + stage * a.acc_cols;
        const uint32_t idesc = (item_n(item) == a.n_tiles - 1) ? a.idesc_last : a.idesc;
        for (int kb = 0; kb < a.k_blocks; ++kb) {
          const bool is8 = kb >= a.kb16;
          const int nk = is8 ? ((kb == a.k_blocks - 1) ? nk_last8 : 4) : ((kb == a.kb16 - 1) ? nk_last : 4);
          mbar_wait(&s.a_full[sa], pa);
          tc_fence_after();
          const uint32_t a_addr = a_ring_addr + sa * kATile;
#pragma unroll
          for (int tap = 0; tap < 3; ++tap) {
            if (!a.resident) {
              mbar_wait(&s.b_full[sb], pb);
              tc_fence_after();
            }
            const uint64_t db = sw_desc<false>(a.resident ? b_region_addr + (tap * a.k_blocks + kb) * b_bytes
                                                          : b_region_addr + sb * b_bytes);
            if (kb == 0 && tap == 0) {       // first touch of this accumulator: both CTAs have drained it
              mbar_wait(&s.tmem_empty[stage][0], acc_phase ^ 1);
              tc_fence_after();
            }
            const uint64_t da = sw_desc<false>(a_addr + tap * 128);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k < nk) {
                if (is8) umma_f8_pair_p(lead, d, da + 2 * k, db + 2 * k, idesc, 1);
                else umma_f16_pair_p(lead, d, da + 2 * k, db + 2 * k, idesc, (kb | tap | k) != 0);
              }
            if (!a.resident) {
              umma_commit_pair_p(lead, &s.b_empty[sb]);
              if (++sb == a.b_stages) {
                sb = 0;
                pb ^= 1;
              }
            }
          }
          umma_commit_pair_p(lead, &s.a_empty[sa]);
          if (++sa == a.a_stages) {
            sa = 0;
            pa ^= 1;
          }
        }
        umma_commit_pair_p(lead, &s.tmem_full[stage]);
        if (++stage == a.acc_stages) {
          stage = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp < 2 + 4 * a.epi_sets) {
    // ===================== epilogue (both CTAs, each its own 128 accumulator rows) =====================
    const int q = warp & 3;
    const int eset = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;
    const int epi_threads = 128 * a.epi_sets;
    const bool odd = lane & 1;
    const int row_elems = a.cout_p * a.out_planes;
    const int lo_off = (a.out_planes == 2 && !a.out_f8) ? a.cout_p : 0;
    int stage = 0, it = -1;
    uint32_t acc_phase = 0;
    PairFlags fl(a.flags, a.n_tiles, pair, n_pairs_grid, n_items, a.nt_magic);
    for (int item = pair; item < n_items; item += n_pairs_grid) {
      if (!fl.take(item)) continue;
      ++it;
      const int m0 = div_nt(item) * 256 + static_cast<int>(rank) * kBlockM;
      const int n_idx = item_n(item);
      const int n_cur = (n_idx == a.n_tiles - 1) ? a.n_last : a.n_tile;
      const int n_chunks = n_cur >> 4;
      const int n0 = n_idx * a.n_tile;
      float* bias_s = s.bias[it & 1];
      for (int i = et; i < n_cur; i += epi_threads) bias_s[i] = a.bias[n0 + i];
      asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
      bool valid = false, writable = false;
      int64_t out_row = 0;
      const int r_even = (m0 + 32 * q + lane) & ~1;
      if (r_even < a.rows_in) {
        const uint32_t pidx = static_cast<uint32_t>(r_even) >> 1;
        const int b = static_cast<int>((static_cast<unsigned long long>(pidx) * a.pair_magic) >> 40);
        const int tp = static_cast<int>(pidx) - b * a.half_lp;
        valid = tp < (__ldg(a.len0 + b) >> a.shift);
        writable = tp < a.Lp_out;
        out_row = static_cast<int64_t>(b) * a.Lp_out + tp;
      }
      mbar_wait(&s.tmem_full[stage], acc_phase);      // the accumulator is complete
      tc_fence_after();
      void* orow = a.out_fp32 ? static_cast<void*>(static_cast<float*>(a.out) + out_row * row_elems + n0)
                              : static_cast<void*>(static_cast<__half*>(a.out) + out_row * row_elems + n0);
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + stage * a.acc_cols;
      for (int c = eset; c < n_chunks; c += a.epi_sets) {
        uint32_t v[16];
        tmem_ld_32x16(t_addr + c * 16, v);
        tmem_ld_wait();
        uint8_t* f8_row = nullptr;
        if (a.out_f8) f8_row = static_cast<uint8_t*>(a.out) + out_row * row_elems * 2 + 2 * a.cout_p + n0;
        epilogue_chunk16(v, bias_s, c * 16, odd, valid, writable, orow, a.out_fp32, lo_off, a.w_inv_scale, f8_row,
                         a.cout_p);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_relaxed(&s.tmem_empty[stage][0], 0);   // on the leader's barrier
      if (++stage == a.acc_stages) {
        stage = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // the peer may still be read by the leader's MMAs / signalled until here
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------
// Per-layer activity flags of the M super-tiles: a super-tile is active when at least one of
// its row pairs has pooled index t' <= valid output length of its read (the "<=" keeps the
// zero row that terminates every read written).  Ragged batches and skipped reads (len 0)
// then cost only the tiles they really need.
__global__ void tile_activity_kernel(const int32_t* __restrict__ len0, ActivityArgs aa, uint8_t* __restrict__ flags) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= aa.total) return;
  int l = 0;
  while (l + 1 < aa.n_layers && idx >= aa.layer[l + 1].flag_off) ++l;
  const ActivityLayer L = aa.layer[l];
  const int sidx = idx - L.flag_off;
  const int row0 = sidx * L.rows_per_super;
  const int row1 = min(row0 + L.rows_per_super, L.rows_in);
  bool active = false;
  for (int b = row0 / L.Lp_in; !active && static_cast<int64_t>(b) * L.Lp_in < row1; ++b) {
    const int t_lo = max(row0 - b * L.Lp_in, 0);
    active = (t_lo >> 1) <= (len0[b] >> L.shift);
  }
  flags[idx] = active ? 1 : 0;
}

// ------------------------------------------------------------------------------------
// head: masked global average pool -> Linear(C, 2) -> softmax.  One CTA per read.
constexpr int kHeadThreads = 128;
__global__ void __launch_bounds__(kHeadThreads)
head_kernel(const float* __restrict__ act, const int32_t* __restrict__ len0, const float* __restrict__ fc_w,
            const float* __restrict__ fc_b, float* __restrict__ probs, float* __restrict__ feat, int B,
            int Lp, int cp, int c, int shift) {
  __shared__ float red[2][kHeadThreads / 32];
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int L = len0[b] >> shift;
  if (L <= 0) {   // shorter than 4096 samples: the reference raises in max_pool1d
    if (threadIdx.x == 0) {
      probs[2 * b] = nanf("");
      probs[2 * b + 1] = nanf("");
    }
    return;
  }
  const float* rows = act + static_cast<int64_t>(b) * Lp * cp;
  const float inv = 1.f / static_cast<float>(L);
  float l0 = 0.f, l1 = 0.f;
  for (int ch = threadIdx.x; ch < c; ch += kHeadThreads) {
    float sum = 0.f;
    for (int t = 0; t < L; ++t) sum += rows[static_cast<int64_t>(t) * cp + ch];
    const float f = sum * inv;
    if (feat) feat[static_cast<int64_t>(b) * c + ch] = f;
    l0 = fmaf(f, __ldg(fc_w + ch), l0);
    l1 = fmaf(f, __ldg(fc_w + c + ch), l1);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    l0 += __shfl_xor_sync(0xffffffffu, l0, d);
    l1 += __shfl_xor_sync(0xffffffffu, l1, d);
  }
  if (lane == 0) {
    red[0][warp] = l0;
    red[1][warp] = l1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    l0 = fc_b[0];
    l1 = fc_b[1];
    for (int w = 0; w < kHeadThreads / 32; ++w) {
      l0 += red[0][w];
      l1 += red[1][w];
    }
    const float m = fmaxf(l0, l1);
    const float e0 = expf(l0 - m), e1 = expf(l1 - m);
    const float inv_s = 1.f / (e0 + e1);
    probs[2 * b] = e0 * inv_s;
    probs[2 * b + 1] = e1 * inv_s;
  }
}

// ------------------------------------------------------------------------------------
// decision rule, riser/control.py:75-82
__global__ void decide_kernel(const float* __restrict__ probs, const int32_t* __restrict__ len, int B, int M,
                              float thr, int mode, int max_len, uint8_t* __restrict__ decision) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int n = len[b];
  if (n <= 0) {
    decision[b] = RISER_SKIPPED;
    return;
  }
  bool any_on = false, all_off = true;
  for (int m = 0; m < M; ++m) {
    const float p_off = probs[(static_cast<int64_t>(m) * B + b) * 2];
    const float p_on = probs[(static_cast<int64_t>(m) * B + b) * 2 + 1];
    any_on |= p_on > thr;
    all_off &= p_off > thr;
  }
  uint8_t d;
  if (any_on) d = (mode == RISER_MODE_ENRICH) ? RISER_ACCEPT : RISER_REJECT;
  else if (all_off) d = (mode == RISER_MODE_DEPLETE) ? RISER_ACCEPT : RISER_REJECT;
  else if (n >= max_len) d = RISER_NO_DECISION;
  else d = RISER_TRY_AGAIN;
  decision[b] = d;
}

// ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* fn) {
  static EncodeTiledFn cached = nullptr;
  if (!cached) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    RISER_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !p)
      return fail(RISER_ECUDA, "cuTensorMapEncodeTiled not available from the driver");
    cached = reinterpret_cast<EncodeTiledFn>(p);
  }
  *fn = cached;
  return RISER_OK;
}

// fp16 [rows][cols] row-major, zero OOB fill; box (64 cols = 128 B, box_rows) with SWIZZLE_128B,
// or (k32) box (32 cols = 64 B, box_rows) with SWIZZLE_64B
int make_tmap(CUtensorMap* tm, void* ptr, uint64_t cols, uint64_t rows, uint32_t box_rows, bool k32 = false) {
  EncodeTiledFn enc;
  int st = get_encode_fn(&enc);
  if (st) return st;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {cols * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(k32 ? 32 : kBlockK), box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptr, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, k32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(RISER_ECUDA, "cuTensorMapEncodeTiled failed (%d) for %llu x %llu box %u", static_cast<int>(r),
                static_cast<unsigned long long>(cols), static_cast<unsigned long long>(rows), box_rows);
  return RISER_OK;
}

// bytes [rows][cols] with row pitch `stride`, zero OOB fill; box (128 B or -- k32 -- 64 B, box_rows), swizzled alike
int make_tmap8(CUtensorMap* tm, void* ptr, uint64_t cols, uint64_t stride, uint64_t rows, uint32_t box_rows, bool k32) {
  EncodeTiledFn enc;
  int st = get_encode_fn(&enc);
  if (st) return st;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {stride};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(k32 ? 64 : 128), box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, ptr, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, k32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(RISER_ECUDA, "cuTensorMapEncodeTiled (bytes) failed (%d) for %llu x %llu box %u", static_cast<int>(r),
                static_cast<unsigned long long>(cols), static_cast<unsigned long long>(rows), box_rows);
  return RISER_OK;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

void plan_lengths(const riser_model* m, int max_len, int* Lmax, int* Lp) {
  Lmax[0] = max_len;
  Lp[0] = 0;
  for (int i = 1; i <= m->n_layers; ++i) {
    Lmax[i] = Lmax[i - 1] / 2;
    Lp[i] = round_up(Lmax[i] + 1, 2);
  }
}

size_t plan_offsets(const riser_model* m, int B, const int* Lp, size_t* off) {
  size_t cur = 0;
  for (int i = 1; i <= m->n_layers; ++i) {
    off[i] = cur;
    const bool last = (i == m->n_layers);
    const size_t elt = last ? 4 : 2;
    const size_t planes = last ? 1 : m->act_planes;
    cur += align_up(static_cast<size_t>(B) * Lp[i] * m->layer[i - 1].cout_p * planes * elt, 1024);
  }
  return cur;
}

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

constexpr int kABoxRows = 136;                               // haloed A tile rows: 130 needed; TMA likes multiples of 8
constexpr size_t kSmemFixed = 1024 + sizeof(ConvSmem) + 64;  // beside a conv kernel's rings: alignment slack, ConvSmem

// Layer i's K blocks and the shared-memory budgets both steps test.  Narrow layers take 32-channel K blocks (64-byte
// rows, SWIZZLE_64B): no zero-filled half rows, twice the pipeline depth / sub-tiles per item in the same memory.
struct LayerBudget {
  bool k32, tc_resident, eo_fits, pair_resident;   // all weights (pair: each CTA's half) stay in shared memory
  int row_bytes, kplanes, kb16, k_blocks, eo_acc, pair_n;   // kplanes: A tiles per K block; eo_acc: [even | odd] TMEM
  size_t avail, b_bytes, w_all, a_group1, eo_group1;   // beside kSmemFixed; weight tile(s); a K block's A / E + O tiles
  size_t pair_a, pair_hb, pair_hw;                 // conv_pair_kernel: A tile; a CTA's half of a weight tile, of all
};
LayerBudget layer_budget(const riser_model* m, int i, int max_smem) {
  const LayerPack& L = m->layer[i];
  LayerBudget g;
  g.k32 = L.cin_p <= 80;
  g.row_bytes = g.k32 ? 64 : 128;
  g.kplanes = L.f8 ? 1 : m->act_planes;
  g.kb16 = (L.cin_p + g.row_bytes / 2 - 1) / (g.row_bytes / 2);
  g.k_blocks = g.kb16 + (L.f8 ? (2 * L.cin_p + g.row_bytes - 1) / g.row_bytes : 0);
  g.eo_acc = round_up(2 * L.n_tile, 32);
  g.pair_n = std::min(kMaxNTile, L.cout_p);
  g.avail = static_cast<size_t>(max_smem) - kSmemFixed;
  g.b_bytes = static_cast<size_t>(L.n_tile) * g.row_bytes;
  g.w_all = static_cast<size_t>(L.passes) * 3 * g.k_blocks * g.b_bytes;
  g.a_group1 = static_cast<size_t>(g.kplanes) * kABoxRows * g.row_bytes;
  g.eo_group1 = static_cast<size_t>(m->act_planes) * 2 * kEoTile;
  g.pair_a = static_cast<size_t>(kABoxRows) * 128;
  g.pair_hb = static_cast<size_t>(g.pair_n / 2) * 128;
  g.pair_hw = static_cast<size_t>(3) * g.k_blocks * g.pair_hb;
  g.tc_resident = L.n_tiles == 1 && g.w_all + 2 * g.a_group1 <= g.avail;
  g.eo_fits = g.w_all + 2 * g.eo_group1 <= g.avail;
  g.pair_resident = L.n_tiles == 1 && g.pair_hw + 3 * g.pair_a <= g.avail;
  return g;
}
void choose_kernels(riser_plan* p, int max_smem) {
  const riser_model* m = p->model;
  // These switches exist so that the test suite can reach, on the shipped network, the kernels that other shapes
  // select on their own.
  const bool fuse_l0 = env_int("RISER_FUSE_L0", 1) != 0, eo_on = env_int("RISER_EO", 1) != 0;
  const bool pair_on = env_int("RISER_PAIR", 1) != 0, kc_on = env_int("RISER_KC", 1) != 0;
  const bool fuse23 = env_int("RISER_FUSE23", 1) != 0;
  constexpr int kPairFrom = 6;
  for (int i = 1; i < m->n_layers; ++i) {
    const LayerPack& L = m->layer[i];
    const LayerBudget g = layer_budget(m, i, max_smem);
    const bool last = (i == m->n_layers - 1);
    LayerPlan& lp = p->layer[i];
    // fused01_kernel stores fp16 rows only: a last layer (the head reads fp32) runs as layer0_kernel + conv_tc_kernel
    if (i == 1 && fuse_l0 && !last && L.cin_p == 32 && L.n_tile == 32 && L.n_tiles == 1 && m->layer[0].cout <= 24) {
      lp.kind = kFused01Kernel;
      lp.kc = (L.wkc && m->layer[0].cout <= 20 && kc_on) ? 1 : 0;
      p->fuse_l0 = 1;
    } else if (eo_on && i >= 2 && i <= 4 && !last && !L.f8 && L.cin_p <= 80 && L.n_tiles == 1 &&
               2 * L.n_tile <= kMaxNTile && g.eo_fits) {   // the narrow resident-weight layers 2..4
      lp.kind = kEoKernel;
      lp.eo = 1;
    } else if (pair_on && L.f8 && !g.tc_resident && !g.k32 && (L.n_tile % 16) == 0 &&
               (i >= kPairFrom || g.pair_resident)) {
      // CTA pairs take the streamed-weight F16_F8 layers from layer kPairFrom on, and earlier ones (layer 5 of the
      // shipped network) only when each CTA's half of the weights stays resident
      lp.kind = kPairKernel;
    }
  }
  // Two consecutive even / odd layers as ONE launch (conv_eo2_kernel): the first such pair (layers 2 + 3 of the shipped
  // network), when both are hi + lo plane layers, the accumulators fit the TMEM and everything fits shared memory.
  for (int i = 2; fuse23 && m->act_planes == 2 && i + 1 < m->n_layers - 1; ++i) {
    const LayerPack &L1 = m->layer[i], &L2 = m->layer[i + 1];
    const LayerBudget g1 = layer_budget(m, i, max_smem), g2 = layer_budget(m, i + 1, max_smem);
    if (p->layer[i].eo && p->layer[i + 1].eo && L1.passes == 2 && L2.passes == 2 && !L1.f8 && !L2.f8 &&
        3 * g1.eo_acc + g2.eo_acc <= kTmemCols && L1.n_tile <= 128 && L2.n_tile <= 128 &&
        conv_eo2_smem(L1.n_tile, L2.n_tile, g1.k_blocks, g2.k_blocks) <= static_cast<size_t>(max_smem)) {
      p->layer[i].kind = p->layer[i + 1].kind = kEo2Kernel;
      p->layer[i + 1].fused_prev = 1;
      break;
    }
  }
}
// The ConvArgs fields all conv kernels share: lengths, K and N tiling, output format and layout, pointers
ConvArgs conv_args(const riser_plan* p, int i, const LayerBudget& g, int m_rows, int n_tile) {
  const LayerPack& L = p->model->layer[i];
  const bool last = (i == p->model->n_layers - 1);
  ConvArgs a = {};
  a.bias = L.bias;
  a.out = p->ws + p->act_off[i + 1];
  a.rows_in = p->B * p->Lp[i];
  a.Lp_in = p->Lp[i];
  a.Lp_out = p->Lp[i + 1];
  a.half_lp = p->Lp[i] / 2;
  a.half_lp_out = p->Lp[i + 1] / 2;
  a.n_pairs_out = p->B * p->Lp[i + 1] / 2;
  a.pair_magic = ((1ull << 40) / static_cast<unsigned long long>(a.half_lp)) + 1ull;
  a.shift = i + 1;
  a.cin_p = L.cin_p;
  a.cout_p = L.cout_p;
  a.kb16 = g.kb16;
  a.k_blocks = g.k_blocks;
  a.k32 = g.k32 ? 1 : 0;
  a.f8 = L.f8;
  a.planes = g.kplanes;
  a.wplanes = L.passes;
  a.a_tx_bytes = kABoxRows * g.row_bytes;
  a.n_tile = n_tile;
  a.n_tiles = (L.cout_p + n_tile - 1) / n_tile;
  a.idesc = umma_idesc_f16(m_rows, n_tile);
  a.w_inv_scale = L.w_inv_scale;
  a.out_fp32 = last ? 1 : 0;
  a.out_planes = last ? 1 : p->model->act_planes;
  a.out_f8 = (!last && p->model->layer[i + 1].f8) ? 1 : 0;   // the epilogue writes the format the next layer reads
  a.out_eo = (!last && p->layer[i + 1].eo) ? 1 : 0;           // ... and the row layout it reads
  a.epi_sets = kMaxEpiSets;
  return a;
}
// Weight maps (box_rows rows): fp16 [plane][tap][cout_p][cin_p]; e4m3 [tap][cout_p][2 cin_p], or a copy when not F16_F8
int weight_maps(CUtensorMap* b, CUtensorMap* b8, const LayerPack& L, uint32_t box_rows, bool k32) {
  const int st = make_tmap(b, L.w, L.cin_p, static_cast<uint64_t>(L.passes) * 3 * L.cout_p, box_rows, k32);
  if (!st && L.f8) return make_tmap8(b8, L.w8, 2ull * L.cin_p, 2ull * L.cin_p, 3ull * L.cout_p, box_rows, k32);
  *b8 = *b;
  return st;
}
int flat_maps(LayerPlan& lp, const riser_plan* p, int i, uint32_t b_rows, bool k32) {
  const LayerPack& L = p->model->layer[i];
  char* act = p->ws + p->act_off[i];
  const int rows = p->B * p->Lp[i];
  int st = make_tmap(&lp.tm_a, act, static_cast<uint64_t>(L.cin_p) * p->model->act_planes, rows, kABoxRows, k32);
  if (!st && L.f8) st = make_tmap8(&lp.tm_a8, act, 4ull * L.cin_p, 4ull * L.cin_p, rows, kABoxRows, k32);
  else lp.tm_a8 = lp.tm_a;
  return st ? st : weight_maps(&lp.tm_b, &lp.tm_b8, L, b_rows, k32);
}
int configure_tc(riser_plan* p, int i, const LayerBudget& g, const void** fn) {
  const LayerPack& L = p->model->layer[i];
  LayerPlan& lp = p->layer[i];
  ConvArgs& a = lp.args = conv_args(p, i, g, kBlockM, L.n_tile);
  a.acc_cols = round_up(L.n_tile, 32);
  a.resident = g.tc_resident ? 1 : 0;
  if (a.resident) {
    // the most 128-row sub-tiles per item that leave >= 2 accumulator stages and A groups (amortises per-item work)
    for (a.ms = 4; a.ms > 1; a.ms >>= 1)
      if (2 * a.ms * a.acc_cols <= kTmemCols && g.w_all + 2 * a.ms * g.a_group1 <= g.avail &&
          static_cast<int64_t>(a.rows_in) / (a.ms * kBlockM) >= 2 * p->model->sm_count)
        break;
    a.b_stages = 1;
    a.a_stages = std::min<int>(kMaxAStages, static_cast<int>((g.avail - g.w_all) / (a.ms * g.a_group1)));
    lp.smem = kSmemFixed + g.w_all + static_cast<size_t>(a.a_stages) * a.ms * g.a_group1;
  } else {
    a.ms = (2 * a.acc_cols <= kTmemCols) ? 2 : 1;
    if (4 * a.acc_cols <= kTmemCols && 2 * 4 * g.a_group1 + 3 * g.b_bytes <= g.avail)
      a.ms = 4;       // more rows per streamed weight tile (narrow layers / 32-channel K blocks)
    // smem split: at least 2 A groups and 2 B stages; a third A group when that still leaves 4+ B stages
    while (a.ms > 1 && 2 * a.ms * g.a_group1 + 2 * g.b_bytes > g.avail) a.ms >>= 1;
    const size_t a_group = a.ms * g.a_group1;
    a.a_stages = (static_cast<int>((g.avail - 2 * a_group) / g.b_bytes) > 4 && 3 * a_group + 4 * g.b_bytes <= g.avail)
                     ? 3 : 2;
    a.b_stages = std::max(2, std::min(kMaxBStages, static_cast<int>((g.avail - a.a_stages * a_group) / g.b_bytes)));
    lp.smem = kSmemFixed + static_cast<size_t>(a.a_stages) * a_group + static_cast<size_t>(a.b_stages) * g.b_bytes;
  }
  a.acc_stages = std::max(1, std::min(kMaxAccStages, kTmemCols / (a.ms * a.acc_cols)));
  a.dual = (a.ms == 2 && !a.resident) ? 1 : 0;
  lp.rows_per_super = a.ms * kBlockM;
  lp.block = 64 + 128 * a.epi_sets + (a.dual ? 32 : 0);
  lp.fn.tc = pick_conv_kernel(a.ms, a.planes, a.wplanes, a.resident, a.k32, a.f8);
  *fn = reinterpret_cast<const void*>(lp.fn.tc);
  return flat_maps(lp, p, i, L.n_tile, g.k32);
}
// layers 0 + 1 on the tensor pipe: work item = 255 pooled outputs = 510 input rows
int configure_fused01(riser_plan* p, const LayerBudget& g, const void** fn) {
  const riser_model* m = p->model;
  const LayerPack& L = m->layer[1];
  LayerPlan& lp = p->layer[1];
  ConvArgs& a = lp.args = conv_args(p, 1, g, kBlockM, L.n_tile);
  a.w0 = m->layer[0].w0;
  a.b0 = m->layer[0].bias;
  a.cout0 = m->layer[0].cout;
  lp.rows_per_super = 2 * kF2Pairs;
  lp.smem = fused01_smem(m->act_planes, L.f8 ? 2 : L.passes);
  lp.fn.fused01 = pick_fused01(lp.kc ? 4 : L.f8 ? 3 : (m->act_planes == 2 ? 2 : (L.passes == 2 ? 1 : 0)));
  lp.block = kF2Threads;
  *fn = reinterpret_cast<const void*>(lp.fn.fused01);
  // kc: the three hi / lo terms concatenated along K, [tap][cout_p][64]; same shared-memory footprint
  if (lp.kc) return make_tmap(&lp.tm_b, L.wkc, 64, 3ull * L.cout_p, 32, false);
  return weight_maps(&lp.tm_b, &lp.tm_b8, L, L.n_tile, true);
}
// conv_eo_kernel; the launch of a conv_eo2_kernel pair reads both layers' maps and arguments (not their launch fields)
int configure_eo(riser_plan* p, int i, const LayerBudget& g, const void** fn) {
  const LayerPack& L = p->model->layer[i];
  LayerPlan& lp = p->layer[i];
  ConvArgs& a = lp.args = conv_args(p, i, g, kBlockM, L.n_tile);
  a.acc_cols = g.eo_acc;
  a.ms = (2 * 2 * a.acc_cols <= kTmemCols && g.w_all + 2 * 2 * g.eo_group1 <= g.avail) ? 2 : 1;
  a.a_stages = std::min<int>(kMaxAStages, static_cast<int>((g.avail - g.w_all) / (a.ms * g.eo_group1)));
  a.acc_stages = std::max(1, std::min(kMaxAccStages, kTmemCols / (a.ms * a.acc_cols)));
  lp.rows_per_super = a.ms * 2 * kBlockM;
  if (lp.kind == kEoKernel) {
    lp.smem = kSmemFixed + g.w_all + static_cast<size_t>(a.a_stages) * a.ms * g.eo_group1;
    lp.block = 64 + 128 * a.epi_sets;
    *fn = reinterpret_cast<const void*>(lp.fn.eo = pick_conv_eo(a.ms, a.planes, a.wplanes));
  }
  // E plane = rows [0, n_pairs), O plane = rows [n_pairs, 2 n_pairs) of the same buffer
  const uint64_t n_pairs = a.rows_in / 2, pitch = static_cast<uint64_t>(L.cin_p) * p->model->act_planes;   // fp16 / row
  int st = make_tmap(&lp.tm_a, p->ws + p->act_off[i], pitch, n_pairs, kABoxRows, true);
  if (!st) st = make_tmap(&lp.tm_a8, p->ws + p->act_off[i] + n_pairs * pitch * 2, pitch, n_pairs, kABoxRows, true);
  return st ? st : weight_maps(&lp.tm_b, &lp.tm_b8, L, L.n_tile, true);
}
// layers i and i + 1, each with its configure_eo arguments, as one conv_eo2_kernel launch
void configure_eo2(riser_plan* p, int i, const void** fn) {
  LayerPlan& l1 = p->layer[i];
  const ConvArgs &a1 = l1.args, &a2 = p->layer[i + 1].args;
  Eo2Args& e = l1.eo2;
  e.kb1 = a1.k_blocks;
  e.kb2 = a2.k_blocks;
  e.n1 = a1.n_tile;
  e.n2 = a2.n_tile;
  e.acc1 = a1.acc_cols;
  e.acc2 = a2.acc_cols;
  e.bias1 = a1.bias;
  e.bias2 = a2.bias;
  e.out = a2.out;
  e.B = p->B;
  e.Lp_out = a2.Lp_out;
  e.n_seg = (e.Lp_out + kE2Rows - 1) / kE2Rows;
  e.half_lp_in = a1.half_lp;
  e.half_lp_out = a2.half_lp_out;
  e.n_pairs_out = a2.n_pairs_out;
  e.out_eo = a2.out_eo;
  e.out_f8 = a2.out_f8;
  e.out_planes = a2.out_planes;
  e.cout_p2 = a2.cout_p;
  e.shift1 = a1.shift;
  e.shift2 = a2.shift;
  e.cin_p1 = a1.cin_p;
  e.idesc1_n = a1.idesc;
  e.idesc1_2n = umma_idesc_f16(kBlockM, 2 * e.n1);
  e.idesc2_n = a2.idesc;
  e.idesc2_2n = umma_idesc_f16(kBlockM, 2 * e.n2);
  e.inv_scale1 = a1.w_inv_scale;
  e.inv_scale2 = a2.w_inv_scale;
  l1.grid = std::min(e.B * e.n_seg, p->model->sm_count);
  l1.smem = conv_eo2_smem(e.n1, e.n2, e.kb1, e.kb2);
  l1.block = kE2Threads;
  *fn = reinterpret_cast<const void*>(l1.fn.eo2 = conv_eo2_kernel);
}
// conv_pair_kernel: M = 256 over two CTAs, each holds 128 rows of A and half of every weight tile
int configure_pair(riser_plan* p, int i, const LayerBudget& g, const void** fn) {
  const LayerPack& L = p->model->layer[i];
  LayerPlan& lp = p->layer[i];
  // N tiles 256 wide (the widest M = 256 MMA: fewest shared-memory operand bytes per MAC) with ONE narrower last tile
  // instead of equal tiles -- cout_p itself (the next layer's K) is unchanged
  ConvArgs& a = lp.args = conv_args(p, i, g, 256, g.pair_n);
  a.n_last = L.cout_p - (a.n_tiles - 1) * a.n_tile;
  a.idesc_last = umma_idesc_f16(256, a.n_last);
  // item / n_tiles by multiply-high; with one N tile the magic would overflow, and the kernel divides instead
  a.nt_magic = a.n_tiles > 1 ? static_cast<uint32_t>((1ull << 32) / static_cast<unsigned>(a.n_tiles)) + 1u : 0u;
  a.acc_cols = round_up(a.n_tile, 32);
  // One 256-row sub-tile per item and two accumulator stages: layers 6-11 in situ 0.38 / 0.47 / 0.37 / 0.38 / 0.46 /
  // 0.49 ms, against 0.41 / 0.47 / 0.40 / 0.43 / 0.48 / 0.55 with two sub-tiles (they leave the TMEM one item deep)
  a.ms = 1;
  int a_st = 5;         // A stages beside streamed weights (the kernel sets up b_stages even when they are resident)
  while (a_st > 2 && a_st * g.pair_a + 4 * g.pair_hb > g.avail) --a_st;
  a.b_stages = std::max(2, std::min<int>(kMaxBStages, static_cast<int>((g.avail - a_st * g.pair_a) / g.pair_hb)));
  a.acc_stages = std::max(1, std::min(kMaxAccStages, kTmemCols / a.acc_cols));
  a.resident = g.pair_resident ? 1 : 0;
  a.a_stages = a.resident ? std::min<int>(kMaxAStages, static_cast<int>((g.avail - g.pair_hw) / g.pair_a)) : a_st;
  lp.rows_per_super = 256;
  lp.smem = kSmemFixed + a.a_stages * g.pair_a + (a.resident ? g.pair_hw : a.b_stages * g.pair_hb);
  lp.block = 64 + 128 * a.epi_sets;
  *fn = reinterpret_cast<const void*>(lp.fn.pair = conv_pair_kernel);
  const int st = flat_maps(lp, p, i, a.n_tile / 2, false);
  return st ? st : weight_maps(&lp.tm_bl, &lp.tm_b8l, L, a.n_last / 2, false);
}
}  // namespace
}  // namespace riser

using namespace riser;

extern "C" int riser_model_create(riser_model** out, int n_layers, const int* channels,
                                  const float* const* conv_w, const float* const* conv_b, const float* fc_w,
                                  const float* fc_b, int precision, int device) {
  RISER_REQUIRE(out && channels && conv_w && conv_b && fc_w && fc_b, "riser_model_create: null pointer");
  RISER_REQUIRE(n_layers >= 2 && n_layers <= kMaxLayers, "riser_model_create: n_layers %d outside [2, %d]",
                n_layers, kMaxLayers);
  RISER_REQUIRE(precision >= RISER_PREC_F16 && precision <= RISER_PREC_F16_F8,
                "riser_model_create: unknown precision %d", precision);
  RISER_REQUIRE(channels[0] <= 64, "riser_model_create: layer 0 supports at most 64 output channels");
  // the caller's current device is left as it was (several models / GPUs per process: shard.py)
  struct DeviceGuard {
    int prev = -1;
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  } guard;
  RISER_CUDA_TRY(cudaGetDevice(&guard.prev));
  RISER_CUDA_TRY(cudaSetDevice(device));
  int major = 0;
  RISER_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(RISER_ECUDA, "device %d is sm_%dx; riser_b200 needs sm_100", device, major);

  riser_model* m = new riser_model();
  m->n_layers = n_layers;
  m->precision = precision;
  m->f8 = (precision == RISER_PREC_F16_F8) ? 1 : 0;
  m->passes = (precision == RISER_PREC_F16 || m->f8) ? 1 : 2;  // fp16 weight planes (hi [, lo])
  m->act_planes = (precision == RISER_PREC_F16_X3 || m->f8) ? 2 : 1;   // activation planes (hi [, lo])
  m->f8_from = std::max(1, env_int("RISER_F8_FROM", 5));
  m->device = device;
  cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device);
  int cin = 1, cin_p = 1;
  for (int i = 0; i < n_layers; ++i) {
    LayerPack& L = m->layer[i];
    L.cin = cin;
    L.cout = channels[i];
    L.cin_p = cin_p;
    L.f8 = (m->f8 && i >= m->f8_from) ? 1 : 0;
    L.passes = m->f8 ? (L.f8 ? 1 : 2) : m->passes;
    L.n_tile = (i == 0) ? round_up(L.cout, 16) : pick_n_tile(L.cout);
    L.cout_p = round_up(L.cout, L.n_tile);
    L.n_tiles = L.cout_p / L.n_tile;
    std::vector<float> bias(L.cout_p, 0.f);
    std::memcpy(bias.data(), conv_b[i], sizeof(float) * L.cout);
    RISER_CUDA_TRY(cudaMalloc(&L.bias, sizeof(float) * L.cout_p));
    RISER_CUDA_TRY(cudaMemcpy(L.bias, bias.data(), sizeof(float) * L.cout_p, cudaMemcpyHostToDevice));
    if (i == 0) {
      RISER_CUDA_TRY(cudaMalloc(&L.w0, sizeof(float) * L.cout * 3));
      RISER_CUDA_TRY(cudaMemcpy(L.w0, conv_w[0], sizeof(float) * L.cout * 3, cudaMemcpyHostToDevice));
    } else {
      // [plane][tap][cout_p][cin_p]: tap-major so that one 2-D tensor map serves all taps
      const size_t per_pass = static_cast<size_t>(3) * L.cout_p * L.cin_p;
      std::vector<__half> w(per_pass * L.passes, __float2half(0.f));
      std::vector<uint8_t> w8(L.f8 ? 2 * per_pass : 0, 0);
      const float* src = conv_w[i];   // [cout][cin][3]
      float wmax = 0.f;
      for (size_t k = 0; k < static_cast<size_t>(L.cout) * L.cin * 3; ++k) wmax = std::max(wmax, std::fabs(src[k]));
      int e = 0;
      if (wmax > 0.f && std::isfinite(wmax)) {
        std::frexp(wmax, &e);          // wmax = f * 2^e, f in [0.5, 1)
        e = 12 - e;                    // scaled max magnitude in [2^11, 2^12)
        e = std::max(-24, std::min(24, e));
      }
      const float scale = std::ldexp(1.f, e);
      L.w_inv_scale = std::ldexp(1.f, -e);
      for (int co = 0; co < L.cout; ++co)
        for (int ci = 0; ci < L.cin; ++ci)
          for (int tap = 0; tap < 3; ++tap) {
            const float v = src[(static_cast<size_t>(co) * L.cin + ci) * 3 + tap] * scale;
            const __half hi = __float2half_rn(v);
            const size_t idx = (static_cast<size_t>(tap) * L.cout_p + co) * L.cin_p + ci;
            w[idx] = hi;
            if (L.passes == 2) w[per_pass + idx] = __float2half_rn(v - __half2float(hi));
            if (L.f8) {   // correction operands: [W_lo * 2^3 | W * 2^-9] e4m3 (pair with a8 and lo8, store_f8_planes)
              const size_t i8 = (static_cast<size_t>(tap) * L.cout_p + co) * (2 * L.cin_p) + ci;
              w8[i8] = __nv_cvt_float_to_fp8((v - __half2float(hi)) * (1.f / kF8AScale), __NV_SATFINITE, __NV_E4M3);
              w8[i8 + L.cin_p] = __nv_cvt_float_to_fp8(v * (1.f / kF8LoScale), __NV_SATFINITE, __NV_E4M3);
            }
          }
      if (L.f8) {
        RISER_CUDA_TRY(cudaMalloc(&L.w8, w8.size()));
        RISER_CUDA_TRY(cudaMemcpy(L.w8, w8.data(), w8.size(), cudaMemcpyHostToDevice));
      }
      RISER_CUDA_TRY(cudaMalloc(&L.w, sizeof(__half) * w.size()));
      RISER_CUDA_TRY(cudaMemcpy(L.w, w.data(), sizeof(__half) * w.size(), cudaMemcpyHostToDevice));
      if (i == 1 && L.passes == 2 && m->act_planes == 2 && !L.f8 && L.cin <= 20 && (L.cin & 1) == 0 && L.cout_p == 32) {
        // K-concatenated operand of fused01_kernel<4>: input channel ci at k = ci (x a_hi), 20 + ci (x a_lo), 40 + ci (x a_hi)
        std::vector<__half> kc(static_cast<size_t>(3) * L.cout_p * 64, __float2half(0.f));
        for (int tap = 0; tap < 3; ++tap)
          for (int co = 0; co < L.cout; ++co)
            for (int ci = 0; ci < L.cin; ++ci) {
              const size_t idx = (static_cast<size_t>(tap) * L.cout_p + co) * L.cin_p + ci;
              __half* row = kc.data() + (static_cast<size_t>(tap) * L.cout_p + co) * 64;
              row[ci] = w[idx];
              row[20 + ci] = w[idx];
              row[40 + ci] = w[per_pass + idx];
            }
        RISER_CUDA_TRY(cudaMalloc(&L.wkc, sizeof(__half) * kc.size()));
        RISER_CUDA_TRY(cudaMemcpy(L.wkc, kc.data(), sizeof(__half) * kc.size(), cudaMemcpyHostToDevice));
      }
    }
    cin = L.cout;
    cin_p = L.cout_p;
  }
  m->c_last = channels[n_layers - 1];
  RISER_CUDA_TRY(cudaMalloc(&m->fc_w, sizeof(float) * 2 * m->c_last));
  RISER_CUDA_TRY(cudaMemcpy(m->fc_w, fc_w, sizeof(float) * 2 * m->c_last, cudaMemcpyHostToDevice));
  RISER_CUDA_TRY(cudaMalloc(&m->fc_b, sizeof(float) * 2));
  RISER_CUDA_TRY(cudaMemcpy(m->fc_b, fc_b, sizeof(float) * 2, cudaMemcpyHostToDevice));
  *out = m;
  return RISER_OK;
}

extern "C" int riser_model_destroy(riser_model* m) {
  if (!m) return RISER_OK;
  for (int i = 0; i < m->n_layers; ++i) {
    cudaFree(m->layer[i].w);
    cudaFree(m->layer[i].w8);
    cudaFree(m->layer[i].wkc);
    cudaFree(m->layer[i].w0);
    cudaFree(m->layer[i].bias);
  }
  cudaFree(m->fc_w);
  cudaFree(m->fc_b);
  delete m;
  return RISER_OK;
}

extern "C" size_t riser_workspace_bytes(const riser_model* m, int B, int max_len) {
  if (!m || B <= 0 || max_len <= 0) return 0;
  int Lmax[kMaxLayers + 1], Lp[kMaxLayers + 1];
  size_t off[kMaxLayers + 1];
  plan_lengths(m, max_len, Lmax, Lp);
  return plan_offsets(m, B, Lp, off);
}

// Two steps: choose_kernels picks the kernel of every conv layer, then that kernel's configure_* function fills in its
// arguments, tensor maps, shared memory, block and kernel pointer.  Both steps test the budgets of layer_budget.
extern "C" int riser_plan_create(riser_plan** out, const riser_model* m, int B, int max_len, void* workspace,
                                 size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(out && m && workspace, "riser_plan_create: null pointer");
  RISER_REQUIRE(B > 0 && max_len >= kMinLen, "riser_plan_create: need B > 0 and max_len >= %d", kMinLen);
  RISER_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "riser_plan_create: workspace not 256-byte aligned");
  std::unique_ptr<riser_plan, int (*)(riser_plan*)> owner(new riser_plan(), riser_plan_destroy);   // freed on every error return
  riser_plan* p = owner.get();
  p->model = m;
  p->B = B;
  p->max_len = max_len;
  p->ws = static_cast<char*>(workspace);
  int Lmax[kMaxLayers + 1];
  plan_lengths(m, max_len, Lmax, p->Lp);
  const size_t need = plan_offsets(m, B, p->Lp, p->act_off);
  if (workspace_bytes < need)
    return fail(RISER_ENOMEM, "riser_plan_create: workspace %zu < %zu bytes", workspace_bytes, need);
  RISER_REQUIRE(static_cast<int64_t>(B) * p->Lp[1] * 8 < (int64_t(1) << 31), "riser_plan_create: B * L too large");
  RISER_CUDA_TRY(cudaMemsetAsync(workspace, 0, need, as_stream(stream)));
  int max_smem = 0;
  RISER_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, m->device));

  choose_kernels(p, max_smem);
  for (int i = 1; i < m->n_layers; ++i) {
    LayerPlan& lp = p->layer[i];
    const LayerBudget g = layer_budget(m, i, max_smem);
    const void* fn = nullptr;      // the kernel this layer launches, if any
    const int st = lp.kind == kFused01Kernel ? configure_fused01(p, g, &fn)
                   : lp.kind == kPairKernel  ? configure_pair(p, i, g, &fn)
                   : lp.kind == kTcKernel    ? configure_tc(p, i, g, &fn)
                                             : configure_eo(p, i, g, &fn);   // also both conv_eo2_kernel layers
    if (st) return st;
    if (lp.fused_prev) configure_eo2(p, i - 1, &fn);   // once the second layer has its arguments
    // every launch covers the whole batch
    ConvArgs& a = lp.args;
    a.n_supers = (a.rows_in + lp.rows_per_super - 1) / lp.rows_per_super;
    if (lp.kind == kPairKernel) lp.grid = std::min(2 * a.n_supers * a.n_tiles, m->sm_count & ~1);
    else if (lp.kind != kEo2Kernel) lp.grid = std::min(a.n_supers * a.n_tiles, m->sm_count);
    if (fn) RISER_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    // tile activity flags (ragged batches / skipped reads): one byte per M super-tile and layer
    p->activity.layer[p->activity.n_layers++] = {a.Lp_in, a.rows_in, lp.rows_per_super, a.shift, a.n_supers,
                                                 p->activity.total};
    p->activity.total += a.n_supers;
  }
  RISER_CUDA_TRY(cudaMalloc(&p->flags, p->activity.total));
  for (int i = 1; i < m->n_layers; ++i) {
    LayerPlan& lp = p->layer[i];
    // fused01_kernel stages its CTA's flags in shared memory; past kF2MaxLocalItems items per CTA it runs every item
    if (lp.kind != kFused01Kernel || (lp.args.n_supers + lp.grid - 1) / lp.grid <= kF2MaxLocalItems)
      lp.args.flags = p->flags + p->activity.layer[i - 1].flag_off;
  }
  *out = owner.release();
  return RISER_OK;
}

extern "C" int riser_plan_destroy(riser_plan* p) {
  if (p) cudaFree(p->flags);
  delete p;
  return RISER_OK;
}

extern "C" int riser_forward_launches(const riser_plan* p) {
  if (!p) return 0;
  // tile_activity_kernel, layer 0, the conv layers and the head, less the layers computed inside another launch
  int inside = p->fuse_l0;
  for (int i = 1; i < p->model->n_layers; ++i) inside += p->layer[i].fused_prev;
  return p->model->n_layers + 2 - inside;
}

extern "C" int riser_plan_fused_layer0(const riser_plan* p) { return p ? p->fuse_l0 : 0; }

extern "C" int riser_plan_layer_eo(const riser_plan* p, int i) {
  return (p && i >= 1 && i < p->model->n_layers) ? p->layer[i].eo : 0;
}

extern "C" int riser_plan_layer_format(const riser_plan* p, int i) {
  if (!p || i < 1 || i >= p->model->n_layers) return 0;
  if (p->layer[i].fused_prev) return -1;      // never materialised: computed inside the previous layer's launch
  if (p->model->layer[i].f8) return 3;
  return p->model->act_planes == 2 ? 2 : 1;
}

extern "C" int riser_plan_layer_kernel(const riser_plan* p, int i) {
  if (!p || i < 1 || i >= p->model->n_layers) return -1;
  return p->layer[i].kind;
}

extern "C" int riser_plan_layer_info(const riser_plan* p, int i, int64_t* offset, int* rows_per_read,
                                     int* channels_padded, int* channels, int* n_tile) {
  RISER_REQUIRE(p && offset && rows_per_read && channels_padded && channels && n_tile,
                "riser_plan_layer_info: null pointer");
  RISER_REQUIRE(i >= 1 && i <= p->model->n_layers, "riser_plan_layer_info: layer %d out of range", i);
  *offset = static_cast<int64_t>(p->act_off[i]);
  *rows_per_read = p->Lp[i];
  *channels_padded = p->model->layer[i - 1].cout_p * (i == p->model->n_layers ? 1 : p->model->act_planes);
  *channels = p->model->layer[i - 1].cout;
  *n_tile = p->model->layer[i - 1].n_tile;
  return RISER_OK;
}

namespace riser {
namespace {

int launch_layer0(const riser_plan* p, const float* x, int64_t ld_x, const int32_t* len, cudaStream_t st) {
  const riser_model* m = p->model;
  if (p->fuse_l0) return RISER_OK;       // computed inside layer 1's kernel
  const LayerPack& L = m->layer[0];
  const int64_t total = static_cast<int64_t>(p->B) * p->Lp[1] * (L.cout_p / 8);
  const int grid = static_cast<int>(std::min<int64_t>((total + 255) / 256, static_cast<int64_t>(m->sm_count) * 32));
  __half* out = reinterpret_cast<__half*>(p->ws + p->act_off[1]);
  layer0_kernel<<<grid, 256, 0, st>>>(x, ld_x, len, L.w0, L.bias, out, p->B, p->Lp[1], L.cout, L.cout_p,
                                      m->act_planes, m->layer[1].f8);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

// conv layer i, through the kernel the plan chose for it
int launch_conv(const riser_plan* p, int i, const float* x, int64_t ld_x, const int32_t* len, cudaStream_t st) {
  const LayerPlan& lp = p->layer[i];
  if (lp.fused_prev) return RISER_OK;      // computed inside layer i - 1's launch
  ConvArgs a = lp.args;
  a.len0 = len;
  switch (lp.kind) {
    case kEo2Kernel: {
      Eo2Args e = lp.eo2;
      e.len0 = len;
      lp.fn.eo2<<<lp.grid, lp.block, lp.smem, st>>>(lp.tm_a, lp.tm_a8, lp.tm_b, p->layer[i + 1].tm_b, e);
      break;
    }
    case kFused01Kernel:
      RISER_REQUIRE(x, "riser_forward: null x");
      RISER_REQUIRE((ld_x & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0,
                    "riser_forward: x must be 16-byte aligned with ld_x a multiple of 4 (bulk copies of the signal)");
      a.x = x;
      a.ld_x = ld_x;
      lp.fn.fused01<<<lp.grid, lp.block, lp.smem, st>>>(lp.tm_b, lp.tm_b8, a);
      break;
    case kPairKernel: {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(static_cast<unsigned>(lp.grid));
      cfg.blockDim = dim3(static_cast<unsigned>(lp.block));
      cfg.dynamicSmemBytes = lp.smem;
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      RISER_CUDA_TRY(cudaLaunchKernelEx(&cfg, lp.fn.pair, lp.tm_a, lp.tm_b, lp.tm_a8, lp.tm_b8, lp.tm_bl, lp.tm_b8l, a));
      return RISER_OK;
    }
    case kEoKernel:
      lp.fn.eo<<<lp.grid, lp.block, lp.smem, st>>>(lp.tm_a, lp.tm_a8, lp.tm_b, a);
      break;
    default:
      lp.fn.tc<<<lp.grid, lp.block, lp.smem, st>>>(lp.tm_a, lp.tm_b, lp.tm_a8, lp.tm_b8, a);
  }
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

}  // namespace
}  // namespace riser

// stage 0: tile activity flags and layer 0 (unless fused into layer 1's launch); stage 1: the conv layers;
// stage 2: head; stage 3: layer 0 alone; stage 16 + i: conv layer i alone.
extern "C" int riser_forward_stage(const riser_plan* p, int stage, const float* x, int64_t ld_x,
                                   const int32_t* len, float* probs, float* feat, riser_stream_t stream) {
  RISER_REQUIRE(p && len, "riser_forward_stage: null pointer");
  const riser_model* m = p->model;
  cudaStream_t st = as_stream(stream);
  int rc = RISER_OK;
  if (stage == 0) {
    RISER_REQUIRE(x, "riser_forward_stage: null x");
    RISER_REQUIRE(ld_x >= p->max_len && (ld_x & 1) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0,
                  "riser_forward: x must be 8-byte aligned with even ld_x >= max_len");
    tile_activity_kernel<<<(p->activity.total + 255) / 256, 256, 0, st>>>(len, p->activity, p->flags);
    RISER_CUDA_TRY(cudaGetLastError());
    return launch_layer0(p, x, ld_x, len, st);
  } else if (stage == 1) {
    for (int i = 1; i < m->n_layers; ++i)
      if ((rc = launch_conv(p, i, x, ld_x, len, st))) return rc;
  } else if (stage == 2) {
    RISER_REQUIRE(probs, "riser_forward_stage: null probs");
    const int n = m->n_layers;
    head_kernel<<<p->B, kHeadThreads, 0, st>>>(reinterpret_cast<const float*>(p->ws + p->act_off[n]), len, m->fc_w,
                                               m->fc_b, probs, feat, p->B, p->Lp[n], m->layer[n - 1].cout_p,
                                               m->c_last, n);
    RISER_CUDA_TRY(cudaGetLastError());
  } else if (stage == 3) {   // layer-0 launch only (timing aid: see bench.py)
    RISER_REQUIRE(x, "riser_forward_stage: null x");
    return launch_layer0(p, x, ld_x, len, st);
  } else if (stage >= 16 && stage < 16 + m->n_layers) {   // conv layer (stage - 16) alone (timing aid: tools/layer_events.py)
    RISER_REQUIRE(stage - 16 >= 1, "riser_forward_stage: single-layer stages need layer >= 1");
    return launch_conv(p, stage - 16, x, ld_x, len, st);
  } else {
    return fail(RISER_EINVAL, "riser_forward_stage: stage %d outside 0..3 / 16..", stage);
  }
  return RISER_OK;
}

extern "C" int riser_forward(const riser_plan* p, const float* x, int64_t ld_x, const int32_t* len, float* probs,
                             float* feat, riser_stream_t stream) {
  RISER_REQUIRE(p && x && len && probs, "riser_forward: null pointer");
  for (int stage = 0; stage < 3; ++stage) {
    const int st = riser_forward_stage(p, stage, x, ld_x, len, probs, feat, stream);
    if (st) return st;
  }
  return RISER_OK;
}

extern "C" int riser_decide(const float* probs, const int32_t* len, int B, int M, float thr, int mode,
                            int max_len, uint8_t* decision, riser_stream_t stream) {
  RISER_REQUIRE(B >= 0 && M >= 1, "riser_decide: bad B / M");
  if (B == 0) return RISER_OK;
  RISER_REQUIRE(probs && len && decision, "riser_decide: null pointer");
  RISER_REQUIRE(mode == RISER_MODE_ENRICH || mode == RISER_MODE_DEPLETE, "riser_decide: bad mode %d", mode);
  decide_kernel<<<(B + 255) / 256, 256, 0, as_stream(stream)>>>(probs, len, B, M, thr, mode, max_len, decision);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
