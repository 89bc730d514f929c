// Training ops of the ResNet variant (riser/nets/resnet.py) that the ConvNet's training path (csrc/train.cu) does not
// cover; riser_b200/training.py's ResNetTrainer drives them.  Layout: fp32 channel-last [B][L_pad][C] with per-read
// valid lengths; rows at or beyond a read's length are never read.
//   * riser_conv1d_dgrad_cl: the input gradient of a strided, padded Conv1d (stride-1 convolutions keep using
//     riser_conv1d_cl with the tap-flipped weight), with an optional gradient to add (the other branch of a block).
//   * riser_bn_stats_cl / riser_bn_apply_cl / riser_bn_bwd_cl: BatchNorm1d in training mode.  Per-channel statistics
//     are over the valid rows of every read (at equal lengths exactly torch's batch statistics), summed in float64:
//     every CTA owns a fixed slice of the rows (kBnParts slices, a constant, so the order does not depend on the
//     device), and a second launch adds the slices in order.  No float atomics: a launch gives the same bits on every
//     run.
//   * riser_bn_{stats,bwd}_{partial,finalize}_cl: the two halves of those reductions for data-parallel replicas
//     (SyncBatchNorm): each replica adds its slices into one float64 partial (valid rows, two sums per channel), and
//     every replica then adds the G partials in device order.  riser_bn_stats_cl / riser_bn_bwd_cl are G = 1 of it
//     without the intermediate partial (0.0 + x is exact), so their bits do not change.
#include "common.cuh"

#include <algorithm>

namespace riser {
namespace {

constexpr int kBnParts = 148;        // row slices of a reduction (a constant: the summation order is fixed)
constexpr int kBnRowLanes = 8;       // threads per channel in a slice (blockDim.y)

int grid_for(int64_t total) { return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, 148 * 16))); }

// ------------------------------------------------------------------ strided dgrad
// dx[b][u][ci] = sum over (t, j) with t * stride + j - pad = u, t < len_out[b] of sum_co w[j][co][ci] dz[b][t][co]
// (+ residual[b][u][ci]) for u < len_in[b]; 0 on the other rows.  Taps in order, channels in order: fixed order.
__global__ void __launch_bounds__(256)
dgrad_cl_kernel(const float* __restrict__ dz, const int32_t* __restrict__ len_out, const float* __restrict__ w,
                const float* __restrict__ residual, float* __restrict__ dx, const int32_t* __restrict__ len_in, int B,
                int Lout_pad, int Lin_pad, int Cin, int Cout, int K, int stride, int pad) {
  const int64_t total = static_cast<int64_t>(B) * Lin_pad * Cin;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(idx % Cin);
    const int64_t bu = idx / Cin;
    const int u = static_cast<int>(bu % Lin_pad);
    const int b = static_cast<int>(bu / Lin_pad);
    if (u >= len_in[b]) {
      dx[idx] = 0.f;
      continue;
    }
    const int Lo = len_out[b];
    float acc = 0.f;
    for (int j = 0; j < K; ++j) {
      const int num = u + pad - j;
      if (num < 0) break;                            // num falls with j
      const int t = num / stride;
      if (t * stride != num || t >= Lo) continue;
      const float* dzr = dz + (static_cast<int64_t>(b) * Lout_pad + t) * Cout;
      const float* wj = w + static_cast<int64_t>(j) * Cout * Cin + ci;
      for (int co = 0; co < Cout; ++co) acc = fmaf(__ldg(dzr + co), __ldg(wj + static_cast<int64_t>(co) * Cin), acc);
    }
    if (residual) acc += residual[idx];
    dx[idx] = acc;
  }
}

// ------------------------------------------------------------------ BatchNorm: per-slice partial sums
// Slice p of the B * L_pad rows, channel c = blockIdx.y * 32 + threadIdx.x, rows threadIdx.y + kBnRowLanes i of the
// slice in order, then the kBnRowLanes lanes in order.  STATS: (sum y, sum y^2); BWD: (sum dy, sum dy xhat) with
// dy = dout * (mask > 0) (mask optional) and xhat = (y - mean) invstd.  part [kBnParts][C][2] float64.
template <bool BWD>
__global__ void __launch_bounds__(32 * kBnRowLanes)
bn_partial_kernel(const float* __restrict__ y, const float* __restrict__ dout, const float* __restrict__ mask,
                  const float* __restrict__ mean, const float* __restrict__ var, float eps,
                  const int32_t* __restrict__ len, int B, int L_pad, int C, double* __restrict__ part) {
  __shared__ double red[kBnRowLanes][32][2];
  const int c = blockIdx.y * 32 + threadIdx.x, p = blockIdx.x;
  const int64_t rows = static_cast<int64_t>(B) * L_pad;
  const int64_t per = (rows + kBnParts - 1) / kBnParts;
  const int64_t r0 = p * per, r1 = std::min<int64_t>(rows, r0 + per);
  double s0 = 0.0, s1 = 0.0;
  if (c < C && r0 + threadIdx.y < r1) {
    double mu = 0.0, inv = 0.0;
    if (BWD) {
      mu = static_cast<double>(mean[c]);
      inv = static_cast<double>(1.f / sqrtf(var[c] + eps));
    }
    int64_t r = r0 + threadIdx.y;
    int b = static_cast<int>(r / L_pad), t = static_cast<int>(r - static_cast<int64_t>(b) * L_pad);
    int n = len[b];
    for (; r < r1; r += kBnRowLanes) {
      if (t < n) {
        const int64_t o = r * C + c;
        const double v = static_cast<double>(y[o]);
        if (BWD) {
          float g = dout[o];
          if (mask && !(mask[o] > 0.f)) g = 0.f;
          const double d = static_cast<double>(g);
          s0 += d;
          s1 += d * (v - mu) * inv;
        } else {
          s0 += v;
          s1 += v * v;
        }
      }
      t += kBnRowLanes;
      while (t >= L_pad && b < B - 1) {
        t -= L_pad;
        n = len[++b];
      }
    }
  }
  red[threadIdx.y][threadIdx.x][0] = s0;
  red[threadIdx.y][threadIdx.x][1] = s1;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    double a0 = 0.0, a1 = 0.0;
    for (int i = 0; i < kBnRowLanes; ++i) {
      a0 += red[i][threadIdx.x][0];
      a1 += red[i][threadIdx.x][1];
    }
    part[(static_cast<int64_t>(p) * C + c) * 2] = a0;
    part[(static_cast<int64_t>(p) * C + c) * 2 + 1] = a1;
  }
}

// number of valid rows, float64 (every thread of the finishing kernels counts it the same way)
__device__ double valid_rows(const int32_t* __restrict__ len, int B) {
  int64_t n = 0;
  for (int b = 0; b < B; ++b) n += len[b];
  return static_cast<double>(n);
}

// The partial sums a finishing kernel adds: G buffers (in device order) of S slices [S][C][2] each.  A replica's
// partial (S = 1) also holds its valid-row count at [2C].
struct BnParts {
  const double* p[RISER_MAX_REPLICAS];
};

__device__ void bn_sums(const BnParts& parts, int G, int S, int C, int c, double& s0, double& s1) {
  s0 = 0.0;
  s1 = 0.0;
  for (int g = 0; g < G; ++g)
    for (int p = 0; p < S; ++p) {
      s0 += parts.p[g][(static_cast<int64_t>(p) * C + c) * 2];
      s1 += parts.p[g][(static_cast<int64_t>(p) * C + c) * 2 + 1];
    }
}

// len != NULL: the rows of this launch's batch; else the replicas' counts (S = 1) in order
__device__ double bn_count(const BnParts& parts, int G, int C, const int32_t* __restrict__ len, int B) {
  if (len) return valid_rows(len, B);
  double n = 0.0;
  for (int g = 0; g < G; ++g) n += parts.p[g][2 * C];
  return n;
}

// A replica's partial: its kBnParts slices in order per channel, and its valid-row count
__global__ void __launch_bounds__(256)
bn_slices_kernel(const double* __restrict__ part, const int32_t* __restrict__ len, int B, int C,
                 double* __restrict__ partial) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  BnParts parts{};
  parts.p[0] = part;
  double s0, s1;
  bn_sums(parts, 1, kBnParts, C, c, s0, s1);
  partial[2 * c] = s0;
  partial[2 * c + 1] = s1;
  if (c == 0) partial[2 * C] = valid_rows(len, B);
}

// Per channel: the slices in order -> mean and biased variance; with update, running = (1 - m) running + m stat
// (unbiased variance n / (n - 1)) and num_batches_tracked + 1.
__global__ void __launch_bounds__(256)
bn_stats_finish_kernel(BnParts parts, int G, int S, const int32_t* __restrict__ len, int B, int C,
                       float* __restrict__ mean, float* __restrict__ var, float* __restrict__ running_mean,
                       float* __restrict__ running_var, int64_t* __restrict__ num_batches, float momentum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s, ss;
  bn_sums(parts, G, S, C, c, s, ss);
  const double n = bn_count(parts, G, C, len, B);
  const double mu = s / n;
  const double v = fmax(ss / n - mu * mu, 0.0);
  mean[c] = static_cast<float>(mu);
  var[c] = static_cast<float>(v);
  if (running_mean) {
    const double m = static_cast<double>(momentum);
    running_mean[c] = static_cast<float>((1.0 - m) * running_mean[c] + m * mu);
    running_var[c] = static_cast<float>((1.0 - m) * running_var[c] + m * v * n / (n - 1.0));
    if (c == 0) *num_batches += 1;
  }
}

// out = act(gamma (y - mean) invstd + beta + r), r = residual, or the BatchNorm of residual with its own parameters
// (res_mean != NULL), or 0; valid rows only.  invstd = 1 / sqrt(var + eps).
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float* __restrict__ y, const int32_t* __restrict__ len, int B, int L_pad, int C,
                const float* __restrict__ mean, const float* __restrict__ var, const float* __restrict__ gamma,
                const float* __restrict__ beta, const float* __restrict__ residual, const float* __restrict__ res_mean,
                const float* __restrict__ res_var, const float* __restrict__ res_gamma,
                const float* __restrict__ res_beta, float eps, int relu, float* __restrict__ out) {
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const int64_t bt = idx / C;
    const int t = static_cast<int>(bt % L_pad);
    const int b = static_cast<int>(bt / L_pad);
    if (t >= len[b]) continue;
    float v = (y[idx] - mean[c]) * (1.f / sqrtf(var[c] + eps)) * gamma[c] + beta[c];
    if (residual) {
      float r = residual[idx];
      if (res_mean) r = (r - res_mean[c]) * (1.f / sqrtf(res_var[c] + eps)) * res_gamma[c] + res_beta[c];
      v += r;
    }
    out[idx] = relu ? fmaxf(v, 0.f) : v;
  }
}

// Per channel: the slices in order -> dgamma = sum dy xhat, dbeta = sum dy (zeros when !owner: a replica whose
// gradients are added to the owner's); sums[c] = (sum dy / n, sum dy xhat / n)
__global__ void __launch_bounds__(256)
bn_bwd_finish_kernel(BnParts parts, int G, int S, const int32_t* __restrict__ len, int B, int C, int owner,
                     float* __restrict__ dgamma, float* __restrict__ dbeta, double* __restrict__ sums) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s0, s1;
  bn_sums(parts, G, S, C, c, s0, s1);
  const double n = bn_count(parts, G, C, len, B);
  dgamma[c] = owner ? static_cast<float>(s1) : 0.f;
  dbeta[c] = owner ? static_cast<float>(s0) : 0.f;
  sums[2 * c] = s0 / n;
  sums[2 * c + 1] = s1 / n;
}

// dx = gamma invstd (dy - sum dy / n - xhat sum dy xhat / n) on valid rows, 0 on the others; dy_out (optional) = dy
__global__ void __launch_bounds__(256)
bn_bwd_dx_kernel(const float* __restrict__ y, const float* __restrict__ dout, const float* __restrict__ mask,
                 const int32_t* __restrict__ len, int B, int L_pad, int C, const float* __restrict__ mean,
                 const float* __restrict__ var, const float* __restrict__ gamma, float eps,
                 const double* __restrict__ sums, float* __restrict__ dx, float* __restrict__ dy_out) {
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const int64_t bt = idx / C;
    const int t = static_cast<int>(bt % L_pad);
    const int b = static_cast<int>(bt / L_pad);
    if (t >= len[b]) {
      dx[idx] = 0.f;
      if (dy_out) dy_out[idx] = 0.f;
      continue;
    }
    float g = dout[idx];
    if (mask && !(mask[idx] > 0.f)) g = 0.f;
    const double inv = static_cast<double>(1.f / sqrtf(var[c] + eps));
    const double xhat = (static_cast<double>(y[idx]) - static_cast<double>(mean[c])) * inv;
    const double d = static_cast<double>(g) - sums[2 * c] - xhat * sums[2 * c + 1];
    dx[idx] = static_cast<float>(static_cast<double>(gamma[c]) * inv * d);
    if (dy_out) dy_out[idx] = g;
  }
}

}  // namespace
}  // namespace riser

using namespace riser;

extern "C" int riser_conv1d_dgrad_cl(const float* dz, const int32_t* len_out, const float* w, const float* residual,
                                     float* dx, const int32_t* len_in, int B, int Lout_pad, int Lin_pad, int Cin,
                                     int Cout, int K, int stride, int pad, riser_stream_t stream) {
  RISER_REQUIRE(dz && len_out && w && dx && len_in, "riser_conv1d_dgrad_cl: null pointer");
  RISER_REQUIRE(B >= 0 && Lout_pad > 0 && Lin_pad > 0 && Cin > 0 && Cout > 0 && K > 0 && stride > 0 && pad >= 0,
                "riser_conv1d_dgrad_cl: bad shape");
  const int64_t total = static_cast<int64_t>(B) * Lin_pad * Cin;
  if (total == 0) return RISER_OK;
  dgrad_cl_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(dz, len_out, w, residual, dx, len_in, B, Lout_pad,
                                                                  Lin_pad, Cin, Cout, K, stride, pad);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" size_t riser_bn_workspace_bytes(int C) {
  if (C <= 0) return 0;
  return (static_cast<size_t>(kBnParts) + 1) * 2 * static_cast<size_t>(C) * sizeof(double);
}

namespace {

BnParts one_part(const double* part) {
  BnParts p{};
  p.p[0] = part;
  return p;
}

int gather_parts(const char* who, const double* const* partials_host, int G, BnParts& parts) {
  RISER_REQUIRE(partials_host && G >= 1 && G <= RISER_MAX_REPLICAS, "%s: %d partials (1 to %d)", who, G,
                RISER_MAX_REPLICAS);
  parts = BnParts{};
  for (int g = 0; g < G; ++g) {
    RISER_REQUIRE(partials_host[g], "%s: partial %d is null", who, g);
    parts.p[g] = partials_host[g];
  }
  return RISER_OK;
}

}  // namespace

extern "C" size_t riser_bn_partial_bytes(int C) {
  if (C <= 0) return 0;
  return (2 * static_cast<size_t>(C) + 1) * sizeof(double);
}

extern "C" int riser_bn_stats_cl(const float* y, const int32_t* len, int B, int L_pad, int C, float* mean, float* var,
                                 float* running_mean, float* running_var, int64_t* num_batches_tracked, float momentum,
                                 void* workspace, size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(y && len && mean && var && workspace, "riser_bn_stats_cl: null pointer");
  RISER_REQUIRE((running_mean == nullptr) == (running_var == nullptr) &&
                    (running_mean == nullptr) == (num_batches_tracked == nullptr),
                "riser_bn_stats_cl: running_mean, running_var and num_batches_tracked go together");
  RISER_REQUIRE(B > 0 && L_pad > 0 && C > 0, "riser_bn_stats_cl: bad shape");
  const size_t need = riser_bn_workspace_bytes(C);
  if (workspace_bytes < need) return fail(RISER_ENOMEM, "riser_bn_stats_cl: workspace %zu bytes < %zu", workspace_bytes, need);
  double* part = static_cast<double*>(workspace);
  bn_partial_kernel<false><<<dim3(kBnParts, (C + 31) / 32), dim3(32, kBnRowLanes), 0, as_stream(stream)>>>(
      y, nullptr, nullptr, nullptr, nullptr, 0.f, len, B, L_pad, C, part);
  RISER_CUDA_TRY(cudaGetLastError());
  bn_stats_finish_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(one_part(part), 1, kBnParts, len, B, C, mean,
                                                                         var, running_mean, running_var,
                                                                         num_batches_tracked, momentum);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_stats_partial_cl(const float* y, const int32_t* len, int B, int L_pad, int C, double* partial,
                                         void* workspace, size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(partial && workspace && (B == 0 || (y && len)), "riser_bn_stats_partial_cl: null pointer");
  RISER_REQUIRE(B >= 0 && L_pad > 0 && C > 0, "riser_bn_stats_partial_cl: bad shape");
  const size_t need = riser_bn_workspace_bytes(C);
  if (workspace_bytes < need)
    return fail(RISER_ENOMEM, "riser_bn_stats_partial_cl: workspace %zu bytes < %zu", workspace_bytes, need);
  if (B == 0) {
    RISER_CUDA_TRY(cudaMemsetAsync(partial, 0, riser_bn_partial_bytes(C), as_stream(stream)));
    return RISER_OK;
  }
  double* part = static_cast<double*>(workspace);
  bn_partial_kernel<false><<<dim3(kBnParts, (C + 31) / 32), dim3(32, kBnRowLanes), 0, as_stream(stream)>>>(
      y, nullptr, nullptr, nullptr, nullptr, 0.f, len, B, L_pad, C, part);
  RISER_CUDA_TRY(cudaGetLastError());
  bn_slices_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(part, len, B, C, partial);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_stats_finalize_cl(const double* const* partials_host, int G, int C, float* mean, float* var,
                                          float* running_mean, float* running_var, int64_t* num_batches_tracked,
                                          float momentum, riser_stream_t stream) {
  RISER_REQUIRE(mean && var, "riser_bn_stats_finalize_cl: null pointer");
  RISER_REQUIRE((running_mean == nullptr) == (running_var == nullptr) &&
                    (running_mean == nullptr) == (num_batches_tracked == nullptr),
                "riser_bn_stats_finalize_cl: running_mean, running_var and num_batches_tracked go together");
  RISER_REQUIRE(C > 0, "riser_bn_stats_finalize_cl: bad shape");
  BnParts parts;
  const int rc = gather_parts("riser_bn_stats_finalize_cl", partials_host, G, parts);
  if (rc != RISER_OK) return rc;
  bn_stats_finish_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(parts, G, 1, nullptr, 0, C, mean, var,
                                                                         running_mean, running_var,
                                                                         num_batches_tracked, momentum);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_apply_cl(const float* y, const int32_t* len, int B, int L_pad, int C, const float* mean,
                                 const float* var, const float* gamma, const float* beta, const float* residual,
                                 const float* res_mean, const float* res_var, const float* res_gamma,
                                 const float* res_beta, float eps, int relu, float* out, riser_stream_t stream) {
  RISER_REQUIRE(y && len && mean && var && gamma && beta && out, "riser_bn_apply_cl: null pointer");
  RISER_REQUIRE(res_mean == nullptr || (residual && res_var && res_gamma && res_beta),
                "riser_bn_apply_cl: a normalised residual needs residual, res_var, res_gamma and res_beta");
  RISER_REQUIRE(B >= 0 && L_pad > 0 && C > 0, "riser_bn_apply_cl: bad shape");
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  if (total == 0) return RISER_OK;
  bn_apply_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(y, len, B, L_pad, C, mean, var, gamma, beta, residual,
                                                                  res_mean, res_var, res_gamma, res_beta, eps, relu, out);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_bwd_cl(const float* dout, const float* mask, const float* y, const int32_t* len, int B,
                               int L_pad, int C, const float* mean, const float* var, const float* gamma, float eps,
                               float* dgamma, float* dbeta, float* dx, float* dy_out, void* workspace,
                               size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(dout && y && len && mean && var && gamma && dgamma && dbeta && dx && workspace,
                "riser_bn_bwd_cl: null pointer");
  RISER_REQUIRE(B > 0 && L_pad > 0 && C > 0, "riser_bn_bwd_cl: bad shape");
  const size_t need = riser_bn_workspace_bytes(C);
  if (workspace_bytes < need) return fail(RISER_ENOMEM, "riser_bn_bwd_cl: workspace %zu bytes < %zu", workspace_bytes, need);
  double* part = static_cast<double*>(workspace);
  double* sums = part + static_cast<size_t>(kBnParts) * 2 * C;
  bn_partial_kernel<true><<<dim3(kBnParts, (C + 31) / 32), dim3(32, kBnRowLanes), 0, as_stream(stream)>>>(
      y, dout, mask, mean, var, eps, len, B, L_pad, C, part);
  RISER_CUDA_TRY(cudaGetLastError());
  bn_bwd_finish_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(one_part(part), 1, kBnParts, len, B, C, 1,
                                                                       dgamma, dbeta, sums);
  RISER_CUDA_TRY(cudaGetLastError());
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  bn_bwd_dx_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(y, dout, mask, len, B, L_pad, C, mean, var, gamma,
                                                                   eps, sums, dx, dy_out);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_bwd_partial_cl(const float* dout, const float* mask, const float* y, const int32_t* len, int B,
                                       int L_pad, int C, const float* mean, const float* var, float eps, double* partial,
                                       void* workspace, size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(partial && workspace && (B == 0 || (dout && y && len && mean && var)),
                "riser_bn_bwd_partial_cl: null pointer");
  RISER_REQUIRE(B >= 0 && L_pad > 0 && C > 0, "riser_bn_bwd_partial_cl: bad shape");
  const size_t need = riser_bn_workspace_bytes(C);
  if (workspace_bytes < need)
    return fail(RISER_ENOMEM, "riser_bn_bwd_partial_cl: workspace %zu bytes < %zu", workspace_bytes, need);
  if (B == 0) {
    RISER_CUDA_TRY(cudaMemsetAsync(partial, 0, riser_bn_partial_bytes(C), as_stream(stream)));
    return RISER_OK;
  }
  double* part = static_cast<double*>(workspace);
  bn_partial_kernel<true><<<dim3(kBnParts, (C + 31) / 32), dim3(32, kBnRowLanes), 0, as_stream(stream)>>>(
      y, dout, mask, mean, var, eps, len, B, L_pad, C, part);
  RISER_CUDA_TRY(cudaGetLastError());
  bn_slices_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(part, len, B, C, partial);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}

extern "C" int riser_bn_bwd_finalize_cl(const double* const* partials_host, int G, int owner, const float* dout,
                                        const float* mask, const float* y, const int32_t* len, int B, int L_pad, int C,
                                        const float* mean, const float* var, const float* gamma, float eps,
                                        float* dgamma, float* dbeta, float* dx, float* dy_out, void* workspace,
                                        size_t workspace_bytes, riser_stream_t stream) {
  RISER_REQUIRE(dgamma && dbeta && workspace && (B == 0 || (dout && y && len && mean && var && gamma && dx)),
                "riser_bn_bwd_finalize_cl: null pointer");
  RISER_REQUIRE(B >= 0 && L_pad > 0 && C > 0, "riser_bn_bwd_finalize_cl: bad shape");
  const size_t need = riser_bn_workspace_bytes(C);
  if (workspace_bytes < need)
    return fail(RISER_ENOMEM, "riser_bn_bwd_finalize_cl: workspace %zu bytes < %zu", workspace_bytes, need);
  BnParts parts;
  const int rc = gather_parts("riser_bn_bwd_finalize_cl", partials_host, G, parts);
  if (rc != RISER_OK) return rc;
  double* sums = static_cast<double*>(workspace) + static_cast<size_t>(kBnParts) * 2 * C;
  bn_bwd_finish_kernel<<<(C + 255) / 256, 256, 0, as_stream(stream)>>>(parts, G, 1, nullptr, 0, C, owner, dgamma,
                                                                       dbeta, sums);
  RISER_CUDA_TRY(cudaGetLastError());
  const int64_t total = static_cast<int64_t>(B) * L_pad * C;
  if (total == 0) return RISER_OK;
  bn_bwd_dx_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(y, dout, mask, len, B, L_pad, C, mean, var, gamma,
                                                                   eps, sums, dx, dy_out);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
