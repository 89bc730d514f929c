// Data-parallel training on the GPUs of one box (riser_b200/parallel.py): peer access between the replicas' devices,
// and the fixed-order fp32 sum of their flat gradient buffers over peer-to-peer loads.  Every replica reduces its own
// slice of the buffer from all of them (one owner per element, so every replica ends up with the same bits), then
// copies the other slices from their owners with the same kernel and one source.
#include "common.cuh"

#include <algorithm>

namespace riser {
namespace {

struct PeerSrc {
  const float* p[RISER_MAX_REPLICAS];
};

__device__ __forceinline__ float sum_in_order(const PeerSrc& src, int G, int64_t i) {
  float a = src.p[0][i];
  for (int g = 1; g < G; ++g) a += src.p[g][i];
  return a;
}

// dst[i] = ((src[0][i] + src[1][i]) + src[2][i]) + ... for i in [lo, hi).  With vec (every pointer 16-byte aligned),
// the elements between the first and last multiple of 4 go as float4 loads and stores, the others one by one.  dst
// may be one of the sources: every element is read and written by the same thread.
__global__ void __launch_bounds__(256)
peer_reduce_kernel(PeerSrc src, int G, float* dst, int64_t lo, int64_t hi, int vec) {
  const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t tid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t head = vec ? std::min<int64_t>(hi, (lo + 3) & ~int64_t{3}) : hi;
  for (int64_t i = lo + tid; i < head; i += step) dst[i] = sum_in_order(src, G, i);
  if (!vec) return;
  const int64_t v1 = hi >> 2;
  for (int64_t v = (head >> 2) + tid; v < v1; v += step) {
    float4 a = reinterpret_cast<const float4*>(src.p[0])[v];
    for (int g = 1; g < G; ++g) {
      const float4 b = reinterpret_cast<const float4*>(src.p[g])[v];
      a.x += b.x;
      a.y += b.y;
      a.z += b.z;
      a.w += b.w;
    }
    reinterpret_cast<float4*>(dst)[v] = a;
  }
  for (int64_t i = std::max(v1 << 2, head) + tid; i < hi; i += step) dst[i] = sum_in_order(src, G, i);
}

}  // namespace
}  // namespace riser

using namespace riser;

extern "C" int riser_peer_enable(const int* devices_host, int G) {
  RISER_REQUIRE(devices_host && G >= 1, "riser_peer_enable: bad device list");
  int current = 0;
  RISER_CUDA_TRY(cudaGetDevice(&current));
  int rc = RISER_OK;
  for (int i = 0; i < G && rc == RISER_OK; ++i) {
    for (int j = 0; j < G && rc == RISER_OK; ++j) {
      const int a = devices_host[i], b = devices_host[j];
      if (a == b) continue;
      int can = 0;
      cudaError_t e = cudaDeviceCanAccessPeer(&can, a, b);
      if (e != cudaSuccess) {
        rc = fail(RISER_ECUDA, "riser_peer_enable: cudaDeviceCanAccessPeer(%d, %d): %s", a, b, cudaGetErrorString(e));
      } else if (!can) {
        rc = fail(RISER_ECUDA, "riser_peer_enable: devices %d and %d cannot access each other's memory (no peer access)",
                  std::min(a, b), std::max(a, b));
      } else if ((e = cudaSetDevice(a)) != cudaSuccess) {
        rc = fail(RISER_ECUDA, "riser_peer_enable: cudaSetDevice(%d): %s", a, cudaGetErrorString(e));
      } else if ((e = cudaDeviceEnablePeerAccess(b, 0)) == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();                          // already enabled in this process: success
      } else if (e != cudaSuccess) {
        rc = fail(RISER_ECUDA, "riser_peer_enable: device %d cannot enable access to device %d: %s", a, b,
                  cudaGetErrorString(e));
      }
    }
  }
  const cudaError_t e = cudaSetDevice(current);
  if (rc == RISER_OK && e != cudaSuccess) rc = fail(RISER_ECUDA, "riser_peer_enable: cudaSetDevice(%d): %s", current,
                                                    cudaGetErrorString(e));
  return rc;
}

extern "C" int riser_peer_reduce_f32(const float* const* src_host, int G, float* dst, int64_t lo, int64_t hi,
                                     riser_stream_t stream) {
  RISER_REQUIRE(src_host && dst, "riser_peer_reduce_f32: null pointer");
  RISER_REQUIRE(G >= 1 && G <= RISER_MAX_REPLICAS, "riser_peer_reduce_f32: %d sources (1 to %d)", G, RISER_MAX_REPLICAS);
  RISER_REQUIRE(0 <= lo && lo <= hi, "riser_peer_reduce_f32: bad range [%lld, %lld)", static_cast<long long>(lo),
                static_cast<long long>(hi));
  PeerSrc src{};
  int vec = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  for (int g = 0; g < G; ++g) {
    RISER_REQUIRE(src_host[g], "riser_peer_reduce_f32: source %d is null", g);
    src.p[g] = src_host[g];
    vec &= (reinterpret_cast<uintptr_t>(src_host[g]) & 15) == 0;
  }
  if (hi == lo) return RISER_OK;
  const int64_t work = vec ? (hi - lo + 3) / 4 + 3 : hi - lo;
  const int grid = static_cast<int>(std::min<int64_t>((work + 255) / 256, 148 * 8));
  peer_reduce_kernel<<<grid, 256, 0, as_stream(stream)>>>(src, G, dst, lo, hi, vec);
  RISER_CUDA_TRY(cudaGetLastError());
  return RISER_OK;
}
