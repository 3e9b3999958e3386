// Host launch helpers: per-device kernel configuration, kernel launches, gemm_tcgen05_kernel grids.
#pragma once
#include <atomic>
#include <mutex>
#include <unordered_set>
#include <utility>

#include "epilogues.cuh"
#include "gemm_sm100.cuh"
#include "tmap.cuh"

namespace vfp {

constexpr int kMaxDevices = 64;

inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}

// SM count of the CURRENT device (cached per device ordinal: one process may drive several GPUs)
inline int device_sm_count() {
  static std::atomic<int> sms[kMaxDevices];
  const int dev = current_device();
  int n = sms[dev].load(std::memory_order_relaxed);
  if (!n) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    sms[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE property of a kernel, so "already configured" is
// remembered per (kernel, device ordinal) - a process-wide flag breaks the second GPU of a process.
inline cudaError_t ensure_dynamic_smem(const void* kernel, int bytes) {
  static std::mutex mu;
  static std::unordered_set<unsigned long long> done;
  const unsigned long long key = (reinterpret_cast<unsigned long long>(kernel) << 6) ^ (unsigned long long)current_device();
  {
    std::lock_guard<std::mutex> g(mu);
    if (done.count(key)) return cudaSuccess;
  }
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) {
    std::lock_guard<std::mutex> g(mu);
    done.insert(key);
  }
  return e;
}

template <class... KArgs, class... Args>
inline cudaError_t launch_kernel_cluster(int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                         Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  int n = 0;
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  return launch_kernel_cluster(1, kernel, grid, block, smem, stream, std::forward<Args>(args)...);
}

template <int BLOCK_N, int BLOCK_K, int STAGES, class Epi, int MT = 1>
inline cudaError_t launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const GemmShape& shape,
                               const typename Epi::Params& ep, cudaStream_t stream) {
  using L = GemmSmemLayout<BLOCK_N, BLOCK_K, STAGES, MT>;
  constexpr int kSmem = L::kTotal + Epi::kExtraSmemBytes;
  static_assert(kSmem <= 232448, "shared memory budget");
  auto kernel = gemm_tcgen05_kernel<BLOCK_N, BLOCK_K, STAGES, Epi, MT>;
  if (cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), kSmem); e != cudaSuccess) return e;
  const int m_super = (shape.m_tiles + MT - 1) / MT;   // super-tiles
  const int total = shape.row_resident ? m_super * shape.n_segments : m_super * shape.n_tiles;
  if (total <= 0) return cudaSuccess;
  const int grid = total < device_sm_count() ? total : device_sm_count();
  return launch_kernel(kernel, dim3(grid), dim3(gemm_threads<BLOCK_N, Epi>()), kSmem, stream, ta, tb, shape, ep);
}

template <int BLOCK_N, int BLOCK_K, int STAGES, int KB, class Epi>
inline cudaError_t launch_gemm_bres(const CUtensorMap& ta, const CUtensorMap& tb, const GemmShape& shape,
                                    const typename Epi::Params& ep, cudaStream_t stream) {
  using L = GemmBresSmemLayout<BLOCK_N, BLOCK_K, STAGES, KB>;
  constexpr int kSmem = L::kTotal + Epi::kExtraSmemBytes;
  static_assert(kSmem <= 232448, "shared memory budget");
  if (shape.k_blocks != KB) return cudaErrorInvalidValue;
  auto kernel = gemm_bres_tcgen05_kernel<BLOCK_N, BLOCK_K, STAGES, KB, Epi>;
  if (cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), kSmem); e != cudaSuccess) return e;
  const long long total = (long long)shape.m_tiles * shape.n_tiles;
  if (total <= 0) return cudaSuccess;
  const int grid = total < device_sm_count() ? (int)total : device_sm_count();
  return launch_kernel(kernel, dim3(grid), dim3(gemm_threads<BLOCK_N, Epi>()), kSmem, stream, ta, tb, shape, ep);
}

template <int STAGES, int KB, class Epi>
inline cudaError_t launch_gemm_ares2(const CUtensorMap& ta, const CUtensorMap& tb, const AresShape& shape,
                                     const typename Epi::Params& ep, cudaStream_t stream) {
  using L = Ares2SmemLayout<STAGES, KB>;
  constexpr int kSmem = L::kTotal + Epi::kExtraSmemBytes;
  static_assert(kSmem <= 232448, "shared memory budget");
  auto kernel = gemm_ares2_tcgen05_kernel<STAGES, KB, Epi>;
  if (cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), kSmem); e != cudaSuccess) return e;
  const long long total = (long long)shape.m_super * shape.n_panels;
  if (total <= 0) return cudaSuccess;
  const int pairs = device_sm_count() / 2;
  const int grid = 2 * (total < pairs ? (int)total : pairs);
  return launch_kernel_cluster(2, kernel, dim3(grid), dim3(gemm_threads<kAres2BlockN, Epi>()), kSmem, stream, ta, tb, shape, ep);
}

// CTA-pair GEMM (BLOCK_N = 256): `tb` must be a tensor map with a box of 128 rows (one CTA's half of the B tile)
template <int BLOCK_K, int STAGES, class Epi>
inline cudaError_t launch_gemm_pair(const CUtensorMap& ta, const CUtensorMap& tb, const GemmShape& shape,
                                    const typename Epi::Params& ep, cudaStream_t stream) {
  using L = GemmPairSmemLayout<BLOCK_K, STAGES>;
  constexpr int kSmem = L::kTotal + Epi::kExtraSmemBytes;
  static_assert(kSmem <= 232448, "shared memory budget");
  auto kernel = gemm_pair_tcgen05_kernel<BLOCK_K, STAGES, Epi>;
  if (cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), kSmem); e != cudaSuccess) return e;
  if (shape.row_resident) return cudaErrorInvalidValue;
  const long long total = (long long)((shape.m_tiles + 1) / 2) * shape.n_tiles;
  if (total <= 0) return cudaSuccess;
  const int pairs = device_sm_count() / 2;
  const int grid = 2 * (total < pairs ? (int)total : pairs);
  return launch_kernel_cluster(2, kernel, dim3(grid), dim3(gemm_threads<256, Epi>()), kSmem, stream, ta, tb, shape, ep);
}

inline GemmShape plain_shape(long long M, int N, int K, int block_n, int block_k, int group_m = 16) {
  GemmShape s{};
  s.m_tiles = (int)((M + kBlockM - 1) / kBlockM);
  s.n_tiles = (N + block_n - 1) / block_n;
  s.k_blocks = K / block_k;
  s.group_m = group_m;
  s.a_conv = 0;
  s.tiles_per_frame = 1;
  s.frames_per_tile = 1;
  s.tile_out_rows = 0;
  s.h_mul = 0;
  s.row_resident = 0;
  s.n_segments = 1;
  return s;
}

// 3x3 / stride-2 / pad-1 convolution read through a stride-2 TMA box: K block kb = tap (kh, kw) x channel slice
inline void conv_taps_strided(GemmShape* s, int cblocks_per_tap) {
  s->h_mul = 2;
  for (int kb = 0; kb < 9 * cblocks_per_tap; ++kb) {
    const int tap = kb / cblocks_per_tap, kh = tap / 3, kw = tap % 3;
    s->tap_c_blk[kb] = (signed char)(kb % cblocks_per_tap);
    s->tap_w[kb] = (signed char)(kw - 1);
    s->tap_h[kb] = (signed char)(kh - 1);
  }
}

}  // namespace vfp
