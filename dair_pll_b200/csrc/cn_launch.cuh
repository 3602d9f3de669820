// Host side of the C entry points: launch status, grids, the SM count, the common workspace and the link-count
// dispatch of the generic chain.  Every translation unit that launches includes this header.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <type_traits>

#include "../../include/dair_pll_b200.h"

namespace cn {

// DPLL_OK, or the error of the last launch (cudaGetLastError) as a positive code
inline int launch_status() {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? DPLL_OK : (int)e;
}

// 1-D grid of `per_block` work items per block: at least one block, at most the grid limit
inline int grid_for(int64_t work, int per_block) {
  const int64_t b = (work + per_block - 1) / per_block;
  return (int)(b < 1 ? 1 : (b > 2147483647LL ? 2147483647LL : b));
}

// SM count of the current device.  Host threads may call the entry points concurrently (the autograd engine runs
// backwards on its own thread per device), so the per-device cache is atomic; a failed query is returned as its
// CUDA error.
inline int sm_count(int* sms) {
  constexpr int kMaxDevices = 64;
  static std::atomic<int> cache[kMaxDevices];       // 0 = not queried yet
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < kMaxDevices && (*sms = cache[dev].load(std::memory_order_relaxed)) > 0) return DPLL_OK;
  e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < kMaxDevices) cache[dev].store(*sms, std::memory_order_relaxed);
  return DPLL_OK;
}

// One resident set of `kernel`'s blocks on the current device: blocks per SM by occupancy (at least one) times the SM
// count, at most max_blocks.
template <typename K>
int resident_cap(K kernel, int threads, size_t smem, int64_t max_blocks, int64_t* cap) {
  int sms = 0, per_sm = 0;
  if (int rc = sm_count(&sms)) return rc;
  const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
  if (e != cudaSuccess) return (int)e;
  if (per_sm < 1) per_sm = 1;
  *cap = (int64_t)sms * per_sm;
  if (*cap > max_blocks) *cap = max_blocks;
  return DPLL_OK;
}

// Grid of a persistent launch that wants `need` blocks: at most one resident set (*cap, resident_cap), at least one
// block.
template <typename K>
int resident_blocks(K kernel, int threads, size_t smem, int64_t need, int64_t max_blocks, int* blocks, int64_t* cap) {
  if (int rc = resident_cap(kernel, threads, smem, max_blocks, cap)) return rc;
  *blocks = (int)(need < *cap ? need : *cap);
  if (*blocks < 1) *blocks = 1;
  return DPLL_OK;
}

// The common workspace of the reductions (dpll_workspace_bytes):
//   [per-block partials | prepared parameters of the box (16 doubles) | chunk counter of the dynamic schedule]
// Each kernel family that writes partials static_asserts that its largest grid fits the partials region.
constexpr size_t kWsPartialsBytes = (size_t)148 * 16 * 32 * sizeof(double);   // 2,368 blocks x 32 accumulators
constexpr size_t kWsParamsOffset = kWsPartialsBytes;
constexpr size_t kWsCounterOffset = kWsParamsOffset + 16 * sizeof(double);
constexpr size_t kWsCounterBytes = 2 * sizeof(unsigned long long);
constexpr size_t kWsBytes = kWsCounterOffset + kWsCounterBytes;

inline bool workspace_ok(const void* ws, size_t bytes) { return ws && bytes >= kWsBytes; }

// Resets the chunk counter of the dynamic schedule (DPLL_LOSS_DYNAMIC) on `st` and points *dyn at it.
inline int dynamic_counter(void* ws, cudaStream_t st, unsigned long long** dyn) {
  *dyn = reinterpret_cast<unsigned long long*>(static_cast<char*>(ws) + kWsCounterOffset);
  const cudaError_t e = cudaMemsetAsync(*dyn, 0, kWsCounterBytes, st);
  return e == cudaSuccess ? DPLL_OK : (int)e;
}

// Calls f(std::integral_constant<int, N>{}) for the generic chain's link count N = 2 .. 6; DPLL_EINVAL for any other.
template <typename F>
int with_links(int n_links, F&& f) {
  switch (n_links) {
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    case 4: return f(std::integral_constant<int, 4>{});
    case 5: return f(std::integral_constant<int, 5>{});
    case 6: return f(std::integral_constant<int, 6>{});
    default: return DPLL_EINVAL;
  }
}

}  // namespace cn
