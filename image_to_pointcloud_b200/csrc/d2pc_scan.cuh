// d2pc_scan.cuh -- exclusive scans of per-tile counts, shared by the translation units that compact in order
// (mesh simplification, mesh components): a tile counts its survivors, one CTA scans the tile counts, and the tile
// then scans its own flags from its offset.
#ifndef D2PC_SCAN_CUH_
#define D2PC_SCAN_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

namespace d2pc {

constexpr int kTileScanThreads = 1024;
constexpr int kTileScanPerThread = 4;

// exclusive scan of one value per thread over the CTA; *total = CTA sum
__device__ __forceinline__ uint32_t tile_excl_scan(uint32_t v, uint32_t *s_warp, uint32_t *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  uint32_t woff = 0, t = 0;
  for (int k = 0; k < nw; ++k) { const uint32_t x = s_warp[k]; if (k < warp) woff += x; t += x; }
  *total = t;
  __syncthreads();
  return woff + incl - v;
}

// exclusive scan in place of one tile-count array (one CTA); the total goes to *total
static __global__ void __launch_bounds__(kTileScanThreads) tile_scan_kernel(uint32_t *arr, uint32_t n, uint32_t *total_out) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n; base += kTileScanThreads * kTileScanPerThread) {
    const uint32_t i0 = base + threadIdx.x * kTileScanPerThread;
    uint32_t v[kTileScanPerThread], sum = 0;
#pragma unroll
    for (int k = 0; k < kTileScanPerThread; ++k) { v[k] = i0 + k < n ? arr[i0 + k] : 0u; sum += v[k]; }
    uint32_t total;
    uint32_t ex = s_carry + tile_excl_scan(sum, s_warp, &total);
#pragma unroll
    for (int k = 0; k < kTileScanPerThread; ++k) {
      if (i0 + k < n) arr[i0 + k] = ex;
      ex += v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = s_carry;
}

}  // namespace d2pc

#endif  // D2PC_SCAN_CUH_
