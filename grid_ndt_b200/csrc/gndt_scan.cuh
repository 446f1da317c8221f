// gndt_scan.cuh — device-wide exclusive scan of u32 values in one pass (CTA scan + grouped
// decoupled look-back), used by the traversability graph (edge offsets) and by the streaming
// fusion (compaction of new / dead voxels, changed-column list).
#pragma once
#include "gndt_device.cuh"

namespace gndt {

struct ScanCtl {
  u32 ticket, total, err, pad;
};

constexpr int kScanItems = 4;
constexpr int kScanTile = 256 * kScanItems;

// out[i] = sum of in[0..i), out[n] = total (also ScanCtl::total).  n = *n_dev when n_dev != NULL.
// `state` and `groups` are lookback_scratch(ceil(n / kScanTile)); `g`, `state` and `groups` are
// zeroed before the launch.
__global__ void __launch_bounds__(256)
exclusive_scan_kernel(ScanCtl *g, const u32 *in, u32 n_fixed, const u32 *n_dev, u32 *out, u64 *state, GroupState *groups) {
  __shared__ u32 warp_sums[32];
  __shared__ u32 s_tile, s_total, s_prefix;
  const int tid = threadIdx.x;
  const u32 n = n_dev ? *n_dev : n_fixed;
  const u32 n_tiles = (n + kScanTile - 1) / kScanTile;
  if (n == 0) {
    if (blockIdx.x == 0 && tid == 0) { out[0] = 0; g->total = 0; }
    return;
  }
  for (;;) {
    __syncthreads();
    if (tid == 0) s_tile = atomicAdd(&g->ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    if (tile >= n_tiles) return;
    const u32 i0 = (tile * 256 + tid) * kScanItems;
    u32 v[kScanItems], sum = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) { v[k] = (i0 + k < n) ? in[i0 + k] : 0u; sum += v[k]; }
    const u32 exc = block_exclusive_scan(sum, warp_sums);
    if (tid == 255) s_total = exc + sum;
    __syncthreads();
    if (tid < 32) {
      const u32 total = s_total;
      const u64 pre = warp_lookback_grouped(state, groups, (int)tile, 0u, total, &g->err);
      if (tid == 0) {
        s_prefix = (u32)pre;
        if (tile == n_tiles - 1) { g->total = (u32)pre + total; out[n] = (u32)pre + total; }
      }
    }
    __syncthreads();
    u32 run = s_prefix + exc;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
      if (i0 + k < n) out[i0 + k] = run;
      run += v[k];
    }
  }
}

}  // namespace gndt
