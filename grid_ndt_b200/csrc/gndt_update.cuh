// gndt_update.cuh — streaming fusion of one scan into the resident map (gndt_update), its
// inverse (gndt_remove) and the list of cells a scan touched (gndt_changed_columns).
//
// Replaces changeCallback + TwoDmap::change2DMap (reference src/receiver.cpp:179-212,
// include/map2D.h:672-822), delCallback + del2DMap (src/receiver.cpp:95-134,214-248,
// include/map2D.h:826-915) and changeMorton_list (src/receiver.cpp:47-56,187,196).  The add
// path is dead code in the reference (uniformDivision never fills the lPoints lists
// change2DMap consumes, its subscription is commented out) and its pooled-covariance formula
// mixes scatters with sample covariances and uses an integer M*N/(M+N) (map2D.h:777-780); the
// delete path is commented out at every call site.  The contract here is batch equivalence:
//   build(A) + update(B)             == build(A ++ B)
//   build(A) + update(B) + remove(B) == build(A)
// The resident state is the sorted table of raw binary64 moments; a scan is reduced to its own
// sorted moments table by the normal front end and merged with Chan's update / its inverse
// (exact in n, mean and centred scatter up to binary64 rounding).
//
// The resident table is never modified: the merged table is written to the alternate buffer,
// and a failed call (capacity, removal of points that were never fused) leaves the map as it
// was.  What is O(resident) is the copy into the alternate table and the relabelling pass.
#pragma once
#include "gndt_device.cuh"
#include "gndt_reduce.cuh"
#include "gndt_scan.cuh"

namespace gndt {

constexpr u32 kNone = 0xFFFFFFFFu;
constexpr u32 kErrUnmatched = 4u;  // gndt_remove: the scan holds points that are not in the map

// persistent (never memset) totals over all clouds fused into the resident map
struct Totals {
  u64 n_points, n_valid, n_dropped, n_outside;
};

// sign >= 0: add the last front end's counters, < 0: subtract them (gndt_remove); reset: start over
__global__ void totals_kernel(Totals *tot, const Ctl *ctl, u64 n_points, int reset, int sign) {
  pdl_wait();
  pdl_trigger();
  if (threadIdx.x || blockIdx.x) return;
  if (reset) { tot->n_points = 0; tot->n_valid = 0; tot->n_dropped = 0; tot->n_outside = 0; }
  if (sign >= 0) { tot->n_points += n_points; tot->n_valid += ctl->n_valid; tot->n_dropped += ctl->n_dropped; tot->n_outside += ctl->n_outside; }
  else { tot->n_points -= n_points; tot->n_valid -= ctl->n_valid; tot->n_dropped -= ctl->n_dropped; tot->n_outside -= ctl->n_outside; }
}

__device__ __forceinline__ u32 lower_bound_key(const VoxMoments *t, u32 n, u64 key) {
  u32 lo = 0, hi = n;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (t[mid].key < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ u32 lower_bound_u64(const u64 *t, u32 n, u64 key) {
  u32 lo = 0, hi = n;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (t[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ void load_moments(const VoxMoments &v, Moments &m) {
  m.n = (double)v.count;
#pragma unroll
  for (int k = 0; k < 3; ++k) m.m[k] = v.m[k];
#pragma unroll
  for (int k = 0; k < 6; ++k) m.s[k] = v.s[k];
}

// Inverse of merge_moments: a = c (+) b  ->  a becomes c.  Needs a.n > b.n.
// Means are relative to the cell centre (gndt_reduce.cuh), so the mean cancellation below loses
// at most the rounding of a cell-sized value.  The scatter c.s = a.s - b.s - d d^T w still cancels
// two large sums when a few points survive a large mass: an entry within a few rounding units of
// that cancellation is noise and is set to 0, so that survivors whose batch scatter is exactly 0
// (identical points) or rank 1 (collinear points) get it back.  The bound of entry (i, j) is
// eps * sqrt(B_i B_j), B_i = |a.s_ii| + |b.s_ii| + d_i^2 w: a PSD matrix's off-diagonal entry is
// bounded by the geometric mean of its diagonal ones, and so is its error.
constexpr double kUnmergeTol = 8.0 * 2.220446049250313e-16;
__device__ __forceinline__ void unmerge_moments(Moments &a, const Moments &b) {
  const double n = a.n - b.n;
  const double c0 = (a.n * a.m[0] - b.n * b.m[0]) / n, c1 = (a.n * a.m[1] - b.n * b.m[1]) / n, c2 = (a.n * a.m[2] - b.n * b.m[2]) / n;
  const double d[3] = {b.m[0] - c0, b.m[1] - c1, b.m[2] - c2};
  const double w = n * b.n / a.n;
  double bound[3];
  const int diag[3] = {0, 3, 5};
#pragma unroll
  for (int i = 0; i < 3; ++i) bound[i] = sqrt(fabs(a.s[diag[i]]) + fabs(b.s[diag[i]]) + d[i] * d[i] * w);
  const int ri[6] = {0, 0, 0, 1, 1, 2}, rj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double s = a.s[k] - (b.s[k] + d[ri[k]] * d[rj[k]] * w);
    a.s[k] = fabs(s) <= kUnmergeTol * bound[ri[k]] * bound[rj[k]] ? 0.0 : s;
  }
  a.m[0] = c0; a.m[1] = c1; a.m[2] = c2;
  a.n = n;
}

// U1: one thread per scan voxel: find the resident voxel with the same key.
//   add:    unmatched scan voxels are new (is_new = 1)
//   remove: unmatched ones (or ones with more points than the map holds) are an error; a resident
//           voxel that loses all its points is dead
// inv[i] = scan voxel matched to resident voxel i (kNone-initialised by the caller).
__global__ void update_match_kernel(Ctl *ctl, const VoxMoments *res, u32 n_res, const VoxMoments *scan, int sign, u32 *inv,
                                    u32 *is_new, u32 *dead) {
  const u32 n_scan = ctl->n_voxels;
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n_scan; j += gridDim.x * blockDim.x) {
    const u64 key = scan[j].key;
    const u32 i = lower_bound_key(res, n_res, key);
    const bool found = i < n_res && res[i].key == key;
    if (found) inv[i] = j;
    if (sign > 0) {
      is_new[j] = found ? 0u : 1u;
    } else {
      is_new[j] = 0u;
      if (!found || scan[j].count > res[i].count) atomicOr(&ctl->err, kErrUnmatched);
      else if (scan[j].count == res[i].count) dead[i] = 1u;
    }
  }
}

// U3: keys of the new voxels, compacted (new_pos = exclusive scan of is_new).
__global__ void update_new_keys_kernel(const Ctl *ctl, const VoxMoments *scan, const u32 *is_new, const u32 *new_pos, u64 *new_keys) {
  const u32 n_scan = ctl->n_voxels;
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n_scan; j += gridDim.x * blockDim.x)
    if (is_new[j]) new_keys[new_pos[j]] = scan[j].key;
}

// U4: size of the merged table, capacity check BEFORE anything is written, control block ready
// for a back-end run.  n_new = new_pos[n_scan], n_dead = dead_pos[n_res] (the scans' totals).
__global__ void update_prepare_kernel(Ctl *ctl, u32 n_res, const u32 *new_pos, const u32 *dead_pos, u32 max_voxels, u32 *n_new_out) {
  if (threadIdx.x || blockIdx.x) return;
  const u32 n_scan = ctl->n_voxels;
  const u32 n_new = new_pos[n_scan], n_dead = dead_pos ? dead_pos[n_res] : 0u;
  *n_new_out = n_new;
  ctl->n_voxels_scan = n_scan;
  if ((u64)n_res + n_new - n_dead > (u64)max_voxels) atomicOr(&ctl->err, kErrCapacity);
  ctl->n_voxels = n_res + n_new - n_dead;
  ctl->ticket[7] = 0;
  ctl->n_columns = 0; ctl->n_slopes = 0; ctl->n_fitted = 0;
}

// U5: resident voxel i moves to i + (new keys below it) - (dead voxels below it), fused with
// (add) or relieved of (remove) the scan voxel matched to it.
__global__ void update_merge_resident_kernel(const Ctl *ctl, const VoxMoments *res, u32 n_res, const VoxMoments *scan, int sign,
                                             const u32 *inv, const u64 *new_keys, const u32 *n_new_p, const u32 *dead,
                                             const u32 *dead_pos, VoxMoments *out) {
  if (ctl->err) return;
  const u32 n_new = *n_new_p;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_res; i += gridDim.x * blockDim.x) {
    if (sign < 0 && dead[i]) continue;
    VoxMoments v = res[i];
    const u32 j = inv[i];
    if (j != kNone) {
      const VoxMoments s = scan[j];
      Moments a, b;
      load_moments(v, a);
      load_moments(s, b);
      if (sign > 0) { merge_moments(a, b); v.first = min(v.first, s.first); }  // resident points came first in the concatenated cloud
      else unmerge_moments(a, b);
      v.count = (u32)a.n;
#pragma unroll
      for (int k = 0; k < 3; ++k) v.m[k] = a.m[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) v.s[k] = a.s[k];
    }
    const u32 dst = i + (n_new ? lower_bound_u64(new_keys, n_new, v.key) : 0u) - (sign < 0 ? dead_pos[i] : 0u);
    out[dst] = v;
  }
}

// U6 (add): new voxel with rank r moves to r + (number of resident keys below it).
__global__ void update_merge_new_kernel(const Ctl *ctl, const VoxMoments *res, u32 n_res, const VoxMoments *scan, const u32 *is_new,
                                        const u32 *new_pos, VoxMoments *out) {
  if (ctl->err) return;
  const u32 n_scan = ctl->n_voxels_scan;
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n_scan; j += gridDim.x * blockDim.x) {
    if (!is_new[j]) continue;
    const VoxMoments v = scan[j];
    out[new_pos[j] + lower_bound_key(res, n_res, v.key)] = v;
  }
}

// ---- the cells a scan touched (changeMorton_list, src/receiver.cpp:47-56: the xy keys of the
// scan's points in first-touched order; republished alone by showInital(change_pub,...,1), :203-206)

// C1: per scan voxel: its column in the NEW column table (binary search on (cx, cy)); keep the
// smallest cloud index that touched the column.
__global__ void changed_mark_kernel(const Ctl *ctl, const VoxMoments *scan, const gndt_column *columns, u32 *touch_first) {
  const u32 n_scan = ctl->n_voxels_scan, C = ctl->n_columns;
  if (ctl->err) return;
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n_scan; j += gridDim.x * blockDim.x) {
    const u64 key = scan[j].key;
    const int cx = (int)(u32)(key >> 32) - kIdxBias, cy = (int)((u32)(key >> 16) & 0xFFFFu) - kIdxBias;
    u32 lo = 0, hi = C;
    while (lo < hi) {
      const u32 mid = (lo + hi) >> 1;
      const int mx = columns[mid].sx > 0 ? columns[mid].sx - 1 : columns[mid].sx, my = columns[mid].sy > 0 ? columns[mid].sy - 1 : columns[mid].sy;
      if (mx < cx || (mx == cx && my < cy)) lo = mid + 1; else hi = mid;
    }
    if (lo < C) {
      const int mx = columns[lo].sx > 0 ? columns[lo].sx - 1 : columns[lo].sx, my = columns[lo].sy > 0 ? columns[lo].sy - 1 : columns[lo].sy;
      if (mx == cx && my == cy) atomicMin(&touch_first[lo], scan[j].first);  // a column that vanished (remove) is not listed
    }
  }
}
// C2: the column whose first touch was scan point k goes to slot k (cloud indices are distinct).
__global__ void changed_order_kernel(const Ctl *ctl, const u32 *touch_first, u32 idx_offset, u32 n_points, u32 *order, u32 *valid) {
  const u32 C = ctl->n_columns;
  if (ctl->err) return;
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    const u32 f = touch_first[c];
    if (f == kNone) continue;
    const u32 k = f - idx_offset;
    if (k < n_points) { order[k] = c; valid[k] = 1u; }
  }
}
// C3: compaction in slot order (pos = exclusive scan of valid).
__global__ void changed_compact_kernel(const u32 *order, const u32 *valid, const u32 *pos, u32 n_points, u32 *changed) {
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < n_points; k += gridDim.x * blockDim.x)
    if (valid[k]) changed[pos[k]] = order[k];
}

}  // namespace gndt
