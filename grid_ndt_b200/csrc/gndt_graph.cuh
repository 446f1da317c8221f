// gndt_graph.cuh — the traversability graph as CSR: for every Slope the list of Slopes that
// TwoDmap::AccessibleNeighbors returns for it.
//
// Replaces, for the host planner, the per-expansion work of AccessibleNeighbors
// (reference include/map2D.h:530-548): substr / strToInt / mortonToXY of the cell key,
// countLRFB (:197-263, four countMorton strings), four map_cell.find() on strings and the
// countReachable scan (:266-296) of each neighbour cell's Slopes with countAngle (:477-482).
// The 4 reach BITS of edges_kernel say "a reachable Slope exists to the L/R/F/B"; the
// cost-map expansion (computeCost, :1285-1397) and A* (GlobalPlan.h:79-83) need the Slopes
// themselves, several layers per neighbour cell.  List order = the reference's: left, right,
// forward, back cell; inside a cell ascending z (std::map<int, Slope*> order).
// Predicate = countReachable with comand 2.5 / 4 and the checkList variant (:284-287,306-315):
// `reachable` of gndt_label.cuh, which also decides the reach bits.  (The 3-D comparison
// variant countReachable3D, :323-338, has no `up` test and is not reproduced.)
//
// Works from a (slopes, columns) table pair alone — a single GPU's or the gathered tables of
// a multi-GPU map — and builds its own x-row directory.
#pragma once
#include "gndt_device.cuh"
#include "gndt_label.cuh"
#include "gndt_scan.cuh"

namespace gndt {

// G1: slope -> column map and the x-row directory of the column table.
__global__ void graph_prepare_kernel(const gndt_column *columns, u32 C, int cx_base, u32 *slope_col, u32 *row_start, u32 *row_end) {
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    const gndt_column col = columns[c];
    for (u32 s = col.slope_begin; s < col.slope_begin + col.slope_count; ++s) slope_col[s] = c;
    const int cx = contiguous_index(col.sx);
    if (c == 0 || contiguous_index(columns[c - 1].sx) != cx) row_start[cx - cx_base] = c;
    if (c + 1 == C || contiguous_index(columns[c + 1].sx) != cx) row_end[cx - cx_base] = c + 1;
  }
}

// Column index of cell (ncx, cy) given the x-row directory, or C if the cell is empty.
__device__ __forceinline__ u32 find_in_row(const gndt_column *columns, u32 C, const u32 *row_start, const u32 *row_end, int cx_base,
                                           int n_rows, int ncx, int cy) {
  const int r = ncx - cx_base;
  if (r < 0 || r >= n_rows) return C;
  u32 lo = row_start[r], hi = row_end[r];
  const u32 end = hi;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (contiguous_index(columns[mid].sy) < cy) lo = mid + 1; else hi = mid;
  }
  return (lo < end && contiguous_index(columns[lo].sy) == cy) ? lo : C;
}

// G2 (FILL = false): number of reachable Slopes per Slope; G4 (FILL = true): the lists.
template <bool FILL>
__global__ void __launch_bounds__(256)
graph_edges_kernel(const gndt_slope *slopes, u32 S, const gndt_column *columns, u32 C, const u32 *slope_col, const u32 *row_start,
                   const u32 *row_end, int cx_base, int n_rows, u32 *deg, const u32 *offsets, u32 *targets, DevParams P) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < S; i += gridDim.x * blockDim.x) {
    const gndt_slope me = slopes[i];
    const int cx = contiguous_index(me.sx), cy = contiguous_index(me.sy);
    const u32 ci = slope_col[i];
    const float n[3] = {me.normal[0], me.normal[1], me.normal[2]};
    const double n_len = normal_length(n);
    u32 nb[4] = {C, C, C, C};  // left (cy-1), right (cy+1), forward (cx+1), back (cx-1): countLRFB in contiguous indices
    if (ci > 0 && contiguous_index(columns[ci - 1].sx) == cx && contiguous_index(columns[ci - 1].sy) == cy - 1) nb[0] = ci - 1;
    if (ci + 1 < C && contiguous_index(columns[ci + 1].sx) == cx && contiguous_index(columns[ci + 1].sy) == cy + 1) nb[1] = ci + 1;
    nb[2] = find_in_row(columns, C, row_start, row_end, cx_base, n_rows, cx + 1, cy);
    nb[3] = find_in_row(columns, C, row_start, row_end, cx_base, n_rows, cx - 1, cy);
    u32 k = 0;
    const u32 base = FILL ? offsets[i] : 0u;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      if (nb[d] == C) continue;
      const gndt_column c = columns[nb[d]];
      for (u32 s = c.slope_begin; s < c.slope_begin + c.slope_count; ++s) {
        const gndt_slope &t = slopes[s];
        if (!reachable(t.normal, t.rough, t.mean[2], t.flags, n, n_len, me.mean[2], P)) continue;
        if (FILL) targets[base + k] = s;
        ++k;
      }
    }
    if (!FILL) deg[i] = k;
  }
}

}  // namespace gndt
