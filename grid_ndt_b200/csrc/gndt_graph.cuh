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

// Rules a caller's (slopes, columns) pair must follow; a violation sets its bit in the word the
// host reads back after the count pass (gndt_build_edges names the rule).
constexpr u32 kGraphBadIndex = 1u;   // a column's sx / sy is 0 or beyond +-GNDT_MAX_INDEX
constexpr u32 kGraphBadOrder = 2u;   // columns not sorted strictly by (cx, cy)
constexpr u32 kGraphBadRange = 4u;   // slope ranges not contiguous from 0 to n_slopes
constexpr u32 kGraphBadCell = 8u;    // a Slope's (sx, sy) is not its column's

__host__ __device__ __forceinline__ bool valid_signed_index(int s) { return s != 0 && s >= -GNDT_MAX_INDEX && s <= GNDT_MAX_INDEX; }

// G1: slope -> column map and the x-row directory of the column table.  Each column first checks
// itself against its predecessor and its own Slopes; one that breaks a rule sets `bad` and writes
// nothing, so every write below stays inside slope_col[0, S) and the rows [cx_lo, cx_hi].
__global__ void graph_prepare_kernel(const gndt_slope *slopes, u32 S, const gndt_column *columns, u32 C, int cx_lo, int cx_hi,
                                     u32 *slope_col, u32 *row_start, u32 *row_end, u32 *bad) {
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    const gndt_column col = columns[c];
    const int cx = contiguous_index(col.sx), cy = contiguous_index(col.sy);
    const u64 begin = col.slope_begin, end = begin + col.slope_count;
    u32 err = 0;
    if (!valid_signed_index(col.sx) || !valid_signed_index(col.sy) || cx < cx_lo || cx > cx_hi) err |= kGraphBadIndex;
    u64 want_begin = 0;
    if (c > 0) {
      const gndt_column prev = columns[c - 1];
      const int px = contiguous_index(prev.sx), py = contiguous_index(prev.sy);
      if (px > cx || (px == cx && py >= cy)) err |= kGraphBadOrder;
      want_begin = (u64)prev.slope_begin + prev.slope_count;
    }
    if (begin != want_begin || end > S || (c + 1 == C && end != S)) err |= kGraphBadRange;
    if (!err)
      for (u32 s = (u32)begin; s < (u32)end; ++s)
        if (slopes[s].sx != col.sx || slopes[s].sy != col.sy) { err |= kGraphBadCell; break; }
    if (err) { atomicOr(bad, err); continue; }
    for (u32 s = (u32)begin; s < (u32)end; ++s) slope_col[s] = c;
    mark_row(columns, C, c, cx, cx_lo, row_start, row_end);
  }
}

// G2 (FILL = false): number of reachable Slopes per Slope; G4 (FILL = true): the lists.  Does
// nothing when G1 found the tables malformed (slope_col and the directory are incomplete then).
template <bool FILL>
__global__ void __launch_bounds__(256)
graph_edges_kernel(const gndt_slope *slopes, u32 S, const gndt_column *columns, u32 C, const u32 *slope_col, const u32 *row_start,
                   const u32 *row_end, int cx_base, int n_rows, u32 *deg, const u32 *offsets, u32 *targets, const u32 *bad, DevParams P) {
  if (*bad) return;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < S; i += gridDim.x * blockDim.x) {
    const gndt_slope me = slopes[i];
    const float n[3] = {me.normal[0], me.normal[1], me.normal[2]};
    const double n_len = normal_length(n);
    u32 nb[4] = {C, C, C, C};
    neighbour_columns(columns, C, slope_col[i], contiguous_index(me.sx), contiguous_index(me.sy), row_start, row_end, cx_base, n_rows,
                      [&](int d, u32 c, const gndt_column &) { nb[d] = c; });
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
