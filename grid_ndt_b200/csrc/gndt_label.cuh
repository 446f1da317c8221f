// gndt_label.cuh — multi-level surface labels, Cell/Slope tables and local traversability.
//
// Replaces OcNode::isSlope (reference include/map2D.h:66-108), Slope::countUp (:147-177),
// the Slope/Cell emission of create2DMap (:598-599,630-660) and the per-edge predicates of
// countLRFB / countReachable / countAngle (:197-296,477-482).
//
// The table is sorted by (cx,cy,cz), so a voxel's vertical neighbours are the adjacent
// records (the contiguous index has no gap at the -1/+1 crossing, map2D.h:69-75) and its
// left/right neighbour cells are the adjacent columns; forward/back cells are found by a
// binary search inside the neighbouring x row.
#pragma once
#include "gndt_device.cuh"
#include "gndt_reduce.cuh"

namespace gndt {

constexpr int kLabelThreads = 256;

__device__ __forceinline__ int contiguous_index(int s) { return s > 0 ? s - 1 : s; }

// isSlope restated in closed form (SURVEY Q8): processing order inside a column is
// ascending first_index; a neighbour u contributes its centroid z only if it was fitted
// BEFORE v (count >= min_points and first(u) < first(v)), else the constructor's 0.
//   up(v)   = exists u at cz+1: |seen_z(u|v) - mean_z(v)| > slope_interval   (binary32)
//   down(v) = same at cz-1;   is_slope = fitted && !up          (demand "slope")
// demand "true": every fitted voxel is a Slope, down = false, up = countUp on FINAL
// centroids (no order dependence).
//
// K4: one thread per voxel, straight from the raw binary64 moments:
//   * finish the voxel — binary32 mean / scatter, closed-form eigen, rough, normal
//     (create2DMap's fit + countRoughNormal, map2D.h:621-623,110-133)
//   * label it — the isSlope / countUp rules restated above, against the adjacent records
//   * compact Slopes and Cells — CTA scan + decoupled look-back over (columns, slopes)
// and write the 96-byte record exactly once.
struct __align__(128) FinSmem {
  VoxMoments in[kLabelThreads + 2];  // in[j] <-> voxel v0 - 1 + j (one halo record on each side)
  float4 out[kLabelThreads * 6];     // the block's 256 finished 96-byte records
  unsigned long long mbar;
  u64 prefix;
  u32 warp_sums[32];
  u32 tile, total;
};

// 256 voxel threads + one helper warp: the helper publishes the block's (columns, slopes)
// counts and resolves their prefix (two L2 round trips) WHILE the voxel warps do the eigen work.
constexpr int kFinThreads = kLabelThreads + 32;
constexpr int kFinMinBlocks = 3;  // resident finalize CTAs per SM (__launch_bounds__)
__global__ void __launch_bounds__(kFinThreads, kFinMinBlocks)
finalize_label_kernel(Ctl *ctl, const VoxMoments *mom, gndt_voxel *table, gndt_slope *slopes,
                      gndt_column *columns, u32 *vfirst, u32 *slope_col, u64 *blk_state, GroupState *blk_groups, u32 *counters,
                      DevParams P) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(128) unsigned char smem_fin[];
  FinSmem &S = *reinterpret_cast<FinSmem *>(smem_fin);
  const int tid = threadIdx.x;
  const bool helper = tid >= kLabelThreads;
  if (ctl->err) return;  // e.g. capacity exceeded: the moments table is incomplete
  const u32 V = ctl->n_voxels;
  const u32 n_blocks = (V + kLabelThreads - 1) / kLabelThreads;
  const float o[3] = {ctl->origin[0], ctl->origin[1], ctl->origin[2]};
  // absolute mean z of a record (the moments hold it relative to the cell centre, gndt_reduce.cuh)
  auto mean_z = [&](const VoxMoments &r) { return (float)(r.m[2] + anchor_axis((u32)r.key & 0xFFFFu, o[2], P.z_len)); };
  if (tid == 0) mbar_init(&S.mbar, 1);
  for (u32 it = 0;; ++it) {
    __syncthreads();  // everyone is done with in[] / out[] of the previous block
    if (tid == 0) S.tile = atomicAdd(&counters[0], 1u);
    __syncthreads();
    const u32 blk = S.tile;
    if (blk >= n_blocks) return;
    const u32 v0 = blk * kLabelThreads;
    const u32 cnt = min((u32)kLabelThreads, V - v0);
    // one TMA bulk copy brings the block's moments plus one neighbour record on each side
    if (tid == 0) {
      const u32 lo = v0 > 0 ? v0 - 1 : 0, hi = min(v0 + cnt + 1, V);
      tma_load_1d(&S.in[lo + 1 - v0], mom + lo, (hi - lo) * (u32)sizeof(VoxMoments), &S.mbar);
    }
    if (!mbar_wait(&S.mbar, it & 1)) atomicOr(&ctl->err, kErrWatchdog);
    const u32 v = v0 + tid;
    const bool live = !helper && tid < (int)cnt;

    // ---- phase 1 (cheap): labels from the record headers
    u64 key = 0;
    u32 count = 0, first = 0, flags = 0;
    float mz = 0.f;
    bool head = false, fitted = false;
    if (live) {
      const VoxMoments &me = S.in[tid + 1];
      key = me.key; count = me.count; first = me.first;
      fitted = (int)count >= P.min_points;
      mz = mean_z(me);
      const bool has_lo = (v > 0) && (S.in[tid].key >> 16) == (key >> 16);
      const bool has_hi = (v + 1 < V) && (S.in[tid + 2].key >> 16) == (key >> 16);
      head = !has_lo;
      if (fitted) {
        flags = GNDT_F_FITTED;
        bool up = false, down = false;
        const bool ordered = (P.demand == GNDT_DEMAND_SLOPE);
        if (has_hi && (S.in[tid + 2].key & 0xFFFFu) == (key & 0xFFFFu) + 1) {
          const VoxMoments &hi = S.in[tid + 2];
          const bool seen = (int)hi.count >= P.min_points && (!ordered || hi.first < first);
          up = fabsf(__fsub_rn(seen ? mean_z(hi) : 0.f, mz)) > P.slope_interval;
        }
        if (ordered && has_lo && (S.in[tid].key & 0xFFFFu) + 1 == (key & 0xFFFFu)) {
          const VoxMoments &lo = S.in[tid];
          const bool seen = (int)lo.count >= P.min_points && lo.first < first;
          down = fabsf(__fsub_rn(seen ? mean_z(lo) : 0.f, mz)) > P.slope_interval;
        }
        if (up) flags |= GNDT_F_UP;
        if (down) flags |= GNDT_F_DOWN;
        if (P.demand == GNDT_DEMAND_TRUE || !up) flags |= GNDT_F_SLOPE;
      }
      if (head) flags |= GNDT_F_COLUMN_HEAD;
    }
    const bool slope = (flags & GNDT_F_SLOPE) != 0;
    const u32 packed = ((head ? 1u : 0u) << 16) | (slope ? 1u : 0u);
    const u32 exc = block_exclusive_scan(packed, S.warp_sums);
    if (tid == kLabelThreads - 1) S.total = exc + packed;
    __syncthreads();

    if (helper) {
      // ---- the block's (columns, slopes) prefix, resolved behind the voxel warps' eigen work
      const u32 total = S.total;
      const u64 pre = warp_lookback_grouped(blk_state, blk_groups, (int)blk, total >> 16, total & 0xFFFFu, &ctl->err);
      if (tid == kLabelThreads) {
        S.prefix = pre;
        if (blk == n_blocks - 1) {
          const u64 incl = pre + pack_pair(total >> 16, total & 0xFFFFu);
          ctl->n_columns = (u32)(incl >> 31);
          ctl->n_slopes = (u32)(incl & 0x7FFFFFFFu);
        }
      }
    } else if (live) {
      // ---- phase 2: finish the voxel (binary32 mean / scatter, eigen) into shared memory
      float f[24];
#pragma unroll
      for (int i = 0; i < 24; ++i) f[i] = 0.f;
      u32 *u = reinterpret_cast<u32 *>(f);
      const int cx = (int)(u32)(key >> 32) - kIdxBias, cy = (int)((u32)(key >> 16) & 0xFFFFu) - kIdxBias,
                cz = (int)((u32)key & 0xFFFFu) - kIdxBias;
      u[0] = (u32)signed_index(cx); u[1] = (u32)signed_index(cy); u[2] = (u32)signed_index(cz);
      u[3] = count; u[4] = first;
      if (fitted) {
        const VoxMoments &me = S.in[tid + 1];
        f[5] = (float)(me.m[0] + anchor_axis((u32)(key >> 32), o[0], P.grid_len));
        f[6] = (float)(me.m[1] + anchor_axis((u32)(key >> 16) & 0xFFFFu, o[1], P.grid_len));
        f[7] = mz;
        double a[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          float sc = (float)me.s[k];
          if (P.normalize_cov) sc = __fdiv_rn(sc, (float)count);
          f[8 + k] = sc;
          a[k] = (double)sc;  // the reference's solver sees the binary32 matrix (map2D.h:111)
        }
        double w[3], Vv[3][3];
        eig3_sym(a, w, Vv);
        // OcNode::countRoughNormal's strict-< chain on the solver's diagonal (map2D.h:114-130)
        const float e0 = (float)w[0], e1 = (float)w[1], e2 = (float)w[2];
        int k;
        if (e0 < e1) k = (e0 < e2) ? 0 : 2; else k = (e1 < e2) ? 1 : 2;
        float rough = (float)w[k];
        if (rough == 0.f) rough = 0.01f;  // map2D.h:131-132
        double s0 = w[0], s1 = w[1], s2 = w[2], t;
        if (s0 > s1) { t = s0; s0 = s1; s1 = t; }
        if (s1 > s2) { t = s1; s1 = s2; s2 = t; }
        if (s0 > s1) { t = s0; s0 = s1; s1 = t; }
        f[14] = (float)s0; f[15] = (float)s1; f[16] = (float)s2;
        f[17] = (float)(k == 0 ? Vv[0][0] : (k == 1 ? Vv[0][1] : Vv[0][2]));
        f[18] = (float)(k == 0 ? Vv[1][0] : (k == 1 ? Vv[1][1] : Vv[1][2]));
        f[19] = (float)(k == 0 ? Vv[2][0] : (k == 1 ? Vv[2][1] : Vv[2][2]));
        f[20] = rough;
      }
      u[21] = flags;
#pragma unroll
      for (int i = 0; i < 6; ++i) S.out[tid * 6 + i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
      vfirst[v] = first;
    }
    const u32 fitted_cnt = __syncthreads_count(live && fitted);  // joins the helper: S.prefix is final
    if (tid == 0 && fitted_cnt) atomicAdd(&ctl->n_fitted, fitted_cnt);

    // ---- phase 3: the compacted indices, Slope and Cell records
    if (live) {
      const u32 cols_before = (u32)(S.prefix >> 31) + (exc >> 16);
      const u32 slopes_before = (u32)(S.prefix & 0x7FFFFFFFu) + (exc & 0xFFFFu);
      const u32 col_idx = cols_before + (head ? 1u : 0u) - 1u;
      float4 *rec = S.out + tid * 6;
      float4 last = rec[5];  // rough flags column slope
      last.z = __uint_as_float(col_idx);
      last.w = __uint_as_float(slope ? slopes_before : 0xFFFFFFFFu);
      rec[5] = last;
      if (slope || head) {
        const float4 r0 = rec[0], r1 = rec[1];  // sx sy sz count | first mean.xyz
        if (slope) {
          const float4 r4 = rec[4];             // evals[2] normal.xyz
          float4 *d = reinterpret_cast<float4 *>(slopes + slopes_before);
          d[0] = make_float4(r0.x, r0.y, r0.z, r1.y);        // sx sy sz mean.x
          d[1] = make_float4(r1.z, r1.w, r4.y, r4.z);        // mean.y mean.z normal.x normal.y
          d[2] = make_float4(r4.w, last.x, __uint_as_float(flags), __uint_as_float(v));
          slope_col[slopes_before] = col_idx;  // compact: the edge kernel need not touch the 96-byte record for it
        }
        if (head) {
          float4 *d = reinterpret_cast<float4 *>(columns + col_idx);
          d[0] = make_float4(r0.x, r0.y, r1.x, __uint_as_float(v));                   // sx sy first voxel_begin
          d[1] = make_float4(0.f, __uint_as_float(slopes_before), 0.f, 0.f);          // count slope_begin count rsvd
        }
      }
    }
    // ---- the 256 records leave shared memory as one TMA bulk store
    tma_store_fence();
    __syncthreads();
    if (tid == 0) {
      tma_store_1d(table + v0, S.out, cnt * (u32)sizeof(gndt_voxel));
      tma_store_wait_read();  // out[] may be overwritten after the next barrier
    }
  }
}

// K4b: one thread per column: extents, first-seen index (position in the reference's
// morton_list, src/receiver.cpp:70), the x-row directory used by the edge search, and the
// voxel ranges of the first and last x row (Ctl::first_row_end / last_row_begin) for the halo.
__global__ void column_finish_kernel(Ctl *ctl, const u32 *vfirst, gndt_column *columns, u32 *row_start, u32 *row_end) {
  pdl_wait();
  pdl_trigger();
  const u32 V = ctl->n_voxels, C = ctl->n_columns, S = ctl->n_slopes;
  const int cx_min = ctl->cx_min, cx_max = ctl->cx_max;
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    gndt_column col = columns[c];
    const u32 v_end = (c + 1 < C) ? columns[c + 1].voxel_begin : V;
    const u32 s_end = (c + 1 < C) ? columns[c + 1].slope_begin : S;
    u32 first = 0xFFFFFFFFu;
    for (u32 v = col.voxel_begin; v < v_end; ++v) first = min(first, vfirst[v]);
    columns[c].first_index = first;
    columns[c].voxel_count = v_end - col.voxel_begin;
    columns[c].slope_count = s_end - col.slope_begin;
    const int cx = contiguous_index(col.sx);
    if (c == 0 || contiguous_index(columns[c - 1].sx) != cx) {
      row_start[cx - cx_min] = c;
      if (cx == cx_max) ctl->last_row_begin = col.voxel_begin;
    }
    if (c + 1 == C || contiguous_index(columns[c + 1].sx) != cx) {
      row_end[cx - cx_min] = c + 1;
      if (cx == cx_min) ctl->first_row_end = v_end;
    }
  }
}

// TwoDmap::countAngle (map2D.h:477-482) in the reference's own mixed precision: binary32
// dot product, binary64 norms (pow(float,int) -> double), quotient stored to float,
// acos(float), degrees via *180 (float) then /M_PI (double) stored to float, folded to
// <= 90.  res > 1 gives NaN, which fails the <= test exactly like the reference.
__device__ __forceinline__ double normal_length(const float a[3]) {
  return sqrt(__dadd_rn(__dadd_rn(__dmul_rn((double)a[0], (double)a[0]), __dmul_rn((double)a[1], (double)a[1])),
                        __dmul_rn((double)a[2], (double)a[2])));
}
// l2 = normal_length(b): the same value for every neighbour of one Slope, computed once.
__device__ __forceinline__ float count_angle(const float a[3], const float b[3], double l2) {
  float dot = __fmul_rn(a[0], b[0]);
  dot = __fadd_rn(dot, __fmul_rn(a[1], b[1]));
  dot = __fadd_rn(dot, __fmul_rn(a[2], b[2]));
  const double l1 = normal_length(a);
  const float res = (float)((double)dot / __dmul_rn(l1, l2));
  const float deg = __fmul_rn(acosf(res), 180.f);
  float an = (float)((double)deg / 3.14159265358979323846);
  if (an > 90.f) an = __fsub_rn(180.f, an);
  return an;
}

// Is the Slope (normal tn, rough, mean z tz, flags) reachable from the Slope with (normal n,
// n_len = normal_length(n), mean z mz)?  countReachable's four tests (map2D.h:276-279 / 284-287;
// thresholds robot.h:38-46).  They are a pure conjunction, so the cheap ones run first and the
// angle (two binary64 divisions, a square root and acosf) only for candidates that pass them.
__device__ __forceinline__ bool reachable(const float tn[3], float rough, float tz, u32 flags, const float n[3], double n_len,
                                          float mz, const DevParams &P) {
  return !(flags & GNDT_F_UP) && rough <= P.rough_max && fabsf(__fsub_rn(tz, mz)) <= P.reach_height &&
         count_angle(tn, n, n_len) <= P.angle_max_deg;
}

// Does neighbour cell `c` hold a Slope reachable from (normal n, mean z)?
__device__ __forceinline__ bool cell_reachable(const gndt_column &c, const gndt_slope *slopes, const float n[3],
                                               double n_len, float mz, const DevParams &P) {
  for (u32 s = c.slope_begin; s < c.slope_begin + c.slope_count; ++s) {
    const gndt_slope &t = slopes[s];
    if (reachable(t.normal, t.rough, t.mean[2], t.flags, n, n_len, mz, P)) return true;
  }
  return false;
}

// K5: one thread per Slope in [begin, begin+count): left/right = adjacent columns of the
// same x row, forward/back = binary search for the same cy in the neighbouring x rows.
// Index arithmetic is in contiguous space, which is countLRFB's quadrant crossing
// (x==1 / y==1 cases, map2D.h:219-253) without the special cases.
__global__ void __launch_bounds__(256)
edges_kernel(Ctl *ctl, gndt_voxel *table, gndt_slope *slopes, const gndt_column *columns, const u32 *slope_col,
             const u32 *row_start, const u32 *row_end, DevParams P) {
  pdl_wait();
  pdl_trigger();
  const u32 S = ctl->n_slopes, C = ctl->n_columns;
  const int cx_base = ctl->cx_min, cx_max = ctl->cx_max;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < S; i += gridDim.x * blockDim.x) {
    gndt_slope me = slopes[i];
    const int cx = contiguous_index(me.sx), cy = contiguous_index(me.sy);
    const u32 ci = slope_col[i];
    const float n[3] = {me.normal[0], me.normal[1], me.normal[2]};
    const double n_len = normal_length(n);
    u32 bits = 0;
    if (ci > 0) {  // left: cy-1
      const gndt_column c = columns[ci - 1];
      if (contiguous_index(c.sx) == cx && contiguous_index(c.sy) == cy - 1 && cell_reachable(c, slopes, n, n_len, me.mean[2], P))
        bits |= GNDT_F_REACH_L;
    }
    if (ci + 1 < C) {  // right: cy+1
      const gndt_column c = columns[ci + 1];
      if (contiguous_index(c.sx) == cx && contiguous_index(c.sy) == cy + 1 && cell_reachable(c, slopes, n, n_len, me.mean[2], P))
        bits |= GNDT_F_REACH_R;
    }
#pragma unroll
    for (int dir = 0; dir < 2; ++dir) {  // forward: cx+1, back: cx-1
      const int ncx = cx + (dir == 0 ? 1 : -1);
      if (ncx < cx_base || ncx > cx_max) continue;
      // first column of the neighbour row with cy' >= cy.  Neighbouring rows of a map are
      // populated alike, so the same offset as in the own row is a good first guess; gallop
      // from it to bracket cy, then bisect the bracket (1-3 probes instead of log2(row)).
      const u32 r_lo = row_start[ncx - cx_base], r_hi = row_end[ncx - cx_base];
      u32 lo = r_lo, hi = r_hi;
      if (r_lo < r_hi) {
        const u32 g = r_lo + min(ci - row_start[cx - cx_base], r_hi - r_lo - 1u);
        if (contiguous_index(columns[g].sy) < cy) {
          lo = g + 1;
          for (u32 step = 1;; step <<= 1) {
            const u32 probe = lo + step - 1;
            if (probe >= r_hi) { hi = r_hi; break; }
            if (contiguous_index(columns[probe].sy) >= cy) { hi = probe; break; }
            lo = probe + 1;
          }
        } else {
          hi = g;
          for (u32 step = 1;; step <<= 1) {
            if (hi < r_lo + step) { lo = r_lo; break; }
            const u32 probe = hi - step;
            if (contiguous_index(columns[probe].sy) < cy) { lo = probe + 1; break; }
            hi = probe;
          }
        }
      }
      while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (contiguous_index(columns[mid].sy) < cy) lo = mid + 1; else hi = mid;
      }
      if (lo < row_end[ncx - cx_base]) {
        const gndt_column c = columns[lo];
        if (contiguous_index(c.sy) == cy && cell_reachable(c, slopes, n, n_len, me.mean[2], P))
          bits |= (dir == 0 ? GNDT_F_REACH_F : GNDT_F_REACH_B);
      }
    }
    if (bits) {
      slopes[i].flags = me.flags | bits;
      table[me.voxel].flags |= bits;
    }
  }
}

}  // namespace gndt
