// gndt_reduce.cuh — per-voxel moments on the partitioned cloud and the closed-form eigen
// solver used to finish a voxel.
//
// Replaces the fitting half of TwoDmap::create2DMap (reference include/map2D.h:606-627:
// pcl::compute3DCentroid + pcl::computeCovarianceMatrix per OcNode with >= MINPOINTSIZE
// points) and OcNode::countRoughNormal (map2D.h:110-133, Eigen::EigenSolver).
//
// Numerics: the reference sums sequentially in binary32.  Here every run (= voxel) is
// accumulated in binary64 about its own first point (differences of two floats are exact in
// binary64), giving (n, mean, centred scatter); runs that straddle tiles are merged with
// Chan's pairwise update.  Results are rounded to binary32 once, in the finalize kernel.
// Shifting by a point of the run keeps the reference's exact zeros (all points sharing a
// coordinate -> that scatter row is exactly 0), which its `roughness == 0 -> 0.01` rule
// (map2D.h:131-132) depends on.
#pragma once
#include "gndt_device.cuh"

namespace gndt {

constexpr int kRedThreads = 256;
constexpr int kRedMinBlocks = 5;                   // resident reduce CTAs per SM (__launch_bounds__)
constexpr int kRedItems = 8;
constexpr int kRedTile = kRedThreads * kRedItems;  // 2048 points
constexpr int kLongRun = 64;                        // longer runs are reduced by a whole warp each
constexpr int kMaxLong = kRedTile / kLongRun;

struct Moments {
  double n;
  double m[3];  // mean
  double s[6];  // centred scatter xx,xy,xz,yy,yz,zz
};

// Device-resident per-voxel state (96 B, 16-byte aligned): what the finalize kernel turns
// into a record and what the streaming merge (gndt_update) accumulates into.
struct __align__(16) VoxMoments {
  u64 key;      // voxel_key(cx,cy,cz)
  u32 count;
  u32 first;    // cloud index of the first point
  double m[3];  // mean relative to the cell centre (cell_anchor)
  double s[6];
  u64 pad;
};

// Centre of a voxel's cell in binary64, from its key, the origin and the cell lengths.  Means are
// kept relative to it: every partial of one voxel shares the anchor, so merges need no change, and
// the inverse merge (unmerge_moments) cancels means of at most a cell's size instead of absolute
// coordinates, whose rounding it would amplify by (points before) / (points after).
__device__ __forceinline__ double anchor_axis(u32 biased, float o, float len) {
  return __fma_rn((double)((int)biased - kIdxBias) + 0.5, (double)len, (double)o);
}
__device__ __forceinline__ void cell_anchor(u64 key, const float o[3], float grid_len, float z_len, double a[3]) {
  a[0] = anchor_axis((u32)(key >> 32), o[0], grid_len);
  a[1] = anchor_axis((u32)(key >> 16) & 0xFFFFu, o[1], grid_len);
  a[2] = anchor_axis((u32)key & 0xFFFFu, o[2], z_len);
}

constexpr u32 kCarryHasLead = 1u, kCarryLeadContinues = 2u, kCarryHasTail = 4u;
struct TileCarry {
  u32 flags;
  u32 tail_slot;
  u32 pad[2];
  Moments lead;  // leading run when it continues a voxel begun in an earlier tile
};

// Chan et al. pairwise combination of two (n, mean, centred scatter) triples.
__device__ __forceinline__ void merge_moments(Moments &a, const Moments &b) {
  if (b.n == 0.0) return;
  if (a.n == 0.0) { a = b; return; }
  const double n = a.n + b.n;
  const double d0 = b.m[0] - a.m[0], d1 = b.m[1] - a.m[1], d2 = b.m[2] - a.m[2];
  const double w = a.n * b.n / n, f = b.n / n;
  a.s[0] += b.s[0] + d0 * d0 * w; a.s[1] += b.s[1] + d0 * d1 * w; a.s[2] += b.s[2] + d0 * d2 * w;
  a.s[3] += b.s[3] + d1 * d1 * w; a.s[4] += b.s[4] + d1 * d2 * w; a.s[5] += b.s[5] + d2 * d2 * w;
  a.m[0] += d0 * f; a.m[1] += d1 * f; a.m[2] += d2 * f;
  a.n = n;
}

// Raw shifted sums (about the run's first point p0) -> (n, mean relative to the cell centre
// `anc`, centred scatter).
__device__ __forceinline__ void close_moments(Moments &mo, double n, const float4 &p0, const double anc[3],
                                              const double sd[3], const double sq[6]) {
  const double inv = 1.0 / n;
  const double m0 = sd[0] * inv, m1 = sd[1] * inv, m2 = sd[2] * inv;
  mo.n = n;
  mo.m[0] = ((double)p0.x - anc[0]) + m0; mo.m[1] = ((double)p0.y - anc[1]) + m1; mo.m[2] = ((double)p0.z - anc[2]) + m2;
  mo.s[0] = sq[0] - sd[0] * m0; mo.s[1] = sq[1] - sd[0] * m1; mo.s[2] = sq[2] - sd[0] * m2;
  mo.s[3] = sq[3] - sd[1] * m1; mo.s[4] = sq[4] - sd[1] * m2; mo.s[5] = sq[5] - sd[2] * m2;
}

// One plane rotation that diagonalises the 2x2 block (app apq; apq aqq): the closed form
// of a single Jacobi step.  Returns the rotated diagonal in place and (c, s).
__device__ __forceinline__ void sym2(double &app, double &aqq, double apq, double &c, double &s) {
  const double theta = (aqq - app) / (2.0 * apq);
  const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  c = 1.0 / sqrt(t * t + 1.0);
  s = t * c;
  app -= t * apq;
  aqq += t * apq;
}

// Closed-form eigen-decomposition of a symmetric 3x3 (a = xx,xy,xz,yy,yz,zz).
// w[k] / column k of V are eigenpairs; when the matrix decouples exactly (an axis whose
// off-diagonals are both 0.0) the pairs stay in axis order so that exact ties (e.g. two
// zero eigenvalues) are broken the same way the reference's strict-< chain breaks them on
// a solver that leaves a diagonal matrix untouched.  Otherwise: trigonometric solution of
// the characteristic cubic, eigenvalues ascending, eigenvectors by the largest cross
// product of rows of (A - wI).
__device__ void eig3_sym(const double a[6], double w[3], double V[3][3]) {
  const double a00 = a[0], a01 = a[1], a02 = a[2], a11 = a[3], a12 = a[4], a22 = a[5];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
  w[0] = a00; w[1] = a11; w[2] = a22;
  const int nz = (a01 != 0.0) + (a02 != 0.0) + (a12 != 0.0);
  if (nz == 0) return;
  if (nz == 1) {
    double c, s;
    if (a01 != 0.0) {
      sym2(w[0], w[1], a01, c, s);
      V[0][0] = c; V[1][0] = -s; V[0][1] = s; V[1][1] = c;
    } else if (a02 != 0.0) {
      sym2(w[0], w[2], a02, c, s);
      V[0][0] = c; V[2][0] = -s; V[0][2] = s; V[2][2] = c;
    } else {
      sym2(w[1], w[2], a12, c, s);
      V[1][1] = c; V[2][1] = -s; V[1][2] = s; V[2][2] = c;
    }
    return;
  }
  // general case, scaled to unit max-norm
  double sc = fmax(fmax(fabs(a00), fabs(a11)), fabs(a22));
  sc = fmax(sc, fmax(fmax(fabs(a01), fabs(a02)), fabs(a12)));
  const double inv = 1.0 / sc;
  const double b00 = a00 * inv, b01 = a01 * inv, b02 = a02 * inv, b11 = a11 * inv, b12 = a12 * inv, b22 = a22 * inv;
  const double q = (b00 + b11 + b22) / 3.0;
  const double c00 = b00 - q, c11 = b11 - q, c22 = b22 - q;
  const double p2 = c00 * c00 + c11 * c11 + c22 * c22 + 2.0 * (b01 * b01 + b02 * b02 + b12 * b12);
  const double p = sqrt(p2 / 6.0);
  const double ip = 1.0 / p;
  const double d00 = c00 * ip, d11 = c11 * ip, d22 = c22 * ip, d01 = b01 * ip, d02 = b02 * ip, d12 = b12 * ip;
  double r = 0.5 * (d00 * (d11 * d22 - d12 * d12) - d01 * (d01 * d22 - d12 * d02) + d02 * (d01 * d12 - d11 * d02));
  r = fmin(1.0, fmax(-1.0, r));
  const double phi = acos(r) / 3.0;
  const double e_max = q + 2.0 * p * cos(phi);
  const double e_min = q + 2.0 * p * cos(phi + 2.0943951023931954923);
  const double e_mid = 3.0 * q - e_max - e_min;
  const double ev[3] = {e_min, e_mid, e_max};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double l = ev[k];
    const double r0[3] = {b00 - l, b01, b02}, r1[3] = {b01, b11 - l, b12}, r2[3] = {b02, b12, b22 - l};
    double x0[3] = {r0[1] * r1[2] - r0[2] * r1[1], r0[2] * r1[0] - r0[0] * r1[2], r0[0] * r1[1] - r0[1] * r1[0]};
    double x1[3] = {r0[1] * r2[2] - r0[2] * r2[1], r0[2] * r2[0] - r0[0] * r2[2], r0[0] * r2[1] - r0[1] * r2[0]};
    double x2[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
    const double n0 = x0[0] * x0[0] + x0[1] * x0[1] + x0[2] * x0[2];
    const double n1 = x1[0] * x1[0] + x1[1] * x1[1] + x1[2] * x1[2];
    const double n2 = x2[0] * x2[0] + x2[1] * x2[1] + x2[2] * x2[2];
    double bx = x0[0], by = x0[1], bz = x0[2], bn = n0;
    if (n1 > bn) { bx = x1[0]; by = x1[1]; bz = x1[2]; bn = n1; }
    if (n2 > bn) { bx = x2[0]; by = x2[1]; bz = x2[2]; bn = n2; }
    if (bn > 0.0) {
      const double in = rsqrt(bn);
      V[0][k] = bx * in; V[1][k] = by * in; V[2][k] = bz * in;
    } else {  // triple eigenvalue: any basis
      V[0][k] = (k == 0); V[1][k] = (k == 1); V[2][k] = (k == 2);
    }
    w[k] = l * sc;
  }
}

struct __align__(128) RedSmem {
  float4 pts_raw[kRedTile + 2];  // [0] last point of the previous tile, [1..cnt] the tile, [cnt+1] first point of the next
  unsigned long long mbar;
  unsigned short run_start[kRedTile + 2];
  unsigned short long_list[kMaxLong];
  u64 row_last_key[kRedItems][8];  // key of the last lane of every (row, warp) for head detection
  u32 seg_cnt[kRedItems][8];
  double red[8][9];
  u64 prev_key, next_key, first_key, last_key;
  u32 n_long, tile_id, n_runs, vox_base;
};

template <bool FAST>
__device__ __forceinline__ u64 point_key(const float4 &p, const float o[3], const DevParams &P) {
  int cx, cy, cz;
  point_indices_masked<FAST>(p.x, p.y, p.z, o, P, 7, cx, cy, cz);  // partitioned points are all valid
  return voxel_key(cx, cy, cz);
}

__device__ __forceinline__ void store_moments(VoxMoments *dst, u64 key, u32 first, const Moments &mo) {
  VoxMoments v;
  v.key = key; v.count = (u32)mo.n; v.first = first;
#pragma unroll
  for (int k = 0; k < 3; ++k) v.m[k] = mo.m[k];
#pragma unroll
  for (int k = 0; k < 6; ++k) v.s[k] = mo.s[k];
  v.pad = 0;
  const double2 *q = reinterpret_cast<const double2 *>(&v);
  double2 *d = reinterpret_cast<double2 *>(dst);
#pragma unroll
  for (int i = 0; i < 6; ++i) d[i] = q[i];
}

// K3: one CTA per tile of 2048 sorted points -> raw moments of every voxel whose run starts
// in the tile; partial runs at the tile edges go to the carry array.
template <bool FAST>
__global__ void __launch_bounds__(kRedThreads, kRedMinBlocks)
reduce_kernel(Ctl *ctl, const float4 *buf_a, const float4 *buf_b, VoxMoments *mom, TileCarry *carry,
              u64 *tile_state, GroupState *tile_groups, DevParams P) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RedSmem &S = *reinterpret_cast<RedSmem *>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { S.tile_id = atomicAdd(&ctl->ticket[6], 1u); S.n_long = 0; mbar_init(&S.mbar, 1); }
  __syncthreads();
  const int tile = (int)S.tile_id;
  const size_t M = (size_t)ctl->n_valid;
  const size_t base = (size_t)tile * kRedTile;
  if (base >= M) return;
  const int cnt = (int)min((size_t)kRedTile, M - base);
  const float4 *src = ((ctl->n_passes - 1) & 1) ? buf_b : buf_a;  // pass p writes A when p is even
  const float o[3] = {ctl->origin[0], ctl->origin[1], ctl->origin[2]};
  float4 *pts = S.pts_raw + 1;

  // ---- stage the tile and its two neighbour points with one TMA bulk copy
  const bool has_prev = base > 0, has_next = base + cnt < M;
  if (tid == 0)
    tma_load_1d(S.pts_raw + (has_prev ? 0 : 1), src + base - (has_prev ? 1 : 0),
                (u32)(cnt + (has_prev ? 1 : 0) + (has_next ? 1 : 0)) * 16u, &S.mbar);
  if (!mbar_wait(&S.mbar, 0)) atomicOr(&ctl->err, kErrWatchdog);
  // voxel key per point in registers
  u64 key[kRedItems];
#pragma unroll
  for (int k = 0; k < kRedItems; ++k) {
    const int i = k * kRedThreads + tid;
    key[k] = ~0ull;
    if (i < cnt) key[k] = point_key<FAST>(pts[i], o, P);
    if (lane == 31) S.row_last_key[k][warp] = key[k];
    if (i == 0) S.first_key = key[k];
    if (i == cnt - 1) S.last_key = key[k];
  }
  if (tid == 0) S.prev_key = has_prev ? point_key<FAST>(S.pts_raw[0], o, P) : ~0ull;
  if (tid == 32) S.next_key = has_next ? point_key<FAST>(pts[cnt], o, P) : ~0ull;
  __syncthreads();

  // ---- run heads (position 0 always starts a run of this tile)
  u32 ball[kRedItems];
#pragma unroll
  for (int k = 0; k < kRedItems; ++k) {
    const int i = k * kRedThreads + tid;
    u64 before = __shfl_up_sync(0xffffffffu, key[k], 1);
    if (lane == 0) before = (warp > 0) ? S.row_last_key[k][warp - 1] : (k > 0 ? S.row_last_key[k - 1][7] : ~key[k]);
    const bool head = (i < cnt) && (i == 0 || key[k] != before);
    ball[k] = __ballot_sync(0xffffffffu, head);
    if (lane == 0) S.seg_cnt[k][warp] = __popc(ball[k]);
  }
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the 64 (k,warp) counts, two per lane
    u32 c0 = (&S.seg_cnt[0][0])[2 * lane], c1 = (&S.seg_cnt[0][0])[2 * lane + 1];
    u32 inc = c0 + c1;
#pragma unroll
    for (int o2 = 1; o2 < 32; o2 <<= 1) {
      u32 t = __shfl_up_sync(0xffffffffu, inc, o2);
      if (lane >= o2) inc += t;
    }
    const u32 exc = inc - (c0 + c1);
    (&S.seg_cnt[0][0])[2 * lane] = exc;
    (&S.seg_cnt[0][0])[2 * lane + 1] = exc + c0;
    if (lane == 31) S.n_runs = inc;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kRedItems; ++k) {
    const int i = k * kRedThreads + tid;
    if (ball[k] & (1u << lane)) S.run_start[S.seg_cnt[k][warp] + __popc(ball[k] & ((1u << lane) - 1u))] = (unsigned short)i;
  }
  const int n_runs = (int)S.n_runs;
  const bool first_is_head = S.prev_key != S.first_key;
  const bool last_complete = S.next_key != S.last_key;
  const u32 heads = (u32)n_runs - (first_is_head ? 0u : 1u);
  if (tid == 0) S.run_start[n_runs] = (unsigned short)cnt;
  __syncthreads();

  // ---- one thread per run: shifted one-pass sums from shared memory (first round kept in
  //      registers so that the look-back below overlaps with nothing but finished work)
  auto run_moments = [&](int j, Moments &mo, u64 &key) -> bool {
    const int s = S.run_start[j], e = S.run_start[j + 1];
    if (e - s > kLongRun) {
      S.long_list[atomicAdd(&S.n_long, 1u)] = (unsigned short)j;
      return false;
    }
    const float4 p0 = pts[s];
    key = point_key<FAST>(p0, o, P);
    double anc[3];
    cell_anchor(key, o, P.grid_len, P.z_len, anc);
    double sd[3] = {0, 0, 0}, sq[6] = {0, 0, 0, 0, 0, 0};
    for (int i = s + 1; i < e; ++i) {
      const float4 p = pts[i];
      const double dx = (double)p.x - (double)p0.x, dy = (double)p.y - (double)p0.y, dz = (double)p.z - (double)p0.z;
      sd[0] += dx; sd[1] += dy; sd[2] += dz;
      sq[0] += dx * dx; sq[1] += dx * dy; sq[2] += dx * dz; sq[3] += dy * dy; sq[4] += dy * dz; sq[5] += dz * dz;
    }
    close_moments(mo, (double)(e - s), p0, anc, sd, sq);
    return true;
  };
  Moments mo0;
  u64 key0;
  const bool have0 = (tid < n_runs) && run_moments(tid, mo0, key0);

  if (warp == kRedThreads / 32 - 1) {  // the last warp has the fewest runs of its own: it resolves the voxel base
    const u64 vb = warp_lookback_grouped(tile_state, tile_groups, tile, 0u, heads, &ctl->err);
    if (lane == 0) S.vox_base = (u32)vb;
  }
  __syncthreads();
  const u32 vox_base = S.vox_base;
  if (tid == 0 && base + cnt == M) ctl->n_voxels = vox_base + heads;
  TileCarry *my_carry = carry + tile;

  auto emit = [&](int j, const Moments &mo, u64 key) {
    const int s = S.run_start[j];
    const bool cont = (j == 0) && !first_is_head;
    const bool open_end = (j == n_runs - 1) && !last_complete;
    const u32 slot = vox_base + (u32)j - (first_is_head ? 0u : 1u);
    if (cont) {
      my_carry->lead = mo;
      atomicOr(&my_carry->flags, kCarryHasLead | (open_end ? kCarryLeadContinues : 0u));
      return;
    }
    if (slot >= P.max_voxels) { atomicOr(&ctl->err, kErrCapacity); return; }
    store_moments(mom + slot, key, __float_as_uint(pts[s].w), mo);
    if (open_end) {
      my_carry->tail_slot = slot;
      atomicOr(&my_carry->flags, kCarryHasTail);
    }
  };
  if (have0) emit(tid, mo0, key0);
  for (int j = tid + kRedThreads; j < n_runs; j += kRedThreads) {
    Moments mo;
    u64 key;
    if (run_moments(j, mo, key)) emit(j, mo, key);
  }
  __syncthreads();

  // ---- longer runs (large cells, heavy voxels): one WARP per run, lanes stride over the
  //      run's points, fixed xor-shuffle tree (deterministic), no CTA-wide barriers
  const int n_long = (int)S.n_long;
  for (int l = warp; l < n_long; l += kRedThreads / 32) {
    const int j = S.long_list[l];
    const int s = S.run_start[j], e = S.run_start[j + 1];
    const float4 p0 = pts[s];
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = s + lane; i < e; i += 32) {
      const float4 p = pts[i];
      const double dx = (double)p.x - (double)p0.x, dy = (double)p.y - (double)p0.y, dz = (double)p.z - (double)p0.z;
      acc[0] += dx; acc[1] += dy; acc[2] += dz;
      acc[3] += dx * dx; acc[4] += dx * dy; acc[5] += dx * dz; acc[6] += dy * dy; acc[7] += dy * dz; acc[8] += dz * dz;
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = warp_sum(acc[k]);
    if (lane == 0) {
      const u64 key = point_key<FAST>(p0, o, P);
      double anc[3];
      cell_anchor(key, o, P.grid_len, P.z_len, anc);
      Moments mo;
      close_moments(mo, (double)(e - s), p0, anc, acc, acc + 3);
      emit(j, mo, key);
    }
  }
}

// K3b: voxels whose run straddles tiles.  One warp per tile: a tile whose last voxel
// continues into later tiles gathers the continuation tiles' leading partial moments 32 at
// a time (one per lane, loaded in parallel), merges them with a fixed shuffle tree
// (deterministic) and folds them into the voxel's stored moments.
__global__ void __launch_bounds__(128) fixup_kernel(Ctl *ctl, VoxMoments *mom, const TileCarry *carry) {
  pdl_wait();
  pdl_trigger();
  const size_t M = (size_t)ctl->n_valid;
  const int n_tiles = (int)((M + kRedTile - 1) / kRedTile);
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  for (int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < n_tiles; t += warps_total) {
    if (!(carry[t].flags & kCarryHasTail)) continue;  // warp-uniform
    Moments acc;
    acc.n = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) acc.m[k] = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) acc.s[k] = 0.0;
    for (int u0 = t + 1; u0 < n_tiles; u0 += 32) {
      const int u = u0 + lane;
      const u32 fl = (u < n_tiles) ? carry[u].flags : 0u;
      const u32 has_lead = __ballot_sync(0xffffffffu, (fl & kCarryHasLead) != 0);
      const u32 ends_here = __ballot_sync(0xffffffffu, (fl & kCarryHasLead) && !(fl & kCarryLeadContinues));
      const int stop_excl = (~has_lead) ? __ffs(~has_lead) - 1 : 32;  // first tile without a lead
      const int stop_incl = ends_here ? __ffs(ends_here) : 33;        // first tile where the voxel ends
      const int n_inc = min(stop_excl, stop_incl);
      Moments mine;
      mine.n = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) mine.m[k] = 0.0;
#pragma unroll
      for (int k = 0; k < 6; ++k) mine.s[k] = 0.0;
      if (lane < n_inc) mine = carry[u].lead;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {  // fixed tree: lane l absorbs lane l+o
        Moments other;
        other.n = __shfl_down_sync(0xffffffffu, mine.n, o);
#pragma unroll
        for (int k = 0; k < 3; ++k) other.m[k] = __shfl_down_sync(0xffffffffu, mine.m[k], o);
#pragma unroll
        for (int k = 0; k < 6; ++k) other.s[k] = __shfl_down_sync(0xffffffffu, mine.s[k], o);
        if (lane + o < 32) merge_moments(mine, other);
      }
      if (lane == 0) merge_moments(acc, mine);
      if (n_inc < 32 || ends_here) break;  // chain ended in this chunk, lane 31 included: later leads are other voxels' (warp-uniform)
    }
    if (lane == 0) {
      VoxMoments *v = mom + carry[t].tail_slot;
      Moments mo;
      mo.n = (double)v->count;
#pragma unroll
      for (int k = 0; k < 3; ++k) mo.m[k] = v->m[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) mo.s[k] = v->s[k];
      merge_moments(mo, acc);
      v->count = (u32)mo.n;
#pragma unroll
      for (int k = 0; k < 3; ++k) v->m[k] = mo.m[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) v->s[k] = mo.s[k];
    }
  }
}

}  // namespace gndt
