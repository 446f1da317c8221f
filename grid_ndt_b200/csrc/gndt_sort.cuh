// gndt_sort.cuh — binning of the cloud by (cx,cy,cz): bounds pass, key-layout plan and a
// single-sweep LSD radix partition that moves the 16-byte points themselves.
//
// Replaces the reference's uniformDivision loop (src/receiver.cpp:41-93,150-154): there,
// every point walks a std::multimap<string,OcNode*> keyed by a decimal Morton string and
// is appended to its voxel's point list.  Here the cloud is stably partitioned so that
// each voxel is one contiguous run (in cloud order) and each x-y column is a contiguous
// run of voxels ordered by z.  Stability gives `first_index` (the first-seen order that
// the reference's isSlope depends on, SURVEY Q8) for free.
//
// Key = (column id << bz) | (cz - cz_min), column id = (cx - cx_min) * ny + (cy - cy_min)
// (mixed radix over the bounding box: no bits are spent on the slack of a power-of-two
// field).  The planner splits the key into the fewest digits of at most kMaxDigitBits bits
// (first digit: at most 8 bits, inside the z field, so that its histogram follows from the
// exact z histogram of the bounds pass).  cfg2 (600 x 400 columns, 46 z levels): 24 bits =
// 3 passes of 6 + 9 + 9 bits, where fixed power-of-two fields with 8-bit digits needed 4.
//
// Traffic per pass: read 16 B + write 16 B per point (one sweep, decoupled look-back).
// A tile is brought into shared memory by ONE TMA bulk copy (cp.async.bulk, completion on
// an mbarrier) and never passes through registers as a whole: threads read the coordinates
// their digit needs, rank, write a 4-byte permutation entry, and the copy-out gathers
// 16-byte points through it.  CTAs are persistent: a launch has (SMs x resident CTAs) of
// them and each takes tiles off a ticket counter in cloud order until none is left, so a
// pass costs one launch however many tiles it has and an unused pass costs a launch only.
#pragma once
#include "gndt_device.cuh"

namespace gndt {

constexpr int kSortThreads = 512;
constexpr int kSortItems = 8;
constexpr int kSortMinBlocks = 2;                     // resident partition CTAs per SM (__launch_bounds__)
constexpr int kSortTile = kSortThreads * kSortItems;  // points per tile
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kFirstMaxBits = 8;                      // first digit: fixed look-back stride, zeroed by the bounds pass
constexpr int kFirstMaxBins = 1 << kFirstMaxBits;
constexpr int kDigitsPerThread = (kMaxBins + kSortThreads - 1) / kSortThreads;
static_assert(kSortThreads % 32 == 0 && kSortTile < 65536 && 32 * kSortItems < 65536, "tile shape");
constexpr int kSortGroup = 16;               // tiles per look-back group
constexpr int kGroupSumBits = 26;            // group word: arrivals << 26 | sum of the tiles' digit counts
static_assert(kSortGroup >= 1 && kSortGroup < 64 && (long long)kSortGroup * kSortTile < (1ll << kGroupSumBits), "group word");

struct __align__(128) SortSmem {
  float4 in[kSortTile];            // the tile, in arrival order (TMA destination)
  u32 slot[kSortTile];             // digit << 16 | source position, in digit order; pass 0 first
                                   // uses this space for the histograms of the later digits
  unsigned short whist[kSortWarps * kMaxBins];  // per-warp digit counts, row stride = bins of the pass
  u32 tile_off[kMaxBins];
  u32 gbase[kMaxBins];
  u64 warp_sums[32];
  unsigned long long mbar;
  u32 tile_id;
  u32 n_valid_tile;
};
// later-digit histograms of pass 0: 16-bit counters packed in pairs, [kMaxPasses-1][kMaxBins]
static_assert((kMaxPasses - 1) * kMaxBins * 2 <= kSortTile * 4, "later-digit histograms alias slot[]");

// Load point i of a strided cloud (first 12 bytes of each record are x,y,z).
__device__ __forceinline__ float4 load_point(const float *in, size_t stride_f, size_t i, bool vec) {
  if (vec) return ld_stream(reinterpret_cast<const float4 *>(in) + i);
  const float *p = in + i * stride_f;
  return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), 0.f);
}

// grid-stride zero fill (16-byte stores) of a look-back region by a whole grid
__device__ __forceinline__ void grid_zero(void *p, size_t bytes) {
  uint4 *q = reinterpret_cast<uint4 *>(p);
  const size_t n = (bytes + 15) / 16;  // regions are 256-byte aligned with slack: rounding up is safe
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    q[i] = make_uint4(0u, 0u, 0u, 0u);
}

// ---------------------------------------------------------------------------------------
// K1a: bounds + exact histogram of the z index modulo kZHistBins + validity counters.
// The index map of transMortonXYZ (map2D.h:950-973) is monotone in each coordinate, so the
// index bounds are the indices of the coordinate bounds: this pass keeps min/max of the raw
// floats of valid points and divides only for the z index.  A point is valid iff
// |p - p0| <= P.max_abs[axis], the largest offset whose index is <= GNDT_MAX_INDEX (found on
// the host with the same IEEE operations).  The grid also zeroes the look-back words of the
// first partition pass (`lb0`, `glb0`).
// ---------------------------------------------------------------------------------------
template <bool FAST>
__global__ void __launch_bounds__(256) bounds_kernel(Ctl *ctl, u32 *zhist, const float *in,
                                                     size_t stride_f, size_t n_in, size_t start,
                                                     void *lb0, size_t lb0_bytes, void *glb0, size_t glb0_bytes,
                                                     DevParams P) {
  pdl_wait();
  pdl_trigger();
  __shared__ u32 sh[kZHistBins];
  __shared__ float red[6][8];
  __shared__ u32 cnt[3];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool vec = (stride_f == 4) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
  float o[3];
  if (P.origin_first) { o[0] = __ldg(in); o[1] = __ldg(in + 1); o[2] = __ldg(in + 2); }
  else { o[0] = P.origin[0]; o[1] = P.origin[1]; o[2] = P.origin[2]; }
  if (blockIdx.x == 0 && tid == 0) { ctl->origin[0] = o[0]; ctl->origin[1] = o[1]; ctl->origin[2] = o[2]; }
  for (int i = tid; i < kZHistBins; i += 256) sh[i] = 0;
  if (tid < 3) cnt[tid] = 0;
  __syncthreads();
  const bool tiled = P.tile_lo < P.tile_hi;
  const float inf = __int_as_float(0x7f800000);
  float lo_x = inf, lo_y = inf, lo_z = inf, hi_x = -inf, hi_y = -inf, hi_z = -inf;
  u32 n_ok = 0, n_drop = 0, n_out = 0;
  // One point of the pass: validity (NaN / Inf / index range), strip filter, bounds, z histogram.
  // All lanes stay converged so that the warp-aggregated histogram update sees full warps.
  auto visit = [&](const float4 &p, bool live) {
    const float ax = fabsf(__fsub_rn(p.x, o[0])), ay = fabsf(__fsub_rn(p.y, o[1])), az = fabsf(__fsub_rn(p.z, o[2]));
    bool ok = live && ax <= P.max_abs[0] && ay <= P.max_abs[0] && az <= P.max_abs[1];
    n_drop += (live && !ok) ? 1u : 0u;
    if (tiled && ok) {
      int cx;
      axis_index<FAST>(p.x, o[0], P.grid_len, P.rinv[0], cx);
      if (cx < P.tile_lo || cx >= P.tile_hi) { n_out++; ok = false; }
    }
    u32 d = kInvalidDigit;
    if (ok) {
      n_ok++;
      lo_x = fminf(lo_x, p.x); lo_y = fminf(lo_y, p.y); lo_z = fminf(lo_z, p.z);
      hi_x = fmaxf(hi_x, p.x); hi_y = fmaxf(hi_y, p.y); hi_z = fmaxf(hi_z, p.z);
      const int cz = axis_index_valid<FAST>(p.z, o[2], P.z_len, P.rinv[1]);
      d = (u32)(cz + kIdxBias) & (u32)(kZHistBins - 1);
    }
    const u32 peers = __match_any_sync(0xffffffffu, d);  // flat scenes: most lanes share a z bin
    if (ok && lane == __ffs(peers) - 1) atomicAdd(&sh[d], (u32)__popc(peers));
  };
  // chunks of 256 x 4 points; whole chunks need no per-point range test
  constexpr int kUnroll = 4, kChunk = 256 * kUnroll;
  const size_t n_pts = n_in - start, n_chunks = (n_pts + kChunk - 1) / kChunk;
  for (size_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    const size_t i0 = start + c * kChunk + tid;
    float4 p[kUnroll];
    if ((c + 1) * kChunk <= n_pts) {
#pragma unroll
      for (int u2 = 0; u2 < kUnroll; ++u2) p[u2] = load_point(in, stride_f, i0 + u2 * 256, vec);
#pragma unroll
      for (int u2 = 0; u2 < kUnroll; ++u2) visit(p[u2], true);
    } else {
#pragma unroll
      for (int u2 = 0; u2 < kUnroll; ++u2) {
        const size_t i = i0 + u2 * 256;
        p[u2] = (i < n_in) ? load_point(in, stride_f, i, vec) : make_float4(inf, inf, inf, 0.f);
      }
#pragma unroll
      for (int u2 = 0; u2 < kUnroll; ++u2) visit(p[u2], i0 + u2 * 256 < n_in);
    }
  }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    lo_x = fminf(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, o2)); lo_y = fminf(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, o2));
    lo_z = fminf(lo_z, __shfl_xor_sync(0xffffffffu, lo_z, o2)); hi_x = fmaxf(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, o2));
    hi_y = fmaxf(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, o2)); hi_z = fmaxf(hi_z, __shfl_xor_sync(0xffffffffu, hi_z, o2));
    n_ok += __shfl_xor_sync(0xffffffffu, n_ok, o2); n_drop += __shfl_xor_sync(0xffffffffu, n_drop, o2);
    n_out += __shfl_xor_sync(0xffffffffu, n_out, o2);
  }
  if (lane == 0) {
    red[0][warp] = hi_x; red[1][warp] = hi_y; red[2][warp] = hi_z; red[3][warp] = lo_x; red[4][warp] = lo_y; red[5][warp] = lo_z;
    atomicAdd(&cnt[0], n_ok); atomicAdd(&cnt[1], n_drop); atomicAdd(&cnt[2], n_out);
  }
  __syncthreads();
  if (tid < 6 && cnt[0]) {
    float m = red[tid][0];
    for (int w = 1; w < 8; ++w) m = (tid < 3) ? fmaxf(m, red[tid][w]) : fminf(m, red[tid][w]);
    const int ax = tid % 3;
    int c;
    axis_index<FAST>(m, o[ax], ax == 2 ? P.z_len : P.grid_len, ax == 2 ? P.rinv[1] : P.rinv[0], c);  // index of the extreme coordinate
    atomicMax(&ctl->max_cx_b + tid, (u32)((tid < 3 ? c : -c) + kIdxBias));
  }
  if (tid == 0) {
    if (cnt[0]) atomicAdd(&ctl->n_valid, (u64)cnt[0]);
    if (cnt[1]) atomicAdd(&ctl->n_dropped, (u64)cnt[1]);
    if (cnt[2]) atomicAdd(&ctl->n_outside, (u64)cnt[2]);
  }
  for (int i = tid; i < kZHistBins; i += 256)
    if (sh[i]) atomicAdd(&zhist[i], sh[i]);
  grid_zero(lb0, lb0_bytes);
  grid_zero(glb0, glb0_bytes);
}

__device__ __forceinline__ int bit_width(u32 v) { return 32 - __clz(v); }

// ---------------------------------------------------------------------------------------
// K1b: derive the key layout from the bounds and split the key into the fewest digits:
// P = smallest pass count for which  first digit <= min(bz, 8)  and every other digit
// <= kMaxDigitBits; the bits are then spread evenly.  The histogram of the first digit
// (a function of cz alone) is folded out of the z histogram.  One CTA of kZHistBins threads.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kZHistBins) plan_kernel(Ctl *ctl, const u32 *zhist, u32 *hist_all) {
  pdl_wait();
  pdl_trigger();
  __shared__ int s_mask0, s_czminb;
  const int tid = threadIdx.x;
  if (tid == 0) {
    if (ctl->n_valid == 0) {
      ctl->cx_min = ctl->cy_min = ctl->cz_min = 0; ctl->ny = 1; ctl->bcol = 1; ctl->bz = 1;
      ctl->n_passes = 1; ctl->shift[0] = 0; ctl->bits[0] = 1; ctl->cx_max = 0;
      s_mask0 = 1; s_czminb = kIdxBias;
    } else {
      const int cx_max = (int)ctl->max_cx_b - kIdxBias, cy_max = (int)ctl->max_cy_b - kIdxBias, cz_max = (int)ctl->max_cz_b - kIdxBias;
      const int cx_min = kIdxBias - (int)ctl->max_ncx_b, cy_min = kIdxBias - (int)ctl->max_ncy_b, cz_min = kIdxBias - (int)ctl->max_ncz_b;
      const u32 nx = (u32)(cx_max - cx_min) + 1u, ny = (u32)(cy_max - cy_min) + 1u, nz = (u32)(cz_max - cz_min) + 1u;
      const int bz = max(1, bit_width(nz - 1u));
      const int bcol = max(1, bit_width(nx * ny - 1u));  // nx, ny <= 65535: the product fits 32 bits
      ctl->cx_min = cx_min; ctl->cy_min = cy_min; ctl->cz_min = cz_min; ctl->cx_max = cx_max;
      ctl->ny = ny; ctl->bz = bz; ctl->bcol = bcol;
      const int B = bz + bcol;
      int P = max(2, (B + kMaxDigitBits - 1) / kMaxDigitBits), b0 = 0;  // B >= bz + 1: never one pass
      for (;; ++P) {
        const int w = (B + P - 1) / P;
        b0 = min(min(bz, kFirstMaxBits), w);
        if ((B - b0 + P - 2) / (P - 1) <= kMaxDigitBits) break;
      }
      if (P > kMaxPasses) { P = kMaxPasses; atomicOr(&ctl->err, kErrWatchdog); }  // cannot happen: B <= 48
      ctl->n_passes = P;
      ctl->shift[0] = 0; ctl->bits[0] = b0;
      int s = b0;
      const int R = B - b0;
      for (int p = 1; p < P; ++p) {
        const int b = R / (P - 1) + (p <= R % (P - 1) ? 1 : 0);
        ctl->shift[p] = s; ctl->bits[p] = b;
        s += b;
      }
      s_mask0 = (1 << b0) - 1;
      s_czminb = cz_min + kIdxBias;
    }
  }
  __syncthreads();
  // first digit = (cz - cz_min) mod 2^b0 = (a - (cz_min + bias)) mod 2^b0 for a = (cz + bias) mod 1024
  const u32 c = zhist[tid];
  if (c) atomicAdd(&hist_all[(u32)(tid - s_czminb) & (u32)s_mask0], c);
}

// 64-bit exclusive scan over the CTA (any multiple of 32 threads up to 1024).
__device__ __forceinline__ u64 block_exclusive_scan64(u64 v, u64 *warp_sums) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  u64 inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u64 t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();  // previous users of warp_sums are done
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  const u64 ws = (lane < n_warps) ? warp_sums[lane] : 0ull;
  u64 winc = ws;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u64 t = __shfl_up_sync(0xffffffffu, winc, o);
    if (lane >= o) winc += t;
  }
  const u64 wexc = __shfl_sync(0xffffffffu, winc - ws, warp);
  return wexc + inc - v;
}

// ---------------------------------------------------------------------------------------
// K2: one radix partition pass.  FIRST=true reads the caller's cloud (any stride), drops
// invalid / out-of-strip points, tags each survivor with its cloud index in .w and builds
// the digit histograms of ALL later passes; FIRST=false moves already-tagged points between
// the two work buffers and evaluates only the key fields its digit covers.
//
// Per tile:
//  1. the tile is fetched into shared memory by one TMA bulk copy (strided / unaligned
//     caller clouds fall back to per-thread loads)
//  2. stable in-tile rank: __match_any_sync groups equal digits inside a warp, per-warp
//     digit counters in shared memory, then a scan across the warps per digit
//  3. tile digit counts are published for the decoupled look-back while the permutation
//     (digit, source position) is written in digit order
//  4. copy-out: consecutive threads gather their point through the permutation and write
//     consecutive addresses inside a digit run
// A pass of up to 2^10 digits gives each of the first ceil(bins / m) threads m consecutive
// digits (m = ceil(bins / threads)).  `lb_next` / `glb_next`: look-back words of the NEXT
// pass, zeroed here by the whole grid (their size depends on that pass's digit width).
// ---------------------------------------------------------------------------------------
template <bool FIRST, bool FAST>
__global__ void __launch_bounds__(kSortThreads, kSortMinBlocks)
sort_pass_kernel(Ctl *ctl, int pass, const float *in_raw, size_t stride_f, size_t n_in, size_t start,
                 const float4 *src, float4 *dst, u32 *lb, u64 *glb, u32 *lb_next, u64 *glb_next, u32 *hist_all,
                 DevParams P) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(128) unsigned char smem_sort[];
  SortSmem &S = *reinterpret_cast<SortSmem *>(smem_sort);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int n_passes = ctl->n_passes;
  if (pass >= n_passes) return;
  const size_t M = FIRST ? (n_in - start) : (size_t)ctl->n_valid;
  const size_t n_tiles = (M + kSortTile - 1) / kSortTile;
  if (pass + 1 < n_passes) {  // the next pass's look-back words (free since pass - 1 finished)
    const size_t n_next = ((size_t)ctl->n_valid + kSortTile - 1) / kSortTile;
    const size_t bins_next = (size_t)1 << ctl->bits[pass + 1];
    grid_zero(lb_next, n_next * bins_next * sizeof(u32));
    grid_zero(glb_next, ((n_next + kSortGroup - 1) / kSortGroup) * bins_next * sizeof(u64));
  }
  if (tid == 0) mbar_init(&S.mbar, 1);

  const int bits = ctl->bits[pass];
  const int n_bins = 1 << bits;  // digits of this pass
  const int m_eff = (n_bins + kSortThreads - 1) / kSortThreads;  // digits per owner thread
  const int d0 = tid * m_eff;                                    // first digit this thread owns
  const KeyLayout L = load_layout(ctl);
  const int shift = ctl->shift[pass];
  const u32 mask = (1u << bits) - 1u;
  const float o[3] = {ctl->origin[0], ctl->origin[1], ctl->origin[2]};
  const bool tiled = P.tile_lo < P.tile_hi;
  // key fields this pass's digit overlaps: z [0,bz), column id [bz, ...)
  const bool need_col = FIRST || (shift + bits > L.bz), need_z = FIRST || (shift < L.bz);
  const int need = (need_col ? 3 : 0) | (need_z ? 4 : 0);
  int q_shift[kMaxPasses];
  u32 q_mask[kMaxPasses];
#pragma unroll
  for (int q = 0; q < kMaxPasses; ++q) {
    q_shift[q] = FIRST ? ctl->shift[q] : 0;
    q_mask[q] = FIRST ? ((1u << ctl->bits[q]) - 1u) : 0u;
  }
  // global digit counts and bases of this pass: the same for every tile
  u32 global_count[kDigitsPerThread];
  u32 digit_base[kDigitsPerThread];
  {
    u64 sum = 0;
#pragma unroll
    for (int j = 0; j < kDigitsPerThread; ++j) {
      const int d = d0 + j;
      global_count[j] = (j < m_eff && d < n_bins) ? hist_all[(size_t)pass * kMaxBins + d] : 0u;
      sum += global_count[j];
    }
    u64 run = block_exclusive_scan64(sum, S.warp_sums);
#pragma unroll
    for (int j = 0; j < kDigitsPerThread; ++j) { digit_base[j] = (u32)run; run += global_count[j]; }
  }
  u32 *later_hist = S.slot;  // packed 16-bit counters [kMaxPasses-1][kMaxBins], pass 0 only
  const bool vec = !FIRST || ((stride_f == 4) && ((reinterpret_cast<uintptr_t>(in_raw) & 15) == 0));

  for (u32 it = 0;; ++it) {
    __syncthreads();  // everyone is done with the previous tile's shared memory
    if (tid == 0) S.tile_id = atomicAdd(&ctl->ticket[pass], 1u);
    for (int i = tid; i < (kSortWarps * n_bins) / 2; i += kSortThreads) reinterpret_cast<u32 *>(S.whist)[i] = 0;
    if (FIRST)
      for (int i = tid; i < (n_passes - 1) * (kMaxBins / 2); i += kSortThreads) later_hist[i] = 0;
    __syncthreads();
    const size_t tile = S.tile_id;
    if (tile >= n_tiles) break;
    const size_t base = tile * kSortTile;
    const int cnt = (int)min((size_t)kSortTile, M - base);

    // ---- 1. tile -> shared memory
    if (vec) {
      if (tid == 0) {
        const float4 *g = FIRST ? reinterpret_cast<const float4 *>(in_raw) + start + base : src + base;
        tma_load_1d(S.in, g, (u32)cnt * 16u, &S.mbar);
      }
      if (!mbar_wait(&S.mbar, it & 1)) atomicOr(&ctl->err, kErrWatchdog);
    } else {
      for (int i = tid; i < cnt; i += kSortThreads) S.in[i] = load_point(in_raw, stride_f, start + base + i, false);
      __syncthreads();
    }

    // ---- digits
    u32 dg[kSortItems];
#pragma unroll
    for (int k = 0; k < kSortItems; ++k) {
      const int i = warp * (32 * kSortItems) + k * 32 + lane;
      dg[k] = kInvalidDigit;
      if (i < cnt) {
        const float4 e = S.in[i];
        int cx, cy, cz;
        if (FIRST) {
          bool ok = point_indices<FAST>(e.x, e.y, e.z, o, P.grid_len, P.z_len, P.rinv[0], P.rinv[1], cx, cy, cz);
          if (ok && tiled && (cx < P.tile_lo || cx >= P.tile_hi)) ok = false;
          if (ok) {
            const u64 key = compact_key(cx, cy, cz, L);
            dg[k] = (u32)key & mask;
#pragma unroll
            for (int q = 1; q < kMaxPasses; ++q)
              if (q < n_passes) {
                const u32 b = (u32)(key >> q_shift[q]) & q_mask[q];
                atomicAdd(&later_hist[(q - 1) * (kMaxBins / 2) + (b >> 1)], (b & 1u) ? 0x10000u : 1u);
              }
          }
        } else {
          point_indices_masked<FAST>(e.x, e.y, e.z, o, P, need, cx, cy, cz);
          u64 key = 0;
          if (need_col) key = (u64)column_id(cx, cy, L) << L.bz;
          if (need_z) key |= (u64)(u32)(cz - L.cz_min);
          dg[k] = (u32)(key >> shift) & mask;
        }
      }
    }

    // ---- 2. stable rank inside the warp's block of points
    unsigned short *my_hist = S.whist + warp * n_bins;
    u32 rank[kSortItems];
#pragma unroll
    for (int k = 0; k < kSortItems; ++k) {
      const u32 peers = __match_any_sync(0xffffffffu, dg[k]);
      const int leader = __ffs(peers) - 1;
      const u32 r = __popc(peers & ((1u << lane) - 1u));
      u32 old = 0;
      if (lane == leader && dg[k] != kInvalidDigit) {
        old = my_hist[dg[k]];
        my_hist[dg[k]] = (unsigned short)(old + __popc(peers));
      }
      old = __shfl_sync(0xffffffffu, old, leader);
      rank[k] = old + r;
      __syncwarp();
    }
    __syncthreads();

    // pass 0: the histograms of the later digits leave shared memory before slot[] reuses it
    if (FIRST) {
      for (int i = tid; i < (n_passes - 1) * (kMaxBins / 2); i += kSortThreads) {
        const u32 c = later_hist[i];
        if (c) {
          u32 *g = hist_all + (size_t)(1 + i / (kMaxBins / 2)) * kMaxBins + 2 * (i % (kMaxBins / 2));
          if (c & 0xFFFFu) atomicAdd(g, c & 0xFFFFu);
          if (c >> 16) atomicAdd(g + 1, c >> 16);
        }
      }
    }

    // ---- 3. per owned digit: scan over the warps, tile count, publication.  A digit takes
    // part in the look-back only if some point of the cloud has it (global count != 0).
    u32 tile_count[kDigitsPerThread];
    u32 *lb_tile = lb + tile * (size_t)n_bins;
    u64 *glb_grp = glb + (tile / kSortGroup) * (size_t)n_bins;
    u32 tsum = 0;
#pragma unroll
    for (int j = 0; j < kDigitsPerThread; ++j) {
      tile_count[j] = 0;
      if (global_count[j]) {
        const int d = d0 + j;
        u32 c = 0;
#pragma unroll 4
        for (int w = 0; w < kSortWarps; ++w) {
          const u32 t = S.whist[w * n_bins + d];
          S.whist[w * n_bins + d] = (unsigned short)c;
          c += t;
        }
        tile_count[j] = c;
        st_relaxed(lb_tile + d, (tile == 0 ? kFlagIncl : kFlagAgg) | c);
        atomicAdd(reinterpret_cast<u32 *>(glb_grp + d), (1u << kGroupSumBits) | c);
      }
      tsum += tile_count[j];
    }
    // exclusive scan of the tile counts over the digits
    u32 toff[kDigitsPerThread];
    {
      u32 run = block_exclusive_scan(tsum, reinterpret_cast<u32 *>(S.warp_sums));
#pragma unroll
      for (int j = 0; j < kDigitsPerThread; ++j) {
        toff[j] = run;
        run += tile_count[j];
        if (j < m_eff && d0 + j < n_bins) S.tile_off[d0 + j] = toff[j];
      }
      if (tid == kSortThreads - 1) S.n_valid_tile = run;
    }
    __syncthreads();  // also orders the later_hist reads above before the slot[] writes below

    // ---- permutation in digit order (stable)
#pragma unroll
    for (int k = 0; k < kSortItems; ++k) {
      if (dg[k] != kInvalidDigit) {
        const u32 pos = S.tile_off[dg[k]] + my_hist[dg[k]] + rank[k];
        S.slot[pos] = (dg[k] << 16) | (u32)(warp * (32 * kSortItems) + k * 32 + lane);
      }
    }

    // ---- decoupled look-back per owned digit, two levels
    // Tiles are also summed per GROUP of kSortGroup consecutive tiles: each tile adds its count
    // to the group's word with one atomic whose top bits count arrivals, so a complete group
    // costs one load instead of kSortGroup.  The walk is: own group's earlier tiles (tile
    // words), then whole groups backwards until a group that already knows its inclusive prefix.
    // The digits a thread owns walk together: every round trip carries the loads of all of them.
    {
      constexpr int kLookBatch = 8;
      u32 prefix[kDigitsPerThread];
      bool done[kDigitsPerThread];
      bool all_done = true;
#pragma unroll
      for (int j = 0; j < kDigitsPerThread; ++j) {
        prefix[j] = 0;
        done[j] = !(j < m_eff && d0 + j < n_bins && tile > 0 && global_count[j] != 0);
        all_done &= done[j];
      }
      const long long grp = (long long)(tile / kSortGroup);
      const long long lo = grp * kSortGroup, tl = (long long)tile;
      for (long long t = tl - 1; t >= lo && !all_done; t -= kLookBatch) {
        u32 w[kDigitsPerThread][kLookBatch];
#pragma unroll
        for (int j = 0; j < kDigitsPerThread; ++j)
#pragma unroll
          for (int q = 0; q < kLookBatch; ++q)
            w[j][q] = (!done[j] && t - q >= lo) ? ld_relaxed(lb_tile + d0 + j - (size_t)(tl - (t - q)) * n_bins) : 0u;
        all_done = true;
#pragma unroll
        for (int j = 0; j < kDigitsPerThread; ++j) {
#pragma unroll
          for (int q = 0; q < kLookBatch; ++q) {
            if (done[j] || t - q < lo) break;
            u32 spins = 0;
            while ((w[j][q] & kFlagMask) == 0 && ++spins < kSpinLimit)
              w[j][q] = ld_relaxed(lb_tile + d0 + j - (size_t)(tl - (t - q)) * n_bins);
            if ((w[j][q] & kFlagMask) == 0) { atomicOr(&ctl->err, kErrWatchdog); done[j] = true; break; }
            prefix[j] += w[j][q] & kValMask;
            if (w[j][q] & kFlagIncl) done[j] = true;
          }
          all_done &= done[j];
        }
      }
      for (long long g = grp - 1; g >= 0 && !all_done; g -= kLookBatch) {
        u64 w[kDigitsPerThread][kLookBatch];
#pragma unroll
        for (int j = 0; j < kDigitsPerThread; ++j)
#pragma unroll
          for (int q = 0; q < kLookBatch; ++q)
            w[j][q] = (!done[j] && g - q >= 0) ? ld_relaxed64(glb + d0 + j + (size_t)(g - q) * n_bins) : 0ull;
        all_done = true;
#pragma unroll
        for (int j = 0; j < kDigitsPerThread; ++j) {
#pragma unroll
          for (int q = 0; q < kLookBatch; ++q) {
            if (done[j] || g - q < 0) break;
            u32 spins = 0;  // ready: inclusive prefix known (high word) or all kSortGroup tiles have arrived
            while (!((u32)(w[j][q] >> 32) & kFlagIncl) && ((u32)w[j][q] >> kGroupSumBits) != (u32)kSortGroup && ++spins < kSpinLimit)
              w[j][q] = ld_relaxed64(glb + d0 + j + (size_t)(g - q) * n_bins);
            const u32 hi = (u32)(w[j][q] >> 32), low = (u32)w[j][q];
            if (hi & kFlagIncl) { prefix[j] += hi & kValMask; done[j] = true; }
            else if ((low >> kGroupSumBits) == (u32)kSortGroup) prefix[j] += low & ((1u << kGroupSumBits) - 1u);
            else { atomicOr(&ctl->err, kErrWatchdog); done[j] = true; }
          }
          all_done &= done[j];
        }
      }
#pragma unroll
      for (int j = 0; j < kDigitsPerThread; ++j) {
        if (j < m_eff && d0 + j < n_bins) {
          const int d = d0 + j;
          if (tile > 0 && global_count[j]) {
            st_relaxed(lb_tile + d, kFlagIncl | (prefix[j] + tile_count[j]));
            if (tl - lo == kSortGroup - 1)  // last tile of its group: the group's inclusive prefix
              st_relaxed(reinterpret_cast<u32 *>(glb_grp + d) + 1, kFlagIncl | (prefix[j] + tile_count[j]));
          }
          S.gbase[d] = digit_base[j] + prefix[j] - toff[j];
        }
      }
    }
    __syncthreads();

    // ---- 4. copy out through the permutation
    const int n_valid_tile = (int)S.n_valid_tile;
    for (int i = tid; i < n_valid_tile; i += kSortThreads) {
      const u32 s = S.slot[i];
      const u32 from = s & 0xFFFFu;
      float4 e = S.in[from];
      if (FIRST) e.w = __uint_as_float(P.idx_offset + (u32)(start + base + from));
      st_stream(dst + S.gbase[s >> 16] + i, e);
    }
  }
}

}  // namespace gndt
