// gndt_exchange.cuh — multi-GPU x strips: thin halo + gather of the finished tables.
//
// SURVEY §8(e): every quantity up to the surface labels depends on one x-y column only, so the
// strips are built without communication.  What crosses GPUs is (1) the first / last x row of a
// strip, for the forward / back reach bits of the neighbour's boundary row (countLRFB's
// neighbours, reference include/map2D.h:219-253, that live on another GPU), and (2) the
// finished tables, so that every GPU (and the host planner behind it) holds the whole map.
//
// The halo row format, its packer, the boundary-edge kernel and the index rule of a gathered voxel
// record serve two transports: the caller's own (gndt_halo_pack / gndt_halo_edges /
// gndt_apply_strip_offsets, e.g. over NCCL) and the library's, through peer-mapped memory
// (NVLink / NVSwitch), no NCCL, no host round trip (gndt_xchg_*).
//
// In the library's transport every rank owns one exchange buffer that its peers map (cudaIpc
// between processes, plain peer access inside one process): a mailbox, two halo rows, and the
// gathered tables.  All traffic is PUSHED by the producer with ordinary stores to the peer's
// buffer, followed by a system-scope fence and an epoch flag in the peer's mailbox; consumers spin
// on flags in their OWN memory.  Strip sizes never visit the host: ranks publish their counts to
// every mailbox and every rank derives the offsets of all strips on the device.
//
//   publish   counts of this strip -> every mailbox
//   halo_send first row -> nearest non-empty lower strip, last row -> nearest non-empty upper strip
//             (empty strips are skipped: their neighbours exchange rows with each other)
//   halo_edges once both rows have arrived
//   push      this strip's voxel / slope / column records, strip-local indices made global on the
//             fly, into every rank's gathered tables at the strip's offset; then a `done` flag
//   wait      until every strip has arrived here
#pragma once
#include "gndt_device.cuh"
#include "gndt_label.cuh"

namespace gndt {

// ---- the halo, shared by both transports --------------------------------------------------

struct HaloHeader {  // occupies the first 96-byte slot of a halo buffer
  u32 count;         // records that follow (0 when the strip is empty or the row did not fit)
  int cx;            // contiguous x index of the packed row
  u32 overflow;      // row larger than the buffer: the receiver raises GNDT_ERR_CAPACITY
  u32 pad[21];
};
static_assert(sizeof(HaloHeader) == sizeof(gndt_voxel), "header uses one record slot");

// Pack the strip's first (last = false) or last x row into `out`: header + up to cap records.
// Called by every thread of one CTA, which copies cooperatively.
__device__ __forceinline__ void pack_halo_row(const Ctl *ctl, const gndt_voxel *table, bool last, gndt_voxel *out, u32 cap) {
  const u32 V = ctl->n_voxels;
  u32 lo = 0, hi = 0;
  int cx = 0;
  if (V && ctl->n_columns && !ctl->err) {
    lo = last ? ctl->last_row_begin : 0u;
    hi = last ? V : ctl->first_row_end;
    cx = last ? ctl->cx_max : ctl->cx_min;
  }
  const u32 n = hi - lo;
  const bool fits = n <= cap;
  HaloHeader *hdr = reinterpret_cast<HaloHeader *>(out);
  if (threadIdx.x == 0) { hdr->count = fits ? n : 0; hdr->cx = cx; hdr->overflow = fits ? 0u : 1u; }
  if (!fits) return;
  const float4 *src = reinterpret_cast<const float4 *>(table + lo);
  float4 *dst = reinterpret_cast<float4 *>(out + 1);
  for (u32 i = threadIdx.x; i < n * 6; i += blockDim.x) dst[i] = src[i];
}

// Block 0 packs the first x row into `first_out`, block 1 the last x row into `last_out`.
__global__ void __launch_bounds__(256)
halo_pack_kernel(const Ctl *ctl, const gndt_voxel *table, gndt_voxel *first_out, gndt_voxel *last_out, u32 cap) {
  const bool last = blockIdx.x == 1;
  pack_halo_row(ctl, table, last, last ? last_out : first_out, cap);
}

// Does the halo row hold, in the column with contiguous y index `cy`, a Slope reachable from
// (normal n, n_len = normal_length(n), mean z)?  Halo records are voxels sorted by (cy, cz).
__device__ __forceinline__ bool halo_reachable(const gndt_voxel *halo, u32 n_halo, int cy, const float n[3], double n_len,
                                               float mz, const DevParams &P) {
  u32 lo = 0, hi = n_halo;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (contiguous_index(halo[mid].sy) < cy) lo = mid + 1; else hi = mid;
  }
  for (u32 v = lo; v < n_halo && contiguous_index(halo[v].sy) == cy; ++v) {
    const gndt_voxel &t = halo[v];
    if ((t.flags & GNDT_F_SLOPE) && reachable(t.normal, t.rough, t.mean[2], t.flags, n, n_len, mz, P)) return true;
  }
  return false;
}

// Fix the forward/back reachability of this strip's boundary rows against the neighbours'
// halo rows: `from_prev` = last row of the strip below in x, `from_next` = first row of the
// strip above.  A row is ignored when its pointer is NULL (an end of the map) or when
// have[0] / have[1] is 0 (no neighbour sent it); have = NULL means the rows given are present.
__global__ void __launch_bounds__(256)
halo_edges_kernel(Ctl *ctl, gndt_voxel *table, gndt_slope *slopes, const gndt_voxel *from_prev, const gndt_voxel *from_next,
                  const int *have, DevParams P) {
  const u32 S = ctl->n_slopes;
  const int cx_lo = ctl->cx_min, cx_hi = ctl->cx_max;
  const HaloHeader *hp = (!have || have[0]) ? reinterpret_cast<const HaloHeader *>(from_prev) : nullptr;
  const HaloHeader *hn = (!have || have[1]) ? reinterpret_cast<const HaloHeader *>(from_next) : nullptr;
  if ((hp && hp->overflow) || (hn && hn->overflow)) { if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&ctl->err, kErrCapacity); return; }
  const bool use_prev = hp && hp->count && hp->cx == cx_lo - 1;  // adjacent x rows only
  const bool use_next = hn && hn->count && hn->cx == cx_hi + 1;
  if (!use_prev && !use_next) return;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < S; i += gridDim.x * blockDim.x) {
    const int cx = contiguous_index(slopes[i].sx);
    if (cx != cx_lo && cx != cx_hi) continue;
    const gndt_slope me = slopes[i];
    const int cy = contiguous_index(me.sy);
    const float n[3] = {me.normal[0], me.normal[1], me.normal[2]};
    const double n_len = normal_length(n);
    u32 bits = 0;
    if (use_prev && cx == cx_lo && halo_reachable(from_prev + 1, hp->count, cy, n, n_len, me.mean[2], P)) bits |= GNDT_F_REACH_B;
    if (use_next && cx == cx_hi && halo_reachable(from_next + 1, hn->count, cy, n, n_len, me.mean[2], P)) bits |= GNDT_F_REACH_F;
    if (bits) {
      slopes[i].flags = me.flags | bits;
      table[me.voxel].flags |= bits;
    }
  }
}

// The strip-local `column` / `slope` indices of a gathered voxel record made global: the strip's
// columns and Slopes before it are added; a voxel without a Slope keeps slope = 0xFFFFFFFF.
__device__ __forceinline__ void globalize_voxel_indices(u32 &column, u32 &slope, u32 cols_before, u32 slopes_before) {
  column += cols_before;
  if (slope != 0xFFFFFFFFu) slope += slopes_before;
}

// After the caller's all-gather: globalize the records [begin, begin+count) of one strip.
__global__ void strip_offsets_kernel(gndt_voxel *table, u64 begin, u64 count, u32 col_off, u32 slope_off) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (u64)gridDim.x * blockDim.x) {
    gndt_voxel *r = table + begin + i;
    globalize_voxel_indices(r->column, r->slope, col_off, slope_off);
  }
}

// ---- the library's transport through peer-mapped memory ------------------------------------

constexpr int kMaxRanks = 16;
constexpr u32 kXWaitLimitNs = 4000000000u;  // a peer that never shows up trips the watchdog after 4 s

// Written by peers (system scope), read by the owner.  Two copies of everything, selected by
// the parity of the epoch: a peer may already be one build ahead on this buffer (it publishes the
// counts of epoch e + 1 as soon as ITS build is done) while the owner's host still reads epoch e;
// it cannot be two ahead, because epoch e + 1 completes only after the owner has joined it.
struct XMail {
  u32 counts[2][kMaxRanks][4];  // {n_voxels, n_columns, n_slopes, epoch} of every strip
  u32 halo_epoch[2][2];         // [.][0] row from the lower neighbour arrived, [.][1] from the upper
  u32 done[2][kMaxRanks];       // strip r has been pushed into this rank's gathered tables
};

struct XLayout {               // byte offsets inside an exchange buffer (identical on all ranks)
  size_t mail, halo[2], voxels, slopes, columns, total;
  size_t cap_records, cap_halo;
};

struct XPeers {                // passed by value to the kernels
  unsigned char *buf[kMaxRanks];
  int rank, world;
};

__device__ __forceinline__ u32 ld_sys(const u32 *p) {
  u32 v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_sys(u32 *p, u32 v) { asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Spin until *p == want (system scope).  false after kXWaitLimitNs.
__device__ __forceinline__ bool wait_word(const u32 *p, u32 want) {
  if (ld_sys(p) == want) return true;
  const unsigned long long t0 = global_ns();
  for (;;) {
    for (int i = 0; i < 64; ++i)
      if (ld_sys(p) == want) { __threadfence_system(); return true; }
    if (global_ns() - t0 > (unsigned long long)kXWaitLimitNs) return false;
  }
}

// X1: this strip's counts into every rank's mailbox (own included).
__global__ void xchg_publish_kernel(const Ctl *ctl, XPeers X, XLayout L, u32 epoch) {
  const int r = threadIdx.x;
  if (r >= X.world) return;
  const bool bad = ctl->err != 0;
  XMail *m = reinterpret_cast<XMail *>(X.buf[r] + L.mail);
  u32 *c = m->counts[epoch & 1][X.rank];
  st_sys(c + 0, bad ? 0u : ctl->n_voxels);
  st_sys(c + 1, bad ? 0u : ctl->n_columns);
  st_sys(c + 2, bad ? 0u : ctl->n_slopes);
  __threadfence_system();
  st_sys(c + 3, epoch);
}

// All strips' counts of this epoch have arrived in the own mailbox (called by one thread).
__device__ __forceinline__ bool wait_counts(const XMail *mine, int world, u32 epoch) {
  bool ok = true;
  for (int r = 0; r < world; ++r) ok &= wait_word(&mine->counts[epoch & 1][r][3], epoch);
  __threadfence_system();
  return ok;
}
__device__ __forceinline__ int nearest_nonempty(const XMail *mine, u32 epoch, int rank, int world, int dir) {
  for (int r = rank + dir; r >= 0 && r < world; r += dir)
    if (ld_sys(&mine->counts[epoch & 1][r][0]) != 0) return r;
  return -1;
}

// X2: block 0 sends the first x row down, block 1 the last x row up.
__global__ void __launch_bounds__(256)
xchg_halo_send_kernel(Ctl *ctl, const gndt_voxel *table, XPeers X, XLayout L, u32 epoch) {
  __shared__ int s_target;
  const bool last = blockIdx.x == 1;
  const XMail *mine = reinterpret_cast<const XMail *>(X.buf[X.rank] + L.mail);
  if (threadIdx.x == 0) {
    int t = -1;
    if (!wait_counts(mine, X.world, epoch)) atomicOr(&ctl->err, kErrWatchdog);
    else if (ld_sys(&mine->counts[epoch & 1][X.rank][0]) != 0) t = nearest_nonempty(mine, epoch, X.rank, X.world, last ? +1 : -1);
    s_target = t;
  }
  __syncthreads();
  const int target = s_target;
  if (target < 0) return;
  // my first row is the target's "from the upper neighbour" row (slot 1), my last row its "from the lower" (slot 0)
  const int slot = last ? 0 : 1;
  pack_halo_row(ctl, table, last, reinterpret_cast<gndt_voxel *>(X.buf[target] + L.halo[slot]), (u32)L.cap_halo);
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    XMail *tm = reinterpret_cast<XMail *>(X.buf[target] + L.mail);
    st_sys(&tm->halo_epoch[epoch & 1][slot], epoch);
  }
}

// X3: wait for the neighbours' rows and tell halo_edges_kernel, which runs next, which of them
// arrived (one thread).
__global__ void xchg_halo_wait_kernel(Ctl *ctl, XPeers X, XLayout L, u32 epoch, int *have /* [2] */) {
  if (threadIdx.x || blockIdx.x) return;
  const XMail *mine = reinterpret_cast<const XMail *>(X.buf[X.rank] + L.mail);
  bool ok = wait_counts(mine, X.world, epoch);
  const bool self = ld_sys(&mine->counts[epoch & 1][X.rank][0]) != 0;
  const int prev = self ? nearest_nonempty(mine, epoch, X.rank, X.world, -1) : -1;
  const int next = self ? nearest_nonempty(mine, epoch, X.rank, X.world, +1) : -1;
  if (prev >= 0) ok &= wait_word(&mine->halo_epoch[epoch & 1][0], epoch);
  if (next >= 0) ok &= wait_word(&mine->halo_epoch[epoch & 1][1], epoch);
  if (!ok) atomicOr(&ctl->err, kErrWatchdog);
  have[0] = prev >= 0 ? 1 : 0;
  have[1] = next >= 0 ? 1 : 0;
}

// X4: push this strip into every rank's gathered tables.  16-byte chunks, each loaded ONCE and
// stored to all `world` destinations; the chunk of a record that holds strip-local indices is
// rewritten with the strip's global offsets on the way.
//   voxel  (6 chunks): chunk 5 = {rough, flags, column, slope}
//   slope  (3 chunks): chunk 2 = {normal.z, rough, flags, voxel}
//   column (2 chunks): chunk 0 = {sx, sy, first_index, voxel_begin}, chunk 1 = {voxel_count, slope_begin, slope_count, reserved}
// The kernel is NVLink-bound, not SM-bound: a small grid with several loads in flight per thread
// leaves the SMs to the next build running beside it.
template <int KIND>  // 0 voxels, 1 slopes, 2 columns
__device__ __forceinline__ void push_table(const uint4 *src, size_t n_chunks, size_t dst_off_bytes, size_t first_chunk, const XPeers &X,
                                           const u32 off[3], int p_lo, int p_hi) {
  constexpr int kU = 8;
  constexpr u32 kPer = KIND == 0 ? 6u : (KIND == 1 ? 3u : 2u);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < n_chunks; i0 += kU * stride) {
    uint4 v[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const size_t i = i0 + u * stride;
      if (i < n_chunks) v[u] = src[i];
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const size_t i = i0 + u * stride;
      if (i >= n_chunks) break;
      const u32 part = (u32)(i % kPer);
      if (KIND == 0) { if (part == 5) globalize_voxel_indices(v[u].z, v[u].w, off[1], off[2]); }
      else if (KIND == 1) { if (part == 2) v[u].w += off[0]; }
      else { if (part == 0) v[u].w += off[0]; else v[u].y += off[2]; }
      for (int p = p_lo; p < p_hi; ++p) reinterpret_cast<uint4 *>(X.buf[p] + dst_off_bytes)[first_chunk + i] = v[u];
    }
  }
}

constexpr int kPushThreads = 256;  // small CTAs: they must fit beside a resident partition-pass CTA (half the register file)
__global__ void __launch_bounds__(kPushThreads, 2)
xchg_push_kernel(Ctl *ctl, const gndt_voxel *table, const gndt_slope *slopes, const gndt_column *columns, XPeers X, XLayout L,
                 int what, u32 epoch, u32 *done_counter, int local_only) {
  const XMail *mine = reinterpret_cast<const XMail *>(X.buf[X.rank] + L.mail);
  u32 off[3] = {0, 0, 0}, total[3] = {0, 0, 0};
  for (int r = 0; r < X.world; ++r)
    for (int k = 0; k < 3; ++k) {
      const u32 c = ld_sys(&mine->counts[epoch & 1][r][k]);  // complete: the halo gate ran before in this stream
      if (r < X.rank) off[k] += c;
      total[k] += c;
    }
  const u32 *own = mine->counts[epoch & 1][X.rank];
  const u32 nv = ld_sys(own + 0), nc = ld_sys(own + 1), ns = ld_sys(own + 2);
  const bool fits = total[0] <= L.cap_records;
  if (!fits && blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&ctl->err, kErrCapacity);
  // local_only: this strip goes (indices made global) into the OWN gathered tables only; the copy engines
  // carry it to the peers from there (gndt_xchg_send) and a separate kernel raises the `done` flags
  const int p_lo = local_only ? X.rank : 0, p_hi = local_only ? X.rank + 1 : X.world;
  if (fits) {
    if (what & 1) push_table<0>(reinterpret_cast<const uint4 *>(table), (size_t)nv * 6, L.voxels, (size_t)off[0] * 6, X, off, p_lo, p_hi);
    if (what & 2) push_table<1>(reinterpret_cast<const uint4 *>(slopes), (size_t)ns * 3, L.slopes, (size_t)off[2] * 3, X, off, p_lo, p_hi);
    if (what & 4) push_table<2>(reinterpret_cast<const uint4 *>(columns), (size_t)nc * 2, L.columns, (size_t)off[1] * 2, X, off, p_lo, p_hi);
  }
  if (local_only) return;
  // completion: the last CTA to finish raises this strip's `done` flag in every mailbox
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const u32 ticket = atomicAdd(done_counter, 1u);
    if (ticket == gridDim.x - 1) {
      *done_counter = 0;
      __threadfence_system();
      for (int p = 0; p < X.world; ++p) st_sys(&reinterpret_cast<XMail *>(X.buf[p] + L.mail)->done[epoch & 1][X.rank], epoch);
    }
  }
}

// X4c (copy-engine transport): the copies of this strip into every peer's tables have completed (stream order);
// raise this strip's `done` flag in every mailbox.
__global__ void xchg_done_kernel(XPeers X, XLayout L, u32 epoch) {
  const int p = threadIdx.x;
  if (p >= X.world) return;
  __threadfence_system();
  st_sys(&reinterpret_cast<XMail *>(X.buf[p] + L.mail)->done[epoch & 1][X.rank], epoch);
}

// X5: every strip has arrived in this rank's gathered tables.
__global__ void xchg_wait_kernel(Ctl *ctl, XPeers X, XLayout L, u32 epoch) {
  const int r = threadIdx.x;
  if (r >= X.world) return;
  const XMail *mine = reinterpret_cast<const XMail *>(X.buf[X.rank] + L.mail);
  if (!wait_word(&mine->done[epoch & 1][r], epoch)) atomicOr(&ctl->err, kErrWatchdog);
  __threadfence_system();
}

}  // namespace gndt
