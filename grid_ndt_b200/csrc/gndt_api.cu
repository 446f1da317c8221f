// gndt_api.cu — C ABI of libgndt.so (include/gndt.h): handle, device workspace, the fixed
// launch sequence of one map build / one streaming update, result accessors and the
// host-side key helpers.
//
// front end : bounds -> plan -> up to 6 partition passes -> reduce -> fixup   (cloud -> moments)
// back end  : finalize+label -> column_finish -> edges                        (moments -> tables)
// All stream-ordered with no host round trip; counts are read back only when asked for.
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "gndt_device.cuh"
#include "gndt_lookup.h"
#include "gndt_label.cuh"
#include "gndt_reduce.cuh"
#include "gndt_sort.cuh"
#include "gndt_update.cuh"
#include "gndt_exchange.cuh"
#include "gndt_graph.cuh"
#include "gndt_ndt.cuh"
#include <unistd.h>

using namespace gndt;

namespace {

thread_local std::string g_create_error;

struct Buffer {
  void *p = nullptr;
  size_t bytes = 0;
};

enum EvId { EV_H2D0, EV_START, EV_KEY, EV_SORT, EV_REDUCE, EV_LABEL, EV_EDGES, EV_COUNT };

struct DivCheck {  // result of the exhaustive hoisted-division check for one cell length
  float len = -1.f;
  float rinv = 0.f;
  int ok = 0;
};

// Device words that outlive a build (h->small)
struct SmallWords {
  Totals tot;           // over every cloud fused into the map (totals_kernel); read back by sync_counts
  u32 fuse_err;         // Ctl::err as the pending update / remove left it (its verdict); read back with tot
  u32 n_new;            // new voxels of the pending update (update_prepare_kernel -> merge)
  struct {
    int have[2];        // which halo rows arrived (xchg_halo_wait_kernel -> halo_edges_kernel)
    u32 done_counter;   // push CTAs finished; the last one resets it
  } x;                  // strip exchange, zeroed by gndt_xchg_create
};
static_assert(sizeof(Totals) == 32 && sizeof(SmallWords) == 56, "SmallWords layout");
static_assert(offsetof(SmallWords, fuse_err) == sizeof(Totals), "fuse_err is read back together with the totals");

}  // namespace

struct gndt_handle {
  int device = 0;
  gndt_params params;
  std::string err;
  // workspace sized by points
  Buffer in_stage, buf_a, buf_b, zero;
  // workspace sized by voxels
  Buffer mom, mom_alt, table, slopes, columns, vfirst, slope_col;
  // PointCloud2 ingest: pinned staging ring for pageable messages, repacked points for odd layouts
  void *ring = nullptr;
  cudaEvent_t ring_ev[4] = {};
  bool ring_used[4] = {};
  Buffer msg_points;
  // streaming fusion scratch
  Buffer mom_scan, upd_work;
  int pending_fuse = 0;        // +1 / -1: a gndt_update / gndt_remove awaits its verdict (sync_counts)
  size_t pending_points = 0;
  Ctl saved_ctl;               // results of the resident map before the pending call
  gndt_params res_params;      // parameters the resident map was built with
  const u32 *changed_dev = nullptr, *changed_count_dev = nullptr;
  size_t n_changed = 0;
  bool n_changed_valid = false;
  Buffer small;  // one SmallWords, never memset by a build
  size_t cap_points = 0, cap_voxels = 0;
  // carved out of `zero`
  Ctl *ctl = nullptr;
  u32 *hist = nullptr;    // digit histograms [kMaxPasses][kMaxBins]
  u32 *zhist = nullptr;   // exact z histogram of the bounds pass [kZHistBins]
  u32 *row_start = nullptr, *row_end = nullptr;
  // look-back words of the partition passes: two regions used alternately (pass p uses region
  // p & 1); never memset from the host: the bounds pass zeroes region 0 for pass 0 and every
  // pass zeroes the other region for its successor (sizes depend on the digit widths)
  u32 *lb[2] = {nullptr, nullptr};
  u64 *glb[2] = {nullptr, nullptr};
  Buffer lookback;
  u64 *tile_state = nullptr;         // reduce: look-back words per tile / per group of tiles
  GroupState *tile_groups = nullptr;
  TileCarry *carry = nullptr;
  u64 *blk_state = nullptr;          // finalize: the same per block of voxels
  GroupState *blk_groups = nullptr;
  size_t zero_bytes_used = 0;
  size_t sort_tiles = 0, sort_groups = 0, red_tiles = 0, label_blocks = 0;
  Buffer f_zero;  // scratch of gndt_plan_tiles (x-column histogram)
  // traversability graph (gndt_build_edges)
  Buffer g_work, g_off, g_tgt;
  size_t g_slopes = 0, g_targets = 0;
  bool g_valid = false;
  // NDT registration (gndt_register): Gaussians of the resident map, scan upload, per-block partials
  Buffer ndt_vox, ndt_pts, ndt_part;
  double *ndt_host = nullptr;  // pinned read-back of one pass
  bool ndt_ready = false;      // ndt_vox describes the resident map (cleared by build / update / remove)
  // coarse levels of gndt_register_levels, by factor: Gaussians, coarse column table, their lengths
  struct NdtLevel { Buffer vox, cov, cols; u32 n_cols = 0, n_vox = 0; } ndt_lv[kNdtMaxFactor + 1];
  uint64_t ndt_lv_ready = 0;   // bit k: ndt_lv[k].vox describes the resident map (cleared with ndt_ready)
  // gndt_register_d2d: the same Gaussians with c = Sigma' (map level, and ndt_lv[k].cov beside the C
  // form; the coarse columns are shared), and the builder of the scan's Gaussians (first D2D call)
  Buffer ndt_cov;
  bool ndt_cov_ready = false;
  uint64_t ndt_lv_cov_ready = 0;
  gndt_handle *ndt_scan = nullptr;
  Buffer ndt_lv_work;          // scratch of a level build
  // peer-mapped strip exchange (gndt_xchg_*)
  Buffer xbuf;
  XLayout xl = {};
  XPeers xp = {};
  void *x_opened[kMaxRanks] = {};  // cudaIpcOpenMemHandle mappings to close
  int x_what = 0;
  cudaStream_t x_stream = nullptr; // high-priority stream of the push: it takes the first slots that free up
  cudaEvent_t x_ev[2] = {};
  // copy-engine transport (gndt_xchg_stage / gndt_xchg_send)
  cudaStream_t x_copy[2] = {};     // the peer copies alternate between two streams (two engines busy)
  cudaEvent_t x_ev_counts = nullptr, x_ev_copy = nullptr;
  u32 *x_counts_host = nullptr;    // pinned: every strip's {voxels, columns, slopes, epoch, failed, ...} of the staged epoch
  bool x_staged = false;
  int x_send_rc = GNDT_OK;         // verdict of the last gndt_xchg_send, reported again by gndt_xchg_view_get
  std::string x_send_err;
  bool x_peer_failed = false;      // the last gndt_xchg_view_get failed because ANOTHER strip failed
  u32 x_epoch = 0;
  bool x_created = false, x_connected = false;
  // state
  bool built = false;
  bool counts_valid = false;
  Ctl host_ctl;
  Totals host_tot, saved_tot;
  u32 host_fuse_err = 0;       // SmallWords::fuse_err, read back with host_tot
  cudaStream_t last_stream = nullptr;
  cudaEvent_t ev[EV_COUNT] = {};
  bool timed_h2d = false;
  bool stage_timing = false;  // per-stage events (they sit between kernels and defeat the programmatic overlap there)
  bool stages_valid = false;  // the last build / update recorded them
  uint64_t launches = 0;      // gndt_launch_count: launch() adds one per kernel, a build / update / remove restarts it
  uint64_t total_points = 0;  // points handed to build + updates so far (host copy)
  int sm_count = 148;
  int sort_ctas_per_sm[2] = {1, 1};  // resident CTAs of the partition pass kernels: [0] first pass, [1] later passes
  DivCheck div[2];            // [0] grid_len, [1] z_len
  uint64_t divcheck_values = 0;
};

namespace {

#define GNDT_CUDA(h, call)                                                                   \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) {                                                                 \
      (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
      return GNDT_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

int ensure(gndt_handle *h, Buffer &b, size_t bytes) {
  if (b.bytes >= bytes) return GNDT_OK;
  if (b.p) GNDT_CUDA(h, cudaFree(b.p));
  b.p = nullptr;
  b.bytes = 0;
  GNDT_CUDA(h, cudaMalloc(&b.p, bytes));
  b.bytes = bytes;
  return GNDT_OK;
}

// grow keeping the first `keep` bytes
int ensure_keep(gndt_handle *h, Buffer &b, size_t bytes, size_t keep, cudaStream_t st) {
  if (b.bytes >= bytes) return GNDT_OK;
  void *np = nullptr;
  GNDT_CUDA(h, cudaMalloc(&np, bytes));
  if (b.p && keep) GNDT_CUDA(h, cudaMemcpyAsync(np, b.p, keep, cudaMemcpyDeviceToDevice, st));
  if (b.p) { GNDT_CUDA(h, cudaStreamSynchronize(st)); GNDT_CUDA(h, cudaFree(b.p)); }
  b.p = np;
  b.bytes = bytes;
  return GNDT_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Sub-allocations of one buffer, each on a 256-byte boundary: take() returns the offset, `bytes`
// is what the buffer needs.
struct Layout {
  size_t bytes = 0;
  size_t take(size_t n) { const size_t o = bytes; bytes = align_up(bytes + n, 256); return o; }
};
template <typename T> T *at(const Buffer &b, size_t off) { return reinterpret_cast<T *>(static_cast<char *>(b.p) + off); }

// Scratch of one exclusive_scan_kernel over up to n items: ScanCtl | state | groups, zeroed together.
struct ScanScratch {
  size_t ctl, state, groups;
  ScanScratch(Layout &L, size_t n) {
    const LookbackScratch s = lookback_scratch((n + kScanTile - 1) / kScanTile);
    ctl = L.take(sizeof(ScanCtl));
    state = L.take(s.words * sizeof(u64));
    groups = L.take(s.groups * sizeof(GroupState));
  }
};

// Every kernel of this file is launched here, and counted once for gndt_launch_count.  With `pdl`
// the launch allows programmatic stream serialization: the kernel's CTAs may be scheduled while its
// predecessor in the stream drains.  Only kernels that start with pdl_wait() may be launched so;
// they touch no memory before the predecessor has completed.
template <typename... KArgs, typename... Args>
void launch(gndt_handle *h, bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
            Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // errors surface at the cudaGetLastError of the caller
  h->launches += 1;
}

// gndt_launch_count covers the map's build / update / remove and the calls on it that follow.  The
// hoisted-division check (create, set_params) and gndt_register promise to leave it unchanged
// (gndt.h): they hold one of these, which puts the count back when they return.
struct KeepLaunchCount {
  gndt_handle *h;
  uint64_t n;
  explicit KeepLaunchCount(gndt_handle *h_) : h(h_), n(h_->launches) {}
  ~KeepLaunchCount() { h->launches = n; }
};

// The cloud as the kernels read it: a host cloud is copied into `stage` on `st` (`h2d0`, when given,
// is recorded just before the copy), a device cloud is read where it is.
int upload(gndt_handle *h, Buffer &stage, const void *xyz, size_t bytes, int mem, cudaStream_t st, cudaEvent_t h2d0,
           const float **d_in) {
  *d_in = static_cast<const float *>(xyz);
  if (mem != GNDT_MEM_HOST) return GNDT_OK;
  const int rc = ensure(h, stage, bytes);
  if (rc != GNDT_OK) return rc;
  if (h2d0) GNDT_CUDA(h, cudaEventRecord(h2d0, st));
  GNDT_CUDA(h, cudaMemcpyAsync(stage.p, xyz, bytes, cudaMemcpyHostToDevice, st));
  *d_in = static_cast<const float *>(stage.p);
  return GNDT_OK;
}

// Largest non-negative float a with (int)ceil(a / len) <= GNDT_MAX_INDEX, by bisection over
// the bit patterns (the test is monotone in a).  Same IEEE binary32 operations as the device
// index arithmetic, so "|p - p0| <= max_abs" is exactly "the point's index is in range".
float max_abs_offset(float len) {
  auto ok = [len](uint32_t b) {
    float a;
    memcpy(&a, &b, 4);
    volatile float q = a / len;
    return std::ceil((float)q) <= (float)GNDT_MAX_INDEX;
  };
  uint32_t lo = 0, hi = 0x7f7fffffu;  // 0.0f is always valid; FLT_MAX usually is not
  if (ok(hi)) lo = hi;
  while (lo + 1 < hi) {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (ok(mid)) lo = mid; else hi = mid;
  }
  float a;
  memcpy(&a, &lo, 4);
  return a;
}

DevParams to_dev(const gndt_params &p, size_t cap_voxels) {
  DevParams d;
  d.max_abs[0] = max_abs_offset(p.grid_len);
  d.max_abs[1] = max_abs_offset(p.z_len);
  d.idx_offset = 0;
  d.fast_div = 0;
  d.rinv[0] = d.rinv[1] = 0.f;
  d.grid_len = p.grid_len; d.z_len = p.z_len; d.slope_interval = p.slope_interval;
  d.demand = p.demand; d.min_points = p.min_points;
  d.rough_max = p.rough_max; d.angle_max_deg = p.angle_max_deg; d.reach_height = p.reach_height;
  d.origin_first = p.origin_is_first_point;
  d.origin[0] = p.origin[0]; d.origin[1] = p.origin[1]; d.origin[2] = p.origin[2];
  d.normalize_cov = p.normalize_cov;
  d.tile_lo = p.tile_lo; d.tile_hi = p.tile_hi;
  d.max_voxels = (u32)cap_voxels;
  return d;
}

// Exhaustive proof-by-enumeration that the hoisted division (gndt_device.cuh) rounds exactly
// like the IEEE division for this cell length: every float a in [len, 2*max_abs] is tried.
// (a < len never divides; beyond 2*max_abs both quotients exceed GNDT_MAX_INDEX by far.)
__global__ void divcheck_kernel(float len, u32 lo_bits, u32 hi_bits, float *rinv_out, unsigned long long *mismatches) {
  const float r = refined_rcp(len);
  if (blockIdx.x == 0 && threadIdx.x == 0) *rinv_out = r;
  unsigned long long bad = 0;
  for (u64 b = (u64)lo_bits + (u64)blockIdx.x * blockDim.x + threadIdx.x; b <= hi_bits; b += (u64)gridDim.x * blockDim.x) {
    const float a = __uint_as_float((u32)b);
    const float exact = ceilf(__fdiv_rn(a, len));
    const float fast = hoisted_div_ceil(a, len, r);
    if (!(exact == fast)) bad++;
  }
  if (bad) atomicAdd(mismatches, bad);
}

int verify_fast_div(gndt_handle *h, float len, DivCheck &out) {
  if (out.len == len) return GNDT_OK;  // cached for this length
  out.len = len;
  out.ok = 0;
  out.rinv = 0.f;
  const char *force = getenv("GNDT_EXACT_DIV");
  if (force && force[0] == '1') return GNDT_OK;
  void *scratch = nullptr;
  GNDT_CUDA(h, cudaMalloc(&scratch, 64));
  GNDT_CUDA(h, cudaMemset(scratch, 0, 64));
  uint32_t lo, hi;
  const float top = 2.f * max_abs_offset(len);
  memcpy(&lo, &len, 4);
  memcpy(&hi, &top, 4);
  KeepLaunchCount keep(h);
  launch(h, false, divcheck_kernel, h->sm_count * 8, 256, 0, nullptr, len, lo, hi, (float *)scratch,
         (unsigned long long *)((char *)scratch + 8));
  unsigned long long host[2] = {0, 0};
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(host, scratch, 16, cudaMemcpyDeviceToHost);
  cudaFree(scratch);
  if (e != cudaSuccess) { h->err = std::string("divcheck: ") + cudaGetErrorString(e); return GNDT_ERR_CUDA; }
  memcpy(&out.rinv, &host[0], 4);
  out.ok = (host[1] == 0) ? 1 : 0;
  h->divcheck_values += (uint64_t)hi - lo + 1;
  return GNDT_OK;
}

DevParams make_dev(gndt_handle *h, const gndt_params &p, size_t cap_voxels) {
  DevParams d = to_dev(p, cap_voxels);
  d.fast_div = (h->div[0].ok && h->div[1].ok && h->div[0].len == p.grid_len && h->div[1].len == p.z_len) ? 1 : 0;
  d.rinv[0] = h->div[0].rinv;
  d.rinv[1] = h->div[1].rinv;
  return d;
}

int validate_params(const gndt_params *p) {
  if (!p) return GNDT_ERR_INVALID_ARG;
  if (!(p->grid_len > 0.f) || !(p->z_len > 0.f) || !std::isfinite(p->grid_len) || !std::isfinite(p->z_len))
    return GNDT_ERR_INVALID_ARG;
  if (p->demand != GNDT_DEMAND_SLOPE && p->demand != GNDT_DEMAND_TRUE) return GNDT_ERR_INVALID_ARG;
  if (p->min_points < 1) return GNDT_ERR_INVALID_ARG;
  return GNDT_OK;
}

// Workspace for n points and cap_vox voxels; carves the zero-initialised region.
// `keep_mom` bytes of the resident moments survive a regrow (streaming update).
int reserve(gndt_handle *h, size_t n, size_t cap_vox, size_t keep_mom, cudaStream_t st) {
  int rc;
  if ((rc = ensure(h, h->buf_a, n * sizeof(float4))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->buf_b, n * sizeof(float4))) != GNDT_OK) return rc;
  if ((rc = ensure_keep(h, h->mom, cap_vox * sizeof(VoxMoments), keep_mom, st)) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->table, cap_vox * sizeof(gndt_voxel))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->slopes, cap_vox * sizeof(gndt_slope))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->columns, cap_vox * sizeof(gndt_column))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->vfirst, cap_vox * sizeof(u32))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->slope_col, cap_vox * sizeof(u32))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->small, sizeof(SmallWords))) != GNDT_OK) return rc;
  h->cap_points = n;
  h->cap_voxels = cap_vox;
  h->sort_tiles = (n + kSortTile - 1) / kSortTile;
  h->sort_groups = (h->sort_tiles + kSortGroup - 1) / kSortGroup;
  h->red_tiles = (n + kRedTile - 1) / kRedTile;
  h->label_blocks = (cap_vox + kLabelThreads - 1) / kLabelThreads;
  const LookbackScratch red = lookback_scratch(h->red_tiles), fin = lookback_scratch(h->label_blocks);
  Layout Z;
  const size_t o_ctl = Z.take(sizeof(Ctl));
  const size_t o_hist = Z.take((size_t)kMaxPasses * kMaxBins * sizeof(u32));
  const size_t o_zh = Z.take(kZHistBins * sizeof(u32));
  const size_t o_rs = Z.take(65536 * sizeof(u32));
  const size_t o_re = Z.take(65536 * sizeof(u32));
  const size_t o_ts = Z.take(red.words * sizeof(u64));
  const size_t o_tg = Z.take(red.groups * sizeof(GroupState));
  const size_t o_ca = Z.take(h->red_tiles * sizeof(TileCarry));
  const size_t o_bs = Z.take(fin.words * sizeof(u64));
  const size_t o_bg = Z.take(fin.groups * sizeof(GroupState));
  if ((rc = ensure(h, h->zero, Z.bytes)) != GNDT_OK) return rc;
  h->ctl = at<Ctl>(h->zero, o_ctl);
  h->hist = at<u32>(h->zero, o_hist);
  h->zhist = at<u32>(h->zero, o_zh);
  h->row_start = at<u32>(h->zero, o_rs);
  h->row_end = at<u32>(h->zero, o_re);
  h->tile_state = at<u64>(h->zero, o_ts);
  h->tile_groups = at<GroupState>(h->zero, o_tg);
  h->carry = at<TileCarry>(h->zero, o_ca);
  h->blk_state = at<u64>(h->zero, o_bs);
  h->blk_groups = at<GroupState>(h->zero, o_bg);
  h->zero_bytes_used = Z.bytes;
  // look-back words of the partition passes (not part of the memset region)
  Layout B;
  const size_t lb_bytes = h->sort_tiles * kMaxBins * sizeof(u32) + 256, glb_bytes = h->sort_groups * kMaxBins * sizeof(u64) + 256;
  const size_t o_lb[2] = {B.take(lb_bytes), B.take(lb_bytes)}, o_glb[2] = {B.take(glb_bytes), B.take(glb_bytes)};
  if ((rc = ensure(h, h->lookback, B.bytes)) != GNDT_OK) return rc;
  for (int k = 0; k < 2; ++k) {
    h->lb[k] = at<u32>(h->lookback, o_lb[k]);
    h->glb[k] = at<u64>(h->lookback, o_glb[k]);
  }
  return GNDT_OK;
}

int grid_for(const gndt_handle *h, size_t work_items, int per_block, int max_waves) {
  size_t blocks = (work_items + per_block - 1) / per_block;
  size_t cap = (size_t)h->sm_count * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

int sync_counts(gndt_handle *h) {
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  if (h->counts_valid) return GNDT_OK;
  // stream-ordered behind the build and nothing else: no legacy-stream copy, so builds of other
  // handles on other streams (a pipelined caller) keep running while this one is read back
  GNDT_CUDA(h, cudaMemcpyAsync(&h->host_ctl, h->ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->last_stream));
  GNDT_CUDA(h, cudaMemcpyAsync(&h->host_tot, h->small.p, sizeof(Totals), cudaMemcpyDeviceToHost, h->last_stream));
  if (h->pending_fuse)
    GNDT_CUDA(h, cudaMemcpyAsync(&h->host_fuse_err, &static_cast<SmallWords *>(h->small.p)->fuse_err, sizeof(u32), cudaMemcpyDeviceToHost,
                                 h->last_stream));
  GNDT_CUDA(h, cudaStreamSynchronize(h->last_stream));
  if (h->pending_fuse) {  // verdict of the last gndt_update / gndt_remove, from ITS error bits: a halo or an
    const int sign = h->pending_fuse;  // exchange enqueued behind it may have raised more since
    h->pending_fuse = 0;
    if (h->host_fuse_err) {
      // failed on the device: the resident moments were never touched and the tables were not rewritten
      // (the back end returns at once when the error word is set); put the counters back
      const u32 e = h->host_fuse_err;
      h->host_ctl = h->saved_ctl;
      h->host_tot = h->saved_tot;
      GNDT_CUDA(h, cudaMemcpyAsync(h->ctl, &h->saved_ctl, sizeof(Ctl), cudaMemcpyHostToDevice, h->last_stream));
      GNDT_CUDA(h, cudaMemcpyAsync(h->small.p, &h->saved_tot, sizeof(Totals), cudaMemcpyHostToDevice, h->last_stream));
      GNDT_CUDA(h, cudaStreamSynchronize(h->last_stream));
      h->counts_valid = true;  // the map before the call stays valid
      if (e & kErrWatchdog) { h->err = "device watchdog tripped (look-back / TMA wait never resolved)"; return GNDT_ERR_INTERNAL; }
      if (e & kErrUnmatched) { h->err = "gndt_remove: the scan holds points that were never fused into the map; map unchanged"; return GNDT_ERR_STATE; }
      h->err = "voxel table capacity (max_voxels) exceeded; map unchanged";
      return GNDT_ERR_CAPACITY;
    }
    std::swap(h->mom, h->mom_alt);
    // the cloud-index counter follows n_input: a remove gives its points' indices back
    if (sign > 0) h->total_points += h->pending_points;
    else h->total_points -= h->pending_points;
    u32 nc = 0;
    GNDT_CUDA(h, cudaMemcpy(&nc, h->changed_count_dev, 4, cudaMemcpyDeviceToHost));
    h->n_changed = nc;
    h->n_changed_valid = true;
  }
  // bits raised by the build (or after the update's verdict, by the halo and the exchange) stay until the next build
  const u32 e = h->host_ctl.err;
  if (e & kErrWatchdog) { h->err = "device watchdog tripped (look-back / TMA / exchange wait never resolved)"; return GNDT_ERR_INTERNAL; }
  if (e & kErrCapacity) { h->err = "voxel table capacity (max_voxels) exceeded"; return GNDT_ERR_CAPACITY; }
  if (e & kErrHaloCapacity) { h->err = "a neighbour strip's halo row exceeds cap_halo_records"; return GNDT_ERR_CAPACITY; }
  if (e & kErrGatherCapacity) { h->err = "gathered map exceeds the exchange capacity (cap_records)"; return GNDT_ERR_CAPACITY; }
  h->counts_valid = true;
  return GNDT_OK;
}

// cloud -> sorted raw moments in `out` (h->ctl->n_voxels entries)
int front_end(gndt_handle *h, cudaStream_t st, const float *d_in, size_t n, size_t stride_f, size_t start,
              const DevParams &dp, VoxMoments *out) {
  GNDT_CUDA(h, cudaMemsetAsync(h->zero.p, 0, h->zero_bytes_used, st));
  // K1: bounds + exact z histogram (+ zeroes the first pass's look-back words), then the key layout
  const size_t tiles = (n + kSortTile - 1) / kSortTile, groups = (tiles + kSortGroup - 1) / kSortGroup;
  auto *bounds = dp.fast_div ? bounds_kernel<true> : bounds_kernel<false>;
  launch(h, true, bounds, grid_for(h, n, 256 * 4, 8), 256, 0, st, h->ctl, h->zhist, d_in, stride_f, n, start, (void *)h->lb[0],
         tiles * kFirstMaxBins * sizeof(u32), (void *)h->glb[0], groups * kFirstMaxBins * sizeof(u64), dp);
  launch(h, true, plan_kernel, 1, kZHistBins, 0, st, h->ctl, (const u32 *)h->zhist, h->hist);
  if (h->stage_timing) GNDT_CUDA(h, cudaEventRecord(h->ev[EV_KEY], st));
  // K2: partition passes (pass p writes buffer A when p is even, B when odd).  Persistent CTAs:
  // a pass beyond the planned count costs one launch of CTAs that return at once.
  float4 *A = static_cast<float4 *>(h->buf_a.p), *B = static_cast<float4 *>(h->buf_b.p);
  // the division mode is a template argument (two instantiations), not a run-time select
  auto *first_pass = dp.fast_div ? sort_pass_kernel<true, true> : sort_pass_kernel<true, false>;
  auto *next_pass = dp.fast_div ? sort_pass_kernel<false, true> : sort_pass_kernel<false, false>;
  const int g0 = (int)std::min<size_t>(tiles, (size_t)h->sm_count * h->sort_ctas_per_sm[0]);
  const int g1 = (int)std::min<size_t>(tiles, (size_t)h->sm_count * h->sort_ctas_per_sm[1]);
  launch(h, true, first_pass, g0, kSortThreads, sizeof(SortSmem), st, h->ctl, 0, d_in, stride_f, n, start, (const float4 *)nullptr, A,
         h->lb[0], h->glb[0], h->lb[1], h->glb[1], h->hist, dp);
  for (int p = 1; p < kMaxPasses; ++p) {
    const float4 *src = (p & 1) ? A : B;
    float4 *dst = (p & 1) ? B : A;
    launch(h, true, next_pass, g1, kSortThreads, sizeof(SortSmem), st, h->ctl, p, (const float *)nullptr, (size_t)4, n, (size_t)0, src, dst,
           h->lb[p & 1], h->glb[p & 1], h->lb[(p + 1) & 1], h->glb[(p + 1) & 1], h->hist, dp);
  }
  if (h->stage_timing) GNDT_CUDA(h, cudaEventRecord(h->ev[EV_SORT], st));
  // K3: per-voxel moments
  const int rtiles = (int)((n + kRedTile - 1) / kRedTile);
  auto *reduce = dp.fast_div ? reduce_kernel<true> : reduce_kernel<false>;
  launch(h, true, reduce, rtiles, kRedThreads, sizeof(RedSmem), st, h->ctl, (const float4 *)A, (const float4 *)B, out, h->carry,
         h->tile_state, h->tile_groups, dp);
  launch(h, true, fixup_kernel, grid_for(h, (size_t)rtiles * 32, 128, 16), 128, 0, st, h->ctl, out, (const TileCarry *)h->carry);
  if (h->stage_timing) GNDT_CUDA(h, cudaEventRecord(h->ev[EV_REDUCE], st));
  return GNDT_OK;
}

__global__ void table_bounds_kernel(Ctl *ctl, const gndt_voxel *table) {
  pdl_wait();
  pdl_trigger();
  const u32 n = ctl->n_voxels;
  if (threadIdx.x == 0 && n && !ctl->err) {
    ctl->cx_min = contiguous_index(table[0].sx);
    ctl->cx_max = contiguous_index(table[n - 1].sx);
  }
}

// sorted raw moments -> voxel / slope / column tables + reachability bits
int back_end(gndt_handle *h, cudaStream_t st, const DevParams &dp, const VoxMoments *mom, bool bounds_from_table) {
  const int g_lab = grid_for(h, h->cap_voxels, kLabelThreads, 8);
  launch(h, true, finalize_label_kernel, g_lab, kFinThreads, sizeof(FinSmem), st, h->ctl, mom, (gndt_voxel *)h->table.p,
         (gndt_slope *)h->slopes.p, (gndt_column *)h->columns.p, (u32 *)h->vfirst.p, (u32 *)h->slope_col.p, h->blk_state, h->blk_groups,
         &h->ctl->ticket[7], dp);
  if (bounds_from_table) launch(h, true, table_bounds_kernel, 1, 32, 0, st, h->ctl, (const gndt_voxel *)h->table.p);
  launch(h, true, column_finish_kernel, g_lab, 256, 0, st, h->ctl, (const u32 *)h->vfirst.p, (gndt_column *)h->columns.p,
         h->row_start, h->row_end);
  if (h->stage_timing) GNDT_CUDA(h, cudaEventRecord(h->ev[EV_LABEL], st));
  launch(h, true, edges_kernel, g_lab, 256, 0, st, h->ctl, (gndt_voxel *)h->table.p, (gndt_slope *)h->slopes.p,
         (const gndt_column *)h->columns.p, (const u32 *)h->slope_col.p, (const u32 *)h->row_start, (const u32 *)h->row_end, dp);
  GNDT_CUDA(h, cudaEventRecord(h->ev[EV_EDGES], st));
  return GNDT_OK;
}

int check_cloud_args(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, const char *who) {
  if (!xyz || n == 0 || stride_bytes < 12 || (stride_bytes & 3) || (mem != GNDT_MEM_HOST && mem != GNDT_MEM_DEVICE)) {
    h->err = std::string(who) + ": bad argument (xyz NULL, n == 0, stride not a multiple of 4 >= 12, or bad mem)";
    return GNDT_ERR_INVALID_ARG;
  }
  if (n > GNDT_MAX_POINTS) { h->err = std::string(who) + ": n exceeds GNDT_MAX_POINTS"; return GNDT_ERR_CAPACITY; }
  return GNDT_OK;
}

}  // namespace

extern "C" {

const char *gndt_version(void) { return "gndt 0.3 (abi 2, sm_100a)"; }

const char *gndt_last_error(const gndt_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

void gndt_default_params(gndt_params *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->grid_len = 0.5f; p->z_len = 0.1f; p->slope_interval = 0.08f;
  p->demand = GNDT_DEMAND_SLOPE; p->min_points = 3;
  p->rough_max = 100.f; p->angle_max_deg = 30.f; p->reach_height = 0.15f;
  p->origin_is_first_point = 1;
}

int gndt_create(const gndt_params *params, int device, gndt_handle **out) {
  if (!out) return GNDT_ERR_INVALID_ARG;
  *out = nullptr;
  if (validate_params(params) != GNDT_OK) { g_create_error = "invalid gndt_params"; return GNDT_ERR_INVALID_ARG; }
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || device < 0 || device >= n_dev) {
    g_create_error = std::string("no usable CUDA device (there is no CPU fallback): ") +
                     (e != cudaSuccess ? cudaGetErrorString(e) : "device index out of range");
    return GNDT_ERR_CUDA;
  }
  gndt_handle *h = new gndt_handle();
  h->device = device;
  h->params = *params;
  if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete h; return GNDT_ERR_CUDA; }
  cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
  for (int i = 0; i < EV_COUNT; ++i)
    if ((e = cudaEventCreate(&h->ev[i])) != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete h; return GNDT_ERR_CUDA; }
  e = cudaFuncSetAttribute(sort_pass_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sort_pass_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sort_pass_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sort_pass_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(reduce_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RedSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(reduce_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RedSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(finalize_label_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FinSmem));
  if (e != cudaSuccess) { g_create_error = std::string("kernel image for sm_100a not loadable on this device: ") + cudaGetErrorString(e); delete h; return GNDT_ERR_CUDA; }
  // persistent partition passes: as many CTAs as stay resident
  for (int k = 0; k < 2; ++k) {
    int nb = 0;
    e = k == 0 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, sort_pass_kernel<true, true>, kSortThreads, sizeof(SortSmem))
               : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, sort_pass_kernel<false, true>, kSortThreads, sizeof(SortSmem));
    if (e != cudaSuccess || nb < 1) { g_create_error = "partition pass kernel does not fit on this device"; delete h; return GNDT_ERR_CUDA; }
    h->sort_ctas_per_sm[k] = nb;
  }
  int rc = verify_fast_div(h, h->params.grid_len, h->div[0]);
  if (rc == GNDT_OK) rc = verify_fast_div(h, h->params.z_len, h->div[1]);
  if (rc != GNDT_OK) { g_create_error = h->err; delete h; return rc; }
  *out = h;
  return GNDT_OK;
}

int gndt_destroy(gndt_handle *h) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  for (int r = 0; r < kMaxRanks; ++r)
    if (h->x_opened[r]) cudaIpcCloseMemHandle(h->x_opened[r]);
  if (h->x_stream) { cudaStreamDestroy(h->x_stream); for (int i = 0; i < 2; ++i) if (h->x_ev[i]) cudaEventDestroy(h->x_ev[i]); }
  for (int i = 0; i < 2; ++i) if (h->x_copy[i]) cudaStreamDestroy(h->x_copy[i]);
  if (h->x_ev_counts) cudaEventDestroy(h->x_ev_counts);
  if (h->x_ev_copy) cudaEventDestroy(h->x_ev_copy);
  if (h->x_counts_host) cudaFreeHost(h->x_counts_host);
  if (h->ndt_host) cudaFreeHost(h->ndt_host);
  if (h->ring) { cudaFreeHost(h->ring); for (int i = 0; i < 4; ++i) if (h->ring_ev[i]) cudaEventDestroy(h->ring_ev[i]); }
  Buffer *bufs[] = {&h->in_stage, &h->buf_a, &h->buf_b, &h->zero, &h->mom, &h->mom_alt, &h->table, &h->slopes,
                    &h->columns, &h->vfirst, &h->slope_col, &h->mom_scan, &h->upd_work, &h->msg_points, &h->small, &h->lookback, &h->f_zero, &h->xbuf, &h->g_work, &h->g_off, &h->g_tgt,
                    &h->ndt_vox, &h->ndt_pts, &h->ndt_part, &h->ndt_lv_work, &h->ndt_cov};
  for (Buffer *b : bufs) if (b->p) cudaFree(b->p);
  for (auto &l : h->ndt_lv) for (Buffer *b : {&l.vox, &l.cov, &l.cols}) if (b->p) cudaFree(b->p);
  if (h->ndt_scan) gndt_destroy(h->ndt_scan);
  for (int i = 0; i < EV_COUNT; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  delete h;
  return GNDT_OK;
}

int gndt_set_params(gndt_handle *h, const gndt_params *params) {
  if (!h || validate_params(params) != GNDT_OK) return GNDT_ERR_INVALID_ARG;
  h->params = *params;
  GNDT_CUDA(h, cudaSetDevice(h->device));
  int rc = verify_fast_div(h, h->params.grid_len, h->div[0]);  // no-op when the length is unchanged
  if (rc == GNDT_OK) rc = verify_fast_div(h, h->params.z_len, h->div[1]);
  return rc;
}

// the build proper, cloud already on the device (reserve() done by the caller)
static int build_device(gndt_handle *h, const float *d_in, size_t n, size_t stride_bytes, cudaStream_t st) {
  const size_t start = h->params.origin_is_first_point ? 1 : 0;
  const DevParams dp = make_dev(h, h->params, h->cap_voxels);
  h->ndt_ready = false;
  h->ndt_lv_ready = 0;
  h->ndt_cov_ready = false;
  h->ndt_lv_cov_ready = 0;
  h->g_valid = false;  // the graph indexes the slope table this build replaces
  GNDT_CUDA(h, cudaEventRecord(h->ev[EV_START], st));
  int rc = front_end(h, st, d_in, n, stride_bytes / 4, start, dp, (VoxMoments *)h->mom.p);
  if (rc != GNDT_OK) return rc;
  launch(h, true, totals_kernel, 1, 32, 0, st, &static_cast<SmallWords *>(h->small.p)->tot, (const Ctl *)h->ctl, (u64)n, 1, 1);
  rc = back_end(h, st, dp, (const VoxMoments *)h->mom.p, false);
  if (rc != GNDT_OK) return rc;
  GNDT_CUDA(h, cudaGetLastError());
  h->built = true;
  h->pending_fuse = 0;
  h->n_changed_valid = false;
  h->res_params = h->params;
  h->stages_valid = h->stage_timing;
  h->total_points = n;
  h->last_stream = st;
  return GNDT_OK;
}

// what a build does before its cloud is on the device: no map until it completes, the launch count
// restarts, the workspace fits n points
static int begin_build(gndt_handle *h, size_t n, cudaStream_t st) {
  GNDT_CUDA(h, cudaSetDevice(h->device));
  h->built = false;
  h->counts_valid = false;
  h->launches = 0;
  const size_t cap_vox = h->params.max_voxels ? (size_t)h->params.max_voxels : n;
  return reserve(h, n, cap_vox, 0, st);
}

int gndt_build(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = check_cloud_args(h, xyz, n, stride_bytes, mem, "gndt_build");
  if (rc != GNDT_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = begin_build(h, n, st)) != GNDT_OK) return rc;
  const float *d_in;
  h->timed_h2d = mem == GNDT_MEM_HOST;
  if ((rc = upload(h, h->in_stage, xyz, n * stride_bytes, mem, st, h->ev[EV_H2D0], &d_in)) != GNDT_OK) return rc;
  return build_device(h, d_in, n, stride_bytes, st);
}

// ---- sensor_msgs/PointCloud2 ingest ------------------------------------------------------
// Any field layout -> packed 16-byte (x, y, z, 0) points: byte-wise reads, optional byte swap.
__global__ void ingest_kernel(const unsigned char *raw, size_t n, u32 point_step, u32 xo, u32 yo, u32 zo, int big_endian, float4 *out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned char *p = raw + i * point_step;
    u32 w[3];
    const u32 offs[3] = {xo, yo, zo};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const unsigned char *q = p + offs[k];
      w[k] = big_endian ? ((u32)q[0] << 24 | (u32)q[1] << 16 | (u32)q[2] << 8 | (u32)q[3])
                        : ((u32)q[3] << 24 | (u32)q[2] << 16 | (u32)q[1] << 8 | (u32)q[0]);
    }
    out[i] = make_float4(__uint_as_float(w[0]), __uint_as_float(w[1]), __uint_as_float(w[2]), 0.f);
  }
}

// Pageable host memory -> device through a ring of pinned chunks: the host copy of chunk i + 1
// (split over a few threads) runs while the DMA engine moves chunk i.  A plain cudaMemcpyAsync
// from pageable memory is staged by the driver one small buffer at a time and blocks the caller.
static int upload_pageable(gndt_handle *h, void *dst, const void *src, size_t bytes, cudaStream_t st) {
  constexpr size_t kChunk = 8u << 20;
  constexpr int kSlots = 4, kThreads = 4;
  if (!h->ring) {
    GNDT_CUDA(h, cudaHostAlloc(&h->ring, kChunk * kSlots, cudaHostAllocDefault));
    for (int i = 0; i < kSlots; ++i) GNDT_CUDA(h, cudaEventCreateWithFlags(&h->ring_ev[i], cudaEventDisableTiming));
  }
  size_t off = 0;
  for (int slot = 0; off < bytes; slot = (slot + 1) % kSlots) {
    const size_t len = std::min(kChunk, bytes - off);
    char *stage = static_cast<char *>(h->ring) + (size_t)slot * kChunk;
    if (h->ring_used[slot]) GNDT_CUDA(h, cudaEventSynchronize(h->ring_ev[slot]));  // its previous DMA is done
    const char *from = static_cast<const char *>(src) + off;
    std::thread workers[kThreads - 1];
    const size_t part = (len + kThreads - 1) / kThreads;
    for (int t = 1; t < kThreads; ++t)
      workers[t - 1] = std::thread([=] { if (t * part < len) memcpy(stage + t * part, from + t * part, std::min(part, len - t * part)); });
    memcpy(stage, from, std::min(part, len));
    for (auto &w : workers) w.join();
    GNDT_CUDA(h, cudaMemcpyAsync(static_cast<char *>(dst) + off, stage, len, cudaMemcpyHostToDevice, st));
    GNDT_CUDA(h, cudaEventRecord(h->ring_ev[slot], st));
    h->ring_used[slot] = true;
    off += len;
  }
  return GNDT_OK;
}

int gndt_build_msg(gndt_handle *h, const gndt_pointcloud2 *msg, void *stream) {
  if (!h || !msg) return GNDT_ERR_INVALID_ARG;
  const size_t n = (size_t)msg->width * msg->height;
  const u32 ps = msg->point_step;
  if (!msg->data || n == 0 || ps < 12 || msg->x_offset + 4 > ps || msg->y_offset + 4 > ps || msg->z_offset + 4 > ps) {
    h->err = "gndt_build_msg: empty message or x/y/z fields outside point_step";
    return GNDT_ERR_INVALID_ARG;
  }
  if (n > GNDT_MAX_POINTS) { h->err = "gndt_build_msg: width * height exceeds GNDT_MAX_POINTS"; return GNDT_ERR_CAPACITY; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = begin_build(h, n, st);
  if (rc == GNDT_OK) rc = ensure(h, h->in_stage, n * ps);
  if (rc != GNDT_OK) return rc;
  GNDT_CUDA(h, cudaEventRecord(h->ev[EV_H2D0], st));
  if (msg->host_pinned) GNDT_CUDA(h, cudaMemcpyAsync(h->in_stage.p, msg->data, n * ps, cudaMemcpyHostToDevice, st));
  else if ((rc = upload_pageable(h, h->in_stage.p, msg->data, n * ps, st)) != GNDT_OK) return rc;
  h->timed_h2d = true;
  // little-endian float32 x, y, z side by side on a 4-byte boundary: the kernels read the message as it is
  const bool direct = !msg->is_bigendian && (ps % 4 == 0) && (msg->x_offset % 4 == 0) && msg->y_offset == msg->x_offset + 4 &&
                      msg->z_offset == msg->x_offset + 8;
  if (direct) return build_device(h, reinterpret_cast<const float *>(static_cast<const char *>(h->in_stage.p) + msg->x_offset), n, ps, st);
  if ((rc = ensure(h, h->msg_points, n * sizeof(float4))) != GNDT_OK) return rc;
  launch(h, false, ingest_kernel, grid_for(h, n, 256, 8), 256, 0, st, static_cast<const unsigned char *>(h->in_stage.p), n, ps,
         msg->x_offset, msg->y_offset, msg->z_offset, msg->is_bigendian ? 1 : 0, static_cast<float4 *>(h->msg_points.p));
  return build_device(h, static_cast<const float *>(h->msg_points.p), n, sizeof(float4), st);
}

// gndt_update (sign = +1) and gndt_remove (sign = -1): reduce the scan to its own sorted moments
// table, merge it with the resident one into the alternate buffer, relabel, list the touched cells.
static int fuse_scan(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, void *stream, int sign) {
  const char *who = sign > 0 ? "gndt_update" : "gndt_remove";
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = check_cloud_args(h, xyz, n, stride_bytes, mem, who);
  if (rc != GNDT_OK) return rc;
  // like the reference (map2D.h:679-680: change2DMap returns false on an empty map) an
  // update needs a resident map; its origin and parameters are kept
  if ((rc = sync_counts(h)) != GNDT_OK) return rc;
  if (h->params.grid_len != h->res_params.grid_len || h->params.z_len != h->res_params.z_len ||
      h->params.tile_lo != h->res_params.tile_lo || h->params.tile_hi != h->res_params.tile_hi) {
    h->err = std::string(who) + ": grid_len / z_len / strip range differ from the resident map's (two key spaces cannot be fused)";
    return GNDT_ERR_STATE;
  }
  if (sign > 0 && h->total_points + n > 0xFFFFFFFFull) { h->err = "gndt_update: more than 2^32 points fused"; return GNDT_ERR_CAPACITY; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const u32 n_res = h->host_ctl.n_voxels;
  const float origin[3] = {h->host_ctl.origin[0], h->host_ctl.origin[1], h->host_ctl.origin[2]};
  h->saved_ctl = h->host_ctl;  // what sync_counts restores if this call fails on the device
  h->saved_tot = h->host_tot;
  h->counts_valid = false;
  h->launches = 0;
  h->n_changed_valid = false;
  h->ndt_ready = false;  // recomputed by the next gndt_register whatever the verdict
  h->ndt_lv_ready = 0;
  h->ndt_cov_ready = false;
  h->ndt_lv_cov_ready = 0;
  h->g_valid = false;    // rebuilt by the next gndt_build_edges whatever the verdict

  // capacity: every scan point could open a new voxel
  size_t cap_vox = h->cap_voxels;
  const size_t need = (size_t)n_res + (sign > 0 ? n : 0);
  if (h->params.max_voxels == 0 && need > cap_vox) cap_vox = need + need / 2;
  rc = reserve(h, n > h->cap_points ? n : h->cap_points, cap_vox, (size_t)n_res * sizeof(VoxMoments), st);
  if (rc != GNDT_OK) return rc;
  if ((rc = ensure(h, h->mom_alt, cap_vox * sizeof(VoxMoments))) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->mom_scan, n * sizeof(VoxMoments))) != GNDT_OK) return rc;
  // scratch: per scan voxel / point (n + 1 words each): is_new, new_pos, order, valid, order_pos, changed; keys (u64)
  //          per resident / merged voxel (cap_vox + 1 words each): inv, dead, dead_pos, touch_first
  //          one per exclusive scan launched (3), each sized for the larger of the two
  Layout W;
  const size_t wn = (n + 1) * 4, wv = (cap_vox + 1) * 4;
  const size_t o_is_new = W.take(wn), o_new_pos = W.take(wn), o_order = W.take(wn), o_valid = W.take(wn), o_order_pos = W.take(wn),
               o_changed = W.take(wn), o_new_keys = W.take(n * 8);
  const size_t o_inv = W.take(wv), o_dead = W.take(wv), o_dead_pos = W.take(wv), o_touch_first = W.take(wv);
  const size_t scan_items = std::max(n, cap_vox);
  const ScanScratch sc[3] = {ScanScratch(W, scan_items), ScanScratch(W, scan_items), ScanScratch(W, scan_items)};
  if ((rc = ensure(h, h->upd_work, W.bytes)) != GNDT_OK) return rc;
  const Buffer &w = h->upd_work;
  u32 *is_new = at<u32>(w, o_is_new), *new_pos = at<u32>(w, o_new_pos), *order = at<u32>(w, o_order), *valid = at<u32>(w, o_valid),
      *order_pos = at<u32>(w, o_order_pos), *changed = at<u32>(w, o_changed);
  u64 *new_keys = at<u64>(w, o_new_keys);
  u32 *inv = at<u32>(w, o_inv), *dead = at<u32>(w, o_dead), *dead_pos = at<u32>(w, o_dead_pos), *touch_first = at<u32>(w, o_touch_first);
  auto exclusive_scan = [&](int k, const u32 *in, u32 n_fixed, const u32 *n_dev, u32 *out, size_t items) {
    launch(h, false, exclusive_scan_kernel, grid_for(h, (items + kScanTile - 1) / kScanTile, 1, 4), 256, 0, st, at<ScanCtl>(w, sc[k].ctl),
           in, n_fixed, n_dev, out, at<u64>(w, sc[k].state), at<GroupState>(w, sc[k].groups));
  };

  const float *d_in;
  h->timed_h2d = mem == GNDT_MEM_HOST;
  if ((rc = upload(h, h->in_stage, xyz, n * stride_bytes, mem, st, h->ev[EV_H2D0], &d_in)) != GNDT_OK) return rc;
  gndt_params p = h->params;  // every point of the scan is binned against the resident origin
  p.origin_is_first_point = 0;
  p.origin[0] = origin[0]; p.origin[1] = origin[1]; p.origin[2] = origin[2];
  DevParams dp = make_dev(h, p, cap_vox);
  dp.idx_offset = sign > 0 ? (u32)h->total_points : 0u;

  GNDT_CUDA(h, cudaEventRecord(h->ev[EV_START], st));
  VoxMoments *res = (VoxMoments *)h->mom.p, *scan = (VoxMoments *)h->mom_scan.p, *merged = (VoxMoments *)h->mom_alt.p;
  rc = front_end(h, st, d_in, n, stride_bytes / 4, 0, dp, scan);
  if (rc != GNDT_OK) return rc;
  SmallWords *small = static_cast<SmallWords *>(h->small.p);
  launch(h, false, totals_kernel, 1, 32, 0, st, &small->tot, h->ctl, (u64)n, 0, sign);
  const int g_scan = grid_for(h, n, 256, 8), g_res = grid_for(h, std::max<size_t>(n_res, 1), 256, 8);
  // zero: is_new .. valid (4 arrays), dead / dead_pos, scan scratch; 0xFF: inv, touch_first
  GNDT_CUDA(h, cudaMemsetAsync(is_new, 0, o_order_pos - o_is_new, st));
  GNDT_CUDA(h, cudaMemsetAsync(dead, 0, o_touch_first - o_dead, st));
  GNDT_CUDA(h, cudaMemsetAsync(at<char>(w, sc[0].ctl), 0, W.bytes - sc[0].ctl, st));
  GNDT_CUDA(h, cudaMemsetAsync(inv, 0xFF, wv, st));
  GNDT_CUDA(h, cudaMemsetAsync(touch_first, 0xFF, wv, st));
  launch(h, false, update_match_kernel, g_scan, 256, 0, st, h->ctl, res, n_res, scan, sign, inv, is_new, dead);
  exclusive_scan(0, is_new, 0u, &h->ctl->n_voxels, new_pos, n);
  if (sign < 0) exclusive_scan(1, dead, n_res, nullptr, dead_pos, n_res);
  launch(h, false, update_new_keys_kernel, g_scan, 256, 0, st, h->ctl, scan, is_new, new_pos, new_keys);
  launch(h, false, update_prepare_kernel, 1, 32, 0, st, h->ctl, n_res, new_pos, sign < 0 ? dead_pos : nullptr, (u32)cap_vox, &small->n_new);
  launch(h, false, update_merge_resident_kernel, g_res, 256, 0, st, h->ctl, res, n_res, scan, sign, inv, new_keys, &small->n_new, dead,
         dead_pos, merged);
  if (sign > 0) launch(h, false, update_merge_new_kernel, g_scan, 256, 0, st, h->ctl, res, n_res, scan, is_new, new_pos, merged);
  rc = back_end(h, st, dp, merged, true);
  if (rc != GNDT_OK) return rc;
  // the cells this scan touched, in first-touched order (changeMorton_list)
  launch(h, false, changed_mark_kernel, g_scan, 256, 0, st, h->ctl, scan, (const gndt_column *)h->columns.p, touch_first);
  launch(h, false, changed_order_kernel, grid_for(h, cap_vox, 256, 8), 256, 0, st, h->ctl, touch_first, dp.idx_offset, (u32)n, order, valid);
  exclusive_scan(2, valid, (u32)n, nullptr, order_pos, n);
  launch(h, false, changed_compact_kernel, g_scan, 256, 0, st, order, valid, order_pos, (u32)n, changed);
  // the verdict: Ctl::err as this call leaves it, before anything enqueued behind it adds bits
  GNDT_CUDA(h, cudaMemcpyAsync(&small->fuse_err, &h->ctl->err, sizeof(u32), cudaMemcpyDeviceToDevice, st));
  GNDT_CUDA(h, cudaGetLastError());
  h->changed_dev = changed;
  h->changed_count_dev = &at<ScanCtl>(w, sc[2].ctl)->total;
  h->pending_fuse = sign;         // resolved by the next sync_counts: swap the moment tables, or roll back
  h->pending_points = n;
  h->stages_valid = h->stage_timing;
  h->last_stream = st;
  return GNDT_OK;
}

int gndt_update(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, void *stream) {
  return fuse_scan(h, xyz, n, stride_bytes, mem, stream, +1);
}

int gndt_remove(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, void *stream) {
  return fuse_scan(h, xyz, n, stride_bytes, mem, stream, -1);
}

int gndt_changed_columns(gndt_handle *h, uint32_t *idx, size_t cap, int dst_mem, size_t *n_out) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  if (!h->n_changed_valid) { h->err = "gndt_changed_columns: the last call on this handle was not a gndt_update / gndt_remove"; return GNDT_ERR_STATE; }
  if (n_out) *n_out = h->n_changed;
  if (!idx) return GNDT_OK;  // size query
  if (h->n_changed > cap) { h->err = "destination capacity too small"; return GNDT_ERR_CAPACITY; }
  if (h->n_changed)
    GNDT_CUDA(h, cudaMemcpy(idx, h->changed_dev, h->n_changed * 4, dst_mem == GNDT_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice));
  return GNDT_OK;
}

int gndt_counts(gndt_handle *h, gndt_counts_t *out) {
  if (!h || !out) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  const Ctl &c = h->host_ctl;
  out->n_input = h->host_tot.n_points;
  out->n_binned = h->host_tot.n_valid;
  out->n_dropped = h->host_tot.n_dropped;
  out->n_outside_tile = h->host_tot.n_outside;
  out->n_columns = c.n_columns;
  out->n_voxels = c.n_voxels;
  out->n_fitted = c.n_fitted;
  out->n_slopes = c.n_slopes;
  return GNDT_OK;
}

static int copy_out(gndt_handle *h, void *dst, size_t cap, int dst_mem, size_t *n_out, const void *src, size_t n,
                    size_t rec) {
  if (!dst && n) return GNDT_ERR_INVALID_ARG;
  if (n > cap) { h->err = "destination capacity too small"; return GNDT_ERR_CAPACITY; }
  if (n) {
    GNDT_CUDA(h, cudaMemcpyAsync(dst, src, n * rec, dst_mem == GNDT_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                 h->last_stream));
    GNDT_CUDA(h, cudaStreamSynchronize(h->last_stream));
  }
  if (n_out) *n_out = n;
  return GNDT_OK;
}

int gndt_copy_voxels(gndt_handle *h, gndt_voxel *dst, size_t cap, int dst_mem, size_t *n_out) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  return copy_out(h, dst, cap, dst_mem, n_out, h->table.p, h->host_ctl.n_voxels, sizeof(gndt_voxel));
}
int gndt_copy_slopes(gndt_handle *h, gndt_slope *dst, size_t cap, int dst_mem, size_t *n_out) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  return copy_out(h, dst, cap, dst_mem, n_out, h->slopes.p, h->host_ctl.n_slopes, sizeof(gndt_slope));
}
int gndt_copy_columns(gndt_handle *h, gndt_column *dst, size_t cap, int dst_mem, size_t *n_out) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  return copy_out(h, dst, cap, dst_mem, n_out, h->columns.p, h->host_ctl.n_columns, sizeof(gndt_column));
}

int gndt_device_voxels(gndt_handle *h, const gndt_voxel **dptr, size_t *n) {
  if (!h || !dptr || !n) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  *dptr = static_cast<const gndt_voxel *>(h->table.p);
  *n = h->host_ctl.n_voxels;
  return GNDT_OK;
}

int gndt_halo_pack(gndt_handle *h, gndt_voxel *first_row_out, gndt_voxel *last_row_out, size_t cap_records, void *stream) {
  if (!h || !first_row_out || !last_row_out || cap_records < 1) return GNDT_ERR_INVALID_ARG;
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  launch(h, false, halo_pack_kernel, 2, 256, 0, st, h->ctl, (const gndt_voxel *)h->table.p, first_row_out, last_row_out,
         (u32)cap_records);
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

int gndt_halo_edges(gndt_handle *h, const gndt_voxel *from_prev, const gndt_voxel *from_next, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const DevParams dp = make_dev(h, h->params, h->cap_voxels);
  launch(h, false, halo_edges_kernel, grid_for(h, h->cap_voxels, 256, 8), 256, 0, st, h->ctl, (gndt_voxel *)h->table.p,
         (gndt_slope *)h->slopes.p, from_prev, from_next, nullptr, dp);
  h->counts_valid = false;
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

int gndt_apply_strip_offsets(gndt_handle *h, gndt_voxel *table, const uint64_t *offsets, const uint32_t *col_offsets,
                             const uint32_t *slope_offsets, int n_strips, void *stream) {
  if (!h || !table || !offsets || !col_offsets || !slope_offsets || n_strips < 1) return GNDT_ERR_INVALID_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  for (int r = 0; r < n_strips; ++r) {
    const uint64_t cnt = offsets[r + 1] - offsets[r];
    if (!cnt || (col_offsets[r] == 0 && slope_offsets[r] == 0)) continue;
    launch(h, false, strip_offsets_kernel, grid_for(h, cnt, 256, 8), 256, 0, st, table, offsets[r], cnt, col_offsets[r], slope_offsets[r]);
  }
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

int gndt_device_count_ptr(gndt_handle *h, const uint32_t **d_n_voxels) {
  if (!h || !d_n_voxels) return GNDT_ERR_INVALID_ARG;
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  *d_n_voxels = &h->ctl->n_voxels;
  return GNDT_OK;
}

int gndt_device_table_ptr(gndt_handle *h, const gndt_voxel **dptr, size_t *capacity) {
  if (!h || !dptr) return GNDT_ERR_INVALID_ARG;
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  *dptr = static_cast<const gndt_voxel *>(h->table.p);
  if (capacity) *capacity = h->cap_voxels;
  return GNDT_OK;
}

// ---- traversability graph (CSR of AccessibleNeighbors) -----------------------------------
int gndt_build_edges(gndt_handle *h, const gndt_slope *slopes, size_t n_slopes, const gndt_column *columns, size_t n_columns,
                     void *stream) {
  if (!h || ((slopes == nullptr) != (columns == nullptr))) return GNDT_ERR_INVALID_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  h->g_valid = false;
  int cx_lo = 0, cx_hi = 0, rc;
  if (!slopes) {  // this handle's own tables
    if ((rc = sync_counts(h)) != GNDT_OK) return rc;
    slopes = static_cast<const gndt_slope *>(h->slopes.p);
    columns = static_cast<const gndt_column *>(h->columns.p);
    n_slopes = h->host_ctl.n_slopes;
    n_columns = h->host_ctl.n_columns;
    if (!st) st = h->last_stream;
  }
  if (n_slopes > 0xFFFFFFFEull || n_columns > 0xFFFFFFFEull) return GNDT_ERR_CAPACITY;
  if (n_slopes && !n_columns) { h->err = "gndt_build_edges: Slopes without a column table"; return GNDT_ERR_INVALID_ARG; }
  if (n_columns) {  // x range of the (sorted) column table
    gndt_column ends[2];
    GNDT_CUDA(h, cudaMemcpyAsync(&ends[0], columns, sizeof(gndt_column), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaMemcpyAsync(&ends[1], columns + n_columns - 1, sizeof(gndt_column), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaStreamSynchronize(st));
    if (!valid_signed_index(ends[0].sx) || !valid_signed_index(ends[1].sx) || contiguous_index(ends[0].sx) > contiguous_index(ends[1].sx)) {
      h->err = "gndt_build_edges: the first and last columns are not an x range of valid indices";
      return GNDT_ERR_INVALID_ARG;
    }
    cx_lo = contiguous_index(ends[0].sx);
    cx_hi = contiguous_index(ends[1].sx);
  }
  const int n_rows = cx_hi - cx_lo + 1;
  const u32 S = (u32)n_slopes, C = (u32)n_columns;
  // work buffer: scan scratch | table check word | rows start/end (zeroed) | slope_col | deg
  Layout W;
  const ScanScratch sc(W, n_slopes);
  const size_t o_bad = W.take(4);
  const size_t o_rs = W.take((size_t)n_rows * 4), o_re = W.take((size_t)n_rows * 4);
  const size_t zero_bytes = W.bytes;
  const size_t o_sc = W.take((n_slopes + 1) * 4), o_dg = W.take((n_slopes + 1) * 4);
  if ((rc = ensure(h, h->g_work, W.bytes)) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->g_off, (n_slopes + 1) * 4)) != GNDT_OK) return rc;
  const Buffer &w = h->g_work;
  ScanCtl *g = at<ScanCtl>(w, sc.ctl);
  u32 *rs = at<u32>(w, o_rs), *re = at<u32>(w, o_re), *slope_col = at<u32>(w, o_sc), *deg = at<u32>(w, o_dg), *bad = at<u32>(w, o_bad);
  GNDT_CUDA(h, cudaMemsetAsync(w.p, 0, zero_bytes, st));
  GNDT_CUDA(h, cudaMemsetAsync(h->g_off.p, 0, (n_slopes + 1) * 4, st));
  h->g_slopes = n_slopes;
  h->g_targets = 0;
  if (S && C) {
    const DevParams dp = make_dev(h, h->params, 0);
    const int grid_c = grid_for(h, C, 256, 8), grid_s = grid_for(h, S, 256, 8);
    launch(h, false, graph_prepare_kernel, grid_c, 256, 0, st, slopes, S, columns, C, cx_lo, cx_hi, slope_col, rs, re, bad);
    launch(h, false, graph_edges_kernel<false>, grid_s, 256, 0, st, slopes, S, columns, C, slope_col, rs, re, cx_lo, n_rows, deg, nullptr,
           nullptr, (const u32 *)bad, dp);
    launch(h, false, exclusive_scan_kernel, grid_for(h, (n_slopes + kScanTile - 1) / kScanTile, 1, 4), 256, 0, st, g, deg, S, nullptr,
           (u32 *)h->g_off.p, at<u64>(w, sc.state), at<GroupState>(w, sc.groups));
    ScanCtl hg;
    u32 hbad = 0;
    GNDT_CUDA(h, cudaMemcpyAsync(&hg, g, sizeof(hg), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaMemcpyAsync(&hbad, bad, sizeof(hbad), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaStreamSynchronize(st));
    if (hbad) {
      h->err = (hbad & kGraphBadIndex)   ? "gndt_build_edges: a column index is 0, beyond +-GNDT_MAX_INDEX or outside the table's x range"
               : (hbad & kGraphBadOrder) ? "gndt_build_edges: the columns are not sorted strictly by (x, y)"
               : (hbad & kGraphBadRange) ? "gndt_build_edges: the columns' slope ranges do not tile [0, n_slopes) in order"
                                         : "gndt_build_edges: a Slope's (sx, sy) differs from its column's";
      return GNDT_ERR_INVALID_ARG;
    }
    if (hg.err) { h->err = "graph scan watchdog"; return GNDT_ERR_INTERNAL; }
    h->g_targets = hg.total;
    if ((rc = ensure(h, h->g_tgt, std::max<size_t>(hg.total, 1) * 4)) != GNDT_OK) return rc;
    launch(h, false, graph_edges_kernel<true>, grid_s, 256, 0, st, slopes, S, columns, C, slope_col, rs, re, cx_lo, n_rows, nullptr,
           (const u32 *)h->g_off.p, (u32 *)h->g_tgt.p, (const u32 *)bad, dp);
    GNDT_CUDA(h, cudaStreamSynchronize(st));
  }
  GNDT_CUDA(h, cudaGetLastError());
  h->g_valid = true;
  return GNDT_OK;
}

int gndt_copy_edges(gndt_handle *h, uint32_t *offsets, size_t cap_offsets, uint32_t *targets, size_t cap_targets, int dst_mem,
                    size_t *n_slopes, size_t *n_targets) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!h->g_valid) { h->err = "gndt_copy_edges: call gndt_build_edges first"; return GNDT_ERR_STATE; }
  if (n_slopes) *n_slopes = h->g_slopes;
  if (n_targets) *n_targets = h->g_targets;
  if (!offsets && !targets) return GNDT_OK;  // size query
  if (cap_offsets < h->g_slopes + 1 || cap_targets < h->g_targets || !offsets || (!targets && h->g_targets)) {
    h->err = "destination capacity too small";
    return GNDT_ERR_CAPACITY;
  }
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const cudaMemcpyKind kind = dst_mem == GNDT_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  GNDT_CUDA(h, cudaMemcpy(offsets, h->g_off.p, (h->g_slopes + 1) * 4, kind));
  if (h->g_targets) GNDT_CUDA(h, cudaMemcpy(targets, h->g_tgt.p, h->g_targets * 4, kind));
  return GNDT_OK;
}

// ---- peer-mapped strip exchange --------------------------------------------------------
static_assert(sizeof(gndt_xchg_info) == 128, "gndt_xchg_info is 128 bytes");
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
constexpr int kPushCtas = 48;  // grid of xchg_push_kernel

int gndt_xchg_create(gndt_handle *h, int rank, int world, size_t cap_records, size_t cap_halo_records, int what,
                     gndt_xchg_info *mine) {
  if (!h || !mine || world < 1 || world > kMaxRanks || rank < 0 || rank >= world || cap_records < 1 || cap_halo_records < 1 ||
      !(what & (GNDT_X_VOXELS | GNDT_X_SLOPES | GNDT_X_COLUMNS)))
    return GNDT_ERR_INVALID_ARG;
  if (cap_records > 0xFFFFFFFEull) return GNDT_ERR_CAPACITY;
  GNDT_CUDA(h, cudaSetDevice(h->device));
  // Load every kernel of the exchange now.  Under lazy module loading (the CUDA 12 default) the first
  // launch of a kernel loads it, and loading may wait for the kernels running on the device.  A rank's
  // halo send spins until every rank has published, so a host thread that drives several ranks and
  // enqueued rank 0's halo send would block loading rank 0's next kernel until the 4 s watchdog fired.
  const void *xk[] = {(const void *)xchg_publish_kernel, (const void *)xchg_halo_send_kernel, (const void *)xchg_halo_wait_kernel,
                      (const void *)halo_edges_kernel,   (const void *)xchg_push_kernel,      (const void *)xchg_done_kernel,
                      (const void *)xchg_wait_kernel};
  for (const void *k : xk) {
    cudaFuncAttributes fa;
    GNDT_CUDA(h, cudaFuncGetAttributes(&fa, k));
  }
  XLayout L = {};
  Layout B;
  L.mail = B.take(sizeof(XMail));
  L.halo[0] = B.take((cap_halo_records + 1) * sizeof(gndt_voxel));
  L.halo[1] = B.take((cap_halo_records + 1) * sizeof(gndt_voxel));
  L.voxels = B.take((what & GNDT_X_VOXELS) ? cap_records * sizeof(gndt_voxel) : 0);
  L.slopes = B.take((what & GNDT_X_SLOPES) ? cap_records * sizeof(gndt_slope) : 0);
  L.columns = B.take((what & GNDT_X_COLUMNS) ? cap_records * sizeof(gndt_column) : 0);
  L.total = B.bytes;
  L.cap_records = cap_records;
  L.cap_halo = cap_halo_records;
  int rc;
  if ((rc = ensure(h, h->xbuf, L.total)) != GNDT_OK) return rc;
  if ((rc = ensure(h, h->small, sizeof(SmallWords))) != GNDT_OK) return rc;
  GNDT_CUDA(h, cudaMemset(h->xbuf.p, 0, sizeof(XMail)));
  GNDT_CUDA(h, cudaMemset(&static_cast<SmallWords *>(h->small.p)->x, 0, sizeof(SmallWords::x)));
  h->xl = L;
  h->xp = XPeers{};
  h->xp.rank = rank;
  h->xp.world = world;
  h->x_what = what;
  h->x_epoch = 0;
  h->x_created = true;
  h->x_connected = false;
  if (!h->x_stream) {
    int lo_p = 0, hi_p = 0;
    GNDT_CUDA(h, cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
    GNDT_CUDA(h, cudaStreamCreateWithPriority(&h->x_stream, cudaStreamNonBlocking, hi_p));
    for (int i = 0; i < 2; ++i) GNDT_CUDA(h, cudaEventCreateWithFlags(&h->x_ev[i], cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) GNDT_CUDA(h, cudaStreamCreateWithFlags(&h->x_copy[i], cudaStreamNonBlocking));
    GNDT_CUDA(h, cudaEventCreateWithFlags(&h->x_ev_counts, cudaEventDisableTiming));
    GNDT_CUDA(h, cudaEventCreateWithFlags(&h->x_ev_copy, cudaEventDisableTiming));
    GNDT_CUDA(h, cudaHostAlloc(reinterpret_cast<void **>(&h->x_counts_host), kMaxRanks * kXCountWords * sizeof(u32), cudaHostAllocDefault));
  }
  h->x_staged = false;
  memset(mine, 0, sizeof(*mine));
  cudaIpcMemHandle_t ipc;
  GNDT_CUDA(h, cudaIpcGetMemHandle(&ipc, h->xbuf.p));
  memcpy(mine->ipc_mem, &ipc, 64);
  mine->ptr = (uint64_t)(uintptr_t)h->xbuf.p;
  mine->bytes = L.total;
  mine->cap_records = cap_records;
  mine->cap_halo = cap_halo_records;
  mine->device = h->device;
  mine->pid = (int32_t)getpid();
  mine->what = what;
  mine->rank = rank;
  return GNDT_OK;
}

int gndt_xchg_connect(gndt_handle *h, const gndt_xchg_info *all, int world) {
  if (!h || !all) return GNDT_ERR_INVALID_ARG;
  if (!h->x_created || world != h->xp.world) { h->err = "gndt_xchg_connect: create the exchange first / world mismatch"; return GNDT_ERR_STATE; }
  GNDT_CUDA(h, cudaSetDevice(h->device));
  for (int r = 0; r < world; ++r) {
    const gndt_xchg_info &in = all[r];
    if (in.rank != r || in.bytes != h->xl.total || in.cap_records != h->xl.cap_records || in.cap_halo != h->xl.cap_halo || in.what != h->x_what) {
      h->err = "gndt_xchg_connect: rank " + std::to_string(r) + " has a different exchange layout";
      return GNDT_ERR_INVALID_ARG;
    }
    if (r == h->xp.rank) { h->xp.buf[r] = static_cast<unsigned char *>(h->xbuf.p); continue; }
    if (in.pid == (int32_t)getpid()) {  // same process: plain peer access
      if (in.device != h->device) {
        int can = 0;
        GNDT_CUDA(h, cudaDeviceCanAccessPeer(&can, h->device, in.device));
        if (!can) { h->err = "no peer access between devices " + std::to_string(h->device) + " and " + std::to_string(in.device); return GNDT_ERR_CUDA; }
        cudaError_t e = cudaDeviceEnablePeerAccess(in.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { h->err = cudaGetErrorString(e); return GNDT_ERR_CUDA; }
        cudaGetLastError();
      }
      h->xp.buf[r] = reinterpret_cast<unsigned char *>((uintptr_t)in.ptr);
    } else {  // another process: map its buffer
      cudaIpcMemHandle_t ipc;
      memcpy(&ipc, in.ipc_mem, 64);
      void *p = nullptr;
      GNDT_CUDA(h, cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
      h->x_opened[r] = p;
      h->xp.buf[r] = static_cast<unsigned char *>(p);
    }
  }
  h->x_connected = true;
  return GNDT_OK;
}

// publish -> halo rows -> boundary reach bits (everything of an exchange that needs no bulk transfer)
static void xchg_front(gndt_handle *h, cudaStream_t st, u32 epoch) {
  const XPeers &X = h->xp;
  const XLayout &L = h->xl;
  int *have = static_cast<SmallWords *>(h->small.p)->x.have;
  const DevParams dp = make_dev(h, h->params, h->cap_voxels);
  unsigned char *mine = X.buf[X.rank];
  launch(h, false, xchg_publish_kernel, 1, 32, 0, st, h->ctl, X, L, epoch);
  launch(h, false, xchg_halo_send_kernel, 2, 256, 0, st, h->ctl, (const gndt_voxel *)h->table.p, X, L, epoch);
  launch(h, false, xchg_halo_wait_kernel, 1, 32, 0, st, h->ctl, X, L, epoch, have);
  launch(h, false, halo_edges_kernel, grid_for(h, h->cap_voxels, 256, 4), 256, 0, st, h->ctl, (gndt_voxel *)h->table.p,
         (gndt_slope *)h->slopes.p, reinterpret_cast<const gndt_voxel *>(mine + L.halo[0]),
         reinterpret_cast<const gndt_voxel *>(mine + L.halo[1]), have, dp);
}

static int xchg_check(gndt_handle *h, const char *who) {
  if (!h->built) { h->err = "no map has been built on this handle"; return GNDT_ERR_STATE; }
  if (!h->x_connected) { h->err = std::string(who) + ": exchange not connected"; return GNDT_ERR_STATE; }
  return GNDT_OK;
}

int gndt_xchg_run(gndt_handle *h, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = xchg_check(h, "gndt_xchg_run");
  if (rc != GNDT_OK) return rc;
  if (h->x_staged) { h->err = "gndt_xchg_run: a staged exchange is waiting for gndt_xchg_send"; return GNDT_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const u32 epoch = ++h->x_epoch;
  const XPeers &X = h->xp;
  const XLayout &L = h->xl;
  u32 *done_counter = &static_cast<SmallWords *>(h->small.p)->x.done_counter;
  h->x_send_rc = GNDT_OK;
  xchg_front(h, st, epoch);
  // the bulk transfer and the final wait run on the high-priority stream, fenced by events on both sides
  GNDT_CUDA(h, cudaEventRecord(h->x_ev[0], st));
  GNDT_CUDA(h, cudaStreamWaitEvent(h->x_stream, h->x_ev[0], 0));
  launch(h, false, xchg_push_kernel, kPushCtas, kPushThreads, 0, h->x_stream, h->ctl, (const gndt_voxel *)h->table.p,
         (const gndt_slope *)h->slopes.p, (const gndt_column *)h->columns.p, X, L, h->x_what, epoch, done_counter, 0);
  launch(h, false, xchg_wait_kernel, 1, 32, 0, h->x_stream, h->ctl, X, L, epoch);
  GNDT_CUDA(h, cudaEventRecord(h->x_ev[1], h->x_stream));
  GNDT_CUDA(h, cudaStreamWaitEvent(st, h->x_ev[1], 0));
  h->counts_valid = false;
  h->last_stream = st;
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

// ---- copy-engine transport: the same exchange with the bulk of the bytes moved by cudaMemcpyAsync ----
// SM-issued stores to peers slow the build that runs beside them on the SENDING GPU (measured:
// profiles/xchg_overlap_r2.md); copy-engine transfers do not.  The engines need sizes and addresses
// on the host, so the exchange is split: gndt_xchg_stage enqueues everything up to the strip sitting,
// indices made global, in this rank's own gathered tables, plus a 512-byte read-back of every strip's
// counts; gndt_xchg_send waits for that read-back (the one host round trip; the next builds are
// already queued behind it) and enqueues the peer copies, the `done` flags and the final wait.
int gndt_xchg_stage(gndt_handle *h, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  int rc = xchg_check(h, "gndt_xchg_stage");
  if (rc != GNDT_OK) return rc;
  if (h->x_staged) { h->err = "gndt_xchg_stage: the previous staged exchange has not been sent"; return GNDT_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const u32 epoch = ++h->x_epoch;
  const XPeers &X = h->xp;
  const XLayout &L = h->xl;
  u32 *done_counter = &static_cast<SmallWords *>(h->small.p)->x.done_counter;
  h->x_send_rc = GNDT_OK;
  xchg_front(h, st, epoch);  // its halo gate has seen every strip's counts of this epoch
  launch(h, false, xchg_push_kernel, kPushCtas, kPushThreads, 0, st, h->ctl, (const gndt_voxel *)h->table.p, (const gndt_slope *)h->slopes.p,
         (const gndt_column *)h->columns.p, X, L, h->x_what, epoch, done_counter, 1);
  const XMail *mail = reinterpret_cast<const XMail *>(X.buf[X.rank] + L.mail);
  GNDT_CUDA(h, cudaMemcpyAsync(h->x_counts_host, mail->counts[epoch & 1], kMaxRanks * kXCountWords * sizeof(u32), cudaMemcpyDeviceToHost, st));
  GNDT_CUDA(h, cudaEventRecord(h->x_ev_counts, st));
  h->x_staged = true;
  h->counts_valid = false;
  h->last_stream = st;
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

int gndt_xchg_counts_ready(gndt_handle *h) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!h->x_staged) return 0;
  const cudaError_t e = cudaEventQuery(h->x_ev_counts);
  if (e == cudaSuccess) return 1;
  if (e == cudaErrorNotReady) return 0;
  h->err = cudaGetErrorString(e);
  return GNDT_ERR_CUDA;
}

int gndt_xchg_send(gndt_handle *h, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!h->x_staged) { h->err = "gndt_xchg_send: nothing staged"; return GNDT_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  GNDT_CUDA(h, cudaEventSynchronize(h->x_ev_counts));
  h->x_staged = false;
  const u32 epoch = h->x_epoch;
  const XPeers &X = h->xp;
  const XLayout &L = h->xl;
  const int W = X.world;
  uint64_t off[3] = {0, 0, 0}, total = 0;  // voxels, columns, slopes before this strip
  for (int r = 0; r < W; ++r) {
    const u32 *c = h->x_counts_host + kXCountWords * r;
    if (c[3] != epoch) {
      h->x_send_err = "gndt_xchg_send: strip " + std::to_string(r) + " never published its counts (watchdog)";
      h->x_send_rc = GNDT_ERR_INTERNAL;
    }
    if (r < X.rank) for (int k = 0; k < 3; ++k) off[k] += c[k];
    total += c[0];
  }
  if (h->x_send_rc == GNDT_OK && total > L.cap_records) {
    h->x_send_err = "gathered map exceeds the exchange capacity: " + std::to_string(total) + " > " + std::to_string(L.cap_records) + " records";
    h->x_send_rc = GNDT_ERR_CAPACITY;
  }
  if (h->x_send_rc != GNDT_OK) {  // nothing was sent: gndt_xchg_view_get reports the same verdict
    h->err = h->x_send_err;
    return h->x_send_rc;
  }
  const u32 *own = h->x_counts_host + kXCountWords * X.rank;
  struct { int bit; size_t base, rec; uint64_t first, n; } tab[3] = {
      {GNDT_X_VOXELS, L.voxels, sizeof(gndt_voxel), off[0], own[0]},
      {GNDT_X_SLOPES, L.slopes, sizeof(gndt_slope), off[2], own[2]},
      {GNDT_X_COLUMNS, L.columns, sizeof(gndt_column), off[1], own[1]}};
  for (int j = 0; j < 2; ++j) GNDT_CUDA(h, cudaStreamWaitEvent(h->x_copy[j], h->x_ev_counts, 0));
  int n_copies = 0;
  for (int d = 1; d < W; ++d) {  // start with the next rank: at any moment every GPU receives from one sender
    const int p = (X.rank + d) % W;
    for (const auto &t : tab) {
      if (!(h->x_what & t.bit) || t.n == 0) continue;
      const size_t at = t.base + (size_t)t.first * t.rec;
      GNDT_CUDA(h, cudaMemcpyAsync(X.buf[p] + at, X.buf[X.rank] + at, (size_t)t.n * t.rec, cudaMemcpyDefault, h->x_copy[n_copies++ & 1]));
    }
  }
  // flags and the final wait: high-priority stream (one warp each; they take the first free slot)
  for (int j = 0; j < 2; ++j) {
    GNDT_CUDA(h, cudaEventRecord(j ? h->x_ev_copy : h->x_ev[0], h->x_copy[j]));
    GNDT_CUDA(h, cudaStreamWaitEvent(h->x_stream, j ? h->x_ev_copy : h->x_ev[0], 0));
  }
  launch(h, false, xchg_done_kernel, 1, 32, 0, h->x_stream, X, L, epoch);
  launch(h, false, xchg_wait_kernel, 1, 32, 0, h->x_stream, h->ctl, X, L, epoch);
  GNDT_CUDA(h, cudaEventRecord(h->x_ev[1], h->x_stream));
  GNDT_CUDA(h, cudaStreamWaitEvent(st, h->x_ev[1], 0));
  h->counts_valid = false;
  h->last_stream = st;
  GNDT_CUDA(h, cudaGetLastError());
  return GNDT_OK;
}

int gndt_xchg_view_get(gndt_handle *h, gndt_xchg_view *out) {
  if (!h || !out) return GNDT_ERR_INVALID_ARG;
  if (!h->x_connected || h->x_epoch == 0) { h->err = "gndt_xchg_view_get: no exchange has run"; return GNDT_ERR_STATE; }
  h->x_peer_failed = false;
  int rc = sync_counts(h);  // synchronises the stream, surfaces watchdog / capacity errors
  if (rc != GNDT_OK) return rc;
  if (h->x_send_rc != GNDT_OK) { h->err = h->x_send_err; return h->x_send_rc; }
  XMail mail;
  GNDT_CUDA(h, cudaMemcpy(&mail, h->xp.buf[h->xp.rank] + h->xl.mail, sizeof(XMail), cudaMemcpyDeviceToHost));
  memset(out, 0, sizeof(*out));
  unsigned char *mine = h->xp.buf[h->xp.rank];
  out->voxels = (h->x_what & GNDT_X_VOXELS) ? reinterpret_cast<const gndt_voxel *>(mine + h->xl.voxels) : nullptr;
  out->slopes = (h->x_what & GNDT_X_SLOPES) ? reinterpret_cast<const gndt_slope *>(mine + h->xl.slopes) : nullptr;
  out->columns = (h->x_what & GNDT_X_COLUMNS) ? reinterpret_cast<const gndt_column *>(mine + h->xl.columns) : nullptr;
  out->world = h->xp.world;
  const int par = h->x_epoch & 1;
  for (int r = 0; r < h->xp.world; ++r) {
    const u32 *c = mail.counts[par][r];
    if (c[3] != h->x_epoch || mail.done[par][r] != h->x_epoch) { h->err = "exchange incomplete (epoch mismatch)"; return GNDT_ERR_INTERNAL; }
    if (c[4]) {  // its records are missing from the gathered tables
      h->err = "strip " + std::to_string(r) + " failed its build / update and sent no records; the gathered map is incomplete";
      h->x_peer_failed = true;
      return GNDT_ERR_STATE;
    }
    out->strip_voxels[r] = c[0];
    out->strip_columns[r] = c[1];
    out->strip_slopes[r] = c[2];
    out->n_voxels += c[0];
    out->n_columns += c[1];
    out->n_slopes += c[2];
  }
  return GNDT_OK;
}

// ---- one process, several GPUs (what the reference's single receiver process would call) ----
struct gndt_multi {
  std::vector<gndt_handle *> h;
  std::vector<int> dev;
  std::vector<cudaStream_t> st;
  std::vector<Buffer> cloud;   // every GPU's copy of the current cloud / scan
  std::vector<int32_t> cuts;
  gndt_params params;
  bool planned = false;
  std::string err;
};

static int multi_fail(gndt_multi *m, int i, int rc, const char *what) {
  m->err = std::string(what) + " (device index " + std::to_string(i) + "): " + (i >= 0 && i < (int)m->h.size() && m->h[i] ? m->h[i]->err : g_create_error);
  return rc;
}

int gndt_multi_create(const gndt_params *params, const int *devices, int ndev, size_t cap_records, size_t cap_halo_records, int what,
                      gndt_multi **out) {
  if (!out || !params || !devices || ndev < 1 || ndev > kMaxRanks) return GNDT_ERR_INVALID_ARG;
  *out = nullptr;
  gndt_multi *m = new gndt_multi();
  m->params = *params;
  m->h.assign(ndev, nullptr);
  m->dev.assign(devices, devices + ndev);
  m->st.assign(ndev, nullptr);
  m->cloud.resize(ndev);
  std::vector<gndt_xchg_info> info(ndev);
  for (int i = 0; i < ndev; ++i) {
    int rc = gndt_create(params, devices[i], &m->h[i]);
    if (rc == GNDT_OK && cudaStreamCreateWithFlags(&m->st[i], cudaStreamNonBlocking) != cudaSuccess) rc = GNDT_ERR_CUDA;
    if (rc == GNDT_OK) rc = gndt_xchg_create(m->h[i], i, ndev, cap_records, cap_halo_records, what, &info[i]);
    if (rc != GNDT_OK) { g_create_error = "gndt_multi_create: device " + std::to_string(devices[i]) + ": " + (m->h[i] ? m->h[i]->err : g_create_error); gndt_multi_destroy(m); return rc; }
  }
  for (int i = 0; i < ndev; ++i) {
    const int rc = gndt_xchg_connect(m->h[i], info.data(), ndev);
    if (rc != GNDT_OK) { g_create_error = "gndt_multi_create: " + m->h[i]->err; gndt_multi_destroy(m); return rc; }
  }
  *out = m;
  return GNDT_OK;
}

int gndt_multi_destroy(gndt_multi *m) {
  if (!m) return GNDT_ERR_INVALID_ARG;
  for (size_t i = 0; i < m->h.size(); ++i) {
    if (!m->h[i]) continue;
    cudaSetDevice(m->dev[i]);
    cudaDeviceSynchronize();
    if (m->cloud[i].p) cudaFree(m->cloud[i].p);
    if (m->st[i]) cudaStreamDestroy(m->st[i]);
    gndt_destroy(m->h[i]);
  }
  delete m;
  return GNDT_OK;
}

const char *gndt_multi_last_error(const gndt_multi *m) { return m ? m->err.c_str() : g_create_error.c_str(); }
gndt_handle *gndt_multi_handle(gndt_multi *m, int index) { return (m && index >= 0 && index < (int)m->h.size()) ? m->h[index] : nullptr; }

// every GPU gets the whole cloud: host input goes up each GPU's own PCIe link, device input (on GPU 0) fans out over NVLink
static int multi_stage(gndt_multi *m, const void *xyz, size_t n, size_t stride_bytes, int mem) {
  const size_t bytes = n * stride_bytes;
  for (size_t i = 0; i < m->h.size(); ++i) {
    gndt_handle *h = m->h[i];
    if (cudaSetDevice(m->dev[i]) != cudaSuccess) return multi_fail(m, (int)i, GNDT_ERR_CUDA, "cudaSetDevice");
    if (mem == GNDT_MEM_DEVICE && i == 0) continue;  // already there
    int rc = ensure(h, m->cloud[i], bytes);
    if (rc != GNDT_OK) return multi_fail(m, (int)i, rc, "cloud staging");
    cudaError_t e = mem == GNDT_MEM_HOST ? cudaMemcpyAsync(m->cloud[i].p, xyz, bytes, cudaMemcpyHostToDevice, m->st[i])
                                         : cudaMemcpyPeerAsync(m->cloud[i].p, m->dev[i], xyz, m->dev[0], bytes, m->st[i]);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return multi_fail(m, (int)i, GNDT_ERR_CUDA, "cloud copy"); }
  }
  return GNDT_OK;
}
static const void *multi_cloud(gndt_multi *m, size_t i, const void *xyz, int mem) { return (mem == GNDT_MEM_DEVICE && i == 0) ? xyz : m->cloud[i].p; }

int gndt_multi_build(gndt_multi *m, const void *xyz, size_t n, size_t stride_bytes, int mem) {
  if (!m || !xyz || n == 0) return GNDT_ERR_INVALID_ARG;
  const int nd = (int)m->h.size();
  int rc = multi_stage(m, xyz, n, stride_bytes, mem);
  if (rc != GNDT_OK) return rc;
  // balanced x strips from GPU 0's histogram of the cloud's x columns; the origin is the same on every GPU
  cudaSetDevice(m->dev[0]);
  m->cuts.assign(nd + 1, 0);
  gndt_params p0 = m->params;
  p0.tile_lo = p0.tile_hi = 0;
  if ((rc = gndt_set_params(m->h[0], &p0)) != GNDT_OK) return multi_fail(m, 0, rc, "set_params");
  if ((rc = gndt_plan_tiles(m->h[0], multi_cloud(m, 0, xyz, mem), n, stride_bytes, GNDT_MEM_DEVICE, nd, m->cuts.data(), m->st[0])) != GNDT_OK)
    return multi_fail(m, 0, rc, "gndt_plan_tiles");
  m->planned = true;
  for (int i = 0; i < nd; ++i) {
    cudaSetDevice(m->dev[i]);
    gndt_params p = m->params;
    const bool empty = nd > 1 && m->cuts[i] >= m->cuts[i + 1];
    p.tile_lo = nd == 1 ? 0 : (empty ? GNDT_MAX_INDEX : m->cuts[i]);
    p.tile_hi = nd == 1 ? 0 : (empty ? GNDT_MAX_INDEX + 1 : m->cuts[i + 1]);
    if ((rc = gndt_set_params(m->h[i], &p)) != GNDT_OK) return multi_fail(m, i, rc, "set_params");
    if ((rc = gndt_build(m->h[i], multi_cloud(m, i, xyz, mem), n, stride_bytes, GNDT_MEM_DEVICE, m->st[i])) != GNDT_OK) return multi_fail(m, i, rc, "gndt_build");
    if ((rc = gndt_xchg_run(m->h[i], m->st[i])) != GNDT_OK) return multi_fail(m, i, rc, "gndt_xchg_run");
  }
  return GNDT_OK;
}

int gndt_multi_update(gndt_multi *m, const void *xyz, size_t n, size_t stride_bytes, int mem) {
  if (!m || !xyz || n == 0) return GNDT_ERR_INVALID_ARG;
  if (!m->planned) { m->err = "gndt_multi_update: no map has been built"; return GNDT_ERR_STATE; }
  int rc = multi_stage(m, xyz, n, stride_bytes, mem);
  if (rc != GNDT_OK) return rc;
  for (size_t i = 0; i < m->h.size(); ++i) {  // every GPU keeps the points of its strip
    cudaSetDevice(m->dev[i]);
    if ((rc = gndt_update(m->h[i], multi_cloud(m, i, xyz, mem), n, stride_bytes, GNDT_MEM_DEVICE, m->st[i])) != GNDT_OK) return multi_fail(m, (int)i, rc, "gndt_update");
    if ((rc = gndt_xchg_run(m->h[i], m->st[i])) != GNDT_OK) return multi_fail(m, (int)i, rc, "gndt_xchg_run");
  }
  return GNDT_OK;
}

int gndt_multi_view(gndt_multi *m, int index, gndt_xchg_view *out) {
  if (!m || !out || index < 0 || index >= (int)m->h.size()) return GNDT_ERR_INVALID_ARG;
  // a strip that failed makes the others fail too (they name it): report the failing strip's own error
  int first = -1, first_rc = GNDT_OK;
  for (size_t i = 0; i < m->h.size(); ++i) {
    cudaSetDevice(m->dev[i]);
    gndt_xchg_view v;
    const int rc = gndt_xchg_view_get(m->h[i], (int)i == index ? out : &v);
    if (rc == GNDT_OK || (first >= 0 && !m->h[first]->x_peer_failed)) continue;
    if (first < 0 || !m->h[i]->x_peer_failed) { first = (int)i; first_rc = rc; }
  }
  return first < 0 ? GNDT_OK : multi_fail(m, first, first_rc, "exchange");
}

int gndt_multi_cuts(gndt_multi *m, int32_t *cuts, int cap) {
  if (!m || !cuts || cap < (int)m->cuts.size()) return GNDT_ERR_INVALID_ARG;
  std::copy(m->cuts.begin(), m->cuts.end(), cuts);
  return GNDT_OK;
}

__global__ void cx_hist_kernel(u32 *hist, const float *in, size_t stride_f, size_t n_in, size_t start, DevParams P) {
  float o[3];
  if (P.origin_first) { o[0] = __ldg(in); o[1] = __ldg(in + 1); o[2] = __ldg(in + 2); }
  else { o[0] = P.origin[0]; o[1] = P.origin[1]; o[2] = P.origin[2]; }
  const bool vec = (stride_f == 4) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
  for (size_t i = start + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_in; i += (size_t)gridDim.x * blockDim.x) {
    float4 p = load_point(in, stride_f, i, vec);
    int cx, cy, cz;
    const bool ok = P.fast_div ? point_indices<true>(p.x, p.y, p.z, o, P.grid_len, P.z_len, P.rinv[0], P.rinv[1], cx, cy, cz)
                               : point_indices<false>(p.x, p.y, p.z, o, P.grid_len, P.z_len, P.rinv[0], P.rinv[1], cx, cy, cz);
    if (ok) atomicAdd(&hist[cx + kIdxBias], 1u);
  }
}

int gndt_plan_tiles(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, int ntiles, int32_t *cuts,
                    void *stream) {
  if (!h || !xyz || !cuts || ntiles < 1 || n == 0 || stride_bytes < 12 || (stride_bytes & 3)) return GNDT_ERR_INVALID_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GNDT_CUDA(h, cudaSetDevice(h->device));
  const float *d_in;
  int rc = upload(h, h->in_stage, xyz, n * stride_bytes, mem, st, nullptr, &d_in);
  if (rc != GNDT_OK) return rc;
  if ((rc = ensure(h, h->f_zero, 65536 * sizeof(u32) + 1024)) != GNDT_OK) return rc;
  GNDT_CUDA(h, cudaMemsetAsync(h->f_zero.p, 0, 65536 * sizeof(u32), st));
  const DevParams dp = make_dev(h, h->params, 0);
  launch(h, false, cx_hist_kernel, grid_for(h, n, 256 * 8, 8), 256, 0, st, (u32 *)h->f_zero.p, d_in, stride_bytes / 4, n,
         h->params.origin_is_first_point ? 1 : 0, dp);
  GNDT_CUDA(h, cudaGetLastError());
  u32 *hist = (u32 *)malloc(65536 * sizeof(u32));
  cudaError_t e = cudaMemcpyAsync(hist, h->f_zero.p, 65536 * sizeof(u32), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { free(hist); h->err = cudaGetErrorString(e); return GNDT_ERR_CUDA; }
  uint64_t total = 0;
  for (int i = 0; i < 65536; ++i) total += hist[i];
  cuts[0] = -kIdxBias;
  cuts[ntiles] = kIdxBias;
  uint64_t acc = 0;
  int t = 1;
  for (int i = 0; i < 65536 && t < ntiles; ++i) {
    acc += hist[i];
    while (t < ntiles && acc * (uint64_t)ntiles >= total * (uint64_t)t) cuts[t++] = i - kIdxBias + 1;
  }
  for (; t < ntiles; ++t) cuts[t] = kIdxBias;
  free(hist);
  return GNDT_OK;
}

int gndt_set_stage_timing(gndt_handle *h, int on) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  h->stage_timing = on != 0;
  return GNDT_OK;
}

int gndt_stage_ms(gndt_handle *h, float ms[GNDT_N_STAGES]) {
  if (!h || !ms) return GNDT_ERR_INVALID_ARG;
  if (!h->built) return GNDT_ERR_STATE;
  GNDT_CUDA(h, cudaStreamSynchronize(h->last_stream));
  for (int i = 0; i < GNDT_N_STAGES; ++i) ms[i] = 0.f;
  if (h->stages_valid) {
    GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_KEY], h->ev[EV_START], h->ev[EV_KEY]));
    GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_SORT], h->ev[EV_KEY], h->ev[EV_SORT]));
    GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_REDUCE], h->ev[EV_SORT], h->ev[EV_REDUCE]));
    GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_LABEL], h->ev[EV_REDUCE], h->ev[EV_LABEL]));
    GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_EDGES], h->ev[EV_LABEL], h->ev[EV_EDGES]));
  }
  GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_TOTAL], h->ev[EV_START], h->ev[EV_EDGES]));
  if (h->timed_h2d) GNDT_CUDA(h, cudaEventElapsedTime(&ms[GNDT_STAGE_H2D], h->ev[EV_H2D0], h->ev[EV_START]));
  return GNDT_OK;
}

int gndt_fast_div_status(gndt_handle *h, int *enabled, uint64_t *values_checked) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (enabled) *enabled = (h->div[0].ok && h->div[1].ok) ? 1 : 0;
  if (values_checked) *values_checked = h->divcheck_values;
  return GNDT_OK;
}

int gndt_launch_count(gndt_handle *h, uint64_t *n_launches) {
  if (!h || !n_launches) return GNDT_ERR_INVALID_ARG;
  *n_launches = h->launches;
  return GNDT_OK;
}

// ---- host key helpers ------------------------------------------------------------------

static int host_axis(float p, float p0, float len, int32_t *s) {
  volatile float d = p - p0;
  volatile float q = std::fabs(d) / len;
  float c = std::ceil(q);
  if (!(c <= (float)GNDT_MAX_INDEX)) return 0;
  int32_t n = (int32_t)c;
  if (n == 0) n = 1;
  *s = (p > p0) ? n : -n;
  return 1;
}

int gndt_trans_morton_xyz(const float origin[3], float grid_len, float z_len, const float pos[3], int32_t *sx,
                          int32_t *sy, int32_t *sz) {
  if (!origin || !pos || !sx || !sy || !sz) return GNDT_ERR_INVALID_ARG;
  if (!host_axis(pos[0], origin[0], grid_len, sx) || !host_axis(pos[1], origin[1], grid_len, sy) ||
      !host_axis(pos[2], origin[2], z_len, sz))
    return GNDT_ERR_INVALID_ARG;
  return GNDT_OK;
}

uint32_t gndt_count_morton(uint32_t nx, uint32_t ny) {
  uint32_t m = 0;
  for (int k = 0; k < 16; ++k) m |= ((nx >> k) & 1u) << (2 * k + 1) | ((ny >> k) & 1u) << (2 * k);
  return m;
}

void gndt_morton_to_xy(uint32_t morton, uint32_t *nx, uint32_t *ny) {
  uint32_t a = 0, b = 0;
  for (int k = 0; k < 16; ++k) { a |= ((morton >> (2 * k + 1)) & 1u) << k; b |= ((morton >> (2 * k)) & 1u) << k; }
  if (nx) *nx = a;
  if (ny) *ny = b;
}

int gndt_morton_string(int32_t sx, int32_t sy, char *buf) {
  if (!buf) return 0;
  const char q = sx > 0 ? (sy > 0 ? 'A' : 'B') : (sy > 0 ? 'C' : 'D');
  return snprintf(buf, 16, "%c%d", q, (int)gndt_count_morton((uint32_t)abs(sx), (uint32_t)abs(sy)));
}

/* TwoDmap::countPositionXYZ (include/map2D.h:918-947): centre of a cell, in metres, with the
 * reference's own float/double mix ((a - 0.5) is double, * gridLen float->double, + origin). */
int gndt_cell_center(const float origin[3], float grid_len, float z_len, int32_t sx, int32_t sy, int32_t sz,
                     float center[3]) {
  if (!origin || !center || sx == 0 || sy == 0 || sz == 0) return GNDT_ERR_INVALID_ARG;
  const double ax = (std::abs(sx) - 0.5) * grid_len, ay = (std::abs(sy) - 0.5) * grid_len, az = (std::abs(sz) - 0.5) * z_len;
  center[0] = (float)(sx > 0 ? ax + origin[0] : origin[0] - ax);
  center[1] = (float)(sy > 0 ? ay + origin[1] : origin[1] - ay);
  center[2] = (float)(sz > 0 ? origin[2] + az : origin[2] - az);
  return GNDT_OK;
}

int gndt_key_layout(gndt_handle *h, int out[4]) {
  if (!h || !out) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  out[0] = h->host_ctl.n_passes; out[1] = h->host_ctl.bcol; out[2] = (int)h->host_ctl.ny; out[3] = h->host_ctl.bz;
  return GNDT_OK;
}

int64_t gndt_find_column(const gndt_column *cols, size_t n_cols, int32_t sx, int32_t sy) {
  return gndtl_find_column(cols, n_cols, sx, sy);
}
int64_t gndt_find_slope(const gndt_column *cols, size_t n_cols, const gndt_slope *slopes, int32_t sx, int32_t sy,
                        int32_t sz) {
  return gndtl_find_slope(cols, n_cols, slopes, sx, sy, sz);
}
int64_t gndt_neighbor_column(const gndt_column *cols, size_t n_cols, int32_t sx, int32_t sy, int dir) {
  return gndtl_neighbor_column(cols, n_cols, sx, sy, dir);
}

int gndt_origin(gndt_handle *h, float origin[3]) {
  if (!h || !origin) return GNDT_ERR_INVALID_ARG;
  int rc = sync_counts(h);
  if (rc != GNDT_OK) return rc;
  for (int i = 0; i < 3; ++i) origin[i] = h->host_ctl.origin[i];
  return GNDT_OK;
}

// ---- NDT scan-to-map registration -------------------------------------------------------

void gndt_default_ndt_params(gndt_ndt_params *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->outlier_ratio = 0.55f;
  p->min_voxel_points = 6;
  p->max_iterations = 100;
  p->translation_epsilon = 1e-4;
  p->rotation_epsilon = 1e-4;
}

namespace {

struct NdtEval {  // one pass at one pose
  double score, g[6], H[36], c[3];
  uint64_t n_points, n_matched, n_pairs;
};

// Exp(phi) of so(3) (Rodrigues), row-major
void so3_exp(const double phi[3], double E[9]) {
  const double th2 = phi[0] * phi[0] + phi[1] * phi[1] + phi[2] * phi[2], th = std::sqrt(th2);
  const double a = th2 < 1e-24 ? 1.0 - th2 / 6.0 : std::sin(th) / th;
  const double b = th2 < 1e-24 ? 0.5 - th2 / 24.0 : (1.0 - std::cos(th)) / th2;
  const double K[9] = {0.0, -phi[2], phi[1], phi[2], 0.0, -phi[0], -phi[1], phi[0], 0.0};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double kk = 0.0;
      for (int m = 0; m < 3; ++m) kk += K[3 * i + m] * K[3 * m + j];
      E[3 * i + j] = (i == j ? 1.0 : 0.0) + a * K[3 * i + j] + b * kk;
    }
}

// Cholesky solve of the 6x6 system A x = b; false if A is not positive definite
bool chol6(const double A_in[36], const double b[6], double x[6]) {
  double L[36] = {};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = A_in[6 * i + j];
      for (int k = 0; k < j; ++k) s -= L[6 * i + k] * L[6 * j + k];
      if (i == j) {
        if (!(s > 0.0) || !std::isfinite(s)) return false;
        L[6 * i + i] = std::sqrt(s);
      } else {
        L[6 * i + j] = s / L[6 * j + j];
      }
    }
  double y[6];
  for (int i = 0; i < 6; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= L[6 * i + k] * y[k];
    y[i] = s / L[6 * i + i];
  }
  for (int i = 5; i >= 0; --i) {
    double s = y[i];
    for (int k = i + 1; k < 6; ++k) s -= L[6 * k + i] * x[k];
    x[i] = s / L[6 * i + i];
  }
  return true;
}

int ndt_check_args(gndt_handle *h, const double *T, const gndt_ndt_params *np) {
  for (int i = 0; i < 16; ++i)
    if (!std::isfinite(T[i])) { h->err = "gndt_register: the guess is not finite"; return GNDT_ERR_INVALID_ARG; }
  if (T[12] != 0.0 || T[13] != 0.0 || T[14] != 0.0 || T[15] != 1.0) { h->err = "gndt_register: the guess's bottom row is not 0 0 0 1"; return GNDT_ERR_INVALID_ARG; }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const double rtr = T[i] * T[j] + T[4 + i] * T[4 + j] + T[8 + i] * T[8 + j];  // (R^T R)_ij
      if (!(std::fabs(rtr - (i == j ? 1.0 : 0.0)) <= 1e-6)) { h->err = "gndt_register: the guess's rotation is not orthonormal"; return GNDT_ERR_INVALID_ARG; }
    }
  if (!(np->outlier_ratio > 0.f && np->outlier_ratio < 1.f) || np->min_voxel_points < 3 || np->max_iterations < 0 || np->reserved != 0 ||
      !(np->translation_epsilon >= 0.0) || !(np->rotation_epsilon >= 0.0) || !std::isfinite(np->translation_epsilon) ||
      !std::isfinite(np->rotation_epsilon)) {
    h->err = "gndt_register: ndt parameter out of range";
    return GNDT_ERR_INVALID_ARG;
  }
  return GNDT_OK;
}

// The tables of the level of factor k (gndt.h, gndt_register_levels), once per map state and factor:
// coarse columns by slab (count, scan, emit), then coarse voxels by coarse column (count, scan,
// emit).  Two read-backs: the map's first and last column (the slab range) and the coarse column
// count.  cov: the voxels go to L.cov with c = Sigma' (D2D); the columns are the same either way.
int ndt_build_level(gndt_handle *h, int k, cudaStream_t st, bool cov) {
  gndt_handle::NdtLevel &L = h->ndt_lv[k];
  Buffer &vox = cov ? L.cov : L.vox;
  const u32 n_vox = h->host_ctl.n_voxels, n_cols = h->host_ctl.n_columns;
  int rc;
  if ((rc = ensure(h, vox, std::max<size_t>(n_vox, 1) * sizeof(NdtVoxel))) != GNDT_OK) return rc;
  if ((rc = ensure(h, L.cols, std::max<size_t>(n_cols, 1) * sizeof(gndt_column))) != GNDT_OK) return rc;
  L.n_cols = L.n_vox = 0;
  if (n_cols) {
    const gndt_column *cols = (const gndt_column *)h->columns.p;
    gndt_column ends[2];
    GNDT_CUDA(h, cudaMemcpyAsync(&ends[0], cols, sizeof(gndt_column), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaMemcpyAsync(&ends[1], cols + n_cols - 1, sizeof(gndt_column), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaStreamSynchronize(st));
    const int X0 = floor_div(contiguous_index(ends[0].sx), k), X1 = floor_div(contiguous_index(ends[1].sx), k);
    const u32 n_slabs = (u32)(X1 - X0 + 1);
    // work: scan scratch of the slabs | of the coarse columns (zeroed) | slab counts, offsets | members | voxel counts, offsets
    Layout W;
    const ScanScratch s1(W, n_slabs), s2(W, n_cols);
    const size_t zero_bytes = W.bytes;
    const size_t o_sc = W.take((size_t)n_slabs * 4), o_sb = W.take(((size_t)n_slabs + 1) * 4), o_m = W.take((size_t)n_cols * 4);
    const size_t o_vc = W.take((size_t)n_cols * 4), o_vb = W.take(((size_t)n_cols + 1) * 4);
    if ((rc = ensure(h, h->ndt_lv_work, W.bytes)) != GNDT_OK) return rc;
    const Buffer &w = h->ndt_lv_work;
    u32 *slab_count = at<u32>(w, o_sc), *slab_begin = at<u32>(w, o_sb), *members = at<u32>(w, o_m);
    u32 *vcount = at<u32>(w, o_vc), *vbegin = at<u32>(w, o_vb);
    gndt_column *ccols = (gndt_column *)L.cols.p;
    GNDT_CUDA(h, cudaMemsetAsync(w.p, 0, zero_bytes, st));
    const int g_slab = (int)(((size_t)n_slabs * 32 + 255) / 256);
    launch(h, false, ndt_level_columns_kernel<false>, g_slab, 256, 0, st, cols, n_cols, k, X0, n_slabs, slab_count, (const u32 *)nullptr,
           ccols, members);
    launch(h, false, exclusive_scan_kernel, grid_for(h, (n_slabs + kScanTile - 1) / kScanTile, 1, 4), 256, 0, st, at<ScanCtl>(w, s1.ctl),
           (const u32 *)slab_count, n_slabs, (const u32 *)nullptr, slab_begin, at<u64>(w, s1.state), at<GroupState>(w, s1.groups));
    launch(h, false, ndt_level_columns_kernel<true>, g_slab, 256, 0, st, cols, n_cols, k, X0, n_slabs, (u32 *)nullptr,
           (const u32 *)slab_begin, ccols, members);
    ScanCtl hs;
    GNDT_CUDA(h, cudaGetLastError());
    GNDT_CUDA(h, cudaMemcpyAsync(&hs, at<ScanCtl>(w, s1.ctl), sizeof(hs), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaStreamSynchronize(st));
    if (hs.err) { h->err = "level column scan watchdog"; return GNDT_ERR_INTERNAL; }
    const u32 nc = hs.total;
    const int g_col = grid_for(h, nc, 256, 8);
    const gndt_voxel *table = (const gndt_voxel *)h->table.p;
    launch(h, false, ndt_level_voxels_kernel<false>, g_col, 256, 0, st, table, cols, (const u32 *)members, k, h->res_params.normalize_cov,
           ccols, nc, vcount, (const u32 *)nullptr, (NdtVoxel *)nullptr);
    launch(h, false, exclusive_scan_kernel, grid_for(h, (nc + kScanTile - 1) / kScanTile, 1, 4), 256, 0, st, at<ScanCtl>(w, s2.ctl),
           (const u32 *)vcount, nc, (const u32 *)nullptr, vbegin, at<u64>(w, s2.state), at<GroupState>(w, s2.groups));
    if (cov)
      launch(h, false, ndt_level_voxels_kernel<true, true>, g_col, 256, 0, st, table, cols, (const u32 *)members, k,
             h->res_params.normalize_cov, ccols, nc, (u32 *)nullptr, (const u32 *)vbegin, (NdtVoxel *)vox.p);
    else
      launch(h, false, ndt_level_voxels_kernel<true>, g_col, 256, 0, st, table, cols, (const u32 *)members, k, h->res_params.normalize_cov,
             ccols, nc, (u32 *)nullptr, (const u32 *)vbegin, (NdtVoxel *)vox.p);
    GNDT_CUDA(h, cudaGetLastError());
    GNDT_CUDA(h, cudaMemcpyAsync(&hs, at<ScanCtl>(w, s2.ctl), sizeof(hs), cudaMemcpyDeviceToHost, st));
    GNDT_CUDA(h, cudaStreamSynchronize(st));
    if (hs.err) { h->err = "level voxel scan watchdog"; return GNDT_ERR_INTERNAL; }
    L.n_cols = nc;
    L.n_vox = hs.total;
  }
  (cov ? h->ndt_lv_cov_ready : h->ndt_lv_ready) |= 1ull << k;
  return GNDT_OK;
}

int ndt_check_levels(gndt_handle *h, const gndt_ndt_level *levels, int n_levels) {
  if (n_levels < 0 || n_levels > GNDT_NDT_MAX_LEVELS || (n_levels > 0 && !levels)) {
    h->err = "gndt_register_levels: n_levels outside [0, GNDT_NDT_MAX_LEVELS] or levels is NULL";
    return GNDT_ERR_INVALID_ARG;
  }
  for (int i = 0; i < n_levels; ++i) {
    const gndt_ndt_level &l = levels[i];
    if (l.factor < 2 || l.factor > kNdtMaxFactor || (i > 0 && l.factor >= levels[i - 1].factor) || l.max_iterations < 0 ||
        !(l.translation_epsilon >= 0.0) || !(l.rotation_epsilon >= 0.0) || !std::isfinite(l.translation_epsilon) ||
        !std::isfinite(l.rotation_epsilon)) {
      h->err = "gndt_register_levels: level " + std::to_string(i) + " out of range (factor in [2, 32] and strictly decreasing, "
               "max_iterations >= 0, epsilons finite and >= 0)";
      return GNDT_ERR_INVALID_ARG;
    }
  }
  return GNDT_OK;
}

// The scan's own Gaussians for gndt_register_d2d, on the builder h->ndt_scan (created here on the first
// call): a gndt_build of the scan with the resident map's parameters and origin, every point binned,
// then its Sigma'-form prepare and level tables.  Launches count on the builder, not on h.
int ndt_scan_gaussians(gndt_handle *h, const float *d_in, size_t n, size_t stride_bytes, const gndt_ndt_level *levels, int n_levels,
                       cudaStream_t st) {
  int rc = GNDT_OK;
  if (!h->ndt_scan && (rc = gndt_create(&h->res_params, h->device, &h->ndt_scan)) != GNDT_OK) {
    h->err = std::string("gndt_register_d2d: scan build: ") + gndt_last_error(nullptr);
    return rc;
  }
  gndt_handle *s = h->ndt_scan;
  gndt_params p = h->res_params;
  p.origin_is_first_point = 0;
  for (int i = 0; i < 3; ++i) p.origin[i] = h->host_ctl.origin[i];
  p.tile_lo = p.tile_hi = 0;
  p.max_voxels = 0;
  if ((rc = gndt_set_params(s, &p)) == GNDT_OK && (rc = gndt_build(s, d_in, n, stride_bytes, GNDT_MEM_DEVICE, st)) == GNDT_OK &&
      (rc = sync_counts(s)) == GNDT_OK && (rc = ensure(s, s->ndt_cov, std::max<size_t>(s->host_ctl.n_voxels, 1) * sizeof(NdtVoxel))) == GNDT_OK) {
    launch(s, false, ndt_prepare_kernel<true>, grid_for(s, s->host_ctl.n_voxels, 256, 8), 256, 0, st, s->ctl, (const gndt_voxel *)s->table.p,
           (NdtVoxel *)s->ndt_cov.p, p.normalize_cov);
    for (int i = 0; i < n_levels && rc == GNDT_OK; ++i) rc = ndt_build_level(s, levels[i].factor, st, true);
  }
  if (rc != GNDT_OK) h->err = "gndt_register_d2d: scan build: " + s->err;
  return rc;
}

// gndt_register / gndt_register_levels (P2D) and gndt_register_d2d: one Levenberg-Marquardt loop per
// level, the derivative pass differs.
int register_levels(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, const double guess[16],
                    const gndt_ndt_params *np, const gndt_ndt_level *levels, int n_levels, gndt_registration *out,
                    gndt_registration *level_out, void *stream, bool d2d) {
  const char *who = d2d ? "gndt_register_d2d" : levels ? "gndt_register_levels" : "gndt_register";
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!guess || !np || !out) { h->err = std::string(who) + ": guess, np and out must not be NULL"; return GNDT_ERR_INVALID_ARG; }
  int rc = check_cloud_args(h, xyz, n, stride_bytes, mem, who);
  if (rc != GNDT_OK) return rc;
  if ((rc = ndt_check_args(h, guess, np)) != GNDT_OK) return rc;
  if ((rc = ndt_check_levels(h, levels, n_levels)) != GNDT_OK) return rc;
  GNDT_CUDA(h, cudaSetDevice(h->device));
  if ((rc = sync_counts(h)) != GNDT_OK) return rc;  // resolves a pending update / remove
  KeepLaunchCount keep(h);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const gndt_params &rp = h->res_params;
  const u32 n_vox = h->host_ctl.n_voxels, n_cols = h->host_ctl.n_columns;

  // the resident map's Gaussians, once per map state and form (C for P2D, Sigma' for D2D); each
  // level's, once per map state, form and factor
  Buffer &map_vox = d2d ? h->ndt_cov : h->ndt_vox;
  if (!(d2d ? h->ndt_cov_ready : h->ndt_ready)) {
    if ((rc = ensure(h, map_vox, std::max<size_t>(n_vox, 1) * sizeof(NdtVoxel))) != GNDT_OK) return rc;
    if (d2d)
      launch(h, false, ndt_prepare_kernel<true>, grid_for(h, n_vox, 256, 8), 256, 0, st, h->ctl, (const gndt_voxel *)h->table.p,
             (NdtVoxel *)map_vox.p, rp.normalize_cov);
    else
      launch(h, false, ndt_prepare_kernel<false>, grid_for(h, n_vox, 256, 8), 256, 0, st, h->ctl, (const gndt_voxel *)h->table.p,
             (NdtVoxel *)map_vox.p, rp.normalize_cov);
  }
  for (int i = 0; i < n_levels; ++i)
    if (!((d2d ? h->ndt_lv_cov_ready : h->ndt_lv_ready) >> levels[i].factor & 1) &&
        (rc = ndt_build_level(h, levels[i].factor, st, d2d)) != GNDT_OK)
      return rc;
  const float *d_in;
  if ((rc = upload(h, h->ndt_pts, xyz, n * stride_bytes, mem, st, nullptr, &d_in)) != GNDT_OK) return rc;
  const int blocks = grid_for(h, n, kNdtThreads, 8);
  if ((rc = ensure(h, h->ndt_part, ((size_t)blocks + 1) * kNdtWidth * sizeof(double))) != GNDT_OK) return rc;
  if (!h->ndt_host) GNDT_CUDA(h, cudaHostAlloc(&h->ndt_host, kNdtWidth * sizeof(double), cudaHostAllocDefault));
  double *part = static_cast<double *>(h->ndt_part.p), *dres = part + (size_t)blocks * kNdtWidth;
  const size_t stride_f = stride_bytes / 4;

  // centre: binary64 mean of the finite points, c = R pbar + t at every pose
  launch(h, false, ndt_mean_kernel, blocks, kNdtThreads, 0, st, d_in, stride_f, n, part);
  launch(h, false, ndt_finish_kernel, 1, 32, 0, st, part, blocks, 4, dres);
  GNDT_CUDA(h, cudaGetLastError());
  GNDT_CUDA(h, cudaMemcpyAsync(h->ndt_host, dres, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  GNDT_CUDA(h, cudaStreamSynchronize(st));
  (d2d ? h->ndt_cov_ready : h->ndt_ready) = true;
  const uint64_t n_points = (uint64_t)h->ndt_host[3];
  const double pbar[3] = {n_points ? h->ndt_host[0] / (double)n_points : 0.0, n_points ? h->ndt_host[1] / (double)n_points : 0.0,
                          n_points ? h->ndt_host[2] / (double)n_points : 0.0};

  if (d2d && (rc = ndt_scan_gaussians(h, d_in, n, stride_bytes, levels, n_levels, st)) != GNDT_OK) return rc;

  // the derivative passes: pass(P) launches one at pose P and returns its number of blocks
  auto p2d = [=](const NdtVoxel *vox, const gndt_column *cols, u32 nc) {
    return [=](const NdtPose &P) {
      launch(h, false, ndt_pass_kernel, blocks, kNdtThreads, 0, st, d_in, stride_f, n, vox, cols, nc, P, part);
      return blocks;
    };
  };
  auto d2d_pass = [=](const Buffer &svox, u32 n_svox, const NdtVoxel *vox, const gndt_column *cols, u32 nc) {
    const int b = grid_for(h, n_svox, kNdtThreads, 8);  // n_svox <= n: the partials fit
    const NdtVoxel *sv = (const NdtVoxel *)svox.p;
    return [=](const NdtPose &P) {
      launch(h, false, ndt_d2d_pass_kernel, b, kNdtThreads, 0, st, sv, n_svox, vox, cols, nc, P, part);
      return b;
    };
  };

  // Levenberg-Marquardt on one level (factor 1: the map) from T_in -> *res
  auto solve = [&](int factor, const auto &pass, int max_iterations, double teps, double reps, const double T_in[16],
                   gndt_registration *res) -> int {
    NdtPose P = {};
    {
      const double p_o = np->outlier_ratio, kg = (double)factor * (double)rp.grid_len, kz = (double)factor * (double)rp.z_len;
      const double V = kg * kg * kz;
      const double c1 = 10.0 * (1.0 - p_o), c2 = p_o / V, d3 = -std::log(c2);
      P.d1 = -std::log(c1 + c2) - d3;
      P.d2 = -2.0 * std::log((-std::log(c1 * std::exp(-0.5) + c2) - d3) / P.d1);
    }
    for (int i = 0; i < 3; ++i) P.origin[i] = h->host_ctl.origin[i];
    P.grid_len = rp.grid_len;
    P.z_len = rp.z_len;
    P.min_points = (u32)np->min_voxel_points;
    P.factor = factor;

    auto eval = [&](const double T[16], NdtEval &e) -> int {
      for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) P.r[3 * i + j] = T[4 * i + j];
        P.t[i] = T[4 * i + 3];
        P.c[i] = T[4 * i] * pbar[0] + T[4 * i + 1] * pbar[1] + T[4 * i + 2] * pbar[2] + T[4 * i + 3];
      }
      const int nb = pass(P);
      launch(h, false, ndt_finish_kernel, 1, 32, 0, st, part, nb, kNdtWidth, dres);
      GNDT_CUDA(h, cudaGetLastError());
      GNDT_CUDA(h, cudaMemcpyAsync(h->ndt_host, dres, kNdtWidth * sizeof(double), cudaMemcpyDeviceToHost, st));
      GNDT_CUDA(h, cudaStreamSynchronize(st));
      const double *r = h->ndt_host;
      e.score = r[0];
      for (int k = 0; k < 6; ++k) e.g[k] = r[1 + k];
      for (int k = 0, idx = 7; k < 6; ++k)
        for (int l = k; l < 6; ++l, ++idx) e.H[6 * k + l] = e.H[6 * l + k] = r[idx];
      for (int i = 0; i < 3; ++i) e.c[i] = P.c[i];
      e.n_points = (uint64_t)r[28];
      e.n_matched = (uint64_t)r[29];
      e.n_pairs = (uint64_t)r[30];
      return GNDT_OK;
    };

    double T[16];
    memcpy(T, T_in, sizeof(T));
    NdtEval cur;
    int rc = eval(T, cur);
    if (rc != GNDT_OK) return rc;
    int term = GNDT_NDT_MAX_ITER;
    uint32_t iters = 0;
    if (cur.n_pairs == 0) {
      term = GNDT_NDT_NO_MATCH;
      cur.score = 0.0;
      memset(cur.g, 0, sizeof(cur.g));
      memset(cur.H, 0, sizeof(cur.H));
    } else {
      // Levenberg-Marquardt on -S: (-H + lambda diag(max(-H_ii, tiny))) delta = g
      constexpr double kLambda0 = 1e-3, kLambdaMin = 1e-12, kLambdaMax = 1e12;
      double lambda = kLambda0;
      while (iters < (uint32_t)max_iterations) {
        double hmax = 0.0;
        for (int i = 0; i < 6; ++i) hmax = std::max(hmax, std::fabs(cur.H[7 * i]));
        const double tiny = std::max(1e-6 * hmax, 1e-300);
        double A[36], delta[6];
        for (int i = 0; i < 36; ++i) A[i] = -cur.H[i];
        for (int i = 0; i < 6; ++i) A[7 * i] += lambda * std::max(-cur.H[7 * i], tiny);
        if (!chol6(A, cur.g, delta)) {
          lambda *= 10.0;
          if (lambda > kLambdaMax) { term = GNDT_NDT_STALLED; break; }
          continue;
        }
        // converged: the (nearly undamped) step to the optimum of the local model is below both
        // epsilons.  Tested before the pass because there S need not rise any more: candidate sets
        // change between poses, and on the tails of thin Gaussians the Hessian is indefinite, lambda
        // grows and steps shrink far from the optimum, so a short damped step says nothing
        const double dr = std::sqrt(delta[0] * delta[0] + delta[1] * delta[1] + delta[2] * delta[2]);
        const double dp = std::sqrt(delta[3] * delta[3] + delta[4] * delta[4] + delta[5] * delta[5]);
        if (lambda < 1.0 && dr < teps && dp < reps) { term = GNDT_NDT_CONVERGED; break; }
        // candidate: T' = (E, c + rho - E c) o T, E = Exp(phi)
        double E[9], Tn[16];
        so3_exp(delta + 3, E);
        memcpy(Tn, T, sizeof(Tn));
        for (int i = 0; i < 3; ++i) {
          double tt = cur.c[i] + delta[i];
          for (int j = 0; j < 3; ++j) {
            Tn[4 * i + j] = E[3 * i] * T[j] + E[3 * i + 1] * T[4 + j] + E[3 * i + 2] * T[8 + j];
            tt += E[3 * i + j] * (T[4 * j + 3] - cur.c[j]);
          }
          Tn[4 * i + 3] = tt;
        }
        NdtEval cand;
        if ((rc = eval(Tn, cand)) != GNDT_OK) return rc;
        ++iters;
        if (cand.score > cur.score) {
          memcpy(T, Tn, sizeof(T));
          cur = cand;
          lambda = std::max(lambda / 10.0, kLambdaMin);
        } else {
          lambda *= 10.0;
          if (lambda > kLambdaMax) { term = GNDT_NDT_STALLED; break; }
        }
      }
    }
    memset(res, 0, sizeof(*res));
    memcpy(res->pose, T, sizeof(T));
    memcpy(res->center, cur.c, sizeof(cur.c));
    res->score = cur.score;
    memcpy(res->gradient, cur.g, sizeof(cur.g));
    memcpy(res->hessian, cur.H, sizeof(cur.H));
    res->n_points = cur.n_points;  // P2D: the finite points, as counted by the mean; D2D: usable scan Gaussians
    res->n_matched = cur.n_matched;
    res->n_pairs = cur.n_pairs;
    res->iterations = iters;
    res->termination = term;
    return GNDT_OK;
  };

  double T[16];
  memcpy(T, guess, sizeof(T));
  for (int i = 0; i < n_levels; ++i) {
    const gndt_ndt_level &l = levels[i];
    const gndt_handle::NdtLevel &L = h->ndt_lv[l.factor];
    const gndt_column *lc = (const gndt_column *)L.cols.p;
    gndt_registration r;
    if (d2d) {
      const gndt_handle::NdtLevel &SL = h->ndt_scan->ndt_lv[l.factor];
      rc = solve(l.factor, d2d_pass(SL.cov, SL.n_vox, (const NdtVoxel *)L.cov.p, lc, L.n_cols), l.max_iterations, l.translation_epsilon,
                 l.rotation_epsilon, T, &r);
    } else {
      rc = solve(l.factor, p2d((const NdtVoxel *)L.vox.p, lc, L.n_cols), l.max_iterations, l.translation_epsilon, l.rotation_epsilon, T, &r);
    }
    if (rc != GNDT_OK) return rc;
    memcpy(T, r.pose, sizeof(T));
    if (level_out) level_out[i] = r;
  }
  const gndt_column *mc = (const gndt_column *)h->columns.p;
  if (d2d)
    return solve(1, d2d_pass(h->ndt_scan->ndt_cov, h->ndt_scan->host_ctl.n_voxels, (const NdtVoxel *)map_vox.p, mc, n_cols),
                 np->max_iterations, np->translation_epsilon, np->rotation_epsilon, T, out);
  return solve(1, p2d((const NdtVoxel *)map_vox.p, mc, n_cols), np->max_iterations, np->translation_epsilon, np->rotation_epsilon, T, out);
}

}  // namespace

int gndt_register(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, const double guess[16],
                  const gndt_ndt_params *np, gndt_registration *out, void *stream) {
  return register_levels(h, xyz, n, stride_bytes, mem, guess, np, nullptr, 0, out, nullptr, stream, false);
}

void gndt_default_ndt_level(gndt_ndt_level *l, int32_t factor) {
  if (!l) return;
  memset(l, 0, sizeof(*l));
  l->factor = factor;
  l->max_iterations = 50;
  l->translation_epsilon = 1e-3;
  l->rotation_epsilon = 1e-3;
}

int gndt_register_levels(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, const double guess[16],
                         const gndt_ndt_params *np, const gndt_ndt_level *levels, int n_levels, gndt_registration *out,
                         gndt_registration *level_out, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!levels && n_levels > 0) { h->err = "gndt_register_levels: levels is NULL with n_levels > 0"; return GNDT_ERR_INVALID_ARG; }
  static const gndt_ndt_level kNone = {};
  return register_levels(h, xyz, n, stride_bytes, mem, guess, np, levels ? levels : &kNone, n_levels, out, level_out, stream, false);
}

int gndt_register_d2d(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem, const double guess[16],
                      const gndt_ndt_params *np, const gndt_ndt_level *levels, int n_levels, gndt_registration *out,
                      gndt_registration *level_out, void *stream) {
  if (!h) return GNDT_ERR_INVALID_ARG;
  if (!levels && n_levels > 0) { h->err = "gndt_register_d2d: levels is NULL with n_levels > 0"; return GNDT_ERR_INVALID_ARG; }
  static const gndt_ndt_level kNone = {};
  return register_levels(h, xyz, n, stride_bytes, mem, guess, np, levels ? levels : &kNone, n_levels, out, level_out, stream, true);
}

}  // extern "C"
