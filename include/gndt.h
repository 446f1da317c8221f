/*
 * gndt.h — C ABI of the B200-native grid-NDT map builder (libgndt.so).
 *
 * This is the drop-in boundary for the map-construction path of daysun/grid_ndt.
 * The reference has no FFI/plugin interface: the boundary there is a pair of
 * in-process C++ call sites and four public containers.  Every entry point below
 * cites the reference interface it replaces (paths relative to the reference
 * tree).  The host adapter that turns the tables returned here back into the
 * reference's `TwoDmap::map_cell / map_xy / morton_list` objects lives in
 * adapter/gndt_twodmap_adapter.h and is NOT part of this ABI.
 *
 * Conventions
 *   - plain C types only; no exceptions, no C++/torch types cross this boundary
 *   - every function returns a gndt_status (0 = ok, negative = error) unless noted
 *   - the caller owns all host buffers; the library owns all device memory
 *   - one handle is used from one thread at a time; all device work is ordered on
 *     the stream passed in (a cudaStream_t cast to void*, NULL = default stream)
 *   - there is no CPU fallback: without a CUDA device gndt_create fails with
 *     GNDT_ERR_CUDA
 */
#ifndef GNDT_H
#define GNDT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNDT_ABI_VERSION 2

typedef enum gndt_status {
  GNDT_OK = 0,
  GNDT_ERR_INVALID_ARG = -1,  /* NULL pointer, bad stride, bad enum, n == 0 ...            */
  GNDT_ERR_CUDA = -2,         /* a CUDA runtime call failed; see gndt_last_error            */
  GNDT_ERR_CAPACITY = -3,     /* caller buffer too small / n exceeds GNDT_MAX_POINTS        */
  GNDT_ERR_STATE = -4,        /* result queried before a successful gndt_build              */
  GNDT_ERR_INTERNAL = -5      /* device-side consistency check tripped (watchdog)           */
} gndt_status;

/* where a caller buffer lives */
typedef enum gndt_mem { GNDT_MEM_HOST = 0, GNDT_MEM_DEVICE = 1 } gndt_mem;

/* `demand` string of the reference (src/receiver.cpp:256, include/map2D.h:630,644) */
typedef enum gndt_demand { GNDT_DEMAND_SLOPE = 0, GNDT_DEMAND_TRUE = 1 } gndt_demand;

#define GNDT_MAX_POINTS ((size_t)1 << 30) /* 30-bit tile-prefix words in the radix partition */
#define GNDT_MAX_INDEX 32767              /* |nx|,|ny|,|nz| limit (Stopwatch.h:102-110 overflow) */

/*
 * Parameters.  Replaces: TwoDmap::TwoDmap(res,zres) + setLen/setZLen/setInterval
 * (include/map2D.h:487-501), the `demand` ROS param (src/receiver.cpp:256),
 * MINPOINTSIZE (include/map2D.h:28) and the RobotSphere thresholds
 * (include/robot.h:38-46).  Floats must be passed already rounded the way the
 * reference rounds them (ROS double param -> float).
 */
typedef struct gndt_params {
  float grid_len;              /* setLen            : x-y cell edge, metres                 */
  float z_len;                 /* setZLen           : z cell edge, metres                   */
  float slope_interval;        /* setInterval       : layer-split threshold on mean.z       */
  int32_t demand;              /* gndt_demand                                               */
  int32_t min_points;          /* MINPOINTSIZE = 3                                          */
  float rough_max;             /* RobotSphere::getRough()           = 100                   */
  float angle_max_deg;         /* RobotSphere::getAngle()           = 30                    */
  float reach_height;          /* RobotSphere::getReachableHeight() = 0.15f                 */
  int32_t origin_is_first_point; /* 1: origin = point 0 and point 0 is not binned
                                    (src/receiver.cpp:145,150); 0: use origin[] and bin all
                                    points (changeCallback loop, src/receiver.cpp:189)      */
  float origin[3];             /* setCloudFirst, used when origin_is_first_point == 0       */
  int32_t normalize_cov;       /* 0 = un-normalised scatter (pcl::computeCovarianceMatrix);
                                  1 = divide by n (computeCovarianceMatrixNormalized)       */
  int32_t tile_lo;             /* multi-GPU x strip: keep columns with tile_lo <= cx <      */
  int32_t tile_hi;             /*   tile_hi, cx = contiguous signed x index (sx>0?sx-1:sx). */
                               /*   tile_lo >= tile_hi disables the filter (single GPU).  An  */
                               /*   EMPTY strip is any range without a valid index, e.g.     */
                               /*   [GNDT_MAX_INDEX, GNDT_MAX_INDEX + 1).                     */
  uint64_t max_voxels;         /* capacity of the device voxel table; 0 = number of points  */
} gndt_params;

/* Fill *p with the reference defaults (receiver.cpp:33-35 + robot.h + map2D.h:28). */
void gndt_default_params(gndt_params *p);

/*
 * One occupied voxel = one OcNode of the reference (include/map2D.h:38-57) plus,
 * when it is a surface, its Slope (include/map2D.h:136-146).  Fixed 96 bytes.
 * Table order: ascending (cx, cy, cz) of the contiguous signed indices, i.e. all
 * voxels of one x-y column are adjacent and sorted bottom-to-top.
 */
typedef struct gndt_voxel {
  int32_t sx, sy, sz;      /* signed NON-ZERO cell indices (map2D.h:965-973); quadrant
                              letter = signs: A(+,+) B(+,-) C(-,+) D(-,-)                */
  uint32_t count;          /* points binned into the voxel (OcNode::N once >= min_points) */
  uint32_t first_index;    /* cloud index of the first point that fell into the voxel     */
  float mean[3];           /* OcNode::xyz_centroid; zeros when count < min_points         */
  float scatter[6];        /* xx,xy,xz,yy,yz,zz of OcNode::covariance_matrix              */
  float evals[3];          /* eigenvalues of the scatter, ascending                       */
  float normal[3];         /* unit eigenvector of evals[0] (sign arbitrary)               */
  float rough;             /* Slope::rough = evals[0], 0 -> 0.01 (map2D.h:131-132)        */
  uint32_t flags;          /* GNDT_F_*                                                    */
  uint32_t column;         /* index of the voxel's Cell in the column table               */
  uint32_t slope;          /* index of its Slope in the slope table, 0xFFFFFFFF if none   */
} gndt_voxel;

#define GNDT_F_FITTED 0x01u   /* count >= min_points: mean/scatter/eigen valid            */
#define GNDT_F_SLOPE 0x02u    /* a Slope object exists for this voxel (map2D.h:630-660)   */
#define GNDT_F_UP 0x04u       /* isSlope()'s `up`  (slope demand) / countUp() (true)      */
#define GNDT_F_DOWN 0x08u     /* isSlope()'s `down`                                       */
#define GNDT_F_REACH_L 0x10u  /* a reachable Slope exists in the left  neighbour cell     */
#define GNDT_F_REACH_R 0x20u  /*   "      right   (countLRFB/countReachable,              */
#define GNDT_F_REACH_F 0x40u  /*   "      forward  map2D.h:197-296)                       */
#define GNDT_F_REACH_B 0x80u  /*   "      back                                            */
#define GNDT_F_COLUMN_HEAD 0x100u /* first voxel of its x-y column (one Cell per column)  */

/* One Slope (include/map2D.h:136-146) — the compacted subset the planner reads. */
typedef struct gndt_slope {
  int32_t sx, sy, sz;      /* Slope::morton_xy (as signed indices) and Slope::morton_z    */
  float mean[3];           /* Slope::mean                                                 */
  float normal[3];         /* Slope::normal                                               */
  float rough;             /* Slope::rough                                                */
  uint32_t flags;          /* same bits as gndt_voxel::flags                              */
  uint32_t voxel;          /* index of the owning record in the voxel table               */
} gndt_slope;

/* One occupied x-y column = one Cell (include/map2D.h:181-187, created at :598-599). */
typedef struct gndt_column {
  int32_t sx, sy;          /* Cell::morton as signed indices                              */
  uint32_t first_index;    /* min first_index over its voxels = position in morton_list   */
  uint32_t voxel_begin;    /* first record of the column in the voxel table               */
  uint32_t voxel_count;    /* records in the column                                       */
  uint32_t slope_begin;    /* first Slope of the column in the slope table                */
  uint32_t slope_count;    /* Cell::map_slope.size()                                      */
  uint32_t reserved;
} gndt_column;

typedef struct gndt_counts_t {
  uint64_t n_input;        /* points handed to the last build/update                      */
  uint64_t n_binned;       /* points that landed in a voxel of this tile                  */
  uint64_t n_dropped;      /* non-finite or |index| > GNDT_MAX_INDEX (undefined in the
                              reference, Stopwatch.h:102-110) — counted, never binned     */
  uint64_t n_outside_tile; /* points of other GPUs' x strips                              */
  uint64_t n_columns;      /* morton_list.size()  (src/receiver.cpp:158)                  */
  uint64_t n_voxels;       /* OcNode count                                                */
  uint64_t n_fitted;       /* voxels with count >= min_points                             */
  uint64_t n_slopes;       /* slope_num (map2D.h:1226)                                    */
} gndt_counts_t;

/* device-timed stages of the last build, milliseconds (cudaEvent on the build stream) */
enum {
  GNDT_STAGE_KEY = 0,      /* bounds + first digit histogram (transMortonXYZ arithmetic)  */
  GNDT_STAGE_SORT = 1,     /* radix partition by (cx,cy,cz) (uniformDivision's binning)   */
  GNDT_STAGE_REDUCE = 2,   /* per-voxel moments + eigen (create2DMap fit)                 */
  GNDT_STAGE_LABEL = 3,    /* isSlope / countUp labels + column/slope tables              */
  GNDT_STAGE_EDGES = 4,    /* neighbour reachability bits (countReachable)                */
  GNDT_STAGE_TOTAL = 5,    /* whole build on the device                                   */
  GNDT_STAGE_H2D = 6,      /* host->device copy of the cloud when mem == GNDT_MEM_HOST    */
  GNDT_N_STAGES = 8
};

typedef struct gndt_handle gndt_handle;

/* library / ABI version string, never NULL */
const char *gndt_version(void);
/* last error text of this handle (or of the failed gndt_create when h == NULL) */
const char *gndt_last_error(const gndt_handle *h);

/*
 * Create a builder bound to CUDA device `device`.
 * Replaces: the global `daysun::TwoDmap map2D(0.5,0.1)` + setters
 * (src/receiver.cpp:35,267-269).
 */
int gndt_create(const gndt_params *params, int device, gndt_handle **out);
int gndt_destroy(gndt_handle *h);
/* change parameters between builds (setLen/setZLen/setInterval, map2D.h:493-501) */
int gndt_set_params(gndt_handle *h, const gndt_params *params);

/*
 * Build the map from one cloud.  `xyz` points at n records of `stride_bytes`
 * bytes each whose first 12 bytes are little-endian float x,y,z (pcl::PointXYZ /
 * the PointCloud2 payload: stride 16).  stride must be a multiple of 4, >= 12.
 * Replaces: chatterCallback's setCloudFirst + uniformDivision loop + create2DMap
 * (src/receiver.cpp:145-160; include/map2D.h:592-668).  Stream-ordered and
 * asynchronous for device input; result queries synchronise the stream.
 */
int gndt_build(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem,
               void *stream);

/*
 * The same build straight from a sensor_msgs/PointCloud2 message — what the receiver holds
 * when its callback fires (src/receiver.cpp:137-143: pcl_conversions::toPCL +
 * pcl::fromPCLPointCloud2 copy the message twice on the host before the division loop;
 * src/publisher.cpp:55 is where pcl::toROSMsg wrote it).  Fill the struct from the message:
 * data = msg.data.data(), width/height/point_step/is_bigendian as they are, *_offset = the
 * `offset` of the fields named "x", "y", "z" (datatype FLOAT32).  The usual layout
 * (little-endian, x y z side by side) is read in place on the device; any other layout is
 * repacked by one small kernel.  host_pinned = 0 (a std::vector<uint8_t> is pageable): the
 * upload runs through an internal ring of pinned chunks, the host copy of one chunk
 * overlapping the DMA of the previous one.
 */
typedef struct gndt_pointcloud2 {
  const void *data;
  uint32_t width, height, point_step;
  uint32_t x_offset, y_offset, z_offset;
  uint8_t is_bigendian;
  uint8_t host_pinned;   /* 1: data is page-locked (cudaHostAlloc / cudaHostRegister) */
  uint8_t reserved[2];
} gndt_pointcloud2;
int gndt_build_msg(gndt_handle *h, const gndt_pointcloud2 *msg, void *stream);

/*
 * Fuse one more scan into the resident map (origin and parameters of the
 * initial build are kept; every point of the scan is binned).
 * Replaces: changeCallback + change2DMap (src/receiver.cpp:179-212;
 * include/map2D.h:672-822) — dead code in the reference (its point lists are
 * never filled); contract here = the result equals one gndt_build over the
 * concatenation of all clouds seen so far.
 */
int gndt_update(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem,
                void *stream);

/*
 * Take a scan out of the resident map again: the inverse of gndt_update (Chan's update run
 * backwards on the binary64 moments; voxels that lose all their points disappear).
 * Replaces: delCallback + uniformDelDivision + del2DMap (src/receiver.cpp:95-134,214-248;
 * include/map2D.h:826-915), commented out at every call site in the reference.  Contract:
 * build(A) + update(B) + remove(B) equals build(A).  A remove gives its points' cloud indices
 * back (n_input and the index of the next update's first point both drop by n), so:
 *   - removing the most recent scan(s) restores the index space exactly: a later update(C)
 *     equals build(A ++ C), first_index and morton_list order included;
 *   - removing an older scan leaves first_index where it was for the voxels later scans
 *     touched first, and a later update may reuse those indices: renumbering them exactly
 *     would need per-point state the map does not keep.  Everything else (cells, counts,
 *     moments, labels under GNDT_DEMAND_TRUE) equals the batch build without that scan.
 * Every point of the scan must have been fused before: otherwise the call fails with
 * GNDT_ERR_STATE at the next result query and the map is left unchanged.
 */
int gndt_remove(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem,
                void *stream);

/*
 * The cells the last gndt_update / gndt_remove touched: indices into the (new) column table,
 * in the order in which the scan's points first touched them.
 * Replaces: changeMorton_list (src/receiver.cpp:47-56,187,196; include/map2D.h:505,674-676),
 * which the reference republishes alone (showInital(change_pub, ..., 1), receiver.cpp:203-206).
 * idx == NULL: size query.  A failed update / remove (GNDT_ERR_CAPACITY, GNDT_ERR_STATE) leaves
 * the resident map exactly as it was before the call.
 */
int gndt_changed_columns(gndt_handle *h, uint32_t *idx, size_t cap, int dst_mem, size_t *n_out);

/* counters the reference prints (receiver.cpp:144,158; map2D.h:1226) and friends */
int gndt_counts(gndt_handle *h, gndt_counts_t *out);

/* Copy result tables out.  cap = capacity of dst in records; returns GNDT_ERR_CAPACITY
 * when too small.  dst_mem says where dst lives.  *n_out (optional) = records written. */
int gndt_copy_voxels(gndt_handle *h, gndt_voxel *dst, size_t cap, int dst_mem, size_t *n_out);
int gndt_copy_slopes(gndt_handle *h, gndt_slope *dst, size_t cap, int dst_mem, size_t *n_out);
int gndt_copy_columns(gndt_handle *h, gndt_column *dst, size_t cap, int dst_mem, size_t *n_out);

/* Zero-copy device view of the voxel table (valid until the next build/update/destroy);
 * used by the multi-GPU tile gather.  Synchronises the build stream. */
int gndt_device_voxels(gndt_handle *h, const gndt_voxel **dptr, size_t *n);

/*
 * Thin-halo protocol for x strips (no host synchronisation, all stream-ordered):
 *   gndt_halo_pack  writes this strip's first and last x row into two caller buffers of
 *                   (1 + cap_records) gndt_voxel slots each (slot 0 is a header);
 *   the caller swaps them with the neighbour strips (rank-1 gets `first`, rank+1 `last`);
 *   gndt_halo_edges completes the forward/back reachability bits of this strip's boundary
 *                   rows from the neighbours' rows (NULL at the ends of the map).  A row
 *                   that did not fit raises GNDT_ERR_CAPACITY at the next result query.
 * After that the strip's records are final and can be all-gathered as they are;
 * gndt_apply_strip_offsets then turns the strip-local `column` / `slope` indices of the
 * gathered records into global ones (offsets = exclusive prefix sums over the strips).
 */
int gndt_halo_pack(gndt_handle *h, gndt_voxel *first_row_out, gndt_voxel *last_row_out, size_t cap_records,
                   void *stream);
int gndt_halo_edges(gndt_handle *h, const gndt_voxel *from_prev, const gndt_voxel *from_next, void *stream);
int gndt_apply_strip_offsets(gndt_handle *h, gndt_voxel *table, const uint64_t *offsets,
                             const uint32_t *col_offsets, const uint32_t *slope_offsets, int n_strips,
                             void *stream);
/* Stream-ordered (non-synchronising) access for collectives: device address of the voxel
 * count of the last build, and of the table with its capacity in records. */
int gndt_device_count_ptr(gndt_handle *h, const uint32_t **d_n_voxels); /* -> {n_voxels, n_columns, n_slopes, n_fitted} */
int gndt_device_table_ptr(gndt_handle *h, const gndt_voxel **dptr, size_t *capacity);

/*
 * The traversability graph as CSR: for Slope i, targets[offsets[i] .. offsets[i+1]) are the
 * indices (into the slope table) of the Slopes TwoDmap::AccessibleNeighbors returns for it
 * (include/map2D.h:530-548: countLRFB :197-263 + countReachable :266-296 + countAngle
 * :477-482), in the reference's order: left, right, forward, back cell, ascending z inside a
 * cell.  The GNDT_F_REACH_* bits only say that such a Slope exists; the cost-map expansion
 * (computeCost, :1285-1397) and A* (GlobalPlan.h:79-83) need the list, several layers per
 * neighbour cell.  slopes / columns: device tables to build from (e.g. the gathered tables of a
 * multi-GPU map), or both NULL for this handle's own map.  Synchronises the stream.
 * adapter/gndt_twodmap_adapter.h (SlopeGraph) serves the planner from it.
 */
int gndt_build_edges(gndt_handle *h, const gndt_slope *slopes, size_t n_slopes, const gndt_column *columns,
                     size_t n_columns, void *stream);
/* offsets: n_slopes + 1 entries, targets: n_targets entries.  offsets == targets == NULL: size query only. */
int gndt_copy_edges(gndt_handle *h, uint32_t *offsets, size_t cap_offsets, uint32_t *targets, size_t cap_targets,
                    int dst_mem, size_t *n_slopes, size_t *n_targets);

/*
 * Strip exchange through peer-mapped memory: the halo rows and the gather of the finished
 * tables without NCCL and without a host round trip (sizes stay on the device).  Every rank
 * (one handle per GPU; ranks may be threads of one process or separate processes) creates an
 * exchange buffer and exports it as a gndt_xchg_info blob; the caller moves the blobs between
 * ranks by any means (MPI, torch.distributed, a pipe) and hands all of them to
 * gndt_xchg_connect.  After each gndt_build / gndt_update of the strips, gndt_xchg_run
 * (stream-ordered, every rank calls it once per build) leaves on EVERY rank the tables of the
 * whole map, strips concatenated in rank order, indices global:
 *   - forward / back reach bits of strip-boundary rows completed from the neighbour strip
 *     (the countLRFB neighbours of include/map2D.h:219-253 that live on another GPU); empty
 *     strips are skipped, their neighbours exchange rows with each other
 *   - `what` selects the tables to gather: the planner reads Slopes and Cells
 *     (GNDT_X_SLOPES | GNDT_X_COLUMNS, 80 B per voxel instead of 176)
 * cap_records bounds the voxels of the WHOLE map, cap_halo_records those of one x row.
 */
#define GNDT_X_VOXELS 1
#define GNDT_X_SLOPES 2
#define GNDT_X_COLUMNS 4
#define GNDT_X_MAX_RANKS 16
typedef struct gndt_xchg_info {
  uint8_t ipc_mem[64];   /* cudaIpcMemHandle_t of the exchange buffer                   */
  uint64_t ptr;          /* its address in the exporting process (same-process peers)   */
  uint64_t bytes, cap_records, cap_halo;
  int32_t device, pid, what, rank;
  uint8_t reserved[16];
} gndt_xchg_info;
typedef struct gndt_xchg_view {
  const gndt_voxel *voxels;    /* device pointers into this rank's gathered tables (NULL if   */
  const gndt_slope *slopes;    /* not selected), valid until the next gndt_xchg_run           */
  const gndt_column *columns;
  uint64_t n_voxels, n_slopes, n_columns;
  int32_t world, reserved;
  uint64_t strip_voxels[GNDT_X_MAX_RANKS], strip_columns[GNDT_X_MAX_RANKS], strip_slopes[GNDT_X_MAX_RANKS];
} gndt_xchg_view;
int gndt_xchg_create(gndt_handle *h, int rank, int world, size_t cap_records, size_t cap_halo_records, int what,
                     gndt_xchg_info *mine);
int gndt_xchg_connect(gndt_handle *h, const gndt_xchg_info *all, int world);
int gndt_xchg_run(gndt_handle *h, void *stream);
/*
 * The same exchange with the bulk of the bytes carried by the copy engines instead of SM stores (the
 * build that runs beside an SM push on the sending GPU loses about as much time as the push takes;
 * copy-engine traffic does not disturb it: profiles/xchg_overlap_r2.md).  gndt_xchg_stage enqueues, on
 * `stream`, everything up to this strip sitting in the rank's own gathered tables (indices global)
 * and a 256-byte read-back of all strips' counts.  gndt_xchg_send blocks the HOST until that
 * read-back has landed (one round trip; enqueue the next builds first), then enqueues the peer
 * copies, the completion flags and the final wait, and makes `stream` wait for them.
 * gndt_xchg_counts_ready: 1 if gndt_xchg_send would not block, 0 if it would, < 0 on error.
 * gndt_xchg_view_get as after gndt_xchg_run.
 */
int gndt_xchg_stage(gndt_handle *h, void *stream);
int gndt_xchg_counts_ready(gndt_handle *h);
int gndt_xchg_send(gndt_handle *h, void *stream);
/* Synchronises the exchange stream; fails with GNDT_ERR_CAPACITY if the map outgrew
 * cap_records / a row outgrew cap_halo_records, GNDT_ERR_INTERNAL if a peer never showed up. */
int gndt_xchg_view_get(gndt_handle *h, gndt_xchg_view *out);

/*
 * One process, several GPUs: the form the reference's receiver (one C++ process, ros::spin,
 * src/receiver.cpp:283) would call.  gndt_multi_create makes one builder per device and
 * connects their exchange buffers; gndt_multi_build takes ONE cloud (host memory, or device
 * memory of devices[0]), plans balanced x strips, gives every GPU the cloud (host: each GPU's
 * own PCIe link; device: NVLink fan-out), builds the strips and runs the exchange, all
 * asynchronously on one private stream per device.  gndt_multi_view(index) then waits for it and
 * returns the tables of the WHOLE map as they lie on GPU `index` (any of them: all are equal).
 * gndt_multi_update fuses one more scan (every GPU keeps the points of its strip).
 * gndt_multi_handle gives the per-device builder (counts, stage times, strip-local tables).
 */
typedef struct gndt_multi gndt_multi;
int gndt_multi_create(const gndt_params *params, const int *devices, int ndev, size_t cap_records,
                      size_t cap_halo_records, int what, gndt_multi **out);
int gndt_multi_destroy(gndt_multi *m);
int gndt_multi_build(gndt_multi *m, const void *xyz, size_t n, size_t stride_bytes, int mem);
int gndt_multi_update(gndt_multi *m, const void *xyz, size_t n, size_t stride_bytes, int mem);
int gndt_multi_view(gndt_multi *m, int index, gndt_xchg_view *out);
int gndt_multi_cuts(gndt_multi *m, int32_t *cuts, int cap); /* ndev + 1 strip boundaries of the last build */
gndt_handle *gndt_multi_handle(gndt_multi *m, int index);
const char *gndt_multi_last_error(const gndt_multi *m);

/*
 * Balanced x strips for `ntiles` GPUs: cuts[0..ntiles] in contiguous signed x index
 * space such that strip t = [cuts[t], cuts[t+1]) holds ~n/ntiles points.  Every rank
 * that passes the same cloud gets the same cuts (no communication needed).
 */
int gndt_plan_tiles(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem,
                    int ntiles, int32_t *cuts, void *stream);

/* Stage events sit between the kernels of a build and keep each stage from overlapping the
 * launch of the next, so they are recorded only on request (default off): with on == 0
 * gndt_stage_ms reports GNDT_STAGE_TOTAL (+ H2D) and zeros for the individual stages.
 * Replaces: the stopwatch() pairs around "division" / "calculate" (src/receiver.cpp:148-162). */
int gndt_set_stage_timing(gndt_handle *h, int on);
int gndt_stage_ms(gndt_handle *h, float ms[GNDT_N_STAGES]);
/* number of kernel launches issued by the last build/update on this handle */
int gndt_launch_count(gndt_handle *h, uint64_t *n_launches);
/* The cell index needs one IEEE binary32 division per axis (map2D.h:965-967).  For the cell
 * lengths of this handle the library verifies on the device, for EVERY float in range, that
 * a division with the reciprocal refinement hoisted out rounds identically; *enabled says
 * whether that check passed (else the plain division is used), *values_checked how many
 * operands were compared.  GNDT_EXACT_DIV=1 in the environment forces the plain division. */
int gndt_fast_div_status(gndt_handle *h, int *enabled, uint64_t *values_checked);

/*
 * NDT scan-to-map registration (Biber & Strasser 2003; Magnusson 2009, ch. 6): the rigid pose
 * T (map <- scan) that maximises the NDT score of a scan against the normal distributions the
 * resident map keeps per voxel.  The usual streaming loop is register, transform, gndt_update.
 *
 * Contract of gndt_register:
 *   - Blocking: returns when the result is in *out.  Scans as for gndt_update (stride, host or
 *     device memory, same argument checks); every point is used, there is no strip filter.
 *   - A gndt_update / gndt_remove still awaiting its verdict is resolved first; if it failed,
 *     its status (GNDT_ERR_CAPACITY / GNDT_ERR_STATE) is returned and the next call registers
 *     against the unchanged map.
 *   - GNDT_ERR_STATE without a successful build.  GNDT_ERR_INVALID_ARG when guess, np or out is
 *     NULL, the guess is not finite, its bottom row is not exactly 0 0 0 1, max|R^T R - I| > 1e-6,
 *     or a parameter is out of range.
 *   - Nothing of the map changes: voxel / slope / column tables, counts, changed columns, key
 *     layout, stage times and gndt_launch_count stay as they were.  The call uses its own
 *     scratch and registers against the map with the parameters and origin it was built with
 *     (later gndt_set_params values do not apply).
 *
 * Objective.  For a finite scan point p (binary32) and pose (R, t): x' = R p + t in binary64,
 * each component ((R_i0 p0 + R_i1 p1) + R_i2 p2) + t_i with every operation rounded on its own
 * (no FMA).  The candidates of x' are the voxels of x' rounded to binary32 (cell as in binning,
 * resident origin and cell lengths; none when the index is out of range) whose column is the
 * point's own or one of its 4 edge neighbours (cx +-1 or cy +-1) and whose |cz_v - cz| <= 1, at
 * most 15, that are GNDT_F_FITTED, have count >= min_voxel_points and a usable Gaussian: mu =
 * mean, Sigma = scatter / (n - 1) (normalize_cov == 0) or scatter * n / (n - 1), eigenvalues
 * raised to >= 0.01 lambda_max (unusable if lambda_max <= 0), C = Sigma'^-1.  With V = grid_len^2
 * z_len, c1 = 10 (1 - p_o), c2 = p_o / V, d3 = -ln c2, d1 = -ln(c1 + c2) - d3,
 * d2 = -2 ln((-ln(c1 e^-1/2 + c2) - d3) / d1), d = x' - mu, every (point, voxel) pair adds
 * -d1 exp(-d2 d^T C d / 2) to the score S.  Gradient and Hessian are those of S over the
 * increment xi = (rho, phi) that maps x' to Exp(phi)(x' - c) + c + rho, at xi = 0, candidates
 * frozen; c = R pbar + t, pbar the binary64 mean of the finite points.  An accepted step
 * updates T <- (Exp(phi), c + rho - Exp(phi) c) o T.
 *
 * Solver: Levenberg-Marquardt on -S on the host, one pass over the scan on the device per
 * pose: (-H + lambda diag(max(-H_ii, 1e-6 max|H_ii|))) delta = g, lambda from 1e-3, / 10 on an
 * accepted step, * 10 on a rejected one or a failed Cholesky, STALLED above 1e12.  A step is
 * accepted only if S strictly rises; out->pose is the last accepted pose (the guess
 * when none was) and score / gradient / hessian / center / counts are those of that pose, so a
 * max_iterations = 0 call at out->pose reproduces them bit for bit.  Results are bitwise
 * repeatable for the same inputs on the same device.
 */
typedef struct gndt_ndt_params {
  float outlier_ratio;        /* Magnusson's p_o in (0, 1); default 0.55 (PCL's default)          */
  int32_t min_voxel_points;   /* voxels with fewer points are not used; default 6, must be >= 3   */
  int32_t max_iterations;     /* derivative passes after the first; 0 = evaluate the guess only   */
  int32_t reserved;           /* must be 0                                                        */
  double translation_epsilon; /* converged when the solved step moves less than this (m) ...      */
  double rotation_epsilon;    /* ... and rotates less than this (rad); |rho| and |phi| of the
                                 step; defaults 1e-4 m and 1e-4 rad, both finite and >= 0        */
} gndt_ndt_params;
void gndt_default_ndt_params(gndt_ndt_params *p);

enum { GNDT_NDT_CONVERGED = 0, GNDT_NDT_STALLED = 1, GNDT_NDT_MAX_ITER = 2, GNDT_NDT_NO_MATCH = 3 };

typedef struct gndt_registration {
  double pose[16];           /* row-major 4x4 map <- scan; the guess when nothing was accepted     */
  double center[3];          /* c of the objective at `pose`: R pbar + t                           */
  double score;              /* S, gradient and Hessian at `pose`                                  */
  double gradient[6];        /* order: rho_x, rho_y, rho_z, phi_x, phi_y, phi_z                     */
  double hessian[36];        /* row-major; -H^-1 is the usual pose covariance estimate              */
  uint64_t n_points;         /* finite points of the scan                                          */
  uint64_t n_matched;        /* points with at least one candidate voxel at `pose`                 */
  uint64_t n_pairs;          /* (point, voxel) pairs at `pose`                                     */
  uint32_t iterations;       /* derivative passes run after the first                              */
  int32_t termination;       /* GNDT_NDT_*: CONVERGED = the solved step at `pose` is below both
                                epsilons with damping lambda < 1 (lambda starts at 1e-3),
                                STALLED = no improving step before the damping limit, MAX_ITER,
                                NO_MATCH = no pair at the guess (pose = guess, S, g, H = 0)       */
} gndt_registration;

int gndt_register(gndt_handle *h, const void *xyz, size_t n, size_t stride_bytes, int mem,
                  const double guess[16], const gndt_ndt_params *np, gndt_registration *out,
                  void *stream);

/* ---- host-side key helpers (pure C, no device) ------------------------------------- */

/* TwoDmap::transMortonXYZ (include/map2D.h:950-976) for one position: signed non-zero
 * indices.  Returns 0, or GNDT_ERR_INVALID_ARG when the position is non-finite / out of
 * the +-GNDT_MAX_INDEX range. */
int gndt_trans_morton_xyz(const float origin[3], float grid_len, float z_len,
                          const float pos[3], int32_t *sx, int32_t *sy, int32_t *sz);
/* countMorton (include/Stopwatch.h:116-147): bits of nx to odd, ny to even positions. */
uint32_t gndt_count_morton(uint32_t nx, uint32_t ny);
/* mortonToXY (include/Stopwatch.h:171-189) */
void gndt_morton_to_xy(uint32_t morton, uint32_t *nx, uint32_t *ny);
/* The reference's string key: quadrant letter + decimal Morton, e.g. "A55".
 * buf must hold >= 16 chars.  Returns the string length. */
int gndt_morton_string(int32_t sx, int32_t sy, char *buf);
/* TwoDmap::countPositionXYZ (include/map2D.h:918-947): centre of cell (sx,sy,sz), metres. */
int gndt_cell_center(const float origin[3], float grid_len, float z_len, int32_t sx, int32_t sy,
                     int32_t sz, float center[3]);
/* Introspection: the sort-key layout the last build / update derived from the cloud's bounds:
 * out[0] = live partition passes (of the 6 launched), out[1] = bits of the column id field
 * ((cx - cx_min) * ny + (cy - cy_min)), out[2] = ny, out[3] = bits of the z field. */
int gndt_key_layout(gndt_handle *h, int out[4]);
/* Integer-keyed replacements for the planner's string lookups `map_cell.find(morton_xy)` /
 * `map_slope.find(morton_z)` (include/map2D.h:269-272,396-398; include/GlobalPlan.h:58-61) and
 * for the neighbour keys of countLRFB (include/map2D.h:197-263), on the caller's copies of the
 * column / slope tables: binary searches, no strings (SURVEY.md section 8(f) rank 2; inline
 * forms in include/gndt_lookup.h).  Return the table index or -1.  dir: 0 left, 1 right,
 * 2 forward, 3 back, as in GNDT_F_REACH_L/R/F/B. */
int64_t gndt_find_column(const gndt_column *cols, size_t n_cols, int32_t sx, int32_t sy);
int64_t gndt_find_slope(const gndt_column *cols, size_t n_cols, const gndt_slope *slopes, int32_t sx, int32_t sy,
                        int32_t sz);
int64_t gndt_neighbor_column(const gndt_column *cols, size_t n_cols, int32_t sx, int32_t sy, int dir);
/* The map origin in use (TwoDmap::cloudFirst, map2D.h:193,490-492): point 0 of the initial
 * cloud when origin_is_first_point, else params.origin. */
int gndt_origin(gndt_handle *h, float origin[3]);

#ifdef __cplusplus
}
#endif
#endif /* GNDT_H */
