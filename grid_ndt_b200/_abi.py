"""ctypes / numpy mirror of include/gndt.h (record layouts, enums, params struct).

Kept in one place so that the product binding (grid_ndt_b200.builder) and the test-side
checker wrapper agree byte-for-byte with the C header.
"""
import ctypes as C

import numpy as np

GNDT_ABI_VERSION = 2
GNDT_OK, GNDT_ERR_INVALID_ARG, GNDT_ERR_CUDA, GNDT_ERR_CAPACITY, GNDT_ERR_STATE, GNDT_ERR_INTERNAL = 0, -1, -2, -3, -4, -5
GNDT_MEM_HOST, GNDT_MEM_DEVICE = 0, 1
GNDT_DEMAND_SLOPE, GNDT_DEMAND_TRUE = 0, 1
GNDT_MAX_INDEX = 32767
GNDT_MAX_POINTS = 1 << 30

F_FITTED, F_SLOPE, F_UP, F_DOWN = 0x01, 0x02, 0x04, 0x08
F_REACH_L, F_REACH_R, F_REACH_F, F_REACH_B = 0x10, 0x20, 0x40, 0x80
F_REACH_ALL = 0xF0
F_COLUMN_HEAD = 0x100

STAGE_NAMES = ("key", "sort", "reduce", "label", "edges", "total", "h2d", "reserved")
N_STAGES = 8


class Params(C.Structure):
    """gndt_params (include/gndt.h)."""

    _fields_ = [
        ("grid_len", C.c_float),
        ("z_len", C.c_float),
        ("slope_interval", C.c_float),
        ("demand", C.c_int32),
        ("min_points", C.c_int32),
        ("rough_max", C.c_float),
        ("angle_max_deg", C.c_float),
        ("reach_height", C.c_float),
        ("origin_is_first_point", C.c_int32),
        ("origin", C.c_float * 3),
        ("normalize_cov", C.c_int32),
        ("tile_lo", C.c_int32),
        ("tile_hi", C.c_int32),
        ("max_voxels", C.c_uint64),
    ]


def default_params(grid_len=0.5, z_len=0.1, slope_interval=0.08, demand="slope", **kw) -> Params:
    """Reference defaults: TwoDmap map2D(0.5,0.1) (src/receiver.cpp:35), MINPOINTSIZE 3
    (include/map2D.h:28), RobotSphere thresholds (include/robot.h:38-46).  Floats are
    rounded double->float exactly like the ROS param path does (receiver.cpp:260-269)."""
    p = Params()
    p.grid_len = np.float32(grid_len)
    p.z_len = np.float32(z_len)
    p.slope_interval = np.float32(slope_interval)
    p.demand = {"slope": GNDT_DEMAND_SLOPE, "true": GNDT_DEMAND_TRUE}[demand] if isinstance(demand, str) else int(demand)
    p.min_points = 3
    p.rough_max = 100.0
    p.angle_max_deg = 30.0
    p.reach_height = np.float32(0.15)
    p.origin_is_first_point = 1
    p.normalize_cov = 0
    p.tile_lo = 0
    p.tile_hi = 0
    p.max_voxels = 0
    for k, v in kw.items():
        if k == "origin":
            for i in range(3):
                p.origin[i] = np.float32(v[i])
        else:
            setattr(p, k, v)
    return p


VOXEL_DTYPE = np.dtype(
    [
        ("sx", "<i4"), ("sy", "<i4"), ("sz", "<i4"),
        ("count", "<u4"), ("first_index", "<u4"),
        ("mean", "<f4", (3,)), ("scatter", "<f4", (6,)), ("evals", "<f4", (3,)),
        ("normal", "<f4", (3,)), ("rough", "<f4"), ("flags", "<u4"), ("column", "<u4"), ("slope", "<u4"),
    ]
)
SLOPE_DTYPE = np.dtype(
    [
        ("sx", "<i4"), ("sy", "<i4"), ("sz", "<i4"),
        ("mean", "<f4", (3,)), ("normal", "<f4", (3,)), ("rough", "<f4"),
        ("flags", "<u4"), ("voxel", "<u4"),
    ]
)
COLUMN_DTYPE = np.dtype(
    [
        ("sx", "<i4"), ("sy", "<i4"), ("first_index", "<u4"),
        ("voxel_begin", "<u4"), ("voxel_count", "<u4"), ("slope_begin", "<u4"), ("slope_count", "<u4"),
        ("reserved", "<u4"),
    ]
)
assert VOXEL_DTYPE.itemsize == 96 and SLOPE_DTYPE.itemsize == 48 and COLUMN_DTYPE.itemsize == 32


class Counts(C.Structure):
    """gndt_counts_t (include/gndt.h)."""

    _fields_ = [(n, C.c_uint64) for n in (
        "n_input", "n_binned", "n_dropped", "n_outside_tile",
        "n_columns", "n_voxels", "n_fitted", "n_slopes")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


X_VOXELS, X_SLOPES, X_COLUMNS = 1, 2, 4
X_MAX_RANKS = 16
TILE_EMPTY = (GNDT_MAX_INDEX, GNDT_MAX_INDEX + 1)  # a strip range that holds no valid index


class XchgInfo(C.Structure):
    """gndt_xchg_info (include/gndt.h): what one rank exports to its peers, 128 bytes."""

    _fields_ = [("ipc_mem", C.c_uint8 * 64), ("ptr", C.c_uint64), ("bytes", C.c_uint64), ("cap_records", C.c_uint64),
                ("cap_halo", C.c_uint64), ("device", C.c_int32), ("pid", C.c_int32), ("what", C.c_int32), ("rank", C.c_int32),
                ("reserved", C.c_uint8 * 16)]


class XchgView(C.Structure):
    """gndt_xchg_view (include/gndt.h)."""

    _fields_ = [("voxels", C.c_void_p), ("slopes", C.c_void_p), ("columns", C.c_void_p),
                ("n_voxels", C.c_uint64), ("n_slopes", C.c_uint64), ("n_columns", C.c_uint64),
                ("world", C.c_int32), ("reserved", C.c_int32),
                ("strip_voxels", C.c_uint64 * X_MAX_RANKS), ("strip_columns", C.c_uint64 * X_MAX_RANKS),
                ("strip_slopes", C.c_uint64 * X_MAX_RANKS)]


assert C.sizeof(XchgInfo) == 128


class PointCloud2(C.Structure):
    """gndt_pointcloud2 (include/gndt.h): the fields of a sensor_msgs/PointCloud2 the path reads."""

    _fields_ = [("data", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("point_step", C.c_uint32),
                ("x_offset", C.c_uint32), ("y_offset", C.c_uint32), ("z_offset", C.c_uint32),
                ("is_bigendian", C.c_uint8), ("host_pinned", C.c_uint8), ("reserved", C.c_uint8 * 2)]


NDT_CONVERGED, NDT_STALLED, NDT_MAX_ITER, NDT_NO_MATCH = 0, 1, 2, 3
NDT_TERMINATION = ("converged", "stalled", "max_iter", "no_match")


class NdtParams(C.Structure):
    """gndt_ndt_params (include/gndt.h): settings of one gndt_register call."""

    _fields_ = [("outlier_ratio", C.c_float), ("min_voxel_points", C.c_int32), ("max_iterations", C.c_int32),
                ("reserved", C.c_int32), ("translation_epsilon", C.c_double), ("rotation_epsilon", C.c_double)]


def default_ndt_params(**kw) -> NdtParams:
    """gndt_default_ndt_params with any field overridden by keyword."""
    p = NdtParams(0.55, 6, 100, 0, 1e-4, 1e-4)
    for k, v in kw.items():
        if k not in dict(NdtParams._fields_):
            raise TypeError(f"unknown NDT parameter {k!r}")
        setattr(p, k, v)
    return p


class Registration(C.Structure):
    """gndt_registration (include/gndt.h): result of gndt_register."""

    _fields_ = [("pose", C.c_double * 16), ("center", C.c_double * 3), ("score", C.c_double), ("gradient", C.c_double * 6),
                ("hessian", C.c_double * 36), ("n_points", C.c_uint64), ("n_matched", C.c_uint64), ("n_pairs", C.c_uint64),
                ("iterations", C.c_uint32), ("termination", C.c_int32)]

    def as_dict(self):
        return {
            "pose": np.array(self.pose[:], np.float64).reshape(4, 4),
            "center": np.array(self.center[:], np.float64),
            "score": float(self.score),
            "gradient": np.array(self.gradient[:], np.float64),
            "hessian": np.array(self.hessian[:], np.float64).reshape(6, 6),
            "n_points": int(self.n_points), "n_matched": int(self.n_matched), "n_pairs": int(self.n_pairs),
            "iterations": int(self.iterations), "termination": int(self.termination),
        }
