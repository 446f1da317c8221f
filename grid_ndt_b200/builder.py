"""Host-side mirror of the reference's map-construction interface, above the C ABI.

`TwoDmap` keeps the names and argument meaning of daysun::TwoDmap for this path
(include/map2D.h:485-507: setLen/setZLen/setInterval/setCloudFirst/getGridLen/...,
create2DMap(demand), change2DMap(), transMortonXYZ, the public containers morton_list /
map_cell / map_xy) and of the receiver's hot loops (src/receiver.cpp:145-162).  All compute
happens in libgndt.so on the GPU; this file only marshals buffers and builds views.
"""
import ctypes as C
from typing import Optional

import numpy as np

from . import _abi
from ._abi import COLUMN_DTYPE, SLOPE_DTYPE, VOXEL_DTYPE, Counts, Params, default_params
from ._lib import GndtError, lib

try:  # torch is only plumbing here: device memory + streams + distributed
    import torch
except Exception:  # pragma: no cover
    torch = None


def _check(h, rc):
    if rc != 0:
        msg = lib().gndt_last_error(h)
        raise GndtError(rc, msg.decode() if msg else "")


def morton_string(sx: int, sy: int) -> str:
    """Quadrant letter + decimal Morton code, the reference's cell key
    (include/map2D.h:971-972, include/Stopwatch.h:116-147)."""
    buf = C.create_string_buffer(16)
    lib().gndt_morton_string(int(sx), int(sy), buf)
    return buf.value.decode()


def morton_strings(sx: np.ndarray, sy: np.ndarray) -> np.ndarray:
    """Vectorised morton_string for arrays of signed indices."""
    ax, ay = np.abs(sx).astype(np.uint64), np.abs(sy).astype(np.uint64)
    m = np.zeros(ax.shape, np.uint64)
    for k in range(16):
        m |= ((ax >> np.uint64(k)) & np.uint64(1)) << np.uint64(2 * k + 1)
        m |= ((ay >> np.uint64(k)) & np.uint64(1)) << np.uint64(2 * k)
    q = np.where(sx > 0, np.where(sy > 0, "A", "B"), np.where(sy > 0, "C", "D"))
    return np.char.add(q, m.astype(np.int64).astype(str))


class Slope:
    """View of one gndt_slope record with the reference's field names (map2D.h:136-146)."""

    __slots__ = ("normal", "rough", "mean", "h", "g", "f", "morton_xy", "morton_z", "up", "down", "father", "flags")

    def __init__(self, rec, key):
        self.normal = np.array(rec["normal"])
        self.rough = float(rec["rough"])
        self.mean = np.array(rec["mean"])
        self.h = self.g = self.f = np.finfo(np.float32).max  # FLT_MAX (map2D.h:637)
        self.morton_xy = key
        self.morton_z = int(rec["sz"])
        self.flags = int(rec["flags"])
        # slope demand: never assigned (map2D.h:636) and never set on a Slope; true demand: the
        # value the lazy Slope::countUp would store (map2D.h:275)
        self.up = bool(self.flags & _abi.F_UP)
        self.down = bool(self.flags & _abi.F_DOWN)
        self.father = None


class Cell:
    """map2D.h:181-187."""

    def __init__(self, morton):
        self._morton = morton
        self.map_slope = {}

    def getMorton(self):
        return self._morton


class TwoDmap:
    """GPU-backed drop-in for daysun::TwoDmap's construction path."""

    def __init__(self, res: float = 0.5, zres: float = 0.1, device: Optional[int] = None):
        self._p = default_params(res, zres)
        self._device = device if device is not None else (torch.cuda.current_device() if torch is not None and torch.cuda.is_available() else 0)
        self._h = C.c_void_p()
        rc = lib().gndt_create(C.byref(self._p), int(self._device), C.byref(self._h))
        if rc != 0:
            raise GndtError(rc, lib().gndt_last_error(None).decode())
        self._cloud = None
        self._keep = None
        self._tables = {}
        self._views = {}

    # ---- parameter setters / getters (map2D.h:487-501) ----------------------------------
    def setLen(self, v): self._p.grid_len = np.float32(v)
    def setZLen(self, v): self._p.z_len = np.float32(v)
    def setInterval(self, v): self._p.slope_interval = np.float32(v)
    def getGridLen(self): return float(self._p.grid_len)
    def getZLen(self): return float(self._p.z_len)
    def getInterval(self): return float(self._p.slope_interval)

    def setCloudFirst(self, p):
        """Explicit origin (map2D.h:490-492).  chatterCallback() uses points[0] instead."""
        self._p.origin_is_first_point = 0
        for i in range(3):
            self._p.origin[i] = np.float32(p[i])

    def setTile(self, lo: int, hi: int):
        """Multi-GPU x strip [lo, hi) in contiguous signed column index; lo >= hi disables."""
        self._p.tile_lo, self._p.tile_hi = int(lo), int(hi)

    @property
    def params(self) -> Params:
        return self._p

    # ---- the hot path --------------------------------------------------------------------
    def _marshal(self, cloud):
        if torch is not None and isinstance(cloud, torch.Tensor):
            if cloud.dtype != torch.float32 or cloud.dim() != 2 or cloud.shape[1] < 3 or not cloud.is_contiguous():
                raise GndtError(-1, "cloud tensor must be contiguous float32 [n, >=3]")
            mem = _abi.GNDT_MEM_DEVICE if cloud.is_cuda else _abi.GNDT_MEM_HOST
            stream = torch.cuda.current_stream(cloud.device).cuda_stream if cloud.is_cuda else 0
            return cloud.data_ptr(), cloud.shape[0], cloud.shape[1] * 4, mem, stream, cloud
        arr = np.ascontiguousarray(cloud, dtype=np.float32)
        if arr.ndim != 2 or arr.shape[1] < 3:
            raise GndtError(-1, "cloud must be float32 [n, >=3]")
        return arr.ctypes.data, arr.shape[0], arr.shape[1] * 4, _abi.GNDT_MEM_HOST, 0, arr

    def uniformDivision(self, cloud):
        """Stage the cloud to be binned: the batched form of the receiver's per-point loop
        (src/receiver.cpp:150-154).  Binning itself runs on the GPU in create2DMap()."""
        self._cloud = cloud

    def create2DMap(self, demand: str = "slope", stream: Optional[int] = None) -> bool:
        """Bin + fit + label the staged cloud (map2D.h:592-668).  Returns True like the
        reference; any other demand string yields no Slopes there and is rejected here."""
        if self._cloud is None:
            raise GndtError(-4, "create2DMap: no cloud staged (call uniformDivision first)")
        if demand not in ("slope", "true"):
            raise GndtError(-1, f"unknown demand {demand!r} (the reference builds no Slopes for it)")
        self._p.demand = _abi.GNDT_DEMAND_SLOPE if demand == "slope" else _abi.GNDT_DEMAND_TRUE
        ptr, n, stride, mem, st, keep = self._marshal(self._cloud)
        if stream is not None:
            st = stream
        L = lib()
        _check(self._h, L.gndt_set_params(self._h, C.byref(self._p)))
        _check(self._h, L.gndt_build(self._h, ptr, n, stride, mem, st))
        self._keep = keep  # device input must outlive the asynchronous build
        self._tables.clear()
        self._views.clear()
        return True

    def chatterCallback(self, cloud, demand: str = "slope") -> bool:
        """setCloudFirst(points[0]) + division loop from i=1 + create2DMap
        (src/receiver.cpp:145-160)."""
        self._p.origin_is_first_point = 1
        self.uniformDivision(cloud)
        return self.create2DMap(demand)

    def chatterCallbackMsg(self, data, width: int, height: int, point_step: int, offsets=(0, 4, 8), is_bigendian: bool = False,
                           demand: str = "slope", stream: int = 0) -> bool:
        """chatterCallback straight from a sensor_msgs/PointCloud2 payload (src/receiver.cpp:137-160):
        `data` = the message's byte buffer (bytes / bytearray / uint8 numpy or torch CPU tensor; a pinned
        torch tensor is uploaded directly, anything else through the library's pinned ring)."""
        if demand not in ("slope", "true"):
            raise GndtError(-1, f"unknown demand {demand!r}")
        self._p.origin_is_first_point = 1
        self._p.demand = _abi.GNDT_DEMAND_SLOPE if demand == "slope" else _abi.GNDT_DEMAND_TRUE
        pinned = False
        if torch is not None and isinstance(data, torch.Tensor):
            pinned, ptr, keep = data.is_pinned(), data.data_ptr(), data
        else:
            keep = np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data).view(np.uint8)
            ptr = keep.ctypes.data
        msg = _abi.PointCloud2(ptr, width, height, point_step, offsets[0], offsets[1], offsets[2], 1 if is_bigendian else 0, 1 if pinned else 0)
        L = lib()
        _check(self._h, L.gndt_set_params(self._h, C.byref(self._p)))
        _check(self._h, L.gndt_build_msg(self._h, C.byref(msg), stream))
        self._keep = keep
        self._tables.clear()
        self._views.clear()
        return True

    def change2DMap(self, scan, stream: Optional[int] = None) -> bool:
        """Fuse one more scan into the resident map (map2D.h:672-822 / receiver.cpp:179-212)."""
        ptr, n, stride, mem, st, keep = self._marshal(scan)
        if stream is not None:
            st = stream
        _check(self._h, lib().gndt_update(self._h, ptr, n, stride, mem, st))
        self._keep = keep
        self._tables.clear()
        self._views.clear()
        return True

    def del2DMap(self, scan, stream: Optional[int] = None) -> bool:
        """Take a scan out of the resident map again (map2D.h:826-915 / receiver.cpp:214-248)."""
        ptr, n, stride, mem, st, keep = self._marshal(scan)
        if stream is not None:
            st = stream
        _check(self._h, lib().gndt_remove(self._h, ptr, n, stride, mem, st))
        self._keep = keep
        self._tables.clear()
        self._views.clear()
        return True

    def register(self, scan, guess=None, stream: Optional[int] = None, levels=None, method: str = "p2d", **ndt) -> dict:
        """NDT registration of a scan against the resident map (gndt_register): the pose
        map <- scan that best fits it, from `guess` (4x4, identity when None).  Keywords set
        gndt_ndt_params fields (outlier_ratio, min_voxel_points, max_iterations,
        translation_epsilon, rotation_epsilon).  Returns the gndt_registration fields as a dict;
        pose is a 4x4 float64 array, termination one of _abi.NDT_*.  The map is not changed.

        levels: coarse-to-fine registration (gndt_register_levels) when not None: a sequence of
        factors, coarsest first, or of dicts with "factor" and any gndt_ndt_level field
        (max_iterations, translation_epsilon, rotation_epsilon); the other fields keep their
        defaults.  The result then has "levels": one dict per level, in the same shape.

        method: "p2d" registers the scan's points; "d2d" registers the scan's own per-cell Gaussians
        (gndt_register_d2d, with or without levels), and the result has the same shape."""
        if method not in ("p2d", "d2d"):
            raise GndtError(-1, f"unknown registration method {method!r} (p2d or d2d)")
        ptr, n, stride, mem, st, keep = self._marshal(scan)
        if stream is not None:
            st = stream
        T = np.eye(4) if guess is None else np.ascontiguousarray(guess, dtype=np.float64)
        if T.shape != (4, 4):
            raise GndtError(-1, "guess must be a 4x4 matrix")
        np_ = _abi.default_ndt_params(**ndt)
        out = _abi.Registration()
        Tp = T.ctypes.data_as(C.POINTER(C.c_double))
        if levels is None and method == "p2d":
            _check(self._h, lib().gndt_register(self._h, ptr, n, stride, mem, Tp, C.byref(np_), C.byref(out), st))
            return out.as_dict()
        lv = [_abi.default_ndt_level(**l) if isinstance(l, dict) else _abi.default_ndt_level(l) for l in levels or ()]
        arr = (_abi.NdtLevel * max(len(lv), 1))(*lv)
        per = (_abi.Registration * max(len(lv), 1))()
        fn = lib().gndt_register_d2d if method == "d2d" else lib().gndt_register_levels
        _check(self._h, fn(self._h, ptr, n, stride, mem, Tp, C.byref(np_), arr, len(lv), C.byref(out), per, st))
        res = out.as_dict()
        if levels is not None:
            res["levels"] = [per[i].as_dict() for i in range(len(lv))]
        return res

    @property
    def changed_columns(self) -> np.ndarray:
        """Indices (into `columns`) of the cells the last change2DMap / del2DMap touched, in
        first-touched order: the reference's changeMorton_list (receiver.cpp:47-56)."""
        n = C.c_size_t()
        _check(self._h, lib().gndt_changed_columns(self._h, None, 0, _abi.GNDT_MEM_HOST, C.byref(n)))
        out = np.zeros(max(n.value, 1), np.uint32)
        _check(self._h, lib().gndt_changed_columns(self._h, out.ctypes.data, len(out), _abi.GNDT_MEM_HOST, C.byref(n)))
        return out[: n.value]

    @property
    def changeMorton_list(self):
        """xy keys of the cells the last scan touched, first-touched order (receiver.cpp:47-56)."""
        cols = self.columns[self.changed_columns]
        return list(morton_strings(cols["sx"], cols["sy"]))

    # ---- results -------------------------------------------------------------------------
    def counts(self) -> dict:
        c = Counts()
        _check(self._h, lib().gndt_counts(self._h, C.byref(c)))
        return c.as_dict()

    def _result_buffer(self, name, dtype, n):
        """Host destination for a result table.  With pinned_results the buffers are
        page-locked (and reused across builds), so the device->host copy runs at PCIe speed."""
        if not getattr(self, "_pinned", False) or torch is None:
            return np.zeros(max(n, 1), dtype)
        need = max(n, 1) * dtype.itemsize
        buf = self._pinned_bufs.get(name)
        if buf is None or buf.numel() < need:
            buf = torch.empty(int(need * 1.25) + 4096, dtype=torch.uint8, pin_memory=True)
            self._pinned_bufs[name] = buf
        return buf.numpy()[:need].view(dtype)

    def pin_results(self, on: bool = True):
        self._pinned = bool(on)
        self._pinned_bufs = getattr(self, "_pinned_bufs", {})
        return self

    def _table(self, name, fn, dtype, n):
        if name not in self._tables:
            out = self._result_buffer(name, dtype, n)
            got = C.c_size_t()
            _check(self._h, fn(self._h, out.ctypes.data, n, _abi.GNDT_MEM_HOST, C.byref(got)))
            self._tables[name] = out[: got.value]
        return self._tables[name]

    @property
    def voxels(self) -> np.ndarray:
        return self._table("voxels", lib().gndt_copy_voxels, VOXEL_DTYPE, self.counts()["n_voxels"])

    @property
    def slopes(self) -> np.ndarray:
        return self._table("slopes", lib().gndt_copy_slopes, SLOPE_DTYPE, self.counts()["n_slopes"])

    @property
    def columns(self) -> np.ndarray:
        return self._table("columns", lib().gndt_copy_columns, COLUMN_DTYPE, self.counts()["n_columns"])

    def device_voxels(self):
        """(device pointer, n) of the resident voxel table (zero copy)."""
        p, n = C.c_void_p(), C.c_size_t()
        _check(self._h, lib().gndt_device_voxels(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def edges(self, slopes_ptr: int = 0, n_slopes: int = 0, columns_ptr: int = 0, n_columns: int = 0):
        """(offsets[n_slopes + 1], targets) — the traversability graph as CSR: for Slope i the Slopes
        AccessibleNeighbors (map2D.h:530-548) returns, in the reference's order.  Built on the GPU
        from this map's tables, or from the device tables given (a gathered multi-GPU map)."""
        L = lib()
        _check(self._h, L.gndt_build_edges(self._h, slopes_ptr or None, n_slopes, columns_ptr or None, n_columns, 0))
        ns, nt = C.c_size_t(), C.c_size_t()
        _check(self._h, L.gndt_copy_edges(self._h, None, 0, None, 0, _abi.GNDT_MEM_HOST, C.byref(ns), C.byref(nt)))
        off, tgt = np.zeros(ns.value + 1, np.uint32), np.zeros(max(nt.value, 1), np.uint32)
        _check(self._h, L.gndt_copy_edges(self._h, off.ctypes.data, len(off), tgt.ctypes.data, len(tgt), _abi.GNDT_MEM_HOST, None, None))
        return off, tgt[: nt.value]

    def plan_tiles(self, cloud, ntiles: int) -> np.ndarray:
        ptr, n, stride, mem, st, keep = self._marshal(cloud)
        cuts = (C.c_int32 * (ntiles + 1))()
        L = lib()
        _check(self._h, L.gndt_set_params(self._h, C.byref(self._p)))
        _check(self._h, L.gndt_plan_tiles(self._h, ptr, n, stride, mem, ntiles, cuts, st))
        return np.array(cuts[:], np.int32)

    def stage_timing(self, on: bool = True):
        """Record per-stage CUDA events in the following builds (off by default: the events keep
        consecutive kernels from overlapping their launches)."""
        _check(self._h, lib().gndt_set_stage_timing(self._h, 1 if on else 0))
        return self

    def stage_ms(self) -> dict:
        ms = (C.c_float * _abi.N_STAGES)()
        _check(self._h, lib().gndt_stage_ms(self._h, ms))
        return {k: float(ms[i]) for i, k in enumerate(_abi.STAGE_NAMES) if k != "reserved"}

    def fast_div_status(self):
        """(enabled, values_checked): whether the hoisted index division passed its exhaustive
        on-device equality check against the IEEE division for this map's cell lengths."""
        en, n = C.c_int(), C.c_uint64()
        _check(self._h, lib().gndt_fast_div_status(self._h, C.byref(en), C.byref(n)))
        return bool(en.value), int(n.value)

    def key_layout(self) -> dict:
        """Sort-key layout of the last build (introspection): live partition passes, bits of the
        column id field, the column id's y radix (ny) and bits of the z field."""
        out = (C.c_int * 4)()
        _check(self._h, lib().gndt_key_layout(self._h, out))
        return {"passes": out[0], "bits_col": out[1], "ny": out[2], "bits_z": out[3]}

    def launch_count(self) -> int:
        n = C.c_uint64()
        _check(self._h, lib().gndt_launch_count(self._h, C.byref(n)))
        return int(n.value)

    def origin(self):
        """The map origin in use (TwoDmap::cloudFirst): point 0 of the initial cloud for
        chatterCallback builds, the setCloudFirst value otherwise."""
        o = (C.c_float * 3)()
        _check(self._h, lib().gndt_origin(self._h, o))
        return np.array(o[:], np.float32)

    def countPositionXYZ(self, sx: int, sy: int, sz: int):
        """Centre of a cell in metres (map2D.h:918-947)."""
        o = (C.c_float * 3)(*self.origin())
        c = (C.c_float * 3)()
        rc = lib().gndt_cell_center(o, self._p.grid_len, self._p.z_len, int(sx), int(sy), int(sz), c)
        if rc != 0:
            raise GndtError(rc, "cell indices are signed and non-zero")
        return np.array(c[:], np.float32)

    def transMortonXYZ(self, position, origin=None):
        """(morton_xy string, morton_z) of a position (map2D.h:950-976)."""
        o = origin if origin is not None else self.origin()
        oo = (C.c_float * 3)(*[np.float32(v) for v in o])
        pp = (C.c_float * 3)(*[np.float32(v) for v in position])
        sx, sy, sz = C.c_int32(), C.c_int32(), C.c_int32()
        rc = lib().gndt_trans_morton_xyz(oo, self._p.grid_len, self._p.z_len, pp, C.byref(sx), C.byref(sy), C.byref(sz))
        if rc != 0:
            raise GndtError(rc, "position outside the supported index range")
        return morton_string(sx.value, sy.value), sz.value

    # ---- integer-keyed lookups (what the planner does with strings; SURVEY §8(f) rank 2) ----
    def find_column(self, sx: int, sy: int) -> int:
        """Index of cell (sx, sy) in `columns`, -1 if empty: map_cell.find(morton_xy) of
        map2D.h:269-272 without building the key string."""
        c = self.columns
        return int(lib().gndt_find_column(c.ctypes.data, len(c), int(sx), int(sy)))

    def find_slope(self, sx: int, sy: int, sz: int) -> int:
        """Index into `slopes` of the Slope at layer sz of cell (sx, sy), -1 if none:
        map_cell[xy]->map_slope.find(z) (GlobalPlan.h:58-61)."""
        c, s = self.columns, self.slopes
        return int(lib().gndt_find_slope(c.ctypes.data, len(c), s.ctypes.data, int(sx), int(sy), int(sz)))

    def neighbor_column(self, sx: int, sy: int, direction: int) -> int:
        """Index of the left/right/forward/back (0..3) neighbour cell of countLRFB
        (map2D.h:197-263), -1 if that cell is empty."""
        c = self.columns
        return int(lib().gndt_neighbor_column(c.ctypes.data, len(c), int(sx), int(sy), int(direction)))

    # ---- the reference's public containers, rebuilt lazily on the host -------------------
    @property
    def morton_list(self):
        """xy keys in first-seen order (receiver.cpp:70): columns sorted by first_index."""
        if "morton_list" not in self._views:
            cols = self.columns
            order = np.argsort(cols["first_index"], kind="stable")
            self._views["morton_list"] = list(morton_strings(cols["sx"][order], cols["sy"][order]))
        return self._views["morton_list"]

    @property
    def map_cell(self):
        """dict key -> Cell with map_slope {z: Slope}; one Cell per occupied column, even
        with no Slope (map2D.h:598-599)."""
        if "map_cell" not in self._views:
            cols, sl = self.columns, self.slopes
            keys = morton_strings(cols["sx"], cols["sy"])
            cells = {}
            for c, key in zip(cols, keys):
                cell = Cell(str(key))
                for s in sl[c["slope_begin"]: c["slope_begin"] + c["slope_count"]]:
                    cell.map_slope[int(s["sz"])] = Slope(s, str(key))
                cells[str(key)] = cell
            self._views["map_cell"] = cells
        return self._views["map_cell"]

    def close(self):
        if self._h:
            lib().gndt_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
