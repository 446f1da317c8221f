"""Loader for libgndt.so (the C-ABI CUDA library).  There is no fallback: if the library is
missing or cannot be loaded this raises, it never routes to a CPU implementation."""
import ctypes as C
import os
import subprocess
import sys

from ._abi import Counts, NdtLevel, NdtParams, Params, PointCloud2, Registration, XchgInfo, XchgView

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
LIB_PATH = os.environ.get("GNDT_LIB") or os.path.join(HERE, "libgndt.so")  # GNDT_LIB: another build, for A/B runs
SOURCES = [os.path.join(HERE, "csrc", f) for f in (
    "gndt_api.cu", "gndt_device.cuh", "gndt_sort.cuh", "gndt_reduce.cuh", "gndt_label.cuh", "gndt_update.cuh",
    "gndt_exchange.cuh", "gndt_graph.cuh", "gndt_scan.cuh", "gndt_ndt.cuh")]
HEADER = os.path.join(REPO, "include", "gndt.h")
LOOKUP_HEADER = os.path.join(REPO, "include", "gndt_lookup.h")

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]


def build_library(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> grid_ndt_b200/libgndt.so (in-tree)."""
    deps = SOURCES + [HEADER, LOOKUP_HEADER]
    if not force and os.path.exists(LIB_PATH) and all(
            os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps if os.path.exists(d)):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", LIB_PATH, SOURCES[0], "-I" + os.path.join(REPO, "include")]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return LIB_PATH


class GndtError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"gndt status {status}: {msg}")
        self.status = status


_lib = None

# every symbol include/gndt.h declares: (name, restype, argtypes)
_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int
SYMBOLS = {
    "gndt_version": (C.c_char_p, []),
    "gndt_last_error": (C.c_char_p, [_vp]),
    "gndt_default_params": (None, [C.POINTER(Params)]),
    "gndt_create": (_i, [C.POINTER(Params), _i, C.POINTER(_vp)]),
    "gndt_destroy": (_i, [_vp]),
    "gndt_set_params": (_i, [_vp, C.POINTER(Params)]),
    "gndt_build": (_i, [_vp, _vp, _sz, _sz, _i, _vp]),
    "gndt_build_msg": (_i, [_vp, C.POINTER(PointCloud2), _vp]),
    "gndt_update": (_i, [_vp, _vp, _sz, _sz, _i, _vp]),
    "gndt_remove": (_i, [_vp, _vp, _sz, _sz, _i, _vp]),
    "gndt_changed_columns": (_i, [_vp, _vp, _sz, _i, C.POINTER(_sz)]),
    "gndt_counts": (_i, [_vp, C.POINTER(Counts)]),
    "gndt_copy_voxels": (_i, [_vp, _vp, _sz, _i, C.POINTER(_sz)]),
    "gndt_copy_slopes": (_i, [_vp, _vp, _sz, _i, C.POINTER(_sz)]),
    "gndt_copy_columns": (_i, [_vp, _vp, _sz, _i, C.POINTER(_sz)]),
    "gndt_device_voxels": (_i, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "gndt_halo_pack": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "gndt_halo_edges": (_i, [_vp, _vp, _vp, _vp]),
    "gndt_apply_strip_offsets": (_i, [_vp, _vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), _i, _vp]),
    "gndt_device_count_ptr": (_i, [_vp, C.POINTER(_vp)]),
    "gndt_device_table_ptr": (_i, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "gndt_build_edges": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "gndt_copy_edges": (_i, [_vp, _vp, _sz, _vp, _sz, _i, C.POINTER(_sz), C.POINTER(_sz)]),
    "gndt_xchg_create": (_i, [_vp, _i, _i, _sz, _sz, _i, C.POINTER(XchgInfo)]),
    "gndt_xchg_connect": (_i, [_vp, C.POINTER(XchgInfo), _i]),
    "gndt_xchg_run": (_i, [_vp, _vp]),
    "gndt_xchg_stage": (_i, [_vp, _vp]),
    "gndt_xchg_counts_ready": (_i, [_vp]),
    "gndt_xchg_send": (_i, [_vp, _vp]),
    "gndt_xchg_view_get": (_i, [_vp, C.POINTER(XchgView)]),
    "gndt_multi_create": (_i, [C.POINTER(Params), C.POINTER(C.c_int), _i, _sz, _sz, _i, C.POINTER(_vp)]),
    "gndt_multi_destroy": (_i, [_vp]),
    "gndt_multi_build": (_i, [_vp, _vp, _sz, _sz, _i]),
    "gndt_multi_update": (_i, [_vp, _vp, _sz, _sz, _i]),
    "gndt_multi_view": (_i, [_vp, _i, C.POINTER(XchgView)]),
    "gndt_multi_cuts": (_i, [_vp, C.POINTER(C.c_int32), _i]),
    "gndt_multi_handle": (_vp, [_vp, _i]),
    "gndt_multi_last_error": (C.c_char_p, [_vp]),
    "gndt_plan_tiles": (_i, [_vp, _vp, _sz, _sz, _i, _i, C.POINTER(C.c_int32), _vp]),
    "gndt_set_stage_timing": (_i, [_vp, _i]),
    "gndt_stage_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "gndt_launch_count": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "gndt_fast_div_status": (_i, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "gndt_trans_morton_xyz": (_i, [C.POINTER(C.c_float), C.c_float, C.c_float, C.POINTER(C.c_float),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "gndt_count_morton": (C.c_uint32, [C.c_uint32, C.c_uint32]),
    "gndt_morton_to_xy": (None, [C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "gndt_morton_string": (_i, [C.c_int32, C.c_int32, C.c_char_p]),
    "gndt_cell_center": (_i, [C.POINTER(C.c_float), C.c_float, C.c_float, C.c_int32, C.c_int32, C.c_int32,
                              C.POINTER(C.c_float)]),
    "gndt_origin": (_i, [_vp, C.POINTER(C.c_float)]),
    "gndt_default_ndt_params": (None, [C.POINTER(NdtParams)]),
    "gndt_register": (_i, [_vp, _vp, _sz, _sz, _i, C.POINTER(C.c_double), C.POINTER(NdtParams), C.POINTER(Registration), _vp]),
    "gndt_default_ndt_level": (None, [C.POINTER(NdtLevel), C.c_int32]),
    "gndt_register_levels": (_i, [_vp, _vp, _sz, _sz, _i, C.POINTER(C.c_double), C.POINTER(NdtParams), C.POINTER(NdtLevel), _i,
                                  C.POINTER(Registration), C.POINTER(Registration), _vp]),
    "gndt_register_d2d": (_i, [_vp, _vp, _sz, _sz, _i, C.POINTER(C.c_double), C.POINTER(NdtParams), C.POINTER(NdtLevel), _i,
                               C.POINTER(Registration), C.POINTER(Registration), _vp]),
    "gndt_key_layout": (_i, [_vp, C.POINTER(C.c_int)]),
    "gndt_find_column": (C.c_int64, [_vp, _sz, C.c_int32, C.c_int32]),
    "gndt_find_slope": (C.c_int64, [_vp, _sz, _vp, C.c_int32, C.c_int32, C.c_int32]),
    "gndt_neighbor_column": (C.c_int64, [_vp, _sz, C.c_int32, C.c_int32, _i]),
}


def lib():
    """The loaded library with typed entry points.  Raises if it is not built/loadable."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GndtError(-2, f"{LIB_PATH} is not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the ABI is incomplete
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib
