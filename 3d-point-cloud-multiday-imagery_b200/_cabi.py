"""ctypes binding of ``libmdkm.so`` (the C ABI in ``include/mdkm.h``).

The library is built in-tree by ``build.py`` (``nvcc -gencode arch=compute_100a,code=sm_100a``).
There is no fallback: if the shared object is missing or no B200 is visible the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_ubyte, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmdkm.so")

MDKM_OK = 0
MEM_HOST, MEM_DEVICE = 0, 1
HM_F32, HM_I16, HM_F32_GTIFF3 = 0, 1, 2
POINTS_AOS, POINTS_SOA = 0, 1
OPT_SETTLE_GROUPS = 1
OPT_RASTER_MIRROR = 2
OPT_CELL_PX, OPT_CELL_ROWS = 3, 4
OPT_TWO_LEVEL = 5
OPT_DEPENDENT_LAUNCH = 6
PHASE_UNPROJECT, PHASE_BUILD, PHASE_STEP, PHASE_FINAL = 0, 1, 2, 3
NCCL_UNIQUE_ID_BYTES = 128
IPC_HANDLE_BYTES = 64

STATUS_NAMES = {
    0: "MDKM_OK",
    -1: "MDKM_ERR_INVALID",
    -2: "MDKM_ERR_CUDA",
    -3: "MDKM_ERR_NO_DEVICE",
    -4: "MDKM_ERR_STATE",
    -5: "MDKM_ERR_NCCL",
    -6: "MDKM_ERR_OOM",
}

STATUS_BY_NAME = {v: k for k, v in STATUS_NAMES.items()}

# name -> (restype, argtypes); mirrors include/mdkm.h one to one
SIGNATURES = {
    "mdkm_version": (c_char_p, []),
    "mdkm_create": (c_int, [POINTER(c_void_p), c_int, c_void_p]),
    "mdkm_destroy": (None, [c_void_p]),
    "mdkm_last_error": (c_char_p, [c_void_p]),
    "mdkm_comm_unique_id": (c_int, [POINTER(c_ubyte)]),
    "mdkm_comm_init": (c_int, [c_void_p, c_int, c_int, POINTER(c_ubyte)]),
    "mdkm_comm_p2p_handle": (c_int, [c_void_p, POINTER(c_ubyte)]),
    "mdkm_comm_p2p_open": (c_int, [c_void_p, POINTER(c_ubyte)]),
    "mdkm_comm_p2p_close": (c_int, [c_void_p]),
    "mdkm_comm_p2p_buffer": (c_int, [c_void_p, POINTER(c_void_p)]),
    "mdkm_comm_p2p_open_ptrs": (c_int, [c_void_p, POINTER(c_void_p)]),
    "mdkm_get_stream": (c_void_p, [c_void_p]),
    "mdkm_set_option": (c_int, [c_void_p, c_int, c_int64]),
    "mdkm_fit_worklist": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "mdkm_unproject": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_int, c_int, c_int,
                               c_int64, c_int64, c_float, c_int, c_int, POINTER(c_int64)]),
    "mdkm_bind_cloud_output": (c_int, [c_void_p, c_void_p, c_int64, c_int]),
    "mdkm_bind_cluster_map": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int]),
    "mdkm_bind_day_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int]),
    "mdkm_bind_day_transitions": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int]),
    "mdkm_bind_regions": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int]),
    "mdkm_region_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdkm_region_table": (c_int, [c_void_p, c_void_p, c_void_p, c_int64]),
    "mdkm_bind_region_overlaps": (c_int, [c_void_p, c_void_p, c_int]),
    "mdkm_region_overlap_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdkm_region_overlap_table": (c_int, [c_void_p, c_void_p, c_int64]),
    "mdkm_bind_tracks": (c_int, [c_void_p, c_double, c_void_p, c_int64, c_int]),
    "mdkm_track_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdkm_track_table": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64]),
    "mdkm_bind_region_adjacency": (c_int, [c_void_p, c_int]),
    "mdkm_region_adjacency_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdkm_region_adjacency_table": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64]),
    "mdkm_set_points": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int]),
    "mdkm_num_points": (c_int64, [c_void_p]),
    "mdkm_num_points_global": (c_int64, [c_void_p]),
    "mdkm_gather_points": (c_int, [c_void_p, POINTER(c_int64), c_int, POINTER(c_float)]),
    "mdkm_get_cloud": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "mdkm_get_cloud_async": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "mdkm_wait": (c_int, [c_void_p]),
    "mdkm_num_segments": (c_int, [c_void_p]),
    "mdkm_segment_offsets": (c_int, [c_void_p, POINTER(c_int64)]),
    "mdkm_ground_level": (c_int, [c_void_p, c_void_p, c_int, POINTER(c_double), POINTER(c_double)]),
    "mdkm_fit": (c_int, [c_void_p, c_int, POINTER(c_double), c_int, c_double, c_void_p, c_int,
                         POINTER(c_double), POINTER(c_int), POINTER(c_double)]),
    "mdkm_fit_stats": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_double)]),
    "mdkm_lloyd_step": (c_int, [c_void_p, c_int, POINTER(c_double), c_void_p, c_int, POINTER(c_double),
                                POINTER(c_int64)]),
    "mdkm_predict": (c_int, [c_void_p, c_int, POINTER(c_double), c_void_p, c_int, POINTER(c_double)]),
    "mdkm_kmeans_plusplus": (c_int, [c_void_p, c_int, c_int64, POINTER(c_double), c_int,
                                     POINTER(c_double), POINTER(c_int64)]),
    "mdkm_drop_caches": (c_int, [c_void_p]),
    "mdkm_profile_enable": (c_int, [c_void_p, c_int]),
    "mdkm_profile_read": (c_int, [c_void_p, POINTER(c_double), POINTER(c_int), POINTER(c_int)]),
    "mdkm_profile_phase": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_int64)]),
}

_lib = None


class MdkmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {msg}")
        self.code = code


def load(path: str | None = None) -> ctypes.CDLL:
    """dlopen libmdkm.so and attach the prototypes.  Raises if the library was not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("MDKM_LIB") or LIB_PATH  # MDKM_LIB: an instrumented build (tools/)
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc; there is no CPU fallback)"
        )
    lib = ctypes.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib
