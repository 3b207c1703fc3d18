"""ctypes binding of libwrgpu.so (include/wr_gpu.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, this module raises.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libwrgpu.so")
CSRC = os.path.join(_HERE, "csrc")

WR_OK = 0
STATUS = {0: "WR_OK", -1: "WR_ERR_INVALID", -2: "WR_ERR_CUDA", -3: "WR_ERR_NOMEM", -4: "WR_ERR_STATE",
          -5: "WR_ERR_NOTFOUND", -6: "WR_ERR_CAPACITY", -7: "WR_ERR_FORMAT"}
WR_ERR_NOTFOUND = -5
UPDATE_FUSED, UPDATE_SPLIT, UPDATE_ATOMIC, UPDATE_RANKSET = 0, 1, 2, 4


class WrError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("%s: %s" % (STATUS.get(status, status), msg))
        self.status = status


class AcsParams(C.Structure):
    """wr_acs_params (include/wr_gpu.h); defaults are the literals of ACSRank_3D.hpp:319-325."""
    _fields_ = [("alpha", C.c_int), ("beta", C.c_float), ("rho", C.c_float), ("tau0", C.c_float),
                ("fixed_colony", C.c_int), ("step_cap", C.c_int), ("K", C.c_int), ("seed", C.c_uint64),
                ("update_mode", C.c_int), ("walk_table_log2", C.c_int)]


# every symbol include/wr_gpu.h declares (tests check the library exports exactly these)
SYMBOLS = """wr_last_error wr_version wr_device_count wr_set_device wr_release_caches wr_stl_parse
wr_grid_create_from_triangles wr_grid_create_from_occupancy wr_grid_destroy wr_grid_dims wr_grid_precision
wr_grid_bbox wr_grid_coords wr_grid_download_bits wr_grid_download_isfree wr_grid_stats
wr_grid_clearance wr_grid_clearance_at wr_grid_inflate wr_grid_clearance_ms wr_grid_shortcut_paths
wr_acs_default_params wr_acs_create wr_acs_destroy wr_acs_set_points wr_acs_set_endpoints wr_acs_snap_points wr_acs_search_pairs wr_acs_search_batch wr_acs_result_path wr_acs_batch_stats wr_acs_begin wr_acs_set_next_search
wr_acs_iterate wr_acs_sync wr_acs_reset wr_acs_best wr_acs_download_pheromone wr_acs_upload_pheromone
wr_acs_last_colony wr_acs_last_ant wr_acs_counters wr_acs_kernel_ms wr_acs_update_stats wr_acs_group_stats wr_acs_walk_stats wr_acs_field_stats wr_acs_field_lines wr_acs_stream_kernel_ms wr_acs_set_timing wr_acs_bench_kernel wr_acs_set_stream
wr_comm_unique_id wr_acs_comm_init wr_acs_set_shard wr_acs_peer_export wr_acs_peer_import wr_acs_peer_set_pointers
wr_gtsp_create wr_gtsp_destroy wr_gtsp_iterate wr_gtsp_solve wr_gtsp_sync wr_gtsp_best wr_gtsp_download_pheromone wr_gtsp_tau0
wr_gtsp_kernel_ms wr_bspline_eval""".split()


def build(verbose=False):
    """Compile libwrgpu.so for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libwrgpu.so failed:\n%s\n%s" % (r.stdout, r.stderr))


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("%s is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, f32, u64, i64 = C.c_void_p, C.c_int, C.c_float, C.c_uint64, C.c_int64
    L.wr_last_error.restype = C.c_char_p
    sig = {
        "wr_device_count": [vp], "wr_set_device": [i32], "wr_release_caches": [],
        "wr_stl_parse": [vp, C.c_size_t, vp, i32, vp],
        "wr_grid_create_from_triangles": [vp, i32, f32, i32, vp],
        "wr_grid_create_from_occupancy": [vp, i32, i32, i32, vp, vp, vp, f32, vp],
        "wr_grid_destroy": [vp], "wr_grid_dims": [vp, vp], "wr_grid_precision": [vp, vp, vp], "wr_grid_bbox": [vp, vp, vp],
        "wr_grid_coords": [vp, vp, vp, vp], "wr_grid_download_bits": [vp, vp, C.c_size_t],
        "wr_grid_download_isfree": [vp, vp, C.c_size_t], "wr_grid_stats": [vp, vp, vp, vp],
        "wr_grid_clearance": [vp, vp, C.c_size_t], "wr_grid_clearance_at": [vp, vp, i32, vp, vp],
        "wr_grid_inflate": [vp, C.c_uint32, vp], "wr_grid_clearance_ms": [vp, vp],
        "wr_grid_shortcut_paths": [vp, vp, vp, i32, C.c_uint32, i32, vp, vp, vp, vp],
        "wr_acs_default_params": [C.POINTER(AcsParams)], "wr_acs_create": [vp, C.POINTER(AcsParams), vp],
        "wr_acs_destroy": [vp], "wr_acs_set_points": [vp, vp, vp, vp], "wr_acs_set_endpoints": [vp, i64, i64],
        "wr_acs_snap_points": [vp, vp, i32, vp], "wr_acs_search_pairs": [vp, vp, vp, i32, f32, i32, vp, vp, vp, vp, i32],
        "wr_acs_search_batch": [vp, vp, vp, i32, f32, i32, vp, vp, vp, vp, i32], "wr_acs_result_path": [vp, i32, vp, vp, i32, vp, vp], "wr_acs_batch_stats": [vp, vp],
        "wr_acs_begin": [vp, f32], "wr_acs_set_next_search": [vp, C.c_uint32], "wr_acs_iterate": [vp, i32], "wr_acs_sync": [vp], "wr_acs_reset": [vp],
        "wr_acs_best": [vp, vp, vp, i32, vp, vp], "wr_acs_download_pheromone": [vp, vp, C.c_size_t],
        "wr_acs_upload_pheromone": [vp, vp, C.c_size_t], "wr_acs_last_colony": [vp, vp, vp, vp],
        "wr_acs_last_ant": [vp, i32, vp, vp, i32, vp, vp, vp], "wr_acs_counters": [vp, vp], "wr_acs_kernel_ms": [vp, vp], "wr_acs_update_stats": [vp, vp], "wr_acs_group_stats": [vp, vp], "wr_acs_walk_stats": [vp, vp], "wr_acs_field_stats": [vp, vp], "wr_acs_field_lines": [vp, vp], "wr_acs_stream_kernel_ms": [vp, vp, vp],
        "wr_acs_set_timing": [vp, i32], "wr_acs_bench_kernel": [vp, i32, i32, vp], "wr_acs_set_stream": [vp, vp], "wr_acs_set_shard": [vp, i32, i32],
        "wr_comm_unique_id": [vp], "wr_acs_comm_init": [vp, vp, i32, i32],
        "wr_acs_peer_export": [vp, vp, vp], "wr_acs_peer_import": [vp, vp], "wr_acs_peer_set_pointers": [vp, vp],
        "wr_gtsp_create": [vp, i32, i32, i32, i32, u64, vp], "wr_gtsp_destroy": [vp], "wr_gtsp_iterate": [vp, i32], "wr_gtsp_solve": [vp, i32, vp, vp, vp],
        "wr_gtsp_sync": [vp], "wr_gtsp_best": [vp, i32, vp, vp, vp], "wr_gtsp_download_pheromone": [vp, i32, vp],
        "wr_gtsp_tau0": [vp, vp], "wr_gtsp_kernel_ms": [vp, vp],
        "wr_bspline_eval": [i32, i32, i32, vp, vp, vp, i32, i32, f32, vp, i32, vp, vp, vp, vp],
    }
    for name, args in sig.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = C.c_int
    _lib = L
    return L


def check(status):
    if status != WR_OK:
        raise WrError(status, lib().wr_last_error().decode(errors="replace"))
    return status


def ptr(a):
    """numpy array -> void* (the array must stay alive for the duration of the call)."""
    return a.ctypes.data_as(C.c_void_p)
