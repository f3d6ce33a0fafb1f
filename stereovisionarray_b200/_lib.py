"""Loads stereovisionarray_b200/libsva_b200.so (the sm_100a CUDA library behind include/sva_c_api.h).

There is NO CPU fallback: a missing library raises, and sva_create() fails on a machine without a B200-class GPU."""
import ctypes as C
import os

from . import abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsva_b200.so")

# every symbol include/sva_c_api.h declares (checked by tests/test_abi.py against the header text)
EXPORTS = [
    "sva_create", "sva_destroy", "sva_last_error", "sva_api_version", "sva_set_stream", "sva_use_own_stream", "sva_synchronize", "sva_kernel_launches",
    "sva_debug_set_guard", "sva_debug_check_guards",
    "sva_camera_project", "sva_camera_inv_project", "sva_bresenham", "sva_get_camera_pairs", "sva_grid_pairs",
    "sva_abs_diff_u8", "sva_match_literal", "sva_shift_perspective_with_disparity", "sva_improve_with_disparity",
    "sva_resize_half_u8", "sva_yaml_write_matrix", "sva_yaml_read_matrix",
    "sva_shift_perspective2", "sva_points3d_to_depth_map", "sva_depth_map_to_points3d", "sva_get_groups", "sva_masked_mean_f64",
    "sva_disparity_to_depth", "sva_depth_from_array", "sva_stream_submit", "sva_stream_wait", "sva_stream_mark", "sva_stream_elapsed",
    "sva_frame_upload", "sva_frame_set_pair_range", "sva_frame_run", "sva_frame_time", "sva_frame_kernel_times", "sva_frame_time_detailed", "sva_timer_start", "sva_timer_stop", "sva_frame_set_debug",
    "sva_frame_download_ad", "sva_frame_download_cost", "sva_frame_download_raw_cost", "sva_frame_download_sgm",
    "sva_frame_download_disparity", "sva_frame_ad_device_ptr", "sva_frame_mark_ad_ready",
    "sva_frame_cost_device_ptr", "sva_frame_set_params", "sva_frame_sgm_directions", "sva_frame_wta_rows", "sva_frame_download_disparity_rows",
    "sva_frame_rows_begin", "sva_frame_sgm_rows",
    "sva_comm_get_unique_id", "sva_comm_init", "sva_comm_destroy", "sva_comm_barrier", "sva_frame_reduce_ad", "sva_depth_pair_sharded",
    "sva_rows_open", "sva_rows_export", "sva_rows_connect", "sva_rows_connect_comm", "sva_rows_connect_local", "sva_rows_block", "sva_rows_run", "sva_rows_run_phase", "sva_rows_run_part", "sva_get_stream",
    "sva_rows_download", "sva_rows_close", "sva_depth_rows_sharded",
    "sva_rows_stream_create", "sva_rows_stream_connect_comm", "sva_rows_stream_submit", "sva_rows_stream_flush", "sva_rows_stream_wait",
    "sva_rows_stream_destroy", "sva_depth_groups", "sva_fuse_maps", "sva_depth_groups_fused",
]

_lib = None


class SvaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("sva error %d: %s" % (code, msg))
        self.code = code


def _preload_nccl():
    """The library binds NCCL at run time (dlopen("libnccl.so.2"), csrc/sva_dist.cu).  A process that imports torch AFTERWARDS would find
    the system's NCCL already mapped under that SONAME instead of the newer copy torch is built against, and fail to import.  So the copy
    torch bundles (site-packages/nvidia/nccl/lib) is mapped first when it exists; without it the library falls back to the system's."""
    import sys
    for base in sys.path:
        cand = os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
            except OSError:
                pass
            return


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libsva_b200.so is not built (run `python -m stereovisionarray_b200.build` or __graft_entry__.build()); "
                              "there is no CPU fallback for the depth path")
        _preload_nccl()
        L = C.CDLL(LIB_PATH)
        L.sva_last_error.restype = C.c_char_p
        L.sva_last_error.argtypes = [C.c_void_p]
        L.sva_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.sva_rows_connect_local.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sva_rows_connect.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        for n in ("sva_rows_open", "sva_comm_init"):
            getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.sva_rows_stream_create.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
        L.sva_rows_stream_submit.argtypes = [C.c_void_p] * 7
        L.sva_rows_stream_wait.argtypes = [C.c_void_p, C.c_int64]
        for n in ("sva_rows_stream_connect_comm", "sva_rows_stream_flush", "sva_rows_stream_destroy"):
            getattr(L, n).argtypes = [C.c_void_p]
        L.sva_depth_groups.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
        L.sva_fuse_maps.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sva_depth_groups_fused.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                             C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        missing = [n for n in EXPORTS if not hasattr(L, n)]
        if missing:
            raise ImportError("libsva_b200.so does not export %s — rebuild it" % missing)
        for name in EXPORTS:
            if name != "sva_last_error":
                getattr(L, name).restype = C.c_int
        _lib = L
    return _lib


def check(ctx, rc):
    if rc < 0:
        msg = lib().sva_last_error(ctx).decode() if ctx else ""
        raise SvaError(rc, msg)
    return rc
