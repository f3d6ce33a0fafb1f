"""Drop-in check: adapter/sva_functions.cpp (the reference-side binding, compiled against the reference's headers, or the stand-ins in
adapter/refshim when no reference tree is given) driven like
the reference's main() — getCameraPairs / Camera / improveWithDisparity / getAbsDiff under their reference names, the loop nest as
one svaMatchLiteral call — must reproduce what the reference's main() produced (tests/golden/main_*.npz)."""
import ctypes as C
import os

import numpy as np
import pytest

from stereovisionarray_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "adapter", "_build", "libsva_adapter_test.so")


def test_adapter_reproduces_reference_driver():
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    for name in ("main_120x160_s7", "main_100x176_s9"):
        g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        h, w, seed = int(g["h"]), int(g["w"]), int(g["seed"])
        sc = synth.make_literal_scene(h, w, seed)
        imgs = [np.ascontiguousarray(i) for i in sc["images"]]
        ptrs = (C.c_void_p * 25)(*[i.ctypes.data for i in imgs])
        mask = np.ascontiguousarray(g["mask"])
        disp = np.zeros((h, w), np.uint8); imp = np.zeros((h, w), np.uint8); sad = C.c_double()
        rc = lib.adapter_driver(ptrs, w, h, mask.ctypes.data_as(C.c_void_p), disp.ctypes.data_as(C.c_void_p), imp.ctypes.data_as(C.c_void_p), C.byref(sad))
        assert rc == 0, lib.adapter_last_error()
        assert np.array_equal(disp, g["disparity"])
        assert np.array_equal(imp, g["improved"])
        assert sad.value == float(np.abs(imgs[12][10:50, 10:50].astype(int) - imgs[11][11:51, 12:52].astype(int)).sum())


def test_adapter_depth_consumers():
    """shiftPerspective2 / DepthMapToPoints3D / Points3DToDepthMap / getGroups through the C++ binding == the reference's fixtures"""
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    lib.adapter_depth_consumers.restype = C.c_longlong
    g = np.load(os.path.join(ROOT, "tests", "golden", "depth_consumers.npz"))
    depth = np.ascontiguousarray(g["depth"])
    h, w = depth.shape
    shifted = np.zeros((h, w)); cloud = np.zeros((h * w, 3)); dmap = np.zeros((h, w)); sizes = np.zeros(16, np.int32)
    n = lib.adapter_depth_consumers(depth.ctypes.data_as(C.c_void_p), w, h, 12, 11, shifted.ctypes.data_as(C.c_void_p), cloud.ctypes.data_as(C.c_void_p),
                                    dmap.ctypes.data_as(C.c_void_p), sizes.ctypes.data_as(C.c_void_p))
    assert n >= 0, lib.adapter_last_error()
    assert np.array_equal(shifted, g["sp2"][0])          # pair (12, 11) is the first fixture pair
    assert np.array_equal(cloud[:n], g["cloud"])
    assert np.array_equal(dmap, g["maps"][1])            # the cloud of camera 12 seen from camera 11
    assert list(sizes[:13]) == list(g["group_sizes"])


def adapter_multi_gpu(lib, device, uid, rank, world, p, ref, others):
    """the C++ host's route to the multi-GPU entry points (adapter/sva_functions.cpp: svaCommInit, svaDepthPairSharded, svaDepthRowsSharded);
    -> (pair-sharded map on rank 0, this rank's rows of the row-sharded maps, y0)"""
    h, w = ref.shape
    others = [np.ascontiguousarray(o) for o in others]
    optr = (C.c_void_p * len(others))(*[o.ctypes.data for o in others])
    dp = np.zeros((h, w), np.uint16); dr = np.zeros((h, w), np.uint16); sr = np.zeros((h, w), np.float32)
    y0, rows = C.c_int(), C.c_int()
    ref = np.ascontiguousarray(ref)
    rc = lib.adapter_multi_gpu(device, (C.c_uint8 * 128).from_buffer_copy(uid), rank, world, C.byref(p), ref.ctypes.data_as(C.c_void_p), optr,
                               dp.ctypes.data_as(C.c_void_p), dr.ctypes.data_as(C.c_void_p), sr.ctypes.data_as(C.c_void_p), C.byref(y0), C.byref(rows))
    assert rc == 0, lib.adapter_last_error()
    return dp, dr[:rows.value], sr[:rows.value], y0.value


def test_adapter_reaches_the_multi_gpu_entry_points(oracle):
    """world of one: the same C++ calls a multi-process host makes (tools/check_sharded.py runs them over several GPUs)"""
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    from stereovisionarray_b200 import abi
    from stereovisionarray_b200._lib import lib as load
    load()  # maps torch's NCCL before the adapter's library binds one (see _lib._preload_nccl)
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    off = [(-1, 0), (1, 0), (0, -1), (0, 1), (1, 1)]
    h, w, D = 64, 96, 64
    sc = synth.make_scene(h, w, D, off, 31)
    p = abi.make_params(w, h, D, off, win_half=4, n_paths=8, lr_gx=-1)
    uid = (C.c_uint8 * 128)()
    assert lib.adapter_comm_id(uid) == 0, lib.adapter_last_error()
    dp, dr, sr, y0 = adapter_multi_gpu(lib, 0, bytes(uid), 0, 1, p, sc["ref"], sc["others"])
    d_o, s_o = oracle.depth_from_array(p, sc["ref"], sc["others"])
    assert y0 == 0 and np.array_equal(dp, d_o) and np.array_equal(dr, d_o) and np.array_equal(sr, s_o)
