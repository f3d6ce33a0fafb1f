"""The C++ adapter's stream of frames through the row-block pipeline (SvaRowsStream in adapter/sva_functions.cpp: world + 1 contexts on one
stream, links connected with sva_rows_stream_connect_comm, submit / flush / wait on cv::Mat images), driven through its test glue with a world
of one: every frame equals the oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from stereovisionarray_b200 import abi, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "adapter", "_build", "libsva_adapter_test.so")


def test_adapter_rows_stream_world_of_one(oracle):
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    from stereovisionarray_b200._lib import lib as load
    load()  # maps torch's NCCL before the adapter's library binds one (see _lib._preload_nccl)
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    off = [(-1, 0), (1, 0), (0, -1), (0, 1), (1, 1)]
    h, w, D, n = 48, 112, 64, 5
    p = abi.make_params(w, h, D, off, win_half=4, n_paths=8, lr_gx=-1)
    scenes = [synth.make_scene(h, w, D, off, 4100 + f, face=f % 2 == 1) for f in range(n)]
    for sc in scenes:  # contiguous u8, as the glue copies width * height bytes per image
        sc["ref"], sc["others"] = np.ascontiguousarray(sc["ref"]), [np.ascontiguousarray(o) for o in sc["others"]]
        sc["mask"] = None if sc["mask"] is None else np.ascontiguousarray(sc["mask"])
    refs = (C.c_void_p * n)(*[sc["ref"].ctypes.data for sc in scenes])
    others = (C.c_void_p * (n * len(off)))(*[o.ctypes.data for sc in scenes for o in sc["others"]])
    masks = (C.c_void_p * n)(*[None if sc["mask"] is None else sc["mask"].ctypes.data for sc in scenes])
    disp = np.zeros((n, h, w), np.uint16)
    sub = np.zeros((n, h, w), np.float32)
    y0, rows = C.c_int(), C.c_int()
    rc = lib.adapter_rows_stream(0, None, 0, 1, C.byref(p), n, refs, others, masks, disp.ctypes.data_as(C.c_void_p), sub.ctypes.data_as(C.c_void_p),
                                 C.byref(y0), C.byref(rows))
    assert rc == 0, lib.adapter_last_error()
    assert (y0.value, rows.value) == (0, h)
    for f, sc in enumerate(scenes):
        d_o, s_o = oracle.depth_from_array(p, sc["ref"], sc["others"], sc["mask"])
        assert np.array_equal(disp[f], d_o), "frame %d: integer disparity" % f
        assert np.array_equal(sub[f], s_o), "frame %d: sub-pixel" % f
