"""The C++ adapter's multi-reference call: svaDepthGroups(p, images, getGroups(cameras, "CHESS"), 5) (adapter/sva_functions.cpp) through its
test glue equals DepthContext.depth_groups on the same frame, masks on every other group."""
import ctypes as C
import os

import numpy as np
import pytest

from stereovisionarray_b200 import abi, reference_api, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "adapter", "_build", "libsva_adapter_test.so")


def test_adapter_depth_groups_equals_python():
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    from stereovisionarray_b200._lib import lib as load
    from stereovisionarray_b200.pipeline import DepthContext
    load()  # maps torch's NCCL before the adapter's library binds one (see _lib._preload_nccl)
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    h, w, D = 120, 160, 32
    sc = synth.make_array_scene(h, w, 5, 5, D, 23)
    images = [np.ascontiguousarray(im) for im in sc["images"]]
    masks = [np.ascontiguousarray(synth.ellipse_mask(h, w)) if g % 2 else None for g in range(13)]
    p = abi.make_params(w, h, D, [(0, 0)] * 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=1)
    p.n_pairs = 0
    disp = np.zeros((13, h, w), np.uint16)
    sub = np.zeros((13, h, w), np.float32)
    rc = lib.adapter_depth_groups(C.byref(p), (C.c_void_p * 25)(*[im.ctypes.data for im in images]),
                                  (C.c_void_p * 13)(*[None if m is None else m.ctypes.data for m in masks]),
                                  disp.ctypes.data_as(C.c_void_p), sub.ctypes.data_as(C.c_void_p))
    assert rc == 13, lib.adapter_last_error()
    ctx = DepthContext(0)
    try:
        d_py, s_py = ctx.depth_groups(p, images, reference_api.getGroups([None] * 25, "CHESS"), 5, masks=masks)
    finally:
        ctx.close()
    assert np.array_equal(disp, d_py)
    assert np.array_equal(sub, s_py)
