"""The C++ adapter's fusion: svaDepthGroupsFused(p, images, getGroups(cameras, "CHESS"), 5, target, f, &subpix, &support), and svaDepthGroups
followed by svaFuseMaps (adapter/sva_functions.cpp) through the test glue, both equal DepthContext.depth_groups_fused on the same frame."""
import ctypes as C
import os

import numpy as np
import pytest

from stereovisionarray_b200 import abi, reference_api, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "adapter", "_build", "libsva_adapter_test.so")


@pytest.mark.parametrize("subpixel,target", [(1, 12), (0, 7)])
def test_adapter_depth_groups_fused_equals_python(subpixel, target):
    assert os.path.exists(SO), "adapter test library not built (__graft_entry__.build() builds it)"
    from stereovisionarray_b200._lib import lib as load
    from stereovisionarray_b200.pipeline import DepthContext
    load()  # maps torch's NCCL before the adapter's library binds one (see _lib._preload_nccl)
    lib = C.CDLL(SO)
    lib.adapter_last_error.restype = C.c_char_p
    h, w, D = 120, 160, 32
    sc = synth.make_array_scene(h, w, 5, 5, D, 23)
    images = [np.ascontiguousarray(im) for im in sc["images"]]
    tmask = np.ascontiguousarray(synth.ellipse_mask(h, w))
    p = abi.make_params(w, h, D, [(0, 0)] * 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=subpixel)
    p.n_pairs = 0
    disp = np.zeros((2, h, w), np.uint16)
    sub = np.zeros((2, h, w), np.float32)
    sup = np.zeros((2, h, w), np.uint8)
    rc = lib.adapter_depth_groups_fused(C.byref(p), (C.c_void_p * 25)(*[im.ctypes.data for im in images]), target, 16, 2,
                                        tmask.ctypes.data_as(C.c_void_p), disp.ctypes.data_as(C.c_void_p), sub.ctypes.data_as(C.c_void_p),
                                        sup.ctypes.data_as(C.c_void_p))
    assert rc == 13, lib.adapter_last_error()
    ctx = DepthContext(0)
    try:
        want = ctx.depth_groups_fused(p, images, reference_api.getGroups([None] * 25, "CHESS"), 5, target, 16, 2, target_mask=tmask)
    finally:
        ctx.close()
    for i, route in enumerate(("svaDepthGroupsFused", "svaDepthGroups + svaFuseMaps")):
        for a, b, name in zip((disp[i], sub[i], sup[i]), want, ("disp", "subpix", "support")):
            assert np.array_equal(a, b), "%s: %s differs from DepthContext.depth_groups_fused" % (route, name)
