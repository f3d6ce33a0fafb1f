"""Memory-safety self-check (the box has no compute-sanitizer): the parity cases again on contexts whose device buffers carry canary
bands and a poisoned payload (sva_debug_set_guard).  An out-of-bounds write shows up as overwritten canary bytes; a read of memory that
no kernel wrote shows up as a parity failure, because the payload starts as 0xCD instead of the zeros cudaMalloc tends to return."""
import os

import numpy as np
import pytest

from stereovisionarray_b200 import abi, synth
from test_gpu_volume import CASES, OFF8

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# frames wide enough for many CTAs per launch: c1-like rows (unpaced SGM) and c2-like rows (W * D * 4 >= 768 KB: paced SGM)
WIDE = [
    (96, 1280, 128, OFF8, dict(win_half=20, n_paths=8, lr_gx=-1)),
    (80, 1024, 192, OFF8, dict(win_half=20, n_paths=8, lr_gx=-1)),
    # c3-wide rows: three directions x 3840 lines exceed one resident wave, so each row-sweeping group runs as ranged launches
    (48, 3840, 256, [(-1, 0), (1, 1)], dict(win_half=4, n_paths=8, lr_gx=-1)),
    (40, 3840, 192, [(-1, 0), (0, -1)], dict(win_half=3, n_paths=8, lr_gx=1)),
    # more rows than one block of W / 16 = 240: each row-sweeping group is marched in two row blocks (240 + 20 rows, run_group_in_blocks),
    # the path-line state handed across the boundary, each block cut by columns into its own set of ranged launches
    (260, 3840, 64, [(-1, 0), (1, 0), (0, 1)], dict(win_half=4, n_paths=8, lr_gx=-1)),
]


@pytest.fixture(scope="module")
def gctx():
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    c.set_guard(True)
    yield c
    c.close()


def _clean(c):
    n, bad = c.check_guards()
    assert n > 0, "no guarded buffers: the guard switch did not take"
    assert bad == 0, "%d canary bytes overwritten (out-of-bounds write)" % bad


@pytest.mark.parametrize("case", range(len(CASES) + len(WIDE)))
def test_guarded_stages(gctx, oracle, case):
    h, w, D, offsets, kw = (CASES + WIDE)[case]
    sc = synth.make_scene(h, w, D, offsets, 500 + case, min_disp=kw.get("min_disp", 0), face=(case % 2 == 0))
    p = abi.make_params(w, h, D, offsets, **kw)
    gctx.set_debug(0, 0)
    gctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    gctx.run(abi.STAGE_AD)
    A_o = oracle.ad_volume(p, sc["ref"], sc["others"])
    assert np.array_equal(gctx.download_ad(), A_o)
    gctx.run(abi.STAGE_BOX)
    C_o = oracle.box_cost(p, A_o)
    assert np.array_equal(gctx.download_cost(), C_o)
    gctx.set_debug(1, 0)
    gctx.run(abi.STAGE_SGM)
    S_o = oracle.sgm_aggregate(p, C_o) if p.n_paths else C_o
    if p.n_paths:
        assert np.array_equal(gctx.download_sgm(), S_o)
    disp, sub = gctx.download_disparity()
    disp_o, sub_o = oracle.wta(p, S_o, sc["mask"])
    assert np.array_equal(disp, disp_o) and np.array_equal(sub, sub_o)
    gctx.set_debug(0, 0)
    # the production order (no debug stores), one call, and a second geometry right after on the same buffers
    d1, s1 = gctx.depth_from_array(p, sc["ref"], sc["others"], sc["mask"])
    assert np.array_equal(d1, disp_o) and np.array_equal(s1, sub_o)
    _clean(gctx)


def test_guarded_stream(gctx, oracle):
    h, w, D = 72, 200, 64
    p = abi.make_params(w, h, D, OFF8, win_half=5, n_paths=8, lr_gx=-1)
    frames = [synth.make_scene(h, w, D, OFF8, 700 + i, face=(i % 2 == 1)) for i in range(4)]
    outs = [(np.empty((h, w), np.uint16), np.empty((h, w), np.float32)) for _ in frames]
    keep = [abi.image_array(f["others"]) for f in frames]
    for t in [gctx.stream_submit(p, f["ref"], k, f["mask"], o[0], o[1]) for f, k, o in zip(frames, keep, outs)]:
        gctx.stream_wait(t)
    for f, o in zip(frames, outs):
        disp_o, sub_o = oracle.depth_from_array(p, f["ref"], f["others"], f["mask"])
        assert np.array_equal(o[0], disp_o) and np.array_equal(o[1], sub_o)
    _clean(gctx)


def test_guard_detects_a_stray_write(gctx):
    """the check itself: four bytes written just below a library buffer are reported, and restoring them clears the report"""
    import torch
    from stereovisionarray_b200.dist import _CudaAlias
    h, w, D = 40, 64, 16
    sc = synth.make_scene(h, w, D, [(-1, 0)], 3)
    gctx.depth_from_array(abi.make_params(w, h, D, [(-1, 0)], win_half=3, n_paths=4, lr_gx=-1), sc["ref"], sc["others"])
    ptr, _ = gctx.cost_device_ptr()
    below = torch.as_tensor(_CudaAlias(ptr - 4, 1), device="cuda")
    below.fill_(0)
    torch.cuda.synchronize()
    assert gctx.check_guards()[1] == 4
    below.fill_(-1515870811)  # 0xA5A5A5A5
    torch.cuda.synchronize()
    _clean(gctx)


def test_guarded_literal_and_consumers(oracle):
    """literal matcher, warp, refine and the depth consumers on a guarded context of the reference-named API"""
    from stereovisionarray_b200 import reference_api as api
    from stereovisionarray_b200._lib import lib
    import ctypes as C
    L = lib()
    if 0 in api._ctx:
        L.sva_destroy(api._ctx.pop(0))
    hctx = api._context(0)
    assert L.sva_debug_set_guard(hctx, 1) == 0

    def clean():
        n, bad = C.c_int64(), C.c_int64()
        assert L.sva_debug_check_guards(hctx, C.byref(n), C.byref(bad)) == 0
        assert n.value > 0 and bad.value == 0, "%d canary bytes overwritten" % bad.value

    from test_gpu_literal import _cams
    g = np.load(os.path.join(G, "main_120x160_s7.npz"))
    h, w, seed = int(g["h"]), int(g["w"]), int(g["seed"])
    sc = synth.make_literal_scene(h, w, seed)
    cams = _cams(api, w)
    disp = api.matchLiteral(sc["images"], cams, [(12, 11)], g["mask"], 20, 0.5, 1.0)
    assert np.array_equal(disp, g["disparity"])
    clean()
    imp = api.improveWithDisparity(disp, sc["images"][12], [sc["images"][11]], [(cams[12], cams[11])], 21, g["mask"])
    assert np.array_equal(imp, g["improved"])
    clean()
    # a multi-pair literal frame against the oracle (no mask: every pixel of the valid area)
    sc2 = synth.make_literal_scene(112, 144, 34, pair=(12, 17))
    pairs = [(12, 18), (12, 11), (12, 17)]
    from test_gpu_literal import _abi_cams
    assert np.array_equal(api.matchLiteral(sc2["images"], _cams(api, 144), pairs, None, 20),
                          oracle.match_literal(sc2["images"], _abi_cams(144), pairs, None, 20, n_threads=8))
    clean()
    wr = np.load(os.path.join(G, "warp_refine.npz"))
    cw = _cams(api, wr["center"].shape[1])
    for (a, b), exp in zip(wr["warp_pairs"], wr["warps"]):
        assert np.array_equal(api.shiftPerspectiveWithDisparity(cw[a], cw[b], wr["disp"], wr["other"]), exp)
    clean()
    dc = np.load(os.path.join(G, "depth_consumers.npz"))
    cd = _cams(api, dc["depth"].shape[1])
    for (a, b), exp in zip(dc["sp2_pairs"], dc["sp2"]):
        assert np.array_equal(api.shiftPerspective2(cd[a], cd[b], dc["depth"]), exp)
    hh, ww = dc["depth"].shape
    cloud = api.DepthMapToPoints3D(dc["depth"], cd[12], (ww, hh))
    assert np.array_equal(cloud, dc["cloud"])
    for ci, exp in zip(dc["maps_cams"], dc["maps"]):
        assert np.array_equal(api.Points3DToDepthMap(cloud, cd[ci], (ww, hh)), exp)
    assert np.array_equal(api.Points3DToDepthMap(cloud, cd[12], (ww // 2, hh // 2)), dc["half_map"])
    clean()
    L.sva_destroy(api._ctx.pop(0))
