"""Multi-view depth fusion on the GPU (DESIGN §3 item 6): sva_fuse_maps bit-exact with the oracle on random and crafted maps;
sva_depth_groups_fused bit-exact with sva_depth_groups + sva_fuse_maps (CHESS with masks, CROSS groups of all 25 cameras in census mode,
c1's geometry); the array scene's ground truth; refusals; guarded buffers; and a capture-stream frame in flight across the call."""
import numpy as np
import pytest

from stereovisionarray_b200 import abi, reference_api, synth
from stereovisionarray_b200 import groups as G
from stereovisionarray_b200.pipeline import fuse_params
from fuse_oracle import fuse_views
from test_gpu_groups import cross_groups, template
from test_oracle_fuse import INVALID, check_ground_truth, random_views

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small():
    """320 x 240, D = 32: the CHESS frame of the array scene, a mask on every other group, a target mask"""
    h, w, D = 240, 320, 32
    sc = synth.make_array_scene(h, w, 5, 5, D, 7)
    groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
    masks = [synth.ellipse_mask(h, w) if g % 2 == 0 else None for g in range(len(groups))]
    tmask = (np.random.default_rng(3).random((h, w)) < 0.9).astype(np.uint8)
    p = template(w, h, D, 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=1)
    return dict(p=p, images=sc["images"], groups=groups, masks=masks, tmask=tmask, scene=sc)


def _equal(got, want, what):
    for a, b, name in zip(got, want, ("disp", "subpix", "support")):
        assert a.shape == b.shape and np.array_equal(a, b), "%s: %s differs" % (what, name)


@pytest.mark.parametrize("n", [1, 2, 13, 25, 32])
def test_fuse_maps_equals_the_oracle_on_random_maps(ctx, n):
    disp, sub, refs = random_views(n, 48, 80, 77 + n)
    mask = (np.random.default_rng(n).random((48, 80)) < 0.8).astype(np.uint8)
    for use_sub in (False, True):
        for tol, ms, m in ((0, 1, None), (16, min(2, n), mask), (4095, n, None)):
            for target in (12, 0, 23):
                s = sub if use_sub else None
                got = ctx.fuse_maps(disp, s, refs, 5, 25, target, tol, ms, m)
                _equal(got, fuse_views(disp, s, refs, 5, target, tol, ms, m), "n=%d sub=%d tol=%d ms=%d t=%d" % (n, use_sub, tol, ms, target))


def test_fuse_maps_on_crafted_cases(ctx):
    """the oracle tests' crafted cases: nearer source of one view, rint and shift ties at negative offsets, equal clusters, identity,
    order of the views"""
    cases = []
    disp = np.full((1, 4, 16), INVALID, np.uint16)
    disp[0, 2, 5], disp[0, 2, 6], disp[0, 2, 10], disp[0, 2, 11] = 3, 2, 2, 3
    cases += [(disp, None, [1], 0, 0, 1), (disp, None, [1], 2, 0, 1)]
    one = np.full((1, 8, 32), INVALID, np.uint16)
    sone = np.full((1, 8, 32), -1.0, np.float32)
    one[0, 4, 10], sone[0, 4, 10] = 1, 1.5
    one[0, 4, 20], sone[0, 4, 20] = 2, 40.5 / 16
    one[0, 5, 20], sone[0, 5, 20] = 2, 41.5 / 16
    cases += [(one, sone, [6], t, 0, 1) for t in (5, 6, 7, 1, 11)]
    clus = np.full((4, 4, 8), INVALID, np.uint16)
    for g, v in enumerate((2, 5, 2, 5)):
        clus[g, 1, 3] = v
    cases += [(clus, None, [12] * 4, 12, 16, 2), (clus, None, [12] * 4, 12, 16, 3)]
    ident, _, _ = random_views(1, 24, 40, 9, max_disp=200)
    cases += [(ident, None, [7], 7, 0, 1)]
    for d, s, refs, t, tol, ms in cases:
        _equal(ctx.fuse_maps(d, s, refs, 5, 25, t, tol, ms), fuse_views(d, s, refs, 5, t, tol, ms), "crafted t=%d" % t)
    got = ctx.fuse_maps(ident, None, [7], 5, 25, 7, 0, 1)
    assert np.array_equal(got[0], ident[0])
    disp, sub, refs = random_views(13, 24, 40, 5)
    base = ctx.fuse_maps(disp, sub, refs, 5, 25, 12, 16, 2)
    perm = np.random.default_rng(1).permutation(13)
    _equal(ctx.fuse_maps(disp[perm], sub[perm], [refs[i] for i in perm], 5, 25, 12, 16, 2), base, "permuted views")


def _fused_vs_composed(ctx, p, images, groups, target, masks=None, tmask=None, tol=16, ms=2):
    fused = ctx.depth_groups_fused(p, images, groups, 5, target, tol, ms, masks=masks, target_mask=tmask)
    d, s = ctx.depth_groups(p, images, groups, 5, masks=masks)
    refs = [g[0][0] for g in groups]
    composed = ctx.fuse_maps(d, s if p.subpixel == 1 else None, refs, 5, len(images), target, tol, ms, tmask)
    _equal(fused, composed, "target %d" % target)
    return fused, (d, s)


def test_chess_fused_equals_groups_then_fuse(ctx, small):
    for target, tmask in ((12, small["tmask"]), (7, None), (0, small["tmask"])):
        _fused_vs_composed(ctx, small["p"], small["images"], small["groups"], target, small["masks"], tmask)
    # integer maps: subpixel off
    p = template(320, 240, 32, 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=0)
    _fused_vs_composed(ctx, p, small["images"], small["groups"], 12, small["masks"], None, tol=0, ms=1)


def test_cross_groups_census_25_views(ctx, small):
    p = template(320, 240, 32, 4, win_half=4, n_paths=4, lr_gx=1, subpixel=1, cost_mode=abi.COST_CENSUS)
    fused, _ = _fused_vs_composed(ctx, p, small["images"], cross_groups(), 12, None, small["tmask"], tol=16, ms=3)
    assert int(fused[2].max()) > 13  # more than 13 views agree somewhere: all 25 took part


def test_c1_geometry_target_12(ctx):
    h, w, D = 960, 1280, 128
    sc = synth.make_array_scene(h, w, 5, 5, D, 1001)
    groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
    p = template(w, h, D, 4, win_half=20, n_paths=8, lr_gx=-1, subpixel=1)
    fused, (d, _) = _fused_vs_composed(ctx, p, sc["images"], groups, 12)
    assert (fused[0] != INVALID).mean() > (d[6] != INVALID).mean()  # group 6 is camera 12's own


def test_fused_maps_find_the_ground_truth(ctx, small):
    """the oracle's thresholds (tests/test_oracle_fuse.py::check_ground_truth) on the GPU's maps"""
    groups = small["groups"]
    refs = [g[0][0] for g in groups]
    d, _ = ctx.depth_groups(small["p"], small["images"], groups, 5)
    own = {t: d[refs.index(t)] for t in (12, 0)}
    fused = {t: ctx.depth_groups_fused(small["p"], small["images"], groups, 5, t, 16, 2)[0] for t in (12, 7, 0)}
    check_ground_truth(small["scene"], refs, own, fused)


def test_refusals_enqueue_nothing(ctx, small):
    from stereovisionarray_b200._lib import SvaError
    p, images, groups = small["p"], small["images"], small["groups"]
    ctx.depth_groups_fused(p, images, groups[:2], 5, 12)  # streams, events and workspaces exist: a refusal must not even start one
    disp, sub, refs = random_views(3, 24, 40, 1)
    ctx.fuse_maps(disp, sub, refs, 5, 25, 12)

    def fp(tol=16, ms=2, res=0):
        f = fuse_params(tol, ms)
        f.reserved[3] = res
        return f

    d3, s3 = list(disp), list(sub)
    fuse_cases = [
        ("no views", [], None, [], 5, 25, 12, fp(ms=1), None),
        ("33 views", [disp[0]] * 33, None, [0] * 33, 5, 25, 12, fp(), None),
        ("reference outside", d3, s3, [0, 1, 25], 5, 25, 12, fp(), None),
        ("negative reference", d3, s3, [0, -1, 2], 5, 25, 12, fp(), None),
        ("target outside", d3, s3, refs, 5, 25, 25, fp(), None),
        ("negative target", d3, s3, refs, 5, 25, -1, fp(), None),
        ("cameras not a multiple of grid_cols", d3, s3, refs, 4, 25, 12, fp(), None),
        ("tol_16 above 4095", d3, s3, refs, 5, 25, 12, fp(tol=4096), None),
        ("negative tol_16", d3, s3, refs, 5, 25, 12, fp(tol=-1), None),
        ("min_support 0", d3, s3, refs, 5, 25, 12, fp(ms=0), None),
        ("min_support above n_views", d3, s3, refs, 5, 25, 12, fp(ms=4), None),
        ("non-zero reserved", d3, s3, refs, 5, 25, 12, fp(res=1), None),
        ("null disp map", [disp[0], None, disp[2]], s3, refs, 5, 25, 12, fp(), None),
        ("null subpix map", d3, [sub[0], None, sub[2]], refs, 5, 25, 12, fp(), None),
        ("mask of the wrong size", d3, s3, refs, 5, 25, 12, fp(), np.ones((24, 39), np.uint8)),
    ]
    for what, dd, ss, rr, cols, ncam, t, f, m in fuse_cases:
        n0 = ctx.launches()
        with pytest.raises(SvaError) as e:
            ctx.fuse_maps_unchecked(dd or [disp[0]], ss, rr, cols, ncam, t, f, m) if dd else _fuse_no_views(ctx, disp[0], f)
        assert e.value.code == abi.SVA_ERR_BAD_ARG, what
        assert ctx.launches() == n0, "%s: kernels were launched" % what
        # the wrapper refuses the same call before it reaches the library (it cannot pass null maps or reserved fields)
        if dd and all(x is not None for x in dd) and (ss is None or all(x is not None for x in ss)) and not any(f.reserved):
            with pytest.raises(ValueError):
                ctx.fuse_maps(np.array(dd), None if ss is None else np.array(ss), rr, cols, ncam, t, f.tol_16, f.min_support, m)

    bad_k = template(320, 240, 32, 4, win_half=57)
    group_cases = [
        ("no groups", p, images, [], 5, None, 12, fp(ms=1), None),
        ("33 groups", p, images, (groups * 3)[:33], 5, None, 12, fp(), None),
        ("target outside", p, images, groups, 5, None, 25, fp(), None),
        ("tol_16 above 4095", p, images, groups, 5, None, 12, fp(tol=4096), None),
        ("min_support above n_views", p, images, groups, 5, None, 12, fp(ms=14), None),
        ("non-zero reserved", p, images, groups, 5, None, 12, fp(res=2), None),
        ("target mask of the wrong size", p, images, groups, 5, None, 12, fp(), np.ones((239, 320), np.uint8)),
        ("mixed reference", p, images, [[(6, 1), (7, 5)]] + groups[1:], 5, None, 12, fp(), None),
        ("images not a multiple of grid_cols", p, images, groups, 7, None, 12, fp(), None),
        ("refused parameters", bad_k, images, groups, 5, None, 12, fp(), None),
        ("camera without data", p, [None] + list(images[1:]), groups, 5, None, 12, fp(), None),
        ("group mask of the wrong size", p, images, groups, 5, [np.zeros((240, 319), np.uint8)] + [None] * 12, 12, fp(), None),
    ]
    for what, pp, ims, grs, cols, masks, t, f, tm in group_cases:
        n0 = ctx.launches()
        with pytest.raises(SvaError) as e:
            ctx.depth_groups_fused_unchecked(pp, ims, grs, cols, t, f, masks, tm)
        assert e.value.code == abi.SVA_ERR_BAD_ARG, what
        assert ctx.launches() == n0, "%s: kernels were launched" % what
        if any(f.reserved):
            continue
        with pytest.raises(ValueError):
            ctx.depth_groups_fused(pp, ims, grs, cols, t, f.tol_16, f.min_support, masks=masks, target_mask=tm)


def _fuse_no_views(ctx, like, f):
    """sva_fuse_maps with n_views = 0 (the wrapper cannot express it)"""
    import ctypes as C
    h, w = like.shape
    out = [np.empty((h, w), t) for t in (np.uint16, np.float32, np.uint8)]
    from stereovisionarray_b200._lib import check
    refs = np.zeros(1, np.int32)
    ptrs = (C.c_void_p * 1)(like.ctypes.data)
    check(ctx._h, ctx._L.sva_fuse_maps(ctx._h, w, h, 5, 25, refs.ctypes.data, 0, ptrs, None, 12, C.byref(f), None, *[a.ctypes.data for a in out]))


def test_guarded_second_call_allocates_nothing(small):
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    try:
        c.set_guard(True)
        args = (small["p"], small["images"], small["groups"], 5, 12)
        kw = dict(masks=small["masks"], target_mask=small["tmask"])
        f1 = c.depth_groups_fused(*args, **kw)
        n1, bad1 = c.check_guards()
        assert n1 > 0 and bad1 == 0, "%d canary bytes overwritten" % bad1
        f2 = c.depth_groups_fused(*args, **kw)
        n2, bad2 = c.check_guards()
        assert bad2 == 0, "%d canary bytes overwritten" % bad2
        assert n2 == n1, "the second call of the same geometry added %d guarded buffers" % (n2 - n1)
        _equal(f1, f2, "second call")
        # the host form, twice
        d, s = c.depth_groups(small["p"], small["images"], small["groups"], 5, masks=small["masks"])
        refs = [g[0][0] for g in small["groups"]]
        h1 = c.fuse_maps(d, s, refs, 5, 25, 12, mask=small["tmask"])
        n3, bad3 = c.check_guards()
        h2 = c.fuse_maps(d, s, refs, 5, 25, 12, mask=small["tmask"])
        n4, bad4 = c.check_guards()
        assert bad3 == 0 and bad4 == 0 and n4 == n3
        _equal(h1, f1, "fuse_maps vs fused call")
        _equal(h2, h1, "fuse_maps second call")
        _equal(h1, fuse_views(d, s, refs, 5, 12, 16, 2, small["tmask"]), "fuse_maps vs oracle")
    finally:
        c.close()


def test_capture_stream_frame_in_flight_survives(oracle, small):
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    try:
        off = [(-1, 0), (1, 0), (0, -1), (0, 1)]
        h, w, D = 96, 160, 64
        frames = [synth.make_scene(h, w, D, off, 7300 + f) for f in range(2)]
        p = abi.make_params(w, h, D, off, win_half=4, n_paths=8, lr_gx=-1)
        outs = [(np.zeros((h, w), np.uint16), np.zeros((h, w), np.float32)) for _ in frames]
        tickets = [c.stream_submit(p, sc["ref"], sc["others"], None, *o) for sc, o in zip(frames, outs)]
        fused = c.depth_groups_fused(small["p"], small["images"], small["groups"][:3], 5, 12, 16, 1)
        for t, sc, (d, s) in zip(tickets, frames, outs):
            c.stream_wait(t)
            d_o, s_o = oracle.depth_from_array(p, sc["ref"], sc["others"])
            assert np.array_equal(d, d_o), "capture-stream ticket %d: integer disparity" % t
            assert float(np.max(np.abs(s - s_o))) <= 0.05
        gd, gs = c.depth_groups(small["p"], small["images"], small["groups"][:3], 5)
        _equal(fused, c.fuse_maps(gd, gs, [g[0][0] for g in small["groups"][:3]], 5, 25, 12, 16, 1), "fused call next to the stream")
        o = (np.zeros((h, w), np.uint16), np.zeros((h, w), np.float32))
        t = c.stream_submit(p, frames[0]["ref"], frames[0]["others"], None, *o)
        c.stream_wait(t)
        assert np.array_equal(o[0], outs[0][0])
    finally:
        c.close()
