"""sva_depth_groups on the GPU: every reference view of one array frame in one call.  The CHESS groups of a 5 x 5 frame (13 groups of 2, 3
or 4 pairs, duplicate pairs, offsets beyond +-2 on the gather K1a) against the oracle; the CROSS groups of every reference in census mode;
the c1-sized CHESS frame against 13 separate sva_depth_from_array calls; sharding emulated as group ranges with partial uploads; the array
scene's ground truth; refusals; guarded buffers; and a capture-stream frame in flight across the call."""
import numpy as np
import pytest

from stereovisionarray_b200 import abi, reference_api, synth
from stereovisionarray_b200 import groups as G
from stereovisionarray_b200.dist import frame_range

pytestmark = pytest.mark.gpu


def template(w, h, D, n_pairs, **kw):
    """make_params' defaults for groups of n_pairs pairs, with no pairs"""
    p = abi.make_params(w, h, D, [(0, 0)] * n_pairs, **kw)
    p.n_pairs = 0
    return p


def cross_groups():
    return [[tuple(pr) for pr in reference_api.gridPairs(5, 5, ref, abi.CROSS)[0]] for ref in range(25)]


@pytest.fixture(scope="module")
def ctx():
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small():
    """320 x 240, D = 32: the CHESS frame of the array scene, a mask on every other group"""
    h, w, D = 240, 320, 32
    sc = synth.make_array_scene(h, w, 5, 5, D, 7)
    groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
    masks = [synth.ellipse_mask(h, w) if g % 2 == 0 else None for g in range(len(groups))]
    p = template(w, h, D, 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=1)
    return dict(p=p, images=sc["images"], groups=groups, masks=masks, scene=sc)


def _check_vs_oracle(oracle, p, images, groups, masks, disp, sub, cols=5):
    for g, grp in enumerate(groups):
        q = G.group_params(p, grp, cols)
        d_o, s_o = oracle.depth_from_array(q, images[grp[0][0]], [images[o] for _, o in grp], None if masks is None else masks[g])
        assert np.array_equal(disp[g], d_o), "group %d (ref %d): integer disparity differs from the oracle" % (g, grp[0][0])
        assert float(np.max(np.abs(sub[g] - s_o))) <= 0.05, "group %d: sub-pixel disparity out of tolerance" % g


def test_chess_groups_vs_oracle(ctx, oracle, small):
    assert len(small["groups"]) == 13 and sorted({len(g) for g in small["groups"]}) == [2, 3, 4]
    disp, sub = ctx.depth_groups(small["p"], small["images"], small["groups"], 5, masks=small["masks"])
    assert disp.shape == (13, 240, 320) and sub.shape == (13, 240, 320)
    _check_vs_oracle(oracle, small["p"], small["images"], small["groups"], small["masks"], disp, sub)


def test_cross_groups_census_vs_oracle(ctx, oracle, small):
    groups = cross_groups()
    p = template(320, 240, 32, 4, win_half=4, n_paths=4, lr_gx=1, subpixel=1, cost_mode=abi.COST_CENSUS)
    disp, sub = ctx.depth_groups(p, small["images"], groups, 5)
    _check_vs_oracle(oracle, p, small["images"], groups, None, disp, sub)


def test_chess_c1_geometry_vs_separate_calls(ctx):
    h, w, D = 960, 1280, 128
    sc = synth.make_array_scene(h, w, 5, 5, D, 1001)
    groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
    p = template(w, h, D, 4, win_half=20, n_paths=8, lr_gx=-1, subpixel=1)
    disp, sub = ctx.depth_groups(p, sc["images"], groups, 5)
    for g, grp in enumerate(groups):
        q = G.group_params(p, grp, 5)
        d1, s1 = ctx.depth_from_array(q, sc["images"][grp[0][0]], [sc["images"][o] for _, o in grp])
        assert np.array_equal(disp[g], d1), "group %d: integer disparity differs from sva_depth_from_array" % g
        assert np.array_equal(sub[g], s1), "group %d: sub-pixel disparity differs from sva_depth_from_array" % g


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_ranges_concatenate_to_the_full_call(ctx, small, world):
    full_d, full_s = ctx.depth_groups(small["p"], small["images"], small["groups"], 5, masks=small["masks"])
    parts_d, parts_s = [], []
    for r in range(world):
        b, e = frame_range(13, world, r)
        mine = set(G.cameras_of(small["groups"][b:e]))
        imgs = [im if i in mine else None for i, im in enumerate(small["images"])]
        d, s = ctx.depth_groups(small["p"], imgs, small["groups"], 5, masks=small["masks"][b:e], group_range=(b, e))
        assert d.shape[0] == e - b
        parts_d.append(d)
        parts_s.append(s)
    assert np.array_equal(np.concatenate(parts_d), full_d)
    assert np.array_equal(np.concatenate(parts_s), full_s)


def test_cross_groups_find_the_ground_truth(ctx, small):
    """the scene's own disparities: on accepted pixels at least 6 px from a layer edge and 8 px from the border, the CROSS groups of all 25
    references find the true integer disparity on >= 90 % (the CPU oracle reaches 93-98 % per reference on this frame)"""
    sc = small["scene"]
    disp, _ = ctx.depth_groups(small["p"], small["images"], cross_groups(), 5)
    for ref in range(25):
        gt = sc["gt"][ref]
        edge = np.zeros(gt.shape, bool)
        for dy in range(-6, 7):
            for dx in range(-6, 7):
                edge |= np.roll(np.roll(gt, dy, 0), dx, 1) != gt
        core = ~edge
        core[:8] = core[-8:] = False
        core[:, :8] = core[:, -8:] = False
        acc = (disp[ref] != abi.SVA_DISP_INVALID) & core
        assert acc.mean() > 0.5, "reference %d: too few accepted pixels" % ref
        assert (disp[ref][acc] == gt[acc]).mean() >= 0.90, "reference %d: %.3f" % (ref, (disp[ref][acc] == gt[acc]).mean())


def test_refusals_enqueue_nothing(ctx, small):
    from stereovisionarray_b200._lib import SvaError
    p, images, groups = small["p"], small["images"], small["groups"]
    ctx.depth_groups(p, images, groups, 5, group_range=(0, 1))  # streams and events exist: a refusal must not even start one
    bad_tpl = template(320, 240, 32, 4, win_half=4)
    bad_tpl.n_pairs = 1
    bad_k = template(320, 240, 32, 4, win_half=57)
    wrong = [im if i != 5 else im[:, :-1] for i, im in enumerate(images)]
    cases = [
        ("mixed reference", p, images, [[(6, 1), (7, 5)]] + groups[1:], 5, None, (0, 13)),
        ("self pair", p, images, [[(0, 0), (0, 1)]] + groups[1:], 5, None, (0, 13)),
        ("index outside", p, images, [[(0, 25)]] + groups[1:], 5, None, (0, 13)),
        ("negative index", p, images, [[(0, -1)]] + groups[1:], 5, None, (0, 13)),
        ("images not a multiple of grid_cols", p, images, groups, 7, None, (0, 13)),
        ("range beyond n_groups", p, images, groups, 5, None, (0, 14)),
        ("negative range", p, images, groups, 5, None, (-1, 2)),
        ("reversed range", p, images, groups, 5, None, (3, 2)),
        ("more than 32 pairs", p, images, [[(12, o) for o in range(25) if o != 12] * 2] + groups[1:], 5, None, (0, 13)),
        ("empty group", p, images, groups[:5] + [[]] + groups[6:], 5, None, (0, 13)),
        ("template with pairs", bad_tpl, images, groups, 5, None, (0, 13)),
        ("refused parameters", bad_k, images, groups, 5, None, (0, 13)),
        ("camera of the wrong size", p, wrong, groups, 5, None, (0, 13)),
        ("camera without data", p, [None] + list(images[1:]), groups, 5, None, (0, 13)),
        ("mask of the wrong size", p, images, groups, 5, [np.zeros((240, 319), np.uint8)], (0, 1)),
    ]
    for what, pp, ims, grs, cols, masks, rng in cases:
        n0 = ctx.launches()
        with pytest.raises(SvaError) as e:
            ctx.depth_groups_unchecked(pp, ims, grs, cols, masks, rng)
        assert e.value.code == abi.SVA_ERR_BAD_ARG, what
        assert ctx.launches() == n0, "%s: kernels were launched" % what
        with pytest.raises(ValueError):  # the wrapper refuses the same call before it reaches the library
            ctx.depth_groups(pp, ims, grs, cols, masks=masks, group_range=rng)
    # camera without data is fine where no group of the range reads it
    ctx.depth_groups_unchecked(p, [None] + list(images[1:]), groups, 5, None, (1, 2))


def test_guarded_second_call_allocates_nothing(oracle, small):
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    try:
        c.set_guard(True)
        d1, s1 = c.depth_groups(small["p"], small["images"], small["groups"], 5, masks=small["masks"])
        n1, bad1 = c.check_guards()
        assert n1 > 0 and bad1 == 0, "%d canary bytes overwritten" % bad1
        d2, s2 = c.depth_groups(small["p"], small["images"], small["groups"], 5, masks=small["masks"])
        n2, bad2 = c.check_guards()
        assert bad2 == 0, "%d canary bytes overwritten" % bad2
        assert n2 == n1, "the second call of the same geometry added %d guarded buffers" % (n2 - n1)
        assert np.array_equal(d1, d2) and np.array_equal(s1, s2)
        _check_vs_oracle(oracle, small["p"], small["images"], small["groups"], small["masks"], d2, s2)
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
        disp, sub = c.depth_groups(small["p"], small["images"], small["groups"], 5, group_range=(0, 3))
        for t, sc, (d, s) in zip(tickets, frames, outs):
            c.stream_wait(t)
            d_o, s_o = oracle.depth_from_array(p, sc["ref"], sc["others"])
            assert np.array_equal(d, d_o), "capture-stream ticket %d: integer disparity" % t
            assert float(np.max(np.abs(s - s_o))) <= 0.05
        _check_vs_oracle(oracle, small["p"], small["images"], small["groups"][:3], None, disp, sub)
        # and the stream goes on after the call
        o = (np.zeros((h, w), np.uint16), np.zeros((h, w), np.float32))
        t = c.stream_submit(p, frames[0]["ref"], frames[0]["others"], None, *o)
        c.stream_wait(t)
        assert np.array_equal(o[0], outs[0][0])
    finally:
        c.close()
