"""Host side of the multi-reference call sva_depth_groups (getGroups, SURVEY §8 f3), without a GPU: the grid offsets derived from the CHESS
groups, the refusal rules the Python wrapper checks before it calls the library, the split of 13 groups over 1-8 ranks, and the consistency
of the array test scene — checked with the oracle against the scene's own layer disparities, which catches a sign error in the offset
convention that a comparison of the GPU with the oracle (both fed the same offsets) cannot."""
import numpy as np
import pytest

from stereovisionarray_b200 import abi, dist, synth
from stereovisionarray_b200 import groups as G

# getCameraPairs(..., CROSS, i) for i = 0, 2, ..., 24, the {cameraNum, +5} quirk included: (ref, [(other, gx, gy), ...])
CHESS = [
    (0, [(5, 0, 1), (1, 1, 0)]),
    (2, [(5, -2, 1), (1, -1, 0), (3, 1, 0)]),
    (4, [(5, -4, 1), (3, -1, 0)]),
    (6, [(1, 0, -1), (5, -1, 0), (5, -1, 0), (7, 1, 0)]),
    (8, [(3, 0, -1), (5, -3, 0), (7, -1, 0), (9, 1, 0)]),
    (10, [(5, 0, -1), (5, 0, -1), (11, 1, 0)]),
    (12, [(7, 0, -1), (5, -2, -1), (11, -1, 0), (13, 1, 0)]),
    (14, [(9, 0, -1), (5, -4, -1), (13, -1, 0)]),
    (16, [(11, 0, -1), (5, -1, -2), (15, -1, 0), (17, 1, 0)]),
    (18, [(13, 0, -1), (5, -3, -2), (17, -1, 0), (19, 1, 0)]),
    (20, [(15, 0, -1), (21, 1, 0)]),
    (22, [(17, 0, -1), (21, -1, 0), (23, 1, 0)]),
    (24, [(19, 0, -1), (23, -1, 0)]),
]


def template(w, h, D, n_pairs, **kw):
    """make_params' defaults for groups of n_pairs pairs (P1, P2, cost shift), with no pairs: a template for sva_depth_groups"""
    p = abi.make_params(w, h, D, [(0, 0)] * n_pairs, **kw)
    p.n_pairs = 0
    return p


def chess_groups():
    return [[(ref, o) for o, _, _ in others] for ref, others in CHESS]


def test_chess_offsets_match_the_table(oracle):
    groups = G.as_groups(oracle.get_groups(25, "CHESS"))
    assert groups == chess_groups()
    for grp, (ref, others) in zip(groups, CHESS):
        assert G.group_offsets(grp, 5) == [(gx, gy) for _, gx, gy in others]
        q = G.group_params(abi.make_params(64, 48, 16, [], win_half=3), grp, 5)
        assert q.n_pairs == len(others)
        assert [(q.pair_gx[j], q.pair_gy[j]) for j in range(q.n_pairs)] == [(gx, gy) for _, gx, gy in others]
    # the groups whose offsets leave +-2 run the gather K1a; the others the image-space tile
    assert [i for i, (_, o) in enumerate(CHESS) if any(abs(gx) > 2 or abs(gy) > 2 for _, gx, gy in o)] == [2, 4, 7, 9]


def test_cameras_of_first_use_order():
    assert G.cameras_of(chess_groups()[:2]) == [0, 5, 1, 2, 3]
    assert sorted(G.cameras_of(chess_groups())) == list(range(25))


def _validate(p=None, groups=None, cols=5, shapes=None, rng=None, masks=None):
    p = abi.make_params(64, 48, 16, [], win_half=3) if p is None else p
    groups = chess_groups() if groups is None else groups
    shapes = [(48, 64)] * 25 if shapes is None else shapes
    return G.validate(p, groups, cols, shapes, rng, masks)


def test_validate_accepts_chess_and_partial_uploads():
    assert _validate() == (0, 13)
    # a rank of 8 with groups [4, 6) needs cameras 8, 3, 5, 7, 9, 10, 11 only
    need = set(G.cameras_of(chess_groups()[4:6]))
    assert need == {8, 3, 5, 7, 9, 10, 11}
    assert _validate(shapes=[(48, 64) if i in need else None for i in range(25)], rng=(4, 6)) == (4, 6)
    assert _validate(rng=(13, 13)) == (13, 13)
    assert _validate(rng=(0, 2), masks=[None, (48, 64)]) == (0, 2)


@pytest.mark.parametrize("what", ["mixed_ref", "self_pair", "index_high", "index_negative", "images_not_multiple", "range_high", "range_negative",
                                  "range_reversed", "too_many_pairs", "bad_params", "empty_group", "template_pairs", "wrong_size", "missing_camera",
                                  "mask_size"])
def test_validate_refuses(what):
    groups = chess_groups()
    p = abi.make_params(64, 48, 16, [], win_half=3)
    kw = {}
    if what == "mixed_ref":
        groups[3] = [(6, 1), (7, 5)]
    elif what == "self_pair":
        groups[0] = [(0, 0), (0, 1)]
    elif what == "index_high":
        groups[0] = [(0, 25)]
    elif what == "index_negative":
        groups[0] = [(0, -1)]
    elif what == "images_not_multiple":
        kw["shapes"] = [(48, 64)] * 24 + [None]
        kw["cols"] = 7
    elif what == "range_high":
        kw["rng"] = (0, 14)
    elif what == "range_negative":
        kw["rng"] = (-1, 3)
    elif what == "range_reversed":
        kw["rng"] = (5, 4)
    elif what == "too_many_pairs":
        groups[0] = [(12, o) for o in range(25) if o != 12] * 2
    elif what == "bad_params":  # a template field the library refuses for every group
        p = abi.make_params(64, 48, 16, [], win_half=57)
    elif what == "empty_group":
        groups[5] = []
    elif what == "template_pairs":
        p = abi.make_params(64, 48, 16, [(1, 0)], win_half=3)
    elif what == "wrong_size":
        kw["shapes"] = [(48, 64)] * 24 + [(48, 63)]
    elif what == "missing_camera":
        kw["shapes"] = [(48, 64)] * 24 + [None]
    elif what == "mask_size":
        kw["rng"] = (0, 2)
        kw["masks"] = [None, (47, 64)]
    with pytest.raises(ValueError):
        _validate(p, groups, **kw)


@pytest.mark.parametrize("world", range(1, 9))
def test_frame_range_covers_13_groups_once(world):
    got = []
    for r in range(world):
        b, e = dist.frame_range(13, world, r)
        got += list(range(b, e))
    assert got == list(range(13))
    if world == 8:
        assert [dist.frame_range(13, 8, r)[1] - dist.frame_range(13, 8, r)[0] for r in range(8)] == [2, 2, 2, 2, 2, 1, 1, 1]


def test_array_scene_views_agree_with_the_layers(oracle):
    """two cameras, WTA on the box cost (no SGM): on a layer's interior the integer disparity is the layer's disparity, whichever direction
    the other camera lies in — only if the scene and the offset convention agree"""
    h, w, D = 96, 128, 32
    sc = synth.make_array_scene(h, w, 3, 3, D, 11)
    gt = sc["gt"][4]
    yy, xx = np.mgrid[0:h, 0:w]
    for other in (1, 3, 5, 7, 8, 0):
        grp = [(4, other)]
        (gx, gy), = G.group_offsets(grp, 3)
        p = G.group_params(template(w, h, D, 1, win_half=4, n_paths=0), grp, 3)
        q = abi.make_params(w, h, D, [(gx, gy)], win_half=4, n_paths=0)
        assert bytes(p) == bytes(q)
        disp, _ = oracle.depth_from_array(p, sc["images"][4], [sc["images"][other]])
        for dl in sc["layers"]:
            # the layer where the other camera sees the same layer point at the offset the convention says: (x - gx*delta, y - gy*delta)
            sx, sy = xx - gx * dl, yy - gy * dl
            ok = (gt == dl) & (sx >= 0) & (sx < w) & (sy >= 0) & (sy < h)
            ok[ok] = sc["gt"][other][sy[ok], sx[ok]] == dl
            for _ in range(p.win_half + 1):  # the whole matching window inside that region
                ok = ok & np.roll(ok, 1, 0) & np.roll(ok, -1, 0) & np.roll(ok, 1, 1) & np.roll(ok, -1, 1)
            ok[:p.win_half] = ok[-p.win_half:] = False
            ok[:, :p.win_half] = ok[:, -p.win_half:] = False
            assert ok.sum() >= 100, (other, dl, ok.sum())
            assert (disp[ok] == dl).mean() > 0.98, (other, dl, (disp[ok] == dl).mean())
