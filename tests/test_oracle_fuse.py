"""The multi-view depth fusion spec (DESIGN §3 item 6) as its CPU restatement states it (tests/fuse_oracle.c): orc_fuse_views against an
independent numpy restatement on random maps, its properties on crafted cases, and what it does on the array scene's ground truth (group
maps from the oracle).  CPU only."""
import itertools

import numpy as np
import pytest

from stereovisionarray_b200 import abi, reference_api, synth
from stereovisionarray_b200 import groups as G
from fuse_oracle import fuse_views

INVALID = abi.SVA_DISP_INVALID


def np_fuse(disp, sub, refs, cols, target, tol, min_support, mask=None):
    """§3 item 6 restated with numpy: a z-buffer per view by np.maximum.at, the vote over all pairs of views at once"""
    n, H, W = disp.shape
    yy, xx = np.mgrid[0:H, 0:W]
    Z = np.zeros((n, H * W), np.int64)
    for g in range(n):
        used = disp[g] != INVALID
        if sub is None:
            q = 16 * disp[g].astype(np.int64)
        else:
            s = sub[g]
            with np.errstate(invalid="ignore"):
                used &= (s >= 0) & (s < 4352)
            q = np.rint(16 * np.where(used, s, 0).astype(np.float32)).astype(np.int64)
        gx, gy = target % cols - refs[g] % cols, target // cols - refs[g] // cols
        xt, yt = xx - ((gx * q + 8) >> 4), yy - ((gy * q + 8) >> 4)
        ok = used & (xt >= 0) & (xt < W) & (yt >= 0) & (yt < H)
        np.maximum.at(Z[g], (yt * W + xt)[ok], q[ok] + 1)
    valid = Z > 0
    c = Z - 1
    agree = (np.abs(c[:, None, :] - c[None, :, :]) <= tol) & valid[:, None, :] & valid[None, :, :]
    support = np.where(valid, agree.sum(1), -1)
    key = np.where(valid, support * (1 << 24) + c, -1)  # largest support, then the larger value (c < 2^21)
    best = np.take_along_axis(c, key.argmax(0)[None], 0)[0]
    M = valid & (np.abs(c - best[None]) <= tol)
    nstar = M.sum(0)
    qh = (np.where(M, c, 0).sum(0) + nstar // 2) // np.maximum(nstar, 1)
    ok = (nstar > 0) & (nstar >= min_support)
    if mask is not None:
        ok &= mask.reshape(-1) != 0
    d = np.where(ok, (qh + 8) >> 4, INVALID).astype(np.uint16)
    s = np.where(ok, qh / 16.0, -1.0).astype(np.float32)
    return d.reshape(H, W), s.reshape(H, W), nstar.astype(np.uint8).reshape(H, W)


def random_views(n, h, w, seed, max_disp=6):
    """n views of a 5 x 5 array (refs drawn from the 25 cameras, repeats allowed beyond 25): small disparities so that many sources
    collide; ~15 % invalid; sub-pixel maps with exact rint ties, negative values, NaN and values at or beyond 4352"""
    rng = np.random.default_rng(seed)
    disp = rng.integers(0, max_disp + 1, (n, h, w)).astype(np.uint16)
    sub = (disp + rng.uniform(-0.5, 0.5, disp.shape)).astype(np.float32)
    ties = rng.random(disp.shape) < 0.1
    sub[ties] = (np.floor(sub[ties] * 16) + 0.5) / 16  # 16 * s = k + 0.5
    sub[rng.random(disp.shape) < 0.01] = -0.25
    sub[rng.random(disp.shape) < 0.01] = np.nan
    sub[rng.random(disp.shape) < 0.005] = 4352.0
    sub[rng.random(disp.shape) < 0.005] = 4351.96875
    disp[rng.random(disp.shape) < 0.15] = INVALID
    refs = list(rng.permutation(25)[:n]) if n <= 25 else list(rng.permutation(25)) + list(rng.integers(0, 25, n - 25))
    return disp, sub, [int(r) for r in refs]


def params_grid():
    for n in (1, 2, 13, 25, 32):
        for use_sub, tol, ms in itertools.product((False, True), (0, 16, 4095), sorted({1, 2, n} - ({2} if n < 2 else set()))):
            yield n, use_sub, tol, ms


@pytest.mark.parametrize("n,use_sub,tol,ms", list(params_grid()))
def test_oracle_equals_numpy_restatement(n, use_sub, tol, ms):
    h, w = 24, 40
    disp, sub, refs = random_views(n, h, w, 1000 * n + tol + ms)
    mask = (np.random.default_rng(n).random((h, w)) < 0.8).astype(np.uint8) if tol == 16 else None
    for target in (12, 0, 23):
        got = fuse_views(disp, sub if use_sub else None, refs, 5, target, tol, ms, mask)
        want = np_fuse(disp, sub if use_sub else None, refs, 5, target, tol, ms, mask)
        for a, b, what in zip(got, want, ("disp", "subpix", "support")):
            assert np.array_equal(a, b), "%s differs (target %d)" % (what, target)


def test_result_does_not_depend_on_the_order_of_the_views():
    disp, sub, refs = random_views(13, 24, 40, 5)
    base = fuse_views(disp, sub, refs, 5, 12, 16, 2)
    for seed in range(3):
        perm = np.random.default_rng(seed).permutation(13)
        got = fuse_views(disp[perm], sub[perm], [refs[i] for i in perm], 5, 12, 16, 2)
        for a, b in zip(got, base):
            assert np.array_equal(a, b)


def test_one_integer_view_onto_its_own_camera_is_that_map():
    disp, _, _ = random_views(1, 24, 40, 9, max_disp=200)
    d, s, n = fuse_views(disp, None, [7], 5, 7, 0, 1)
    assert np.array_equal(d, disp[0])
    valid = disp[0] != INVALID
    assert np.array_equal(s[valid], disp[0][valid].astype(np.float32)) and np.all(s[~valid] == -1.0)
    assert np.array_equal(n, valid.astype(np.uint8))


def test_the_nearer_of_two_sources_of_one_view_wins():
    """whichever of the two the scan visits first: view of camera 1 into camera 0 (gx = -1, x' = x + d): x = 5 at d = 3 and x = 6 at d = 2
    land on x' = 8; into camera 2 (gx = +1, x' = x - d): x = 10 at d = 2 and x = 11 at d = 3 land on x' = 8"""
    for target, srcs in ((0, ((5, 3), (6, 2))), (2, ((10, 2), (11, 3)))):
        disp = np.full((1, 4, 16), INVALID, np.uint16)
        for x, v in srcs:
            disp[0, 2, x] = v
        d, s, n = fuse_views(disp, None, [1], 5, target, 0, 1)
        assert d[2, 8] == 3 and s[2, 8] == 3.0 and n[2, 8] == 1, target
        assert np.count_nonzero(d != INVALID) == 1


def test_rounding_ties():
    """rint(16 s) rounds half to even; (gx q + 8) >> 4 rounds half towards +inf, also for negative gx q"""
    disp = np.full((1, 8, 32), INVALID, np.uint16)
    sub = np.full((1, 8, 32), -1.0, np.float32)
    disp[0, 4, 10], sub[0, 4, 10] = 2, 40.5 / 16   # q = 40 (even)
    disp[0, 4, 20], sub[0, 4, 20] = 2, 41.5 / 16   # q = 42
    d, s, _ = fuse_views(disp, sub, [6], 5, 6, 0, 1)  # own camera: no shift
    assert s[4, 10] == 40 / 16 and s[4, 20] == 42 / 16
    assert d[4, 10] == 3 and d[4, 20] == 3  # (40 + 8) >> 4 = 3, (42 + 8) >> 4 = 3
    one = np.full((1, 8, 32), INVALID, np.uint16)
    sone = np.full((1, 8, 32), -1.0, np.float32)
    one[0, 4, 10], sone[0, 4, 10] = 1, 1.5  # q = 24: gx q = -24 -> (-16) >> 4 = -1; +24 -> 32 >> 4 = 2
    for target, x_want in ((5, 11), (7, 8)):  # ref 6; target 5: gx = -1; target 7: gx = +1
        d, s, _ = fuse_views(one, sone, [6], 5, target, 0, 1)
        assert d[4, x_want] == 2 and s[4, x_want] == 1.5 and np.count_nonzero(d != INVALID) == 1, target
    for target, y_want in ((1, 5), (11, 2)):  # ref 6; target 1: gy = -1; target 11: gy = +1
        d, s, _ = fuse_views(one, sone, [6], 5, target, 0, 1)
        assert d[y_want, 10] == 2 and np.count_nonzero(d != INVALID) == 1, target


def test_two_clusters_of_equal_support_the_nearer_wins():
    disp = np.full((4, 4, 8), INVALID, np.uint16)
    for g, v in enumerate((2, 5, 2, 5)):
        disp[g, 1, 3] = v
    d, s, n = fuse_views(disp, None, [12] * 4, 5, 12, 16, 2)
    assert d[1, 3] == 5 and s[1, 3] == 5.0 and n[1, 3] == 2
    d, s, n = fuse_views(disp, None, [12] * 4, 5, 12, 16, 3)
    assert d[1, 3] == INVALID and s[1, 3] == -1.0 and n[1, 3] == 2
    # a spread cluster: 32, 40, 48 at tol 16 -> 40 has support 3, the mean of all three is the result
    sub = np.full((3, 4, 8), -1.0, np.float32)
    sub[:, 1, 3] = (2.0, 2.5, 3.0)
    d, s, n = fuse_views(np.where(sub >= 0, 2, INVALID).astype(np.uint16), sub, [12] * 3, 5, 12, 16, 2)
    assert s[1, 3] == 2.5 and n[1, 3] == 3


# ---- the array scene (tests/test_gpu_groups.py's frame): the CHESS groups' maps, fused ----
def array_scene_groups(oracle):
    h, w, D = 240, 320, 32
    sc = synth.make_array_scene(h, w, 5, 5, D, 7)
    groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
    p = abi.make_params(w, h, D, [(0, 0)] * 4, win_half=4, n_paths=8, lr_gx=-1, subpixel=1)
    p.n_pairs = 0
    ds, ss = [], []
    for grp in groups:
        d, s = oracle.depth_from_array(G.group_params(p, grp, 5), sc["images"][grp[0][0]], [sc["images"][o] for _, o in grp])
        ds.append(d)
        ss.append(s)
    return sc, groups, p, np.array(ds), np.array(ss)


def core_of(gt):
    """at least 6 px from a layer edge and 8 px from the border"""
    edge = np.zeros(gt.shape, bool)
    for dy in range(-6, 7):
        for dx in range(-6, 7):
            edge |= np.roll(np.roll(gt, dy, 0), dx, 1) != gt
    core = ~edge
    core[:8] = core[-8:] = False
    core[:, :8] = core[:, -8:] = False
    return core


def scores(d, gt):
    """(valid share, share of the frame with the true integer disparity, accuracy on accepted core pixels)"""
    v = d != INVALID
    acc = v & core_of(gt)
    return v.mean(), (v & (d == gt)).mean(), (d[acc] == gt[acc]).mean()


def check_ground_truth(sc, refs, own, fused):
    """The oracle, on this frame (tol 1 px, min_support 2): target 12 own group 88.8 % valid / 79.6 % correct / 93.5 % core accuracy, fused
    98.5 / 90.6 / 94.5; target 7 (no group's reference) fused 96.9 / 91.4 / 95.9; target 0 own 89.1 / 83.3 / 96.5, fused 95.9 / 90.0 / 96.7.
    Asserted with margins: at targets 12 and 0 the fused map is correct on >= 5 points more of the frame than the own group, with core
    accuracy at most 1 point lower; at target 7 it is >= 90 % valid, >= 85 % correct and >= 93 % accurate on the core."""
    for t in (12, 0):
        o_valid, o_corr, o_acc = scores(own[t], sc["gt"][t])
        f_valid, f_corr, f_acc = scores(fused[t], sc["gt"][t])
        assert f_corr >= o_corr + 0.05, "target %d: fused correct %.3f vs own %.3f" % (t, f_corr, o_corr)
        assert f_acc >= o_acc - 0.01, "target %d: fused core accuracy %.3f vs own %.3f" % (t, f_acc, o_acc)
        assert f_valid > o_valid
    f_valid, f_corr, f_acc = scores(fused[7], sc["gt"][7])
    assert 7 not in refs
    assert f_valid >= 0.90 and f_corr >= 0.85 and f_acc >= 0.93, (f_valid, f_corr, f_acc)


def test_fusion_finds_the_ground_truth(oracle):
    sc, groups, p, ds, ss = array_scene_groups(oracle)
    refs = [g[0][0] for g in groups]
    own = {t: ds[refs.index(t)] for t in (12, 0)}
    fused = {t: fuse_views(ds, ss, refs, 5, t, 16, 2)[0] for t in (12, 7, 0)}
    check_ground_truth(sc, refs, own, fused)
