"""Every kernel variant the A/B switches of DESIGN §8a select, against the oracle, on guarded contexts.  Needs a B200: -m gpu.

The switches are environment variables read at sva_create (SVA_SGM_NO_* also where the SGM launches are planned), so each check sets its
variables for the whole test and creates a fresh context.  SWITCHES has one entry per variant: the variables, the cases that reach the
variant, the stages it can change and a witness — what the timing labels of one production run must show for the switch to have taken
effect — where the library exposes one.  tests/test_switch_inventory.py checks that every switch the library reads has an entry here."""
import re
import zlib
from typing import Callable, NamedTuple, Optional

import numpy as np
import pytest

from stereovisionarray_b200 import abi, synth
from test_gpu_guard import WIDE
from test_gpu_volume import CASES, OFF8, OFF15, ROW_BLOCKS, check_row_block_pipeline

pytestmark = pytest.mark.gpu

PAIR2 = [(-1, 0), (1, 0)]

# geometries by name: h, w, D, pair offsets, make_params keywords
GEOM = {"c%d" % i: c for i, c in enumerate(CASES)}
GEOM.update({"wide%d" % i: c for i, c in enumerate(WIDE[:4])})
GEOM["mblk"] = WIDE[4]  # 3840 x 260: each row-sweeping group marched in two row blocks, each cut by columns
GEOM.update({
    "d160": (64, 200, 160, OFF8, dict(win_half=4, n_paths=8, lr_gx=-1)),  # SGM with NR = 4 on 20 lanes, K3 on k_wta_tile
    # forced pacing: >= 150 rows give 15 or more rounds of 9 rows (more than any window tested), >= 300 columns give a resident wave of
    # at least one line per CTA (pacing needs W >= grid)
    "pace64": (160, 320, 64, OFF8, dict(win_half=4, n_paths=8, lr_gx=-1)),
    "pace128": (150, 300, 128, PAIR2, dict(win_half=5, n_paths=8, lr_gx=1, min_disp=2)),
    "pace192": (152, 310, 192, OFF8, dict(win_half=3, n_paths=8, lr_gx=-1)),
    "pace256": (150, 300, 256, [(-1, 0), (0, -1)], dict(win_half=6, n_paths=8, lr_gx=0)),
    # the capture stream at a small width and at a width where the SGM launches are paced (W * D * 4 >= 768 KB)
    "stream136": (80, 136, 64, OFF8, dict(win_half=4, n_paths=8, lr_gx=-1)),
    "stream1024": (64, 1024, 192, OFF8, dict(win_half=4, n_paths=8, lr_gx=-1)),
})
# K3's register march for each D it exists for x the three LR modes; 333 columns end every segment length in a partial segment
WTA = []
for _i, (_D, _lr) in enumerate((D, lr) for D in (64, 128, 192, 256) for lr in (-1, 0, 1)):
    WTA.append("wta%d%s" % (_D, "lr-+"[_lr + 1] if _lr else "lr0"))
    GEOM[WTA[-1]] = (44, 333, _D, PAIR2, dict(win_half=3, n_paths=8 if _i % 2 else 4, lr_gx=_lr, min_disp=_i % 4 * 2 + (_i % 3)))
ROWS = ["rows%d" % i for i in range(len(ROW_BLOCKS))]  # the row-block pipeline of test_gpu_volume (check_row_block_pipeline)


def _face(name):
    return not (name.startswith("c") and int(name[1:]) % 2 == 0)  # as test_stages_bit_exact: the even CASES without a mask


class Sw(NamedTuple):
    env: dict                       # variables set for the whole test
    cases: tuple                    # names in GEOM / ROWS that reach the variant
    stages: str                     # what the variant can change: K1a, K1b, K2 (SGM), K3, stream
    witness: Optional[Callable]     # (timing labels, params) -> bool; None: the library exposes no trace of the choice
    why: str = ""                   # where witness is None: why the cases reach the variant
    dirs: tuple = ()                # cases on which every single SGM direction is checked too
    kind: str = "stages"            # "stream": the capture stream over several distinct frames


def _sgm_args(labels):
    """template arguments <NR, PF, FULL, STORE, BL, ROWS, BULK> of every k_sgm_acc launch"""
    return [[int(a) for a in re.match(r"k_sgm_acc<([^>]*)>", l).group(1).split(",")] for l in labels if l.startswith("k_sgm_acc<")]


def _ranged(labels, group):
    return sum(1 for l in labels if re.search(r"/red_%s\d_ranged$" % group, l))


def _bulk(v):
    return lambda L, p: bool(_sgm_args(L)) and all(a[6] == v for a in _sgm_args(L))


def _stores(L):
    return [l for l in L if "/store_" in l]


_one_hstore = lambda L, p: len(_stores(L)) == 1 and _stores(L)[0].endswith("/store_horizontal1")
_no_ranged = lambda L, p: bool(_sgm_args(L)) and not any("_ranged" in l for l in L)

BOX4 = ("c0", "c11", "c13", "c12")  # win_half 4, 12, 20, 28: the register form of K1b (win_half % 8 == 4) with 1, 3, 5, 7 lanes per window
BULK_D = ("c5", "c0", "c1", "d160", "c2", "c3")  # D = 16 (NR 1, 8 lanes, 4 paths), 64 (NR 1, full warp, 4 paths), 128 (NR 2), 160 (NR 4, 20 lanes), 192 / 256 (block layout, 24 / 32 lanes)
PACE_D = ("pace64", "pace128", "pace192", "pace256")

SWITCHES = [
    # K1a (k_ad2.cu): the tile height the frame-size rule picks only where the grid keeps five waves (full-size frames); OFF8 runs 8-row
    # passes (c1; c2 with 70 rows ends in a partial tile), OFF15 16-row passes (c4, c12), c0 the one-pair set, c10 the generic kernel,
    # rows1 row blocks that start at rows 9, 10 and 55
    *[Sw({"SVA_AD_TH": v}, ("c1", "c2", "c4", "c12", "c0", "c10", "rows1"), "K1a", None, "tall tiles exist only above the small frames' five-wave limit")
      for v in ("16", "24", "32", "48")],
    Sw({"SVA_AD_SET": "0"}, ("c1", "c4", "c0"), "K1a", lambda L, p: "k_ad_tile" in L and "k_ad_tile_set" not in L),
    Sw({"SVA_AD_GATHER": "1"}, ("c1", "c3"), "K1a", lambda L, p: "k_ad_planar" in L and not any(l.startswith("k_ad_tile") for l in L)),
    # K1b (k_box.cu)
    Sw({"SVA_BOX_SHFL": "0"}, BOX4, "K1b", lambda L, p: "k_box_planar" in L and "k_box_planar_shfl" not in L),
    *[Sw({"SVA_BOX_OCC": v}, BOX4 + ("c14",), "K1b", None, "the cost model picks 2 or 3 CTAs per SM per launch; the switch pins one (c14: ragged width)")
      for v in ("2", "3")],
    # 4096 bands: one row per band, shorter than any window (a band the cost model never picks)
    *[Sw({"SVA_BOX_BANDS": v}, ("c0", "c13", "c7", "rows0"), "K1b", None, "the band count is otherwise the cost model's (c7: the prefix-table kernel, k = 7)")
      for v in ("1", "2", "5", "4096")],
    Sw({"SVA_BOX_L2": "1"}, ("c0", "c13"), "K1b", None, "the eviction hints are compiled into the register form, which c0 (k = 4) and c13 (k = 20) run"),
    # K2 (k_sgm.cu)
    *[Sw({"SVA_SGM_BULK": v}, BULK_D + tuple(ROWS) + ("mblk",), "K2", _bulk(int(v)), dirs=BULK_D) for v in ("1", "2")],
    *[Sw({"SVA_SGM_PACE": "1", "SVA_SGM_PACE_WINDOW": wnd}, PACE_D, "K2", None, "frames this small are not paced by default; their rounds exceed the window")
      for wnd in ("1", "2", "4")],
    Sw({"SVA_SGM_PACE": "0"}, ("wide1", "mblk"), "K2", _no_ranged),
    Sw({"SVA_SGM_DIAG_SPLIT": "0"}, ("c1", "c2", "wide0"), "K2", None, "unpaced 8-path frames run the split diagonal march by default"),
    Sw({"SVA_SGM_DIAG_SPLIT": "2"}, ("wide1",), "K2", None, "wide1 is paced: by default its diagonals take the generic march"),
    Sw({"SVA_SGM_DIAG_SPLIT": "2", "SVA_SGM_PACE": "1"}, ("pace64", "pace192"), "K2", None, "forced pacing with the split diagonal march"),
    *[Sw({"SVA_SGM_HSTORE": "0", "SVA_PREZERO": z}, ("c1", "c2", "wide1"), "K2", lambda L, p: not _stores(L)) for z in ("0", "1")],
    *[Sw({"SVA_SGM_HSTORE": v}, ("c1", "wide1"), "K2", _one_hstore) for v in ("1", "3")],
    Sw({"SVA_PREZERO": "0"}, ("c0", "c5"), "K2", None, "4-path frames zero S next to K1 by default; 0 = a memset in line"),
    Sw({"SVA_SGM_SPLIT": "0"}, ("c1", "c2", "wide1"), "K2", lambda L, p: any(l.endswith("/red_mixed8") for l in L)),
    Sw({"SVA_SGM_NO_BLK": "1"}, ("c2", "c3", "pace256"), "K2",
       lambda L, p: any(a[0] == 4 for a in _sgm_args(L)) and all(a[4] == 0 for a in _sgm_args(L))),
    Sw({"SVA_SGM_NO_RANGED": "1"}, ("mblk",), "K2", _no_ranged),
    # without the column cut the group is one set of ranged launches for the whole frame: 3 W lines in launches of at least W lines = 1 to
    # 3 per group, against one such set per row block (two blocks here) by default
    Sw({"SVA_SGM_NO_COLSPLIT": "1"}, ("mblk",), "K2", lambda L, p: 1 <= _ranged(L, "down") <= 3 and 1 <= _ranged(L, "up") <= 3),
    Sw({}, ("mblk",), "K2", lambda L, p: _ranged(L, "down") >= 4 and _ranged(L, "up") >= 4),
    # K3 (k_wta.cu): 0 = the shared-memory tile kernel (+ the LR check where lr_gx != 0); the segment lengths the frame-size rule never picks
    # at these sizes (160 with D = 192 leaves a partial rotation in every segment; 4096 = one segment per row)
    Sw({"SVA_WTA_SEG": "0"}, tuple(WTA), "K3",
       lambda L, p: "k_wta_tile" in L and "k_wta_seg" not in L and ("k_lr_check" in L) == (p.lr_gx != 0)),
    *[Sw({"SVA_WTA_SEG": v}, tuple(WTA), "K3", lambda L, p: "k_wta_seg" in L and "k_wta_tile" not in L) for v in ("16", "48", "96", "160", "4096")],
    # the capture stream (sva_api.cu): K1a of the next frame next to this frame's SGM, not at paced widths unless 2
    *[Sw({"SVA_STREAM_AD_AHEAD": v}, ("stream136", "stream1024"), "stream", None, "five distinct frames in flight, each checked", kind="stream")
      for v in ("0", "1", "2")],
]


def _entry_id(e):
    return "-".join("%s=%s" % (k[4:], v) for k, v in e.env.items()) or "default"


_ORACLE = {}  # (case, what) -> oracle result: many switch values share a case, and the oracle is the slow part


def _scene(name):
    h, w, D, offs, kw = GEOM[name]
    return synth.make_scene(h, w, D, offs, zlib.crc32(name.encode()) % 10000, min_disp=kw.get("min_disp", 0), face=_face(name))


def _expected(oracle, name):
    if name not in _ORACLE:
        h, w, D, offs, kw = GEOM[name]
        sc = _scene(name)
        p = abi.make_params(w, h, D, offs, **kw)
        A = oracle.ad_volume(p, sc["ref"], sc["others"])
        C = oracle.box_cost(p, A)
        S = oracle.sgm_aggregate(p, C) if p.n_paths else C
        _ORACLE[name] = dict(sc=sc, p=p, A=A, C=C, S=S, maps=oracle.wta(p, S, sc["mask"]))
    return _ORACLE[name]


def _single_path(oracle, name, d):
    if (name, d) not in _ORACLE:
        e = _expected(oracle, name)
        _ORACLE[name, d] = oracle.sgm_single_path(e["p"], e["C"], d)
    return _ORACLE[name, d]


def _clean(c):
    n, bad = c.check_guards()
    assert n > 0, "no guarded buffers: the guard switch did not take"
    assert bad == 0, "%d canary bytes overwritten (out-of-bounds write)" % bad


def _new_ctx(monkeypatch, env):
    from stereovisionarray_b200.pipeline import DepthContext
    for k, v in env.items():
        monkeypatch.setenv(k, v)  # kept for the whole test: SVA_SGM_NO_* are read at launch time
    c = DepthContext(0)
    c.set_guard(True)
    return c


def _labels(ctx):
    return [n for n, _ in ctx.kernel_times(abi.STAGE_ALL)]


def _check_stages(ctx, oracle, e, name):
    x = _expected(oracle, name)
    p, sc = x["p"], x["sc"]
    ctx.set_debug(0, 0)
    ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    ctx.run(abi.STAGE_AD)
    if "K1a" in e.stages:
        assert np.array_equal(ctx.download_ad(), x["A"]), "AD volume"
    ctx.run(abi.STAGE_BOX)
    assert np.array_equal(ctx.download_cost(), x["C"]), "cost volume"
    if name in e.dirs and p.n_paths:
        for d in range(p.n_paths):
            ctx.set_debug(0, 1 << d)  # one direction alone: the storing launch
            ctx.run(abi.STAGE_SGM)
            assert np.array_equal(ctx.download_sgm(), _single_path(oracle, name, d)), "direction %d" % d
    ctx.set_debug(1, 0)
    ctx.run(abi.STAGE_SGM)
    if p.n_paths:
        assert np.array_equal(ctx.download_sgm(), x["S"]), "S total"
    disp, sub = ctx.download_disparity()
    assert np.array_equal(disp, x["maps"][0]), "integer disparity"
    assert np.array_equal(sub, x["maps"][1]), "sub-pixel disparity"
    ctx.set_debug(0, 0)
    # the production order: the launches set_debug does not reproduce (S written by the first horizontal launch, the side stream, ...)
    d1, s1 = ctx.depth_from_array(p, sc["ref"], sc["others"], sc["mask"])
    assert np.array_equal(d1, x["maps"][0]) and np.array_equal(s1, x["maps"][1]), "one-call path"
    return p


STAGE_CHECKS = [(e, c) for e in SWITCHES if e.kind == "stages" for c in e.cases]


@pytest.mark.parametrize("e,case", STAGE_CHECKS, ids=["%s-%s" % (_entry_id(e), c) for e, c in STAGE_CHECKS])
def test_switch_variant_matches_oracle(monkeypatch, oracle, e, case):
    ctx = _new_ctx(monkeypatch, e.env)
    try:
        if case in ROWS:
            h, w, D, blocks = ROW_BLOCKS[ROWS.index(case)]
            check_row_block_pipeline(ctx, h, w, D, blocks, oracle)  # the block contexts are created under the same switches
            p = ctx.params
        else:
            p = _check_stages(ctx, oracle, e, case)
        if e.witness is not None:
            L = _labels(ctx)  # one more production run, timed launch by launch
            assert e.witness(L, p), "the switch did not take effect: %s" % L
            if case not in ROWS:
                x = _expected(oracle, case)
                d, s = ctx.download_disparity()
                assert np.array_equal(d, x["maps"][0]) and np.array_equal(s, x["maps"][1])
        _clean(ctx)
    finally:
        ctx.close()


STREAM_CHECKS = [(e, c) for e in SWITCHES if e.kind == "stream" for c in e.cases]


@pytest.mark.parametrize("e,case", STREAM_CHECKS, ids=["%s-%s" % (_entry_id(e), c) for e, c in STREAM_CHECKS])
def test_switch_capture_stream_matches_oracle(monkeypatch, oracle, e, case):
    """as test_stream_of_frames_matches_the_one_call_path: distinct frames through sva_stream_submit / sva_stream_wait, every frame's maps
    against the oracle"""
    h, w, D, offs, kw = GEOM[case]
    p = abi.make_params(w, h, D, offs, **kw)
    frames = [synth.make_scene(h, w, D, offs, 330 + i, face=(i % 2 == 0)) for i in range(6)]
    if (case, "stream") not in _ORACLE:
        _ORACLE[case, "stream"] = [oracle.depth_from_array(p, f["ref"], f["others"], f["mask"]) for f in frames]
    expected = _ORACLE[case, "stream"]
    ctx = _new_ctx(monkeypatch, e.env)
    try:
        outs = [(np.empty((h, w), np.uint16), np.empty((h, w), np.float32)) for _ in frames]
        keep = [abi.image_array(f["others"]) for f in frames]
        tickets = [ctx.stream_submit(p, f["ref"], k, f["mask"], o[0], o[1]) for f, k, o in zip(frames, keep, outs)]
        for t in tickets:
            ctx.stream_wait(t)
        for i, (o, (d_o, s_o)) in enumerate(zip(outs, expected)):
            assert np.array_equal(o[0], d_o) and np.array_equal(o[1], s_o), "frame %d" % i
        d1, s1 = ctx.depth_from_array(p, frames[1]["ref"], frames[1]["others"], frames[1]["mask"])
        assert np.array_equal(d1, expected[1][0]) and np.array_equal(s1, expected[1][1])
        _clean(ctx)
    finally:
        ctx.close()


@pytest.mark.parametrize("var,value", [("SVA_BOX_OCC", "1"), ("SVA_SGM_SPLIT", "off"), ("SVA_SGM_PACE_WINDOW", "0"), ("SVA_SGM_BULK", "3"),
                                       ("SVA_SGM_HSTORE", "4"), ("SVA_SGM_DIAG_SPLIT", "-1"), ("SVA_SGM_PACE", "2"), ("SVA_WTA_SEG", "-2"),
                                       ("SVA_AD_TH", "-8"), ("SVA_BOX_BANDS", "2x"), ("SVA_AD_SET", ""), ("SVA_STREAM_AD_AHEAD", "3"),
                                       ("SVA_SGM_NO_BLK", "0")])
def test_bad_switch_value_is_refused(monkeypatch, var, value):
    """a value outside the documented set fails sva_create, naming the variable, instead of running some other schedule (SVA_BOX_OCC=1
    used to leave K1b without a launch shape: no cost volume written, and the stale one used).  No kernel runs here."""
    from stereovisionarray_b200._lib import SvaError
    from stereovisionarray_b200.pipeline import DepthContext
    monkeypatch.setenv(var, value)
    with pytest.raises(SvaError, match=var) as ei:
        DepthContext(0)
    assert ei.value.code == abi.SVA_ERR_BAD_ARG
    monkeypatch.delenv(var)
    DepthContext(0).close()  # and the next create, without it, works


@pytest.mark.parametrize("value", ["abc", "0", "-5"])
def test_bad_rows_timeout_is_refused(monkeypatch, value):
    """SVA_ROWS_TIMEOUT_MS of text or <= 0 would be a time-out that fires at once: sva_rows_open refuses it (the local two-rank setup of
    test_rows_direct_times_out_instead_of_hanging)"""
    from stereovisionarray_b200._lib import SvaError
    from stereovisionarray_b200.pipeline import DepthContext
    monkeypatch.setenv("SVA_ROWS_TIMEOUT_MS", value)
    h, w, D = 48, 64, 64
    sc = synth.make_scene(h, w, D, OFF8, 5)
    p = abi.make_params(w, h, D, OFF8, win_half=3, n_paths=8, lr_gx=-1)
    a, b = DepthContext(0), DepthContext(0)
    try:
        for r, c in enumerate((a, b)):
            c.upload(p, sc["ref"], sc["others"])
            with pytest.raises(SvaError, match="SVA_ROWS_TIMEOUT_MS") as ei:
                c.rows_open(p, r, 2)
            assert ei.value.code == abi.SVA_ERR_BAD_ARG
        monkeypatch.setenv("SVA_ROWS_TIMEOUT_MS", "5000")
        a.rows_open(p, 0, 2)
    finally:
        a.close(); b.close()
