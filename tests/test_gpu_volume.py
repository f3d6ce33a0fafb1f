"""CUDA volume pipeline vs the CPU oracle, bit-exact, through the C ABI (libsva_b200.so).  Needs a B200: -m gpu."""
import numpy as np
import pytest

from stereovisionarray_b200 import abi, synth

pytestmark = pytest.mark.gpu

OFF8 = [(-1, -1), (0, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (0, 1), (1, 1)]
OFF15 = [(gx, gy) for gy in range(-1, 3) for gx in range(-1, 3) if (gx, gy) != (0, 0)]


@pytest.fixture(scope="module")
def ctx():
    from stereovisionarray_b200.pipeline import DepthContext
    c = DepthContext(0)
    yield c
    c.close()


CASES = [
    # h, w, D, offsets, kwargs
    (64, 96, 64, [(-1, 0)], dict(win_half=4, n_paths=4, lr_gx=-1)),
    (72, 100, 128, OFF8, dict(win_half=5, n_paths=8, lr_gx=-1)),
    (70, 90, 192, OFF8, dict(win_half=3, n_paths=8, lr_gx=1)),
    (66, 120, 256, [(-1, 0), (1, 0)], dict(win_half=6, n_paths=8, lr_gx=-1, min_disp=3)),
    (60, 88, 32, OFF15, dict(win_half=20, n_paths=8, lr_gx=0)),
    (61, 83, 16, [(0, -1), (2, 1)], dict(win_half=2, n_paths=4, lr_gx=-1, subpixel=0)),
    (50, 70, 96, [(-1, 0), (0, 1)], dict(win_half=13, n_paths=0, lr_gx=-1)),
    (40, 611, 40, OFF8, dict(win_half=7, n_paths=4, lr_gx=-1)),   # several 256-column box strips, win_half % 4 != 0, D % 16 != 0, ragged width
    (150, 300, 24, [(1, 0), (0, -1), (-1, 1)], dict(win_half=9, n_paths=8, lr_gx=1, min_disp=2)),  # several row bands
    (90, 200, 16, [(3, 0), (-3, 1), (1, -4)], dict(win_half=3, n_paths=4, lr_gx=-1)),  # pair offsets beyond +-2: the line-image gather AD kernel
    (48, 260, 64, [(2, -2), (-2, 2), (0, 2), (2, 0)], dict(win_half=4, n_paths=8, lr_gx=1, min_disp=5)),  # |g| = 2 bodies of the image-space AD kernel, min_disp % 4 != 0
    # the register form of the box filter (win_half % 8 == 4) beyond the configurations' 20: one lane, three lanes, seven lanes per window;
    # several strips and row bands, ragged width, D % 16 != 0, the 3 x 3 and 4 x 4 pair-set kernels of K1a with tiles taller than one pass
    (130, 530, 40, OFF8, dict(win_half=12, n_paths=8, lr_gx=-1, min_disp=1)),
    (200, 300, 24, OFF15, dict(win_half=28, n_paths=4, lr_gx=1)),
    (200, 280, 48, OFF8, dict(win_half=20, n_paths=8, lr_gx=-1)),
    (97, 515, 72, [(-1, 0)], dict(win_half=4, n_paths=8, lr_gx=-1)),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_stages_bit_exact(ctx, oracle, case):
    h, w, D, offsets, kw = CASES[case]
    sc = synth.make_scene(h, w, D, offsets, 100 + case, min_disp=kw.get("min_disp", 0), face=(case % 2 == 1))
    p = abi.make_params(w, h, D, offsets, **kw)
    ctx.set_debug(0, 0)
    ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    ctx.run(abi.STAGE_AD)
    A = ctx.download_ad()
    A_o = oracle.ad_volume(p, sc["ref"], sc["others"])
    assert np.array_equal(A, A_o), "AD volume"
    ctx.run(abi.STAGE_BOX)
    Cg = ctx.download_cost()
    C_o, C32_o = oracle.box_cost(p, A_o, raw=True)
    assert np.array_equal(Cg, C_o), "packed cost"
    assert np.array_equal(ctx.download_raw_cost(), C32_o), "raw cost"
    # every single SGM direction on its own, then the full aggregation (debug: last pass also stores S_total)
    if p.n_paths:
        for di in range(p.n_paths):
            ctx.set_debug(0, 1 << di)
            ctx.run(abi.STAGE_SGM)
            assert np.array_equal(ctx.download_sgm(), oracle.sgm_single_path(p, C_o, di)), "direction %d" % di
    ctx.set_debug(1, 0)
    ctx.run(abi.STAGE_SGM)
    S_o = oracle.sgm_aggregate(p, C_o) if p.n_paths else C_o
    if p.n_paths:
        assert np.array_equal(ctx.download_sgm(), S_o), "S total"
    disp, sub = ctx.download_disparity()
    disp_o, sub_o = oracle.wta(p, S_o, sc["mask"])
    assert np.array_equal(disp, disp_o), "integer disparity"
    assert (disp != abi.SVA_DISP_INVALID).sum() > 0 or case == 4
    assert np.max(np.abs(sub - sub_o)) <= 0.05  # stated tolerance (north_star); in practice bit-equal
    assert np.array_equal(sub, sub_o)
    ctx.set_debug(0, 0)


def test_one_call_matches_oracle_pipeline(ctx, oracle):
    h, w, D = 96, 128, 64
    sc = synth.make_scene(h, w, D, OFF8, 7)
    p = abi.make_params(w, h, D, OFF8, win_half=4, n_paths=8, lr_gx=-1)
    disp, sub = ctx.depth_from_array(p, sc["ref"], sc["others"])
    disp_o, sub_o = oracle.depth_from_array(p, sc["ref"], sc["others"])
    assert np.array_equal(disp, disp_o) and np.array_equal(sub, sub_o)
    assert ctx.launches() > 0


def test_stream_of_frames_matches_the_one_call_path(ctx, oracle):
    """capture stream (c4): the double-buffered submit / wait pipeline returns, frame by frame, exactly what the one-call path returns"""
    h, w, D = 80, 136, 64
    p = abi.make_params(w, h, D, OFF8, win_half=4, n_paths=8, lr_gx=-1)
    frames = [synth.make_scene(h, w, D, OFF8, 300 + i, face=(i % 2 == 0)) for i in range(5)]
    outs = [(np.empty((h, w), np.uint16), np.empty((h, w), np.float32)) for _ in frames]
    keep = [abi.image_array(f["others"]) for f in frames]
    tickets = [ctx.stream_submit(p, f["ref"], k, f["mask"], o[0], o[1]) for f, k, o in zip(frames, keep, outs)]
    assert tickets == sorted(tickets) and len(set(tickets)) == len(tickets)
    for t in tickets:
        ctx.stream_wait(t)
    for f, o in zip(frames, outs):
        disp_o, sub_o = oracle.depth_from_array(p, f["ref"], f["others"], f["mask"])
        assert np.array_equal(o[0], disp_o) and np.array_equal(o[1], sub_o)
    # and the context is still good for the one-call path afterwards
    d1, s1 = ctx.depth_from_array(p, frames[0]["ref"], frames[0]["others"], frames[0]["mask"])
    assert np.array_equal(d1, outs[0][0]) and np.array_equal(s1, outs[0][1])


@pytest.mark.parametrize("D,G", [(64, 4), (96, 2), (128, 8)])
def test_slice_direction_row_sharding_emulated_on_one_gpu(ctx, oracle, D, G):
    """dist.slice_sharded_depth's building blocks, with the collectives replaced by local concatenation / addition: 4 disparity slices ->
    slice-major cost volume -> direction shares summed -> row blocks through K3 == the oracle's whole pipeline, bit for bit"""
    import torch
    from stereovisionarray_b200 import dist as sdist
    h, w = 70, 150
    sc = synth.make_scene(h, w, D, OFF8, 41, min_disp=2, face=True)
    p = abi.make_params(w, h, D, OFF8, win_half=5, n_paths=8, lr_gx=-1, min_disp=2)
    alias = lambda ptr, nbytes: torch.as_tensor(sdist._CudaAlias(ptr, nbytes // 4), device="cuda")
    slices = []
    for r in range(G):
        ctx.upload(sdist.slice_params(p, r, G), sc["ref"], sc["others"], sc["mask"])
        ctx.run(abi.STAGE_AD)
        ctx.run(abi.STAGE_BOX)
        ctx.synchronize()
        slices.append(alias(*ctx.cost_device_ptr()).clone())
    call = torch.cat(slices)
    torch.cuda.synchronize()
    ctx.set_params(p)
    rows_per, blocks = sdist.row_blocks(h, G)
    total = None
    for r in range(G):
        sptr, sbytes = ctx.sgm_directions(call.data_ptr(), D // G, sdist.direction_masks(8, G)[r], rows_per * G)
        ctx.synchronize()
        part = alias(sptr, sbytes).clone()
        total = part if total is None else total + part
    torch.cuda.synchronize()
    C_o = oracle.box_cost(p, oracle.ad_volume(p, sc["ref"], sc["others"]))
    S_o = oracle.sgm_aggregate(p, C_o)
    S_g = total.cpu().numpy().view(np.uint16).reshape(rows_per * G, w, D)
    assert np.array_equal(S_g[:h], S_o) and not S_g[h:].any()
    disp = np.empty((h, w), np.uint16)
    sub = np.empty((h, w), np.float32)
    words_row = w * D // 2
    for y0, y1 in blocks:
        if y1 > y0:
            rows = total[y0 * words_row:y1 * words_row].clone()
            torch.cuda.synchronize()
            ctx.wta_rows(rows.data_ptr(), y0, y1 - y0)
            disp[y0:y1], sub[y0:y1] = ctx.download_disparity_rows(y1 - y0)
    disp_o, sub_o = oracle.wta(p, S_o, sc["mask"])
    assert np.array_equal(disp, disp_o) and np.array_equal(sub, sub_o)
    # and the world-size-1 path of the real function (it needs the library on torch's stream)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        d1, s1 = sdist.slice_sharded_depth(ctx, p, sc["ref"], sc["others"], sc["mask"], 0, 1)
    finally:
        ctx.use_own_stream()
    assert np.array_equal(d1, disp_o) and np.array_equal(s1, sub_o)


def test_pair_range_partials_sum_to_full(ctx, oracle):
    """what the pair-sharded multi-GPU reduce relies on: AD partials over disjoint pair ranges add up exactly"""
    h, w, D = 48, 64, 32
    sc = synth.make_scene(h, w, D, OFF15, 9)
    p = abi.make_params(w, h, D, OFF15, win_half=4)
    ctx.upload(p, sc["ref"], sc["others"])
    tot = np.zeros((h, w, D), np.uint32)
    for b, e in [(0, 2), (2, 4), (4, 6), (6, 8), (8, 10), (10, 12), (12, 14), (14, 15)]:
        ctx.set_pair_range(b, e)
        ctx.run(abi.STAGE_AD)
        part = ctx.download_ad()
        assert np.array_equal(part, oracle.ad_volume(p, sc["ref"], sc["others"], b, e))
        tot += part
    assert np.array_equal(tot, oracle.ad_volume(p, sc["ref"], sc["others"]))


def test_bad_arguments_fail_loudly(ctx):
    from stereovisionarray_b200._lib import SvaError
    sc = synth.make_scene(32, 40, 16, [(-1, 0)], 3)
    p = abi.make_params(40, 32, 20, [(-1, 0)], win_half=2)  # D not a multiple of 8
    with pytest.raises(SvaError):
        ctx.upload(p, sc["ref"], sc["others"])
    p = abi.make_params(40, 32, 16, [(-1, 0)], win_half=2)
    with pytest.raises(SvaError):
        ctx.upload(p, sc["ref"][:, :30], sc["others"])  # wrong size
    # a volume the 32-bit element cursors cannot address is refused before anything is allocated
    p = abi.make_params(65536, 32768, 8, [(-1, 0)], win_half=2)
    with pytest.raises(SvaError, match="2\\^32"):
        ctx.upload(p, sc["ref"], sc["others"])
    for bad in (dict(n_paths=3), dict(win_half=0), dict(win_half=57), dict(lr_gx=2), dict(min_disp=-1)):
        with pytest.raises(SvaError):
            ctx.upload(abi.make_params(40, 32, 16, [(-1, 0)], **{**dict(win_half=2), **bad}), sc["ref"], sc["others"])
    p = abi.make_params(40, 32, 16, [(-1, 0)], win_half=2)
    p.p1, p.p2 = 9, 8  # P2 < P1
    with pytest.raises(SvaError):
        ctx.upload(p, sc["ref"], sc["others"])
    # a refused upload leaves the context as it was, and usable
    p = abi.make_params(40, 32, 16, [(-1, 0)], win_half=2, n_paths=4, lr_gx=-1)
    disp, _ = ctx.depth_from_array(p, sc["ref"], sc["others"])
    assert disp.shape == (32, 40)


ROW_BLOCKS = [(67, 96, 64, [(0, 20), (20, 47), (47, 67)]), (90, 140, 128, [(0, 9), (9, 10), (10, 55), (55, 90)]),
              (64, 70, 256, [(0, 33), (33, 64)]), (58, 3840, 192, [(0, 30), (30, 58)])]


@pytest.mark.parametrize("h,w,D,blocks", ROW_BLOCKS)
def test_row_block_pipeline_emulated_on_one_gpu(ctx, h, w, D, blocks):
    """the row-block scheme's building blocks (sva_frame_rows_begin / sva_frame_sgm_rows / sva_frame_wta_rows with the path-line state
    handed from block to block) reproduce the whole-frame aggregation and maps bit for bit; blocks as small as one row, diagonals that
    wrap at a block boundary, rows wide enough for ranged launches"""
    check_row_block_pipeline(ctx, h, w, D, blocks)


def check_row_block_pipeline(ctx, h, w, D, blocks, oracle=None):
    """the row-block pipeline on a second, guarded context against the whole-frame run on ctx (and, given the oracle, that run against
    the oracle: cost volume, aggregation and maps); test_gpu_switches runs it under the A/B switches"""
    import torch
    sc = synth.make_scene(h, w, D, OFF8[:3] if w > 1000 else OFF8, 900 + D, face=True)
    offs = OFF8[:3] if w > 1000 else OFF8
    p = abi.make_params(w, h, D, offs, win_half=4, n_paths=8, lr_gx=-1)
    ctx.set_debug(0, 0)
    ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    ctx.run(abi.STAGE_AD)
    ctx.run(abi.STAGE_BOX)
    ctx.run(abi.STAGE_SGM)
    S_full = ctx.download_sgm()
    d_full, s_full = ctx.download_disparity()
    C_full = ctx.download_cost()
    if oracle is not None:
        C_o = oracle.box_cost(p, oracle.ad_volume(p, sc["ref"], sc["others"]))
        S_o = oracle.sgm_aggregate(p, C_o)
        d_o, s_o = oracle.wta(p, S_o, sc["mask"])
        assert np.array_equal(C_full, C_o) and np.array_equal(S_full, S_o), "whole frame: cost volume / aggregation"
        assert np.array_equal(d_full, d_o) and np.array_equal(s_full, s_o), "whole frame: maps"
    state = [torch.empty(3 * w * D, dtype=torch.int16, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    # the cost volume block by block on a second, poisoned context (bottom block first: a block must not lean on its neighbours' rows)
    from stereovisionarray_b200.pipeline import DepthContext
    blk = DepthContext(0)
    blk.set_guard(True)
    blk.upload(p, sc["ref"], sc["others"], sc["mask"])
    for y0, y1 in reversed(blocks):
        blk.rows_begin(y0, y1 - y0)
        blk.run(abi.STAGE_AD)
        blk.run(abi.STAGE_BOX)
        assert np.array_equal(blk.download_cost()[y0:y1], C_full[y0:y1]), "cost rows %d..%d" % (y0, y1)
    assert blk.check_guards()[1] == 0
    full, ctx = ctx, blk
    for y0, y1 in blocks:
        ctx.sgm_rows(2, y0, y1 - y0)
    for i, (y0, y1) in enumerate(blocks):                      # down sweep: top block first
        ctx.sgm_rows(0, y0, y1 - y0, state[(i + 1) % 2].data_ptr(), state[i % 2].data_ptr())
    for i, (y0, y1) in enumerate(reversed(blocks)):            # up sweep: bottom block first
        ctx.sgm_rows(1, y0, y1 - y0, state[(i + 1) % 2].data_ptr(), state[i % 2].data_ptr())
    ctx.synchronize()
    assert np.array_equal(ctx.download_sgm(), S_full)
    for y0, y1 in blocks:
        ctx.wta_rows(None, y0, y1 - y0)
        d, s = ctx.download_disparity_rows(y1 - y0)
        assert np.array_equal(d, d_full[y0:y1]) and np.array_equal(s, s_full[y0:y1])
    assert blk.check_guards()[1] == 0
    blk.close()


def test_state_guards_of_the_staged_api(ctx, oracle):
    """round-1 review findings, each as the sequence that used to go wrong silently:
    (1) set_params to a further disparity reach than the upload staged the views for, then K1a; (2) a bad frame in the middle of a
    capture stream; (3) a whole-frame SGM over a cost volume of which only a row block was computed"""
    from stereovisionarray_b200._lib import SvaError
    h, w, D = 64, 96, 64
    sc = synth.make_scene(h, w, D, OFF8, 77)
    p = abi.make_params(w, h, D, OFF8, win_half=4, n_paths=8, lr_gx=-1)
    # (1)
    p_small = abi.make_params(w, h, 32, OFF8, win_half=4, n_paths=8, lr_gx=-1)
    ctx.upload(p_small, sc["ref"], sc["others"])
    ctx.set_params(p)  # reaches 32 disparities further than the zero borders of the staged views
    with pytest.raises(SvaError, match="upload the frame again"):
        ctx.run(abi.STAGE_AD)
    ctx.set_params(p_small)  # back inside the staged reach: fine, and exact
    ctx.run(abi.STAGE_AD)
    assert np.array_equal(ctx.download_ad(), oracle.ad_volume(p_small, sc["ref"], sc["others"]))
    p_shift = abi.make_params(w, h, 32, OFF8, win_half=4, n_paths=8, lr_gx=-1, min_disp=1)  # same reach, other column phase
    ctx.set_params(p_shift)
    with pytest.raises(SvaError):
        ctx.run(abi.STAGE_AD)
    # (2)
    frames = [synth.make_scene(h, w, D, OFF8, 500 + i) for i in range(4)]
    outs = [(np.empty((h, w), np.uint16), np.empty((h, w), np.float32)) for _ in frames]
    keep = [abi.image_array(f["others"]) for f in frames]
    tickets = []
    for i, (f, k, o) in enumerate(zip(frames, keep, outs)):
        if i == 2:
            with pytest.raises(SvaError):  # wrong image size: refused before anything of the frames in flight is touched
                ctx.stream_submit(p, f["ref"][:, :50], k, None, o[0], o[1])
        tickets.append(ctx.stream_submit(p, f["ref"], k, None, o[0], o[1]))
    assert tickets == list(range(tickets[0], tickets[0] + 4))
    for t in tickets:
        ctx.stream_wait(t)
    for f, o in zip(frames, outs):
        d_o, s_o = oracle.depth_from_array(p, f["ref"], f["others"])
        assert np.array_equal(o[0], d_o) and np.array_equal(o[1], s_o)
    # (3)
    ctx.upload(p, sc["ref"], sc["others"])
    ctx.rows_begin(16, 20)
    ctx.run(abi.STAGE_AD)
    ctx.run(abi.STAGE_BOX)
    with pytest.raises(SvaError, match="cost volume was not computed for these rows"):
        ctx.sgm_rows(2, 0, 16)
    ctx.rows_begin(0, h)  # "whole frame" again, but C still holds only rows 16..36
    with pytest.raises(SvaError, match="only a row block"):
        ctx.run(abi.STAGE_SGM)
    ctx.run(abi.STAGE_AD)
    ctx.run(abi.STAGE_BOX)
    ctx.run(abi.STAGE_SGM)
    d, s = ctx.download_disparity()
    d_o, s_o = oracle.depth_from_array(p, sc["ref"], sc["others"])
    assert np.array_equal(d, d_o) and np.array_equal(s, s_o)


@pytest.mark.parametrize("h,w,D,offs,kw", [(64, 96, 64, OFF8, dict(win_half=4, n_paths=8, lr_gx=-1)), (57, 203, 40, [(-1, 0), (2, 1), (0, -3)], dict(win_half=2, n_paths=4, lr_gx=1, min_disp=3)),
                                           (70, 150, 192, OFF15, dict(win_half=5, n_paths=8, lr_gx=-1))])
def test_census_cost_mode_bit_exact(ctx, oracle, h, w, D, offs, kw):
    """census cost (north_star names it; no reference counterpart: parity is against the spec frozen in the oracle): Hamming volume, cost
    volume and the maps of the whole pipeline, plus pair-range partials (the pair-sharded reduce) and the one-call path"""
    sc = synth.make_scene(h, w, D, offs, 640 + D, min_disp=kw.get("min_disp", 0), face=True)
    p = abi.make_params(w, h, D, offs, cost_mode=abi.COST_CENSUS, **kw)
    ctx.set_debug(1, 0)
    ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    ctx.run(abi.STAGE_AD)
    A_o = oracle.ad_volume(p, sc["ref"], sc["others"])
    assert np.array_equal(ctx.download_ad(), A_o), "Hamming volume"
    ctx.run(abi.STAGE_BOX)
    C_o = oracle.box_cost(p, A_o)
    assert np.array_equal(ctx.download_cost(), C_o), "cost volume"
    ctx.run(abi.STAGE_SGM)
    S_o = oracle.sgm_aggregate(p, C_o)
    assert np.array_equal(ctx.download_sgm(), S_o)
    disp, sub = ctx.download_disparity()
    disp_o, sub_o = oracle.wta(p, S_o, sc["mask"])
    assert np.array_equal(disp, disp_o) and np.array_equal(sub, sub_o)
    ctx.set_debug(0, 0)
    if len(offs) > 2:
        ctx.set_pair_range(1, len(offs))
        ctx.run(abi.STAGE_AD)
        assert np.array_equal(ctx.download_ad(), oracle.ad_volume(p, sc["ref"], sc["others"], 1, len(offs)))
    d1, s1 = ctx.depth_from_array(p, sc["ref"], sc["others"], sc["mask"])
    assert np.array_equal(d1, disp_o) and np.array_equal(s1, sub_o)
    # and back to SAD on the same context
    p_sad = abi.make_params(w, h, D, offs, **kw)
    d2, _ = ctx.depth_from_array(p_sad, sc["ref"], sc["others"], sc["mask"])
    assert np.array_equal(d2, oracle.depth_from_array(p_sad, sc["ref"], sc["others"], sc["mask"])[0])
