"""The stream of frames in the order skewed by chain position (dist.rows_direct_stream_steps) on CPU: where the upload and download hooks are
called, that a host blocking in them never waits for work nobody has enqueued yet, and — with the oracle — that the GPU test of this stream
(tests/test_gpu_rows_stream.py) can see every stale hand-off it is meant to catch."""
import numpy as np
import pytest

from stereovisionarray_b200 import dist as sdist
from test_gpu_rows_stream import GEOMETRIES, stream_frame, stream_frames, stream_params

_DONE = object()


class _Ctx:
    """stands in for a DepthContext: logs its parts; a context's k-th part 0 is frame slot + k * (world + 1)"""

    def __init__(self, log, rank, slot, P):
        self.log, self.rank, self.slot, self.P = log, rank, slot, P
        self.started = 0

    def rows_run_part(self, part):
        if part == 0:
            self.started += 1
        self.log.append(("part", self.rank, part, self.slot + (self.started - 1) * self.P))


def _hooks(log):
    return (lambda ctx, f: log.append(("upload", ctx.rank, ctx.slot, f)),
            lambda ctx, f: log.append(("download", ctx.rank, ctx.slot, f)))


def _waits(rank, world, part, f):
    """what sva_rows_run_part(part) of frame f on `rank` waits for, as (rank, part, frame) of the neighbour's part that signals it.  The sweep
    that reaches a rank first is its part 1 (csrc/sva_dist.cu: down_first); a sweep waits for the state from the rank it comes from (same
    frame) and for the ack of the rank it goes to (the link's previous frame, f - world - 1)"""
    if part == 0:
        return []
    down_first = lambda r: r < (world + 1) // 2
    down = (part == 1) == down_first(rank)
    part_of = lambda r: 1 if down == down_first(r) else 2
    frm, to = (rank - 1, rank + 1) if down else (rank + 1, rank - 1)
    out = []
    if 0 <= frm < world:
        out.append((frm, part_of(frm), f))
    if 0 <= to < world and f - world - 1 >= 0:
        out.append((to, part_of(to), f - world - 1))
    return out


@pytest.mark.parametrize("world", range(1, 9))
def test_stream_hooks_are_called_where_the_contexts_allow(world):
    P = world + 1
    for frames in range(1, 3 * P + 3):
        for rank in range(world):
            log = []
            ctxs = [_Ctx(log, rank, j, P) for j in range(P)]
            up, down = _hooks(log)
            iterations = 0
            for _ in sdist.rows_direct_stream_steps(ctxs, rank, world, frames, up, down):
                iterations += 1
            assert iterations == frames + world
            at = {e: i for i, e in enumerate(log)}
            assert len(at) == len(log) == 5 * frames, "every hook and part exactly once per frame"
            part = lambda k, f: at[("part", rank, k, f)]
            for f in range(frames):
                slot = f % P
                assert part(0, f) < part(1, f) < part(2, f)
                assert at[("upload", rank, slot, f)] < part(0, f), "upload before the frame's part 0"
                assert at[("download", rank, slot, f)] > part(2, f), "download after the frame is complete"
                if f >= P:
                    assert part(2, f - P) < at[("upload", rank, slot, f)], "no upload into a context whose frame is still running"
                if f + P < frames:
                    assert at[("download", rank, slot, f)] < min(at[("upload", rank, slot, f + P)], part(0, f + P)), "download before the context is reused"
            last_part = max(i for i, e in enumerate(log) if e[0] == "part")
            flushed = [e[3] for e in log[last_part + 1:]]
            assert flushed == list(range(max(0, frames - P), frames)), "the final flush: exactly the frames still in the contexts, in frame order"
            assert all(e[0] == "download" for e in log[last_part + 1:])

            plain = []
            sdist.rows_direct_stream([_Ctx(plain, rank, j, P) for j in range(P)], rank, world, frames, *_hooks(plain))
            assert plain == log, "the plain call enqueues what the generator does"
            bare = []
            sdist.rows_direct_stream([_Ctx(bare, rank, j, P) for j in range(P)], rank, world, frames)
            assert bare == [e for e in log if e[0] == "part"], "no hooks: the same parts"
    with pytest.raises(ValueError):
        next(sdist.rows_direct_stream_steps([None] * world, 0, world, 4))


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("reverse", [False, True])
def test_a_host_blocking_in_a_hook_never_waits_for_unenqueued_work(world, reverse):
    """one process plays every rank and advances the ranks' generators round-robin.  Whenever a hook runs (where a download synchronises),
    every wait any rank has enqueued has its producer enqueued already, so blocking there cannot sit out the hand-off time-out"""
    P = world + 1
    frames = 3 * P + 2
    log, calls = [], [0]

    def hook(ctx, f):
        enqueued = {e[1:] for e in log}
        for r, k, g in enqueued:
            for w in _waits(r, world, k, g):
                assert w in enqueued, "hook of rank %d, frame %d: rank %d's part %d of frame %d waits for %s, not enqueued yet" % (ctx.rank, f, r, k, g, w)
        calls[0] += 1

    order = list(reversed(range(world))) if reverse else list(range(world))
    gens = {r: sdist.rows_direct_stream_steps([_Ctx(log, r, j, P) for j in range(P)], r, world, frames, hook, hook) for r in order}
    live = list(order)
    while live:
        for r in list(live):
            if next(gens[r], _DONE) is _DONE:
                live.remove(r)
    assert calls[0] == 2 * frames * world
    enqueued = {e[1:] for e in log}
    assert all(w in enqueued for e in enqueued for w in _waits(e[0], world, e[1], e[2])) and len(enqueued) == 3 * frames * world


DOWN, UP = (0, 4, 5), (1, 6, 7)  # the oracle's row-sweeping directions: the down-sweeping and the up-sweeping group


def _boundary_states(orc, p, C, blocks):
    """{direction: {b: L at the boundary between blocks b - 1 and b, as the sweep crosses it}} for b = 1 .. G - 1: what a rank hands on"""
    G = len(blocks)
    scratch = np.zeros((p.height, p.width, p.num_disp), np.uint16)
    out = {}
    for di in DOWN + UP:
        out[di], prev = {}, None
        for b in (range(G) if di in DOWN else reversed(range(G))):
            y0, y1 = blocks[b]
            state = np.zeros((p.width, p.num_disp), np.uint16)
            orc.sgm_rows(p, C, di, y0, y1 - y0, prev, scratch, state)
            prev = state
            edge = b + 1 if di in DOWN else b
            if 0 < edge < G:
                out[di][edge] = state
    return out


def _blind_hand_offs(orc, geom):
    """every (sweep, boundary, frame) of the stream whose maps do NOT change when the consumer reads the state that the link's previous frame
    (f - G - 1) left at that boundary instead of its own — only the consuming block's rows are recomputed, the rest of the frame is right"""
    h, w, D, G, offs, k = geom
    P, F = G + 1, stream_frames(G)
    p = stream_params(geom)
    _, blocks = sdist.row_blocks(h, G)
    frames, costs, states = [], [], []
    for i in range(F):
        sc = stream_frame(geom, i)
        C = orc.box_cost(p, orc.ad_volume(p, sc["ref"], sc["others"]))
        frames.append(sc); costs.append(C); states.append(_boundary_states(orc, p, C, blocks))
    blind = []
    good, bad = np.zeros((h, w, D), np.uint16), np.zeros((h, w, D), np.uint16)
    for f in range(P, F):
        S = orc.sgm_aggregate(p, costs[f])
        maps = orc.wta(p, S, frames[f]["mask"])
        for name, group in (("down", DOWN), ("up", UP)):
            for b in range(1, G):
                y0, y1 = blocks[b] if group is DOWN else blocks[b - 1]
                S_stale = S.astype(np.int64)
                for di in group:
                    good[y0:y1] = 0; bad[y0:y1] = 0
                    orc.sgm_rows(p, costs[f], di, y0, y1 - y0, states[f][di][b], good, None)
                    orc.sgm_rows(p, costs[f], di, y0, y1 - y0, states[f - P][di][b], bad, None)
                    S_stale[y0:y1] += bad[y0:y1].astype(np.int64) - good[y0:y1]
                assert S_stale.min() >= 0 and S_stale.max() < 1 << 16
                stale = orc.wta(p, S_stale.astype(np.uint16), frames[f]["mask"])
                if np.array_equal(stale[0], maps[0]) and np.array_equal(stale[1], maps[1]):
                    blind.append((name, b, f))
    return blind


@pytest.mark.parametrize("geom", GEOMETRIES, ids=["%dx%dx%d_G%d" % (g[1], g[0], g[2], g[3]) for g in GEOMETRIES])
def test_every_hand_off_of_the_gpu_stream_test_is_observable(oracle, geom):
    """for every geometry of tests/test_gpu_rows_stream.py, every boundary of both sweeps and every frame that follows another on its link:
    a consumer that read the previous frame's state there changes the frame's integer or sub-pixel map.  A stale hand-off can leave the maps
    alone (a 1-row block inside the border band: its S changes, its pixels are invalid anyway) — a geometry with such a blind boundary would
    let the GPU test pass over a broken flag, so it must not be in the list"""
    assert _blind_hand_offs(oracle, geom) == []
