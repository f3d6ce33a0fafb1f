"""A stream of distinct frames through the peer-direct row-block pipeline in the order skewed by chain position (dist.rows_direct_stream_steps),
on one GPU: G local ranks x (G + 1) contexts, one stream per rank, connected with sva_rows_connect_local — the same kernels, flags, acks and
hand-off stores as across GPUs.  Every frame has its own seed (the mask on odd frames), and each context carries three of them, so every link
carries three different frames: a consumer that read the state of the link's previous frame, or a producer that overwrote a state before it was
read, changes the maps (tests/test_rows_stream_hooks.py proves that for every hand-off of these geometries with the oracle)."""
import numpy as np
import pytest

from stereovisionarray_b200 import abi, dist as sdist, synth

pytestmark = pytest.mark.gpu
OFF8 = [(-1, -1), (0, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (0, 1), (1, 1)]

# (height, width, D, G ranks, camera offsets, win_half)
GEOMETRIES = [
    (40, 96, 64, 2, OFF8, 4),
    (70, 120, 64, 3, OFF8, 4),
    (72, 112, 64, 4, OFF8, 4),
    (96, 120, 64, 8, OFF8, 3),         # 12-row blocks: none lies wholly inside the 3-row border band at the top or the bottom
    (32, 3840, 192, 2, OFF8[:3], 4),   # paced rows whose 3 x W lines exceed one resident wave: the row launches are cut by columns
    (60, 200, 160, 3, OFF8, 4),        # D = 160: the marches on the plain NR = 4 layout on 20 lanes, K3 on k_wta_tile
]


def stream_frames(G):
    """frames in the stream: three per context, so every link carries three different frames"""
    return 3 * (G + 1)


def stream_params(geom):
    h, w, D, G, offs, k = geom
    return abi.make_params(w, h, D, offs, win_half=k, n_paths=8, lr_gx=-1)


def stream_frame(geom, i):
    h, w, D, G, offs, k = geom
    return synth.make_scene(h, w, D, offs, 6000 + 97 * GEOMETRIES.index(geom) + i, face=(i % 2 == 1))


_expected = {}
_DONE = object()


def _frames_and_oracle(oracle, geom):
    key = GEOMETRIES.index(geom)
    if key not in _expected:
        p = stream_params(geom)
        frames = [stream_frame(geom, i) for i in range(stream_frames(geom[3]))]
        _expected[key] = frames, [oracle.depth_from_array(p, f["ref"], f["others"], f["mask"]) for f in frames]
    return _expected[key]


class _Ranks:
    """G ranks x (G + 1) guarded contexts; context j of every rank is one link of the chain"""

    def __init__(self, geom, frames):
        self.G = geom[3]
        self.p = stream_params(geom)
        self.ctxs = []
        try:
            self._open(frames)
        except BaseException:
            self.close()
            raise

    def _open(self, frames):
        from stereovisionarray_b200.pipeline import DepthContext
        G, p = self.G, self.p
        for r in range(G):
            row = []
            self.ctxs.append(row)
            for j in range(G + 1):
                c = DepthContext(0)
                row.append(c)
                c.set_guard(True)
                if j:
                    c.set_stream(row[0].get_stream())
                c.rows_open(p, r, G)
        for r in range(G):
            for j, c in enumerate(self.ctxs[r]):
                c.rows_connect_local(self.ctxs[r - 1][j] if r > 0 else None, self.ctxs[r + 1][j] if r < G - 1 else None)
        # every allocation before the stream, masked and unmasked: a buffer that grew inside the stream would synchronise the device
        assert frames[0]["mask"] is None and frames[1]["mask"] is not None
        for f in (frames[1], frames[0]):
            for row in self.ctxs:
                for c in row:
                    y0, n = c.rows_block()
                    c.upload(p, f["ref"], f["others"], f["mask"])
                    c.rows_begin(y0, n); c.run(abi.STAGE_AD); c.run(abi.STAGE_BOX); c.sgm_rows(2, y0, n); c.wta_rows(None, y0, n); c.synchronize()

    def run(self, frames, rank_order, hooked):
        """the stream, each rank's generator advanced one iteration at a time in rank_order -> {frame: [rank's (disp, sub) rows]}"""
        P, p = self.G + 1, self.p
        got = {}

        def upload(ctx, f):
            ctx.upload(p, frames[f]["ref"], frames[f]["others"], frames[f]["mask"])

        def download(r):
            def hook(ctx, f):
                assert ctx is self.ctxs[r][f % P]
                got.setdefault(f, [None] * self.G)[r] = ctx.rows_download()
            return hook

        gens = {r: sdist.rows_direct_stream_steps(self.ctxs[r], r, self.G, len(frames), upload, download(r) if hooked else None) for r in rank_order}
        live = list(rank_order)
        while live:  # one iteration per rank: when a rank blocks in a download, every rank has enqueued the previous iteration
            for r in list(live):
                if next(gens[r], _DONE) is _DONE:
                    live.remove(r)
        return got

    def idle_and_guarded(self):
        for row in self.ctxs:
            for c in row:
                c.synchronize()
        for row in self.ctxs:  # check_guards allocates: only once every stream is idle
            for c in row:
                n, bad = c.check_guards()
                assert n > 0 and bad == 0, "%d canary bytes overwritten" % bad

    def close(self):
        for row in self.ctxs:
            for c in reversed(row):  # the borrowers first: row[0] owns the stream they run on
                c.close()


@pytest.fixture
def ranks_for(oracle):
    made = []

    def make(geom):
        frames, want = _frames_and_oracle(oracle, geom)
        made.append(_Ranks(geom, frames))
        return made[-1], frames, want
    yield make
    for m in made:
        m.close()


def _assemble(parts):
    return np.concatenate([d for d, _ in parts]), np.concatenate([s for _, s in parts])


@pytest.mark.parametrize("reverse", [False, True], ids=["ranks_ascending", "ranks_descending"])
@pytest.mark.parametrize("geom", GEOMETRIES, ids=["%dx%dx%d_G%d" % (g[1], g[0], g[2], g[3]) for g in GEOMETRIES])
def test_every_frame_of_the_skewed_stream_equals_the_oracle(ranks_for, geom, reverse):
    """the download hook collects every frame from its context before the context is reused: all 3 (G + 1) frames, bit for bit against the
    oracle, integer and sub-pixel maps; the enqueue order of the ranks inside an iteration must not matter"""
    rk, frames, want = ranks_for(geom)
    order = list(reversed(range(rk.G))) if reverse else list(range(rk.G))
    got = rk.run(frames, order, hooked=True)
    rk.idle_and_guarded()
    assert sorted(got) == list(range(len(frames)))
    for f in range(len(frames)):
        disp, sub = _assemble(got[f])
        assert np.array_equal(disp, want[f][0]), "frame %d: integer disparity" % f
        assert np.array_equal(sub, want[f][1]), "frame %d: sub-pixel" % f


@pytest.mark.parametrize("geom", GEOMETRIES, ids=["%dx%dx%d_G%d" % (g[1], g[0], g[2], g[3]) for g in GEOMETRIES])
def test_free_running_skewed_stream_leaves_the_last_frames_right(ranks_for, geom):
    """no download hook and no host synchronisation until the stream is drained: the last G + 1 frames, still in their contexts, equal the
    oracle — each differs from the frame its link carried before"""
    rk, frames, want = ranks_for(geom)
    P = rk.G + 1
    assert rk.run(frames, list(range(rk.G)), hooked=False) == {}
    rk.idle_and_guarded()
    for f in range(len(frames) - P, len(frames)):
        assert not np.array_equal(want[f][0], want[f - P][0])
        disp, sub = _assemble([rk.ctxs[r][f % P].rows_download() for r in range(rk.G)])
        assert np.array_equal(disp, want[f][0]), "frame %d: integer disparity" % f
        assert np.array_equal(sub, want[f][1]), "frame %d: sub-pixel" % f
