"""The skewed row-pipeline stream behind one C call per frame (sva_rows_stream_*, pipeline.RowsStream), on one GPU: G local ranks x (G + 1)
guarded contexts, one stream per rank, linked with sva_rows_connect_local, and one RowsStream per rank, the ranks advanced one call each,
round-robin — a process that blocks where the skewed order forbids it dead-locks here.  The frames, geometries and oracle results are those of
tests/test_gpu_rows_stream.py, where the Python driver (dist.rows_direct_stream_steps) runs the same order."""
import random

import numpy as np
import pytest

from stereovisionarray_b200 import abi
from test_gpu_rows_stream import GEOMETRIES, _frames_and_oracle, _Ranks, stream_params

pytestmark = pytest.mark.gpu
IDS = ["%dx%dx%d_G%d" % (g[1], g[0], g[2], g[3]) for g in GEOMETRIES]
SENTINEL_D = 0x1234


class _Streams:
    """G ranks x (G + 1) guarded contexts (context j of every rank is one chain) and a RowsStream per rank"""

    def __init__(self, geom, connect=True):
        self.G = geom[3]
        self.p = stream_params(geom)
        self.ctxs, self.streams = [], []
        try:
            self._open(connect)
        except BaseException:
            self.close()
            raise

    def _open(self, connect):
        from stereovisionarray_b200.pipeline import DepthContext, RowsStream
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
        if connect:
            self.connect()
        for r in range(G):
            self.streams.append(RowsStream(self.ctxs[r], p))

    def connect(self):
        G = self.G
        for r in range(G):
            for j, c in enumerate(self.ctxs[r]):
                c.rows_connect_local(self.ctxs[r - 1][j] if r > 0 else None, self.ctxs[r + 1][j] if r < G - 1 else None)

    def launches(self):
        return [[c.launches() for c in row] for row in self.ctxs]

    def guards(self):
        """-> per context (guarded buffers, overwritten canary bytes); synchronises the device"""
        return [[c.check_guards() for c in row] for row in self.ctxs]

    def outputs(self, n):
        """per rank and frame: sentinel-filled (disp, subpix) rows, so a buffer the library never wrote shows"""
        out = []
        for r in range(self.G):
            rows = self.streams[r].rows
            out.append([(np.full((rows, self.p.width), SENTINEL_D, np.uint16), np.full((rows, self.p.width), np.nan, np.float32)) for _ in range(n)])
        return out

    def close(self):
        for s in self.streams:
            s.close()
        for row in self.ctxs:
            for c in reversed(row):  # the borrowers first: row[0] owns the stream
                c.close()


@pytest.fixture
def streams_for(oracle):
    made = []

    def make(geom, connect=True):
        frames, want = _frames_and_oracle(oracle, geom)
        made.append(_Streams(geom, connect))
        return made[-1], frames, want
    yield make
    for m in made:
        m.close()


def _pinned(frames):
    """the frames in page-locked host memory (torch pin_memory tensors viewed as numpy)"""
    import torch

    def pin(a):
        return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    return [{"ref": pin(f["ref"]), "others": [pin(o) for o in f["others"]], "mask": pin(f["mask"])} for f in frames]


def _submit_round(st, order, frame, outs, f):
    """one submit per rank, round-robin, of frame `f` -> the tickets"""
    tickets = []
    for r in order:
        d, s = outs[r][f]
        tickets.append(st.streams[r].submit(frame["ref"], frame["others"], frame["mask"], d, s))
    return tickets


def _raises(code, fn):
    from stereovisionarray_b200._lib import SvaError
    with pytest.raises(SvaError) as e:
        fn()
    assert e.value.code == code, str(e.value)


def _check_frame(outs, want, f, G):
    disp = np.concatenate([outs[r][f][0] for r in range(G)])
    sub = np.concatenate([outs[r][f][1] for r in range(G)])
    assert np.array_equal(disp, want[f][0]), "frame %d: integer disparity" % f
    assert np.array_equal(sub, want[f][1]), "frame %d: sub-pixel" % f


@pytest.mark.parametrize("order,inputs", [("ascending", "pageable"), ("descending", "pinned")])
@pytest.mark.parametrize("geom", GEOMETRIES, ids=IDS)
def test_every_frame_of_the_c_stream_equals_the_oracle(streams_for, geom, order, inputs):
    """all 3 (G + 1) distinct frames (masks on odd frames) through one RowsStream per rank, bit for bit against the oracle.  Some tickets are
    waited for in the stream, the others only after their slot was reused: their buffers hold the right maps before any wait, and the waits
    after the flush, in a shuffled order, all succeed.  The contexts launch exactly what the Python driver launches for the same frames, and
    nothing is allocated after create."""
    st, frames, want = streams_for(geom)
    G, n = st.G, len(frames)
    ranks = list(range(G)) if order == "ascending" else list(reversed(range(G)))
    feed = _pinned(frames) if inputs == "pinned" else frames
    guards0, launches0 = st.guards(), st.launches()
    outs = st.outputs(n)
    waited = set()
    for f in range(n):
        assert _submit_round(st, ranks, feed[f], outs, f) == [f] * G
        t = f - G - 1  # its part 2 is at least one iteration old on every rank; its slot is reused one submit later
        if t >= 0 and t % 3 == 0:
            for r in ranks:
                st.streams[r].wait(t)
            waited.add(t)
    slots = G + 2
    for t in range(n - slots):  # retired when ticket t + G + 2 reused their slot: written without a wait
        if t not in waited:
            _check_frame(outs, want, t, G)
    for r in ranks:
        _raises(abi.SVA_ERR_STATE, lambda: st.streams[r].wait(n - 1))  # the last frame's part 2 is not enqueued before the flush
        st.streams[r].flush()
    shuffled = list(range(n))
    random.Random(n).shuffle(shuffled)
    for t in shuffled:
        for r in ranks:
            st.streams[r].wait(t)
    for f in range(n):
        _check_frame(outs, want, f, G)
    for r in ranks:
        for bad in (-1, n):
            _raises(abi.SVA_ERR_BAD_ARG, lambda: st.streams[r].wait(bad))
    launches = st.launches()
    guards = st.guards()
    for r in range(G):
        for j in range(G + 1):
            assert guards[r][j][0] == guards0[r][j][0] > 0, "rank %d context %d: a device buffer was allocated inside the stream" % (r, j)
            assert guards[r][j][1] == 0, "rank %d context %d: %d canary bytes overwritten" % (r, j, guards[r][j][1])
    if inputs == "pinned":  # the Python driver on contexts of its own, the same frames
        rk = _Ranks(geom, frames)
        try:
            py0 = [[c.launches() for c in row] for row in rk.ctxs]
            rk.run(frames, list(range(G)), hooked=False)
            rk.idle_and_guarded()
            py = [[c.launches() - c0 for c, c0 in zip(row, row0)] for row, row0 in zip(rk.ctxs, py0)]
        finally:
            rk.close()
        assert [[a - b for a, b in zip(row, row0)] for row, row0 in zip(launches, launches0)] == py


@pytest.mark.parametrize("geom", GEOMETRIES, ids=IDS)
def test_flushes_between_fills(streams_for, geom):
    """a stream of one frame, a flush, G + 2 frames, a flush, the rest, a flush: every frame right, tickets continuing across the fills"""
    st, frames, want = streams_for(geom)
    G, n = st.G, len(frames)
    outs = st.outputs(n)
    f = 0
    for fill in (1, G + 2, n - G - 3):
        for _ in range(fill):
            assert _submit_round(st, range(G), frames[f], outs, f) == [f] * G
            f += 1
        for s in st.streams:
            s.flush()
            s.flush()  # nothing left to drain: no-op
        for t in range(f - fill, f):
            for s in st.streams:
                s.wait(t)
            _check_frame(outs, want, t, G)
    assert f == n


def test_refusals_leave_the_stream_working(streams_for):
    """each refusal enqueues nothing, and the stream works afterwards"""
    from stereovisionarray_b200.pipeline import DepthContext, RowsStream
    geom = GEOMETRIES[0]
    st, frames, want = streams_for(geom, connect=False)
    G, p, n = st.G, st.p, len(frames)
    extra = []

    def refused(code, fn):
        before = st.launches()
        _raises(code, fn)
        assert st.launches() == before
    try:
        row = st.ctxs[0]
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row[:G], p))                      # world + 1 contexts are needed
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row + [row[0]], p))               # and no more
        other = DepthContext(0)                                                           # a context on a stream of its own
        extra.append(other)
        other.rows_open(p, 0, G)
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row[:G] + [other], p))
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row[:G] + [st.ctxs[1][G]], p))   # a context of another rank
        h, w, D, _, offs, k = geom
        p2 = abi.make_params(w, h + 8, D, offs, win_half=k, n_paths=8, lr_gx=-1)          # a context of another geometry
        odd = DepthContext(0)
        extra.append(odd)
        odd.set_stream(row[0].get_stream())
        odd.rows_open(p2, 0, G)
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row[:G] + [odd], p))
        refused(abi.SVA_ERR_BAD_ARG, lambda: RowsStream(row, p2))                          # parameters the links were not opened for
        outs = st.outputs(n)
        f0 = frames[0]
        refused(abi.SVA_ERR_STATE, lambda: st.streams[0].submit(f0["ref"], f0["others"], None, *outs[0][0]))  # links not connected
        st.connect()
        small = np.ascontiguousarray(f0["ref"][:-1])
        refused(abi.SVA_ERR_BAD_ARG, lambda: st.streams[0].submit(small, f0["others"], None, *outs[0][0]))     # image of another size
        for f in range(n):
            assert _submit_round(st, range(G), frames[f], outs, f) == [f] * G
        for s in st.streams:
            s.flush()
        for f in range(n):
            for s in st.streams:
                s.wait(f)
            _check_frame(outs, want, f, G)
    finally:
        for c in extra:
            c.close()
