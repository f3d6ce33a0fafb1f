"""torchrun check: every multi-GPU scheme of ONE frame over WORLD_SIZE GPUs against the CPU ORACLE (rank 0 compares), bit for bit.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/check_sharded.py [--c3] [--time]

Schemes: pairs (C: sva_depth_pair_sharded, NCCL reduce from the library), slices and rows (Python + torch.distributed), rows_direct
(C: sva_rows_*, peer-direct hand-off over CUDA IPC), rows_stream (rows_direct over a stream of distinct frames in the order skewed by chain
position, dist.rows_direct_stream, every frame checked), rows_stream_c (the same stream through the C library's one call per frame,
sva_rows_stream_* via pipeline.RowsStream, links connected with dist.rows_stream_connect).  Small frames are checked against a live oracle run; --c3 checks the full
3840x2160x256 frame against the oracle digests in tests/golden/c3_full_oracle.json (tests/golden/make_c3_hash.py) and the streams on c3's
width, D and pairs at 24 rows per rank (+ the border bands) against a live oracle run, and --time adds device-timed runs of the row pipelines at full size.
Exit code 1 on any mismatch."""
import argparse
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stereovisionarray_b200 import abi, configs, dist as sdist, synth  # noqa: E402
from stereovisionarray_b200.pipeline import DepthContext  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--c3", action="store_true", help="the full c3 frame against the committed oracle digests")
ap.add_argument("--time", action="store_true", help="with --c3: device-timed row pipelines")
ap.add_argument("--schemes", default="pairs,slices,rows,rows_direct,rows_stream,rows_stream_c,adapter")
args = ap.parse_args()

rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
OFF15 = [(gx, gy) for gy in range(-1, 3) for gx in range(-1, 3) if (gx, gy) != (0, 0)]
schemes = args.schemes.split(",")
ok = True
ADAPTER_UID = None


def say(msg):
    if rank == 0:
        print(msg, flush=True)


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def run_schemes(p, sc, tag):
    """-> {scheme: (disp, subpix)} on rank 0"""
    out = {}
    ctx = DepthContext(local)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    if "pairs" in schemes:
        uid = [DepthContext.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
        for _ in range(2):
            r = ctx.depth_pair_sharded(p, sc["ref"], sc["others"], sc["mask"], 0)
        out["pairs"] = r
        ctx.comm_barrier()
        ctx.comm_destroy()
    if "slices" in schemes and p.num_disp % world == 0 and (p.num_disp // world) % 8 == 0:
        keep = {}
        for _ in range(2):  # twice: cached buffers, re-upload
            out["slices"] = sdist.slice_sharded_depth(ctx, p, sc["ref"], sc["others"], sc["mask"], rank, world, None, keep)
    if "rows" in schemes:
        keep = {}
        for _ in range(2):
            out["rows"] = sdist.row_sharded_depth(ctx, p, sc["ref"], sc["others"], sc["mask"], rank, world, None, keep)
    if "rows_direct" in schemes:
        ctx.use_own_stream()  # nothing of torch's is ordered against these kernels: upload, hand-off and download all happen in the library
        sdist.rows_direct_connect(ctx, p, rank, world)
        for _ in range(3):  # several frames through the same link: the flags count frames
            out["rows_direct"] = sdist.rows_direct_depth(ctx, p, sc["ref"], sc["others"], sc["mask"], rank, world)
        dist.barrier()
        ctx.rows_close()
    torch.cuda.synchronize()
    dist.barrier()
    ctx.close()
    if "adapter" in schemes and not args.c3:
        # a C++ host's route: adapter/sva_functions.cpp (svaCommInit, svaDepthPairSharded, svaDepthRowsSharded) through its C test glue
        import ctypes as C
        so = os.path.join(ROOT, "adapter", "_build", "libsva_adapter_test.so")
        if os.path.exists(so):
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from test_gpu_adapter import adapter_multi_gpu
            lib = C.CDLL(so)
            lib.adapter_last_error.restype = C.c_char_p
            uid = [None]
            if rank == 0:
                buf = (C.c_uint8 * 128)()
                assert lib.adapter_comm_id(buf) == 0
                uid = [bytes(buf)]
            global ADAPTER_UID
            if ADAPTER_UID is None:  # the adapter holds ONE communicator per process
                dist.broadcast_object_list(uid, src=0)
                ADAPTER_UID = uid[0]
            dp, dr, sr, y0 = adapter_multi_gpu(lib, local, ADAPTER_UID, rank, world, p, sc["ref"], sc["others"])
            rows_per = sdist.row_blocks(p.height, world)[0]
            d_t = torch.full((rows_per, p.width), abi.SVA_DISP_INVALID, dtype=torch.int32, device="cuda")
            s_t = torch.full((rows_per, p.width), -1.0, dtype=torch.float32, device="cuda")
            d_t[:dr.shape[0]] = torch.from_numpy(dr.astype(np.int32)).cuda()
            s_t[:dr.shape[0]] = torch.from_numpy(sr).cuda()
            d_all = [torch.empty_like(d_t) for _ in range(world)] if rank == 0 else None
            s_all = [torch.empty_like(s_t) for _ in range(world)] if rank == 0 else None
            dist.gather(d_t, d_all, dst=0)
            dist.gather(s_t, s_all, dst=0)
            if rank == 0:
                out["adapter_rows"] = (torch.cat(d_all)[:p.height].cpu().numpy().astype(np.uint16), torch.cat(s_all)[:p.height].cpu().numpy())
                out["adapter_pairs"] = (dp, out["adapter_rows"][1])  # the pair-sharded wrapper returns the integer map
    return out


def rows_stream(p, scenes):
    """the frames `scenes` through rows_direct in the order skewed by chain position (dist.rows_direct_stream): world + 1 contexts on one
    stream, each its own link; the download hook gathers every frame's rows on rank 0 before its context is reused.  -> [(frame, (disp,
    subpix))] in download order on rank 0"""
    P = world + 1
    ctxs, got = [], []
    try:
        for j in range(P):
            c = DepthContext(local)
            ctxs.append(c)
            if j:
                c.set_stream(ctxs[0].get_stream())
            sdist.rows_direct_connect(c, p, rank, world)
        assert scenes[0]["mask"] is None and scenes[1]["mask"] is not None
        for sc in scenes[:2]:  # every buffer, masked and unmasked, before the stream: a buffer that grew there would synchronise the device
            for c in ctxs:
                c.upload(p, sc["ref"], sc["others"], sc["mask"])
                c.rows_run()
                c.rows_download()

        def upload(c, f):
            c.upload(p, scenes[f]["ref"], scenes[f]["others"], scenes[f]["mask"])

        def download(c, f):
            d, s = c.rows_download()
            got.append((f, sdist.gather_rows(d, s, p, rank, world)))
        sdist.rows_direct_stream(ctxs, rank, world, len(scenes), upload, download)
        dist.barrier()  # nobody unmaps a link a neighbour still writes into
        for c in reversed(ctxs):  # the borrowers first: ctxs[0] owns the stream
            c.rows_close()
    finally:
        for c in reversed(ctxs):
            c.close()
    return got


def rows_stream_c(p, scenes):
    """the frames `scenes` through the C library's stream (pipeline.RowsStream: one sva_rows_stream_submit per frame, uploads and downloads on
    copy streams), world + 1 contexts on one stream linked with dist.rows_stream_connect; every frame's rows are gathered on rank 0 after a
    flush.  -> [(frame, (disp, subpix))] on rank 0"""
    from stereovisionarray_b200.pipeline import RowsStream
    ctxs, got, s = [], [], None
    try:
        for j in range(world + 1):
            c = DepthContext(local)
            ctxs.append(c)
            if j:
                c.set_stream(ctxs[0].get_stream())
        sdist.rows_stream_connect(ctxs, p, rank, world)
        s = RowsStream(ctxs, p)
        outs = [(np.empty((s.rows, p.width), np.uint16), np.empty((s.rows, p.width), np.float32)) for _ in scenes]
        tickets = [s.submit(sc["ref"], sc["others"], sc["mask"], *o) for sc, o in zip(scenes, outs)]
        s.flush()
        for t in tickets:
            s.wait(t)
            got.append((t, sdist.gather_rows(outs[t][0], outs[t][1], p, rank, world)))
        dist.barrier()  # nobody unmaps a link a neighbour still writes into
    finally:
        if s is not None:
            s.close()
        for c in reversed(ctxs):  # the borrowers first: ctxs[0] owns the stream
            c.close()
    return got


def check_stream(p, scenes, tag, name="rows_stream", run=rows_stream):
    global ok
    got = run(p, scenes)
    if rank != 0:
        return
    from oracle.oracle import Oracle
    if [f for f, _ in got] != list(range(len(scenes))):
        say("%s %s over %d GPUs vs oracle: MISMATCH (frames downloaded: %s)" % (name, tag, world, [f for f, _ in got]))
        ok = False
    for f, (d, s) in got:
        d0, s0 = Oracle().depth_from_array(p, scenes[f]["ref"], scenes[f]["others"], scenes[f]["mask"])
        same = np.array_equal(d, d0) and np.array_equal(s, s0) and bool((d0 != 0xFFFF).any())  # a frame with no valid pixel checks nothing
        say("%s %s frame %d over %d GPUs vs oracle: %s (valid %.3f)" % (name, tag, f, world, "bit-exact" if same else "MISMATCH", float((d0 != 0xFFFF).mean())))
        ok = ok and same


def stream_scenes(h, w, D, off):
    """3 (world + 1) distinct frames — every link of the skewed order carries three — the mask on odd frames"""
    return [synth.make_scene(h, w, D, off, 7700 + f, face=f % 2 == 1) for f in range(3 * (world + 1))]


if not args.c3:
    from oracle.oracle import Oracle  # test infrastructure: the checker
    for (h, w, D, off, k, face) in [(270, 480, 256, OFF15, 20, True), (203, 333, 128, OFF15[:8], 7, True), (131, 3840, 192, OFF15[:3], 4, False)]:
        sc = synth.make_scene(h, w, D, off, 77, face=face)
        p = abi.make_params(w, h, D, off, win_half=k, n_paths=8, lr_gx=-1)
        out = run_schemes(p, sc, "%dx%dx%d" % (w, h, D))
        if rank == 0:
            d0, s0 = Oracle().depth_from_array(p, sc["ref"], sc["others"], sc["mask"])
            d0n, s0n = Oracle().depth_from_array(p, sc["ref"], sc["others"], None) if any(k.startswith("adapter") for k in out) else (None, None)
            for name, o in out.items():
                dref, sref = (d0n, s0n) if name.startswith("adapter") else (d0, s0)  # the adapter's test glue passes no mask
                same = np.array_equal(o[0], dref) and np.array_equal(o[1], sref)
                say("%s %dx%dx%d over %d GPUs vs oracle: %s (valid %.3f)" % (name, w, h, D, world, "bit-exact" if same else "MISMATCH", float((d0 != 0xFFFF).mean())))
                ok = ok and same
        if "rows_stream" in schemes:
            check_stream(p, stream_scenes(h, w, D, off), "%dx%dx%d" % (w, h, D))
        if "rows_stream_c" in schemes:
            check_stream(p, stream_scenes(h, w, D, off), "%dx%dx%d" % (w, h, D), "rows_stream_c", rows_stream_c)
else:
    with open(os.path.join(ROOT, "tests", "golden", "c3_full_oracle.json")) as f:
        gold = json.load(f)
    sc = configs.scene("c3")
    p = configs.params("c3")
    if rank == 0:
        same_in = digest(np.stack([sc["ref"]] + list(sc["others"]))) == gold["inputs_sha256"]
        say("c3 synthetic inputs: %s" % ("same bytes as the oracle run" if same_in else "DIFFERENT from the oracle run"))
        ok = ok and same_in
    out = run_schemes(p, sc, "c3")
    if rank == 0:
        for name, o in out.items():
            same_d = digest(o[0]) == gold["disp_sha256"]
            same_s = digest(o[1]) == gold["subpix_sha256"]
            say("%s c3 3840x2160x256, 15 pairs, %d GPUs vs oracle digests: integer map %s, sub-pixel map %s (valid pixels %d / %d)"
                % (name, world, "bit-exact" if same_d else "MISMATCH", "bit-exact" if same_s else "MISMATCH", int((o[0] != 0xFFFF).sum()), gold["valid_pixels"]))
            ok = ok and same_d and same_s
    # distinct full-size c3 frames would cost a minute of oracle time each: the streams run c3's width, D and pairs at a height of 24 rows per
    # rank plus the two border bands of win_half rows, which hold no valid pixel
    ps = configs.params("c3")
    ps.height = 24 * world + 2 * ps.win_half
    for name, run in (("rows_stream", rows_stream), ("rows_stream_c", rows_stream_c)):
        if name in schemes:
            check_stream(ps, stream_scenes(ps.height, ps.width, ps.num_disp, configs.offsets("c3")), "c3 3840x%dx256" % ps.height, name, run)
    if args.time:
        ctx = DepthContext(local)
        stream = torch.cuda.current_stream()
        ctx.set_stream(stream.cuda_stream)
        ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
        sdist.rows_direct_connect(ctx, p, rank, world)
        keep = {}
        for name, step in (("rows (NCCL send/recv hops)", lambda: sdist.row_sharded_compute(ctx, p, rank, world, None, keep)), ("rows_direct (peer stores + flags)", ctx.rows_run)):
            for _ in range(2):
                step()
            res = []
            for frames, per_frame_barrier in ((5, True), (8, False)):
                tot = 0.0
                for _ in range(frames if per_frame_barrier else 1):
                    torch.cuda.synchronize()
                    dist.barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(1 if per_frame_barrier else frames):
                        step()
                    e1.record(stream)
                    torch.cuda.synchronize()
                    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    tot += float(t.item())
                res.append(tot / frames)
            say("%s c3, %d GPUs: %.3f ms latency of one frame (all ranks start together), %.3f ms per frame back to back (device time, max over ranks)"
                % (name, world, res[0], res[1]))
        dist.barrier()
        ctx.rows_close()
        ctx.close()
flag = torch.tensor([0 if ok else 1], device="cuda")
dist.broadcast(flag, src=0)
dist.barrier()
dist.destroy_process_group()
sys.exit(int(flag.item()))
