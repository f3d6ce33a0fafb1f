"""torchrun: c3 (3840x2160, 16 cameras, D = 256) end to end through the C stream of the row-block pipeline, from pinned host buffers.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/bench_rows_stream.py [--steps K] [--out FILE]
    python tools/bench_rows_stream.py [--steps K] [--out FILE]        # a world of one

Three figures on the same ranks and contexts (world + 1 per GPU, one stream):
  * stream: ms per frame through sva_rows_stream_submit (pipeline.RowsStream) — every frame's 16 images uploaded from pinned host memory on the
    object's copy stream, the rows copied back on its second copy stream into pinned output buffers;
  * resident: ms per frame of the Python skewed loop (dist.rows_direct_stream) with each context's frame uploaded once, as bench.py times it;
  * upload alone: device time of one frame's H2D copies (the same pinned images into device memory, every rank at once, nothing else running).
Each ms per frame is the steady-state slope between a K- and a 3K-frame run (device clock: CUDA events on the compute stream, max over ranks),
as bench.py reports the skewed order.  Rank 0 prints one JSON line and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stereovisionarray_b200 import configs, dist as sdist  # noqa: E402
from stereovisionarray_b200.pipeline import DepthContext, RowsStream  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10, help="frames of the short run (the long run has 3x as many)")
ap.add_argument("--warmup", type=int, default=4)
ap.add_argument("--out", help="also write the JSON line to this file")
args = ap.parse_args()

rank, local, world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(local)
dist = None
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def barrier():
    if dist:
        dist.barrier()
    torch.cuda.synchronize()


def rank_max(v):
    if not dist:
        return v
    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(local), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def pin(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


p = configs.params("c3")
sc = configs.scene("c3")
frame = {"ref": pin(sc["ref"]), "others": [pin(o) for o in sc["others"]], "mask": pin(sc["mask"])}
images = [frame["ref"]] + frame["others"] + ([frame["mask"]] if frame["mask"] is not None else [])
h2d_bytes = sum(a.nbytes for a in images)

ctxs, s = [], None
try:
    for j in range(world + 1):
        c = DepthContext(local)
        ctxs.append(c)
        if j:
            c.set_stream(ctxs[0].get_stream())
    sdist.rows_stream_connect(ctxs, p, rank, world)
    s = RowsStream(ctxs, p)
    outs = [(torch.empty((s.rows, p.width), dtype=torch.int16).pin_memory().numpy().view(np.uint16),
             torch.empty((s.rows, p.width), dtype=torch.float32).pin_memory().numpy()) for _ in range(s.slots)]

    def stream_run(frames):
        """frames through the C stream, then the drain -> device ms from the first submit to the end of the drain (max over ranks)"""
        barrier()
        ctxs[0].timer_start()
        for k in range(frames):  # output buffer k % slots is reused only once the ticket that last used it has been retired
            t = s.submit(frame["ref"], frame["others"], frame["mask"], *outs[k % s.slots])
        s.flush()
        ms = ctxs[0].timer_stop()
        for k in range(max(0, t + 1 - s.slots), t + 1):  # the tickets whose slot was not reused; raises on a hand-off time-out
            s.wait(k)
        return rank_max(ms)

    stream_run(args.warmup)
    short, long = args.steps, 3 * args.steps
    t_stream = {n: stream_run(n) for n in (short, long)}
    s.close()
    s = None

    def resident_run(frames):
        barrier()
        ctxs[0].timer_start()
        sdist.rows_direct_stream(ctxs, rank, world, frames)
        ms = ctxs[0].timer_stop()
        for c in ctxs:
            c.rows_download()  # raises on a hand-off time-out
        return rank_max(ms)

    for c in ctxs:
        c.upload(p, frame["ref"], frame["others"], frame["mask"])
    resident_run(args.warmup)
    t_res = {n: resident_run(n) for n in (short, long)}

    # the upload on its own: the same pinned images into device memory, every rank at once, with nothing else running
    dev = [torch.empty(a.nbytes, dtype=torch.uint8, device="cuda") for a in images]
    host = [torch.from_numpy(a.reshape(-1)) for a in images]
    up = []
    for _ in range(5):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for d, hst in zip(dev, host):
            d.copy_(hst, non_blocking=True)
        e1.record()
        e1.synchronize()
        up.append(rank_max(e0.elapsed_time(e1)))
    barrier()
finally:
    if s is not None:
        s.close()
    for c in reversed(ctxs):  # the borrowers first: ctxs[0] owns the stream
        c.close()

slope = lambda t: round((t[long] - t[short]) / (long - short), 3)  # noqa: E731
upload_ms = min(up)
res = {
    "workload": "c3: " + configs.CONFIGS["c3"]["desc"], "n_gpus": world, "contexts_per_gpu": world + 1, "frames_per_run": [short, long],
    "stream_ms_per_frame_steady_state": slope(t_stream), "stream_ms_per_frame_long_run": round(t_stream[long] / long, 3),
    "stream_inputs": "pinned host buffers, uploaded every frame on the stream's copy stream; rows copied back into pinned host buffers",
    "resident_ms_per_frame_steady_state": slope(t_res), "resident_ms_per_frame_long_run": round(t_res[long] / long, 3),
    "resident": "Python skewed loop (dist.rows_direct_stream), each context's frame uploaded once before the runs",
    "h2d_bytes_per_frame_and_rank": h2d_bytes, "h2d_images_per_frame": len(images),
    "upload_alone_ms_per_frame": round(upload_ms, 3), "upload_alone_gb_per_s": round(h2d_bytes / upload_ms / 1e6, 1),
    "upload_alone": "the same pinned images copied H2D with nothing else running, every rank at once, best of 5 (max over ranks)",
    "timing": "CUDA events on the compute stream (device clock), steady state = slope between the two runs, max over ranks",
    "card": card(),
}
if rank == 0:
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
if dist:
    dist.barrier()
    dist.destroy_process_group()
