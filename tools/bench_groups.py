"""The 13 CHESS groups of a 25-camera frame (getGroups(cameras, "CHESS") on a 5 x 5 array) at c1's geometry (1280 x 960, D = 128, k = 20,
8 paths, LR and sub-pixel on), host buffers in and out, pinned inputs and outputs in every arm.

    python tools/bench_groups.py [--steps K] [--warmup W] [--out FILE]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/bench_groups.py [--steps K] [--out FILE]

One GPU: five arms in the same process, alternating round by round (so clock and thermal drift hit them alike):
  (a) groups:   one sva_depth_groups call — 25 uploads, each group staged from the device stack, the groups pipelined;
  (b) separate: 13 synchronous sva_depth_from_array calls — 55 uploads;
  (c) stream:   13 sva_stream_submit calls with host views, then waits for the last two tickets — 55 uploads, frames pipelined;
  (d) fused:    one sva_depth_groups_fused call into camera 12's view (tol 1 px, min_support 2): the group maps never leave the device;
  (e) groups_then_fuse: (a), then sva_fuse_maps on its 13 host maps into the same view.
After the timed rounds, the two fusion kernels (k_fuse_splat, k_fuse_consensus) are timed alone with torch.profiler over --steps
sva_fuse_maps calls: the device time of each launch, from the CUDA activity trace.
Several ranks: groups_sharded_depth, rank r computing the groups frame_range(13, N, r) from only the cameras they read; the slowest rank's
compute and the gather of the maps to rank 0 are reported separately.
Each figure is the median over --steps rounds of a host clock around work that ends with every map in host memory.  Rates: groups/s, and
GMDE/s counted as 13 x W x H x D matching-disparity evaluations per frame.  Rank 0 prints one JSON line (with the card's name and power
limit, read in the same run) and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stereovisionarray_b200 import abi, dist as sdist, reference_api, synth  # noqa: E402
from stereovisionarray_b200 import groups as G  # noqa: E402
from stereovisionarray_b200.pipeline import DepthContext  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10, help="timed rounds")
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", help="also write the JSON line to this file")
args = ap.parse_args()
if args.steps < 1:
    ap.error("--steps must be at least 1")

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
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


H, W, D = 960, 1280, 128
sc = synth.make_array_scene(H, W, 5, 5, D, 1001)
images = [pin(im) for im in sc["images"]]
groups = G.as_groups(reference_api.getGroups([None] * 25, "CHESS"))
p = abi.make_params(W, H, D, [(0, 0)] * 4, win_half=20, n_paths=8, lr_gx=-1, subpixel=1)
p.n_pairs = 0
NG = len(groups)
params = [G.group_params(p, g, 5) for g in groups]
gmde = NG * W * H * D / 1e9


TARGET = 12  # the centre camera


def fuse_kernel_times(fn, n):
    """device time of the fusion kernels over n calls of fn, from torch.profiler's CUDA activity trace -> {kernel: {mean_us, launches}}"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        for k in ("k_fuse_splat", "k_fuse_consensus"):
            if k in ev.name and ev.device_type.name == "CUDA":
                e = out.setdefault(k, {"total_us": 0.0, "launches": 0})
                e["total_us"] += ev.device_time
                e["launches"] += 1
    for e in out.values():
        e["mean_us"] = round(e["total_us"] / max(1, e["launches"]), 2)
        e["total_us"] = round(e["total_us"], 1)
    if set(out) != {"k_fuse_splat", "k_fuse_consensus"}:
        return {"not_measured": "the profiler trace holds only %r of the two fusion kernels" % sorted(out)}
    return out


def timed(fn):
    barrier()
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


ctx = DepthContext(local)
res = {"workload": "13 CHESS groups of a 5x5 array frame, %dx%d, D=%d, k=20, 8 paths, LR + sub-pixel; pinned host inputs and outputs" % (W, H, D),
       "n_gpus": world, "rounds": args.steps, "timing": "host clock around work ending with every map in host memory, median over rounds",
       "gmde_per_frame": round(gmde, 3)}
try:
    if world == 1:
        outs = [(torch.empty((H, W), dtype=torch.int16).pin_memory().numpy().view(np.uint16), torch.empty((H, W), dtype=torch.float32).pin_memory().numpy())
                for _ in range(NG)]

        g_disp = torch.empty((NG, H, W), dtype=torch.int16).pin_memory().numpy().view(np.uint16)
        g_sub = torch.empty((NG, H, W), dtype=torch.float32).pin_memory().numpy()

        def arm_groups():
            ctx.depth_groups(p, images, groups, 5, disp=g_disp, sub=g_sub)

        def arm_separate():
            for q, g, (d, s) in zip(params, groups, outs):
                ctx.depth_from_array(q, images[g[0][0]], [images[o] for _, o in g], None, d, s)

        def arm_stream():
            t = [ctx.stream_submit(q, images[g[0][0]], [images[o] for _, o in g], None, *out) for q, g, out in zip(params, groups, outs)]
            ctx.stream_wait(t[-2])
            ctx.stream_wait(t[-1])

        refs = [g[0][0] for g in groups]

        def arm_fused():
            ctx.depth_groups_fused(p, images, groups, 5, TARGET, 16, 2)

        def arm_groups_then_fuse():
            ctx.depth_groups(p, images, groups, 5, disp=g_disp, sub=g_sub)
            ctx.fuse_maps(g_disp, g_sub, refs, 5, 25, TARGET, 16, 2)

        arms = {"groups": arm_groups, "separate": arm_separate, "stream": arm_stream, "fused": arm_fused, "groups_then_fuse": arm_groups_then_fuse}
        for _ in range(args.warmup):
            for fn in arms.values():
                fn()
        times = {k: [] for k in arms}
        for _ in range(args.steps):
            for k, fn in arms.items():
                times[k].append(timed(fn))
        for k in arms:
            ms = float(np.median(times[k]))
            res[k] = {"ms_per_frame": round(ms, 3), "groups_per_s": round(NG / ms * 1e3, 1), "gmde_per_s": round(gmde / ms * 1e3, 2),
                      "ms_all_rounds": [round(t, 3) for t in times[k]]}
        res["arms"] = {"groups": "sva_depth_groups: 25 uploads, groups staged from the device stack and pipelined",
                       "separate": "13 synchronous sva_depth_from_array calls (55 uploads)",
                       "stream": "13 sva_stream_submit calls with host views (55 uploads), then waits for the last two tickets",
                       "fused": "sva_depth_groups_fused into camera %d (tol_16 16, min_support 2): one fused map downloaded" % TARGET,
                       "groups_then_fuse": "sva_depth_groups (13 maps downloaded), then sva_fuse_maps on them (13 maps uploaded again)"}
        res["groups_speedup_vs_stream"] = round(res["stream"]["ms_per_frame"] / res["groups"]["ms_per_frame"], 3)
        res["groups_speedup_vs_separate"] = round(res["separate"]["ms_per_frame"] / res["groups"]["ms_per_frame"], 3)
        res["fused_minus_groups_ms"] = round(res["fused"]["ms_per_frame"] - res["groups"]["ms_per_frame"], 3)
        res["fused_speedup_vs_groups_then_fuse"] = round(res["groups_then_fuse"]["ms_per_frame"] / res["fused"]["ms_per_frame"], 3)
        res["fuse_kernels"] = fuse_kernel_times(lambda: ctx.fuse_maps(g_disp, g_sub, refs, 5, 25, TARGET, 16, 2), args.steps)
    else:
        b, e = sdist.frame_range(NG, world, rank)
        mine = set(G.cameras_of(groups[b:e]))
        imgs = [im if i in mine else None for i, im in enumerate(images)]
        r_disp = torch.empty((e - b, H, W), dtype=torch.int16).pin_memory().numpy().view(np.uint16)
        r_sub = torch.empty((e - b, H, W), dtype=torch.float32).pin_memory().numpy()
        comp, gath, total = [], [], []
        for it in range(args.warmup + args.steps):
            barrier()
            t0 = time.perf_counter()
            d, s = ctx.depth_groups(p, imgs, groups, 5, group_range=(b, e), disp=r_disp, sub=r_sub)
            t1 = time.perf_counter()
            out = sdist.gather_groups(d, s, p, NG, rank, world)
            t2 = time.perf_counter()
            if it >= args.warmup:
                comp.append(rank_max((t1 - t0) * 1e3))
                gath.append(rank_max((t2 - t1) * 1e3))
                total.append(rank_max((t2 - t0) * 1e3))
        if rank == 0:
            assert out[0].shape == (NG, H, W)
        ms = float(np.median(total))
        res["sharded"] = {"groups_per_rank": [sdist.frame_range(NG, world, r)[1] - sdist.frame_range(NG, world, r)[0] for r in range(world)],
                          "compute_ms_slowest_rank": round(float(np.median(comp)), 3), "gather_to_rank0_ms": round(float(np.median(gath)), 3),
                          "ms_per_frame": round(ms, 3), "groups_per_s": round(NG / ms * 1e3, 1), "gmde_per_s": round(gmde / ms * 1e3, 2)}
    res["card"] = card()
finally:
    ctx.close()

if rank == 0:
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
if dist:
    dist.barrier()
    dist.destroy_process_group()
