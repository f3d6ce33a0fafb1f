#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the multi-camera depth hot path.

  python bench.py --gpus N --steps K --warmup W [--config c1] [--win-half 20] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path (K1a AD volume -> K1b box/pack -> 8-path SGM -> WTA/LR/sub-pixel) over one synthetic
frame per rank.  `value` = whole-job MDE/s with inputs resident in HBM (CUDA events on the library's stream, max over ranks);
`e2e` = the same metric through the host-buffer C-ABI call sva_depth_from_array (pinned host inputs, H2D + D2H inside the timed
region).  Volumes (>= 300 MB each at c1) exceed the 126 MB L2, so no L2 flush is needed between iterations.
`--impl reference` times the reference's own CPU code (oracle/_ref: the unmodified sources compiled against oracle/cvshim) on
bounded bands of the same resolution; rank 0 only."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from stereovisionarray_b200 import abi, configs, synth  # noqa: E402

FALLBACK_HBM_GBS = 6650.0


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.p:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            text = self.p.communicate(timeout=5)[0]
        except Exception:
            return out
        sm, mx, reasons = [], [], set()
        for line in text.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def split_label(label):
    """timing label of the library: '<kernel symbol as ncu prints it>/<what the launch carries>' (plain symbol for the other kernels)"""
    sym, _, what = label.partition("/")
    return sym, what


def schedule_bytes(label, p, n_cam):
    """Minimum DRAM bytes ONE launch of this kernel has to move in the schedule the library runs (DESIGN.md §4; s_C = s_S = 2 bytes per cell):
    what `roofline.achieved` is computed from.  A launch that carries several row-sweeping SGM directions streams C once and
    read-modify-writes S once for all of them (they share the lines in L2): 6 B/DE; the two horizontal directions cannot share: 12 B/DE."""
    de = p.width * p.height * p.num_disp
    px = p.width * p.height
    sym, what = split_label(label)
    if sym in ("k_ad_planar", "k_ad_tile") or sym.startswith("k_ad_tile"):
        return n_cam * px + 2 * de          # views in, A out
    if sym in ("k_box_cost", "k_box_planar") or sym.startswith("k_box_planar"):
        return 4 * de                       # A in, C out
    if sym.startswith("k_sgm_acc"):
        n = int(what[-1]) if what and what[-1].isdigit() else 1
        if what.startswith("store_"):
            return 4 * de * n
        if "horizontal" in what or "mixed" in what:
            return 6 * de * n               # every direction streams C and read-modify-writes S on its own
        return 6 * de                       # row-sweeping directions of one launch share C and S (each ranged launch streams them once)
    if sym.startswith("k_wta_seg") or sym.startswith("k_wta_tile"):
        return 2 * de + 6 * px              # S once, winner map + the other view's key map
    if sym.startswith("k_wta_finish"):
        return 18 * px                      # winner, key, mask, three S cells, u16 + f32 outputs
    if sym.startswith("k_lr_check"):
        return 10 * px
    return None


def textbook_bytes(label, p, n_cam):
    """SURVEY §8(d)'s per-path count for the same launch: every SGM direction streams C once and read-modify-writes S once (6 B/DE each)"""
    de = p.width * p.height * p.num_disp
    sym, what = split_label(label)
    if sym.startswith("k_sgm_acc") and not what.startswith("store_"):
        n = int(what[-1]) if what and what[-1].isdigit() else 1
        return 6 * de * n
    return schedule_bytes(label, p, n_cam)


def load_traffic(key, order):
    """profiles/traffic.json (tools/traffic_from_ncu.py): ncu records of the launches of one frame of THIS configuration, paired with
    the library's own launch list of a frame (`order`: timing labels in launch order) -> {label: averaged record}; {} without a capture"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            recs = json.load(f).get(key, {}).get("launches", [])
    except Exception:
        return {}
    norm = lambda s: s.replace(" ", "")
    if len(recs) != len(order) or any(norm(split_label(l)[0]) not in norm(r["kernel"]) for l, r in zip(order, recs)):
        return {}  # the capture is of another build / schedule: refuse rather than print stale numbers
    out = {}
    for l, r in zip(order, recs):
        out.setdefault(l, []).append(r)
    avg = {}
    for l, rs in out.items():
        a = {"dram_bytes": sum(r["dram_bytes"] for r in rs) / len(rs), "bound": max(set(r["bound"] for r in rs), key=[r["bound"] for r in rs].count)}
        for k in ("hbm_pct", "l1tex_pct", "alu_pct", "lsu_pct", "issue_pct", "warps_pct"):
            v = [r[k] for r in rs if r.get(k) is not None]
            a[k] = round(sum(v) / len(v), 1) if v else None
        avg[l] = a
    return avg


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class Ranks:
    """barrier / max-over-ranks plumbing (torch.distributed over NCCL when launched by torchrun)"""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank, self.local_rank, self.world = dist_env()
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        if not self.dist:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def run_sva(args):
    import torch
    R = Ranks()
    rank, local_rank, world = R.rank, R.local_rank, R.world
    from stereovisionarray_b200.pipeline import DepthContext
    name = args.config
    if name == "literal":
        return run_literal(args, R)
    cfg = configs.CONFIGS[name]
    p = configs.params(name, win_half=args.win_half)
    n_cam = p.n_pairs + 1
    if name == "c3":
        out = run_c3(args, R, headline=True)
        if rank == 0:
            emit(json.dumps(out))
        R.close()
        return
    # capture batch: c4 has 64 frames per step split over the ranks (strong scaling); the others one frame per rank per step (weak)
    from stereovisionarray_b200 import dist as sdist
    batch = cfg["frames"]
    fb, fe = sdist.frame_range(batch, world, rank) if batch > 1 else (rank, rank + 1)
    frames_rank = fe - fb
    frames_step_total = batch if batch > 1 else world
    sc = configs.scene(name, frame=fb)  # every rank works on its own frames of the capture batch
    ctx = DepthContext(local_rank)

    # ---- resident: inputs already in HBM ----
    ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
    for _ in range(args.warmup):
        ctx.run(abi.STAGE_ALL)
    ctx.synchronize()
    l0 = ctx.launches()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    R.barrier()
    total_ms, kern_main = ctx.time_detailed(abi.STAGE_ALL, args.steps * frames_rank)
    R.barrier()
    launches = ctx.launches() - l0
    total_ms = R.max(total_ms)
    if args.dump_outputs and rank == 0:
        disp, sub = ctx.download_disparity()  # the maps the last timed step left on the device
        dump_outputs(args.dump_outputs, {"disparity": disp, "subpixel": sub})
    # Per-kernel table: the default schedule runs the second horizontal SGM direction on a second stream NEXT TO the first row-sweeping
    # group (where the launches are not paced), so event times of those launches overlap and say little about each kernel.  The table,
    # the roofline of the dominant kernel and the ncu pairing therefore come from a second pass of the same frames with that one overlap
    # switched off (SVA_SGM_HSTORE=1: same kernels, same launches, one after the other — what ncu sees as well); `value` is the default pass.
    sgm_wall_ms = kern_main.get("stage:k2_sgm", (0.0, 0))[0] / max(1, args.steps * frames_rank)
    kern, serial_ms, order = kern_main, None, None
    if rank == 0:
        prev = os.environ.get("SVA_SGM_HSTORE")
        if prev is None:
            os.environ["SVA_SGM_HSTORE"] = "1"
        ctx2 = DepthContext(local_rank)
        if prev is None:
            del os.environ["SVA_SGM_HSTORE"]
        ctx2.upload(p, sc["ref"], sc["others"], sc["mask"])
        for _ in range(args.warmup):
            ctx2.run(abi.STAGE_ALL)
        ctx2.synchronize()
        order = [n for n, _ in ctx2.kernel_times(abi.STAGE_ALL) if not n.startswith("stage:")]  # the launches of one frame, in order
        serial_ms, kern = ctx2.time_detailed(abi.STAGE_ALL, args.steps * frames_rank)
        ctx2.close()
    sgm_serial_ms = kern.get("stage:k2_sgm", (0.0, 0))[0] / max(1, args.steps * frames_rank)
    kern = {k: v for k, v in kern.items() if not k.startswith("stage:")}
    mde = configs.mde_per_frame(name)
    value = frames_step_total * mde * args.steps / (total_ms / 1e3)

    # ---- end to end: pinned host buffers -> C-ABI call -> host results ----
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = [pinned(sc["ref"])] + [pinned(o) for o in sc["others"]] + ([pinned(sc["mask"])] if sc["mask"] is not None else [])
    ref_h = keep[0][1]; others_h = [k[1] for k in keep[1:1 + p.n_pairs]]; mask_h = keep[-1][1] if sc["mask"] is not None else None
    others_c = abi.image_array(others_h)
    outs = []
    for _ in range(2):  # two frames are in flight: two sets of pinned result buffers
        disp_t = torch.empty((p.height, p.width), dtype=torch.uint16).pin_memory(); sub_t = torch.empty((p.height, p.width), dtype=torch.float32).pin_memory()
        outs.append((disp_t, sub_t, disp_t.numpy(), sub_t.numpy()))
    disp_h, sub_h = outs[0][2], outs[0][3]
    # (a) one synchronous call per frame: upload, kernels and download back to back
    for _ in range(max(1, args.warmup)):
        ctx.depth_from_array(p, ref_h, others_c, mask_h, disp_h, sub_h)
    R.barrier()
    ctx.timer_start()
    for _ in range(args.steps * frames_rank):
        ctx.depth_from_array(p, ref_h, others_c, mask_h, disp_h, sub_h)
    single_ms = ctx.timer_stop()
    # (b) the capture-stream API (what a user with a stream of frames calls): same work per frame, but frame t+1's upload and frame
    # t-1's download overlap frame t's kernels.  Timed on the device from the first upload to the end of the last download.
    for i in range(max(2, args.warmup)):
        ctx.stream_wait(ctx.stream_submit(p, ref_h, others_c, mask_h, outs[i % 2][2], outs[i % 2][3]))
    R.barrier()
    ctx.stream_mark()
    last = None
    for i in range(args.steps * frames_rank):
        last = ctx.stream_submit(p, ref_h, others_c, mask_h, outs[i % 2][2], outs[i % 2][3])
    e2e_ms = ctx.stream_elapsed(last)
    R.barrier()
    clocks = sampler.stop() if sampler else None
    e2e_ms = R.max(e2e_ms)
    single_ms = R.max(single_ms)
    e2e_value = frames_step_total * mde * args.steps / (e2e_ms / 1e3)
    h2d = frames_rank * (n_cam * p.width * p.height + (p.width * p.height if mask_h is not None else 0))
    d2h = frames_rank * p.width * p.height * (2 + 4)
    ctx.close()

    out = None
    if rank == 0:
        # ---- roofline of the dominant kernel + the per-kernel table ----
        peak, peak_src = measured_peak()
        traffic = load_traffic("%s_k%d" % (name, args.win_half), order)
        de = p.width * p.height * p.num_disp
        rows = []
        for kname, (sum_ms, cnt) in kern.items():
            sb, tb = schedule_bytes(kname, p, n_cam), textbook_bytes(kname, p, n_cam)
            avg_ms = sum_ms / max(1, cnt)
            sym, what = split_label(kname)
            tr = traffic.get(kname)
            # bytes the launch has to move: the schedule's count, or the measured DRAM traffic where the L2 serves part of that count (the
            # horizontal SGM launch: -> and <- meet in the middle of a row) — so the fraction is of real HBM work and cannot exceed ~1
            fb = min(sb, tr["dram_bytes"]) if (sb and tr) else sb
            rows.append({"kernel": sym, "launch": what or None, "launches_per_step": cnt / args.steps / frames_rank, "avg_ms": round(avg_ms, 4), "share": round(sum_ms / serial_ms, 4),
                         "schedule_bytes": sb, "achieved_gbs": round(fb / avg_ms / 1e6, 1) if fb else None, "frac": round(fb / avg_ms / 1e6 / peak, 4) if fb else None,
                         "frac_schedule": round(sb / avg_ms / 1e6 / peak, 4) if sb else None,
                         "frac_textbook": round(tb / avg_ms / 1e6 / peak, 4) if tb else None,
                         "traffic": int(tr["dram_bytes"]) if tr else None, "dram_frac": round(tr["dram_bytes"] / avg_ms / 1e6 / peak, 4) if tr else None,
                         "bound": tr["bound"] if tr else None, "ncu_pct": {k[:-4]: tr[k] for k in ("hbm_pct", "l1tex_pct", "alu_pct", "lsu_pct", "issue_pct", "warps_pct")} if tr else None})
        rows.sort(key=lambda r: -r["share"])
        dom = next(r for r in rows if r["schedule_bytes"])
        per_frame = lambda pred: sum(s for k, (s, c) in kern.items() if pred(split_label(k)[0])) / args.steps / frames_rank
        sgm_ms = per_frame(lambda s: s.startswith("k_sgm"))
        sgm_sched = sum(schedule_bytes(k, p, n_cam) * c for k, (s, c) in kern.items() if split_label(k)[0].startswith("k_sgm")) / args.steps / frames_rank
        sgm_text = (6 * p.n_paths - 4) * de if p.n_paths else 0
        k1_ms = per_frame(lambda s: s.startswith("k_ad") or s.startswith("k_box"))
        k1_bytes = n_cam * p.width * p.height + 2 * de  # SURVEY §8(d): the views in, the packed cost volume out (A is an implementation detail)
        stage = lambda b, ms: {"bytes": int(b), "ms": round(ms, 4), "achieved_gbs": round(b / ms / 1e6, 1) if ms else None, "frac": round(b / ms / 1e6 / peak, 4) if ms else None}
        roofline = {"bound": ("hbm" if dom["bound"] in (None, "hbm") else dom["bound"]) if dom["traffic"] else "hbm",
                    "bound_source": "ncu capture of this configuration (profiles/traffic.json)" if dom["traffic"] else "assumed: no ncu capture of this configuration and build in profiles/traffic.json",
                    "kernel": dom["kernel"], "launch": dom["launch"], "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                    "frac_definition": "min(schedule bytes, measured DRAM bytes of the ncu capture) / event-timed launch / measured HBM peak; schedule bytes = what this launch must move given which directions share C and S in L2 (DESIGN.md §6)",
                    "frac_schedule": dom["frac_schedule"],
                    "frac_textbook": dom["frac_textbook"], "frac_of_8000": round(dom["achieved_gbs"] / 8000.0, 4),
                    "traffic": dom["traffic"], "dram_frac": dom["dram_frac"], "peak_source": peak_src,
                    "sgm_stage": dict(stage(sgm_sched, sgm_wall_ms or sgm_ms), textbook_bytes=int(sgm_text), frac_textbook=round(sgm_text / (sgm_wall_ms or sgm_ms) / 1e6 / peak, 4) if sgm_ms else None,
                                      ms_launches_one_after_the_other=round(sgm_serial_ms or sgm_ms, 4),
                                      note="wall time of the stage in the default pass (first launch to last, launches may overlap) against the bytes its schedule must move"),
                    "kernel_table_pass": {"ms_per_step": round(serial_ms / args.steps, 4), "what": "same frames, SVA_SGM_HSTORE=1: the launches one after the other (kernel times, shares, roofline of the dominant kernel); `value` is the default, overlapped pass"},
                    "cost_volume_stage": dict(stage(k1_bytes, k1_ms), note="K1a + K1b against SURVEY §8(d)'s N_cam*H*W + 2*H*W*D; bound by the integer pipe / L1TEX, not by HBM (DESIGN.md §4)")}
        out = {
            "metric": "MDE/s", "value": round(value, 1), "unit": "MDE/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(total_ms / args.steps, 4), "higher_is_better": True, "scaling": "strong" if batch > 1 else "weak", "vs_baseline": None, "dtype": "u16",
            "data": "synthetic", "frames_per_s": round(frames_step_total * args.steps / (total_ms / 1e3), 2),
            "config": {"workload": "%s: %s" % (name, cfg["desc"]), "width": p.width, "height": p.height, "num_disp": p.num_disp, "cameras": n_cam,
                       "pairs": p.n_pairs, "win_half": p.win_half, "sgm_paths": p.n_paths, "frames_per_step_per_gpu": frames_rank,
                       "partitioning": "independent frames per GPU, no data-path collective" if world > 1 else "single GPU",
                       "l2": "no flush: each volume (%.0f MB) exceeds the 126 MB L2" % (p.width * p.height * p.num_disp * 2 / 1e6)},
            "e2e": {"value": round(e2e_value, 1), "unit": "MDE/s", "ms_per_step": round(e2e_ms / args.steps, 4), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "sva_stream_submit / sva_stream_wait (C ABI, pinned host buffers, two frames in flight: a THROUGHPUT figure)",
                    "single_call_ms_per_step": round(single_ms / args.steps, 4), "single_call_api": "sva_depth_from_array, one synchronous call per frame (the latency a one-frame user sees)"},
            "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks, "kernels": rows,
        }
        # ---- CPU baselines (rank 0, N = 1): bounded samples on the box's host cores ----
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline_legs(args, name, p)
            try:
                out["literal_mode"] = literal_mode_line(p.width, p.height)
            except Exception as ex:  # reported, never fatal for the headline line
                out["literal_mode"] = {"error": str(ex)[:200]}
        else:
            out["cpu_baseline"] = None
    # ---- the multi-GPU configurations north_star names, on the same ranks: extra keys of the same line ----
    if not args.no_extras:
        with Watchdog(args.extras_timeout, rank, out):
            ex = {}
            for key, fn in (("c4_strong", run_c4_strong), ("c3", run_c3)):
                try:
                    ex[key] = fn(args, R)
                except Exception as e:  # noqa: BLE001 — reported in the line
                    ex[key] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
            if out is not None:
                out.update(ex)
    if rank == 0:
        emit(json.dumps(out))
    R.close()


class Watchdog:
    """the extra configurations must never cost the headline line: after `seconds` rank 0 prints the line it has and every rank exits"""

    def __init__(self, seconds, rank, out):
        import threading
        self.t = threading.Timer(seconds, self.fire)
        self.t.daemon = True
        self.rank, self.out, self.seconds = rank, out, seconds

    def fire(self):
        if self.rank == 0 and self.out is not None:
            self.out["extras_error"] = "the multi-GPU extras did not finish within %d s" % self.seconds
            emit(json.dumps(self.out))
        os._exit(0)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.t.cancel()
        return False


def cpu_baseline_legs(args, name, p):
    """BASELINE.md §4 on the GPU box's host cores, each a bounded sample: CPU-fast (the parity oracle's OpenMP volume pipeline — the headline
    `value`, same unit as the GPU line), CPU-ref-1T and CPU-ref-MT (the reference's algorithm restated: per-candidate brute-force 40x40 SAD
    over Bresenham candidates, one thread as the reference runs, and OpenMP over rows), in the reference arm's unit."""
    from oracle.oracle import Oracle
    orc = Oracle()
    band = min(p.height, args.cpu_band)
    scb = configs.scene(name, frame=0, height=band)
    pb = abi.make_params(p.width, band, p.num_disp, configs.offsets(name), win_half=args.win_half, n_paths=p.n_paths, lr_gx=-1, subpixel=1)
    orc.depth_from_array(pb, scb["ref"], scb["others"], scb["mask"])  # warm-up
    best = 1e30
    for _ in range(3):
        t0 = time.perf_counter()
        orc.depth_from_array(pb, scb["ref"], scb["others"], scb["mask"])
        best = min(best, time.perf_counter() - t0)
    cpu = {"value": round(p.width * band * p.num_disp / 1e6 / best, 2), "unit": "MDE/s", "cores": orc.num_threads(), "kind": "port",
           "sample": "CPU-fast: oracle/sva_oracle.c volume pipeline (OpenMP) on a %dx%d row band of the %s frame, D=%d, %d pairs, best of 3" % (p.width, band, name, p.num_disp, p.n_pairs)}
    try:
        w, rows = p.width, 64
        lit = synth.make_literal_scene(rows, w, 7000)
        cams = [abi.camera(*c) for c in synth.reference_cameras(w)]
        mask = np.zeros((rows, w), np.uint8)
        mask[20:rows - 20, 20:w - 20] = 255
        ev = literal_evals(w, rows)
        legs = {}
        for key, nt in (("ref_1t", 1), ("ref_mt", orc.num_threads())):
            best = 1e30
            for _ in range(2):
                t0 = time.perf_counter()
                orc.match_literal(lit["images"], cams, [(12, 11)], mask, 20, 0.5, 1.0, n_threads=nt)
                best = min(best, time.perf_counter() - t0)
            legs[key] = {"value": round(ev / 1e6 / best, 3), "unit": "MDE/s (pixel x candidate evaluations)", "cores": nt, "seconds": round(best, 3)}
        cpu["reference_algorithm"] = dict(legs, sample="oracle restatement of src/CameraStereoVision.cpp:49-95 on a %dx%d band, pair {12,11}, best of 2; "
                                          "full-frame time = linear extrapolation by rows (x %.1f)" % (w, rows, (p.height - 40) / (rows - 40)))
    except Exception as ex:  # noqa: BLE001
        cpu["reference_algorithm"] = {"error": str(ex)[:200]}
    return cpu


def run_c4_strong(args, R):
    """c4 (64 frames x 1920x1080, 9 cameras, D = 192): the frames of the batch partitioned over the ranks, no data-path collective.
    Strong scaling: `ms_per_step` is the whole 64-frame batch."""
    from stereovisionarray_b200 import dist as sdist
    from stereovisionarray_b200.pipeline import DepthContext
    name = "c4"
    p = configs.params(name, win_half=args.win_half)
    batch = configs.CONFIGS[name]["frames"]
    fb, fe = sdist.frame_range(batch, R.world, R.rank)
    sc = configs.scene(name, frame=fb)
    ctx = DepthContext(R.local_rank)
    try:
        ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
        for _ in range(3):
            ctx.run(abi.STAGE_ALL)
        ctx.synchronize()
        steps = args.steps
        R.barrier()
        ms = ctx.time(abi.STAGE_ALL, steps * (fe - fb))
        R.barrier()
        ms = R.max(ms) / steps
    finally:
        ctx.close()
    return {"workload": "c4: " + configs.CONFIGS[name]["desc"], "scaling": "strong", "n_gpus": R.world, "frames_per_step": batch, "frames_per_gpu": fe - fb,
            "ms_per_step": round(ms, 3), "frames_per_s": round(batch / (ms / 1e3), 2), "value": round(batch * configs.mde_per_frame(name) / (ms / 1e3), 1), "unit": "MDE/s",
            "steps": steps, "timing": "CUDA events on the library's stream, inputs resident, max over ranks"}


def run_c3(args, R, headline=False):
    """c3 (one 3840x2160x256 frame, 16 cameras): on one GPU the whole frame; on several the row-block pipeline with peer-direct hand-off
    (sva_rows_*: no volume ever crosses GPUs, the path-line state of the row-sweeping directions is stored straight into the next GPU's
    memory).  Two figures: the latency of one frame with all ranks starting together, and frames back to back with `in_flight` contexts per
    GPU (the sweeps of consecutive frames fill each other's pipeline bubbles)."""
    from stereovisionarray_b200 import dist as sdist
    from stereovisionarray_b200.pipeline import DepthContext
    name = "c3"
    cfg = configs.CONFIGS[name]
    p = configs.params(name, win_half=args.win_half)
    sc = configs.scene(name, frame=0)
    mde = configs.mde_per_frame(name)
    world, rank = R.world, R.rank
    steps = args.steps
    base = {"workload": "c3: " + cfg["desc"], "scaling": "strong", "n_gpus": world, "unit": "MDE/s", "steps": steps,
            "timing": "CUDA events on the library's streams, inputs resident, max over ranks"}
    if world == 1:
        ctx = DepthContext(R.local_rank)
        try:
            ctx.upload(p, sc["ref"], sc["others"], sc["mask"])
            for _ in range(2):
                ctx.run(abi.STAGE_ALL)
            ctx.synchronize()
            l0 = ctx.launches()
            ms = ctx.time(abi.STAGE_ALL, steps) / steps
            launches = ctx.launches() - l0
            if headline and args.dump_outputs:
                disp, sub = ctx.download_disparity()  # the maps the last timed step left on the device
                dump_outputs(args.dump_outputs, {"disparity": disp, "subpixel": sub})
        finally:
            ctx.close()
        res = dict(base, scheme="single GPU: the whole frame, no exchange", latency_ms=round(ms, 3), ms_per_frame=round(ms, 3), frames_per_s=round(1e3 / ms, 2),
                   value=round(mde / (ms / 1e3), 1))
    elif headline and args.c3_scheme != "rows_direct":
        res = dict(base, **run_c3_host_sequenced(args, R, p, sc, steps))
        launches = res.pop("launches")
    else:
        max_in_flight = 3
        ctxs = [DepthContext(R.local_rank) for _ in range(max_in_flight)]
        try:
            for c in ctxs[1:]:  # ONE stream for all of them: frames are interleaved by enqueue order, never by concurrent kernels
                c.set_stream(ctxs[0].get_stream())
            for c in ctxs:
                c.upload(p, sc["ref"], sc["others"], sc["mask"])
                sdist.rows_direct_connect(c, p, rank, world)
            for c in ctxs:  # warm-up: allocates every workspace
                c.rows_run()
            for c in ctxs:
                c.rows_download()
            l0 = ctxs[0].launches()
            lat = 0.0
            for _ in range(steps):  # latency: one frame, all ranks start together
                R.barrier()
                ctxs[0].timer_start()
                ctxs[0].rows_run()
                lat += R.max(ctxs[0].timer_stop())
                ctxs[0].rows_download()  # checks the hand-off time-outs
            lat /= steps
            launches = (ctxs[0].launches() - l0) // steps
            # frames back to back (`steps` frames per run) with P = 1, 2, 3 frames in flight per GPU (P contexts on one stream): phase 0 of
            # frame f is enqueued before phase 1 of frame f - P + 1, so a rank spends the wait for the far end of its second sweep on the next
            # frames' first halves
            by_in_flight = {}
            for in_flight in range(1, max_in_flight + 1):
                frames = steps
                use = ctxs[:in_flight]
                R.barrier()
                ctxs[0].timer_start()
                for f in range(frames + in_flight - 1):
                    if f < frames:
                        use[f % in_flight].rows_run_phase(0)
                    if f - in_flight + 1 >= 0:
                        use[(f - in_flight + 1) % in_flight].rows_run_phase(1)
                by_in_flight[in_flight] = R.max(ctxs[0].timer_stop()) / frames
                for c in use:
                    c.rows_download()
            # three frames in flight in the three-part form (sva_rows_run_part): part 0 of frame f, part 1 of frame f - 1, part 2 of frame f - 2 —
            # every wait for a neighbour's state sits behind a later frame's cost volume, which needs no neighbour
            if max_in_flight >= 3:
                frames = steps
                use = ctxs[:3]
                R.barrier()
                ctxs[0].timer_start()
                for f in range(frames + 2):
                    if f < frames:
                        use[f % 3].rows_run_part(0)
                    if 0 <= f - 1 < frames:
                        use[(f - 1) % 3].rows_run_part(1)
                    if f - 2 >= 0:
                        use[(f - 2) % 3].rows_run_part(2)
                by_in_flight["3 (three parts)"] = R.max(ctxs[0].timer_stop()) / frames
                for c in use:
                    c.rows_download()
            R.barrier()
            # The sweeps as a software pipeline ACROSS the ranks.  In the orders above every rank enqueues "its sweep of frame f" at the same point
            # of the same iteration, so the hand-off still ripples rank by rank inside one iteration and each rank idles while it does.  Skewed
            # by chain position, iteration i of rank r runs the cost volume of frame i, its FIRST sweep of frame i - 1 - min(pd, pu) and its second
            # sweep + K3 of frame i - 1 - max(pd, pu) (pd = r, pu = G - 1 - r: hops from the start of the down / up chain): the state a sweep needs
            # was produced by the neighbour ONE ITERATION EARLIER, so no wait ever blocks.  Needs G + 1 contexts per GPU (frames in flight);
            # reported as the steady-state slope between a `steps`- and a 3 x `steps`-frame run and as the average of the longer run (fill and
            # drain included).
            skew = None
            try:
                G = world
                P = G + 1
                while len(ctxs) < P:
                    c = DepthContext(R.local_rank)
                    ctxs.append(c)
                    c.set_stream(ctxs[0].get_stream())
                    c.upload(p, sc["ref"], sc["others"], sc["mask"])
                    sdist.rows_direct_connect(c, p, rank, world)
                    c.rows_run()
                    c.rows_download()
                pd, pu = rank, G - 1 - rank
                lag1, lag2 = 1 + min(pd, pu), 1 + max(pd, pu)
                t_run = {}
                short, long = steps, 3 * steps
                for frames in (short, long):
                    R.barrier()
                    ctxs[0].timer_start()
                    for i in range(frames + G):
                        if i < frames:
                            ctxs[i % P].rows_run_part(0)
                        if 0 <= i - lag1 < frames:
                            ctxs[(i - lag1) % P].rows_run_part(1)
                        if 0 <= i - lag2 < frames:
                            ctxs[(i - lag2) % P].rows_run_part(2)
                    t_run[frames] = R.max(ctxs[0].timer_stop())
                    for c in ctxs:
                        c.rows_download()
                skew = {"contexts_per_gpu": P, "frames_per_run": [short, long], "ms_per_frame_steady_state": round((t_run[long] - t_run[short]) / (long - short), 3),
                        "ms_per_frame_long_run": round(t_run[long] / long, 3),
                        "order": "iteration i of rank r: part 0 of frame i, part 1 of frame i - 1 - min(r, G-1-r), part 2 of frame i - 1 - max(r, G-1-r) (sva_rows_run_part)"}
                by_in_flight["%d (skewed by chain position, %d frames incl. fill and drain)" % (P, long)] = t_run[long] / long
            except Exception as e:  # noqa: BLE001 — the figures above stand on their own
                skew = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
            R.barrier()
            in_flight = min(by_in_flight, key=by_in_flight.get)
            thr = by_in_flight[in_flight]
        finally:
            for c in reversed(ctxs):  # the borrowers first: ctxs[0] owns the stream they run on
                c.close()
        blocks = sdist.row_blocks(p.height, world)[1]
        res = dict(base, scheme="row blocks %s end to end (sva_rows_*): cost volume and horizontal paths local, row-sweeping paths continue across GPUs — each march stores "
                                "%.1f MB of path state straight into the next GPU's memory (CUDA IPC over NVLink), sequenced by device flags; no volume collective, no NCCL on the data path"
                                % (blocks, 3 * p.width * p.num_disp * 2 / 1e6),
                   latency_ms=round(lat, 3), latency_value=round(mde / (lat / 1e3), 1), in_flight=in_flight, ms_per_frame=round(thr, 3), frames_per_s=round(1e3 / thr, 2),
                   ms_per_frame_by_in_flight={str(k): round(v, 3) for k, v in by_in_flight.items()}, skewed_pipeline=skew,
                   value=round(mde / (thr / 1e3), 1), parity="tools/check_sharded.py --c3: bit-exact against the oracle digests (profiles/)")
    if not headline:
        return res
    # `--config c3` as the headline: the contract's keys, value = frames back to back
    peak, peak_src = measured_peak()
    return {"metric": "MDE/s", "value": res["value"], "unit": "MDE/s", "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": res["ms_per_frame"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u16", "data": "synthetic", "frames_per_s": res["frames_per_s"],
            "config": {"workload": res["workload"], "width": p.width, "height": p.height, "num_disp": p.num_disp, "cameras": p.n_pairs + 1, "pairs": p.n_pairs, "win_half": p.win_half,
                       "sgm_paths": p.n_paths, "partitioning": res["scheme"], "l2": "no flush: each volume (%.0f MB) exceeds the 126 MB L2" % (p.width * p.height * p.num_disp * 2 / 1e6)},
            "c3": res, "e2e": None, "gpu_launches": int(launches), "roofline": {"bound": "hbm", "peak": peak, "peak_source": peak_src, "note": "see the c1 line for per-kernel rooflines"},
            "cpu_baseline": None}


def run_c3_host_sequenced(args, R, p, sc, steps):
    """the schemes whose exchange steps are NCCL collectives issued from Python (kept for comparison, DESIGN.md §7): 'pairs' = north_star's pair
    sharding + packed reduce of the AD volume onto rank 0; 'slices' = disparity slices / directions / row blocks; 'rows' = the row-block pipeline
    with NCCL send / recv hops.  Timed with CUDA events on torch's current stream, which the library is told to run on."""
    import torch
    import torch.distributed as dist
    from stereovisionarray_b200 import dist as sdist
    from stereovisionarray_b200.pipeline import DepthContext
    rank, world = R.rank, R.world
    ctx = DepthContext(R.local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    scheme, keep = args.c3_scheme, {}
    b, e = sdist.pair_ranges(p.n_pairs, world)[rank]
    ctx.upload(sdist.slice_params(p, rank, world) if scheme == "slices" else p, sc["ref"], sc["others"], sc["mask"])
    if scheme == "pairs":
        ptr, nbytes = ctx.ad_device_ptr()
        vol = torch.as_tensor(sdist._CudaAlias(ptr, nbytes // 4), device="cuda")

    def step():
        if scheme == "slices":
            sdist.slice_sharded_compute(ctx, p, rank, world, None, keep)
        elif scheme == "rows":
            sdist.row_sharded_compute(ctx, p, rank, world, None, keep)
        else:
            if e > b:
                ctx.set_pair_range(b, e)
                ctx.run(abi.STAGE_AD)
            else:
                vol.zero_()
            dist.reduce(vol, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                ctx.mark_ad_ready()
                ctx.run(abi.STAGE_BOX)
                ctx.run(abi.STAGE_SGM)
    try:
        for _ in range(2):
            step()
        l0 = ctx.launches()
        R.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        R.barrier()
        ms = R.max(e0.elapsed_time(e1)) / steps
        launches = (ctx.launches() - l0) // steps
    finally:
        ctx.close()
    mde = configs.mde_per_frame("c3")
    return {"scheme": "%s (host-sequenced NCCL exchange; see DESIGN.md §7)" % scheme, "latency_ms": round(ms, 3), "ms_per_frame": round(ms, 3), "frames_per_s": round(1e3 / ms, 2),
            "value": round(mde / (ms / 1e3), 1), "launches": launches}


def run_literal(args, R):
    """`--config literal`: the REFERENCE'S OWN algorithm (src/CameraStereoVision.cpp:49-95 + improveWithDisparity) on the GPU, in the
    reference arm's unit and on its frame size, so that this line and `--impl reference --config literal` are like for like:
    MDE = pixel x candidate evaluations of pair {12,11} on a 1280-wide frame."""
    import ctypes as C
    from stereovisionarray_b200 import reference_api as api
    from stereovisionarray_b200._lib import lib
    w, h = configs.CONFIGS["c1"]["width"], configs.CONFIGS["c1"]["height"]
    sc = synth.make_literal_scene(h, w, 7000)
    cams = [api.Camera(f, pos, ps) for pos, f, ps in synth.reference_cameras(w)]
    mask = np.zeros((h, w), np.uint8)
    mask[20:h - 20, 20:w - 20] = 255
    hnd = api._context(R.local_rank)
    L = lib()

    def step():
        return api.improveWithDisparity(api.matchLiteral(sc["images"], cams, [(12, 11)], mask, 20, 0.5, 1.0), sc["images"][12], [sc["images"][11]], [(cams[12], cams[11])], 21, mask)
    for _ in range(args.warmup):
        step()
    n0 = C.c_uint64(); L.sva_kernel_launches(hnd, C.byref(n0))
    sampler = ClockSampler(R.local_rank) if R.rank == 0 else None
    R.barrier()
    L.sva_timer_start(hnd)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        improved = step()
    wall = time.perf_counter() - t0
    ms = C.c_float(); L.sva_timer_stop(hnd, C.byref(ms))
    R.barrier()
    clocks = sampler.stop() if sampler else None
    n1 = C.c_uint64(); L.sva_kernel_launches(hnd, C.byref(n1))
    dev_ms, wall_ms = R.max(ms.value), R.max(wall * 1e3)
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"improved": improved})
    ev = literal_evals(w, h, stride=64) / 1e6
    if R.rank == 0:
        peak, peak_src = measured_peak()
        out = {"metric": "MDE/s", "value": round(R.world * ev * args.steps / (dev_ms / 1e3), 1), "unit": "MDE/s", "n_gpus": R.world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": round(dev_ms / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
               "config": {"workload": "literal: the reference driver's loop nest (SAD 40x40 over Bresenham candidates, first-min WTA) + improveWithDisparity, pair {12,11}",
                          "width": w, "height": h, "mde_definition": "pixel x candidate evaluations, as --impl reference", "mde_per_frame": round(ev, 2),
                          "value_timing": "CUDA events on the library's stream around the host-buffer calls (the copies are on that stream too: this API has no resident form)"},
               "e2e": {"value": round(R.world * ev * args.steps / (wall_ms / 1e3), 1), "unit": "MDE/s", "ms_per_step": round(wall_ms / args.steps, 4),
                       "h2d_bytes_per_step": 4 * w * h + 4 * w * h, "d2h_bytes_per_step": 2 * w * h,
                       "api": "sva_match_literal + sva_improve_with_disparity (host buffers in and out, wall clock around the calls)"},
               "gpu_launches": int(n1.value - n0.value), "roofline": {"bound": "alu", "peak": peak, "peak_source": peak_src, "note": "plane SAD + raw box sums per candidate offset: integer-pipe bound, see DESIGN.md §2"},
               "cpu_baseline": None, "clocks": clocks}
        emit(json.dumps(out))
    R.close()


def _ref_band_worker(job):
    """one band through the reference's own main() (loop nest src/CameraStereoVision.cpp:49-95); returns (seconds, pixel*candidate evaluations)"""
    w, band, seed = job
    import contextlib
    import io
    from oracle.oracle import Oracle, Reference
    r = Reference()
    sc = synth.make_literal_scene(band, w, seed)
    mask = np.zeros((band, w), np.uint8)
    mask[20:band - 20, 20:w - 20] = 255
    up = [np.repeat(np.repeat(i, 2, axis=0), 2, axis=1) for i in sc["images"]]
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)  # the driver prints to std::cout
    try:
        t0 = time.perf_counter()
        disp, _, _ = r.main_run(up, mask)
        dt = time.perf_counter() - t0
    finally:
        os.dup2(saved, 1); os.close(devnull); os.close(saved)
    return dt, literal_evals(w, band)


def literal_evals(w, h, stride=16):
    """pixel x candidate evaluations of the reference's loop nest for pair {12,11} on a w x h frame (geometry only; every `stride`-th
    column is walked and scaled)"""
    from oracle.oracle import Oracle
    o = Oracle()
    cams = [abi.camera(*c) for c in synth.reference_cameras(w)]
    hx, hy = w // 2, h // 2
    evals = 0
    for y in range(20, h - 20):
        for x in range(20, w - 20, stride):
            ray = o.camera_inv_project(cams[12], (x - hx, y - hy))
            a = o.camera_project(cams[11], [cams[12].pos[i] + ray[i] * 0.5 for i in range(3)])
            b = o.camera_project(cams[11], [cams[12].pos[i] + ray[i] * 1.0 for i in range(3)])
            a, b = (a[0] + hx, a[1] + hy), (b[0] + hx, b[1] + hy)
            if min(a[0], b[0]) < 20 or max(a[0], b[0]) > w - 20 or min(a[1], b[1]) < 20 or max(a[1], b[1]) > h - 20:
                continue
            evals += stride * (max(abs(a[0] - b[0]), abs(a[1] - b[1])) + 1)
    return evals


def literal_mode_line(w, h, reps=5):
    """the reference's OWN algorithm (SAD 40x40 over the Bresenham candidates, first-min WTA, improveWithDisparity) on the GPU through the
    C ABI, whole w x h frame, host buffers in and out — the like-for-like counterpart of `--impl reference` (same MDE definition)"""
    from stereovisionarray_b200 import reference_api as api
    sc = synth.make_literal_scene(h, w, 7000)
    cams = [api.Camera(f, pos, ps) for pos, f, ps in synth.reference_cameras(w)]
    mask = np.zeros((h, w), np.uint8)
    mask[20:h - 20, 20:w - 20] = 255
    run = lambda: api.improveWithDisparity(api.matchLiteral(sc["images"], cams, [(12, 11)], mask, 20, 0.5, 1.0), sc["images"][12], [sc["images"][11]],
                                           [(cams[12], cams[11])], 21, mask)
    run()
    t0 = time.perf_counter()
    for _ in range(reps):
        run()
    dt = (time.perf_counter() - t0) / reps
    ev = literal_evals(w, h, stride=64)
    return {"ms_per_frame": round(dt * 1e3, 3), "value": round(ev / 1e6 / dt, 1), "unit": "MDE/s (pixel x candidate evaluations, as --impl reference)",
            "api": "sva_match_literal + sva_improve_with_disparity (host buffers, wall clock)", "frame": "%dx%d, pair {12,11}, mask = interior" % (w, h)}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    from oracle.oracle import Reference
    name = args.config
    cfg = configs.CONFIGS["c1" if name == "literal" else name]
    if not Reference.available():
        emit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libsva_ref.so missing (built only where /root/reference exists)"}))
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    w, band = cfg["width"], args.ref_band
    ctxm = mp.get_context("fork")
    times = []
    with ctxm.Pool(cores) as pool:
        for step in range(args.warmup + args.steps):
            res = pool.map(_ref_band_worker, [(w, band, 7000 + 100 * step + i) for i in range(cores)])
            if step >= args.warmup:  # the bands run concurrently: a step lasts as long as its slowest band (scene synthesis is not timed)
                times.append((max(t for t, _ in res), sum(e for _, e in res)))
    tot_t = sum(t for t, _ in times)
    tot_e = sum(e for _, e in times)
    v = tot_e / 1e6 / tot_t
    sample = ("UNMODIFIED reference main() (oracle/_ref): SAD 40x40 + first-min WTA + improveWithDisparity on %d independent %dx%d bands per step "
              "(one per core; the reference is single-threaded and has no multi-pair sum / SGM), pair {12,11}, MDE = pixel x candidate evaluations.  "
              "Like for like with `bench.py --config literal` (the same algorithm on the GPU, same unit and frame width), NOT with the default c1 line (8-pair volume + 8-path SGM, "
              "array-level cells).  Caveat: compiled against oracle/cvshim, whose Mat expression path allocates and zero-fills a temporary per getAbsDiff call (~1.6 us per 40x40 SAD); "
              "a real OpenCV 4.2 build is likely 2-4x faster" % (cores, w, band))
    out = {"impl": "reference", "metric": "MDE/s", "value": round(v, 3), "unit": "MDE/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": round(1e3 * tot_t / max(1, len(times)), 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": {"workload": ("literal: the reference driver's loop nest (SAD 40x40 over Bresenham candidates, first-min WTA) + improveWithDisparity, pair {12,11}" if name == "literal"
                                   else "%s: %s" % (name, cfg["desc"])), "width": w, "band_rows": band, "mde_definition": "pixel x candidate evaluations"},
           "cpu_baseline": {"value": round(v, 3), "unit": "MDE/s", "cores": cores, "kind": "reference", "sample": sample},
           "e2e": {"value": round(v, 3), "unit": "MDE/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(json.dumps(out))


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every map as <out_dir>/<name>.npy in float32 (u8 / u16 disparities are exact in float32).  Maps of more than
    DUMP_BYTES in all (c3) keep a fixed sample of rows drawn with seed 0, the same rows of every map, listed in sample_rows.npy."""
    arrays = {name: np.asarray(a, dtype=np.float32) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        h = next(iter(arrays.values())).shape[0]
        keep = h * (DUMP_BYTES - 2**20) // total  # 1 MiB left for the row list and the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(h, keep, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class StdoutToStderr:
    """NCCL / torchrun print banners on fd 1; the contract is ONE JSON line on stdout, so everything else goes to stderr"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


_real_print = print


def emit(line):
    """the single JSON line, written to the REAL stdout even while fd 1 is redirected"""
    os.write(_STDOUT_FD, (line + "\n").encode())


_STDOUT_FD = os.dup(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c1", choices=sorted(configs.CONFIGS) + ["literal"],
                    help="c0..c4 = BASELINE.json's configurations (volume pipeline); literal = the reference's own algorithm, like for like with --impl reference")
    ap.add_argument("--win-half", type=int, default=20)
    ap.add_argument("--impl", default="sva", choices=["sva", "reference"])
    ap.add_argument("--cpu-band", type=int, default=256, help="rows of the CPU-baseline sample")
    ap.add_argument("--ref-band", type=int, default=44, help="rows per band of the reference arm (40 + valid rows)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--c3-scheme", default="rows_direct", choices=["pairs", "slices", "rows", "rows_direct"],
                    help="--config c3 only: 'rows_direct' (default) = row blocks end to end with peer-direct hand-off (sva_rows_*); 'rows' = the same pipeline with NCCL send/recv hops; "
                         "'pairs' = north_star's pair sharding + NCCL reduce of the AD volume; 'slices' = disparity-slice / direction / row sharding (DESIGN.md §7)")
    ap.add_argument("--no-extras", action="store_true", help="skip the c4-strong and c3 runs that the default line carries as extra keys")
    ap.add_argument("--extras-timeout", type=int, default=420, help="seconds after which the line is printed without the extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the maps rank 0 received in the last timed step as DIR/<name>.npy "
                                                          "(float32): disparity and subpixel, or improved for --config literal; c3 keeps a seeded sample of "
                                                          "rows (sample_rows.npy) and is dumped on one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "sva" or (args.config == "c3" and dist_env()[2] > 1)):
        ap.error("--dump-outputs covers --impl sva, and --config c3 on one GPU")
    args.warmup = max(args.warmup, 3) if args.impl == "sva" else args.warmup
    with StdoutToStderr():
        if args.impl == "reference":
            run_reference(args)
        else:
            run_sva(args)


if __name__ == "__main__":
    main()
