"""Multi-GPU sharding of the depth path on one 8xB200 box (SURVEY §8e) — one process per GPU, torch.distributed for plumbing.

Natural partitions, nothing else:
  * frames of a capture batch are independent units -> rank r takes frames [r*F/G, (r+1)*F/G); NO data-path collective;
  * camera pairs of ONE frame: the cost volume is a sum over pairs (integer, associative, commutative), so each rank
    computes the AD partial of its pair range over the full [H][W][D] volume and the partials are sum-reduced onto the
    rank that owns the reference view, which then runs the box filter, SGM and WTA.  NCCL has no 16-bit integer type, so
    the u16 volume is reduced as packed int32 (two cells per word): totals are <= 255 * n_pairs <= 8160 < 2^15, so no
    carry crosses the half-word boundary and the sign bit is never set — bit-exact in any reduction order.

The compute backend is an object with upload / set_pair_range / run / ad_device_ptr ... (stereovisionarray_b200.pipeline.
DepthContext on GPUs).  The helper functions below are pure host logic and are exercised on CPU with the gloo backend."""
import numpy as np


def frame_range(n_frames, world, rank):
    """contiguous, balanced: the first (n_frames % world) ranks get one extra frame"""
    base, extra = divmod(n_frames, world)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def pair_ranges(n_pairs, world):
    """balanced contiguous pair ranges, e.g. 15 pairs over 8 ranks -> 2,2,2,2,2,2,2,1 (ranks beyond the pairs get empty ranges)"""
    out = []
    base, extra = divmod(n_pairs, world)
    b = 0
    for r in range(world):
        e = b + base + (1 if r < extra else 0)
        out.append((b, e))
        b = e
    return out


def packed_no_carry(n_pairs):
    """the packed-int32 reduce is exact iff the full sum of a cell stays below 2^15"""
    return 255 * n_pairs < (1 << 15)


def reduce_packed_u16(t_int32, dst, group=None):
    """sum-reduce a packed-u16x2 volume (viewed as int32) onto rank `dst`; in place on dst"""
    import torch.distributed as dist
    dist.reduce(t_int32, dst=dst, op=dist.ReduceOp.SUM, group=group)
    return t_int32


class _CudaAlias:
    """zero-copy torch view of a device buffer owned by libsva_b200.so"""

    def __init__(self, ptr, n_int32):
        self.__cuda_array_interface__ = {"shape": (n_int32,), "typestr": "<i4", "data": (ptr, False), "version": 3, "strides": None}


def pair_sharded_depth(ctx, p, ref, others, mask, rank, world, owner=0, group=None):
    """One frame, pairs sharded over `world` GPUs (config c3).  Every rank holds the frame's images; returns (disp, subpix) on the
    owner rank and None elsewhere.  ctx must run on torch's current stream (ctx.set_stream) so NCCL and the kernels are ordered."""
    import torch
    from . import abi
    if not packed_no_carry(p.n_pairs):
        raise ValueError("too many pairs for the packed-int32 reduce")
    b, e = pair_ranges(p.n_pairs, world)[rank]
    ctx.upload(p, ref, others, mask)
    ptr, nbytes = ctx.ad_device_ptr()
    vol = torch.as_tensor(_CudaAlias(ptr, nbytes // 4), device="cuda")
    if e > b:
        ctx.set_pair_range(b, e)
        ctx.run(abi.STAGE_AD)
    else:
        vol.zero_()
    if world > 1:
        reduce_packed_u16(vol, owner, group)
    if rank != owner:
        return None
    ctx.mark_ad_ready()
    ctx.run(abi.STAGE_BOX)
    ctx.run(abi.STAGE_SGM)
    return ctx.download_disparity()


def direction_masks(n_paths, world):
    """path directions dealt round-robin: rank r aggregates directions r, r + world, ... (bit i = direction i of the C ABI's order)"""
    return [sum(1 << d for d in range(r, n_paths, world)) for r in range(world)]


def row_blocks(height, world):
    """equal row blocks for the reduce-scatter of the partial aggregation volumes: (rows per block, [(y0, y1)] per rank); the last blocks
    may be short or empty, the volume is padded to rows_per * world rows"""
    rows_per = -(-height // world)
    return rows_per, [(min(height, r * rows_per), min(height, (r + 1) * rows_per)) for r in range(world)]


def slice_params(p, rank, world):
    """rank's disparity slice of p: D / world disparities starting at min_disp + rank * D / world (same pairs, shift, cap, penalties)"""
    if p.num_disp % world or (p.num_disp // world) % 8:
        raise ValueError("num_disp must split into %d slices of a multiple of 8 disparities" % world)
    ps = type(p).from_buffer_copy(p)
    ps.num_disp = p.num_disp // world
    ps.min_disp = p.min_disp + rank * ps.num_disp
    return ps


def slice_sharded_compute(ctx, p, rank, world, group=None, keep=None):
    """Device part of slice_sharded_depth for a frame that is already uploaded on every rank WITH THE RANK'S SLICE PARAMETERS
    (slice_params(p, rank, world): the view staging is laid out for the upload's disparity reach, and the library refuses to run K1a for
    any other — sva_frame_set_params): steps 1-5 below; afterwards the rank's rows of the maps are in the library
    (ctx.download_disparity_rows).  Returns (y0, y1)."""
    import torch
    import torch.distributed as dist
    from . import abi
    keep = keep if keep is not None else {}
    ds = p.num_disp // world
    ctx.set_params(slice_params(p, rank, world))
    ctx.run(abi.STAGE_AD)
    ctx.run(abi.STAGE_BOX)
    cptr, cbytes = ctx.cost_device_ptr()
    cslice = torch.as_tensor(_CudaAlias(cptr, cbytes // 4), device="cuda")
    if keep.get("call") is None or keep["call"].numel() != world * cslice.numel():
        keep["call"] = torch.empty(world * cslice.numel(), dtype=torch.int32, device="cuda")
    call = keep["call"]
    if world > 1:
        dist.all_gather_into_tensor(call, cslice, group=group)
    else:
        call.copy_(cslice)
    ctx.set_params(p)
    rows_per, blocks = row_blocks(p.height, world)
    bits = direction_masks(p.n_paths, world)[rank]
    words_row = p.width * p.num_disp // 2
    if bits:
        sptr, sbytes = ctx.sgm_directions(call.data_ptr(), ds, bits, rows_per * world)
        spart = torch.as_tensor(_CudaAlias(sptr, sbytes // 4), device="cuda")
    else:  # more ranks than directions: nothing to add
        if keep.get("zero") is None or keep["zero"].numel() != rows_per * world * words_row:
            keep["zero"] = torch.zeros(rows_per * world * words_row, dtype=torch.int32, device="cuda")
        spart = keep["zero"]
    if keep.get("srows") is None or keep["srows"].numel() != rows_per * words_row:
        keep["srows"] = torch.empty(rows_per * words_row, dtype=torch.int32, device="cuda")
    srows = keep["srows"]
    if world > 1:
        dist.reduce_scatter_tensor(srows, spart, op=dist.ReduceOp.SUM, group=group)
    else:
        srows.copy_(spart[:srows.numel()])
    y0, y1 = blocks[rank]
    if y1 > y0:
        ctx.wta_rows(srows.data_ptr(), y0, y1 - y0)
    return y0, y1


def slice_sharded_depth(ctx, p, ref, others, mask, rank, world, group=None, keep=None):
    """One frame sharded WITHOUT a volume reduction (the alternative to pair_sharded_depth for configuration c3):
      1. rank r computes its DISPARITY SLICE of the cost volume from all pairs (K1a + K1b, no exchange);
      2. all-gather of the slices (slice-major volume on every rank);
      3. rank r aggregates its share of the SGM DIRECTIONS over the whole volume;
      4. reduce-scatter of the partial sums by ROW BLOCKS (packed int32: 8 paths x 8190 <= 65520, carry-free, bit-exact in any order);
      5. rank r runs WTA / left-right check / sub-pixel on its rows; the maps are gathered on rank 0.
    Every rank holds the frame's images.  ctx must run on torch's current stream.  Returns (disp, subpix) on rank 0, None elsewhere.
    `keep` (a dict) caches the gather / scatter buffers across frames."""
    import torch
    import torch.distributed as dist
    from . import abi
    ctx.upload(slice_params(p, rank, world), ref, others, mask)
    y0, y1 = slice_sharded_compute(ctx, p, rank, world, group, keep)
    rows_per = row_blocks(p.height, world)[0]
    d_t = torch.full((rows_per, p.width), abi.SVA_DISP_INVALID, dtype=torch.int32)
    s_t = torch.full((rows_per, p.width), -1.0, dtype=torch.float32)
    if y1 > y0:
        d, s = ctx.download_disparity_rows(y1 - y0)
        d_t[:y1 - y0] = torch.from_numpy(d.astype(np.int32))
        s_t[:y1 - y0] = torch.from_numpy(s)
    if world == 1:
        return d_t[:p.height].numpy().astype(np.uint16), s_t[:p.height].numpy()
    d_all = [torch.empty_like(d_t, device="cuda") for _ in range(world)] if rank == 0 else None
    s_all = [torch.empty_like(s_t, device="cuda") for _ in range(world)] if rank == 0 else None
    dist.gather(d_t.cuda(), d_all, dst=0, group=group)
    dist.gather(s_t.cuda(), s_all, dst=0, group=group)
    if rank != 0:
        return None
    disp = torch.cat(d_all)[:p.height].cpu().numpy().astype(np.uint16)
    sub = torch.cat(s_all)[:p.height].cpu().numpy()
    return disp, sub


def row_pipeline_steps(rank, world):
    """Hop schedule of the row-block pipeline.  Step s (0 <= s < world - 1) moves the down-sweep state from rank s to s + 1 and the
    up-sweep state from rank world - 1 - s to world - 2 - s.  Returns, per step, what THIS rank does:
    (send_down_to, recv_down_from, send_up_to, recv_up_from), None where it takes no part.  Every rank walks the steps in the same
    order and issues a step's transfers as one batch, so two neighbours that exchange both states in the same step (the middle of
    the array) cannot dead-lock."""
    steps = []
    for s in range(world - 1):
        steps.append((s + 1 if rank == s else None, s if rank == s + 1 else None,
                      world - 2 - s if rank == world - 1 - s else None, world - 1 - s if rank == world - 2 - s else None))
    return steps


def row_sharded_compute(ctx, p, rank, world, group=None, keep=None, device="cuda"):
    """Device part of row_sharded_depth for a frame already uploaded on every rank: the rank's block of image rows end to end.
    Afterwards the block's maps are in the library (ctx.download_disparity_rows).  Returns (y0, y1)."""
    import torch
    import torch.distributed as dist
    from . import abi
    keep = keep if keep is not None else {}
    _, blocks = row_blocks(p.height, world)
    if any(b[1] <= b[0] for b in blocks):
        raise ValueError("row-block pipeline: %d rows do not give every one of %d ranks a block" % (p.height, world))
    y0, y1 = blocks[rank]
    n = y1 - y0
    words = 3 * p.width * p.num_disp // 2  # u16 pairs as int32: NCCL has no 16-bit integer type
    if keep.get("state") is None or keep["state"][0].numel() != words or keep["state"][0].device.type != torch.device(device).type:
        keep["state"] = [torch.empty(words, dtype=torch.int32, device=device) for _ in range(4)]
    d_in, d_out, u_in, u_out = keep["state"]
    ctx.rows_begin(y0, n)
    ctx.run(abi.STAGE_AD)
    ctx.run(abi.STAGE_BOX)
    starts_chain = world > 1 and rank in (0, world - 1)  # these run their (local) horizontal paths after their first block, off the serial chain
    if not starts_chain:
        ctx.sgm_rows(2, y0, n)
    if rank == 0:
        ctx.sgm_rows(0, y0, n, 0, d_out.data_ptr())
    if rank == world - 1:
        ctx.sgm_rows(1, y0, n, 0, u_out.data_ptr())
    if starts_chain:
        ctx.sgm_rows(2, y0, n)
    for send_d, recv_d, send_u, recv_u in row_pipeline_steps(rank, world):
        ops = []
        if send_d is not None:
            ops.append(dist.P2POp(dist.isend, d_out, send_d, group))
        if recv_d is not None:
            ops.append(dist.P2POp(dist.irecv, d_in, recv_d, group))
        if send_u is not None:
            ops.append(dist.P2POp(dist.isend, u_out, send_u, group))
        if recv_u is not None:
            ops.append(dist.P2POp(dist.irecv, u_in, recv_u, group))
        if ops:
            for r in dist.batch_isend_irecv(ops):
                r.wait()
        if recv_d is not None:
            ctx.sgm_rows(0, y0, n, d_in.data_ptr(), d_out.data_ptr())
        if recv_u is not None:
            ctx.sgm_rows(1, y0, n, u_in.data_ptr(), u_out.data_ptr())
    ctx.wta_rows(None, y0, n)
    return y0, y1


def row_sharded_depth(ctx, p, ref, others, mask, rank, world, group=None, keep=None):
    """One frame sharded by ROW BLOCKS end to end — no volume ever crosses GPUs (c3, DESIGN.md §7):
      1. rank r computes the cost volume of its block of image rows (K1a + K1b; the box window reaches win_half rows into the neighbours'
         rows of the IMAGES, which every rank holds — nothing is exchanged);
      2. the horizontal path directions are local to a row;
      3. the three down-sweeping directions run as a pipeline 0 -> G-1, the three up-sweeping ones as a pipeline G-1 -> 0: a rank
         aggregates its block and hands L of every path line at its last row (3 * W * D u16, a few MB) to the next rank;
      4. K3 on the rank's rows; the maps are gathered on rank 0.
    Every rank holds the frame's images.  ctx must run on torch's current stream.  Returns (disp, subpix) on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from . import abi
    ctx.upload(p, ref, others, mask)
    y0, y1 = row_sharded_compute(ctx, p, rank, world, group, keep)
    rows_per = row_blocks(p.height, world)[0]
    d_t = torch.full((rows_per, p.width), abi.SVA_DISP_INVALID, dtype=torch.int32)
    s_t = torch.full((rows_per, p.width), -1.0, dtype=torch.float32)
    d, s = ctx.download_disparity_rows(y1 - y0)
    d_t[:y1 - y0] = torch.from_numpy(d.astype(np.int32))
    s_t[:y1 - y0] = torch.from_numpy(s)
    if world == 1:
        return d_t[:p.height].numpy().astype(np.uint16), s_t[:p.height].numpy()
    d_all = [torch.empty_like(d_t, device="cuda") for _ in range(world)] if rank == 0 else None
    s_all = [torch.empty_like(s_t, device="cuda") for _ in range(world)] if rank == 0 else None
    dist.gather(d_t.cuda(), d_all, dst=0, group=group)
    dist.gather(s_t.cuda(), s_all, dst=0, group=group)
    if rank != 0:
        return None
    return torch.cat(d_all)[:p.height].cpu().numpy().astype(np.uint16), torch.cat(s_all)[:p.height].cpu().numpy()


def rows_direct_connect(ctx, p, rank, world, group=None):
    """Open the C library's row-block link on this rank and map the neighbours' state buffers (CUDA IPC): the 64-byte handles travel over
    torch.distributed as plain bytes (host plumbing; a C++ host would use sva_rows_connect_comm or its own channel).  Collective."""
    import torch.distributed as dist
    ctx.rows_open(p, rank, world)
    if world == 1:
        return
    handles = [None] * world
    dist.all_gather_object(handles, ctx.rows_export(), group=group)
    ctx.rows_connect(handles[rank - 1] if rank > 0 else None, handles[rank + 1] if rank < world - 1 else None)
    dist.barrier(group=group)  # nobody runs ahead of a neighbour that has not mapped its side yet


def rows_stream_connect(ctxs, p, rank, world, group=None):
    """rows_direct_connect for the world + 1 contexts of a pipeline.RowsStream (context j of every rank is one chain): opens every link and
    maps the neighbours' state buffers, with one all-gather of this rank's world + 1 handles.  Collective; create the RowsStream afterwards."""
    import torch.distributed as dist
    if len(ctxs) != world + 1:
        raise ValueError("the skewed order keeps world + 1 = %d frames in flight: that many contexts per GPU" % (world + 1))
    for c in ctxs:
        c.rows_open(p, rank, world)
    if world == 1:
        return
    handles = [None] * world
    dist.all_gather_object(handles, [c.rows_export() for c in ctxs], group=group)
    for j, c in enumerate(ctxs):
        c.rows_connect(handles[rank - 1][j] if rank > 0 else None, handles[rank + 1][j] if rank < world - 1 else None)
    dist.barrier(group=group)


def rows_direct_depth(ctx, p, ref, others, mask, rank, world, group=None):
    """One frame through the peer-direct row-block pipeline (sva_rows_*; rows_direct_connect first): the path-line state is stored by the
    neighbour's march kernel straight into this GPU's memory and sequenced by device flags.  Returns (disp, subpix) on rank 0, None elsewhere."""
    ctx.upload(p, ref, others, mask)
    ctx.rows_run()
    d, s = ctx.rows_download()
    return gather_rows(d, s, p, rank, world, group)


def gather_rows(d, s, p, rank, world, group=None):
    """this rank's block of the maps (DepthContext.rows_download) -> the whole maps (disp, subpix) on rank 0, None elsewhere.  Collective."""
    import torch
    import torch.distributed as dist
    from . import abi
    if world == 1:
        return d, s
    rows_per = row_blocks(p.height, world)[0]
    d_t = torch.full((rows_per, p.width), abi.SVA_DISP_INVALID, dtype=torch.int32)
    s_t = torch.full((rows_per, p.width), -1.0, dtype=torch.float32)
    d_t[:d.shape[0]] = torch.from_numpy(d.astype(np.int32))
    s_t[:d.shape[0]] = torch.from_numpy(s)
    d_all = [torch.empty_like(d_t, device="cuda") for _ in range(world)] if rank == 0 else None
    s_all = [torch.empty_like(s_t, device="cuda") for _ in range(world)] if rank == 0 else None
    dist.gather(d_t.cuda(), d_all, dst=0, group=group)
    dist.gather(s_t.cuda(), s_all, dst=0, group=group)
    if rank != 0:
        return None
    return torch.cat(d_all)[:p.height].cpu().numpy().astype(np.uint16), torch.cat(s_all)[:p.height].cpu().numpy()


def rows_skewed_order(rank, world, frames):
    """Enqueue order of a STREAM of frames through the peer-direct row-block pipeline as a software pipeline across the ranks (DESIGN.md §7):
    -> one list per iteration of (part, frame) pairs for `sva_rows_run_part`, to be enqueued in that order on the rank's one stream, frame f on
    context f % (world + 1).

    A sweep reaches rank r after pd = r hops (down chain) resp. pu = world - 1 - r hops (up chain).  Iteration i of rank r runs part 0 (cost
    volume) of frame i, its first sweep (part 1) of frame i - 1 - min(pd, pu) and its second sweep + K3 (part 2) of frame i - 1 - max(pd, pu):
    the down sweep of a frame then runs on rank r exactly one iteration after it ran on rank r - 1 (and the up sweep one iteration after
    rank r + 1), so the state it waits for is already there and no rank idles inside an iteration — measured on 8 B200: 2.55 ms per c3 frame
    against 4.37 ms when all ranks enqueue a frame's sweeps in the same iteration.  world + 1 contexts per GPU keep the frames in flight."""
    pd, pu = rank, world - 1 - rank
    lag1, lag2 = 1 + min(pd, pu), 1 + max(pd, pu)
    order = []
    for i in range(frames + world):
        step = []
        if i < frames:
            step.append((0, i))
        if 0 <= i - lag1 < frames:
            step.append((1, i - lag1))
        if 0 <= i - lag2 < frames:
            step.append((2, i - lag2))
        order.append(step)
    return order


def rows_direct_stream_steps(ctxs, rank, world, frames, upload=None, download=None):
    """Generator form of rows_direct_stream: each next() enqueues one iteration of rows_skewed_order(rank, world, frames) on this rank, and the
    next() after the last iteration downloads the frames still in the contexts and stops.  One process per GPU simply exhausts it; a process
    that plays several ranks advances one generator per rank round-robin, one iteration each, and runs the same code as production.

    upload(ctx, f) is called right before part 0 of frame f.  download(ctx, f) is called exactly once per frame: at the start of the iteration
    that reuses frame f's context (before upload and part 0 of frame f + world + 1), and for the last min(world + 1, frames) frames after the
    loop, in frame order.  A download may synchronise the device: in the skewed order every wait enqueued on any rank depends only on work
    its neighbour enqueued in an EARLIER iteration (the sweep's state one iteration before, the ack of the context's previous frame at least
    world iterations before), so a host that blocks at the start of iteration i — every rank having enqueued iteration i - 1 — never blocks on
    work that is not enqueued yet."""
    P = world + 1
    if len(ctxs) < P:
        raise ValueError("the skewed order keeps world + 1 = %d frames in flight: that many contexts per GPU" % P)
    for step in rows_skewed_order(rank, world, frames):
        for part, f in step:
            if part == 0:
                if download is not None and f >= P:
                    download(ctxs[(f - P) % P], f - P)
                if upload is not None:
                    upload(ctxs[f % P], f)
            ctxs[f % P].rows_run_part(part)
        yield
    if download is not None:
        for f in range(max(0, frames - P), frames):
            download(ctxs[f % P], f)


def rows_direct_stream(ctxs, rank, world, frames, upload=None, download=None):
    """Drives `frames` frames through world + 1 contexts of this rank (all on ONE stream, each connected with rows_direct_connect) in the
    skewed order (rows_direct_stream_steps: where upload(ctx, f) and download(ctx, f) are called).  Without a download hook a frame's maps
    stay in its context (rows_download) until frame f + world + 1 overwrites them."""
    for _ in rows_direct_stream_steps(ctxs, rank, world, frames, upload, download):
        pass


def numpy_pack(a_u16):
    """[H][W][D] u16 (D even) -> int32 view, the layout the GPU path reduces"""
    return np.ascontiguousarray(a_u16).view(np.int32)


def groups_sharded_depth(ctx, p, images, groups, grid_cols, rank, world, group=None):
    """Every reference view of one array frame (sva_depth_groups), the groups sharded over `world` GPUs: rank r computes the groups
    frame_range(n_groups, world, r) (13 CHESS groups on 8 ranks: 2,2,2,2,2,1,1,1) and passes only the cameras they read, so nothing crosses
    GPUs on the data path.  The maps are gathered on rank 0 -> (disp (G, H, W) uint16, subpix (G, H, W) float32) there, None elsewhere.
    Collective (the gather)."""
    from . import groups as _groups
    groups = _groups.as_groups(groups)
    b, e = frame_range(len(groups), world, rank)
    mine = set(_groups.cameras_of(groups[b:e]))
    d, s = ctx.depth_groups(p, [im if i in mine else None for i, im in enumerate(images)], groups, grid_cols, group_range=(b, e))
    return gather_groups(d, s, p, len(groups), rank, world, group)


def gather_groups(d, s, p, n_groups, rank, world, group=None):
    """this rank's maps of its groups (frame_range) -> all groups' maps on rank 0, None elsewhere.  Collective."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return d, s
    per = frame_range(n_groups, world, 0)[1]  # the largest share
    d_t = torch.zeros((per, p.height, p.width), dtype=torch.int32)
    s_t = torch.zeros((per, p.height, p.width), dtype=torch.float32)
    d_t[:d.shape[0]] = torch.from_numpy(d.astype(np.int32))
    s_t[:d.shape[0]] = torch.from_numpy(s)
    d_all = [torch.empty_like(d_t, device="cuda") for _ in range(world)] if rank == 0 else None
    s_all = [torch.empty_like(s_t, device="cuda") for _ in range(world)] if rank == 0 else None
    dist.gather(d_t.cuda(), d_all, dst=0, group=group)
    dist.gather(s_t.cuda(), s_all, dst=0, group=group)
    if rank != 0:
        return None
    counts = [frame_range(n_groups, world, r)[1] - frame_range(n_groups, world, r)[0] for r in range(world)]
    disp = torch.cat([t[:n] for t, n in zip(d_all, counts)]).cpu().numpy().astype(np.uint16)
    sub = torch.cat([t[:n] for t, n in zip(s_all, counts)]).cpu().numpy()
    return disp, sub
