"""Host-side driver of the volume-mode depth pipeline over the C ABI (one DepthContext per GPU).

Stages (DESIGN.md §4): K1a AD volume -> K1b box/pack -> K2 SGM (four launches for 8 paths: -> storing S, <-, the down-sweeping and the up-sweeping group) -> K3 (WTA / LR / sub-pixel).
All compute happens in libsva_b200.so on the GPU; this module only marshals numpy buffers."""
import ctypes as C

import numpy as np

from . import abi
from . import groups as _groups
from ._lib import SvaError, check, lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _groups_args(images, groups, masks, n_masks):
    """the C layout of sva_depth_groups' frame arguments -> (images, flat pairs, sizes, masks or None, keepalive)"""
    keep = [None if im is None else np.ascontiguousarray(im, dtype=np.uint8) for im in images]
    ims = (abi.SvaImageU8 * max(1, len(keep)))()
    for i, a in enumerate(keep):
        if a is not None:
            ims[i] = abi.SvaImageU8(a.ctypes.data, a.shape[0], a.shape[1], a.strides[0])
    flat = np.array([v for g in groups for pr in g for v in pr] or [0], np.int32)
    sizes = np.array([len(g) for g in groups] or [0], np.int32)
    m_arr = None
    if masks is not None:
        m_arr = (abi.SvaImageU8 * max(1, n_masks))()
        for i, m in enumerate(masks):
            if m is not None:
                a = np.ascontiguousarray(m, dtype=np.uint8)
                keep.append(a)
                m_arr[i] = abi.SvaImageU8(a.ctypes.data, a.shape[0], a.shape[1], a.strides[0])
    return ims, flat, sizes, m_arr, keep


def fuse_params(tol_16=16, min_support=2):
    f = abi.SvaFuseParams()
    f.tol_16, f.min_support = int(tol_16), int(min_support)
    return f


class DepthContext:
    def __init__(self, device=0):
        self._L = lib()
        h = C.c_void_p()
        rc = self._L.sva_create(device, C.byref(h))
        if rc == abi.SVA_ERR_BAD_ARG:  # an A/B switch (DESIGN §8a) outside its documented set
            raise SvaError(rc, "sva_create: " + self._L.sva_last_error(None).decode())
        if rc != 0:
            raise RuntimeError("sva_create(device=%d) failed with %d — a B200 (sm_100) GPU is required; there is no CPU fallback" % (device, rc))
        self._h = h
        self.params = None

    def close(self):
        if self._h:
            self._L.sva_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- staged / resident ----
    def upload(self, p, ref, others, mask=None):
        r, rk = abi.image_u8(np.ascontiguousarray(ref, dtype=np.uint8) if not isinstance(ref, np.ndarray) or ref.dtype != np.uint8 else ref)
        o, ok = abi.image_array(others) if not isinstance(others, tuple) else others
        m = None
        if mask is not None:
            m, mk = abi.image_u8(mask)
        check(self._h, self._L.sva_frame_upload(self._h, C.byref(p), C.byref(r), o, C.byref(m) if m is not None else None))
        self.params = p

    def set_pair_range(self, b, e):
        check(self._h, self._L.sva_frame_set_pair_range(self._h, b, e))

    def set_debug(self, store_full_s=0, sgm_dir_mask=0):
        check(self._h, self._L.sva_frame_set_debug(self._h, int(store_full_s), C.c_uint32(sgm_dir_mask)))

    def run(self, stage=abi.STAGE_ALL):
        check(self._h, self._L.sva_frame_run(self._h, stage))

    def time(self, stage, iters):
        ms = C.c_float()
        check(self._h, self._L.sva_frame_time(self._h, stage, iters, C.byref(ms)))
        return ms.value

    def kernel_times(self, stage=abi.STAGE_ALL):
        names = (C.c_char_p * 64)()
        ms = (C.c_float * 64)()
        n = check(self._h, self._L.sva_frame_kernel_times(self._h, stage, names, ms, 64))
        return [(names[i].decode(), ms[i]) for i in range(min(n, 64))]

    def time_detailed(self, stage, iters):
        """-> (total_ms, {kernel name: (sum_ms, launches)}) with CUDA events on the ctx stream"""
        names = (C.c_char_p * 64)()
        sums = (C.c_float * 64)()
        cnts = (C.c_int32 * 64)()
        tot = C.c_float()
        n = check(self._h, self._L.sva_frame_time_detailed(self._h, stage, iters, C.byref(tot), names, sums, cnts, 64))
        return tot.value, {names[i].decode(): (sums[i], cnts[i]) for i in range(n)}

    def timer_start(self):
        check(self._h, self._L.sva_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float()
        check(self._h, self._L.sva_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def synchronize(self):
        check(self._h, self._L.sva_synchronize(self._h))

    def set_stream(self, stream_ptr):
        """run on a caller-owned CUDA stream (torch.cuda.current_stream().cuda_stream; 0 = the legacy default stream)"""
        check(self._h, self._L.sva_set_stream(self._h, C.c_void_p(stream_ptr)))

    def use_own_stream(self):
        check(self._h, self._L.sva_use_own_stream(self._h))

    def launches(self):
        n = C.c_uint64()
        check(self._h, self._L.sva_kernel_launches(self._h, C.byref(n)))
        return n.value

    def set_guard(self, on=True):
        """debug: device buffers allocated from now on get canary bands and a poisoned payload (see check_guards)"""
        check(self._h, self._L.sva_debug_set_guard(self._h, int(on)))

    def check_guards(self):
        """-> (guarded buffers, overwritten canary bytes); the second number must be 0"""
        n, bad = C.c_int64(), C.c_int64()
        check(self._h, self._L.sva_debug_check_guards(self._h, C.byref(n), C.byref(bad)))
        return n.value, bad.value

    def _shape(self):
        p = self.params
        return (p.height, p.width, p.num_disp)

    def download_ad(self):
        out = np.empty(self._shape(), np.uint16)
        check(self._h, self._L.sva_frame_download_ad(self._h, _p(out, C.c_uint16)))
        return out

    def download_cost(self):
        out = np.empty(self._shape(), np.uint16)
        check(self._h, self._L.sva_frame_download_cost(self._h, _p(out, C.c_uint16)))
        return out

    def download_raw_cost(self):
        out = np.empty(self._shape(), np.uint32)
        check(self._h, self._L.sva_frame_download_raw_cost(self._h, _p(out, C.c_uint32)))
        return out

    def download_sgm(self):
        out = np.empty(self._shape(), np.uint16)
        check(self._h, self._L.sva_frame_download_sgm(self._h, _p(out, C.c_uint16)))
        return out

    def download_disparity(self, disp=None, sub=None):
        p = self.params
        disp = np.empty((p.height, p.width), np.uint16) if disp is None else disp
        sub = np.empty((p.height, p.width), np.float32) if sub is None else sub
        check(self._h, self._L.sva_frame_download_disparity(self._h, _p(disp, C.c_uint16), _p(sub, C.c_float)))
        return disp, sub

    def ad_device_ptr(self):
        ptr, n = C.c_void_p(), C.c_size_t()
        check(self._h, self._L.sva_frame_ad_device_ptr(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def mark_ad_ready(self):
        check(self._h, self._L.sva_frame_mark_ad_ready(self._h))

    # ---- multi-GPU building blocks: disparity-slice / direction / row sharding of one frame (dist.slice_sharded_depth) ----
    def cost_device_ptr(self):
        ptr, n = C.c_void_p(), C.c_size_t()
        check(self._h, self._L.sva_frame_cost_device_ptr(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def set_params(self, p):
        check(self._h, self._L.sva_frame_set_params(self._h, C.byref(p)))
        self.params = p

    def sgm_directions(self, cost_ptr, slice_disp, dir_mask, rows_alloc=0):
        """aggregate the directions of dir_mask on a device cost volume (slice-major when slice_disp > 0) -> (device ptr, bytes) of the partial S"""
        ptr, n = C.c_void_p(), C.c_size_t()
        check(self._h, self._L.sva_frame_sgm_directions(self._h, C.c_void_p(cost_ptr), int(slice_disp), C.c_uint32(dir_mask), int(rows_alloc), C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def wta_rows(self, s_rows_ptr, y0, rows):
        """K3 on image rows [y0, y0 + rows) of S given by device pointer (None / 0: the context's own volume)"""
        check(self._h, self._L.sva_frame_wta_rows(self._h, C.c_void_p(s_rows_ptr or None), int(y0), int(rows)))

    def rows_begin(self, y0, rows):
        """row-block pipeline: zero image rows [y0, y0 + rows) of the aggregation volume"""
        check(self._h, self._L.sva_frame_rows_begin(self._h, int(y0), int(rows)))

    def sgm_rows(self, group, y0, rows, state_in=0, state_out=0):
        """one direction group (0 down-sweeping, 1 up-sweeping, 2 horizontal) on image rows [y0, y0 + rows); state_* = device pointers
        to 3 * W * D u16 (0 = none: the sweep starts / ends in this block)"""
        check(self._h, self._L.sva_frame_sgm_rows(self._h, int(group), int(y0), int(rows), C.c_void_p(state_in or None), C.c_void_p(state_out or None)))

    def download_disparity_rows(self, rows):
        p = self.params
        disp = np.empty((rows, p.width), np.uint16)
        sub = np.empty((rows, p.width), np.float32)
        check(self._h, self._L.sva_frame_download_disparity_rows(self._h, int(rows), _p(disp, C.c_uint16), _p(sub, C.c_float)))
        return disp, sub

    # ---- multi-GPU from C: NCCL communicator, pair-sharded reduce, row-block pipeline with peer-direct hand-off (csrc/sva_dist.cu) ----
    @staticmethod
    def comm_unique_id():
        """rank 0: the 128-byte NCCL id to hand to every rank (bytes)"""
        buf = (C.c_uint8 * abi.SVA_COMM_ID_BYTES)()
        rc = lib().sva_comm_get_unique_id(buf)
        if rc != 0:
            raise RuntimeError("sva_comm_get_unique_id failed with %d (libnccl.so.2 not loadable?)" % rc)
        return bytes(buf)

    def comm_init(self, uid, rank, world):
        check(self._h, self._L.sva_comm_init(self._h, (C.c_uint8 * abi.SVA_COMM_ID_BYTES).from_buffer_copy(uid), int(rank), int(world)))

    def comm_barrier(self):
        check(self._h, self._L.sva_comm_barrier(self._h))

    def comm_destroy(self):
        check(self._h, self._L.sva_comm_destroy(self._h))

    def reduce_ad(self, root=0):
        check(self._h, self._L.sva_frame_reduce_ad(self._h, int(root)))

    def depth_pair_sharded(self, p, ref, others, mask=None, root=0):
        """collective; returns (disp, subpix) on root and None elsewhere"""
        r, rk = abi.image_u8(ref)
        o, ok = abi.image_array(others) if not isinstance(others, tuple) else others
        m = None
        if mask is not None:
            m, mk = abi.image_u8(mask)
        disp = np.empty((p.height, p.width), np.uint16)
        sub = np.empty((p.height, p.width), np.float32)
        check(self._h, self._L.sva_depth_pair_sharded(self._h, C.byref(p), C.byref(r), o, C.byref(m) if m is not None else None, int(root),
                                                       _p(disp, C.c_uint16), _p(sub, C.c_float)))
        self.params = p
        return disp, sub

    def rows_open(self, p, rank, world):
        check(self._h, self._L.sva_rows_open(self._h, C.byref(p), int(rank), int(world)))

    def rows_export(self):
        buf = (C.c_uint8 * abi.SVA_IPC_HANDLE_BYTES)()
        check(self._h, self._L.sva_rows_export(self._h, buf))
        return bytes(buf)

    def rows_connect(self, prev_handle, next_handle):
        mk = lambda h: (C.c_uint8 * abi.SVA_IPC_HANDLE_BYTES).from_buffer_copy(h) if h is not None else None
        check(self._h, self._L.sva_rows_connect(self._h, mk(prev_handle), mk(next_handle)))

    def rows_connect_comm(self):
        check(self._h, self._L.sva_rows_connect_comm(self._h))

    def rows_connect_local(self, prev_ctx, next_ctx):
        check(self._h, self._L.sva_rows_connect_local(self._h, prev_ctx._h if prev_ctx is not None else None, next_ctx._h if next_ctx is not None else None))

    def rows_block(self):
        y0, n = C.c_int32(), C.c_int32()
        check(self._h, self._L.sva_rows_block(self._h, C.byref(y0), C.byref(n)))
        return y0.value, n.value

    def rows_run(self):
        """enqueue this rank's block of the uploaded frame (asynchronous)"""
        check(self._h, self._L.sva_rows_run(self._h))

    def rows_run_part(self, part):
        """part 0: cost volume (+ horizontal paths off the chain's ends); part 1: first sweep; part 2: second sweep + K3 (see sva_rows_run_part)"""
        check(self._h, self._L.sva_rows_run_part(self._h, int(part)))

    def rows_run_phase(self, phase):
        """phase 0: cost volume, horizontal paths, first sweep; phase 1: second sweep + K3 (see sva_rows_run_phase)"""
        check(self._h, self._L.sva_rows_run_phase(self._h, int(phase)))

    def get_stream(self):
        s = C.c_void_p()
        check(self._h, self._L.sva_get_stream(self._h, C.byref(s)))
        return s.value or 0

    def rows_download(self):
        y0, n = self.rows_block()
        disp = np.empty((n, self.params.width), np.uint16)
        sub = np.empty((n, self.params.width), np.float32)
        check(self._h, self._L.sva_rows_download(self._h, _p(disp, C.c_uint16), _p(sub, C.c_float)))
        return disp, sub

    def rows_close(self):
        check(self._h, self._L.sva_rows_close(self._h))

    # ---- one call, host in / host out (the e2e path) ----
    def depth_from_array(self, p, ref, others, mask=None, disp=None, sub=None):
        r, rk = abi.image_u8(ref)
        o, ok = abi.image_array(others) if not isinstance(others, tuple) else others
        m = None
        if mask is not None:
            m, mk = abi.image_u8(mask)
        disp = np.empty((p.height, p.width), np.uint16) if disp is None else disp
        sub = np.empty((p.height, p.width), np.float32) if sub is None else sub
        check(self._h, self._L.sva_depth_from_array(self._h, C.byref(p), C.byref(r), o, C.byref(m) if m is not None else None,
                                                     _p(disp, C.c_uint16), _p(sub, C.c_float)))
        self.params = p
        return disp, sub

    # ---- every reference view of one array frame (getGroups, SURVEY §8 f3) ----
    def depth_groups(self, p, images, groups, grid_cols, masks=None, group_range=None, disp=None, sub=None):
        """The depth maps of the groups [begin, end) = group_range (default: all) of one array frame in one call (sva_depth_groups).
        images: one 2-D uint8 array per camera of a grid of grid_cols columns, or None for a camera no group of the range reads; groups: what
        reference_api.getGroups or oracle.get_groups return; p: template parameters with no pairs; masks: None, or one per group of the range
        (None: no mask).  -> (disp (G, H, W) uint16, subpix (G, H, W) float32), G = end - begin, written into disp / sub when given (C-contiguous;
        pinned memory lets each map's download overlap the groups after it).  ValueError for what the library refuses."""
        groups = _groups.as_groups(groups)
        begin, end = _groups.validate(p, groups, grid_cols, [None if im is None else im.shape for im in images], group_range,
                                      None if masks is None else [None if m is None else m.shape for m in masks])
        for a, dt in ((disp, np.uint16), (sub, np.float32)):
            if a is not None and (a.dtype != dt or a.shape != (end - begin, p.height, p.width) or not a.flags.c_contiguous):
                raise ValueError("output must be a C-contiguous (%d, %d, %d) %s array" % (end - begin, p.height, p.width, np.dtype(dt).name))
        return self.depth_groups_unchecked(p, images, groups, grid_cols, masks, (begin, end), disp, sub)

    def depth_groups_unchecked(self, p, images, groups, grid_cols, masks, group_range, disp=None, sub=None):
        """depth_groups without the Python-side validation: the library's own refusals raise SvaError"""
        begin, end = group_range
        n = max(0, end - begin)
        ims, flat, sizes, m_arr, keep = _groups_args(images, groups, masks, n)
        disp = np.empty((n, p.height, p.width), np.uint16) if disp is None else disp
        sub = np.empty((n, p.height, p.width), np.float32) if sub is None else sub
        d_ptr = (C.c_void_p * max(1, n))(*[disp[i].ctypes.data for i in range(n)])
        s_ptr = (C.c_void_p * max(1, n))(*[sub[i].ctypes.data for i in range(n)])
        check(self._h, self._L.sva_depth_groups(self._h, C.byref(p), int(grid_cols), ims, len(images), flat.ctypes.data, sizes.ctypes.data, len(groups),
                                                 int(begin), int(end), m_arr, d_ptr, s_ptr))
        return disp, sub

    # ---- multi-view depth fusion (DESIGN §3 item 6) ----
    def fuse_maps(self, disp, sub, refs, grid_cols, n_cameras, target, tol_16=16, min_support=2, mask=None):
        """The maps of several reference views of one array frame fused into camera target's view (sva_fuse_maps).  disp: (G, H, W) uint16
        (e.g. depth_groups' output); sub: (G, H, W) float32, or None to fuse the integer maps; refs[g]: view g's reference camera on a grid of
        grid_cols columns and n_cameras cameras; mask: None or (H, W) uint8 of the target (0 = reject).  -> (disp (H, W) uint16,
        subpix (H, W) float32, support (H, W) uint8: how many views agree).  ValueError for what the library refuses."""
        disp = np.asarray(disp)
        if disp.ndim != 3 or disp.dtype != np.uint16:
            raise ValueError("disp must be a (G, H, W) uint16 array")
        if sub is not None and (np.shape(sub) != disp.shape or np.asarray(sub).dtype != np.float32):
            raise ValueError("sub must be None or a float32 array of disp's shape")
        _groups.validate_fuse(disp.shape[0], refs, grid_cols, n_cameras, target, tol_16, min_support, disp.shape[1:],
                              None if mask is None else np.shape(mask))
        return self.fuse_maps_unchecked(list(disp), None if sub is None else list(sub), refs, grid_cols, n_cameras, target,
                                        fuse_params(tol_16, min_support), mask)

    def fuse_maps_unchecked(self, disp, sub, refs, grid_cols, n_cameras, target, f, mask=None):
        """fuse_maps without the Python-side validation: disp / sub are lists of (H, W) maps (None: a null pointer), f an abi.SvaFuseParams;
        the library's own refusals raise SvaError"""
        H, W = next(d.shape for d in disp if d is not None)
        keep = [None if d is None else np.ascontiguousarray(d, dtype=np.uint16) for d in disp]
        d_ptr = (C.c_void_p * max(1, len(keep)))(*[None if d is None else d.ctypes.data for d in keep])
        s_keep = None if sub is None else [None if s is None else np.ascontiguousarray(s, dtype=np.float32) for s in sub]
        s_ptr = None if sub is None else (C.c_void_p * max(1, len(s_keep)))(*[None if s is None else s.ctypes.data for s in s_keep])
        refs = np.array(list(refs) or [0], np.int32)
        m, mk = (None, None) if mask is None else abi.image_u8(np.ascontiguousarray(mask, dtype=np.uint8))
        out = (np.empty((H, W), np.uint16), np.empty((H, W), np.float32), np.empty((H, W), np.uint8))
        check(self._h, self._L.sva_fuse_maps(self._h, W, H, int(grid_cols), int(n_cameras), refs.ctypes.data, len(keep), d_ptr, s_ptr, int(target),
                                              C.byref(f), None if m is None else C.byref(m), *[a.ctypes.data for a in out]))
        return out

    def depth_groups_fused(self, p, images, groups, grid_cols, target, tol_16=16, min_support=2, masks=None, target_mask=None):
        """Every group of one array frame (as depth_groups computes them, masks one per group or None) fused into camera target's view in one
        call (sva_depth_groups_fused): the group maps never leave the device.  The sub-pixel maps are fused iff p.subpixel == 1.  Equal to
        fuse_maps(*depth_groups(...), refs=[g[0][0] for g in groups], ...) bit for bit.  -> (disp, subpix, support) as fuse_maps returns."""
        groups = _groups.as_groups(groups)
        _groups.validate(p, groups, grid_cols, [None if im is None else im.shape for im in images], None,
                         None if masks is None else [None if m is None else m.shape for m in masks])
        _groups.validate_fuse(len(groups), [g[0][0] for g in groups], grid_cols, len(images), target, tol_16, min_support, (p.height, p.width),
                              None if target_mask is None else np.shape(target_mask))
        return self.depth_groups_fused_unchecked(p, images, groups, grid_cols, target, fuse_params(tol_16, min_support), masks, target_mask)

    def depth_groups_fused_unchecked(self, p, images, groups, grid_cols, target, f, masks=None, target_mask=None):
        """depth_groups_fused without the Python-side validation (f: abi.SvaFuseParams): the library's own refusals raise SvaError"""
        ims, flat, sizes, m_arr, keep = _groups_args(images, groups, masks, len(groups))
        m, mk = (None, None) if target_mask is None else abi.image_u8(np.ascontiguousarray(target_mask, dtype=np.uint8))
        out = (np.empty((p.height, p.width), np.uint16), np.empty((p.height, p.width), np.float32), np.empty((p.height, p.width), np.uint8))
        check(self._h, self._L.sva_depth_groups_fused(self._h, C.byref(p), int(grid_cols), ims, len(images), flat.ctypes.data, sizes.ctypes.data,
                                                       len(groups), m_arr, int(target), C.byref(f), None if m is None else C.byref(m),
                                                       *[a.ctypes.data for a in out]))
        return out

    # ---- capture stream: two frames in flight (upload of t+1 | kernels of t | download of t-1) ----
    def stream_submit(self, p, ref, others, mask, disp, sub):
        """enqueue one frame; every numpy buffer must stay alive and untouched until stream_wait(ticket) (pin them for real overlap)"""
        r, rk = abi.image_u8(ref)
        o, ok = abi.image_array(others) if not isinstance(others, tuple) else others
        m = None
        if mask is not None:
            m, mk = abi.image_u8(mask)
        t = C.c_int64()
        check(self._h, self._L.sva_stream_submit(self._h, C.byref(p), C.byref(r), o, C.byref(m) if m is not None else None,
                                                  _p(disp, C.c_uint16), _p(sub, C.c_float) if sub is not None else None, C.byref(t)))
        self.params = p
        return t.value

    def stream_wait(self, ticket):
        check(self._h, self._L.sva_stream_wait(self._h, C.c_int64(ticket)))

    def stream_mark(self):
        check(self._h, self._L.sva_stream_mark(self._h))

    def stream_elapsed(self, ticket):
        ms = C.c_float()
        check(self._h, self._L.sva_stream_elapsed(self._h, C.c_int64(ticket), C.byref(ms)))
        return ms.value


class RowsStream:
    """A stream of frames through the peer-direct row-block pipeline in the order skewed by chain position, one call per frame and rank
    (sva_rows_stream_*, DESIGN.md §7).  ctxs: this rank's world + 1 DepthContexts, all on one stream, each through rows_open(p, rank, world)
    (dist.rows_stream_connect opens and connects them; or connect them after creating the stream with connect_comm).  The contexts are
    borrowed: close the stream before them.

    submit() uploads on a copy stream and returns a ticket; the block's rows (rows_block() of the contexts) reach disp_out / sub_out in
    wait(ticket) or when the ticket's slot is reused world + 2 frames later, whichever comes first.  Until then the input images and the output
    arrays must stay untouched (this object keeps them alive); pinned inputs (torch pin_memory tensors viewed as numpy) let the upload overlap
    the marches.  flush() enqueues the drain: afterwards every submitted frame completes."""

    def __init__(self, ctxs, p):
        self._L = lib()
        self._h = None
        self._ctxs = list(ctxs)  # the stream borrows them: keep them alive as long as it exists
        self._err = ctxs[0]._h
        arr = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
        h = C.c_void_p()
        check(self._err, self._L.sva_rows_stream_create(arr, len(ctxs), C.byref(p), C.byref(h)))
        self._h = h
        self.params = p
        self.slots = len(ctxs) + 1  # world + 2
        self.rows = ctxs[0].rows_block()[1]
        self._keep = {}

    def connect_comm(self):
        """collective: connect all world + 1 links over the communicator of ctxs[0] (comm_init)"""
        check(self._err, self._L.sva_rows_stream_connect_comm(self._h))

    def submit(self, ref, others, mask, disp_out, sub_out=None):
        """enqueue one iteration of the skewed order for a new frame -> ticket.  disp_out: (rows, width) uint16, sub_out: (rows, width)
        float32 or None"""
        p = self.params
        for a, dt in ((disp_out, np.uint16), (sub_out, np.float32)):
            if a is not None and (a.dtype != dt or a.shape != (self.rows, p.width) or not a.flags.c_contiguous):
                raise ValueError("output must be a C-contiguous (%d, %d) %s array" % (self.rows, p.width, np.dtype(dt).name))
        r, rk = abi.image_u8(ref)
        o, ok = abi.image_array(others) if not isinstance(others, tuple) else others
        m = mk = None
        if mask is not None:
            m, mk = abi.image_u8(mask)
        t = C.c_int64()
        check(self._err, self._L.sva_rows_stream_submit(self._h, C.byref(r), o, C.byref(m) if m is not None else None, _p(disp_out, C.c_uint16),
                                                         _p(sub_out, C.c_float) if sub_out is not None else None, C.byref(t)))
        self._keep[t.value] = (rk, ok, mk, disp_out, sub_out)
        for old in [k for k in self._keep if k <= t.value - self.slots]:  # retired when their slot was reused
            del self._keep[old]
        return t.value

    def flush(self):
        check(self._err, self._L.sva_rows_stream_flush(self._h))

    def wait(self, ticket):
        """blocks until the ticket's rows are in its output arrays; SvaError with code SVA_ERR_COMM if a hand-off timed out"""
        try:
            check(self._err, self._L.sva_rows_stream_wait(self._h, C.c_int64(ticket)))
        except SvaError as e:
            if e.code == abi.SVA_ERR_COMM:
                self._keep.pop(ticket, None)
            raise
        self._keep.pop(ticket, None)

    def close(self):
        if self._h:
            self._L.sva_rows_stream_destroy(self._h)
            self._h = None
            self._keep.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
