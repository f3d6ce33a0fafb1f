"""Host-side driver of the volume-mode depth pipeline over the C ABI (one DepthContext per GPU).

Stages (DESIGN.md §4): K1a AD volume -> K1b box/pack -> K2 SGM (four launches for 8 paths: -> storing S, <-, the down-sweeping and the up-sweeping group) -> K3 (WTA / LR / sub-pixel).
All compute happens in libsva_b200.so on the GPU; this module only marshals numpy buffers."""
import ctypes as C

import numpy as np

from . import abi
from ._lib import SvaError, check, lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


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
