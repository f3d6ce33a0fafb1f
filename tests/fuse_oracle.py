"""TEST INFRASTRUCTURE ONLY — ctypes wrapper over tests/fuse_oracle.c, the CPU restatement of the multi-view depth fusion spec
(DESIGN §3 item 6).  The library is compiled on first use into the temporary directory, under a name derived from its sources, so the
repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "fuse_oracle.c"), os.path.join(HERE, "..", "include", "sva_c_api.h")]
_lib = None


def _load():
    global _lib
    if _lib is None:
        digest = hashlib.sha256(b"".join(open(s, "rb").read() for s in SOURCES)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "sva_fuse_oracle_%d_%s.so" % (os.getuid(), digest))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            r = subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", SOURCES[0], "-o", tmp, "-lm"],
                               capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("building the fusion oracle failed:\n" + r.stdout + r.stderr)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def fuse_views(disp, sub, refs, grid_cols, target, tol_16=16, min_support=2, mask=None):
    """disp (G, H, W) uint16 (and sub (G, H, W) float32, or None) of the views with reference cameras refs, fused into camera target's view
    -> (disp (H, W) uint16, sub (H, W) float32, support (H, W) uint8)"""
    d = np.ascontiguousarray(disp, dtype=np.uint16)
    G, H, W = d.shape
    s = None if sub is None else np.ascontiguousarray(sub, dtype=np.float32)
    dp = (C.c_void_p * G)(*[d[g].ctypes.data for g in range(G)])
    sp = None if s is None else (C.c_void_p * G)(*[s[g].ctypes.data for g in range(G)])
    m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
    refs = np.ascontiguousarray(refs, dtype=np.int32)
    out_d = np.zeros((H, W), np.uint16)
    out_s = np.zeros((H, W), np.float32)
    out_n = np.zeros((H, W), np.uint8)
    rc = _load().orc_fuse_views(W, H, grid_cols, _ptr(refs, C.c_int32), G, dp, sp, target, tol_16, min_support,
                                None if m is None else _ptr(m, C.c_uint8), _ptr(out_d, C.c_uint16), _ptr(out_s, C.c_float), _ptr(out_n, C.c_uint8))
    assert rc == 0, rc
    return out_d, out_s, out_n
