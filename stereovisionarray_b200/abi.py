"""ctypes mirror of include/sva_c_api.h (structs, enums, status codes).  No compute here."""
import ctypes as C

import numpy as np

SVA_MAX_PAIRS = 32
SVA_COST_CAP_MAX = 4095
SVA_COST_INVALID_U32 = 0xFFFFFFFF
SVA_DISP_INVALID = 0xFFFF
SVA_SUBPIX_INVALID = -1.0

SVA_OK = 0
SVA_ERR_BAD_ARG = -1
SVA_ERR_ROI = -2
SVA_ERR_CUDA = -3
SVA_ERR_NO_DEVICE = -4
SVA_ERR_STATE = -5
SVA_ERR_NOMEM = -6
SVA_ERR_COMM = -7
SVA_COMM_ID_BYTES = 128
SVA_IPC_HANDLE_BYTES = 64

# enum pairType — reference include/functions.h:8-19
ORTHOGONAL, DIAGONAL, TO_CENTER, LINE_HORIZONTAL, LINE_VERTICAL, CROSS, JUMP_CROSS, TO_CENTER_SMALL, MID_LEFT, MID_TOP = range(10)

STAGE_AD, STAGE_BOX, STAGE_SGM, STAGE_ALL = 1, 2, 3, 100
COST_SAD, COST_CENSUS = 0, 1  # sva_cost_mode (params.reserved[0])


class SvaCamera(C.Structure):
    """class Camera — reference include/Camera.h:6-21 (pos3D, f, pixel_size)."""
    _fields_ = [("pos", C.c_double * 3), ("f", C.c_double), ("pixel_size", C.c_double)]


class SvaImageU8(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_int32), ("cols", C.c_int32), ("step", C.c_size_t)]


class SvaParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("num_disp", C.c_int32), ("min_disp", C.c_int32),
        ("win_half", C.c_int32), ("n_pairs", C.c_int32),
        ("pair_gx", C.c_int32 * SVA_MAX_PAIRS), ("pair_gy", C.c_int32 * SVA_MAX_PAIRS),
        ("cost_shift", C.c_int32), ("cost_cap", C.c_int32), ("p1", C.c_int32), ("p2", C.c_int32),
        ("n_paths", C.c_int32), ("lr_gx", C.c_int32), ("lr_max_diff", C.c_int32), ("subpixel", C.c_int32),
        ("reserved", C.c_int32 * 8),
    ]


class SvaFuseParams(C.Structure):
    """sva_fuse_params: candidates within tol_16 / 16 px agree; min_support views must agree (DESIGN §3 item 6)"""
    _fields_ = [("tol_16", C.c_int32), ("min_support", C.c_int32), ("reserved", C.c_int32 * 6)]


def make_params(width, height, num_disp, pairs, win_half=20, min_disp=0, cost_shift=None, cost_cap=SVA_COST_CAP_MAX,
                p1=None, p2=None, n_paths=8, lr_gx=0, lr_max_diff=1, subpixel=1, cost_mode=COST_SAD):
    """pairs: list of (gx, gy) grid offsets of the other cameras.  Defaults follow SURVEY §8(d):
    P1 = 8*Np, P2 = 32*Np in PACK_U16 units; shift = smallest s with (4k^2 * 255 * Np) >> s <= cap (census: 62 instead of 255)."""
    p = SvaParams()
    p.width, p.height, p.num_disp, p.min_disp, p.win_half = width, height, num_disp, min_disp, win_half
    p.n_pairs = len(pairs)
    for i, (gx, gy) in enumerate(pairs):
        p.pair_gx[i], p.pair_gy[i] = gx, gy
    if cost_shift is None:
        full = 4 * win_half * win_half * (62 if cost_mode == COST_CENSUS else 255) * len(pairs)
        cost_shift = 0
        while (full >> cost_shift) > cost_cap:
            cost_shift += 1
    p.cost_shift, p.cost_cap = cost_shift, cost_cap
    p.p1 = 8 * len(pairs) if p1 is None else p1
    p.p2 = 32 * len(pairs) if p2 is None else p2
    p.n_paths, p.lr_gx, p.lr_max_diff, p.subpixel = n_paths, lr_gx, lr_max_diff, subpixel
    p.reserved[0] = cost_mode
    return p


def image_u8(a):
    """numpy 2-D uint8 (C-order along x) -> (SvaImageU8, keepalive)."""
    if a.dtype != np.uint8 or a.ndim != 2 or a.strides[1] != 1:
        raise ValueError("expected a 2-D uint8 array with unit x stride")
    return SvaImageU8(a.ctypes.data, a.shape[0], a.shape[1], a.strides[0]), a


def image_array(arrs):
    """list of 2-D uint8 arrays -> (ctypes array of SvaImageU8, keepalive list)."""
    arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in arrs]
    out = (SvaImageU8 * len(arrs))()
    for i, a in enumerate(arrs):
        out[i] = SvaImageU8(a.ctypes.data, a.shape[0], a.shape[1], a.strides[0])
    return out, arrs


def camera(pos, f, pixel_size):
    c = SvaCamera()
    c.pos[0], c.pos[1], c.pos[2] = float(pos[0]), float(pos[1]), float(pos[2])
    c.f, c.pixel_size = float(f), float(pixel_size)
    return c


def camera_array(cams):
    out = (SvaCamera * len(cams))()
    for i, c in enumerate(cams):
        out[i] = c
    return out
