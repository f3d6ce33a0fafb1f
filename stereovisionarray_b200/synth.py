"""Deterministic synthetic textured scenes with known ground-truth disparity (SURVEY §8d).

The same bytes feed the CPU oracle and the GPU path.  numpy only (no cv2) so it runs anywhere.
  texture   : uniform u8 noise, separable Gaussian blur (sigma 1.5), min-max stretched to 0..255
  disparity : background plane at dmin + D/4, four rectangles at dmin + {D/2, 5D/8, 3D/4, 7D/8-2}, one
              horizontally slanted strip (integer-rounded); optional ellipsoidal "face" bump + elliptical mask
  views     : camera at grid offset (gx, gy) sees R(y, x) at (y - gy*delta, x - gx*delta); rendered far-to-near
              (z-buffer by delta); disocclusions filled from an independent noise texture (seed + 1 + k)
  seed      : 1000 * config_index + frame_index
"""
import numpy as np


def _gauss_blur(a, sigma=1.5):
    r = int(3 * sigma + 0.5)
    x = np.arange(-r, r + 1, dtype=np.float64)
    k = np.exp(-0.5 * (x / sigma) ** 2)
    k /= k.sum()
    a = np.pad(a.astype(np.float64), r, mode="reflect")
    a = sum(k[i] * a[:, i:i + a.shape[1] - 2 * r] for i in range(2 * r + 1))
    a = sum(k[i] * a[i:i + a.shape[0] - 2 * r, :] for i in range(2 * r + 1))
    return a


def texture(h, w, seed):
    rng = np.random.default_rng(seed)
    t = _gauss_blur(rng.integers(0, 256, size=(h, w), dtype=np.uint8))
    t = (t - t.min()) / max(1e-9, t.max() - t.min())
    return np.clip(np.rint(t * 255.0), 0, 255).astype(np.uint8)


def gt_disparity(h, w, num_disp, min_disp=0, face=False, seed=0):
    D = num_disp
    d = np.full((h, w), min_disp + D // 4, dtype=np.int32)
    levels = [D // 2, (5 * D) // 8, (3 * D) // 4, (7 * D) // 8 - 2]
    rects = [(0.08, 0.06, 0.30, 0.32), (0.55, 0.10, 0.36, 0.30), (0.12, 0.55, 0.28, 0.34), (0.60, 0.58, 0.30, 0.30)]
    for lv, (fx, fy, fw, fh) in zip(levels, rects):
        d[int(fy * h):int((fy + fh) * h), int(fx * w):int((fx + fw) * w)] = min_disp + max(0, lv)
    # slanted strip across the middle: gradient 0.08 px/px, rounded to integers
    y0, y1 = int(0.44 * h), int(0.52 * h)
    ramp = np.rint(min_disp + D // 4 + 0.08 * np.arange(w)).astype(np.int32)
    d[y0:y1, :] = np.minimum(ramp, min_disp + D - 2)[None, :]
    if face:
        yy, xx = np.mgrid[0:h, 0:w]
        e = ((xx - w / 2) / (0.30 * w)) ** 2 + ((yy - h / 2) / (0.38 * h)) ** 2
        bump = np.rint(min_disp + D // 3 + (D // 3) * np.sqrt(np.clip(1 - e, 0, 1))).astype(np.int32)
        d = np.where(e < 1, np.minimum(bump, min_disp + D - 2), d)
    return np.clip(d, min_disp, min_disp + D - 1).astype(np.int32)


def ellipse_mask(h, w):
    """elliptical u8 mask, the stand-in for getFaceCircle's output (reference src/dlibFaceSelect.cpp:51-62)."""
    yy, xx = np.mgrid[0:h, 0:w]
    e = ((xx - w / 2) / (0.34 * w)) ** 2 + ((yy - h / 2) / (0.42 * h)) ** 2
    return np.where(e < 1, 255, 0).astype(np.uint8)


def render_view(ref, disp, gx, gy, fill, order=None):
    """forward-warp ref into the camera at grid offset (gx, gy); nearer (larger delta) wins; holes <- fill.
    One scatter in ascending-disparity order (numpy keeps the LAST value written to a repeated index), i.e. far first, near overwrites;
    `order` = np.argsort(disp.ravel(), kind="stable"), shared by the views of a scene."""
    h, w = ref.shape
    out = fill.copy()
    if order is None:
        order = np.argsort(disp.ravel(), kind="stable")
    lv = disp.ravel()[order]
    ty = order // w - gy * lv
    tx = order % w - gx * lv
    ok = (ty >= 0) & (ty < h) & (tx >= 0) & (tx < w)
    out[ty[ok], tx[ok]] = ref.ravel()[order[ok]]
    return out


def make_scene(h, w, num_disp, offsets, seed, min_disp=0, face=False):
    """returns dict(ref, others[list], gt[int32 disparity], mask[u8 or None])."""
    ref = texture(h, w, seed)
    gt = gt_disparity(h, w, num_disp, min_disp, face=face, seed=seed)
    order = np.argsort(gt.ravel(), kind="stable")
    others = [render_view(ref, gt, gx, gy, texture(h, w, seed + 1 + k), order) for k, (gx, gy) in enumerate(offsets)]
    return {"ref": ref, "others": others, "gt": gt, "mask": ellipse_mask(h, w) if face else None}


# ---- literal-mode scenes in the reference driver's own geometry (src/CameraStereoVision.cpp:24-39) ----
REF_F = 0.05
REF_SENSOR = 0.036
REF_PITCH = 0.05
REF_Z = -0.75


def reference_cameras(width):
    """the 5x5 grid of src/CameraStereoVision.cpp:33-39 as (pos, f, pixel_size) tuples; index = 5*row + col."""
    ps = REF_SENSOR / width
    return [((-0.1 + x * REF_PITCH, -0.1 + y * REF_PITCH, REF_Z), REF_F, ps) for y in range(5) for x in range(5)]


def make_literal_scene(h, w, seed, pair=(12, 11)):
    """A centre image (camera 12) and the `pair[1]` view of a piecewise-planar scene whose disparities fall in the range the
    driver searches (ray length 0.5..1.0 -> roughly 0.07W .. 0.14W px per baseline).  Returns 25 images (unused views = noise)."""
    lo, hi = int(0.075 * w), int(0.135 * w)
    ref = texture(h, w, seed)
    gt = gt_disparity(h, w, hi - lo, lo, seed=seed)
    r0, c0 = divmod(pair[0], 5)
    r1, c1 = divmod(pair[1], 5)
    gx, gy = c1 - c0, r1 - r0
    other = render_view(ref, gt, gx, gy, texture(h, w, seed + 1))
    images = [texture(h, w, seed + 100 + i) for i in range(25)]
    images[pair[0]], images[pair[1]] = ref, other
    return {"images": images, "gt": gt, "mask": ellipse_mask(h, w)}


def make_depth_scene(h, w, seed=0):
    """f64 depth map in the reference's metric range (the scene sits ~0.75 in front of the array, CameraStereoVision.cpp:37): smooth
    background + two closer blobs, with holes (0 = no depth, skipped by shiftPerspective2's `depth < 0.5` and DepthMapToPoints3D's `> 0.1`)"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    d = 0.95 + 0.05 * np.sin(xx / w * 3.0) + 0.03 * np.cos(yy / h * 2.0)
    for cx, cy, r, dz in ((0.35, 0.4, 0.18, 0.22), (0.7, 0.6, 0.12, 0.3)):
        m = ((xx / w - cx) ** 2 + (yy / h - cy) ** 2) < r * r
        d[m] -= dz
    d[rng.random((h, w)) < 0.03] = 0.0
    d[:2, :] = 0.3  # below shiftPerspective2's 0.5 threshold but above DepthMapToPoints3D's 0.1
    return d


# ---- one scene seen by every camera of an array (multi-reference groups, sva_depth_groups) ----
def make_array_scene(h, w, grid_rows, grid_cols, num_disp, seed, min_disp=0):
    """Fronto-parallel textured layers at integer disparities, rendered consistently into every camera of a grid_rows x grid_cols array.
    Pixel (x, y) of camera (c, r) (index r * grid_cols + c) shows layer l's texture at (x + c * delta_l, y + r * delta_l) of the layer's
    reference plane; of the layers whose support covers that point the nearest (largest delta) wins.  So a texture point at (u, v) appears in
    camera (c, r) at (u - c * delta, v - r * delta): seen from camera i, the match of (x, y) in camera j is (x - gx * delta, y - gy * delta)
    with (gx, gy) = (col j - col i, row j - row i), the convention of configs.grid_offsets.
    Layers: a background covering everything at min_disp + D/4 and three rectangles at min_disp + {D/2, 5D/8 + 1, 7D/8 - 2}, placed in the
    centre camera's image.  -> dict(images[list of u8 (h, w)], gt[list of int32 (h, w)]: each camera's disparity, layers[list of delta])."""
    D = num_disp
    deltas = [min_disp + D // 4, min_disp + D // 2, min_disp + (5 * D) // 8 + 1, min_disp + (7 * D) // 8 - 2]
    cm, rm = (grid_cols - 1) / 2.0, (grid_rows - 1) / 2.0
    # supports in reference-plane coordinates (u0, v0, u1, v1): rectangles of the centre camera's image, shifted by its delta
    rects = [None]
    for (fx, fy, fw, fh), dl in zip([(0.10, 0.12, 0.34, 0.36), (0.52, 0.18, 0.32, 0.30), (0.30, 0.56, 0.30, 0.30)], deltas[1:]):
        rects.append((fx * w + cm * dl, fy * h + rm * dl, (fx + fw) * w + cm * dl, (fy + fh) * h + rm * dl))
    texs = []
    for i, dl in enumerate(deltas):
        texs.append(texture(h + (grid_rows - 1) * dl + 1, w + (grid_cols - 1) * dl + 1, seed * 16 + i))
    yy, xx = np.mgrid[0:h, 0:w]
    images, gts = [], []
    for r in range(grid_rows):
        for c in range(grid_cols):
            img = np.zeros((h, w), np.uint8)
            gt = np.zeros((h, w), np.int32)
            for tex, dl, rc in zip(texs, deltas, rects):  # ascending delta: nearer layers overwrite
                u, v = xx + c * dl, yy + r * dl
                inside = np.ones((h, w), bool) if rc is None else (u >= rc[0]) & (u < rc[2]) & (v >= rc[1]) & (v < rc[3])
                img[inside] = tex[v[inside], u[inside]]
                gt[inside] = dl
            images.append(img)
            gts.append(gt)
    return {"images": images, "gt": gts, "layers": deltas}
