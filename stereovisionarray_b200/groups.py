"""Host logic of the multi-reference calls sva_depth_groups (getGroups, SURVEY §8 f3) and of the depth fusion (sva_fuse_maps,
sva_depth_groups_fused): grid offsets of a group's pairs, the flattened layout the C ABI takes, and the refusal rules, checked here before the
library is called so that a caller gets a ValueError naming the problem.  Pure Python: no library, no GPU."""
from . import abi


def as_groups(groups):
    """reference_api.getGroups / oracle.get_groups output (lists of (ref, other) pairs or (n, 2) arrays) -> list of lists of (int, int)"""
    return [[(int(a), int(b)) for a, b in g] for g in groups]


def group_offsets(group, grid_cols):
    """(gx, gy) of each pair of a group on a grid of grid_cols columns: gx = col(other) - col(ref), gy = row(other) - row(ref)
    (configs.grid_offsets' convention)"""
    return [(o % grid_cols - r % grid_cols, o // grid_cols - r // grid_cols) for r, o in group]


def group_params(p, group, grid_cols):
    """the template p with the group's pairs: what sva_depth_groups computes that group with"""
    q = abi.SvaParams.from_buffer_copy(p)
    q.n_pairs = len(group)
    for j, (gx, gy) in enumerate(group_offsets(group, grid_cols)):
        q.pair_gx[j], q.pair_gy[j] = gx, gy
    return q


def cameras_of(groups):
    """cameras the groups read, in order of first use"""
    seen = []
    for g in groups:
        for pr in g:
            for cam in pr:
                if cam not in seen:
                    seen.append(cam)
    return seen


def _params_ok(q):
    """the checks of sva_api.cu's check_params on a derived parameter set -> reason or None"""
    if q.width < 8 or q.height < 8:
        return "image smaller than 8x8"
    if q.num_disp < 8 or q.num_disp > 256 or q.num_disp % 8:
        return "num_disp must be a multiple of 8 in 8..256"
    if q.min_disp < 0 or q.min_disp > 4096:
        return "min_disp must be in 0..4096"
    if q.win_half < 1 or q.win_half > 56:
        return "win_half must be in 1..56"
    if q.n_pairs < 1 or q.n_pairs > abi.SVA_MAX_PAIRS:
        return "n_pairs must be in 1..32"
    if q.cost_cap < 1 or q.cost_cap > abi.SVA_COST_CAP_MAX or q.cost_shift < 0 or q.cost_shift > 31:
        return "bad cost_cap / cost_shift"
    if q.p1 < 0 or q.p2 < q.p1 or q.p2 > 4095:
        return "need 0 <= p1 <= p2 <= 4095"
    if q.n_paths not in (0, 4, 8):
        return "n_paths must be 0, 4 or 8"
    if q.lr_gx not in (-1, 0, 1):
        return "lr_gx must be -1, 0 or +1"
    if q.reserved[0] not in (abi.COST_SAD, abi.COST_CENSUS) or any(q.reserved[i] for i in range(1, 8)):
        return "unknown cost mode or non-zero reserved fields"
    if 4.0 * q.win_half * q.win_half * 255.0 * q.n_pairs > 4.0e9:
        return "window sum overflows u32"
    if float(q.width) * q.height * q.num_disp >= 2.0 ** 32:
        return "frame too large"
    return None


def validate(p, groups, grid_cols, shapes, group_range=None, mask_shapes=None):
    """Raise ValueError where sva_depth_groups would return SVA_ERR_BAD_ARG.  shapes[i] = (rows, cols) of camera i, or None for a camera
    without data; mask_shapes: None, or one entry per group of the range ((rows, cols), or None for no mask).  -> (begin, end)"""
    n_images = len(shapes)
    begin, end = (0, len(groups)) if group_range is None else (int(group_range[0]), int(group_range[1]))
    if not (0 <= begin <= end <= len(groups)):
        raise ValueError("group range %r outside [0, %d]" % ((begin, end), len(groups)))
    if grid_cols < 1 or n_images < 1 or n_images % grid_cols:
        raise ValueError("%d images are not a positive multiple of grid_cols = %d" % (n_images, grid_cols))
    if p.n_pairs != 0 or any(p.pair_gx[i] or p.pair_gy[i] for i in range(abi.SVA_MAX_PAIRS)):
        raise ValueError("the template's n_pairs, pair_gx and pair_gy must be zero: each group's come from its pairs")
    for g, grp in enumerate(groups):
        for r, o in grp:
            if not (0 <= r < n_images and 0 <= o < n_images):
                raise ValueError("group %d names a camera outside [0, %d)" % (g, n_images))
            if r != grp[0][0]:
                raise ValueError("the pairs of group %d do not share one reference" % g)
            if o == r:
                raise ValueError("group %d pairs camera %d with itself" % (g, r))
        if len(grp) > abi.SVA_MAX_PAIRS:
            raise ValueError("group %d has more than 32 pairs" % g)
        why = _params_ok(group_params(p, grp, grid_cols))
        if why:
            raise ValueError("group %d: %s" % (g, why))
    for g in range(begin, end):
        for cam in cameras_of([groups[g]]):
            if shapes[cam] is None:
                raise ValueError("camera %d is read by group %d but has no data" % (cam, g))
            if tuple(shapes[cam]) != (p.height, p.width):
                raise ValueError("camera %d is %r, not %dx%d" % (cam, tuple(shapes[cam]), p.height, p.width))
    if mask_shapes is not None:
        if len(mask_shapes) != end - begin:
            raise ValueError("masks: one per group of the range")
        for i, m in enumerate(mask_shapes):
            if m is not None and tuple(m) != (p.height, p.width):
                raise ValueError("mask of group %d is %r, not %dx%d" % (begin + i, tuple(m), p.height, p.width))
    return begin, end


def validate_fuse(n_views, refs, grid_cols, n_cameras, target, tol_16, min_support, shape, mask_shape=None):
    """Raise ValueError where sva_fuse_maps (and the fusion part of sva_depth_groups_fused) would return SVA_ERR_BAD_ARG.  shape: (rows, cols)
    of the maps; mask_shape: None or the target mask's (rows, cols)."""
    if not 1 <= n_views <= 32:
        raise ValueError("%d views: fusion takes 1..32" % n_views)
    if len(refs) != n_views:
        raise ValueError("one reference camera per view")
    if grid_cols < 1 or n_cameras < 1 or n_cameras % grid_cols:
        raise ValueError("%d cameras are not a positive multiple of grid_cols = %d" % (n_cameras, grid_cols))
    for g, r in enumerate(refs):
        if not 0 <= r < n_cameras:
            raise ValueError("reference %d of view %d outside [0, %d)" % (r, g, n_cameras))
    if not 0 <= target < n_cameras:
        raise ValueError("target %d outside [0, %d)" % (target, n_cameras))
    if not 0 <= tol_16 <= 4095:
        raise ValueError("tol_16 must be in 0..4095")
    if not 1 <= min_support <= n_views:
        raise ValueError("min_support must be in 1..%d" % n_views)
    if min(shape) < 1:
        raise ValueError("empty maps")
    if mask_shape is not None and tuple(mask_shape) != tuple(shape):
        raise ValueError("target mask is %r, not %r" % (tuple(mask_shape), tuple(shape)))
