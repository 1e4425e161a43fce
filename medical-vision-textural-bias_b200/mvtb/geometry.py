"""Host geometry of the resampling at the front of the reference's pipelines (127_...FLAIR.py:120-129, utils.py:186-198):

    Spacingd(["image", "label"], pixdim=(1.5, 1.5, 2.0), mode=("bilinear", "nearest")) -> Orientationd(..., axcodes="RAS")

Restated from MONAI 0.5 (monai/data/utils.py: zoom_affine, compute_shape_offset, to_affine_nd; monai/networks/utils.py:
normalize_transform, to_norm_affine; monai/networks/layers/spatial_transforms.py: AffineTransform's reversed indexing;
monai/transforms/spatial/array.py: Spacing, Orientation) and nibabel (nibabel/orientations.py: io_orientation,
axcodes2ornt, ornt_transform, apply_orientation, inv_ornt_aff) with numpy and torch only.  Everything here is small
and runs once per geometry; the voxels are moved by mvtb_resample_f32 (csrc/resample.cuh) through mvtb/spatial.py.

`plan()` composes the two transforms into one description of the gather: the source -> grid transform of Spacingd,
Orientationd's signed axis permutation of the grid, the resulting shape and affine.  `index_map()` folds an optional
window and flip on top, and `axis_taps()` gives the per-axis interpolation tables of an axis-aligned transform,
computed with torch's own affine_grid so that nearest-neighbour labels pick the voxel torch picks, ties included."""
from typing import NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

LABELS = (("L", "R"), ("P", "A"), ("I", "S"))


# ----------------------------------------------------------------------------- MONAI 0.5: monai/data/utils.py

def to_affine_nd(r, affine) -> np.ndarray:
    """`affine` embedded in an (r+1)x(r+1) identity (r an int), or copied into the shape of the array `r`"""
    affine_np = np.array(affine, dtype=np.float64)
    if affine_np.ndim != 2:
        raise ValueError(f"affine must have 2 dimensions, got {affine_np.ndim}")
    new_affine = np.array(r, dtype=np.float64, copy=True)
    if new_affine.ndim == 0:
        sr = int(new_affine)
        if not np.isfinite(new_affine) or sr < 0:
            raise ValueError(f"r must be positive, got {sr}")
        new_affine = np.eye(sr + 1, dtype=np.float64)
    d = max(min(len(new_affine) - 1, len(affine_np) - 1), 1)
    new_affine[:d, :d] = affine_np[:d, :d]
    if d > 1:
        new_affine[:d, -1] = affine_np[:d, -1]
    return new_affine


def zoom_affine(affine, scale, diagonal: bool = True) -> np.ndarray:
    """affine with voxel size `scale`: diagonal, or keeping the rotation of `affine` (Cholesky of its RZS)"""
    affine = np.array(affine, dtype=float, copy=True)
    if len(affine) != len(affine[0]):
        raise ValueError(f"affine must be n x n, got {len(affine)} x {len(affine[0])}")
    scale_np = np.array(scale, dtype=float, copy=True)
    d = len(affine) - 1
    if len(scale_np) < d:                                   # missing entries: the affine's own voxel size
        norm = np.sqrt(np.sum(np.square(affine), 0))[:-1]
        scale_np = np.append(scale_np, norm[len(scale_np):])
    scale_np = scale_np[:d]
    scale_np[scale_np == 0] = 1.0
    if diagonal:
        return np.diag(np.append(scale_np, [1.0]))
    rzs = affine[:-1, :-1]
    zs = np.linalg.cholesky(rzs.T @ rzs).T
    rotation = rzs @ np.linalg.inv(zs)
    s = np.sign(np.diag(zs)) * np.abs(scale_np)
    new_affine = np.eye(len(affine))
    new_affine[:-1, :-1] = rotation @ np.diag(s)
    return new_affine


def compute_shape_offset(spatial_shape, in_affine, out_affine) -> Tuple[np.ndarray, np.ndarray]:
    """output grid shape covering the input's corner voxels, and its origin (world coordinates)"""
    shape = np.array(spatial_shape, copy=True, dtype=float)
    sr = len(shape)
    in_affine = to_affine_nd(sr, in_affine)
    out_affine = to_affine_nd(sr, out_affine)
    in_coords = [(0.0, dim - 1.0) for dim in shape]
    corners = np.asarray(np.meshgrid(*in_coords, indexing="ij")).reshape((len(shape), -1))
    corners = np.concatenate((corners, np.ones_like(corners[:1])))
    corners = in_affine @ corners
    corners_out = np.linalg.inv(out_affine) @ corners
    corners_out = corners_out[:-1] / corners_out[-1]
    out_shape = np.round(np.ptp(corners_out, axis=1) + 1.0)
    if np.allclose(io_orientation(in_affine), io_orientation(out_affine)):
        offset = in_affine @ ([0] * sr + [1])                # same orientation: the input's origin
        offset = offset[:-1] / offset[-1]
    else:
        corners = corners[:-1] / corners[-1]                 # else the lowest corner
        offset = np.min(corners, 1)
    return out_shape.astype(int), offset


# ----------------------------------------------------------------------------- nibabel/orientations.py

def io_orientation(affine, tol=None) -> np.ndarray:
    """(p, 2) orientation of the voxel axes in world space: row = (world axis, +-1), NaN for a dropped axis"""
    affine = np.asarray(affine)
    q, p = affine.shape[0] - 1, affine.shape[1] - 1
    RZS = affine[:q, :p]
    zooms = np.sqrt(np.sum(RZS * RZS, axis=0))
    zooms[zooms == 0] = 1
    RS = RZS / zooms
    P, S, Qs = np.linalg.svd(RS, full_matrices=False)        # polar decomposition: the closest shear-free matrix
    if tol is None:
        tol = S.max() * max(RS.shape) * np.finfo(np.float64).eps
    keep = S > tol
    R = np.dot(P[:, keep], Qs[keep])
    ornt = np.ones((p, 2), dtype=np.int8) * np.nan
    for in_ax in range(p):
        col = R[:, in_ax]
        if not np.allclose(col, 0):
            out_ax = np.argmax(np.abs(col))
            ornt[in_ax, 0] = out_ax
            ornt[in_ax, 1] = -1 if col[out_ax] < 0 else 1
            R[out_ax, :] = 0                                 # ties: each world axis is taken once
    return ornt


def axcodes2ornt(axcodes, labels=None) -> np.ndarray:
    labels = list(zip("LPI", "RAS")) if labels is None else labels
    allowed_labels = sum([list(L) for L in labels], []) + [None]
    if len(allowed_labels) != len(set(allowed_labels)):
        raise ValueError(f"Duplicate labels in {allowed_labels}")
    if not set(axcodes).issubset(allowed_labels):
        raise ValueError(f"Not all axis codes {list(axcodes)} in label set {allowed_labels}")
    ornt = np.ones((len(axcodes), 2), dtype=np.int8) * np.nan
    for code_idx, code in enumerate(axcodes):
        for label_idx, codes in enumerate(labels):
            if code is None:
                continue
            if code in codes:
                ornt[code_idx, :] = [label_idx, -1 if code == codes[0] else 1]
                break
    return ornt


def ornt_transform(start_ornt, end_ornt) -> np.ndarray:
    """the orientation that takes an array in start_ornt to end_ornt"""
    start_ornt = np.asarray(start_ornt)
    end_ornt = np.asarray(end_ornt)
    if start_ornt.shape != end_ornt.shape:
        raise ValueError("The orientations must have the same shape")
    if start_ornt.shape[1] != 2:
        raise ValueError(f"Invalid shape for an orientation: {start_ornt.shape}")
    result = np.empty_like(start_ornt)
    for end_in_idx, (end_out_idx, end_flip) in enumerate(end_ornt):
        for start_in_idx, (start_out_idx, start_flip) in enumerate(start_ornt):
            if end_out_idx == start_out_idx:
                result[start_in_idx, :] = [end_in_idx, 1 if start_flip == end_flip else -1]
                break
        else:
            raise ValueError(f"Unable to find out axis {end_out_idx} in start_ornt")
    return result


def apply_orientation(arr, ornt) -> np.ndarray:
    """flip every axis with ornt[:, 1] == -1, then move axis i to ornt[i, 0]"""
    t_arr = np.asarray(arr)
    ornt = np.asarray(ornt)
    n = ornt.shape[0]
    if t_arr.ndim < n:
        raise ValueError("Data array has fewer dimensions than orientation")
    if np.any(np.isnan(ornt[:, 0])):
        raise ValueError("Cannot drop coordinates when applying orientation to data")
    for ax, flip in enumerate(ornt[:, 1]):
        if flip == -1:
            t_arr = np.flip(t_arr, axis=ax)
    full_transpose = np.arange(t_arr.ndim)
    full_transpose[:n] = np.argsort(ornt[:, 0])
    return t_arr.transpose(full_transpose)


def inv_ornt_aff(ornt, shape) -> np.ndarray:
    """the voxel affine that undoes apply_orientation(ornt) on an array of `shape`"""
    ornt = np.asarray(ornt)
    if np.any(np.isnan(ornt)):
        raise ValueError("We cannot invert orientation transform")
    p = ornt.shape[0]
    shape = np.array(shape)[:p]
    axis_transpose = [int(v) for v in ornt[:, 0]]
    undo_reorder = np.eye(p + 1)[axis_transpose + [p], :]
    undo_flip = np.diag(list(ornt[:, 1]) + [1.0])
    center_trans = -(shape - 1) / 2.0
    undo_flip[:p, p] = (ornt[:, 1] * center_trans) - center_trans
    return np.dot(undo_flip, undo_reorder)


# ----------------------------------------------------------------------------- MONAI 0.5: monai/networks/utils.py

def normalize_transform(shape, align_corners: bool = False) -> torch.Tensor:
    """(1, r+1, r+1) float64 map from voxel index to grid_sample's [-1, 1] coordinates"""
    norm = torch.tensor(shape, dtype=torch.float64)
    if align_corners:
        norm[norm <= 1.0] = 2.0
        norm = 2.0 / (norm - 1.0)
        norm = torch.diag(torch.cat((norm, torch.ones((1,), dtype=torch.float64))))
        norm[:-1, -1] = -1.0
    else:
        norm[norm <= 0.0] = 2.0
        norm = 2.0 / norm
        norm = torch.diag(torch.cat((norm, torch.ones((1,), dtype=torch.float64))))
        norm[:-1, -1] = 1.0 / torch.tensor(shape, dtype=torch.float64) - 1.0
    return norm.unsqueeze(0)


def to_norm_affine(affine: torch.Tensor, src_size, dst_size, align_corners: bool = False) -> torch.Tensor:
    sr = affine.shape[1] - 1
    if affine.ndimension() != 3 or affine.shape[1] != affine.shape[2] or sr != len(src_size) or sr != len(dst_size):
        raise ValueError(f"affine of shape {tuple(affine.shape)} does not fit sizes {src_size} -> {dst_size}")
    src_xform = normalize_transform(src_size, align_corners).to(affine.dtype)
    dst_xform = normalize_transform(dst_size, align_corners).to(affine.dtype)
    return src_xform @ affine @ torch.inverse(dst_xform)


def affine_theta(transform, src_shape, dst_shape) -> torch.Tensor:
    """AffineTransform(normalized=False, reverse_indexing=True, align_corners=False)'s theta: (1, 4, 4) float64, what
    affine_grid receives (its first three rows)"""
    theta = torch.as_tensor(np.ascontiguousarray(transform), dtype=torch.float64)[None].clone()
    theta = to_norm_affine(theta, tuple(src_shape), tuple(dst_shape), align_corners=False)
    rev = torch.as_tensor([2, 1, 0])
    theta[:, :3] = theta[:, rev]
    theta[:, :, :3] = theta[:, :, rev]
    return theta


# ----------------------------------------------------------------------------- Spacing / Orientation composed

class SpacingGeom(NamedTuple):
    transform: np.ndarray     # 4x4: Spacingd's grid index -> source index (what MONAI hands AffineTransform)
    shape: Tuple[int, ...]    # the grid's shape
    affine: np.ndarray        # the new affine
    identity: bool            # MONAI's shortcut: transform within 1e-3 of I -> the data is copied, not resampled


def spacing(affine, spatial_shape: Sequence[int], pixdim, diagonal: bool = False) -> SpacingGeom:
    """Spacing.__call__'s geometry for a 3-D (C, H, W, D) array"""
    sr = 3
    if len(spatial_shape) != sr:
        raise ValueError(f"Spacing here takes 3 spatial axes, got {len(spatial_shape)}")
    affine_ = np.eye(sr + 1, dtype=np.float64) if affine is None else to_affine_nd(sr, affine)
    out_d = np.array(pixdim if isinstance(pixdim, (list, tuple, np.ndarray)) else (pixdim,), dtype=np.float64)[:sr]
    if np.any(out_d <= 0):
        raise ValueError(f"pixdim must be positive, got {out_d}")
    new_affine = zoom_affine(affine_, out_d, diagonal=diagonal)
    output_shape, offset = compute_shape_offset(spatial_shape, affine_, new_affine)
    new_affine[:sr, -1] = offset[:sr]
    transform = to_affine_nd(sr, np.linalg.inv(affine_) @ new_affine)
    identity = bool(np.allclose(transform, np.diag(np.ones(len(transform))), atol=1e-3))
    shape = tuple(int(s) for s in (spatial_shape if identity else output_shape))
    new_affine = to_affine_nd(np.eye(sr + 1) if affine is None else affine, new_affine)
    return SpacingGeom(transform, shape, new_affine, identity)


def orientation(affine, spatial_shape: Sequence[int], axcodes=None, as_closest_canonical: bool = False,
                labels=LABELS) -> Tuple[np.ndarray, Tuple[int, ...], np.ndarray]:
    """Orientation.__call__'s geometry: (spatial ornt (3, 2) ints, new shape, new affine)"""
    sr = len(spatial_shape)
    affine_ = np.eye(sr + 1, dtype=np.float64) if affine is None else to_affine_nd(sr, affine)
    src = io_orientation(affine_)
    if as_closest_canonical:
        spatial_ornt = src
    else:
        if axcodes is None:
            raise ValueError("Incompatible values: axcodes=None and as_closest_canonical=True.")
        dst = axcodes2ornt(axcodes[:sr], labels=labels)
        if len(dst) < sr:
            raise ValueError(f"axcodes must match data_array spatially, got axcodes={len(axcodes)}D data_array={sr}D")
        spatial_ornt = ornt_transform(src, dst)
    if np.any(np.isnan(spatial_ornt)):
        raise ValueError("Cannot drop coordinates when applying orientation to data")
    new_affine = to_affine_nd(np.eye(sr + 1) if affine is None else affine, affine_ @ inv_ornt_aff(spatial_ornt, spatial_shape))
    ornt = spatial_ornt.astype(int)
    shape = [0] * sr
    for i in range(sr):
        shape[ornt[i, 0]] = int(spatial_shape[i])
    return ornt, tuple(shape), new_affine


class Plan(NamedTuple):
    in_shape: Tuple[int, ...]   # source (H, W, D)
    spacing: SpacingGeom        # source -> grid (identity when there is no Spacingd)
    ornt: np.ndarray            # grid axis i -> output axis ornt[i, 0], reversed when ornt[i, 1] == -1
    shape: Tuple[int, ...]      # shape after both transforms
    affine: np.ndarray          # affine after both transforms


def plan(affine, spatial_shape: Sequence[int], pixdim=None, diagonal: bool = False, axcodes=None,
         as_closest_canonical: bool = False, labels=LABELS) -> Plan:
    """Spacingd (when pixdim is given) followed by Orientationd (when axcodes is given or as_closest_canonical), as
    MONAI chains them: Orientationd sees the affine and shape that come out of Spacingd."""
    in_shape = tuple(int(s) for s in spatial_shape)
    if pixdim is None:
        a = np.eye(4) if affine is None else to_affine_nd(np.eye(4), affine)
        sp = SpacingGeom(np.eye(4), in_shape, a, True)
    else:
        sp = spacing(affine, in_shape, pixdim, diagonal)
    if axcodes is None and not as_closest_canonical:
        return Plan(in_shape, sp, np.array([[0, 1], [1, 1], [2, 1]]), sp.shape, sp.affine)
    ornt, shape, new_affine = orientation(sp.affine, sp.shape, axcodes, as_closest_canonical, labels)
    return Plan(in_shape, sp, ornt, shape, new_affine)


def index_map(p: Plan, start: Sequence[int], size: Sequence[int], flip_axes_mask: int = 0):
    """output index j of the window (start, size) of the oriented array, flipped on the axes of flip_axes_mask ->
    grid index q[i] = base[i] + step[i] * j[axis[i]]; returns (axis, base, step)"""
    axis, base, step = [], [], []
    for i in range(3):
        a = int(p.ornt[i, 0])
        if not (0 <= start[a] and start[a] + size[a] <= p.shape[a]):
            raise ValueError(f"window {tuple(start)} + {tuple(size)} does not fit in {p.shape}")
        b, s = (start[a] + size[a] - 1, -1) if flip_axes_mask >> a & 1 else (start[a], 1)
        if p.ornt[i, 1] < 0:
            b, s = p.spacing.shape[i] - 1 - b, -s
        axis.append(a); base.append(int(b)); step.append(s)
    return axis, base, step


TAP_DTYPE = np.dtype([("i0", np.int32), ("i1", np.int32), ("w0", np.float32), ("w1", np.float32)])


def axis_taps(p: Plan, nearest: bool) -> Optional[Tuple[Sequence[int], np.ndarray]]:
    """Per-axis interpolation tables when Spacingd's transform maps each grid axis to one source axis, else None.

    Source axis k follows grid axis tap_grid[k]; its table has one entry per grid index.  The coordinates are torch's:
    affine_grid evaluated on the one line of the grid along that axis gives, bit for bit, the coordinate it gives on
    every line of the full grid (the other axes meet exact zeros in theta), then grid_sample's unnormalisation
    ((x + 1) n - 1) / 2 and border clip in float64.  Nearest rounds half to even (nearbyint); bilinear keeps the two
    taps and grid_sample's weights (i0 + 1 - x, x - i0)."""
    sp, src, grid = p.spacing, p.in_shape, p.spacing.shape
    if sp.identity:
        tap_grid = [0, 1, 2]
        coords = [np.arange(n, dtype=np.float64) for n in src]
        nearest = True
    else:
        theta = affine_theta(sp.transform, src, grid)
        nz = theta[0, :3, :3].numpy() != 0
        if not ((nz.sum(0) == 1).all() and (nz.sum(1) == 1).all()):
            return None
        # theta row r / column c: source / grid axis 2 - r / 2 - c (affine_grid's x is the last axis)
        tap_grid = [2 - int(np.flatnonzero(nz[2 - k])[0]) for k in range(3)]
        coords = []
        for k in range(3):
            c = tap_grid[k]
            size = [1, 1, 1, 1, 1]
            size[2 + c] = grid[c]
            line = F.affine_grid(theta[:, :3], size, align_corners=False)[..., 2 - k].reshape(-1).numpy()
            n = src[k]
            ix = ((line + 1) * n - 1) / 2
            coords.append(np.minimum(float(n - 1), np.maximum(ix, 0.0)))
    parts = []
    for k in range(3):
        ix, n = coords[k], src[k]
        t = np.empty(len(ix), dtype=TAP_DTYPE)
        if nearest:
            i0 = np.rint(ix)
            t["i0"], t["i1"], t["w0"], t["w1"] = i0, i0, 1.0, 0.0
        else:
            f = np.floor(ix)
            t["i0"], t["i1"] = f, np.minimum(f + 1, n - 1)
            t["w0"], t["w1"] = (f + 1) - ix, ix - f
        parts.append(t)
    return tap_grid, parts
