"""TEST INFRASTRUCTURE ONLY (tests/, tools/bench_resample.py): the MONAI 0.5 resampling at the front of the reference's
pipelines (10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:120-129, utils.py:186-198):

    Spacingd(["image", "label"], pixdim=(1.5, 1.5, 2.0), mode=("bilinear", "nearest")) -> Orientationd(axcodes="RAS")

MONAI and nibabel are not dependencies of this project, so this restates their published algorithm
(monai/transforms/spatial/array.py: Spacing, Orientation; monai/networks/layers/spatial_transforms.py: AffineTransform).
The affine and shape arithmetic is the numpy restatement in mvtb/geometry.py, pinned by known-answer tests
(tests/test_resample.py); the voxels are moved the way MONAI moves them: torch.nn.functional.affine_grid + grid_sample
on the CPU in float64 over the full grid (align_corners=False, border padding), cast to float32, and nibabel's
apply_orientation (np.flip, then transpose).  PARITY UNPINNED against MONAI itself."""
import numpy as np
import torch
import torch.nn.functional as F

from mvtb import geometry as G


def spacing(img: np.ndarray, affine, pixdim, diagonal: bool = False, mode: str = "bilinear"):
    """Spacing.__call__ on a (C, H, W, D) array -> (float32 array, new affine)"""
    sp = G.spacing(affine, img.shape[1:], pixdim, diagonal)
    if sp.identity:
        return img.copy().astype(np.float32), sp.affine
    src = torch.as_tensor(np.ascontiguousarray(img).astype(np.float64)).unsqueeze(0)
    grid = F.affine_grid(G.affine_theta(sp.transform, img.shape[1:], sp.shape)[:, :3], [1, img.shape[0]] + list(sp.shape),
                         align_corners=False)
    out = F.grid_sample(src, grid, mode=mode, padding_mode="border", align_corners=False)
    return out.squeeze(0).numpy().astype(np.float32), sp.affine


def source_coords(shape, affine, pixdim, diagonal: bool = False) -> np.ndarray:
    """the source index grid_sample computes for every voxel of Spacing's grid, (3, s0, s1, s2) float64, source axis
    order, before the border clip"""
    sp = G.spacing(affine, shape, pixdim, diagonal)
    grid = F.affine_grid(G.affine_theta(sp.transform, shape, sp.shape)[:, :3], [1, 1] + list(sp.shape), align_corners=False)
    return np.stack([((grid[0, ..., 2 - k].numpy() + 1) * shape[k] - 1) / 2 for k in range(3)])


def orientation(img: np.ndarray, affine, axcodes=None, as_closest_canonical: bool = False, labels=G.LABELS):
    """Orientation.__call__ on a (C, H, W, D) array -> (array, new affine)"""
    ornt, _, new_affine = G.orientation(affine, img.shape[1:], axcodes, as_closest_canonical, labels)
    full = np.concatenate([np.array([[0, 1]]), np.column_stack([ornt[:, 0] + 1, ornt[:, 1]])])
    return np.ascontiguousarray(G.apply_orientation(img, full)), new_affine


def spacing_orientation(img: np.ndarray, affine, pixdim, axcodes="RAS", diagonal: bool = False, mode: str = "bilinear"):
    out, a = spacing(img, affine, pixdim, diagonal, mode)
    return orientation(out, a, axcodes)
