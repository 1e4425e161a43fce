"""The spatial part of the reference's training pipelines on the GPU: drop-ins for the MONAI 0.5 dictionary transforms between
the resampled volume and the intensity prologue
(10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:130-133, :153)

    RandSpatialCropd(keys, roi_size, random_center=True, random_size=True) -> RandFlipd(keys, prob, spatial_axis)
    CenterSpatialCropd(keys, roi_size)

with MONAI's constructor arguments and random draw order (one `R.randint(0, N - roi + 1)` per axis that is larger than the
roi, in axis order; one `R.random() < prob` for the flip), and `CropFlipd`, the two as one gather.  The data movement is
`mvtb_crop_flip_f32` in libmvtb.so (csrc/spatial.cu); no CPU fallback.  Every key of a sample shares the drawn window and
flip, as in MONAI (the window is drawn from the first key's shape).

In front of them, `Spacingd` -> `Orientationd` (127_...FLAIR.py:120-129) resample the loaded volume to the training grid:
`resample` runs both, plus an optional window and flip, as one gather (`mvtb_resample_f32`, csrc/resample.cuh) on the
geometry of mvtb/geometry.py; `SpacingOrientationd` is the two drop-ins in one pass."""
import ctypes as C
import threading
from collections import OrderedDict
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib, functional as Fn, geometry as Geo
from ._monai_compat import KeysCollection, MapTransform, Randomizable, RandomizableTransform


def _fall_back(roi_size, img_size: Sequence[int]) -> Tuple[int, ...]:
    nd = len(img_size)
    user = tuple(roi_size) if isinstance(roi_size, (list, tuple, np.ndarray)) else (roi_size,) * nd
    if len(user) != nd:
        raise ValueError(f"roi_size has {len(user)} entries for {nd} spatial axes")
    return tuple(int(d) if (u is None or u <= 0) else int(u) for u, d in zip(user, img_size))


def _flip_mask(spatial_axis: Optional[Union[int, Sequence[int]]], nd: int) -> int:
    if spatial_axis is None:
        axes = range(nd)
    elif isinstance(spatial_axis, int):
        axes = (spatial_axis,)
    else:
        axes = tuple(spatial_axis)
    m = 0
    for a in axes:
        a = a + nd if a < 0 else a
        if not 0 <= a < nd:
            raise ValueError(f"spatial_axis {a} outside the {nd} spatial axes")
        m |= 1 << a
    return m


def crop_flip(x, start: Sequence[int], size: Sequence[int], flip_axes_mask: int = 0):
    """out = flip(x[:, start : start + size]) for a (C, H, W, D) (or (C, H, W)) sample; result on x's device, in x's precision."""
    xd, org = Fn.to_device(x)
    nd = xd.dim() - 1
    if nd not in (2, 3):
        raise ValueError(f"crop_flip expects a (C, H, W[, D]) sample, got rank {xd.dim()}")
    shp = tuple(xd.shape[1:]) if nd == 3 else (1,) + tuple(xd.shape[1:])          # 2-D: a leading axis of length 1
    st = tuple(int(v) for v in start) if nd == 3 else (0,) + tuple(int(v) for v in start)
    sz = tuple(int(v) for v in size) if nd == 3 else (1,) + tuple(int(v) for v in size)
    fm = flip_axes_mask if nd == 3 else flip_axes_mask << 1
    out = torch.empty((xd.shape[0],) + (sz if nd == 3 else sz[1:]), dtype=torch.float32, device=xd.device)
    L = _lib.lib()
    i3 = C.c_int32 * 3
    with torch.cuda.device(xd.device):
        rc = L.mvtb_crop_flip_f32(Fn._ptr(xd), Fn._ptr(out), int(xd.shape[0]), i3(*shp), i3(*sz), i3(*st), int(fm), Fn._stream(xd.device))
    _lib.check(L, rc)
    return Fn.back(out, org)


def crop_flip_batch(x: torch.Tensor, starts, size: Sequence[int], flip_masks) -> torch.Tensor:
    """out[b] = flip_b(x[b, :, start_b : start_b + size]) for a CUDA batch (B, C, H, W, D) in one launch; starts: (B, 3) ints,
    flip_masks: (B,) ints (bit a = spatial axis a), as tensors or sequences."""
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous() or x.dim() != 5:
        raise ValueError("crop_flip_batch expects a contiguous float32 CUDA tensor (B, C, H, W, D)")
    B_, C_ = int(x.shape[0]), int(x.shape[1])
    st = torch.as_tensor(starts, dtype=torch.int32).reshape(B_, 3)
    fm = torch.as_tensor(flip_masks, dtype=torch.int32).reshape(B_)
    sz = tuple(int(v) for v in size)
    if bool((st < 0).any()) or any(int(st[:, a].max()) + sz[a] > int(x.shape[2 + a]) for a in range(3)):
        raise ValueError("crop_flip_batch: a window does not fit in the volume")
    st, fm = st.to(x.device), fm.to(x.device)
    out = torch.empty((B_, C_) + sz, dtype=torch.float32, device=x.device)
    L = _lib.lib()
    i3 = C.c_int32 * 3
    with torch.cuda.device(x.device):
        rc = L.mvtb_crop_flip_batch_f32(Fn._ptr(x), Fn._ptr(out), B_, C_, i3(*[int(v) for v in x.shape[2:]]), i3(*sz), Fn._ptr(st), Fn._ptr(fm),
                                        Fn._stream(x.device))
    _lib.check(L, rc)
    return out


def _center_start(img_size: Sequence[int], roi: Sequence[int]):
    """CenterSpatialCrop -> SpatialCrop(roi_center=[i // 2], roi_size): start = max(center - roi // 2, 0), clipped at the end"""
    start = [max(n // 2 - r // 2, 0) for n, r in zip(img_size, roi)]
    size = [min(s + r, n) - s for s, r, n in zip(start, roi, img_size)]
    return start, size


class CenterSpatialCropd(MapTransform):
    def __init__(self, keys: KeysCollection, roi_size, allow_missing_keys: bool = False) -> None:
        super().__init__(keys, allow_missing_keys)
        self.roi_size = roi_size

    def __call__(self, data):
        d = dict(data)
        for key in self.key_iterator(d):
            img_size = tuple(d[key].shape[1:])
            start, size = _center_start(img_size, _fall_back(self.roi_size, img_size))
            d[key] = crop_flip(d[key], start, size, 0)
        return d


class RandSpatialCropd(Randomizable, MapTransform):
    def __init__(self, keys: KeysCollection, roi_size, random_center: bool = True, random_size: bool = True,
                 allow_missing_keys: bool = False) -> None:
        MapTransform.__init__(self, keys, allow_missing_keys)
        self.roi_size, self.random_center, self.random_size = roi_size, random_center, random_size
        self._start: Optional[Sequence[int]] = None
        self._size: Optional[Sequence[int]] = None

    def randomize(self, img_size: Sequence[int]) -> None:
        self._size = _fall_back(self.roi_size, img_size)
        if self.random_size:
            self._size = tuple(self.R.randint(low=self._size[i], high=img_size[i] + 1) for i in range(len(img_size)))
        if self.random_center:
            valid = tuple(min(ms, ps or ms) for ms, ps in zip(img_size, self._size))
            self._start = tuple(self.R.randint(low=0, high=ms - ps + 1) if ms > ps else 0 for ms, ps in zip(img_size, valid))
            self._size = valid
        else:
            self._start, self._size = _center_start(img_size, self._size)

    def __call__(self, data):
        d = dict(data)
        self.randomize(tuple(d[self.keys[0]].shape[1:]))             # the first key's shape, as in MONAI
        for key in self.key_iterator(d):
            d[key] = crop_flip(d[key], self._start, self._size, 0)
        return d


class RandFlipd(RandomizableTransform, MapTransform):
    def __init__(self, keys: KeysCollection, prob: float = 0.1, spatial_axis: Optional[Union[Sequence[int], int]] = None,
                 allow_missing_keys: bool = False) -> None:
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, prob)
        self.spatial_axis = spatial_axis

    def __call__(self, data):
        self.randomize(None)
        d = dict(data)
        if not self._do_transform:
            return d
        for key in self.key_iterator(d):
            nd = d[key].dim() - 1 if isinstance(d[key], torch.Tensor) else np.ndim(d[key]) - 1
            d[key] = crop_flip(d[key], (0,) * nd, tuple(d[key].shape[1:]), _flip_mask(self.spatial_axis, nd))
        return d


class CropFlipd(Randomizable, MapTransform):
    """RandSpatialCropd(random_size=False) followed by RandFlipd as ONE pass over the crop: the same draws in the same order
    from two random states (set_random_state seeds both the way Compose seeds two consecutive transforms)."""

    def __init__(self, keys: KeysCollection, roi_size, prob: float = 0.5, spatial_axis=0, allow_missing_keys: bool = False) -> None:
        MapTransform.__init__(self, keys, allow_missing_keys)
        self.crop = RandSpatialCropd(keys, roi_size, random_center=True, random_size=False, allow_missing_keys=allow_missing_keys)
        self.flipper = RandFlipd(keys, prob, spatial_axis, allow_missing_keys=allow_missing_keys)

    def set_random_state(self, seed: Optional[int] = None, state: Optional[np.random.RandomState] = None):
        Randomizable.set_random_state(self, seed, state)
        MAX_SEED = np.iinfo(np.uint32).max + 1
        self.crop.set_random_state(seed=int(self.R.randint(MAX_SEED, dtype="uint32")))
        self.flipper.set_random_state(seed=int(self.R.randint(MAX_SEED, dtype="uint32")))
        return self

    def randomize(self, data=None) -> None:
        pass

    def __call__(self, data):
        d = dict(data)
        self.crop.randomize(tuple(d[self.keys[0]].shape[1:]))
        self.flipper.randomize(None)
        for key in self.key_iterator(d):
            nd = len(self.crop._size)
            fm = _flip_mask(self.flipper.spatial_axis, nd) if self.flipper._do_transform else 0
            d[key] = crop_flip(d[key], self.crop._start, self.crop._size, fm)
        return d


# ----------------------------------------------------------------------------- Spacingd / Orientationd

# per-axis tap tables on the device, per (device, geometry, mode): a cache fill of equal-shape volumes uploads them once
_TAPS_MAX = 32
_taps_lock = threading.Lock()
_taps_cache: "OrderedDict" = OrderedDict()


def tap_tables(p: Geo.Plan, nearest: bool):
    """(tap_grid, first entry per source axis, one mvtb_resample_tap array) of geometry.axis_taps, or None"""
    t = Geo.axis_taps(p, nearest)
    if t is None:
        return None
    tap_grid, parts = t
    return tap_grid, np.cumsum([0] + [len(q) for q in parts[:-1]]).tolist(), np.concatenate(parts)


def _device_taps(p: Geo.Plan, nearest: bool, dev: torch.device):
    key = (dev.index, p.in_shape, p.spacing.shape, p.spacing.transform.tobytes(), p.spacing.identity, nearest)
    with _taps_lock:
        hit = _taps_cache.get(key, False)
        if hit is not False:
            _taps_cache.move_to_end(key)
            return hit
    t = tap_tables(p, nearest)
    if t is not None:
        t = (t[0], t[1], torch.from_numpy(t[2].view(np.uint8).copy()).to(dev))
    with _taps_lock:
        _taps_cache[key] = t
        while len(_taps_cache) > _TAPS_MAX:
            _taps_cache.popitem(last=False)
    return t


def resample_geom(p: Geo.Plan, nearest: bool, window=None, flip_axes_mask: int = 0, taps=None, taps_ptr: int = 0):
    """the mvtb_resample_geom of `p` with an optional window (start, size) and flip; taps: tap_tables(p, nearest) (its
    array at address taps_ptr), None for the general path.  Returns (geom, output spatial shape)."""
    start, size = ((0, 0, 0), p.shape) if window is None else (tuple(int(v) for v in window[0]), tuple(int(v) for v in window[1]))
    if flip_axes_mask & ~7:
        raise ValueError(f"flip_axes_mask {flip_axes_mask} has bits beyond the 3 spatial axes")
    axis, base, step = Geo.index_map(p, start, size, flip_axes_mask)
    i3 = C.c_int32 * 3
    g = _lib.ResampleGeom(in_shape=i3(*p.in_shape), grid_shape=i3(*p.spacing.shape), out_shape=i3(*size), axis=i3(*axis),
                          base=i3(*base), step=i3(*step),
                          mode=_lib.RESAMPLE_NEAREST if (nearest or p.spacing.identity) else _lib.RESAMPLE_BILINEAR)
    if taps is not None:
        g.tap_grid, g.tap_off, g.n_taps, g.taps = i3(*taps[0]), i3(*taps[1]), taps[2].nbytes // C.sizeof(_lib.ResampleTap), taps_ptr
    else:
        g.matrix = (C.c_double * 12)(*p.spacing.transform[:3].ravel().tolist())
    return g, tuple(size)


def _check_options(mode, padding_mode, align_corners, dtype) -> bool:
    """True for nearest; the options no script of the reference uses raise"""
    if mode not in ("bilinear", "nearest"):
        raise NotImplementedError(f"mode {mode!r}: only 'bilinear' and 'nearest' are implemented")
    if padding_mode != "border":
        raise NotImplementedError(f"padding_mode {padding_mode!r}: only 'border' is implemented")
    if align_corners:
        raise NotImplementedError("align_corners=True is not implemented")
    if dtype is not None and np.dtype(dtype) != np.float64:
        raise NotImplementedError(f"dtype {dtype}: the coordinates are computed in float64 only")
    return mode == "nearest"


def center_window(shape: Sequence[int], roi_size):
    """CenterSpatialCropd's window (start, size) on an array of spatial `shape`"""
    return _center_start(tuple(shape), _fall_back(roi_size, tuple(shape)))


def resample(x, p: Geo.Plan, mode: str = "bilinear", window=None, flip_axes_mask: int = 0, padding_mode: str = "border",
             align_corners: bool = False, dtype=np.float64):
    """Spacingd -> Orientationd of a (C, H, W, D) volume as one gather, as described by `p` (geometry.plan), then the
    window (start, size) of the oriented array (default: all of it) flipped on the axes of flip_axes_mask (bit a =
    spatial axis a).  C may stack channels and samples of the same geometry.  float32 result: a CUDA input stays on
    its device, a CPU tensor comes back as a CPU tensor, a numpy array as a numpy array."""
    nearest = _check_options(mode, padding_mode, align_corners, dtype)
    is_np = isinstance(x, np.ndarray)
    xd, org = Fn.to_device(x)
    if xd.dim() != 4 or tuple(xd.shape[1:]) != tuple(p.in_shape):
        raise ValueError(f"resample expects a (C, {', '.join(map(str, p.in_shape))}) array, got {tuple(xd.shape)}")
    taps = _device_taps(p, nearest, xd.device)
    g, size = resample_geom(p, nearest, window, flip_axes_mask, taps, 0 if taps is None else taps[2].data_ptr())
    if taps is not None:
        taps[2].record_stream(torch.cuda.current_stream(xd.device))      # the cache may drop it while the gather runs
    out = torch.empty((xd.shape[0],) + size, dtype=torch.float32, device=xd.device)
    L = _lib.lib()
    with torch.cuda.device(xd.device):
        rc = L.mvtb_resample_f32(Fn._ptr(xd), Fn._ptr(out), int(xd.shape[0]), C.byref(g), Fn._stream(xd.device))
    _lib.check(L, rc)
    if out.device != org.device:
        out = out.to(org.device)
    return out.numpy() if is_np else out


def _per_key(v, n: int, name: str):
    if isinstance(v, (list, tuple)):
        if len(v) != n:
            raise ValueError(f"{name} has {len(v)} entries for {n} keys")
        return tuple(v)
    return (v,) * n


class _Resampled(MapTransform):
    """shared by the three drop-ins: per key, read d[f"{key}_{postfix}"]["affine"], resample, write the new affine back"""

    def __init__(self, keys, pixdim, diagonal, mode, padding_mode, align_corners, dtype, axcodes, as_closest_canonical,
                 labels, meta_key_postfix, allow_missing_keys):
        MapTransform.__init__(self, keys, allow_missing_keys)
        n = len(self.keys)
        self.pixdim, self.diagonal = pixdim, diagonal
        self.mode = _per_key(mode, n, "mode")
        self.padding_mode = _per_key(padding_mode, n, "padding_mode")
        self.align_corners = _per_key(align_corners, n, "align_corners")
        self.dtype = _per_key(dtype, n, "dtype")
        for m, pm, ac, dt in zip(self.mode, self.padding_mode, self.align_corners, self.dtype):
            _check_options(m, pm, ac, dt)
        self.axcodes, self.as_closest_canonical, self.labels = axcodes, as_closest_canonical, labels
        self.meta_key_postfix = meta_key_postfix

    def __call__(self, data):
        d = dict(data)
        for key, mode, pm, ac, dt in self.key_iterator(d, self.mode, self.padding_mode, self.align_corners, self.dtype):
            meta = d[f"{key}_{self.meta_key_postfix}"]
            p = Geo.plan(meta["affine"], tuple(d[key].shape[1:]), self.pixdim, self.diagonal, self.axcodes,
                         self.as_closest_canonical, self.labels)
            d[key] = resample(d[key], p, mode, padding_mode=pm, align_corners=ac, dtype=dt)
            meta["affine"] = p.affine
        return d


class Spacingd(_Resampled):
    """MONAI 0.5 Spacingd on the GPU: resample to voxel size `pixdim` (one mode per key, as the scripts pass it)."""

    def __init__(self, keys: KeysCollection, pixdim, diagonal: bool = False, mode="bilinear", padding_mode="border",
                 align_corners=False, dtype=np.float64, meta_key_postfix: str = "meta_dict", allow_missing_keys: bool = False):
        super().__init__(keys, pixdim, diagonal, mode, padding_mode, align_corners, dtype, None, False, Geo.LABELS,
                         meta_key_postfix, allow_missing_keys)


class Orientationd(_Resampled):
    """MONAI 0.5 Orientationd on the GPU: reorder and flip the axes to `axcodes` (a copy of the data)."""

    def __init__(self, keys: KeysCollection, axcodes=None, as_closest_canonical: bool = False, labels=Geo.LABELS,
                 meta_key_postfix: str = "meta_dict", allow_missing_keys: bool = False):
        if axcodes is None and not as_closest_canonical:
            raise ValueError("Incompatible values: axcodes=None and as_closest_canonical=True.")
        super().__init__(keys, None, False, "nearest", "border", False, np.float64, axcodes, as_closest_canonical, labels,
                         meta_key_postfix, allow_missing_keys)


class SpacingOrientationd(_Resampled):
    """Spacingd followed by Orientationd in one gather; the same bits and the same affine as the two in sequence."""

    def __init__(self, keys: KeysCollection, pixdim, axcodes=None, diagonal: bool = False, mode="bilinear",
                 padding_mode="border", align_corners=False, dtype=np.float64, as_closest_canonical: bool = False,
                 labels=Geo.LABELS, meta_key_postfix: str = "meta_dict", allow_missing_keys: bool = False):
        if axcodes is None and not as_closest_canonical:
            raise ValueError("Incompatible values: axcodes=None and as_closest_canonical=True.")
        super().__init__(keys, pixdim, diagonal, mode, padding_mode, align_corners, dtype, axcodes, as_closest_canonical,
                         labels, meta_key_postfix, allow_missing_keys)
