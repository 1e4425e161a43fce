"""The training loader of the reference's 127-family scripts on the GPU
(10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:117-141): a device-resident sample cache and the
random tail of the Compose applied to a whole batch.

    DeviceCache(data, prefix)      runs the deterministic prefix (LoadImaged -> AsChannelFirstd -> ConvertToMultiChannel ->
                                   Spacingd / Orientationd, ...) once per item, on threads, and keeps every key of every item
                                   in one flat float32 device buffer per key (what MONAI's CacheDataset holds, on the GPU)
    TrainStage(cache, transforms)  the random tail (RandSpatialCropd -> RandFlipd -> intensity prologue -> disk -> plane wave
                                   -> wrap -> salt-and-pepper, each optional, SelectChanneld anywhere) as a handful of launches
                                   per batch: one crop + flip gather per key (mvtb_crop_flip_gather_f32), one statistics pass,
                                   one k-space chain call with the intensity map on the way in and the select on the way out

`draw` asks every transform object for its random parameters with its own `randomize`, sample after sample, in the order the
per-sample Compose would, so a batch gets exactly what the same objects would draw one sample at a time and leaves them in
the same state.  `apply` runs the batch on the device.  Parity is defined against the per-sample GPU drop-ins (mvtb.spatial,
mvtb.intensity, filters_and_operators): the same windows, flips, gates, spike locations and salt-and-pepper positions; the
image to float32 rounding (the k-space stages run as one chain instead of three), labels bit for bit.

Only the transforms listed in TrainStage's docstring, in that order, are accepted; anything else raises NotImplementedError
when the stage is built."""
import ctypes as C
import math
import types
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
from torch.utils.data import BatchSampler, RandomSampler, SequentialSampler

from . import _lib, functional as Fn, host, intensity as I, nifti as N, spatial as S


def _ops():
    import filters_and_operators as F                # the drop-in module lives next to the package
    return F


def _name(t) -> str:
    return type(t).__name__


def _keys(t) -> List[str]:
    return list(t.keys)


# ----------------------------------------------------------------------------------------------------------------- cache

class DeviceCache:
    """Every item of `data` (the scripts' list of dicts, e.g. {"image": path, "label": path}) after the deterministic
    `prefix`, on the device.  Allowed in the prefix: mvtb.nifti.LoadImaged / AsChannelFirstd, filters_and_operators'
    ConvertToMultiChannelBasedOnBratsClassesd / SelectChanneld, mvtb.spatial.Spacingd / Orientationd / SpacingOrientationd.

    The prefix runs per item on `num_workers` threads (the loaders and the resampling are thread-safe).  Each array key
    (a (C, H, W, D) volume; C equal for all items, H, W, D free, as Spacingd makes them) then lives in one flat float32
    buffer `buffers[key]`, with per-entry element offsets and spatial shapes in `offsets[key]` / `shapes[key]` (host numpy)
    and `offsets_dev[key]` / `shapes_dev[key]` (device).  Everything else of an item (the meta dicts) stays on the host in
    `meta[i]`.  Every item is cached; while the cache is filled the per-item results and the flat buffers coexist."""

    def __init__(self, data: Sequence[dict], prefix: Sequence, num_workers: int = 4, device: Optional[torch.device] = None):
        F = _ops()
        allowed = (N.LoadImaged, N.AsChannelFirstd, F.ConvertToMultiChannelBasedOnBratsClassesd, F.SelectChanneld,
                   S.Spacingd, S.Orientationd, S.SpacingOrientationd)
        for t in prefix:
            if not isinstance(t, allowed):
                raise NotImplementedError(f"DeviceCache: {_name(t)} is not a supported prefix transform "
                                          f"(supported: {', '.join(a.__name__ for a in allowed)})")
        Fn.require_cuda()
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        prefix = list(prefix)

        def one(item):
            d = dict(item)
            with torch.cuda.device(self.device):
                for t in prefix:
                    d = t(d)
                torch.cuda.current_stream(self.device).synchronize()
            return d

        if not len(data):
            raise ValueError("DeviceCache: no items")
        with ThreadPoolExecutor(max(1, int(num_workers))) as ex:
            items = list(ex.map(one, data))
        self.keys = [k for k, v in items[0].items() if isinstance(v, (torch.Tensor, np.ndarray)) and v.ndim == 4]
        if not self.keys:
            raise ValueError("DeviceCache: the prefix produced no (C, H, W, D) array")
        self.channels: Dict[str, int] = {}
        self.buffers: Dict[str, torch.Tensor] = {}
        self.offsets: Dict[str, np.ndarray] = {}
        self.shapes: Dict[str, np.ndarray] = {}
        self.offsets_dev: Dict[str, torch.Tensor] = {}
        self.shapes_dev: Dict[str, torch.Tensor] = {}
        for k in self.keys:
            vols = [it[k] for it in items]
            if any(not isinstance(v, (torch.Tensor, np.ndarray)) or v.ndim != 4 for v in vols):
                raise ValueError(f"DeviceCache: key {k!r} is not a (C, H, W, D) array in every item")
            ch = {int(v.shape[0]) for v in vols}
            if len(ch) != 1:
                raise ValueError(f"DeviceCache: key {k!r} has {sorted(ch)} channels across items; one count is needed")
            self.channels[k] = ch.pop()
            shp = np.array([v.shape[1:] for v in vols], dtype=np.int32)
            sizes = self.channels[k] * shp.astype(np.int64).prod(axis=1)
            off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
            buf = torch.empty(int(sizes.sum()), dtype=torch.float32, device=self.device)
            for i, v in enumerate(vols):
                buf[int(off[i]):int(off[i] + sizes[i])].copy_(torch.as_tensor(v).reshape(-1))
            for it in items:
                it[k] = None                            # release the per-item volume as soon as it is in the buffer
            self.buffers[k], self.offsets[k], self.shapes[k] = buf, off, shp
            self.offsets_dev[k] = torch.from_numpy(off).to(self.device)
            self.shapes_dev[k] = torch.from_numpy(shp.reshape(-1).copy()).to(self.device)
        self.meta = [{k: v for k, v in it.items() if k not in self.keys} for it in items]
        torch.cuda.synchronize(self.device)

    def __len__(self) -> int:
        return len(self.meta)

    def item(self, i: int) -> dict:
        """Item i as the prefix left it: (C, H, W, D) views of the cache plus its meta entries."""
        d = dict(self.meta[i])
        for k in self.keys:
            o, shp = int(self.offsets[k][i]), tuple(int(s) for s in self.shapes[k][i])
            d[k] = self.buffers[k][o:o + self.channels[k] * math.prod(shp)].view((self.channels[k],) + shp)
        return d


# ----------------------------------------------------------------------------------------------------------------- stage

# position of each supported transform in the 127 scripts' order; SelectChanneld and ToTensord may sit anywhere
_RANK = {"RandSpatialCropd": 0, "RandFlipd": 1, "NormalizeIntensityd": 2, "RandScaleIntensityd": 3, "RandShiftIntensityd": 4,
         "IntensityPrologued": (2, 4), "RandFourierDiskMaskd": 5, "RandPlaneWaves_ellipsoid": 6, "WrapArtifactd": 7,
         "SaltAndPepper": 8}


class TrainStage:
    """The random tail of the 127 scripts' training Compose on a DeviceCache, per batch.  Supported, in this order, each
    optional:

        mvtb.spatial.RandSpatialCropd(random_size=False) -> RandFlipd      over all cached keys
        mvtb.intensity.NormalizeIntensityd(nonzero=True, channel_wise=True) -> RandScaleIntensityd -> RandShiftIntensityd,
            or IntensityPrologued (scale / shift need the normalisation in front of them)
        filters_and_operators.RandFourierDiskMaskd(inside_off=False) -> RandPlaneWaves_ellipsoid -> WrapArtifactd
            -> SaltAndPepper(prob=1, rng="philox" or "philox-sparse")

    with filters_and_operators.SelectChanneld anywhere and MONAI's ToTensord as a no-op.  The intensity and k-space
    transforms act on one key (the image).  A SelectChanneld in front of the salt-and-pepper is folded into the gather;
    one behind it (the select takes its min / max over all channels) is applied to the result.

    `draw(indices)` (host only) returns a record of every random parameter; `apply(record)` returns the batch as CUDA
    float32 tensors (B, C, *roi) per key, plus per-sample lists of the meta dicts.  `loader(...)` yields
    apply(draw(batch)) in the order of a DataLoader on the same sampler.  `stage[i]` is draw([i]): a small host object
    that a forked DataLoader worker can produce (`DataLoader(stage, batch_size, collate_fn=list)` and apply on the
    collated list in the main process); each worker then draws from its own copy of the transforms, and MONAI's
    per-worker reseeding (worker_init_fn) changes the draws, as it does for the reference.  The copies include the
    salt-and-pepper `offset`, which starts equal in every worker and never advances in the main process: give each worker
    its own `sp.seed` in worker_init_fn (records carry the seed they were drawn with), or the workers' salt-and-pepper
    patterns repeat."""

    def __init__(self, cache: DeviceCache, transforms: Sequence):
        F = _ops()
        self.cache = cache
        self.tail = list(transforms)
        cached = set(cache.keys)
        ch = {k: list(range(cache.channels[k])) for k in cache.keys}     # current channel map per key (into the cache)
        self.pre_select = None                          # channel maps at the salt-and-pepper (what the gather reads)
        self.post_select: Dict[str, List[int]] = {}     # channels of the result kept after the salt-and-pepper
        self.crop = self.flip = self.norm = self.scale = self.shift = self.disk = self.wave = self.wrap = self.sp = None
        self.image_key = None
        last = -1
        for t in self.tail:
            n = _name(t)
            if n == "ToTensord":
                continue
            if isinstance(t, F.SelectChanneld):
                self._select(t, ch, cached)
                continue
            supported = {"RandSpatialCropd": S.RandSpatialCropd, "RandFlipd": S.RandFlipd, "NormalizeIntensityd": I.NormalizeIntensityd,
                         "RandScaleIntensityd": I.RandScaleIntensityd, "RandShiftIntensityd": I.RandShiftIntensityd,
                         "IntensityPrologued": I.IntensityPrologued, "RandFourierDiskMaskd": F.RandFourierDiskMaskd,
                         "RandPlaneWaves_ellipsoid": F.RandPlaneWaves_ellipsoid, "WrapArtifactd": F.WrapArtifactd,
                         "SaltAndPepper": F.SaltAndPepper}
            if n not in supported or not isinstance(t, supported[n]):
                raise NotImplementedError(f"TrainStage: {n} is not supported")
            lo, hi = _RANK[n] if isinstance(_RANK[n], tuple) else (_RANK[n], _RANK[n])
            if lo <= last:
                raise NotImplementedError(f"TrainStage: {n} after a transform that comes later in the 127 scripts' order "
                                          "(crop -> flip -> intensity -> disk -> plane wave -> wrap -> salt-and-pepper)")
            last = hi
            if n in ("RandSpatialCropd", "RandFlipd"):
                if set(_keys(t)) != cached:
                    raise NotImplementedError(f"TrainStage: {n} must act on every cached key {sorted(cached)}, not {_keys(t)}")
                if n == "RandSpatialCropd":
                    if t.random_size:
                        raise NotImplementedError("TrainStage: RandSpatialCropd(random_size=True) is not supported")
                    self.crop = t
                else:
                    self.flip = t
                continue
            keys = _keys(t) if n != "SaltAndPepper" else list(t.keys)
            if len(keys) != 1 or keys[0] not in cached or (self.image_key is not None and keys[0] != self.image_key):
                raise NotImplementedError(f"TrainStage: {n} must act on one cached key, the same for every intensity and "
                                          f"k-space transform (got {keys})")
            self.image_key = keys[0]
            if n == "NormalizeIntensityd":
                if not (t.nonzero and t.channel_wise):
                    raise NotImplementedError("TrainStage: only NormalizeIntensityd(nonzero=True, channel_wise=True)")
                self.norm = t
            elif n == "IntensityPrologued":
                self.norm, self.scale, self.shift = t, t.scale, t.shift
            elif n in ("RandScaleIntensityd", "RandShiftIntensityd"):
                if self.norm is None:
                    raise NotImplementedError(f"TrainStage: {n} without NormalizeIntensityd in front of it")
                if n == "RandScaleIntensityd":
                    self.scale = t
                else:
                    self.shift = t
            elif n == "RandFourierDiskMaskd":
                if t.inside_off:
                    raise NotImplementedError("TrainStage: RandFourierDiskMaskd(inside_off=True) is not supported")
                self.disk = t
            elif n == "RandPlaneWaves_ellipsoid":
                self.wave = t
            elif n == "WrapArtifactd":
                self.wrap = t
            else:
                if t.rng not in ("philox", "philox-sparse"):
                    raise NotImplementedError(f"TrainStage: SaltAndPepper(rng={t.rng!r}) draws on the host; use rng='philox' "
                                              "or 'philox-sparse'")
                if t.prob != 1:
                    raise NotImplementedError("TrainStage: SaltAndPepper needs prob=1")
                self.sp = t
                self.pre_select = {k: list(v) for k, v in ch.items()}
                ch = {k: list(range(len(v))) for k, v in ch.items()}
        if self.pre_select is None:
            self.pre_select = ch
        else:
            self.post_select = {k: v for k, v in ch.items() if v != list(range(len(self.pre_select[k])))}
        for k, v in self.pre_select.items():
            if len(v) > 8:
                raise NotImplementedError(f"TrainStage: {len(v)} channels of {k!r} in the gather; at most 8")
        if self.image_key is None:
            self.image_key = cache.keys[0]
        self._descs: dict = {}

    def _select(self, t, ch, cached):
        cn = t.chan_num
        keys = _keys(t)
        if any(k not in cached for k in keys):
            raise NotImplementedError(f"TrainStage: SelectChanneld on a key that is not cached ({keys})")
        per_key = isinstance(cn, (list, tuple)) and len(cn) > 1
        picks = list(zip(keys, cn)) if per_key else [(k, cn[0] if isinstance(cn, (list, tuple)) else cn) for k in keys]
        for k, c in picks:
            n = len(ch[k])
            c = int(c)
            if not -n <= c < n:
                raise ValueError(f"TrainStage: SelectChanneld channel {c} of {n} for key {k!r}")
            ch[k] = [ch[k][c]]

    # ---- host side
    def draw(self, indices: Sequence[int]) -> dict:
        """Every random parameter of the batch `indices`, sample after sample, from the transforms' own randomize (and the
        salt-and-pepper offsets, which advance as per-sample calls advance them).  Touches no CUDA state."""
        rec = {k: [] for k in ("index", "start", "size", "flip", "scale_gate", "factor", "shift_gate", "offset", "disk_gate",
                               "r", "spike_gate", "spike_idx", "sp_gate", "sp_seed", "sp_offset", "sp_blocks")}
        first = self.crop.keys[0] if self.crop is not None else self.cache.keys[0]
        for i in indices:
            i = int(i)
            rec["index"].append(i)
            shape = tuple(int(s) for s in self.cache.shapes[first][i])
            start, size = (0, 0, 0), shape
            fm = 0
            for t in self.tail:
                if t is self.crop:
                    t.randomize(shape)
                    start, size = tuple(int(v) for v in t._start), tuple(int(v) for v in t._size)
                elif t is self.flip:
                    t.randomize(None)
                    fm = S._flip_mask(t.spatial_axis, 3) if t._do_transform else 0
                elif isinstance(t, I.IntensityPrologued):
                    t.scale.randomize()
                    t.shift.randomize()
                elif t is self.scale:
                    t.randomize()
                elif t is self.shift:
                    t.randomize()
                elif t is self.disk:
                    t.randomize()
                    rec["disk_gate"].append(bool(t._do_transform))
                    rec["r"].append(float(t.r) if not isinstance(t.r, list) else None)
                elif t is self.wave:
                    t.randomize(None)
                    idx = None
                    if t._do_transform:
                        t.idx = t.ellipsoid.sample_ellipsoid(types.SimpleNamespace(shape=size))
                        idx = tuple(int(v) for v in t.idx)
                    rec["spike_gate"].append(bool(t._do_transform))
                    rec["spike_idx"].append(idx)
                elif t is self.sp:
                    t.randomize(None)
                    n = len(self.pre_select[self.image_key]) * math.prod(size)
                    blocks = (n + 255) // 256 if t.rng == "philox-sparse" else (n + 3) // 4
                    rec["sp_gate"].append(bool(t._do_transform))
                    rec["sp_seed"].append(int(t.seed))
                    rec["sp_offset"].append(int(t.offset))
                    rec["sp_blocks"].append(blocks)
                    if t._do_transform:
                        t.offset += blocks
            if self.scale is not None:
                rec["scale_gate"].append(bool(self.scale._do_transform))
                rec["factor"].append(float(self.scale.factor))
            if self.shift is not None:
                rec["shift_gate"].append(bool(self.shift._do_transform))
                rec["offset"].append(float(self.shift._offset))
            rec["start"].append(start)
            rec["size"].append(size)
            rec["flip"].append(fm)
        return rec

    def __len__(self) -> int:
        return len(self.cache)

    def __getitem__(self, i: int) -> dict:
        return self.draw([i])

    # ---- device side
    def _desc(self, roi, r, idx):
        key = (roi, r, idx)
        d = self._descs.get(key)
        if d is None:
            kw = {}
            if r is not None:
                kw.update(mask_kind=_lib.MASK_DISK, mask_ndim=3, mask_thresh=host.disk_threshold(r, roi))
            if idx is not None:
                kw["spikes"] = [(idx, host.exp_f32(self.wave.intensity_value))]
            if self.wrap is not None:
                kw["wrap_alpha"] = float(self.wrap.transform.alpha)
            d = host.make_desc(**kw)
            if len(self._descs) >= 4096:
                self._descs.clear()
            self._descs[key] = d
        return d

    def apply(self, record) -> dict:
        """The batch of `record` (a draw, or a list of draws) on the device: {key: (B, C, *roi) float32 CUDA tensor,
        meta key: [one meta entry per sample]}."""
        if isinstance(record, (list, tuple)):
            rec = {k: [v for r in record for v in r[k]] for k in record[0]}
        else:
            rec = record
        cache, dev = self.cache, self.cache.device
        B = len(rec["index"])
        sizes = {tuple(s) for s in rec["size"]}
        if len(sizes) != 1:
            raise ValueError(f"TrainStage: the batch has crops of different sizes {sorted(sizes)}; a batch needs one")
        roi = sizes.pop()
        idx = np.asarray(rec["index"], dtype=np.int64)
        starts = np.asarray(rec["start"], dtype=np.int32).reshape(B, 3)
        if idx.min() < 0 or idx.max() >= len(cache):
            raise IndexError(f"TrainStage: sample index outside the {len(cache)} cached items")
        for k in cache.keys:
            shp = cache.shapes[k][idx]
            if (starts < 0).any() or (starts + np.asarray(roi, dtype=np.int32) > shp).any():
                raise ValueError(f"TrainStage: a window does not fit in its cached {k!r} volume")
        ik = self.image_key
        c_img = len(self.pre_select[ik])
        has_int = self.norm is not None
        # the per-sample arrays of every step, uploaded in one copy from pinned memory
        n_int = 5 * B
        n_flt = 2 * B * c_img if has_int else 0
        pinned = torch.empty(n_int + n_flt, dtype=torch.int32, pin_memory=True)
        pv = pinned.numpy()
        pv[:B] = idx
        pv[B:4 * B] = starts.reshape(-1)
        pv[4 * B:5 * B] = rec["flip"]
        if has_int:
            sc = np.ones(B, dtype=np.float32) if self.scale is None else \
                np.where(rec["scale_gate"], 1.0 + np.asarray(rec["factor"], dtype=np.float64), 1.0).astype(np.float32)
            sh = np.zeros(B, dtype=np.float32) if self.shift is None else \
                np.where(rec["shift_gate"], np.asarray(rec["offset"], dtype=np.float64), 0.0).astype(np.float32)
            fv = pv[n_int:].view(np.float32)
            fv[:B * c_img] = np.repeat(sc, c_img)
            fv[B * c_img:] = np.repeat(sh, c_img)
        up = pinned.to(dev, non_blocking=True)
        entry_d, starts_d, flips_d = up[:B], up[B:4 * B], up[4 * B:5 * B]
        L = _lib.lib()
        i3 = C.c_int32 * 3
        out = {}
        with torch.cuda.device(dev):
            stream = Fn._stream(dev)
            for k in cache.keys:
                chans = self.pre_select[k]
                y = torch.empty((B, len(chans)) + roi, dtype=torch.float32, device=dev)
                rc = L.mvtb_crop_flip_gather_f32(Fn._ptr(cache.buffers[k]), Fn._ptr(y), B, len(chans), Fn._ptr(cache.offsets_dev[k]),
                                                 Fn._ptr(cache.shapes_dev[k]), cache.channels[k], (C.c_int32 * len(chans))(*chans),
                                                 i3(*roi), Fn._ptr(entry_d), Fn._ptr(starts_d), Fn._ptr(flips_d), stream)
                _lib.check(L, rc)
                out[k] = y
            x = out[ik]
            abt = None
            if has_int:
                scale_d = up[n_int:n_int + B * c_img].view(torch.float32)
                shift_d = up[n_int + B * c_img:].view(torch.float32)
                abt = Fn.intensity_coeffs(x, B * c_img, scale=scale_d, shift=shift_d)
            if self.disk or self.wave or self.wrap or self.sp:
                x = self._chain(x, rec, roi, B, c_img, abt)
            elif abt is not None:
                x = Fn.intensity_affine(x, abt, out=x)
            out[ik] = x
        for k, chans in self.post_select.items():
            out[k] = out[k][:, chans].contiguous()
        for mk in (cache.meta[0].keys() if cache.meta else ()):
            out[mk] = [cache.meta[i][mk] for i in rec["index"]]
        return out

    def _chain(self, x, rec, roi, B, c_img, abt):
        descs = []
        for b in range(B):
            r = rec["r"][b] if self.disk is not None and rec["disk_gate"][b] else None
            idx = rec["spike_idx"][b] if self.wave is not None else None
            descs.extend([self._desc(roi, r, idx)] * c_img)
        descs = host.desc_array(descs)
        sp = self.sp
        if sp is None or not any(rec["sp_gate"]):
            return Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, out=x)
        off, blocks, seed = rec["sp_offset"], rec["sp_blocks"], rec["sp_seed"]
        # one select call when the batch's counters follow each other as per-sample calls would have used them
        contiguous = all(rec["sp_gate"]) and all(off[b] == off[0] + b * blocks[0] and blocks[b] == blocks[0] and seed[b] == seed[0]
                                                 for b in range(B))
        sparse = sp.rng == "philox-sparse"
        if sparse and contiguous:
            return Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, sp=(float(sp.p), seed[0], off[0], blocks[0]), vols_per_sample=c_img,
                                      out=x)[0]
        y, mm = Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, want_minmax=True, vols_per_sample=c_img, out=x)
        n = y[0].numel()
        if not sparse and contiguous and n % 4 == 0:      # dense Philox: element i of the batch uses counter offset + i / 4
            return Fn.salt_pepper(y, float(sp.p), seed=seed[0], offset=off[0], n_samples=B, mm=mm, out=y)
        for b in range(B):
            if rec["sp_gate"][b]:
                Fn.salt_pepper(y[b], float(sp.p), seed=seed[b], offset=off[b], n_samples=1, mm=mm[b:b + 1], out=y[b], sparse=sparse)
        return y

    def loader(self, batch_size: int, shuffle: bool = True, drop_last: bool = False, generator: Optional[torch.Generator] = None):
        """apply(draw(batch)) for the batches of BatchSampler(RandomSampler / SequentialSampler): the order of a DataLoader
        with the same arguments and generator."""
        src = range(len(self.cache))
        sampler = RandomSampler(src, generator=generator) if shuffle else SequentialSampler(src)
        for batch in BatchSampler(sampler, batch_size, drop_last):
            yield self.apply(self.draw(batch))
