"""The training loader of the reference's 127-family scripts on the GPU
(10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:117-141): a device-resident sample cache and the
random tail of the Compose applied to a whole batch.

    DeviceCache(data, prefix)      runs the deterministic prefix (LoadImaged -> AsChannelFirstd -> ConvertToMultiChannel ->
                                   Spacingd / Orientationd, ...) once per item, on threads, and keeps every key of every item
                                   in one flat float32 device buffer per key (what MONAI's CacheDataset holds, on the GPU);
                                   for validation the prefix ends in CenterSpatialCropd, fused into the resampling gather
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
from collections.abc import Sequence as _SeqABC
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

class ResampleCenterCrop:
    """A Spacingd / Orientationd / SpacingOrientationd and the CenterSpatialCropd right behind it, on some of its keys, as one
    step of a cache fill: each cropped key is one windowed gather (mvtb.spatial's resample_crop)."""

    def __init__(self, resample, crop):
        self.resample, self.crop = resample, crop

    def __call__(self, data):
        return self.resample.resample_crop(data, self.crop)


def fill_steps(prefix: Sequence) -> list:
    """The steps a DeviceCache runs for `prefix`: the transforms themselves, except that a CenterSpatialCropd directly behind
    a resampling transform, acting on a subset of its keys, joins it as one ResampleCenterCrop."""
    steps: list = []
    for t in prefix:
        prev = steps[-1] if steps else None
        if (isinstance(t, S.CenterSpatialCropd) and isinstance(prev, (S.Spacingd, S.Orientationd, S.SpacingOrientationd))
                and set(_keys(t)) <= set(_keys(prev))):
            steps[-1] = ResampleCenterCrop(prev, t)
        else:
            steps.append(t)
    return steps


class DeviceCache:
    """Every item of `data` (the scripts' list of dicts, e.g. {"image": path, "label": path}) after the deterministic
    `prefix`, on the device.  Allowed in the prefix: mvtb.nifti.LoadImaged / AsChannelFirstd, filters_and_operators'
    ConvertToMultiChannelBasedOnBratsClassesd / WholeTumorTCGA / SelectChanneld, mvtb.spatial.Spacingd / Orientationd /
    SpacingOrientationd / CenterSpatialCropd.

    A CenterSpatialCropd directly behind Spacingd, Orientationd or SpacingOrientationd, on a subset of its keys (the
    validation prefix), is fused into the resampling gather of those keys (`fill_steps`): the fill then reads the loaded
    volume once and writes only the crop, with the same bits and meta dicts as the two transforms in sequence.  Anywhere
    else it runs as the drop-in.  As in MONAI, a volume smaller than the roi on some axis gives a smaller crop; the cache
    holds it like any other ragged entry, and TrainStage.apply refuses a batch of different sizes with ValueError.

    The prefix runs per item on `num_workers` threads (the loaders and the resampling are thread-safe).  Each array key
    (a (C, H, W, D) volume; C equal for all items, H, W, D free, as Spacingd makes them) then lives in one flat float32
    buffer `buffers[key]`, with per-entry element offsets and spatial shapes in `offsets[key]` / `shapes[key]` (host numpy)
    and `offsets_dev[key]` / `shapes_dev[key]` (device).  Everything else of an item (the meta dicts) stays on the host in
    `meta[i]`.  Every item is cached; while the cache is filled the per-item results and the flat buffers coexist."""

    def __init__(self, data: Sequence[dict], prefix: Sequence, num_workers: int = 4, device: Optional[torch.device] = None):
        F = _ops()
        allowed = (N.LoadImaged, N.AsChannelFirstd, F.ConvertToMultiChannelBasedOnBratsClassesd, F.WholeTumorTCGA,
                   F.SelectChanneld, S.Spacingd, S.Orientationd, S.SpacingOrientationd, S.CenterSpatialCropd)
        for t in prefix:
            if not isinstance(t, allowed):
                raise NotImplementedError(f"DeviceCache: {_name(t)} is not a supported prefix transform "
                                          f"(supported: {', '.join(a.__name__ for a in allowed)})")
        Fn.require_cuda()
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        prefix = fill_steps(prefix)

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
         "SaltAndPepper": 8, "RandGibbsNoised": 5, "RandKSpaceSpikeNoised": 6}
# the augmentation transforms, accepted with kspace_augment=True; each takes the slot of the one it cannot share a tail with
_AUGMENT = {"RandGibbsNoised": "RandFourierDiskMaskd", "RandKSpaceSpikeNoised": "RandPlaneWaves_ellipsoid"}


class TrainStage:
    """The random tail of the 127 scripts' training Compose on a DeviceCache, per batch.  Supported, in this order, each
    optional:

        mvtb.spatial.RandSpatialCropd(random_size=False) -> RandFlipd      over all cached keys
        mvtb.intensity.NormalizeIntensityd(nonzero=True, channel_wise=True) -> RandScaleIntensityd -> RandShiftIntensityd,
            or IntensityPrologued (scale / shift need the normalisation in front of them)
        filters_and_operators.RandFourierDiskMaskd(inside_off=False) -> RandPlaneWaves_ellipsoid -> WrapArtifactd
            -> SaltAndPepper(prob=1, rng="philox" or "philox-sparse"; rng="torch" with torch_generator=True)

    with filters_and_operators.SelectChanneld anywhere and MONAI's ToTensord as a no-op.  The intensity and k-space
    transforms act on one key (the image).  A SelectChanneld in front of the salt-and-pepper is folded into the gather;
    one behind it (the select takes its min / max over all channels) is applied to the result.

    Without a RandSpatialCropd the stage gathers whole entries, so every sample of a batch needs the same cached shape
    (ValueError otherwise).  On a cache whose prefix ends in CenterSpatialCropd this is the scripts' validation tail
    (SelectChanneld -> NormalizeIntensityd -> disk -> plane wave -> wrap -> salt-and-pepper), and loader(batch_size,
    shuffle=False) visits the samples in the validation DataLoader's order.

    `draw(indices)` (host only) returns a record of every random parameter; `apply(record)` returns the batch as CUDA
    float32 tensors (B, C, *roi) per key, plus per-sample lists of the meta dicts.  `loader(...)` yields
    apply(draw(batch)) in the order of a DataLoader on the same sampler.  `stage[i]` is draw([i]): a small host object
    that a forked DataLoader worker can produce (`DataLoader(stage, batch_size, collate_fn=list)` and apply on the
    collated list in the main process); each worker then draws from its own copy of the transforms, and MONAI's
    per-worker reseeding (worker_init_fn) changes the draws, as it does for the reference.  The copies include the
    salt-and-pepper `offset`, which starts equal in every worker and never advances in the main process: give each worker
    its own `sp.seed` in worker_init_fn (records carry the seed they were drawn with), or the workers' salt-and-pepper
    patterns repeat.

    SaltAndPepper(rng="torch") draws its uniforms from torch's process-wide CPU generator, as the reference does; a stage
    takes it only with `torch_generator=True`, since consuming that generator is a side effect.  Per-sample torch.rand calls
    consume the stream one after another, so `draw` records the generator's state at its first sample (the others continue
    that stream) and advances the generator on the host by jump-ahead, once, by what all its samples' torch.rand would take:
    a batch leaves it where per-sample calls would.  `apply` makes the uniforms on the device from the recorded states
    (mvtb_mt19937_uniform_f32) and selects with them.  In forked DataLoader workers each worker's generator is seeded by
    torch per worker, as for the reference.

    `kspace_augment=True` also accepts the k-space augmentation of the 20_Gibbs_filters and 30_augmentation scripts, on
    the image key:

        filters_and_operators.RandGibbsNoised(as_tensor_output=True)       in the disk's slot (1 to 8 channels)
        filters_and_operators.RandKSpaceSpikeNoised(intensity_ranges={image: ...}, as_tensor_output=True)
                                                                            in the plane wave's slot; channel_wise and
                                                                            common_sampling either way

    Without the keyword both are refused, as before.  The Gibbs transform cannot share a tail with the disk, nor the spikes
    with the plane wave (a chain descriptor holds one mask and one spike source); the spikes need a given intensity range
    (the default one is computed from the image's spectrum, which `draw` cannot see), and no SelectChanneld on the image
    between them and the salt-and-pepper (their draws are per channel).  `draw` calls the objects' own `_randomize`
    sample after sample: the Gibbs gate and alpha, the spikes' global gate, the common_sampling reseed and the inner
    per-channel gates, locations and intensities, on a shape-only stand-in of the (C, *roi) image.  `apply` builds one
    chain descriptor per channel volume and runs the k-space chain only on the samples with something to do (a gate on,
    or a WrapArtifactd in the tail): those are compacted, chained with their intensity map, and put back; the others
    get the intensity map alone and are what the per-sample drop-ins leave, bit for bit.  The salt-and-pepper then
    runs over the whole batch with the counters per-sample calls use."""

    def __init__(self, cache: DeviceCache, transforms: Sequence, torch_generator: bool = False, kspace_augment: bool = False):
        F = _ops()
        self.cache = cache
        self.tail = list(transforms)
        self.torch_generator = bool(torch_generator)
        self.kspace_augment = bool(kspace_augment)
        cached = set(cache.keys)
        ch = {k: list(range(cache.channels[k])) for k in cache.keys}     # current channel map per key (into the cache)
        self.pre_select = None                          # channel maps at the salt-and-pepper (what the gather reads)
        self.post_select: Dict[str, List[int]] = {}     # channels of the result kept after the salt-and-pepper
        self.crop = self.flip = self.norm = self.scale = self.shift = self.disk = self.wave = self.wrap = self.sp = None
        self.gibbs = self.kspike = None
        kspike_ch = None                                # the image's channel map where the spikes are drawn
        self.image_key = None
        last = -1
        seen = set()
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
            if self.kspace_augment:
                supported.update(RandGibbsNoised=F.RandGibbsNoised, RandKSpaceSpikeNoised=F.RandKSpaceSpikeNoised)
            elif n in _AUGMENT:
                raise NotImplementedError(f"TrainStage: {n} is not supported; pass kspace_augment=True to run it in the stage")
            if n not in supported or not isinstance(t, supported[n]):
                raise NotImplementedError(f"TrainStage: {n} is not supported")
            for a, b in _AUGMENT.items():
                if (n == a and b in seen) or (n == b and a in seen):
                    raise NotImplementedError(f"TrainStage: {a} and {b} in one tail; a chain descriptor holds one "
                                              + ("mask" if a == "RandGibbsNoised" else "spike source"))
            seen.add(n)
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
            elif n == "RandGibbsNoised":
                if not t.as_tensor_output:
                    raise NotImplementedError("TrainStage: RandGibbsNoised(as_tensor_output=False) returns numpy arrays")
                self.gibbs = t
            elif n == "RandKSpaceSpikeNoised":
                inner = t.transforms[keys[0]]
                if not t.as_tensor_output:
                    raise NotImplementedError("TrainStage: RandKSpaceSpikeNoised(as_tensor_output=False) returns numpy arrays")
                if inner.intensity_range is None:
                    raise NotImplementedError("TrainStage: RandKSpaceSpikeNoised without intensity_ranges for the image key; the "
                                              "default range comes from the image's spectrum, which draw() cannot see")
                rng = inner.intensity_range
                if isinstance(rng[0], _SeqABC) and len(rng) != len(ch[keys[0]]):
                    raise ValueError(f"TrainStage: RandKSpaceSpikeNoised has {len(rng)} intensity ranges for an image of "
                                     f"{len(ch[keys[0]])} channels; one per channel is needed")
                self.kspike, kspike_ch = t, list(ch[keys[0]])
            else:
                if t.rng not in ("philox", "philox-sparse") and not (t.rng == "torch" and self.torch_generator):
                    raise NotImplementedError(f"TrainStage: SaltAndPepper(rng={t.rng!r}) draws from torch's global generator; "
                                              "pass torch_generator=True to let the stage consume it, or use rng='philox' "
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
        if self.kspike is not None and kspike_ch != self.pre_select[self.image_key]:
            raise NotImplementedError("TrainStage: a SelectChanneld on the image between RandKSpaceSpikeNoised and the "
                                      "salt-and-pepper (or the end); the spikes are drawn per channel of the image they see")
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
                               "r", "spike_gate", "spike_idx", "sp_gate", "sp_seed", "sp_offset", "sp_blocks", "sp_state")}
        if self.gibbs is not None:
            rec.update(gibbs_gate=[], alpha=[])
        if self.kspike is not None:
            rec.update(kspike_gate=[], kspikes=[])
        first = self.crop.keys[0] if self.crop is not None else self.cache.keys[0]
        mt = None                                       # rng="torch": the generator at the draw's start, and the draws taken
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
                elif t is self.gibbs:
                    t._randomize(None)                  # the gate, then alpha, which is always drawn
                    rec["gibbs_gate"].append(bool(t._do_transform))
                    rec["alpha"].append(float(t.sampled_alpha))
                elif t is self.kspike:
                    gate, spikes = self._draw_kspikes(t, size)
                    rec["kspike_gate"].append(gate)
                    rec["kspikes"].append(spikes)
                elif t is self.sp:
                    t.randomize(None)
                    n = len(self.pre_select[self.image_key]) * math.prod(size)
                    if t.rng == "torch":                # prob=1: every sample draws torch.rand(n)
                        if torch.get_default_dtype() != torch.float32:
                            raise RuntimeError("TrainStage: SaltAndPepper(rng='torch') draws float32 uniforms; torch.rand "
                                               f"would draw {torch.get_default_dtype()} under this default dtype")
                        # the samples' streams follow each other: the first records its start state, the others continue it
                        if mt is None:
                            mt = [Fn.mt19937_take(0, 1)[0], 0]
                            rec["sp_state"].append(mt[0])
                        else:
                            rec["sp_state"].append(None)
                        mt[1] += n
                    blocks = (n + 255) // 256 if t.rng == "philox-sparse" else (n + 3) // 4
                    rec["sp_gate"].append(bool(t._do_transform))
                    rec["sp_seed"].append(int(t.seed))
                    rec["sp_offset"].append(int(t.offset))
                    rec["sp_blocks"].append(blocks)
                    if t._do_transform and t.rng != "torch":
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
        if mt is not None:                              # one host jump for the whole draw
            st = torch.get_rng_state()
            words, nx, lf = Fn.mt19937_advance(mt[0][:624].view(np.uint32).copy(), int(mt[0][624]), int(mt[0][625]), mt[1])
            torch.set_rng_state(Fn.mt19937_pack(words, nx, lf, st))
        return rec

    def _draw_kspikes(self, t, size):
        """RandKSpaceSpikeNoised's draws for one sample, as its __call__ makes them: the global gate, the common_sampling
        reseed, then the inner transform's per-channel draws on a (C, *size) stand-in of the image (shape only, no memory).
        Returns the gate and, when it is on, one (fftshift-ed (x, y, z), log-intensity) or None per channel."""
        t.randomize(None)
        if t.common_sampling:
            for k in t.keys:
                t.transforms[k].set_random_state(t.common_seed)
        if not t._do_transform:
            return False, None
        inner = t.transforms[self.image_key]
        img = np.broadcast_to(np.zeros((), np.uint8), (len(self.pre_select[self.image_key]),) + tuple(size))
        inner.sampled_k_intensity, inner.sampled_locs = [], []
        inner._randomize(img, inner._make_sequence(img))
        spikes = [None] * img.shape[0]
        for loc, v in zip(inner.sampled_locs, inner.sampled_k_intensity):
            spikes[loc[0]] = (tuple(int(i) for i in loc[1:]), float(v))
        return True, tuple(spikes)

    def __len__(self) -> int:
        return len(self.cache)

    def __getitem__(self, i: int) -> dict:
        return self.draw([i])

    # ---- device side
    def _desc(self, roi, mask, spikes):
        """mask: None, ("disk", r) or ("gibbs", alpha); spikes: ((fftshift-ed (x, y, z), log-intensity), ...)"""
        key = (roi, mask, spikes)
        d = self._descs.get(key)
        if d is None:
            kw = {}
            if mask is not None and mask[0] == "disk":
                kw.update(mask_kind=_lib.MASK_DISK, mask_ndim=3, mask_thresh=host.disk_threshold(mask[1], roi))
            elif mask is not None:
                kw.update(mask_kind=_lib.MASK_CENTRED, mask_ndim=3, mask_thresh=host.gibbs_threshold(mask[1], roi))
            if spikes:
                kw["spikes"] = [(idx, host.exp_f32(v)) for idx, v in spikes]
            if self.wrap is not None:
                kw["wrap_alpha"] = float(self.wrap.transform.alpha)
            d = host.make_desc(**kw)
            if len(self._descs) >= 4096:
                self._descs.clear()
            self._descs[key] = d
        return d

    def _sample_descs(self, rec, b, roi, c_img):
        """The chain descriptors of sample b, one per channel volume, and whether the chain has anything to do on it"""
        mask = None
        if self.disk is not None and rec["disk_gate"][b]:
            mask = ("disk", rec["r"][b])
        elif self.gibbs is not None and rec["gibbs_gate"][b]:
            mask = ("gibbs", rec["alpha"][b])
        spikes = [()] * c_img
        if self.wave is not None and rec["spike_idx"][b] is not None:
            spikes = [((rec["spike_idx"][b], self.wave.intensity_value),)] * c_img
        elif self.kspike is not None and rec["kspikes"][b] is not None:
            spikes = [() if s is None else (s,) for s in rec["kspikes"][b]]
        busy = mask is not None or any(spikes) or self.wrap is not None
        return [self._desc(roi, mask, s) for s in spikes], busy

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
        torch_sp = self.sp is not None and self.sp.rng == "torch"
        runs = [b for b in range(B) if rec["sp_state"][b] is not None] if torch_sp else []
        n_mt = len(runs) * _lib.MT_STATE_WORDS
        descs, gated = None, None                       # kspace_augment: the samples the chain runs on, when not all
        if self.gibbs is not None or self.kspike is not None:
            per = [self._sample_descs(rec, b, roi, c_img) for b in range(B)]
            descs = [d for ds, busy in per if busy for d in ds]
            if not all(busy for _, busy in per):
                gated = [b for b in range(B) if per[b][1]]
        o_g = n_int + n_flt + n_mt + (n_int + n_flt + n_mt) % 2        # int64 indices at an 8-byte boundary
        pinned = torch.empty(o_g + 2 * len(gated) if gated else n_int + n_flt + n_mt, dtype=torch.int32, pin_memory=True)
        pv = pinned.numpy()
        pv[:B] = idx
        pv[B:4 * B] = starts.reshape(-1)
        pv[4 * B:5 * B] = rec["flip"]
        if has_int:
            sc = np.ones(B, dtype=np.float32) if self.scale is None else \
                np.where(rec["scale_gate"], 1.0 + np.asarray(rec["factor"], dtype=np.float64), 1.0).astype(np.float32)
            sh = np.zeros(B, dtype=np.float32) if self.shift is None else \
                np.where(rec["shift_gate"], np.asarray(rec["offset"], dtype=np.float64), 0.0).astype(np.float32)
            fv = pv[n_int:n_int + n_flt].view(np.float32)
            fv[:B * c_img] = np.repeat(sc, c_img)
            fv[B * c_img:] = np.repeat(sh, c_img)
        if torch_sp:
            pv[n_int + n_flt:n_int + n_flt + n_mt] = np.stack([rec["sp_state"][b] for b in runs]).reshape(-1)
        if gated:
            pv[o_g:].view(np.int64)[:] = gated
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
                shift_d = up[n_int + B * c_img:n_int + n_flt].view(torch.float32)
                abt = Fn.intensity_coeffs(x, B * c_img, scale=scale_d, shift=shift_d)
            if self.disk or self.wave or self.wrap or self.sp or self.gibbs is not None or self.kspike is not None:
                states = (runs, up[n_int + n_flt:n_int + n_flt + n_mt].view(len(runs), _lib.MT_STATE_WORDS)) if torch_sp else None
                if gated is None:
                    x = self._chain(x, rec, roi, B, c_img, abt, states, descs)
                else:
                    x = self._chain_gated(x, rec, B, c_img, abt, states, descs, up[o_g:].view(torch.int64) if gated else None)
            elif abt is not None:
                x = Fn.intensity_affine(x, abt, out=x)
            out[ik] = x
        for k, chans in self.post_select.items():
            out[k] = out[k][:, chans].contiguous()
        for mk in (cache.meta[0].keys() if cache.meta else ()):
            out[mk] = [cache.meta[i][mk] for i in rec["index"]]
        return out

    def _chain(self, x, rec, roi, B, c_img, abt, states=None, descs=None):
        if descs is None:
            descs = [d for b in range(B) for d in self._sample_descs(rec, b, roi, c_img)[0]]
        descs = host.desc_array(descs)
        sp = self.sp
        if sp is None or not any(rec["sp_gate"]):
            return Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, out=x)
        if states is None and sp.rng == "philox-sparse" and self._sp_contiguous(rec, B):
            off, blocks, seed = rec["sp_offset"], rec["sp_blocks"], rec["sp_seed"]
            return Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, sp=(float(sp.p), seed[0], off[0], blocks[0]), vols_per_sample=c_img,
                                      out=x)[0]
        y, mm = Fn.kspace_chain_ex(x, 3, descs, pre_abt=abt, want_minmax=True, vols_per_sample=c_img, out=x)
        return self._salt_pepper(y, mm, rec, B, states)

    def _chain_gated(self, x, rec, B, c_img, abt, states, descs, g):
        """The k-space chain on the samples `g` (int64 indices on the device; None: no sample) alone: compacted, chained with
        their slice of the intensity map, put back.  The others get the intensity map alone, as the per-sample drop-ins
        pass them through without an FFT.  The salt-and-pepper then runs over the whole batch."""
        if g is not None:
            xg = x.index_select(0, g)
            abt_g = None if abt is None else abt.view(B, c_img, 3).index_select(0, g).view(-1, 3)
        if abt is not None:
            Fn.intensity_affine(x, abt, out=x)
        if g is not None:
            x.index_copy_(0, g, Fn.kspace_chain_ex(xg, 3, host.desc_array(descs), pre_abt=abt_g, out=xg))
        if self.sp is None or not any(rec["sp_gate"]):
            return x
        return self._salt_pepper(x, Fn.minmax(x, B), rec, B, states)

    @staticmethod
    def _sp_contiguous(rec, B):
        """do the batch's salt-and-pepper counters follow each other as per-sample calls would have used them?"""
        off, blocks, seed = rec["sp_offset"], rec["sp_blocks"], rec["sp_seed"]
        return all(rec["sp_gate"]) and all(off[b] == off[0] + b * blocks[0] and blocks[b] == blocks[0] and seed[b] == seed[0]
                                           for b in range(B))

    def _salt_pepper(self, y, mm, rec, B, states=None):
        """The select on the batch y (min / max per sample in mm) with the recorded counters or torch states"""
        sp = self.sp
        off, blocks, seed = rec["sp_offset"], rec["sp_blocks"], rec["sp_seed"]
        # one select call when the batch's counters follow each other as per-sample calls would have used them
        contiguous = self._sp_contiguous(rec, B)
        sparse = sp.rng == "philox-sparse"
        if states is not None:                          # rng="torch": the uniforms of every sample's torch.rand
            starts, st = states                         # sample starts[j] .. starts[j + 1] - 1 continue one stream
            n = y[0].numel()
            bounds = starts + [B]
            lens = {bounds[j + 1] - bounds[j] for j in range(len(starts))}
            u = torch.empty_like(y)
            if len(lens) == 1:                          # runs of equal length: one call, a segment per run
                Fn.mt19937_uniform(st, lens.pop() * n, out=u.view(len(starts), -1))
            else:
                for j in range(len(starts)):
                    Fn.mt19937_uniform(st[j:j + 1], (bounds[j + 1] - bounds[j]) * n, out=u[bounds[j]:bounds[j + 1]].view(1, -1))
            return Fn.salt_pepper(y, float(sp.p), u=u, n_samples=B, mm=mm, out=y)
        # philox-sparse: the standalone select numbers a batch's spans per sample, not by the offsets per-sample calls use, so
        # it runs sample by sample (the stride that fixes that is only in the chain's fused select)
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
        if self.torch_generator:
            # a DataLoader draws its base seed before the sampler's: the generator then ends an epoch where one leaves it
            torch.empty((), dtype=torch.int64).random_(generator=generator)
        sampler = RandomSampler(src, generator=generator) if shuffle else SequentialSampler(src)
        for batch in BatchSampler(sampler, batch_size, drop_last):
            yield self.apply(self.draw(batch))
