"""The training loader's batch stage without a GPU: the ragged-cache crop + flip gather through the DEBUG emulator against
numpy slicing, the C entry's argument checks, TrainStage.draw against the same seeded transforms randomized one sample at
a time, and the transforms and orders the stage refuses."""
import ctypes as C
import shutil
import types

import numpy as np
import pytest

emu_only = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++ for the emulator build")

SHAPES = [(9, 7, 8), (6, 10, 5), (8, 6, 11)]         # three entries of different shapes
C_IN = 3
ROI = (4, 5, 5)


def _cache_arrays():
    rng = np.random.RandomState(3)
    vols = [rng.standard_normal((C_IN,) + s).astype(np.float32) for s in SHAPES]
    sizes = [v.size for v in vols]
    offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    return vols, np.concatenate([v.ravel() for v in vols]), offsets, np.array(SHAPES, dtype=np.int32).reshape(-1)


def _gather(L, flat, offsets, shapes, entries, starts, flips, channels, roi=ROI):
    from cuemu import emu
    B_ = len(entries)
    n_out = C_IN if channels is None else len(channels)
    out = np.full((B_, n_out) + roi, -7.0, dtype=np.float32)
    e = np.asarray(entries, dtype=np.int32)
    st = np.asarray(starts, dtype=np.int32).reshape(-1)
    fl = np.asarray(flips, dtype=np.int32)
    ch = None if channels is None else (C.c_int32 * len(channels))(*channels)
    rc = L.mvtb_crop_flip_gather_f32(emu.ptr(flat), emu.ptr(out), B_, n_out, emu.ptr(offsets), emu.ptr(shapes), C_IN, ch,
                                     (C.c_int32 * 3)(*roi), emu.ptr(e), emu.ptr(st), emu.ptr(fl), None)
    return rc, out


def _want(vol, start, flip, channels, roi=ROI):
    x = vol if channels is None else vol[list(channels)]
    x = x[:, start[0]:start[0] + roi[0], start[1]:start[1] + roi[1], start[2]:start[2] + roi[2]]
    axes = tuple(1 + a for a in range(3) if flip >> a & 1)
    return np.flip(x, axes) if axes else x


@emu_only
@pytest.mark.parametrize("channels", [None, [2, 0], [1], [2, 1, 0]])
def test_emulated_gather_is_slicing_and_flip(channels):
    from cuemu import emu
    from mvtb import _lib as B
    L = emu.lib()
    vols, flat, offsets, shapes = _cache_arrays()
    entries = [2, 0, 0, 1, 2, 1, 0, 2, 1, 1, 0, 2]                 # repeated and out of order
    starts, flips = [], []
    for b, e in enumerate(entries):
        s = SHAPES[e]
        hi = [s[a] - ROI[a] for a in range(3)]
        # windows at the low border, the high border and in between, on every axis
        starts.append([(0, hi[a], hi[a] // 2)[(b + a) % 3] for a in range(3)])
        flips.append(b % 8)                                        # all 8 masks
    rc, out = _gather(L, flat, offsets, shapes, entries, starts, flips, channels)
    B.check(L, rc)
    for b, e in enumerate(entries):
        assert np.array_equal(out[b], _want(vols[e], starts[b], flips[b], channels)), b


@emu_only
def test_emulated_gather_argument_checks():
    from cuemu import emu
    L = emu.lib()
    vols, flat, offsets, shapes = _cache_arrays()
    e, st, fl = np.zeros(1, np.int32), np.zeros(3, np.int32), np.zeros(1, np.int32)
    out = np.zeros((1, C_IN) + ROI, np.float32)
    i3 = C.c_int32 * 3

    def call(cache=flat, dst=out, n=1, n_out=C_IN, off=offsets, shp=shapes, n_in=C_IN, ch=None, roi=ROI, ent=e, starts=st, flips=fl):
        return L.mvtb_crop_flip_gather_f32(emu.ptr(cache), emu.ptr(dst), n, n_out, emu.ptr(off), emu.ptr(shp), n_in, ch,
                                           None if roi is None else i3(*roi), emu.ptr(ent), emu.ptr(starts), emu.ptr(flips), None)

    assert call() == 0
    for kw in ({"cache": None}, {"dst": None}, {"off": None}, {"shp": None}, {"roi": None}, {"ent": None}, {"starts": None},
               {"flips": None}):
        assert call(**kw) == -1, kw                                                    # null pointers
    assert call(dst=flat) == -1                                                        # in place
    assert call(n=-1) == -1 and call(n_out=-1) == -1 and call(n_in=-1) == -1           # negative counts
    nine = (C.c_int32 * 9)(*([0] * 9))
    assert call(n_out=9, ch=nine) == -1                                                # more than 8 output channels
    assert call(n_out=2) == -1                                                         # NULL channels = all of them
    assert call(n_out=1, ch=(C.c_int32 * 1)(3)) == -1                                  # channel out of range
    assert call(n_out=1, ch=(C.c_int32 * 1)(-1)) == -1
    for roi in ((0, 5, 5), (4, -1, 5), (4, 5, 0)):
        assert call(roi=roi) == -1                                                     # empty output shape
    assert call(n=0) == 0


def test_gather_symbol_is_exported():
    from mvtb import _lib as B
    assert "mvtb_crop_flip_gather_f32" in B.exported_symbols()


# ----------------------------------------------------------------------------------------------------------------- draw

def _fake_cache(shapes, channels=None):
    """What TrainStage reads of a DeviceCache on the host (no device buffers)."""
    from mvtb.train_stage import DeviceCache
    c = DeviceCache.__new__(DeviceCache)
    c.keys = ["image", "label"]
    c.channels = channels or {"image": 4, "label": 3}
    c.shapes = {k: np.array(shapes, dtype=np.int32) for k in c.keys}
    c.meta = [{} for _ in shapes]
    return c


def _tail(seed, rng="philox-sparse", select_after=False, prologue=False):
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(["image", "label"], roi_size=[12, 10, 6], random_size=False),
         S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0)]
    if not select_after:
        t.append(F.SelectChanneld("image", 0))
    if prologue:
        t.append(I.IntensityPrologued("image", factors=0.1, offsets=0.1, prob=0.5))
    else:
        t += [I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), I.RandScaleIntensityd("image", factors=0.1, prob=0.5),
              I.RandShiftIntensityd("image", offsets=0.1, prob=0.5)]
    t += [F.RandFourierDiskMaskd("image", r=[4.0, 9.0], inside_off=False, prob=0.7),
          F.RandPlaneWaves_ellipsoid("image", 5, 4, 2, intensity_value=12, prob=0.6),
          F.WrapArtifactd("image", alpha=0.5),
          F.SaltAndPepper(0.05, "image", prob=1.0, rng=rng, seed=11)]
    if select_after:
        t.append(F.SelectChanneld("image", 0))
    t.append(type("ToTensord", (), {"keys": ["image", "label"]})())
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 100 + k)
    return t


def _per_sample(tail, shape, c_sp):
    """What each transform's __call__ draws for one sample of spatial `shape` (mvtb.spatial, mvtb.intensity,
    filters_and_operators), without touching the data."""
    from mvtb import intensity as I, spatial as S
    import filters_and_operators as F
    got = {}
    size = shape
    for t in tail:
        if isinstance(t, S.RandSpatialCropd):
            t.randomize(shape)
            got["start"], size = tuple(t._start), tuple(t._size)
        elif isinstance(t, S.RandFlipd):
            t.randomize(None)
            got["flip"] = t._do_transform
        elif isinstance(t, I.IntensityPrologued):
            t.scale.randomize()
            t.shift.randomize()
            got["scale"] = (t.scale._do_transform, t.scale.factor)
            got["shift"] = (t.shift._do_transform, t.shift._offset)
        elif isinstance(t, I.RandScaleIntensityd):
            t.randomize()
            got["scale"] = (t._do_transform, t.factor)
        elif isinstance(t, I.RandShiftIntensityd):
            t.randomize()
            got["shift"] = (t._do_transform, t._offset)
        elif isinstance(t, F.RandFourierDiskMaskd):
            t.randomize()
            got["disk"] = (t._do_transform, t.r)
        elif isinstance(t, F.RandPlaneWaves_ellipsoid):
            t.randomize(None)
            got["spike"] = (t._do_transform, tuple(int(v) for v in t.ellipsoid.sample_ellipsoid(np.empty(size)))
                            if t._do_transform else None)
        elif isinstance(t, F.SaltAndPepper):
            t.randomize(None)
            got["sp"] = (t._do_transform, t.offset)
            n = c_sp * int(np.prod(size))
            if t._do_transform:
                t.offset += (n + 255) // 256 if t.rng == "philox-sparse" else (n + 3) // 4
        elif isinstance(t, F.SelectChanneld):
            pass
    return got


def _states(tail):
    out = []
    for t in tail:
        for o in (t, getattr(t, "scale", None), getattr(t, "shift", None), getattr(t, "ellipsoid", None)):
            if o is not None and "R" in vars(o):
                st = o.R.get_state()
                out.append((st[1].tobytes(), st[2]))
        if hasattr(t, "offset") and isinstance(t.offset, int):
            out.append(t.offset)
    return out


@pytest.mark.parametrize("rng", ["philox-sparse", "philox"])
@pytest.mark.parametrize("select_after", [False, True])
@pytest.mark.parametrize("prologue", [False, True])
def test_draw_matches_per_sample_randomize(rng, select_after, prologue):
    from mvtb.train_stage import TrainStage
    shapes = [(20, 18, 9), (16, 14, 8), (12, 10, 6), (21, 11, 7)]
    cache = _fake_cache(shapes)
    for seed in range(2):
        a, b = _tail(seed, rng, select_after, prologue), _tail(seed, rng, select_after, prologue)
        for t in a + b:                               # the ellipsoids are seeded too (their R draws the spike location)
            if hasattr(t, "ellipsoid"):
                t.ellipsoid.set_random_state(seed=seed + 7)
        stage = TrainStage(cache, a)
        order = [3, 0, 2, 2, 1, 0, 3, 1, 0, 0, 2, 3, 1, 2, 0, 3]      # 16 samples, repeats and out of order
        rec = stage.draw(order[:5])
        rec2 = stage.draw(order[5:])
        rec = {k: rec[k] + rec2[k] for k in rec}
        for j, i in enumerate(order):
            want = _per_sample(b, shapes[i], 4 if select_after else 1)     # the channels the select pass sees
            assert rec["start"][j] == want["start"]
            assert rec["flip"][j] == (1 if want["flip"] else 0)
            assert (rec["scale_gate"][j], rec["factor"][j]) == want["scale"]
            assert (rec["shift_gate"][j], rec["offset"][j]) == want["shift"]
            assert (rec["disk_gate"][j], rec["r"][j]) == want["disk"]
            assert (rec["spike_gate"][j], rec["spike_idx"][j]) == want["spike"]
            assert rec["sp_gate"][j] == want["sp"][0]
            assert rec["sp_offset"][j] == want["sp"][1]
        assert _states(a) == _states(b)


def test_draw_counts_sp_blocks_over_the_channels_the_select_sees():
    from mvtb.train_stage import TrainStage
    cache = _fake_cache([(20, 18, 9)] * 3)
    for after, c in ((False, 1), (True, 4)):
        stage = TrainStage(cache, _tail(0, "philox-sparse", select_after=after))
        rec = stage.draw([0, 1, 2])
        n = c * 12 * 10 * 6
        assert rec["sp_blocks"] == [(n + 255) // 256] * 3
        assert rec["sp_offset"] == [0, (n + 255) // 256, 2 * ((n + 255) // 256)]
        assert stage.sp.offset == 3 * ((n + 255) // 256)
        assert rec["sp_seed"] == [11] * 3                 # records carry the seed they were drawn with


def test_draw_touches_no_cuda(monkeypatch):
    import torch
    from mvtb.train_stage import TrainStage

    def boom(*a, **k):
        raise AssertionError("draw touched CUDA")
    monkeypatch.setattr(torch.cuda, "is_available", boom)
    monkeypatch.setattr(torch.cuda, "current_device", boom)
    stage = TrainStage(_fake_cache([(20, 18, 9)] * 2), _tail(0))
    assert len(stage[1]["index"]) == 1


def _refused():
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    crop = lambda: S.RandSpatialCropd(["image", "label"], roi_size=[12, 10, 6], random_size=False)   # noqa: E731
    flip = lambda: S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0)                          # noqa: E731
    norm = lambda: I.NormalizeIntensityd("image", nonzero=True, channel_wise=True)                   # noqa: E731
    disk = lambda: F.RandFourierDiskMaskd("image", r=8.0, prob=1.0)                                   # noqa: E731
    wave = lambda: F.RandPlaneWaves_ellipsoid("image", 5, 4, 2, intensity_value=12, prob=1.0)         # noqa: E731
    wrap = lambda: F.WrapArtifactd("image", alpha=0.5)                                                # noqa: E731
    sp = lambda **k: F.SaltAndPepper(0.05, "image", rng=k.pop("rng", "philox-sparse"), **k)            # noqa: E731
    return {
        "random_size": [S.RandSpatialCropd(["image", "label"], roi_size=[12, 10, 6], random_size=True)],
        "crop_one_key": [S.RandSpatialCropd(["image"], roi_size=[12, 10, 6], random_size=False)],
        "flip_one_key": [crop(), S.RandFlipd(["image"], prob=0.5)],
        "flip_before_crop": [flip(), crop()],
        "normalize_zero": [crop(), I.NormalizeIntensityd("image", nonzero=False, channel_wise=True)],
        "normalize_global": [crop(), I.NormalizeIntensityd("image", nonzero=True, channel_wise=False)],
        "scale_without_normalize": [crop(), I.RandScaleIntensityd("image", factors=0.1, prob=0.5)],
        "shift_before_scale": [crop(), norm(), I.RandShiftIntensityd("image", 0.1), I.RandScaleIntensityd("image", 0.1)],
        "normalize_twice": [crop(), norm(), norm()],
        "intensity_after_disk": [crop(), disk(), norm()],
        "disk_inside_off": [crop(), F.RandFourierDiskMaskd("image", r=8.0, inside_off=True)],
        "wave_before_disk": [crop(), wave(), disk()],
        "wrap_before_wave": [crop(), wrap(), wave()],
        "sp_before_wrap": [crop(), sp(), wrap()],
        "sp_torch": [crop(), sp(rng="torch")],
        "sp_prob": [crop(), sp(prob=0.5)],
        "chain_two_keys": [crop(), F.RandFourierDiskMaskd(["image", "label"], r=8.0)],
        "two_image_keys": [crop(), norm(), F.RandFourierDiskMaskd("label", r=8.0)],
        "kspace_spike": [crop(), F.RandKSpaceSpikeNoised("image", prob=1.0)],
        "gibbs": [crop(), F.RandGibbsNoised("image", prob=1.0)],
        "center_crop": [S.CenterSpatialCropd(["image", "label"], roi_size=[12, 10, 6])],
        "crop_flip_fused": [S.CropFlipd(["image", "label"], roi_size=[12, 10, 6])],
        "wrap_plain": [crop(), F.WrapArtifact(0.5)],
        "select_unknown_key": [crop(), F.SelectChanneld("mask", 0)],
        "too_many_channels": [crop(), F.SelectChanneld("image", 0)],     # replaced below: a 9-channel cache
        "other": [types.SimpleNamespace(keys=["image"])],
    }


@pytest.mark.parametrize("case", sorted(_refused()))
def test_unsupported_transforms_and_orders_raise(case):
    from mvtb.train_stage import TrainStage
    tail = _refused()[case]
    cache = _fake_cache([(20, 18, 9)] * 2, {"image": 9, "label": 3} if case == "too_many_channels" else None)
    if case == "too_many_channels":
        tail = tail[:1]
    with pytest.raises(NotImplementedError):
        TrainStage(cache, tail)


def test_cache_prefix_is_checked():
    import filters_and_operators as F
    from mvtb.train_stage import DeviceCache
    with pytest.raises(NotImplementedError, match="RandFourierDiskMaskd"):
        DeviceCache([{"image": "x.nii"}], [F.RandFourierDiskMaskd("image", r=8.0)])
