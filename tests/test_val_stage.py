"""Validation on the device without a GPU: the prefix transforms DeviceCache accepts (CenterSpatialCropd and WholeTumorTCGA
among them), which CenterSpatialCropd the fill fuses into the resampling gather (spies on mvtb.spatial.resample and the
crop's gather; the fused steps give the arrays and meta dicts of the transforms in sequence), WholeTumorTCGA's numpy
branch, and the validation TrainStage's draws and use of torch's generator for a loader with shuffle=False."""
import shutil
import types

import numpy as np
import pytest
import torch

ROI = (8, 6, 4)
LPS = np.array([[-1.5, 0, 0, 10], [0, -1.2, 0, 20], [0, 0, 2.5, -5], [0, 0, 0, 1]])


class _Reached(Exception):
    pass


def _allowed_prefix():
    import filters_and_operators as F
    from mvtb import nifti as N, spatial as S
    return [N.LoadImaged(["image", "label"]), N.AsChannelFirstd("image"), F.WholeTumorTCGA("label"),
            F.ConvertToMultiChannelBasedOnBratsClassesd("label"), F.SelectChanneld("image", 0),
            S.Spacingd(["image", "label"], (1.0, 1.5, 2.0)), S.Orientationd(["image", "label"], axcodes="RAS"),
            S.SpacingOrientationd(["image", "label"], (1.0, 1.5, 2.0), axcodes="RAS"),
            S.CenterSpatialCropd(["image", "label"], list(ROI))]


def test_cache_accepts_center_crop_and_whole_tumor(monkeypatch):
    from mvtb import functional as Fn
    from mvtb.train_stage import DeviceCache

    def reached():
        raise _Reached
    monkeypatch.setattr(Fn, "require_cuda", reached)      # the prefix check passed; stop before the device is needed
    for t in _allowed_prefix():
        with pytest.raises(_Reached):
            DeviceCache([{"image": "x.nii", "label": "y.nii"}], [t])
    with pytest.raises(_Reached):
        DeviceCache([{"image": "x.nii", "label": "y.nii"}], _allowed_prefix())


def _refused_prefix():
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    return {"rand_crop": S.RandSpatialCropd(["image", "label"], list(ROI), random_size=False),
            "flip": S.RandFlipd(["image", "label"], prob=0.5), "crop_flip": S.CropFlipd(["image", "label"], list(ROI)),
            "normalize": I.NormalizeIntensityd("image", nonzero=True, channel_wise=True),
            "disk": F.RandFourierDiskMaskd("image", r=8.0), "sp": F.SaltAndPepper(0.05, "image", rng="philox-sparse"),
            "gibbs": F.RandGibbsNoised("image", prob=1.0), "slices": F.SegmentationSlicesd(["image", "label"], seed=0),
            "other": types.SimpleNamespace(keys=["image"])}


@pytest.mark.parametrize("case", sorted(_refused_prefix()))
def test_cache_still_refuses_the_rest(case):
    from mvtb.train_stage import DeviceCache
    with pytest.raises(NotImplementedError, match="WholeTumorTCGA.*CenterSpatialCropd"):
        DeviceCache([{"image": "x.nii"}], _allowed_prefix()[:2] + [_refused_prefix()[case]])


# ---------------------------------------------------------------------------------------------------------- fused crop

def _fill_cases():
    from mvtb import spatial as S
    keys = ["image", "label"]
    sp = lambda k=keys: S.Spacingd(k, (1.0, 1.5, 2.0), mode=("bilinear", "nearest")[:len(k)])    # noqa: E731
    orient = lambda k=keys: S.Orientationd(k, axcodes="RAS")                                      # noqa: E731
    both = lambda k=keys: S.SpacingOrientationd(k, (1.0, 1.5, 2.0), axcodes="RAS",               # noqa: E731
                                                mode=("bilinear", "nearest")[:len(k)])
    crop = lambda k=keys, roi=ROI: S.CenterSpatialCropd(k, list(roi))                              # noqa: E731
    # (prefix, the (resampling transform, crop) positions in the prefix of each pair that is fused)
    return {
        "spacing_orientation": ([both(), crop()], [(0, 1)]),
        "spacing": ([sp(), crop()], [(0, 1)]),
        "orientation": ([orient(), crop()], [(0, 1)]),
        "spacing_then_orientation": ([sp(), orient(), crop()], [(1, 2)]),
        "crop_one_key": ([both(), crop(["label"])], [(0, 1)]),
        "crop_roi_larger": ([both(), crop(roi=(64, 6, 40))], [(0, 1)]),
        "crop_other_key": ([both(["image"]), crop()], []),
        "crop_before": ([crop(), both()], []),
        "crop_after_select": ([both(), _select(), crop()], []),
        "two_crops": ([both(), crop(), crop(roi=(4, 4, 4))], [(0, 1)]),
        "crop_twice_resampled": ([sp(), crop(), orient(), crop(roi=(4, 4, 4))], [(0, 1), (2, 3)]),
    }


def _select():
    import filters_and_operators as F
    return F.SelectChanneld("image", 0)


def _item(shape=(18, 14, 9)):
    rng = np.random.RandomState(0)
    return {"image": rng.standard_normal((2,) + shape).astype(np.float32),
            "label": (rng.rand(3, *shape) < 0.3).astype(np.float32),
            "image_meta_dict": {"affine": LPS.copy()}, "label_meta_dict": {"affine": LPS.copy()}}


class _Spies:
    """mvtb.spatial.resample and crop_flip without a device: resample writes each output voxel's grid coordinates (and the
    mode), the crop slices; both record their calls."""

    def __init__(self, monkeypatch):
        from mvtb import spatial as S
        self.resamples, self.crops = [], []
        monkeypatch.setattr(S, "resample", self.resample)
        monkeypatch.setattr(S, "crop_flip", self.crop_flip)

    def resample(self, x, p, mode="bilinear", window=None, flip_axes_mask=0, **kw):
        self.resamples.append((tuple(x.shape), p.shape, mode, window))
        assert flip_axes_mask == 0
        start, size = ((0, 0, 0), p.shape) if window is None else window
        g = np.meshgrid(*[np.arange(s, s + n) for s, n in zip(start, size)], indexing="ij")
        v = (g[0] * 1000 + g[1]) * 1000 + g[2] + (0.5 if mode == "nearest" else 0.0)
        return np.stack([v + 1e7 * c for c in range(x.shape[0])]).astype(np.float64)

    def crop_flip(self, x, start, size, flip_axes_mask=0):
        self.crops.append((tuple(x.shape), tuple(start), tuple(size)))
        assert flip_axes_mask == 0
        return x[:, start[0]:start[0] + size[0], start[1]:start[1] + size[1], start[2]:start[2] + size[2]]


def _run(steps, d):
    for t in steps:
        d = t(d)
    return d


@pytest.mark.parametrize("case", sorted(_fill_cases()))
def test_fill_fuses_a_center_crop_right_behind_a_resample(case, monkeypatch):
    from mvtb import geometry as G
    from mvtb.train_stage import ResampleCenterCrop, fill_steps
    prefix, fused = _fill_cases()[case]
    steps = fill_steps(prefix)
    # the fused pairs, and every other transform as itself, in order
    want, j = [], 0
    pairs = dict(fused)
    while j < len(prefix):
        if j in pairs:
            want.append((prefix[j], prefix[pairs[j]]))
            j = pairs[j] + 1
        else:
            want.append(prefix[j])
            j += 1
    assert len(steps) == len(want)
    for s, w in zip(steps, want):
        if isinstance(w, tuple):
            assert isinstance(s, ResampleCenterCrop) and s.resample is w[0] and s.crop is w[1]
        else:
            assert s is w
    spies = _Spies(monkeypatch)
    got = _run(steps, _item())
    n_fused_crop_keys = sum(len(prefix[c].keys) for _, c in fused)
    n_crop_calls = len(spies.crops)
    n_resample_calls = len(spies.resamples)
    spies.resamples.clear()
    spies.crops.clear()
    ref = _run(prefix, _item())                           # the transforms one after another
    # every fused key is one windowed gather in place of a gather and a crop
    assert n_crop_calls == len(spies.crops) - n_fused_crop_keys
    assert n_resample_calls == len(spies.resamples)
    windows = [w for (_, _, _, w) in spies.resamples]
    assert windows == [None] * len(windows)
    assert set(got) == set(ref)
    for k in ref:
        if k.endswith("_meta_dict"):
            assert got[k].keys() == ref[k].keys() and np.array_equal(got[k]["affine"], ref[k]["affine"]), k
        else:
            assert got[k].shape == ref[k].shape and np.array_equal(got[k], ref[k]), k
    if case == "crop_roi_larger":                         # MONAI's size where the roi is larger than the volume
        grid = G.plan(LPS, (18, 14, 9), (1.0, 1.5, 2.0), axcodes="RAS").shape
        assert got["image"].shape[1:] == tuple(min(r, n) for r, n in zip((64, 6, 40), grid)) != (64, 6, 40)


def test_fused_windows_are_the_center_crop(monkeypatch):
    from mvtb import geometry as G, spatial as S
    from mvtb.train_stage import fill_steps
    both = S.SpacingOrientationd(["image", "label"], (1.0, 1.5, 2.0), axcodes="RAS", mode=("bilinear", "nearest"))
    spies = _Spies(monkeypatch)
    _run(fill_steps([both, S.CenterSpatialCropd(["label"], list(ROI))]), _item())
    p = G.plan(LPS, (18, 14, 9), (1.0, 1.5, 2.0), axcodes="RAS")
    assert spies.resamples == [((2, 18, 14, 9), p.shape, "bilinear", None),
                               ((3, 18, 14, 9), p.shape, "nearest", S.center_window(p.shape, ROI))]
    assert spies.crops == []


def test_fused_crop_keeps_missing_key_rules(monkeypatch):
    from mvtb import spatial as S
    from mvtb.train_stage import fill_steps
    _Spies(monkeypatch)
    d = _item()
    del d["label"]
    steps = fill_steps([S.SpacingOrientationd(["image", "label"], (1.0, 1.5, 2.0), axcodes="RAS", allow_missing_keys=True),
                        S.CenterSpatialCropd(["image", "label"], list(ROI))])
    with pytest.raises(KeyError):
        _run(steps, d)
    steps = fill_steps([S.SpacingOrientationd(["image", "label"], (1.0, 1.5, 2.0), axcodes="RAS", allow_missing_keys=True),
                        S.CenterSpatialCropd(["image", "label"], list(ROI), allow_missing_keys=True)])
    assert _run(steps, d)["image"].shape[1:] == ROI
    with pytest.raises(ValueError, match="not all among"):
        S.Spacingd("image", (1.0, 1.0, 1.0)).resample_crop(_item(), S.CenterSpatialCropd("label", list(ROI)))


# ------------------------------------------------------------------------------------------------------ WholeTumorTCGA

def test_whole_tumor_numpy_branch_is_unchanged():
    import filters_and_operators as F
    rng = np.random.RandomState(4)
    for lab in (rng.randint(-2, 5, size=(9, 7, 5)).astype(np.int16), rng.randint(0, 3, size=(6, 5, 4)).astype(np.uint8),
                np.where(rng.rand(5, 4, 3) < 0.5, 0.0, rng.standard_normal((5, 4, 3))), np.array([0, 2, 4])):
        out = F.WholeTumorTCGA("label")({"label": lab, "image": "kept"})
        want = (lab != 0)[None, :].astype(np.float32)
        assert isinstance(out["label"], np.ndarray) and out["label"].dtype == np.float32
        assert out["label"].shape == (1,) + lab.shape and np.array_equal(out["label"], want)
        assert out["image"] == "kept"
    with pytest.raises(KeyError):
        F.WholeTumorTCGA("label")({"image": 0})
    assert F.WholeTumorTCGA("label", allow_missing_keys=True)({"image": 0}) == {"image": 0}


# ---------------------------------------------------------------------------------------------------- validation tail

@pytest.fixture(scope="module")
def L():
    if shutil.which("g++") is None:
        pytest.skip("needs g++ for the emulator build")
    from cuemu import emu
    return emu.lib()


def _val_tail(rng):
    import filters_and_operators as F
    from mvtb import intensity as I
    t = [F.SelectChanneld("image", 0), I.NormalizeIntensityd("image", nonzero=True, channel_wise=True),
         F.RandFourierDiskMaskd("image", r=3.0, inside_off=False, prob=1.0),
         F.RandPlaneWaves_ellipsoid("image", 3, 2, 1, intensity_value=8, prob=1.0), F.WrapArtifactd("image", alpha=0.5),
         F.SaltAndPepper(0.05, "image", prob=1.0, rng=rng, seed=3)]
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=10 + k)
    return t


def test_validation_draw_gathers_whole_entries():
    from mvtb.train_stage import TrainStage
    from test_train_stage import _fake_cache
    stage = TrainStage(_fake_cache([ROI] * 5), _val_tail("philox-sparse"))
    assert stage.crop is None and stage.flip is None and stage.pre_select["image"] == [0]
    rec = stage.draw([0, 1, 2])
    assert rec["start"] == [(0, 0, 0)] * 3 and rec["size"] == [ROI] * 3 and rec["flip"] == [0] * 3
    n = (ROI[0] * ROI[1] * ROI[2] + 255) // 256
    assert rec["sp_offset"] == [0, n, 2 * n] and stage.sp.offset == 3 * n


def test_validation_loader_consumes_the_generator_as_a_dataloader(L, monkeypatch):
    """shuffle=False: a DataLoader still draws its base seed, then the per-sample torch.rand calls follow in order"""
    from torch.utils.data import DataLoader
    from mvtb import _lib
    from mvtb.train_stage import TrainStage
    from test_train_stage import _fake_cache
    monkeypatch.setattr(_lib, "_lib", L)
    n_vox = ROI[0] * ROI[1] * ROI[2]
    for n_items, bs in ((5, 2), (6, 5), (3, 1)):
        stage = TrainStage(_fake_cache([ROI] * n_items), _val_tail("torch"), torch_generator=True)
        monkeypatch.setattr(stage, "apply", lambda rec: rec)
        torch.manual_seed(n_items)
        got = [r["index"] for r in stage.loader(bs, shuffle=False)]
        got_state = torch.get_rng_state()
        torch.manual_seed(n_items)
        want = []
        for batch in DataLoader(range(n_items), batch_size=bs, shuffle=False, num_workers=0, collate_fn=list):
            for _ in batch:
                torch.rand(1 * n_vox)                     # the per-sample SaltAndPepper: one channel of the entry
            want.append(batch)
        assert got == want
        assert torch.equal(torch.get_rng_state(), got_state), (n_items, bs)
