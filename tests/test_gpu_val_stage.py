"""Validation on the GPU: a DeviceCache whose prefix ends in CenterSpatialCropd (the crop fused into the resampling gather)
against the per-file prefix run transform by transform, bit for bit; the scripts' validation tail through TrainStage.loader
(shuffle=False) against the per-sample drop-ins applied to the cached items, with philox-sparse and with torch's generator;
WholeTumorTCGA on the device and a TCGA-style prefix; and volumes smaller than the roi."""
import numpy as np
import pytest
import torch

from oracle import monai_spatial as O, nifti_writer as W

PIXDIM_IN, PIXDIM = (1.5, 1.2, 2.5), (1.0, 1.5, 2.0)
AFFINES = {"identity": np.diag(PIXDIM_IN + (1.0,))[:3],
           "lps": np.array([[-1.5, 0, 0, 10], [0, -1.2, 0, 20], [0, 0, 2.5, -5]]),
           "swapped": np.array([[0, 1.2, 0, 3], [-1.5, 0, 0, 5], [0, 0, 2.5, -7]])}
ROI = (20, 20, 16)                      # inside every resampled grid below (23 voxels or more per axis)


def _files(tmp_path, sform, n=6, tcga=False):
    data = []
    for i in range(n):
        r = np.random.RandomState(i)
        shp = (30 + 4 * (i % 3), 28, 20 + 2 * (i % 2))
        if tcga:
            img = r.standard_normal(shp + (1,)).astype(np.float32)
            lab = r.choice(np.array([0, 1, 2, 4], dtype=np.uint8), size=shp, p=[0.7, 0.1, 0.1, 0.1])
        else:
            img = (r.standard_normal(shp + (4,)) * 100).astype(np.int16)
            lab = r.randint(0, 4, size=shp).astype(np.uint8)
        sfx = ".nii.gz" if i % 2 else ".nii"
        kw = dict(sform=sform, pixdim=PIXDIM_IN, gzip_members=1 if i % 2 else 0, level=1)
        data.append({"image": str(W.write(tmp_path / f"i{i}{sfx}", img, **kw)),
                     "label": str(W.write(tmp_path / f"l{i}{sfx}", lab, **kw))})
    return data


def _prefix(tcga=False, roi=ROI):
    import filters_and_operators as F
    from mvtb import nifti as N, spatial as S
    label = F.WholeTumorTCGA("label") if tcga else F.ConvertToMultiChannelBasedOnBratsClassesd("label")
    return [N.LoadImaged(["image", "label"]), N.AsChannelFirstd("image"), label,
            S.SpacingOrientationd(["image", "label"], PIXDIM, axcodes="RAS", mode=("bilinear", "nearest")),
            S.CenterSpatialCropd(["image", "label"], list(roi))]


def _per_file(item, prefix):
    d = dict(item)
    for t in prefix:
        d = t(d)
    return d


def _assert_cache_equals_per_file(cache, data, tcga=False):
    for i, item in enumerate(data):
        want = _per_file(item, _prefix(tcga))
        got = cache.item(i)
        for k in ("image", "label"):
            assert torch.equal(got[k], want[k]), (i, k)
            gm, wm = got[f"{k}_meta_dict"], want[f"{k}_meta_dict"]
            assert gm.keys() == wm.keys() and np.array_equal(gm["affine"], wm["affine"]), (i, k)
            assert np.array_equal(gm["original_affine"], wm["original_affine"]), (i, k)


@pytest.mark.gpu
@pytest.mark.parametrize("affine", sorted(AFFINES))
def test_gpu_fused_fill_equals_the_prefix_per_file(cuda_device, tmp_path, affine):
    from mvtb.train_stage import DeviceCache, ResampleCenterCrop, fill_steps
    assert isinstance(fill_steps(_prefix())[-1], ResampleCenterCrop)
    data = _files(tmp_path, AFFINES[affine])
    cache = DeviceCache(data, _prefix(), num_workers=4)
    assert [tuple(s) for s in cache.shapes["image"]] == [ROI] * len(data)
    assert cache.channels == {"image": 4, "label": 3}
    _assert_cache_equals_per_file(cache, data)


# ---------------------------------------------------------------------------------------------------- validation tail

VROI = (16, 14, 10)
GRIDS = [(20, 18, 12), (22, 17, 13), (19, 20, 11)]
LPS4 = np.array([[-1.0, 0, 0, 4], [0, -1.0, 0, 2], [0, 0, 1.0, -3], [0, 0, 0, 1]])


def _val_items(dev, n, grids, channels):
    """volumes on the device with an LPS affine (new dicts each call: the resampling writes the new affine into them)"""
    items = []
    for i in range(n):
        g = torch.Generator(device="cpu").manual_seed(200 + i)
        shp = grids[i % len(grids)]
        img = torch.randn((channels,) + shp, generator=g).abs_() + 0.1
        img[:, :2] = 0                                            # zero background, as in the scans
        lab = (torch.rand((3,) + shp, generator=g) < 0.3).to(torch.float32)
        items.append({"image": img.to(dev), "label": lab.to(dev), "idx": i,
                      "image_meta_dict": {"affine": LPS4.copy()}, "label_meta_dict": {"affine": LPS4.copy()}})
    return items


def _resample():
    from mvtb import spatial as S
    return S.SpacingOrientationd(["image", "label"], (1.0, 1.0, 1.0), axcodes="RAS", mode=("bilinear", "nearest"))


def _val_cache(dev, n=7, roi=VROI, grids=GRIDS, channels=4):
    """the items resampled (LPS -> RAS at the same voxel size) and centre-cropped by the fill"""
    from mvtb import spatial as S
    from mvtb.train_stage import DeviceCache
    return DeviceCache(_val_items(dev, n, grids, channels), [_resample(), S.CenterSpatialCropd(["image", "label"], list(roi))],
                       num_workers=2)


def _val_tail(seed, rng="philox-sparse", r=5.0, shell=(4, 3, 2), intensity=8):
    """the scripts' validation tail after the centre crop; rng=None: without the salt-and-pepper"""
    import filters_and_operators as F
    from mvtb import intensity as I
    t = [F.SelectChanneld("image", 0), I.NormalizeIntensityd("image", nonzero=True, channel_wise=True),
         # the ball keeps every bin of the spike shell: the plane wave rewrites a bin whose phase is well defined
         F.RandFourierDiskMaskd("image", r=r, inside_off=False, prob=1.0),
         F.RandPlaneWaves_ellipsoid("image", *shell, intensity_value=intensity, prob=1.0), F.WrapArtifactd("image", alpha=0.5)]
    if rng is not None:
        t.append(F.SaltAndPepper(0.05, "image", prob=1.0, rng=rng, seed=2024))
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
        if hasattr(x, "ellipsoid"):
            x.ellipsoid.set_random_state(seed=seed + 77)
    return t


def _per_sample(cache, tail, indices):
    out = []
    for i in indices:
        d = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in cache.item(i).items()}
        for t in tail:
            d = t(d)
        out.append(d)
    return out


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.gpu
def test_gpu_validation_loader_philox_sparse(cuda_device):
    from mvtb.train_stage import TrainStage
    cache = _val_cache(cuda_device)
    n = len(cache)
    for seed in range(4):
        for bs in (2, 5):
            stage, plain = TrainStage(cache, _val_tail(seed)), TrainStage(cache, _val_tail(seed, None))
            ref_t, ref_plain_t = _val_tail(seed), _val_tail(seed, None)
            batches = [list(range(n))[j:j + bs] for j in range(0, n, bs)]
            for batch, got, got_plain in zip(batches, stage.loader(bs, shuffle=False), plain.loader(bs, shuffle=False),
                                             strict=True):
                assert got["idx"] == batch
                want, want_plain = _per_sample(cache, ref_t, batch), _per_sample(cache, ref_plain_t, batch)
                assert got["image"].shape == (len(batch), 1) + VROI and got["label"].shape == (len(batch), 3) + VROI
                for b in range(len(batch)):
                    assert torch.equal(got["label"][b], want[b]["label"]), (seed, bs, b)
                    err = _rel(got["image"][b], want[b]["image"])
                    assert err <= 1e-5, (seed, bs, b, err)
                    hit, hit_ref = got["image"][b] != got_plain["image"][b], want[b]["image"] != want_plain[b]["image"]
                    assert hit.any() and torch.equal(hit, hit_ref), (seed, bs, b)
            assert stage.sp.offset == ref_t[-1].offset > 0


@pytest.mark.gpu
def test_gpu_validation_loader_torch_generator(cuda_device):
    from torch.utils.data import DataLoader
    from mvtb.train_stage import TrainStage
    cache = _val_cache(cuda_device)
    for seed in range(4):
        for bs in (2, 5):
            stage = TrainStage(cache, _val_tail(seed, "torch"), torch_generator=True)
            plain = TrainStage(cache, _val_tail(seed, None))
            ref_t, ref_plain_t = _val_tail(seed, "torch"), _val_tail(seed, None)
            torch.manual_seed(60 + seed)
            got = list(stage.loader(bs, shuffle=False))
            got_state = torch.get_rng_state()
            got_plain = [plain.apply(plain.draw(g["idx"])) for g in got]
            torch.manual_seed(60 + seed)
            dl = DataLoader(range(len(cache)), batch_size=bs, shuffle=False, num_workers=0, collate_fn=list)
            want = [_per_sample(cache, ref_t, batch) for batch in dl]
            assert torch.equal(torch.get_rng_state(), got_state), (seed, bs)
            want_plain = [_per_sample(cache, ref_plain_t, [d["idx"] for d in w]) for w in want]
            assert len(got) == len(want)
            for g, gp, w, wp in zip(got, got_plain, want, want_plain):
                assert g["idx"] == [d["idx"] for d in w]
                for b in range(len(w)):
                    assert torch.equal(g["label"][b], w[b]["label"])
                    assert _rel(g["image"][b], w[b]["image"]) <= 1e-5, (seed, bs, b)
                    # the stage's select takes its min / max from the chain on the way, so away from the hits it equals the
                    # plain stage to rounding, and at the reference's hits it holds the reference's values
                    hit_ref = w[b]["image"] != wp[b]["image"]
                    assert hit_ref.any(), (seed, bs, b)
                    torch.testing.assert_close(g["image"][b][hit_ref], w[b]["image"][hit_ref], rtol=1e-4, atol=1e-6)
                    scale = float(gp["image"][b].abs().max())
                    assert float((g["image"][b] - gp["image"][b])[~hit_ref].abs().max()) <= 1e-5 * scale, (seed, bs, b)


@pytest.mark.gpu
def test_gpu_validation_at_the_scripts_crop(cuda_device):
    """128 x 128 x 64 centre crops with the disk of radius 12.5: the band-limited chain with the select fused into its inverse
    kernel, on whole cached entries"""
    from mvtb.train_stage import TrainStage
    roi = (128, 128, 64)
    cache = _val_cache(cuda_device, 4, roi, [(136, 132, 70), (140, 130, 66)], channels=2)
    assert [tuple(s) for s in cache.shapes["image"]] == [roi] * 4
    tail = lambda sp: _val_tail(3, "philox-sparse" if sp else None, 12.5, (8, 7, 5), 15)    # noqa: E731
    stage, plain, ref_t, ref_plain_t = TrainStage(cache, tail(True)), TrainStage(cache, tail(False)), tail(True), tail(False)
    for batch, got, got_plain in zip(([0, 1], [2, 3]), stage.loader(2, shuffle=False), plain.loader(2, shuffle=False), strict=True):
        want, want_plain = _per_sample(cache, ref_t, batch), _per_sample(cache, ref_plain_t, batch)
        for b in range(2):
            assert torch.equal(got["label"][b], want[b]["label"]), b
            assert _rel(got["image"][b], want[b]["image"]) <= 1e-5, b
            hit, hit_ref = got["image"][b] != got_plain["image"][b], want[b]["image"] != want_plain[b]["image"]
            assert 0.045 < float(hit.float().mean()) < 0.055 and torch.equal(hit, hit_ref), b


# ----------------------------------------------------------------------------------------------------------------- TCGA

@pytest.mark.gpu
def test_gpu_whole_tumor_on_the_device_equals_numpy(cuda_device):
    import filters_and_operators as F
    r = np.random.RandomState(7)
    for lab in (r.randint(0, 5, size=(9, 7, 5)).astype(np.uint8), r.randint(-3, 3, size=(6, 5, 4)).astype(np.int16),
                np.where(r.rand(5, 4, 3) < 0.5, 0.0, r.standard_normal((5, 4, 3))).astype(np.float32)):
        want = F.WholeTumorTCGA("label")({"label": lab})["label"]
        got = F.WholeTumorTCGA("label")({"label": torch.from_numpy(lab).to(cuda_device)})["label"]
        assert got.is_cuda and got.dtype == torch.float32 and got.is_contiguous()
        assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.gpu
def test_gpu_tcga_prefix_fills_the_cache(cuda_device, tmp_path):
    import filters_and_operators as F
    from mvtb import nifti as N
    from mvtb.train_stage import DeviceCache
    data = _files(tmp_path, AFFINES["lps"], n=4, tcga=True)
    cache = DeviceCache(data, _prefix(tcga=True), num_workers=4)
    assert cache.channels == {"image": 1, "label": 1}
    _assert_cache_equals_per_file(cache, data, tcga=True)
    for item in data:                                   # the device branch on a loaded label is the numpy branch
        lab = N.LoadImaged("label")(item)["label"]
        want = F.WholeTumorTCGA("label")({"label": lab.cpu().numpy()})["label"]
        assert np.array_equal(F.WholeTumorTCGA("label")({"label": lab})["label"].cpu().numpy(), want)


# ---------------------------------------------------------------------------------------------------------- ragged crop

@pytest.mark.gpu
def test_gpu_volume_smaller_than_the_roi(cuda_device):
    from mvtb.train_stage import TrainStage
    grids = [(20, 18, 12), (14, 18, 12), (20, 13, 9)]
    cache = _val_cache(cuda_device, 3, VROI, grids)
    want_shapes = [tuple(min(r, n) for r, n in zip(VROI, g)) for g in grids]
    assert [tuple(s) for s in cache.shapes["image"]] == want_shapes == [VROI, (14, 14, 10), (16, 13, 9)]
    for i, item in enumerate(_val_items(cuda_device, 3, grids, 4)):     # MONAI's centre crop of the whole resampled volume
        full = _resample()(item)
        for k in ("image", "label"):
            sl = (slice(None),) + O.center_crop_slices(tuple(full[k].shape[1:]), VROI)
            assert torch.equal(cache.item(i)[k], full[k][sl]), (i, k)
    stage = TrainStage(cache, _val_tail(0))
    assert stage.apply(stage.draw([0]))["image"].shape == (1, 1) + VROI
    assert stage.apply(stage.draw([1]))["image"].shape == (1, 1, 14, 14, 10)
    with pytest.raises(ValueError, match="different sizes"):
        stage.apply(stage.draw([0, 1]))
    with pytest.raises(ValueError, match="different sizes"):
        list(stage.loader(2, shuffle=False))
