"""The training loader's batch stage on the GPU against the per-sample drop-ins: a DeviceCache of volumes on two grids and
the full 127 tail (crop -> flip -> intensity prologue -> disk -> plane wave -> wrap -> philox-sparse salt-and-pepper) batch
by batch from TrainStage.loader, against the same seeded transform objects applied one sample at a time; the cache filled
from NIfTI files against the per-file prefix; and the loader's epoch order against RandomSampler."""
import math

import numpy as np
import pytest
import torch

from oracle import nifti_writer as W

ROI = (12, 10, 8)
GRIDS = [(20, 18, 12), (16, 14, 10)]


def _items(dev, n=6):
    items = []
    for i in range(n):
        g = torch.Generator(device="cpu").manual_seed(100 + i)
        shp = GRIDS[i % 2]
        img = torch.randn((4,) + shp, generator=g).abs_() + 0.1
        img[:, :2] = 0                                            # zero background, as in the scans
        lab = (torch.rand((3,) + shp, generator=g) < 0.3).to(torch.float32)
        items.append({"image": img.to(dev), "label": lab.to(dev), "idx": i, "image_meta_dict": {"affine": np.eye(4) * (i + 1)}})
    return items


def _tail(seed, select_after=False, sp=True, rng="philox-sparse"):
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(["image", "label"], roi_size=list(ROI), random_size=False),
         S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0)]
    if not select_after:
        t.append(F.SelectChanneld("image", 2))
    t += [I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), I.RandScaleIntensityd("image", factors=0.1, prob=0.5),
          I.RandShiftIntensityd("image", offsets=0.1, prob=0.5),
          # the ball keeps every bin of the spike shell (|k - centre| <= 4): the per-sample plane wave then rewrites a bin that
          # holds data, whose phase is well defined (on a bin the disk zeroed it is the phase of rounding noise)
          F.RandFourierDiskMaskd("image", r=[5.0, 7.0], inside_off=False, prob=0.7),
          F.RandPlaneWaves_ellipsoid("image", 4, 3, 2, intensity_value=8, prob=0.6),
          F.WrapArtifactd("image", alpha=0.5)]
    if sp:
        t.append(F.SaltAndPepper(0.05, "image", prob=1.0, rng=rng, seed=2024))
    if select_after:
        t.append(F.SelectChanneld("image", 1))
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
        if hasattr(x, "ellipsoid"):
            x.ellipsoid.set_random_state(seed=seed + 77)
    return t


def _per_sample(cache, tail, indices):
    out = []
    for i in indices:
        d = cache.item(i)
        d = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}
        for t in tail:
            d = t(d)
        out.append(d)
    return out


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.gpu
@pytest.mark.parametrize("select_after", [False, True])
@pytest.mark.parametrize("rng", ["philox-sparse", "philox"])
def test_gpu_batches_equal_per_sample_dropins(cuda_device, select_after, rng):
    from torch.utils.data import BatchSampler, RandomSampler
    from mvtb.train_stage import DeviceCache, TrainStage
    cache = DeviceCache(_items(cuda_device), [], num_workers=2)
    assert [tuple(s) for s in cache.shapes["image"]] == [GRIDS[i % 2] for i in range(6)]
    for seed in range(4):
        for bs in (2, 5):
            stage = TrainStage(cache, _tail(seed, select_after, rng=rng))
            plain = TrainStage(cache, _tail(seed, select_after, sp=False))           # the same draws without the select
            ref_t, ref_plain_t = _tail(seed, select_after, rng=rng), _tail(seed, select_after, sp=False)
            g, g2, g3 = (torch.Generator().manual_seed(seed) for _ in range(3))
            batches = list(BatchSampler(RandomSampler(range(len(cache)), generator=g3), bs, False))
            for batch, got, got_plain in zip(batches, stage.loader(bs, generator=g), plain.loader(bs, generator=g2)):
                assert got["idx"] == list(batch)
                want = _per_sample(cache, ref_t, batch)
                want_plain = _per_sample(cache, ref_plain_t, batch)
                assert got["image"].shape == (len(batch), 1) + ROI and got["label"].shape == (len(batch), 3) + ROI
                for b in range(len(batch)):
                    assert torch.equal(got["label"][b], want[b]["label"]), (seed, bs, b)
                    err = _rel(got["image"][b], want[b]["image"])
                    assert err <= 1e-5, (seed, bs, b, err)
                    hit = got["image"][b] != got_plain["image"][b]
                    hit_ref = want[b]["image"] != want_plain[b]["image"]
                    assert hit.any() and torch.equal(hit, hit_ref), (seed, bs, b)
            assert stage.sp.offset == ref_t[-2 if select_after else -1].offset


@pytest.mark.gpu
def test_gpu_loader_epoch_order(cuda_device):
    from torch.utils.data import RandomSampler
    from mvtb.train_stage import DeviceCache, TrainStage
    cache = DeviceCache(_items(cuda_device, 7), [], num_workers=1)
    stage = TrainStage(cache, _tail(0))
    seen = [i for out in stage.loader(3, shuffle=True, generator=torch.Generator().manual_seed(9)) for i in out["idx"]]
    assert seen == list(RandomSampler(range(7), generator=torch.Generator().manual_seed(9)))
    seen = [i for out in stage.loader(3, shuffle=False, drop_last=True) for i in out["idx"]]
    assert seen == list(range(6))
    # records drawn one sample at a time (as DataLoader workers would) and applied as a collated list
    rec = [stage[i] for i in (4, 1)]
    out = stage.apply(rec)
    assert out["idx"] == [4, 1] and out["image"].shape == (2, 1) + ROI


@pytest.mark.gpu
def test_gpu_cache_from_nifti_equals_prefix_per_file(cuda_device, tmp_path):
    import filters_and_operators as F
    from mvtb import nifti as N, spatial as S
    from mvtb.train_stage import DeviceCache
    lps = np.array([[-1.5, 0, 0, 10], [0, -1.2, 0, 20], [0, 0, 2.5, -5]])
    data = []
    for n in range(6):
        r = np.random.RandomState(n)
        shp = (30 + 4 * (n % 3), 28, 20 + 2 * (n % 2))
        img = (r.standard_normal(shp + (4,)) * 100).astype(np.int16)
        lab = r.randint(0, 4, size=shp).astype(np.uint8)
        sfx = ".nii.gz" if n % 2 else ".nii"
        data.append({"image": str(W.write(tmp_path / f"i{n}{sfx}", img, sform=lps, pixdim=(1.5, 1.2, 2.5),
                                          gzip_members=1 if n % 2 else 0, level=1)),
                     "label": str(W.write(tmp_path / f"l{n}{sfx}", lab, sform=lps, pixdim=(1.5, 1.2, 2.5),
                                          gzip_members=1 if n % 2 else 0, level=1))})

    def prefix():
        return [N.LoadImaged(["image", "label"]), N.AsChannelFirstd("image"), F.ConvertToMultiChannelBasedOnBratsClassesd("label"),
                S.SpacingOrientationd(["image", "label"], (1.0, 1.5, 2.0), axcodes="RAS", mode=("bilinear", "nearest"))]

    cache = DeviceCache(data, prefix(), num_workers=4)
    assert len({tuple(s) for s in cache.shapes["image"]}) > 1                   # a ragged cache
    for i, item in enumerate(data):
        d = dict(item)
        for t in prefix():
            d = t(d)
        got = cache.item(i)
        for k in ("image", "label"):
            assert torch.equal(got[k], d[k]), (i, k)
            assert np.array_equal(got[f"{k}_meta_dict"]["affine"], d[f"{k}_meta_dict"]["affine"]), (i, k)


@pytest.mark.gpu
def test_gpu_batches_at_the_scripts_crop(cuda_device):
    """128 x 128 x 64 crops with the disk of radius 12.5: the band-limited chain with the select pass fused into its inverse
    kernel, whose Philox spans then follow the per-sample SaltAndPepper offsets (4096 blocks a sample, 128 spans)."""
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    from mvtb.train_stage import DeviceCache, TrainStage
    roi = (128, 128, 64)
    items = []
    for i, shp in enumerate([(136, 132, 70), (144, 130, 66), (136, 132, 70), (144, 130, 66)]):
        g = torch.Generator(device="cpu").manual_seed(300 + i)
        img = torch.randn((2,) + shp, generator=g).abs_()
        img *= img > 0.3
        lab = (torch.rand((3,) + shp, generator=g) < 0.3).to(torch.float32)
        items.append({"image": img.to(cuda_device), "label": lab.to(cuda_device), "idx": i})
    cache = DeviceCache(items, [], num_workers=2)

    def tail(sp=True):
        t = [S.RandSpatialCropd(["image", "label"], roi_size=list(roi), random_size=False),
             S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0), F.SelectChanneld("image", 1),
             I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), I.RandScaleIntensityd("image", factors=0.1, prob=0.5),
             I.RandShiftIntensityd("image", offsets=0.1, prob=0.5), F.RandFourierDiskMaskd("image", r=12.5, prob=1.0),
             # a shell inside the ball, so that the per-sample plane wave rewrites a bin with a well-defined phase
             F.RandPlaneWaves_ellipsoid("image", 8, 7, 5, intensity_value=15, prob=1.0), F.WrapArtifactd("image", alpha=0.5)]
        if sp:
            t.append(F.SaltAndPepper(0.05, "image", prob=1.0, rng="philox-sparse", seed=7))
        for k, x in enumerate(t):
            if hasattr(x, "set_random_state"):
                x.set_random_state(seed=50 + k)
            if hasattr(x, "ellipsoid"):
                x.ellipsoid.set_random_state(seed=51)
        return t

    stage, plain, ref_t, ref_plain_t = TrainStage(cache, tail()), TrainStage(cache, tail(False)), tail(), tail(False)
    for batch in ([2, 0], [3, 1]):
        got, got_plain = stage.apply(stage.draw(batch)), plain.apply(plain.draw(batch))
        want, want_plain = _per_sample(cache, ref_t, batch), _per_sample(cache, ref_plain_t, batch)
        for b in range(2):
            assert torch.equal(got["label"][b], want[b]["label"]), b
            assert _rel(got["image"][b], want[b]["image"]) <= 1e-5, b
            hit, hit_ref = got["image"][b] != got_plain["image"][b], want[b]["image"] != want_plain[b]["image"]
            assert 0.045 < float(hit.float().mean()) < 0.055 and torch.equal(hit, hit_ref), b
    assert stage.sp.offset == ref_t[-1].offset == 4 * (math.prod(roi) // 256)
