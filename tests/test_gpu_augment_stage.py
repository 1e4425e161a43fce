"""The k-space augmentation scripts' tails through TrainStage(kspace_augment=True) on the GPU, against the same seeded
transform objects applied one sample at a time through the drop-ins: RandGibbsNoised on 1 and 4 channels,
RandKSpaceSpikeNoised channel-wise and shared, both in one tail, a philox-sparse salt-and-pepper behind them, and a
128 x 128 x 64 batch whose Gibbs balls take the band-limited and the general chain path.  Labels and the samples whose
gates are all off are equal bit for bit; gated samples are within rel-L2 1e-5."""
import numpy as np
import pytest
import torch

ROI = (12, 10, 8)
GRIDS = [(20, 18, 12), (16, 14, 10)]
REL = 1e-5


def _items(dev, n=7):
    items = []
    for i in range(n):
        g = torch.Generator(device="cpu").manual_seed(400 + i)
        shp = GRIDS[i % 2]
        img = torch.randn((4,) + shp, generator=g).abs_() + 0.1
        img[:, :2] = 0                                            # zero background, as in the scans
        lab = (torch.rand((3,) + shp, generator=g) < 0.3).to(torch.float32)
        items.append({"image": img.to(dev), "label": lab.to(dev), "idx": i})
    return items


@pytest.fixture(scope="module")
def cache(cuda_device):
    from mvtb.train_stage import DeviceCache
    return DeviceCache(_items(cuda_device), [], num_workers=2)


def _gibbs(prob=0.5, alpha=(0.0, 0.3)):
    import filters_and_operators as F
    return [F.RandGibbsNoised("image", prob, alpha=alpha)]


def _spikes(global_prob=0.5, prob=0.6, rng=(9, 11), channel_wise=True):
    import filters_and_operators as F
    return [F.RandKSpaceSpikeNoised("image", global_prob, prob, intensity_ranges={"image": rng}, channel_wise=channel_wise)]


AUG = {"gibbs": lambda: _gibbs(), "gibbs_all": lambda: _gibbs(1.0, (0.0, 0.5)),
       "spikes": lambda: _spikes(), "spikes_shared": lambda: _spikes(0.5, 0.7, (10, 11), False),
       "spikes_scripts": lambda: _spikes(0.1, 1.0, (10, 11)), "both": lambda: _gibbs(0.5, (0.0, 0.4)) + _spikes(0.5, 0.5)}


def _tail(seed, aug, channels, sp=True):
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(["image", "label"], roi_size=list(ROI), random_size=False),
         S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0)]
    if channels == 1:
        t.append(F.SelectChanneld("image", 2))
    t.append(I.IntensityPrologued("image", factors=0.1, offsets=0.1, prob=0.5))
    t += AUG[aug]()
    if sp:
        t.append(F.SaltAndPepper(0.05, "image", prob=1.0, rng="philox-sparse", seed=2024))
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
        for inner in getattr(x, "transforms", {}).values():
            inner.set_random_state(seed=seed * 1000 + k + 500)
    return t


def _per_sample(cache, tail, indices):
    """the drop-ins one sample at a time; with each result, whether a gate was on and the spikes per channel"""
    import filters_and_operators as F
    out = []
    for i in indices:
        d = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in cache.item(i).items()}
        gated, spikes = False, {}
        for t in tail:
            d = t(d)
            if isinstance(t, F.RandGibbsNoised):
                gated |= bool(t._do_transform)
            elif isinstance(t, F.RandKSpaceSpikeNoised) and t._do_transform:
                locs = t.transforms["image"].sampled_locs
                gated |= bool(locs)
                spikes = {int(loc[0]): tuple(int(v) for v in loc[1:]) for loc in locs}
        out.append((d, gated, spikes))
    return out


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _remove_plane_waves(y, spikes):
    """each channel less its +-f plane wave (the phase of a spike on a bin the Gibbs mask zeroed is rounding noise in the
    per-sample pipeline, SURVEY section 0); returns the residual and the amplitudes"""
    y = y.double().cpu().numpy().copy()
    amps = []
    for ch, idx in spikes.items():
        shape = y.shape[-3:]
        grids = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
        ph = 2 * np.pi * sum((i - n // 2) * g / n for i, g, n in zip(idx, grids, shape))
        c, s = np.cos(ph), np.sin(ph)
        a = (y[ch] * c).sum() / (c * c).sum()
        b = (y[ch] * s).sum() / max((s * s).sum(), 1e-30)
        y[ch] -= a * c + b * s
        amps.append(np.hypot(a, b))
    return torch.from_numpy(y), np.array(amps)


def _compare(cache, aug, channels, seed, bs, project=False):
    from torch.utils.data import BatchSampler, RandomSampler
    from mvtb.train_stage import TrainStage
    stage = TrainStage(cache, _tail(seed, aug, channels), kspace_augment=True)
    plain = TrainStage(cache, _tail(seed, aug, channels, sp=False), kspace_augment=True)
    ref_t, ref_plain_t = _tail(seed, aug, channels), _tail(seed, aug, channels, sp=False)
    g, g2, g3 = (torch.Generator().manual_seed(seed) for _ in range(3))
    batches = list(BatchSampler(RandomSampler(range(len(cache)), generator=g3), bs, False))
    counts = [0, 0]
    for batch, got, got_plain in zip(batches, stage.loader(bs, generator=g), plain.loader(bs, generator=g2), strict=True):
        assert got["idx"] == list(batch)
        want, want_plain = _per_sample(cache, ref_t, batch), _per_sample(cache, ref_plain_t, batch)
        assert got["image"].shape == (len(batch), channels) + ROI
        for b, ((w, gated, spikes), (wp, _, _)) in enumerate(zip(want, want_plain)):
            where = (aug, channels, seed, bs, b)
            assert torch.equal(got["label"][b], w["label"]), where
            counts[gated] += 1
            if not gated:
                assert torch.equal(got["image"][b], w["image"]), where
                assert torch.equal(got_plain["image"][b], wp["image"]), where
                continue
            if project and spikes:
                (ga, gamp), (wa, wamp) = _remove_plane_waves(got_plain["image"][b], spikes), _remove_plane_waves(wp["image"], spikes)
                err = _rel(ga, wa)
                assert np.allclose(gamp, wamp, rtol=1e-3), (where, gamp, wamp)
            else:
                err = _rel(got["image"][b], w["image"])
                assert _rel(got_plain["image"][b], wp["image"]) <= REL, where
            assert err <= REL, (where, err)
            # the salt-and-pepper hits the per-sample positions
            hit, hit_ref = got["image"][b] != got_plain["image"][b], w["image"] != wp["image"]
            assert hit.any() and torch.equal(hit, hit_ref), where
    assert stage.sp.offset == ref_t[-1].offset > 0
    return counts


@pytest.mark.gpu
@pytest.mark.parametrize("aug,channels", [("gibbs", 1), ("gibbs", 4), ("gibbs_all", 1), ("spikes", 1), ("spikes", 4),
                                          ("spikes_shared", 4), ("spikes_scripts", 1)])
def test_gpu_loader_equals_per_sample_dropins(cache, aug, channels):
    counts = [0, 0]
    for seed in range(4):
        for bs in (2, 5):
            c = _compare(cache, aug, channels, seed, bs)
            counts = [counts[0] + c[0], counts[1] + c[1]]
    assert counts[1] > 0 and (counts[0] > 0) == (aug != "gibbs_all"), counts


@pytest.mark.gpu
def test_gpu_spikes_after_gibbs(cache):
    """a spike on a bin the Gibbs mask zeroed: compared after removing each channel's plane wave, amplitudes checked"""
    counts = [0, 0]
    for seed in range(4):
        for bs in (2, 5):
            c = _compare(cache, "both", 4, seed, bs, project=True)
            counts = [counts[0] + c[0], counts[1] + c[1]]
    assert counts[0] > 0 and counts[1] > 0, counts


def _kinds(plan):
    import ctypes as C
    from mvtb import _lib
    L = _lib.lib()
    ms, cn = (C.c_double * _lib.K_KINDS)(), (C.c_int * _lib.K_KINDS)()
    _lib.check(L, L.mvtb_plan_profile_read(plan, ms, cn))
    _lib.check(L, L.mvtb_plan_profile(plan, 0))
    return {L.mvtb_kernel_name(k).decode() for k in range(_lib.K_KINDS) if cn[k]}


@pytest.mark.gpu
def test_gpu_gibbs_band_limited_and_general_path(cuda_device):
    """at the scripts' 128 x 128 x 64: alpha 0.95 keeps a small ball (band-limited path), alpha 0.3 a large one (r >= 45,
    general path); a batch of both takes the general path, a batch of two equal small balls the band-limited one, and each sample
    equals GibbsNoise(alpha) on the normalised sample"""
    import filters_and_operators as F
    from mvtb import _lib, functional as Fn, intensity as I
    from mvtb.train_stage import DeviceCache, TrainStage
    roi = (128, 128, 64)
    items = []
    for i in range(3):
        g = torch.Generator(device="cpu").manual_seed(500 + i)
        img = torch.randn((1,) + roi, generator=g).abs_()
        img *= img > 0.3
        items.append({"image": img.to(cuda_device), "label": (img > 1.0).to(torch.float32).to(cuda_device)})
    cache = DeviceCache(items, [], num_workers=1)
    stage = TrainStage(cache, [I.NormalizeIntensityd("image", nonzero=True, channel_wise=True),
                               F.RandGibbsNoised("image", 1.0, alpha=(0.0, 1.0))], kspace_augment=True)
    L = _lib.lib()
    plan = Fn.get_plan(roi, 2, cuda_device)
    # the band-limited path needs one mask threshold in the call: the same alpha twice
    for alphas, band_limited in (((0.95, 0.3), False), ((0.95, 0.95), True), ((0.3, 0.5), False)):
        rec = stage.draw([0, 2])
        rec["alpha"] = list(alphas)
        _lib.check(L, L.mvtb_plan_profile(plan, 1))
        got = stage.apply(rec)
        torch.cuda.synchronize()
        kinds = _kinds(plan)
        assert any(k.startswith("k_bl_") for k in kinds) == band_limited, (alphas, kinds)
        for b, (i, a) in enumerate(zip((0, 2), alphas)):
            x = I.NormalizeIntensityd("image", nonzero=True, channel_wise=True)({"image": cache.item(i)["image"].clone()})["image"]
            want = F.GibbsNoise(a)(x)
            assert _rel(got["image"][b], want) <= REL, (alphas, b)
            assert torch.equal(got["label"][b], cache.item(i)["label"])
