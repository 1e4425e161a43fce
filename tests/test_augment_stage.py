"""The k-space augmentation scripts' transforms in the training stage without a GPU: TrainStage(kspace_augment=True).draw
against RandGibbsNoised / RandKSpaceSpikeNoised called one sample at a time on deep copies (their k-space work stubbed
out, every draw real), the tails the stage refuses with and without the keyword, and the chain descriptors it builds."""
import copy

import numpy as np
import pytest
import torch

ROI = [12, 10, 6]
SHAPES = [(20, 18, 9), (16, 14, 8), (12, 10, 6), (21, 11, 7)]
ORDER = [3, 0, 2, 2, 1, 0, 3, 1, 0, 0, 2, 3, 1, 2, 0, 3]          # 16 samples, repeats and out of order


def _fake_cache(shapes, channels=None):
    """What TrainStage reads of a DeviceCache on the host (no device buffers)."""
    from mvtb.train_stage import DeviceCache
    c = DeviceCache.__new__(DeviceCache)
    c.keys = ["image", "label"]
    c.channels = channels or {"image": 4, "label": 3}
    c.shapes = {k: np.array(shapes, dtype=np.int32) for k in c.keys}
    c.meta = [{} for _ in shapes]
    return c


def _tail(seed, aug, channels=1, sp=True):
    """crop -> flip -> [SelectChanneld] -> intensity -> aug -> [salt-and-pepper], every object seeded"""
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(["image", "label"], roi_size=ROI, random_size=False),
         S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0)]
    if channels == 1:
        t.append(F.SelectChanneld("image", 2))
    t.append(I.IntensityPrologued("image", factors=0.1, offsets=0.1, prob=0.5))
    t += aug()
    if sp:
        t.append(F.SaltAndPepper(0.05, "image", prob=1.0, rng="philox-sparse", seed=11))
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 100 + k)
        for inner in getattr(x, "transforms", {}).values():      # RandKSpaceSpikeNoised's per-key transforms
            inner.set_random_state(seed=seed * 100 + k + 50)
    return t


def _gibbs(prob=0.5, alpha=(0.0, 0.3)):
    import filters_and_operators as F
    return lambda: [F.RandGibbsNoised("image", prob, alpha=alpha)]


def _spikes(global_prob=0.5, prob=0.6, rng=(9, 11), channel_wise=True, common=False):
    import filters_and_operators as F
    return lambda: [F.RandKSpaceSpikeNoised("image", global_prob, prob, intensity_ranges={"image": rng}, channel_wise=channel_wise,
                                            common_sampling=common, common_seed=5)]


@pytest.fixture
def no_kspace(monkeypatch):
    """the per-sample transforms with their k-space work replaced by the identity: every random draw still runs"""
    import filters_and_operators as F
    monkeypatch.setattr(F.GibbsNoise, "__call__", lambda self, img: img)
    monkeypatch.setattr(F.KSpaceSpikeNoise, "__call__", lambda self, img: img)


def _per_sample(tail, shape, c_img):
    """What one sample's per-sample Compose draws: the stage's own transforms through randomize, the augmentation through
    its __call__ on a (c_img, *roi) CPU tensor."""
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    got, size = {}, shape
    for t in tail:
        if isinstance(t, S.RandSpatialCropd):
            t.randomize(shape)
            got["start"], size = tuple(t._start), tuple(t._size)
        elif isinstance(t, S.RandFlipd):
            t.randomize(None)
        elif isinstance(t, I.IntensityPrologued):
            t.scale.randomize()
            t.shift.randomize()
        elif isinstance(t, F.RandGibbsNoised):
            t({"image": torch.zeros((c_img,) + size)})
            got["gibbs"] = (bool(t._do_transform), float(t.sampled_alpha))
        elif isinstance(t, F.RandKSpaceSpikeNoised):
            inner = t.transforms["image"]
            inner.sampled_locs, inner.sampled_k_intensity = [], []
            t({"image": torch.zeros((c_img,) + size)})
            spikes = None
            if t._do_transform:
                spikes = [None] * c_img
                for loc, v in zip(inner.sampled_locs, inner.sampled_k_intensity):
                    spikes[loc[0]] = (tuple(int(i) for i in loc[1:]), float(v))
                spikes = tuple(spikes)
            got["kspike"] = (bool(t._do_transform), spikes)
        elif isinstance(t, F.SaltAndPepper):
            t.randomize(None)
            got["sp"] = (bool(t._do_transform), t.offset)
            n = c_img * int(np.prod(size))
            if t._do_transform:
                t.offset += (n + 255) // 256
    return got


def _states(tail):
    out = []
    for t in tail:
        objs = [t, getattr(t, "scale", None), getattr(t, "shift", None)] + list(getattr(t, "transforms", {}).values())
        for o in objs:
            if o is not None and "R" in vars(o):
                st = o.R.get_state()
                out.append((st[1].tobytes(), st[2], st[3], st[4]))
        if hasattr(t, "offset") and isinstance(t.offset, int):
            out.append(t.offset)
    return out


def _check_draws(aug, channels, no_kspace):
    from mvtb.train_stage import TrainStage
    cache = _fake_cache(SHAPES)
    for seed in range(3):
        a = _tail(seed, aug, channels)
        b = copy.deepcopy(a)
        stage = TrainStage(cache, a, kspace_augment=True)
        rec = stage.draw(ORDER[:5])
        rec2 = stage.draw(ORDER[5:])
        rec = {k: rec[k] + rec2[k] for k in rec}
        gates = {}
        for j, i in enumerate(ORDER):
            want = _per_sample(b, SHAPES[i], channels)
            assert rec["start"][j] == want["start"]
            if "gibbs" in want:
                assert (rec["gibbs_gate"][j], rec["alpha"][j]) == want["gibbs"], (seed, j)
                gates.setdefault("gibbs", set()).add(want["gibbs"][0])
            if "kspike" in want:
                assert (rec["kspike_gate"][j], rec["kspikes"][j]) == want["kspike"], (seed, j)
                gates.setdefault("kspike", set()).add(want["kspike"][0])
            assert (rec["sp_gate"][j], rec["sp_offset"][j]) == want["sp"]
        assert gates and all(v == {False, True} for v in gates.values())     # both gate values were drawn
        assert _states(a) == _states(b), seed


@pytest.mark.parametrize("channels", [1, 4])
@pytest.mark.parametrize("prob", [0.5, 1.0])
def test_gibbs_draw_matches_per_sample(no_kspace, channels, prob):
    if prob == 1.0:                                     # every gate on: check the alpha draws
        from mvtb.train_stage import TrainStage
        a = _tail(0, _gibbs(1.0), channels)
        b = copy.deepcopy(a)
        rec = TrainStage(_fake_cache(SHAPES), a, kspace_augment=True).draw(ORDER)
        want = [_per_sample(b, SHAPES[i], channels)["gibbs"] for i in ORDER]
        assert list(zip(rec["gibbs_gate"], rec["alpha"])) == want and all(g for g, _ in want)
        assert _states(a) == _states(b)
        return
    _check_draws(_gibbs(prob), channels, no_kspace)


@pytest.mark.parametrize("channels", [1, 4])
@pytest.mark.parametrize("channel_wise", [True, False])
@pytest.mark.parametrize("common", [False, True])
def test_spike_draw_matches_per_sample(no_kspace, channels, channel_wise, common):
    _check_draws(_spikes(channel_wise=channel_wise, common=common), channels, no_kspace)


def test_spike_draw_with_per_channel_ranges(no_kspace):
    _check_draws(_spikes(rng=[(9, 10), (10, 11), (11, 12), (5, 6)]), 4, no_kspace)


def test_spike_draw_the_scripts_settings(no_kspace):
    """global_prob=0.1, prob=1.0, (10, 11): gated samples have a spike in every channel"""
    from mvtb.train_stage import TrainStage
    a = _tail(1, _spikes(0.1, 1.0, (10, 11)), 4)
    b = copy.deepcopy(a)
    order = list(range(4)) * 10
    rec = TrainStage(_fake_cache(SHAPES), a, kspace_augment=True).draw(order)
    for j, i in enumerate(order):
        assert (rec["kspike_gate"][j], rec["kspikes"][j]) == _per_sample(b, SHAPES[i], 4)["kspike"]
        if rec["kspike_gate"][j]:
            assert all(s is not None and 10 <= s[1] < 11 for s in rec["kspikes"][j])
    assert 0 < sum(rec["kspike_gate"]) < len(order)
    assert _states(a) == _states(b)


def test_both_augmentations_in_one_tail(no_kspace):
    def both():
        return _gibbs(0.5)() + _spikes(0.5, 0.5)()
    _check_draws(both, 4, no_kspace)


# ----------------------------------------------------------------------------------------------------------- refusals

def _refused():
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    crop = lambda: S.RandSpatialCropd(["image", "label"], roi_size=ROI, random_size=False)        # noqa: E731
    norm = lambda: I.NormalizeIntensityd("image", nonzero=True, channel_wise=True)               # noqa: E731
    gibbs = lambda **k: F.RandGibbsNoised(k.pop("keys", "image"), 0.1, alpha=(0.0, 0.3), **k)    # noqa: E731
    spike = lambda **k: F.RandKSpaceSpikeNoised(k.pop("keys", "image"), 0.1, 1.0, **k)           # noqa: E731
    rng = {"intensity_ranges": {"image": (10, 11)}}
    disk = lambda: F.RandFourierDiskMaskd("image", r=8.0, prob=1.0)                               # noqa: E731
    wave = lambda: F.RandPlaneWaves_ellipsoid("image", 5, 4, 2, intensity_value=12, prob=1.0)     # noqa: E731
    wrap = lambda: F.WrapArtifactd("image", alpha=0.5)                                            # noqa: E731
    sp = lambda: F.SaltAndPepper(0.05, "image", rng="philox-sparse")                               # noqa: E731
    # case: (tail, what the keyword changes it to: the exception and a part of its message)
    return {
        "spike_default_range": ([crop(), spike()], (NotImplementedError, "intensity_ranges")),
        "spike_range_of_another_key": ([crop(), F.RandKSpaceSpikeNoised(["image"], 0.1, 1.0, intensity_ranges=[(10, 11)])],
                                       (NotImplementedError, "intensity_ranges")),
        "gibbs_numpy": ([crop(), gibbs(as_tensor_output=False)], (NotImplementedError, "numpy")),
        "spike_numpy": ([crop(), spike(as_tensor_output=False, **rng)], (NotImplementedError, "numpy")),
        "gibbs_and_disk": ([crop(), norm(), disk(), gibbs()], (NotImplementedError, "one mask")),
        "disk_and_gibbs": ([crop(), norm(), gibbs(), disk()], (NotImplementedError, "one mask")),
        "spike_and_wave": ([crop(), wave(), spike(**rng)], (NotImplementedError, "one spike source")),
        "wave_and_spike": ([crop(), spike(**rng), wave()], (NotImplementedError, "one spike source")),
        "gibbs_before_intensity": ([crop(), gibbs(), norm()], (NotImplementedError, "order")),
        "gibbs_after_wrap": ([crop(), wrap(), gibbs()], (NotImplementedError, "order")),
        "gibbs_after_sp": ([crop(), sp(), gibbs()], (NotImplementedError, "order")),
        "spike_before_gibbs": ([crop(), spike(**rng), gibbs()], (NotImplementedError, "order")),
        "spike_after_wrap": ([crop(), wrap(), spike(**rng)], (NotImplementedError, "order")),
        "gibbs_on_label": ([crop(), norm(), gibbs(keys="label")], (NotImplementedError, "one cached key")),
        "gibbs_two_keys": ([crop(), gibbs(keys=["image", "label"])], (NotImplementedError, "one cached key")),
        "spike_two_keys": ([crop(), spike(keys=["image", "label"], intensity_ranges={"image": (10, 11), "label": (1, 2)})],
                           (NotImplementedError, "one cached key")),
        "select_between_spike_and_sp": ([crop(), spike(**rng), F.SelectChanneld("image", 0), sp()],
                                        (NotImplementedError, "drawn per channel")),
        "select_after_spike": ([crop(), spike(**rng), F.SelectChanneld("image", 0)], (NotImplementedError, "drawn per channel")),
        "spike_ranges_per_channel_count": ([crop(), spike(intensity_ranges={"image": [(9, 10), (10, 11)]})],
                                           (ValueError, "one per channel")),
        "gibbs_array_transform": ([crop(), F.RandGibbsNoise(0.1)], (NotImplementedError, "not supported")),
        "spike_array_transform": ([crop(), F.RandKSpaceSpikeNoise(0.1, (10, 11))], (NotImplementedError, "not supported")),
    }


@pytest.mark.parametrize("keyword", [False, True])
@pytest.mark.parametrize("case", sorted(_refused()))
def test_refusals(case, keyword):
    from mvtb.train_stage import TrainStage
    tail, (exc, msg) = _refused()[case]
    cache = _fake_cache([(20, 18, 9)] * 2)
    if not keyword:
        with pytest.raises(NotImplementedError):
            TrainStage(cache, tail)
        return
    with pytest.raises(exc, match=msg):
        TrainStage(cache, tail, kspace_augment=True)


def test_gibbs_up_to_eight_channels():
    from mvtb.train_stage import TrainStage
    TrainStage(_fake_cache([(20, 18, 9)] * 2, {"image": 8, "label": 3}), _tail(0, _gibbs(), 8), kspace_augment=True)
    with pytest.raises(NotImplementedError, match="at most 8"):
        TrainStage(_fake_cache([(20, 18, 9)] * 2, {"image": 9, "label": 3}), _tail(0, _gibbs(), 9), kspace_augment=True)


def test_without_the_keyword_the_message_names_it():
    import filters_and_operators as F
    from mvtb.train_stage import TrainStage
    for t in (F.RandGibbsNoised("image", 1.0), F.RandKSpaceSpikeNoised("image", 0.1, 1.0, intensity_ranges={"image": (10, 11)})):
        with pytest.raises(NotImplementedError, match="kspace_augment=True"):
            TrainStage(_fake_cache([(20, 18, 9)] * 2), [t])


def test_keyword_leaves_other_tails_alone():
    """the same draws and descriptors for a tail without the augmentation transforms, with and without the keyword"""
    from mvtb.train_stage import TrainStage
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S

    def tail():
        t = [S.RandSpatialCropd(["image", "label"], roi_size=ROI, random_size=False), F.SelectChanneld("image", 0),
             I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), F.RandFourierDiskMaskd("image", r=[4.0, 9.0], prob=0.7),
             F.RandPlaneWaves_ellipsoid("image", 5, 4, 2, intensity_value=12, prob=0.6), F.WrapArtifactd("image", alpha=0.5)]
        for k, x in enumerate(t):
            if hasattr(x, "set_random_state"):
                x.set_random_state(seed=k)
            if hasattr(x, "ellipsoid"):
                x.ellipsoid.set_random_state(seed=9)
        return t
    cache = _fake_cache(SHAPES)
    a, b = TrainStage(cache, tail()), TrainStage(cache, tail(), kspace_augment=True)
    ra, rb = a.draw(ORDER), b.draw(ORDER)
    assert ra == rb
    for j in range(len(ORDER)):
        da, busy_a = a._sample_descs(ra, j, tuple(ROI), 1)
        db, busy_b = b._sample_descs(rb, j, tuple(ROI), 1)
        assert bytes(da[0]) == bytes(db[0]) and busy_a and busy_b


# -------------------------------------------------------------------------------------------------------- descriptors

def test_descriptors_per_channel_volume():
    from mvtb import _lib, host
    from mvtb.train_stage import TrainStage

    def both():
        return _gibbs(0.6, (0.0, 0.9))() + _spikes(0.7, 0.5, (9, 11))()
    stage = TrainStage(_fake_cache(SHAPES), _tail(0, both, 4), kspace_augment=True)
    rec = stage.draw(ORDER * 2)
    roi = tuple(ROI)
    seen = set()
    for b in range(len(rec["index"])):
        descs, busy = stage._sample_descs(rec, b, roi, 4)
        assert len(descs) == 4
        g, spikes = rec["gibbs_gate"][b], rec["kspikes"][b]
        assert busy == (g or (spikes is not None and any(s is not None for s in spikes)))
        for c, d in enumerate(descs):
            if g:
                assert d.mask_kind == _lib.MASK_CENTRED and d.mask_ndim == 3
                assert d.mask_thresh == host.gibbs_threshold(rec["alpha"][b], roi)
            else:
                assert d.mask_kind == _lib.MASK_NONE
            s = None if spikes is None else spikes[c]
            assert d.n_spikes == (s is not None)
            if s is not None:
                assert tuple(d.spikes[0].idx[:3]) == s[0] and d.spikes[0].amplitude == host.exp_f32(s[1])
                assert all(0 <= i < n for i, n in zip(s[0], roi))
            assert d.wrap_naxes == 0
            seen.add((g, s is not None))
    assert seen == {(False, False), (False, True), (True, False), (True, True)}


def test_wrap_sends_every_sample_through_the_chain():
    import filters_and_operators as F
    from mvtb.train_stage import TrainStage

    def gibbs_wrap():
        return _gibbs(0.3)() + [F.WrapArtifactd("image", alpha=0.5)]
    stage = TrainStage(_fake_cache(SHAPES), _tail(0, gibbs_wrap), kspace_augment=True)
    rec = stage.draw(ORDER)
    assert not all(rec["gibbs_gate"])
    for b in range(len(ORDER)):
        descs, busy = stage._sample_descs(rec, b, tuple(ROI), 1)
        assert busy and descs[0].wrap_naxes == 3 and descs[0].wrap_alpha == 0.5
