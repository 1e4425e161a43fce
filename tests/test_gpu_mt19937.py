"""torch's CPU generator made on the device: mvtb.functional.torch_uniform against torch.rand from the same state, the
SaltAndPepper(rng="torch") drop-in against its host path, and TrainStage(torch_generator=True) batches against the
per-sample drop-ins in a DataLoader on the same generator."""
import pytest
import torch

SIZES = [(1, 128, 128, 64), (1, 240, 240, 155), (4, 240, 240, 155), (1,), (7,), (623,), (625,), (3, 5, 7, 11), (100003,)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SIZES)
@pytest.mark.parametrize("pre", [0, 1, 624, 1000])
def test_gpu_torch_uniform_equals_torch_rand(cuda_device, shape, pre):
    from mvtb import functional as Fn
    segments = 2 if len(shape) > 1 and shape[0] == 1 else 1
    torch.manual_seed(1000 + pre)
    if pre:
        torch.rand(pre)
    start = torch.get_rng_state()
    want = torch.stack([torch.rand(shape) for _ in range(segments)])
    want_state = torch.get_rng_state()
    torch.set_rng_state(start)
    got = Fn.torch_uniform(shape, segments, cuda_device)
    assert got.shape == (segments,) + shape and got.dtype == torch.float32 and got.is_cuda
    assert torch.equal(torch.get_rng_state(), want_state)
    assert torch.equal(got.cpu(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 128, 128, 64), (2, 17, 9, 5)])
def test_gpu_dropin_equals_host_path(cuda_device, shape):
    import filters_and_operators as F
    x = torch.randn(shape, generator=torch.Generator().manual_seed(3)).to(cuda_device)
    for seed in range(3):
        torch.manual_seed(seed)
        u = torch.rand(shape)
        want = F.SaltAndPepper(0.05).salt_and_pepper(x, u=u)
        want_state = torch.get_rng_state()
        torch.manual_seed(seed)
        got = F.SaltAndPepper(0.05).salt_and_pepper(x)
        assert torch.equal(got, want)
        assert torch.equal(torch.get_rng_state(), want_state)


@pytest.mark.gpu
def test_gpu_dropin_keeps_torch_rand_under_a_float64_default(cuda_device):
    import filters_and_operators as F
    x = torch.randn((2, 9, 7, 5), generator=torch.Generator().manual_seed(4)).to(cuda_device)
    old = torch.get_default_dtype()
    try:
        torch.set_default_dtype(torch.float64)
        torch.manual_seed(8)
        u = torch.rand(x.size())
        torch.manual_seed(8)
        got = F.SaltAndPepper(0.1).salt_and_pepper(x)
    finally:
        torch.set_default_dtype(old)
    assert torch.equal(got, F.SaltAndPepper(0.1).salt_and_pepper(x, u=u))


@pytest.mark.gpu
def test_gpu_loader_equals_per_sample_dropins_in_a_dataloader(cuda_device):
    from torch.utils.data import DataLoader
    from mvtb.train_stage import DeviceCache, TrainStage
    from test_gpu_train_stage import ROI, _items, _per_sample, _rel, _tail
    cache = DeviceCache(_items(cuda_device), [], num_workers=2)
    for seed in range(4):
        for bs in (2, 5):
            stage = TrainStage(cache, _tail(seed, rng="torch"), torch_generator=True)
            plain = TrainStage(cache, _tail(seed, sp=False))
            ref_t, ref_plain_t = _tail(seed, rng="torch"), _tail(seed, sp=False)
            torch.manual_seed(50 + seed)
            got = list(stage.loader(bs, generator=torch.Generator().manual_seed(seed)))
            got_state = torch.get_rng_state()
            got_plain = [plain.apply(plain.draw(g["idx"])) for g in got]     # the same batches without the select
            torch.manual_seed(50 + seed)
            dl = DataLoader(range(len(cache)), batch_size=bs, shuffle=True, num_workers=0,
                            generator=torch.Generator().manual_seed(seed), collate_fn=list)
            want = [_per_sample(cache, ref_t, batch) for batch in dl]
            assert torch.equal(torch.get_rng_state(), got_state), (seed, bs)
            want_plain = [_per_sample(cache, ref_plain_t, [d["idx"] for d in w]) for w in want]
            assert len(got) == len(want)
            for g, gp, w, wp in zip(got, got_plain, want, want_plain):
                assert g["idx"] == [d["idx"] for d in w]
                assert g["image"].shape == (len(w), 1) + ROI
                for b in range(len(w)):
                    assert torch.equal(g["label"][b], w[b]["label"])
                    assert _rel(g["image"][b], w[b]["image"]) <= 1e-5, (seed, bs, b)
                    # the per-sample select runs behind the same chain call with and without it: its hits are exact.  The
                    # stage's chain takes its min / max on the way, so its output equals the plain stage's to rounding: the
                    # stage must hold the reference's min / 2, max / 2 at those hits and the plain chain everywhere else.
                    hit_ref = w[b]["image"] != wp[b]["image"]
                    assert hit_ref.any(), (seed, bs, b)
                    torch.testing.assert_close(g["image"][b][hit_ref], w[b]["image"][hit_ref], rtol=1e-4, atol=1e-6)
                    scale = float(gp["image"][b].abs().max())
                    assert float((g["image"][b] - gp["image"][b])[~hit_ref].abs().max()) <= 1e-5 * scale, (seed, bs, b)


@pytest.mark.gpu
def test_gpu_loader_without_a_generator_draws_as_a_dataloader(cuda_device):
    from torch.utils.data import DataLoader
    from mvtb.train_stage import DeviceCache, TrainStage
    from test_gpu_train_stage import _items, _tail
    cache = DeviceCache(_items(cuda_device), [], num_workers=2)
    stage = TrainStage(cache, _tail(0, rng="torch"), torch_generator=True)
    torch.manual_seed(9)
    got = [b["idx"] for b in stage.loader(2)]
    got_state = torch.get_rng_state()
    torch.manual_seed(9)
    ref = _tail(0, rng="torch")
    from test_gpu_train_stage import _per_sample
    want = []
    for batch in DataLoader(range(len(cache)), batch_size=2, shuffle=True, num_workers=0, collate_fn=list):
        want.append(list(batch))
        _per_sample(cache, ref, batch)
    assert got == want
    assert torch.equal(torch.get_rng_state(), got_state)
