"""Spacingd -> Orientationd on the GPU at the scripts' size against the oracle (torch affine_grid + grid_sample in float64 on
the CPU): labels equal, images within rtol 1e-6 / atol 1e-6 max|ref|, meta affines equal; the fused and windowed forms
equal the two-step result bit for bit."""
import numpy as np
import pytest
import torch

from oracle import monai_resample as O, ref_port as P

PIXDIM = (1.5, 1.5, 2.0)
LPS = np.diag([-1.0, -1.0, 1.0, 1.0]) @ np.array([[1, 0, 0, -120.0], [0, 1, 0, -120.0], [0, 0, 1, -77.0], [0, 0, 0, 1]])
SWAP = np.array([[0, 1.0, 0, 3], [-1.0, 0, 0, 5], [0, 0, 1.0, -7], [0, 0, 0, 1]])


def _close(got, want):
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6 * float(np.abs(want).max()))


def _sample(seed, affine, shape=(240, 240, 155)):
    img = P.synthetic_volume(seed, (4,) + shape).numpy()
    lab = (P.synthetic_volume(seed + 1, (3,) + shape).numpy() > 0.5).astype(np.float32)
    return {"image": img, "label": lab, "image_meta_dict": {"affine": affine.copy()}, "label_meta_dict": {"affine": affine.copy()}}


@pytest.mark.gpu
@pytest.mark.parametrize("affine", [np.eye(4), LPS, SWAP], ids=["identity", "lps", "swapped"])
def test_gpu_spacing_orientation_matches_oracle(cuda_device, affine):
    from mvtb import spatial as S
    d = _sample(30, affine)
    dev = dict(d, image=torch.from_numpy(d["image"]).to(cuda_device), label=torch.from_numpy(d["label"]).to(cuda_device),
               image_meta_dict=dict(d["image_meta_dict"]), label_meta_dict=dict(d["label_meta_dict"]))
    keys = ["image", "label"]
    out = S.Orientationd(keys, axcodes="RAS")(S.Spacingd(keys, PIXDIM, mode=("bilinear", "nearest"))(dev))
    for k, mode in (("image", "bilinear"), ("label", "nearest")):
        want, aff = O.spacing_orientation(d[k], affine, PIXDIM, "RAS", mode=mode)
        got = out[k]
        assert got.is_cuda and got.dtype == torch.float32
        if mode == "nearest":
            assert torch.equal(got.cpu(), torch.from_numpy(want))
        else:
            _close(got.cpu().numpy(), want)
        assert np.array_equal(out[f"{k}_meta_dict"]["affine"], aff)
    # one pass: the same bits and affines
    both = S.SpacingOrientationd(keys, PIXDIM, axcodes="RAS", mode=("bilinear", "nearest"))(
        dict(dev, image_meta_dict=dict(d["image_meta_dict"]), label_meta_dict=dict(d["label_meta_dict"])))
    for k in keys:
        assert torch.equal(both[k], out[k]) and np.array_equal(both[f"{k}_meta_dict"]["affine"], out[f"{k}_meta_dict"]["affine"])


@pytest.mark.gpu
def test_gpu_windowed_call_is_the_crop(cuda_device):
    """Spacingd -> Orientationd -> CenterSpatialCropd (the validation pipeline) as one gather, and a flipped window"""
    from mvtb import geometry as G, spatial as S
    d = _sample(40, LPS)
    x = torch.from_numpy(d["image"]).to(cuda_device)
    p = G.plan(LPS, x.shape[1:], PIXDIM, axcodes="RAS")
    full = S.resample(x, p, "bilinear")
    start, size = S.center_window(p.shape, (128, 128, 64))
    got = S.resample(x, p, "bilinear", window=(start, size))
    assert torch.equal(got, full[:, start[0]:start[0] + 128, start[1]:start[1] + 128, start[2]:start[2] + 64])
    assert torch.equal(S.CenterSpatialCropd("image", (128, 128, 64))({"image": full})["image"], got)
    got = S.resample(x, p, "bilinear", window=((5, 17, 3), (100, 90, 60)), flip_axes_mask=5)
    assert torch.equal(got, full[:, 5:105, 17:107, 3:63].flip(1).flip(3))


@pytest.mark.gpu
def test_gpu_oblique_takes_the_general_path(cuda_device):
    from mvtb import geometry as G, spatial as S
    c, s = np.cos(np.radians(10)), np.sin(np.radians(10))
    rot = np.array([[c, -s, 0, 3.0], [s, c, 0, -2.0], [0, 0, 1, 1.0], [0, 0, 0, 1]])
    shape = (120, 110, 60)
    d = _sample(50, rot, shape)
    p = G.plan(rot, shape, PIXDIM, diagonal=True)
    assert S.tap_tables(p, False) is None
    for k, mode in (("image", "bilinear"), ("label", "nearest")):
        want, aff = O.spacing(d[k], rot, PIXDIM, diagonal=True, mode=mode)
        got = S.Spacingd(k, PIXDIM, diagonal=True, mode=mode)({k: torch.from_numpy(d[k]).to(cuda_device),
                                                               f"{k}_meta_dict": {"affine": rot.copy()}})
        assert np.array_equal(got[f"{k}_meta_dict"]["affine"], aff)
        got = got[k].cpu().numpy()
        if mode == "bilinear":
            _close(got, want)
        else:
            coords = O.source_coords(shape, rot, PIXDIM, diagonal=True)
            tie = (np.abs(coords - np.floor(coords) - 0.5) < 1e-9).any(0)
            assert np.array_equal(got[:, ~tie], want[:, ~tie])


@pytest.mark.gpu
def test_gpu_inputs_come_back_in_their_own_kind(cuda_device):
    from mvtb import spatial as S
    x = P.synthetic_volume(60, (2, 40, 36, 31)).numpy()
    meta = lambda: {"affine": LPS.copy()}
    t = S.SpacingOrientationd("image", PIXDIM, axcodes="RAS")
    from_np = t({"image": x, "image_meta_dict": meta()})["image"]
    from_cpu = t({"image": torch.from_numpy(x), "image_meta_dict": meta()})["image"]
    from_dev = t({"image": torch.from_numpy(x).to(cuda_device), "image_meta_dict": meta()})["image"]
    assert isinstance(from_np, np.ndarray) and from_np.dtype == np.float32
    assert isinstance(from_cpu, torch.Tensor) and not from_cpu.is_cuda and from_cpu.dtype == torch.float32
    assert from_dev.is_cuda
    assert np.array_equal(from_np, from_cpu.numpy()) and torch.equal(from_cpu, from_dev.cpu())
    with pytest.raises(KeyError):
        t({"image": x})
