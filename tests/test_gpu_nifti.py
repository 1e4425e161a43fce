"""mvtb.nifti.load on the GPU against oracle/nifti_writer.decode_reference (torch.equal) over every datatype, byte order,
scaling and container, and the scripts' loading pipeline at BraTS size against the host path:
    LoadImaged -> AsChannelFirstd -> ConvertToMultiChannelBasedOnBratsClassesd -> SpacingOrientationd
    decode_reference -> np.moveaxis -> numpy ConvertToMultiChannelBasedOnBratsClassesd -> the same SpacingOrientationd
plus concurrent loads from several threads."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from oracle import nifti_writer as W, ref_port as P

LPS = np.array([[-1.0, 0, 0, 120.0], [0, -1.0, 0, 120.0], [0, 0, 1.0, -77.0]])
PIXDIM = (1.5, 1.5, 2.0)


def _vol(code, shape, seed):
    r = np.random.RandomState(seed)
    dt = np.dtype(W.DTYPES[code])
    if dt.kind == "f":
        return (r.standard_normal(shape) * 1e3 + 1e-9).astype(dt)
    info = np.iinfo(dt)
    x = r.randint(info.min, info.max, size=shape, dtype=np.uint64 if dt == np.uint32 else np.int64).astype(dt)
    x.flat[0], x.flat[-1] = info.min, info.max
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(33, 17, 9, 2), (5, 3, 2), (240, 37, 155)])
@pytest.mark.parametrize("code", sorted(W.DTYPES))
def test_gpu_load_matches_reference(cuda_device, tmp_path, code, shape):
    from mvtb import nifti as N
    x = _vol(code, shape, code)
    for n, (order, scale, members, chunk) in enumerate([("<", (0.0, 0.0), 0, 4 << 20), (">", (0.37, -2.5), 2, 7),
                                                         ("<", (1.5, 4.0), 1, 4096), (">", (0.0, 0.0), 0, 1000)]):
        p = W.write(tmp_path / f"a{n}.nii", x, byteorder=order, slope=scale[0], inter=scale[1], gzip_members=members,
                    version=1 + n % 2, sform=LPS, level=1)
        got, h = N.load(p, _chunk_bytes=chunk)
        want = torch.from_numpy(W.decode_reference(p))
        assert got.is_cuda and got.dtype == torch.float32 and got.is_contiguous() and got.shape == want.shape
        assert torch.equal(got.cpu(), want), (order, scale, members)
        assert np.array_equal(h.affine[:3], LPS)


def _brats(tmp_path):
    img = P.synthetic_volume(70, (4, 240, 240, 155)).numpy()
    lab = np.zeros((240, 240, 155), np.uint8)
    r = np.random.RandomState(5)
    lab[60:180, 50:190, 30:120] = r.randint(0, 4, size=(120, 140, 90))
    ip = W.write(tmp_path / "img.nii.gz", np.moveaxis(img, 0, -1), sform=LPS, gzip_members=1, level=1)
    lp = W.write(tmp_path / "seg.nii.gz", lab, sform=LPS, gzip_members=1, level=1)
    return str(ip), str(lp)


@pytest.mark.gpu
def test_gpu_brats_pipeline_equals_host_path(cuda_device, tmp_path):
    import filters_and_operators as F
    from mvtb import nifti as N, spatial as S
    ip, lp = _brats(tmp_path)
    keys = ["image", "label"]
    resample = S.SpacingOrientationd(keys, PIXDIM, axcodes="RAS", mode=("bilinear", "nearest"))

    d = N.LoadImaged(keys)({"image": ip, "label": lp})
    assert d["image"].shape == (240, 240, 155, 4) and d["label"].shape == (240, 240, 155)
    assert d["image_meta_dict"]["filename_or_obj"] == ip and list(d["label_meta_dict"]["spatial_shape"]) == [240, 240, 155]
    d = N.AsChannelFirstd("image")(d)
    assert d["image"].is_contiguous() and d["image"].shape == (4, 240, 240, 155)
    d = F.ConvertToMultiChannelBasedOnBratsClassesd("label")(d)
    assert d["label"].is_cuda and d["label"].dtype == torch.float32
    gpu = resample(d)

    img = np.moveaxis(W.decode_reference(ip), 0, -1)            # MONAI's (X, Y, Z, C)
    h = {"image": np.moveaxis(img, -1, 0), "label": W.decode_reference(lp)[0],
         "image_meta_dict": {"affine": d["image_meta_dict"]["original_affine"].copy()},
         "label_meta_dict": {"affine": d["label_meta_dict"]["original_affine"].copy()}}
    h = F.ConvertToMultiChannelBasedOnBratsClassesd("label")(h)
    host = resample(h)
    for k in keys:
        assert torch.equal(gpu[k].cpu(), torch.from_numpy(host[k])), k
        assert np.array_equal(gpu[f"{k}_meta_dict"]["affine"], host[f"{k}_meta_dict"]["affine"])
    assert gpu["image"].shape == (4, 160, 160, 78) and gpu["label"].shape == (3, 160, 160, 78)


@pytest.mark.gpu
def test_gpu_concurrent_loads_equal_sequential(cuda_device, tmp_path):
    from mvtb import nifti as N
    paths = []
    for n in range(8):
        code = sorted(W.DTYPES)[n]
        paths.append(W.write(tmp_path / (f"v{n}.nii" + (".gz" if n % 2 else "")), _vol(code, (96, 80, 40, 2), n),
                             byteorder="<>"[n % 2], slope=0.5 * (n % 3), inter=1.0, gzip_members=n % 3, level=1))
    seq = [N.load(p, _chunk_bytes=64 << 10)[0] for p in paths]

    def one(p):
        out = N.load(p, _chunk_bytes=64 << 10)[0]
        torch.cuda.current_stream().synchronize()
        return out

    with ThreadPoolExecutor(8) as ex:
        par = list(ex.map(one, paths))
    torch.cuda.synchronize()
    for a, b, p in zip(seq, par, paths):
        assert torch.equal(a, b), p
        assert torch.equal(a.cpu(), torch.from_numpy(W.decode_reference(p))), p
