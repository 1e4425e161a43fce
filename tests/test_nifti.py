"""NIfTI loading (mvtb/nifti.py, csrc/nifti.cuh): header and affine known answers, error cases, the chunked gzip reader
against the gzip module, and the decode kernel through the DEBUG emulator against oracle/nifti_writer.decode_reference
for every datatype, both byte orders, scaled and unscaled, on shapes that do not fill the 32 x 32 tile."""
import ctypes as C
import gzip
import math
import shutil
import struct

import numpy as np
import pytest

from mvtb import _lib as B, nifti as N
from oracle import nifti_writer as W

emu_only = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++ for the emulator build")
LPS = np.array([[-1.0, 0, 0, 120.0], [0, -1.0, 0, 120.0], [0, 0, 1.0, -77.0]])


def _vol(dtype, shape, seed=0):
    """values spanning the type, incl. its extremes (float: values float32 cannot hold exactly)"""
    r = np.random.RandomState(seed)
    dt = np.dtype(dtype)
    if dt.kind == "f":
        x = r.standard_normal(shape) * 1e3
        if dt == np.float64:
            x = x + 1e-9
        return x.astype(dt)
    info = np.iinfo(dt)
    x = r.randint(info.min, info.max, size=shape, dtype=np.int64 if dt != np.uint32 else np.uint64).astype(dt)
    x.flat[0], x.flat[-1] = info.min, info.max
    if dt.itemsize == 4:
        x.flat[1] = (1 << 24) + 1                                   # rounds to nearest even in float32
    return x


def test_identity_sform(tmp_path):
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6), np.float32), sform=np.eye(4), pixdim=(2, 3, 4))
    h = N.read_header(p)
    assert np.array_equal(h.affine, np.eye(4)) and h.shape == (4, 5, 6) and h.vox_offset == 352 and h.version == 1


def test_lps_sform_nifti2_big_endian(tmp_path):
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6, 2), np.int16), sform=LPS, version=2, byteorder=">")
    h = N.read_header(p)
    assert h.version == 2 and h.byteorder == ">" and h.shape == (4, 5, 6, 2) and h.vox_offset == 544
    assert np.array_equal(h.affine[:3], LPS) and np.array_equal(h.affine[3], [0, 0, 0, 1])


def test_qform_qfac_minus_one(tmp_path):
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6), np.uint8), qform=(0, 0, 0, 1.5, -2.5, 3.0), pixdim=(2, 3, 4), qfac=-1)
    assert np.array_equal(N.read_header(p).affine, [[2, 0, 0, 1.5], [0, 3, 0, -2.5], [0, 0, -4, 3], [0, 0, 0, 1]])


def test_qform_90_degrees_about_z(tmp_path):
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6), np.uint8), qform=(0, 0, math.sqrt(0.5), 0, 0, 0), pixdim=(2, 3, 4))
    np.testing.assert_allclose(N.read_header(p).affine, [[0, -3, 0, 0], [2, 0, 0, 0], [0, 0, 4, 0], [0, 0, 0, 1]], atol=1e-6)


def test_qform_fixes_nibabel_makes_at_load(tmp_path):
    """qfac 0 reads as 1; negative pixdim reads as its absolute value"""
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6), np.uint8), qform=(0, 0, 0, 0, 0, 0), pixdim=(-2, 3, -4), qfac=0)
    h = N.read_header(p)
    assert np.array_equal(h.affine, np.diag([2.0, 3, 4, 1])) and h.pixdim[:4] == (1.0, 2.0, 3.0, 4.0)


def test_sform_wins_over_qform(tmp_path):
    p = W.write(tmp_path / "a.nii", np.zeros((4, 5, 6), np.uint8), qform=(0, 0, 0, 9, 9, 9), sform=LPS)
    assert np.array_equal(N.read_header(p).affine[:3], LPS)


def test_fallback_affine(tmp_path):
    p = W.write(tmp_path / "a.nii.gz", np.zeros((4, 5, 6, 3), np.float32), pixdim=(2, 3, 4), gzip_members=1)
    assert np.array_equal(N.read_header(p).affine, [[-2, 0, 0, 3], [0, 3, 0, -6], [0, 0, 4, -10], [0, 0, 0, 1]])


@pytest.mark.parametrize("chunk", [1, 7, 4096])
def test_header_straddles_chunks(tmp_path, chunk):
    p = W.write(tmp_path / "a.nii.gz", np.zeros((4, 5, 6), np.float32), sform=LPS, version=2, gzip_members=3,
                extensions=[(6, b"x" * 37), (4, b"y" * 100)])
    h = N.read_header(p, chunk)
    assert h.vox_offset == 544 + 48 + 112 and np.array_equal(h.affine[:3], LPS)


# ------------------------------------------------------------------ errors

def _nii(tmp_path, name="a.nii", data=None, **kw):
    return W.write(tmp_path / name, np.zeros((4, 5, 6), np.int16) if data is None else data, **kw)


def _read_all(p, chunk=4096):
    """header and payload through the chunked reader (the host half of load) into a ring of two bytearray chunks"""
    views = [memoryview(bytearray(chunk)) for _ in range(2)]
    got = bytearray()
    with N._Source(p) as src:
        h = N._header(src, chunk)
        N._read_payload(src, h, views, lambda slot: None, lambda slot, off, n: got.extend(views[slot][:n]))
    return h, bytes(got)


@pytest.mark.parametrize("kw,what", [
    (dict(magic=b"n+9\0"), "magic"),
    (dict(version=2, magic=b"n+9\0\r\n\x1a\n"), "magic"),
    (dict(vox_offset=300), "inside"),
    (dict(version=2, vox_offset=500), "inside"),
    (dict(payload=b"\0" * 239), "240 needed"),
])
def test_malformed_files_raise_value_error(tmp_path, kw, what):
    p = _nii(tmp_path, **kw)
    with pytest.raises(ValueError, match=what):
        _read_all(p)


def test_short_payload_names_path_and_counts(tmp_path):
    p = _nii(tmp_path, payload=b"\0" * 239)
    with pytest.raises(ValueError, match=r"a\.nii: 239 payload bytes .* 240 needed"):
        _read_all(p)


def test_truncated_and_garbled_files(tmp_path):
    p = tmp_path / "short.nii"
    p.write_bytes(open(_nii(tmp_path), "rb").read()[:200])
    with pytest.raises(ValueError, match="file ends .* into the header"):
        N.read_header(p)
    p.write_bytes(struct.pack("<i", 123) + b"\0" * 400)
    with pytest.raises(ValueError, match="sizeof_hdr"):
        N.read_header(p)
    gz = open(_nii(tmp_path, "b.nii.gz", gzip_members=1), "rb").read()
    p.write_bytes(gz[:len(gz) // 2])
    with pytest.raises(ValueError, match="ends inside a member"):
        _read_all(p)
    p.write_bytes(gz[:20] + bytes(b ^ 0x5A for b in gz[20:40]) + gz[40:])
    with pytest.raises(ValueError, match="gzip"):
        _read_all(p)
    p.write_bytes(gz + b"not gzip")                       # as the gzip module: garbage after a member is an error ...
    with pytest.raises(ValueError, match="gzip"), N._Source(p) as src:
        src.readinto(memoryview(bytearray(len(gz) * 100)))
    assert _read_all(p)[1] == b"\0" * 240                # ... once it is read: a load stops at the payload's end


@pytest.mark.parametrize("kw", [
    dict(magic=b"ni1\0"),
    dict(version=2, magic=b"ni2\0\r\n\x1a\n"),
    dict(data=np.zeros((4, 5), np.int16)),
    dict(data=np.zeros((4, 5, 6, 2, 2), np.int16)),
    dict(datatype=32),          # complex64
    dict(datatype=128),         # RGB
    dict(datatype=1024),        # int64
    dict(datatype=1536),        # float128
])
def test_unsupported_input_raises(tmp_path, kw):
    with pytest.raises(NotImplementedError):
        N.read_header(_nii(tmp_path, **kw))


def test_transform_options_no_script_uses_raise():
    with pytest.raises(NotImplementedError):
        N.LoadImaged("image", reader="ITKReader")
    with pytest.raises(NotImplementedError):
        N.LoadImaged("image", dtype=np.float64)
    N.LoadImaged("image", reader="NibabelReader")


def test_as_channel_first_numpy_is_monai_moveaxis():
    x = np.arange(24.0).reshape(2, 3, 4)
    assert np.array_equal(N.AsChannelFirstd("image")({"image": x})["image"], np.moveaxis(x, -1, 0))


# ------------------------------------------------------------------ the chunked reader

@pytest.mark.parametrize("members", [0, 1, 4])
@pytest.mark.parametrize("chunk", [1, 7, 4096])
def test_chunked_reader_matches_gzip(tmp_path, members, chunk):
    x = _vol(np.int16, (9, 7, 5, 2), 3)
    p = W.write(tmp_path / "a.nii.gz", x, gzip_members=members, level=1)
    blob = open(p, "rb").read()
    want = gzip.decompress(blob) if members else blob
    got = bytearray()
    buf = bytearray(chunk)
    with N._Source(p) as src:
        while True:
            k = src.readinto(memoryview(buf))
            got += buf[:k]
            if k < chunk:
                break
    assert bytes(got) == want


@pytest.mark.parametrize("chunk", [1, 7, 4096])
def test_header_and_payload_through_chunks(tmp_path, chunk):
    x = _vol(np.float32, (9, 7, 5), 4)
    p = W.write(tmp_path / "a.nii.gz", x, gzip_members=3, sform=LPS, extensions=[(4, b"z" * 21)])
    h, payload = _read_all(p, chunk)
    assert np.array_equal(h.affine[:3], LPS) and payload == x.astype("<f4").tobytes(order="F")


def test_chunked_reader_skips_zero_padding_between_members(tmp_path):
    p = tmp_path / "a.nii.gz"
    p.write_bytes(gzip.compress(b"abc") + b"\0" * 9 + gzip.compress(b"defg") + b"\0\0")
    with N._Source(p) as src:
        buf = bytearray(16)
        assert src.readinto(memoryview(buf)) == 7 and bytes(buf[:7]) == b"abcdefg"


# ------------------------------------------------------------------ the kernel through the emulator

SCALES = [(0.0, 0.0), (0.37, -2.5)]


def _emu_decode(p):
    from cuemu import emu
    L = emu.lib()
    h = N.read_header(p)
    blob = open(p, "rb").read()
    blob = gzip.decompress(blob) if blob[:2] == b"\x1f\x8b" else blob
    raw = np.frombuffer(blob, np.uint8, h.payload_bytes, h.vox_offset).copy()
    al = np.empty(raw.nbytes + 8, np.uint8)               # an 8-byte aligned copy
    a = al[(-al.ctypes.data) % 8:][:raw.nbytes]
    a[:] = raw
    out = np.full((h.channels,) + h.shape[:3], -7.0, np.float32)
    B.check(L, L.mvtb_nifti_decode_f32(emu.ptr(a), emu.ptr(out), *N.decode_args(h), None))
    return out


@emu_only
@pytest.mark.parametrize("shape", [(33, 17, 9, 2), (5, 3, 2)])
@pytest.mark.parametrize("scale", SCALES, ids=["raw", "scaled"])
@pytest.mark.parametrize("order", "<>")
@pytest.mark.parametrize("code", sorted(W.DTYPES))
def test_emulated_decode_matches_reference(tmp_path, code, order, scale, shape):
    x = _vol(W.DTYPES[code], shape, code)
    p = W.write(tmp_path / "a.nii", x, byteorder=order, slope=scale[0], inter=scale[1], version=len(shape) - 2)
    want = W.decode_reference(p)
    if not scale[0]:
        assert np.array_equal(want, (np.moveaxis(x, 3, 0) if len(shape) == 4 else x[None]).astype(np.float32))
    assert np.array_equal(_emu_decode(p), want)


@emu_only
@pytest.mark.parametrize("slope,inter,scaled", [(float("nan"), 3.0, False), (np.inf, 3.0, False), (0.0, 3.0, False),
                                                (1.0, 0.0, False), (2.0, float("inf"), True), (1.0, 0.5, True)])
def test_emulated_decode_value_rule_edges(tmp_path, slope, inter, scaled):
    x = _vol(np.int32, (6, 4, 3), 9)
    p = W.write(tmp_path / "a.nii", x, slope=slope, inter=inter)
    want = W.decode_reference(p)
    assert N.value_rule(N.read_header(p))[0] == scaled
    if not scaled:
        assert np.array_equal(want, x[None].astype(np.float32))
    assert np.array_equal(_emu_decode(p), want)


def test_reference_value_rule_known_answers(tmp_path):
    x = np.array([1 << 24 | 1, 3, -(1 << 24) - 3], np.int32).reshape(3, 1, 1)
    p = W.write(tmp_path / "a.nii", x)
    assert W.decode_reference(p).ravel().tolist() == [16777216.0, 3.0, -16777220.0]          # nearest even
    p = W.write(tmp_path / "b.nii", np.array([3], np.int16).reshape(1, 1, 1), slope=0.1, inter=0.2)
    assert W.decode_reference(p).ravel()[0] == np.float32(np.float32(3) * np.float32(0.1)) + np.float32(0.2)


@emu_only
def test_emulated_decode_rejects_bad_arguments():
    from cuemu import emu
    L = emu.lib()
    raw = np.zeros(64, np.float64)
    out = np.zeros(64, np.float32)
    i64 = C.c_int64 * 4

    def call(src=raw.ctypes.data, dst=out.ctypes.data, dt=16, dims=(2, 2, 2, 1)):
        return L.mvtb_nifti_decode_f32(C.c_void_p(src), C.c_void_p(dst), dt, 0, None if dims is None else i64(*dims), 1.0, 0.0, 0, None)

    assert call() == B.MVTB_OK
    assert call(src=None) == B.MVTB_EINVAL
    assert call(dst=None) == B.MVTB_EINVAL
    assert call(dims=None) == B.MVTB_EINVAL
    assert call(dst=raw.ctypes.data) == B.MVTB_EINVAL                                   # in place
    assert call(dt=32) == B.MVTB_EUNSUPPORTED                                           # complex64
    assert call(dt=1024) == B.MVTB_EUNSUPPORTED                                         # int64
    assert call(dims=(2, 0, 2, 1)) == B.MVTB_EINVAL
    assert call(dims=(2, 2, 2, -1)) == B.MVTB_EINVAL
    assert call(dims=(1 << 16, 1 << 15, 2, 1)) == B.MVTB_EINVAL                         # 2^32 voxels per channel
    assert call(src=raw.ctypes.data + 2) == B.MVTB_EINVAL                               # float32 payload not 4-byte aligned
    assert "aligned" in B.last_error(L)
    assert call(src=raw.ctypes.data + 2, dt=4) == B.MVTB_OK                             # int16 at 2 bytes is fine
