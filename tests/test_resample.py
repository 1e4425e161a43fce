"""Spacingd -> Orientationd (SURVEY 8(f) rank 4): the MONAI 0.5 / nibabel geometry restatement against known answers, the
per-axis tables against torch's full affine_grid, and the gather kernel through the DEBUG emulator against the oracle
(oracle/monai_resample.py: torch affine_grid + grid_sample in float64)."""
import ctypes as C
import shutil

import numpy as np
import pytest
import torch

from mvtb import _lib as B, geometry as G, spatial as S
from oracle import monai_resample as O, ref_port as P

emu_only = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++ for the emulator build")

SWAP = np.array([[0, 1.2, 0, 3], [-0.9, 0, 0, 5], [0, 0, 1.1, -7], [0, 0, 0, 1]])       # voxel axes 0 and 1 swapped


def test_spacing_scripts_geometry():
    sp = G.spacing(np.eye(4), (240, 240, 155), (1.5, 1.5, 2.0))
    assert sp.shape == (160, 160, 78) and not sp.identity
    assert np.array_equal(sp.affine, np.diag([1.5, 1.5, 2.0, 1.0]))             # offset 0: same orientation, origin 0
    assert np.array_equal(sp.transform, np.diag([1.5, 1.5, 2.0, 1.0]))


def test_io_orientation_known_answers():
    assert np.array_equal(G.io_orientation(np.diag([2.0, 3, 4, 1])), [[0, 1], [1, 1], [2, 1]])
    a = np.array([[0, 1, 0, 0], [-1, 0, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]])     # first voxel axis along -y
    assert np.array_equal(G.io_orientation(a), [[1, -1], [0, 1], [2, 1]])
    assert np.array_equal(G.axcodes2ornt("RAS"), [[0, 1], [1, 1], [2, 1]])
    assert np.array_equal(G.axcodes2ornt("LPS"), [[0, -1], [1, -1], [2, 1]])


def test_orientation_flips_and_transposes():
    ornt, shape, aff = G.orientation(np.diag([-1.0, -1, 1, 1]), (4, 5, 6), "RAS")
    assert np.array_equal(ornt, [[0, -1], [1, -1], [2, 1]]) and shape == (4, 5, 6)
    assert np.allclose(aff, np.array([[1, 0, 0, -3], [0, 1, 0, -4], [0, 0, 1, 0], [0, 0, 0, 1.0]]))
    x = np.arange(120.0).reshape(1, 4, 5, 6)
    got, _ = O.orientation(x, np.diag([-1.0, -1, 1, 1]), "RAS")
    assert np.array_equal(got, x[:, ::-1, ::-1, :])
    ornt, shape, aff = G.orientation(SWAP, (4, 5, 6), "RAS")
    assert np.array_equal(ornt, [[1, -1], [0, 1], [2, 1]]) and shape == (5, 4, 6)
    got, _ = O.orientation(x, SWAP, "RAS")
    assert np.array_equal(got, np.transpose(x[:, ::-1], (0, 2, 1, 3)))
    # the new affine maps the reoriented voxel to the same world point
    w = SWAP @ [3, 1, 2, 1]
    assert np.allclose(aff @ [1, 0, 2, 1], w)


def test_identity_spacing_copies():
    sp = G.spacing(np.eye(4), (6, 7, 8), (1.0005, 1.0, 1.0))
    assert sp.identity and sp.shape == (6, 7, 8)
    x = P.synthetic_volume(1, (2, 6, 7, 8)).numpy().astype(np.float64)
    got, _ = O.spacing(x, np.eye(4), (1.0005, 1.0, 1.0))
    assert got.dtype == np.float32 and np.array_equal(got, x.astype(np.float32))
    tg, parts = G.axis_taps(G.plan(np.eye(4), (6, 7, 8), (1.0005, 1.0, 1.0)), False)
    assert all(np.array_equal(parts[k]["i0"], np.arange(n)) for k, n in enumerate((6, 7, 8)))


def test_nearest_tie_follows_torch():
    """1.5 o on the H axis: torch's float64 grid puts odd o just off the half-integer; o = 5 lands on 7.499999999999998"""
    tg, parts = G.axis_taps(G.plan(np.eye(4), (240, 240, 155), (1.5, 1.5, 2.0), axcodes="RAS"), True)
    assert tg == [0, 1, 2] and parts[0]["i0"][5] == 7 and parts[0]["i0"][1] == 2 and parts[0]["i0"][3] == 4


@pytest.mark.parametrize("shape,pixdim,affine,diagonal", [
    ((240, 240, 155), (1.5, 1.5, 2.0), np.eye(4), False),
    ((161, 97, 33), (1.5, 0.7, 2.0), np.array([[1.0, 0, 0, 4.5], [0, 1, 0, -2], [0, 0, 1, 3], [0, 0, 0, 1]]), False),
    ((17, 13, 11), (1.5, 0.7, 2.0), np.diag([-1.0, -1, 1, 1]), False),
    ((31, 23, 19), (1.5, 1.5, 2.0), SWAP, True),                                  # a permuted transform
])
def test_axis_tables_equal_the_full_grid(shape, pixdim, affine, diagonal):
    p = G.plan(affine, shape, pixdim, diagonal)
    full = O.source_coords(shape, affine, pixdim, diagonal)
    for nearest in (True, False):
        tg, parts = G.axis_taps(p, nearest)
        for k in range(3):
            ix = np.minimum(shape[k] - 1.0, np.maximum(full[k], 0.0))
            lines = np.moveaxis(ix, tg[k], -1).reshape(-1, ix.shape[tg[k]])
            assert (lines == lines[:1]).all()                                    # depends on one grid axis only
            want = np.rint(lines[0]) if nearest else np.floor(lines[0])
            assert np.array_equal(parts[k]["i0"], want)
            if not nearest:
                assert np.array_equal(parts[k]["w1"], (lines[0] - want).astype(np.float32))
    if diagonal:
        assert G.axis_taps(p, True)[0] == [1, 0, 2]


def test_oblique_transform_has_no_tables():
    c, s = np.cos(np.radians(10)), np.sin(np.radians(10))
    rot = np.array([[c, -s, 0, 0], [s, c, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]])
    assert G.axis_taps(G.plan(rot, (20, 18, 9), (1.5, 1.5, 2.0), diagonal=True), False) is None


def test_options_no_script_uses_raise():
    with pytest.raises(NotImplementedError):
        S.Spacingd("image", (1.5, 1.5, 2.0), padding_mode="zeros")
    with pytest.raises(NotImplementedError):
        S.Spacingd("image", (1.5, 1.5, 2.0), align_corners=True)
    with pytest.raises(NotImplementedError):
        S.Spacingd(["image", "label"], (1.5, 1.5, 2.0), mode=("bilinear", "bicubic"))
    with pytest.raises(ValueError):
        S.Spacingd(["image", "label"], (1.5, 1.5, 2.0), mode=("bilinear",))


# ------------------------------------------------------------------ the kernel through the emulator

def _emu_resample(x, p, mode, window=None, flip=0, general=False):
    from cuemu import emu
    L = emu.lib()
    nearest = mode == "nearest"
    taps = None if general else S.tap_tables(p, nearest)
    tap_arr = None if taps is None else np.ascontiguousarray(taps[2])
    g, size = S.resample_geom(p, nearest, window, flip, taps, 0 if taps is None else tap_arr.ctypes.data)
    out = np.full((x.shape[0],) + size, -7.0, dtype=np.float32)
    B.check(L, L.mvtb_resample_f32(emu.ptr(x), emu.ptr(out), x.shape[0], C.byref(g), None))
    return out


def _close(got, want):
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6 * float(np.abs(want).max()))


CASES = [  # affine, axcodes, window (start, size) or None, flip mask
    (np.eye(4), "RAS", None, 0),
    (np.diag([-1.0, -1, 1, 1]), "RAS", ((1, 2, 0), (9, 12, 5)), 5),
    (SWAP, "RAS", ((2, 0, 1), (8, 9, 5)), 2),
    (np.diag([1.0, -1, 1, 1]), "LPS", None, 7),
]


@emu_only
@pytest.mark.parametrize("affine,axcodes,window,flip", CASES)
def test_emulated_kernel_matches_the_oracle(affine, axcodes, window, flip):
    shape, pixdim = (2, 17, 13, 11), (1.5, 0.7, 2.0)
    x = P.synthetic_volume(3, shape).numpy()
    lab = (P.synthetic_volume(4, shape).numpy() > 0.4).astype(np.float32)
    p = G.plan(affine, shape[1:], pixdim, axcodes=axcodes)
    assert S.tap_tables(p, False) is not None
    def crop_flip(a):
        if window is not None:
            a = a[(slice(None),) + tuple(slice(s, s + n) for s, n in zip(*window))]
        for ax in range(3):
            if flip >> ax & 1:
                a = np.flip(a, ax + 1)
        return a

    # voxels whose source coordinate is a half-integer on some axis: there the fp64 matrix may round the other way
    coords = O.source_coords(shape[1:], affine, pixdim)
    tie = (np.abs(coords - np.floor(coords) - 0.5) < 1e-9).any(0).astype(np.float32)[None]
    tie = crop_flip(O.orientation(tie, p.spacing.affine, axcodes)[0])[0] > 0
    for img, mode in ((x, "bilinear"), (lab, "nearest")):
        want, aff = O.spacing_orientation(img, affine, pixdim, axcodes, mode=mode)
        assert np.array_equal(aff, p.affine)
        want = crop_flip(want)
        got = _emu_resample(img, p, mode, window, flip)
        gen = _emu_resample(img, p, mode, window, flip, general=True)
        if mode == "nearest":
            assert np.array_equal(got, want)
            assert tie.any() and np.array_equal(gen[:, ~tie], want[:, ~tie])
        else:
            _close(got, want)
            _close(gen, want)


@emu_only
def test_emulated_general_path_oblique():
    c, s = np.cos(np.radians(10)), np.sin(np.radians(10))
    rot = np.array([[c, -s, 0, 2], [s, c, 0, -1], [0, 0, 1, 0], [0, 0, 0, 1.0]])
    x = P.synthetic_volume(5, (1, 15, 12, 9)).numpy()
    p = G.plan(rot, (15, 12, 9), (1.5, 0.7, 2.0), diagonal=True)
    assert S.tap_tables(p, False) is None
    want, _ = O.spacing(x, rot, (1.5, 0.7, 2.0), diagonal=True)
    _close(_emu_resample(x, p, "bilinear"), want)


@emu_only
def test_emulated_kernel_rejects_bad_arguments():
    from cuemu import emu
    L = emu.lib()
    x = np.zeros((1, 8, 8, 8), dtype=np.float32)
    out = np.zeros((1, 4, 4, 4), dtype=np.float32)
    p = G.plan(np.eye(4), (8, 8, 8), (2.0, 2.0, 2.0))
    taps = S.tap_tables(p, False)
    arr = np.ascontiguousarray(taps[2])

    def call(src=x, dst=out, n=1, **kw):
        g, _ = S.resample_geom(p, False, None, 0, taps, arr.ctypes.data)
        for k, v in kw.items():
            setattr(g, k, v)
        return L.mvtb_resample_f32(emu.ptr(src), emu.ptr(dst), n, C.byref(g), None)

    i3 = C.c_int32 * 3
    assert call() == B.MVTB_OK
    assert call(dst=x) == B.MVTB_EINVAL                                             # in place
    assert call(n=-1) == B.MVTB_EINVAL
    assert call(mode=2) == B.MVTB_EINVAL
    assert call(axis=i3(0, 0, 2)) == B.MVTB_EINVAL                                  # not a permutation
    assert call(step=i3(1, 2, 1)) == B.MVTB_EINVAL
    assert call(base=i3(1, 0, 0)) == B.MVTB_EINVAL                                  # 1 + 3 leaves the grid of 4
    assert call(n_taps=11) == B.MVTB_EINVAL                                         # tables shorter than the grid
    assert call(tap_grid=i3(0, 1, 1)) == B.MVTB_EINVAL
    assert call(in_shape=i3(8, 0, 8)) == B.MVTB_EINVAL
    assert L.mvtb_resample_f32(emu.ptr(x), emu.ptr(out), 1, None, None) == B.MVTB_EINVAL
