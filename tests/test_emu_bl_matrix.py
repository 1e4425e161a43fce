"""Band-limited chain over every NF bucket, run through the DEBUG emulator, against the float64 reference of
oracle/bl_matrix.py.

The emulator runs the CUDA-core H-axis kernels (its profile names every forward variant k_bl_fwd_h and every
inverse k_bl_inv_h) and both forms of the W/D stage; the fused inverse + select and the tensor-core kernels exist
only in the CUDA build and are covered by tests/test_gpu_bl_matrix.py with the same case table.  Every case asserts
which kernels ran, because a shape the band-limited path does not take silently runs the general FFT path and still
gives the right numbers.

Regression: D = 2F + 1 (the kept box spans the whole last axis) made the fused W/D kernel k_bl_midw overwrite its
D-axis twiddles with the bins of the way back; every such case here failed at rel-L2 ~ 0.9."""
import ctypes as C
import shutil

import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++ for the emulator build")

from cuemu import emu  # noqa: E402
from mvtb import _lib as B, host  # noqa: E402
from oracle import bl_matrix as M, ref_port as P  # noqa: E402

REL_L2 = 1e-5        # image domain, the project's bar
BIN = 2e-5           # any k-space bin, relative to the RMS of the reference's nonzero bins


def white(seed, shape):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float32).numpy()


def matrix_inputs(case):
    x, spec = M.inputs(case)
    assert spec[1] == host.disk_threshold(M.disk_radius(case.F), case.shape)
    kind, thr, sp, alphas = spec
    descs = [host.make_desc(mask_kind=B.MASK_DISK, mask_ndim=3, mask_thresh=thr, spikes=s, wrap_alpha=a) for s, a in zip(sp, alphas)]
    return x, descs, spec


_refs = {}


def reference(case, x, spec, abt=None):
    key = (case, abt is not None)
    if key not in _refs:
        kind, thr, sp, alphas = spec
        _refs[key] = M.chain_ref(x, kind, thr, sp, alphas, abt)
    return _refs[key]


def run(x, descs, path, abt=None, vps=1):
    L = emu.lib()
    plan = emu.Plan(x.shape[-3:], 4)
    B.check(L, L.mvtb_plan_set_path(plan.h, path))
    B.check(L, L.mvtb_plan_profile(plan.h, 1))
    nvol = x.shape[0]
    y = np.empty_like(x)
    mm = np.zeros(2 * nvol // vps, dtype=np.float32)
    arr = host.desc_array(descs)
    if abt is None:
        B.check(L, L.mvtb_kspace_chain_f32(plan.h, emu.ptr(x), emu.ptr(y), nvol, arr, len(descs), emu.ptr(mm), vps, None))
    else:
        B.check(L, L.mvtb_kspace_chain_ex_f32(plan.h, emu.ptr(x), emu.ptr(y), nvol, arr, len(descs), emu.ptr(abt),
                                              emu.ptr(mm), vps, None, None))
    ms, cn = (C.c_double * B.K_KINDS)(), (C.c_int * B.K_KINDS)()
    B.check(L, L.mvtb_plan_profile_read(plan.h, ms, cn))
    kinds = {L.mvtb_kernel_name(k).decode() for k in range(B.K_KINDS) if cn[k]}
    return y, mm.reshape(-1, 2), kinds


def expected_kinds(case, path):
    if not case.bl:
        return M.GENERAL_KINDS
    # the profile names every CUDA-core forward k_bl_fwd_h and every inverse k_bl_inv_h (bandlimited.cu:1031, 1251)
    return {"k_bl_fwd_h", "k_bl_inv_h"} | (M.BL_KINDS_SPLIT if path == 3 else M.BL_KINDS_MID)


def check_numbers(y, ref, mm=None, vps=1):
    l2, b = M.errors(y, ref)
    assert l2 <= REL_L2, f"rel-L2 {l2:.3e}"
    assert b <= BIN, f"worst bin {b:.3e} of the kept bins' RMS"
    if mm is not None:
        ys = y.reshape(mm.shape[0], -1)
        assert np.array_equal(mm[:, 0], ys.min(axis=1)) and np.array_equal(mm[:, 1], ys.max(axis=1))
    return l2, b


# ------------------------------------------------------------------------------------------------ the reference


@pytest.mark.parametrize("shape,r,idx,intensity,alpha", [((1, 16, 12, 9), 3.5, (9, 7, 4), 9.0, 0.5),         # spike in the ball
                                                         ((2, 15, 14, 11), 4.5, (2, 13, 1), 11.0, 0.25),     # on a masked bin
                                                         ((1, 20, 9, 10), 2.5, (10, 4, 5), 8.0, 1.0)])       # the DC bin
def test_reference_matches_chain_127_exact_phase(shape, r, idx, intensity, alpha):
    x = white(7, shape)
    want = P.chain_127_exact_phase(torch.from_numpy(x), r, idx, intensity, alpha).numpy()
    thr = host.disk_threshold(r, shape[-3:])
    amp = float(np.exp(np.float64(intensity)))
    got = M.chain_ref(x, M.MASK_DISK, thr, [[(idx, amp)]] * shape[0], alpha)
    assert rel_l2(got, want) <= 1e-12


@pytest.mark.parametrize("shape,alpha", [((2, 16, 12, 8), 0.8), ((1, 15, 13, 9), 0.7), ((1, 9, 15, 7), 0.75), ((1, 20, 18, 15), 0.9)])
def test_reference_matches_gibbs_noise(shape, alpha):
    x = white(8, shape)
    want = P.gibbs_noise(torch.from_numpy(x).double(), alpha).numpy()
    got = M.chain_ref(x, M.MASK_CENTRED, host.gibbs_threshold(alpha, shape[1:]))
    assert rel_l2(got, want) <= 1e-12
    assert np.abs(got).max() > 0


def test_reference_prologue_map():
    x = white(9, (2, 8, 6, 5))
    x[:, 0] = 0.0
    abt = np.array([[1.5, -0.25, 0.75], [0.5, 2.0, -1.0]])
    mapped = np.where(x != 0, abt[:, 0, None, None, None] * x + abt[:, 1, None, None, None], abt[:, 2, None, None, None])
    got = M.chain_ref(x, M.MASK_DISK, 10 ** 6, abt=abt)                  # a mask that keeps every bin: the identity
    assert rel_l2(got, mapped) <= 1e-13


def test_case_table_covers_every_bucket_edge():
    fs = M.bucket_ends()
    assert fs == (0, 3, 4, 7, 8, 12, 13, 15, 16, 19, 20, 25, 26, 31)
    assert {M.nf_bucket(F) for F in fs} == set(M.BUCKETS)
    for c in M.cases():
        H, W, D = c.shape
        assert max(c.shape) <= 70
        if c.bl:
            assert H >= 2 * c.NF - 1 and min(W, D) >= 2 * c.F + 1
        else:
            assert H == 2 * c.NF - 2 or W == 2 * c.F
    kinds = {c.kind: c for c in M.cases() if c.F == 31}
    assert kinds["tc"].shape[0] % 16 == 0 and (kinds["tc"].shape[1] * kinds["tc"].shape[2]) % 4 == 0
    assert kinds["quad"].shape[0] % 4 == 0 and kinds["quad"].shape[0] % 16 != 0
    assert kinds["h2"].shape[0] % 4 == 2 and kinds["odd"].shape[0] % 2 == 1


# ------------------------------------------------------------------------------------------------ the matrix


def _matrix_params():
    """Path 0 on every case; path 2 (pair kernels) where it differs, on band-limited shapes with H % 4 == 0; path 3
    (the three-kernel W/D stage, independent of H) on two shapes per F, one of them with D = 2F + 1."""
    out = []
    for c in M.cases():
        for path, name in ((0, "auto"), (2, "pairs"), (3, "split")):
            if path and not c.bl or path == 2 and c.shape[0] % 4 or path == 3 and c.kind not in ("tc", "h2"):
                continue
            out.append(pytest.param(c, path, id=f"{c.id}-{name}"))
    return out


@pytest.mark.parametrize("case,path", _matrix_params())
def test_emu_matrix(case, path):
    x, descs, spec = matrix_inputs(case)
    y, mm, kinds = run(x, descs, path)
    assert kinds == expected_kinds(case, path)
    check_numbers(y, reference(case, x, spec), mm)


@pytest.mark.parametrize("case", M.cases(("quad", "h2", "fb_h")), ids=lambda c: c.id)
def test_emu_matrix_prologue(case):
    """mvtb_kspace_chain_ex_f32 with the intensity map: the emulator's forward kernel never applies it, so the
    separate affine pass runs into `out` first (bandlimited.cu:1074); some voxels are 0 to take the `t` branch."""
    x, descs, spec = matrix_inputs(case)
    x[:, :, 0, :] = 0.0
    # near-zero b, as NormalizeIntensity makes it: a large DC bin would dominate the kept bins' RMS
    abt = np.array([[1.75, -0.05, 0.25], [0.5, 0.03, -0.2]], dtype=np.float32)
    y, mm, kinds = run(x, descs, 0, abt=abt)
    assert kinds == expected_kinds(case, 0)
    kind, thr, sp, alphas = spec
    check_numbers(y, M.chain_ref(x, kind, thr, sp, alphas, abt), mm)


@pytest.mark.parametrize("F", [F for F in M.bucket_ends() if F > 0])
def test_emu_matrix_centred_mask(F):
    """A centred (GibbsNoise) mask sized to keep |f| <= F exactly: M_eff is 1/2 on the box faces of the even axes."""
    shape = M.shape_for(F, "quad")
    thr = M.centred_threshold(F)
    x = white(2000 + F, (2,) + shape)
    d = host.make_desc(mask_kind=B.MASK_CENTRED, mask_ndim=3, mask_thresh=thr)
    y, mm, kinds = run(x, [d], 0)
    assert kinds == expected_kinds(M.Case(F, "quad", shape, True), 0)
    check_numbers(y, M.chain_ref(x, M.MASK_CENTRED, thr), mm)
