"""Every band-limited kernel variant at every NF bucket against the float64 reference of oracle/bl_matrix.py.

`bl_chain` instantiates `bl_run<NF>` for NF in {4, 8, 13, 16, 20, 26, 32}, and `bl_run` picks its H-axis kernels
from the shape, the pointer alignment, W*D and the plan options.  The case table takes F at both ends of every
bucket (and F = 0) and, per F, shapes that select each variant; the variants are driven by the plan's path
(mvtb_plan_set_path 0 / 2 / 3 / 4 / 5), the options read at plan creation (MVTB_NO_ASYNC, MVTB_NO_FUSEMID,
MVTB_NO_FUSESP, MVTB_TC_INV) and input or output views one float off 16-byte alignment.  Every call asserts the
kernel kinds it expects, because a shape the band-limited path does not take runs the general FFT path silently
and still gives the right numbers.

Checks: image-domain rel-L2 <= 1e-5 and, over all bins, max |FFT(y) - FFT(ref)| <= 2e-5 x RMS(nonzero bins of
ref); the per-sample (min, max) bit-equal to y's; the fused select bit-equal to the chain followed by the sparse
select; tensor cores against CUDA cores at rel-L2 <= 5e-6; no tensor-core kernel gave up a wait."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import rel_l2
from oracle import bl_matrix as M

pytestmark = pytest.mark.gpu

REL_L2 = 1e-5
BIN = 2e-5
TC_VS_CC = 5e-6
ENVS = ("MVTB_NO_ASYNC", "MVTB_NO_FUSEMID", "MVTB_NO_FUSESP", "MVTB_TC_INV")
PATHS = {"auto": 0, "pairs": 2, "split": 3, "cc": 4, "tc": 5}

_worst = {}          # NF -> [rel-L2, bin error]: printed at the end of the module (pytest -s)


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if _worst:
        print("\nband-limited matrix, worst errors per NF bucket (rel-L2, bin error / RMS of the kept bins):")
        for nf in sorted(_worst):
            print(f"  NF {nf:2d}: {_worst[nf][0]:.3e}  {_worst[nf][1]:.3e}")


@pytest.fixture
def env(monkeypatch):
    """Sets plan-creation options; plans are destroyed before and after, so that the options take effect and end."""
    from mvtb import functional as Fn

    def set_(**kv):
        for k in ENVS:
            monkeypatch.delenv(k, raising=False)
        for k, v in kv.items():
            monkeypatch.setenv(k, str(v))
        Fn._destroy_plans()
    yield set_
    Fn._destroy_plans()


def descs_for(spec):
    from mvtb import _lib, host
    kind, thr, sp, alphas = spec
    return [host.make_desc(mask_kind=_lib.MASK_DISK if kind == M.MASK_DISK else _lib.MASK_CENTRED, mask_ndim=3,
                           mask_thresh=thr, spikes=s, wrap_alpha=a) for s, a in zip(sp, alphas)]


def inputs(case):
    x, spec = M.inputs(case)
    return x, spec, descs_for(spec)


_refs = {}


def reference(case, x, spec, abt=None):
    key = (case, None if abt is None else abt.tobytes())
    if key not in _refs:
        _refs[key] = M.chain_ref(x, *spec, abt=abt)
    return _refs[key]


def check(case, y, ref, mm=None):
    y = y.cpu().numpy()
    l2, b = M.errors(y, ref)
    w = _worst.setdefault(case.NF, [0.0, 0.0])
    w[0], w[1] = max(w[0], l2), max(w[1], b)
    assert l2 <= REL_L2, f"rel-L2 {l2:.3e}"
    assert b <= BIN, f"worst bin {b:.3e} of the kept bins' RMS"
    if mm is not None:
        mm = mm.cpu().numpy()
        ys = y.reshape(mm.shape[0], -1)
        assert np.array_equal(mm[:, 0], ys.min(axis=1)) and np.array_equal(mm[:, 1], ys.max(axis=1))


class Kinds:
    """Pins the plan of x's shape to a path with the per-kernel profile on; .kinds after the block.  Asserts that no
    tensor-core kernel gave up on a wait."""

    def __init__(self, shape3, n, path):
        from mvtb import _lib, functional as Fn
        self.L, self.lib = _lib.lib(), _lib
        self.plan = Fn.get_plan(shape3, n, torch.device("cuda:0"))
        self.path = path

    def __enter__(self):
        self.lib.check(self.L, self.L.mvtb_plan_set_path(self.plan, self.path))
        self.lib.check(self.L, self.L.mvtb_plan_profile(self.plan, 1))
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        ms, cn = (C.c_double * self.lib.K_KINDS)(), (C.c_int * self.lib.K_KINDS)()
        self.lib.check(self.L, self.L.mvtb_plan_profile_read(self.plan, ms, cn))
        self.kinds = {self.L.mvtb_kernel_name(k).decode() for k in range(self.lib.K_KINDS) if cn[k]}
        st = self.L.mvtb_plan_tc_status(self.plan)
        self.lib.check(self.L, self.L.mvtb_plan_profile(self.plan, 0))
        self.lib.check(self.L, self.L.mvtb_plan_set_path(self.plan, 0))
        assert st == 0, f"a tensor-core kernel gave up on an mbarrier wait (code {st})"
        return False


def expected(case, path, env=None, in_al=True, out_al=True, sp=False):
    """The kernel kinds bl_run launches (bandlimited.cu) for this case, path, environment and alignment."""
    if not case.bl:
        return M.GENERAL_KINDS                                  # bl_eligible, bandlimited.cu:609
    env = env or {}
    H, W, D = case.shape
    NC, NF = W * D, case.NF
    opt_tc = path != 4                                          # plan.cu:396
    opt_tc_inv = 1 if path == 5 else int(env.get("MVTB_TC_INV", 0))
    quad = H % 4 == 0 and path != 2                             # bandlimited.cu:830
    # bandlimited.cu:1027 -- otherwise k_bl_fwd_h4a (1073: quad, NF <= 16, W*D % 4 == 0, 16-byte input, async on),
    # k_bl_fwd_h4 (1085: quad) or k_bl_fwd_h (1090), all profiled as k_bl_fwd_h
    tc_fwd = opt_tc and H % 16 == 0 and NC % 4 == 0 and in_al
    kinds = {"k_bl_fwd_tc" if tc_fwd else "k_bl_fwd_h"}
    kinds |= M.BL_KINDS_SPLIT if path == 3 or "MVTB_NO_FUSEMID" in env else M.BL_KINDS_MID     # bandlimited.cu:815
    tc_inv = opt_tc and opt_tc_inv and H % 16 == 0 and 16 <= H <= 256                         # bandlimited.cu:859
    if tc_inv:                                                  # bandlimited.cu:862-865, 1193-1234
        kinds |= ({"k_bl_inv_tc"} if not sp or opt_tc_inv == 2 else {"k_bl_mm_tc", "k_sp_bits", "k_bl_inv_tc"})
    elif sp and "MVTB_NO_FUSESP" not in env and quad and NF <= 16 and NC % 2 == 0 and out_al and H >= 8:
        kinds.add("k_bl_inv_sp")                                # bandlimited.cu:840
    else:
        # k_bl_inv_h4v (1252: quad, CPT == 2 i.e. NF <= 16, W*D even, 8-byte output), else k_bl_inv_h4 / k_bl_inv_h
        # (1259), all profiled as k_bl_inv_h
        kinds.add("k_bl_inv_h")
    return kinds


def run_chain(x, descs, path, *, out=None, minmax=True):
    from mvtb import functional as Fn
    with Kinds(x.shape[-3:], x.shape[0], path) as k:
        r = Fn.kspace_chain(x, 3, descs, want_minmax=minmax, out=out)
    y, mm = r if minmax else (r, None)
    return y.clone(), mm, k.kinds


def offset_view(t):
    """A contiguous copy of t whose data pointer is 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device=t.device)
    v = buf[1:1 + t.numel()].view(t.shape)
    assert v.data_ptr() % 16 == 4
    return v.copy_(t)


def _params(variants, kinds=tuple(M.SHAPE_KINDS), bl_only=False):
    out = []
    for c in M.cases(kinds):
        if bl_only and not c.bl:
            continue
        for v in (variants if c.bl else variants[:1]):
            out.append(pytest.param(c, v, id=f"{c.id}-{v}"))
    return out


# ------------------------------------------------------------------------------------------------ paths


@pytest.mark.parametrize("case,variant", _params(("auto", "cc", "tc", "pairs", "split")))
def test_matrix_paths(cuda_device, case, variant):
    """kspace_chain with per-sample (min, max) on every case of the table under each plan path."""
    path = PATHS[variant]
    x, spec, descs = inputs(case)
    y, mm, kinds = run_chain(torch.from_numpy(x).to(cuda_device), descs, path)
    assert kinds == expected(case, path)
    check(case, y, reference(case, x, spec), mm)


@pytest.mark.parametrize("case", [c for c in M.cases(("tc", "quad", "odd")) if c.bl], ids=lambda c: c.id)
def test_matrix_tensor_cores_agree_with_cuda_cores(cuda_device, case):
    x, spec, descs = inputs(case)
    xt = torch.from_numpy(x).to(cuda_device)
    y_tc, _, k_tc = run_chain(xt, descs, 5)
    y_cc, _, k_cc = run_chain(xt, descs, 4)
    assert not ({"k_bl_fwd_tc", "k_bl_inv_tc"} & k_cc)
    if case.kind == "tc":
        assert {"k_bl_fwd_tc", "k_bl_inv_tc"} <= k_tc
    assert rel_l2(y_tc.cpu().numpy(), y_cc.cpu().numpy()) <= TC_VS_CC


# ------------------------------------------------------------------------------------------------ plan options


@pytest.mark.parametrize("case,opt", _params(("NO_ASYNC", "NO_FUSEMID", "TC_INV=1", "TC_INV=2"), ("tc", "quad"), bl_only=True))
def test_matrix_plan_options(cuda_device, env, case, opt):
    """MVTB_NO_ASYNC takes k_bl_fwd_h4 for k_bl_fwd_h4a (quad, NF <= 16) under the CUDA-core path; MVTB_NO_FUSEMID the
    three-kernel W/D stage; MVTB_TC_INV=1/2 the tensor-core inverse on the automatic path."""
    name, _, val = opt.partition("=")
    e = {"MVTB_" + name: val or "1"}
    env(**e)
    path = 4 if name == "NO_ASYNC" else 0
    x, spec, descs = inputs(case)
    y, mm, kinds = run_chain(torch.from_numpy(x).to(cuda_device), descs, path)
    assert kinds == expected(case, path, e)
    check(case, y, reference(case, x, spec), mm)


# ------------------------------------------------------------------------------------------------ select


SELECTS = ("cc", "tc", "TC_INV=2", "NO_FUSESP")


@pytest.mark.parametrize("case,variant", _params(SELECTS, ("tc", "quad", "h2"), bl_only=True))
def test_matrix_select_equals_chain_then_sparse_select(cuda_device, env, case, variant):
    """kspace_chain_sp == kspace_chain(want_minmax) + salt_pepper(sparse=True) bit for bit, whichever kernel selects:
    k_bl_inv_sp (CUDA cores, quad, NF <= 16), k_bl_mm_tc + k_sp_bits + k_bl_inv_tc (tensor cores), k_bl_inv_tc alone
    (MVTB_TC_INV=2), or the separate sampler after the inverse pass."""
    from mvtb import functional as Fn
    e = {}
    if "=" in variant or variant.startswith("NO_"):
        name, _, val = variant.partition("=")
        e = {"MVTB_" + name: val or "1"}
    env(**e)
    path = {"cc": 4, "tc": 5}.get(variant, 0)
    x, spec, descs = inputs(case)
    xt = torch.from_numpy(x).to(cuda_device)
    y, mm, _ = run_chain(xt, descs, path)
    check(case, y, reference(case, x, spec), mm)
    p, seed, offset = 0.3, 11 + case.F, 1000 * case.F
    want = Fn.salt_pepper(y.clone(), p, seed=seed, offset=offset, n_samples=x.shape[0], mm=mm, sparse=True)
    with Kinds(case.shape, x.shape[0], path) as k:
        got, mm2 = Fn.kspace_chain_sp(xt, 3, descs, p, seed=seed, offset=offset)
        got = got.clone()
    assert k.kinds == expected(case, path, e, sp=True)
    assert torch.equal(mm, mm2)
    assert torch.equal(got, want) and not torch.equal(got, y)


# ------------------------------------------------------------------------------------------------ alignment


@pytest.mark.parametrize("case,side", _params(("in", "out", "both"), ("tc", "quad"), bl_only=True))
def test_matrix_unaligned_views(cuda_device, case, side):
    """An input 4 bytes off 16-byte alignment takes neither k_bl_fwd_tc nor k_bl_fwd_h4a; an output 4 bytes off
    8-byte alignment takes k_bl_inv_h4 for k_bl_inv_h4v and the separate select for k_bl_inv_sp."""
    from mvtb import functional as Fn
    x, spec, descs = inputs(case)
    xt = torch.from_numpy(x).to(cuda_device)
    xin = offset_view(xt) if side in ("in", "both") else xt
    out = offset_view(torch.zeros_like(xt)) if side in ("out", "both") else None
    ia, oa = side == "out", side == "in"
    for path in (0, 4):
        y, mm, kinds = run_chain(xin, descs, path, out=out)
        assert kinds == expected(case, path, in_al=ia, out_al=oa)
        check(case, y, reference(case, x, spec), mm)
    want = Fn.salt_pepper(y.clone(), 0.2, seed=5, offset=7, n_samples=x.shape[0], mm=mm, sparse=True)
    with Kinds(case.shape, x.shape[0], 4) as k:
        got, mm2 = Fn.kspace_chain_sp(xin, 3, descs, 0.2, seed=5, offset=7, out=out)
        got = got.clone()
    assert k.kinds == expected(case, 4, in_al=ia, out_al=oa, sp=True)
    assert torch.equal(mm, mm2) and torch.equal(got, want)


# ------------------------------------------------------------------------------------------------ intensity prologue


def _abt(n):
    # near-zero b, as NormalizeIntensity makes it; t reached by the zero voxels of the input
    return np.array([[1.75, -0.05, 0.25], [0.5, 0.03, -0.2]][:n], dtype=np.float32)


@pytest.mark.parametrize("case,where", _params(("auto", "cc", "unaligned", "inplace"), ("tc", "quad", "h2"), bl_only=True))
def test_matrix_prologue(cuda_device, case, where):
    """kspace_chain_ex(pre_abt) at all three places the map can run: in the converters of k_bl_fwd_tc (auto on the
    tc shapes), as k_bl_fwd_h4a<NF, true> reads (cc on the tc and quad shapes with NF <= 16; bandlimited.cu:1073), and
    as the separate affine pass into `out` before any other forward kernel (bandlimited.cu:1074: the h2 shapes, NF > 16,
    an unaligned input, and in place with out = x)."""
    from mvtb import functional as Fn
    path = 4 if where == "cc" else 0
    x, spec, descs = inputs(case)
    x[:, :, 0, :] = 0.0
    abt = _abt(x.shape[0])
    xt = torch.from_numpy(x).to(cuda_device)
    if where == "unaligned":
        xt = offset_view(xt)
    out = xt if where == "inplace" else None
    with Kinds(case.shape, x.shape[0], path) as k:
        y, mm = Fn.kspace_chain_ex(xt, 3, descs, pre_abt=torch.from_numpy(abt).to(cuda_device), want_minmax=True, out=out)
        y = y.clone()
    assert k.kinds == expected(case, path, in_al=where != "unaligned")
    check(case, y, reference(case, x, spec, abt), mm)
    if where == "inplace":
        assert torch.equal(xt, y)


# ------------------------------------------------------------------------------------------------ production shapes


@pytest.mark.parametrize("shape,r", [((2, 240, 240, 155), 17.5), ((2, 128, 128, 64), 18.0)])
@pytest.mark.parametrize("variant", ["auto", "cc", "tc"])
def test_matrix_production_shapes_nf20(cuda_device, shape, r, variant):
    from mvtb import host
    path = PATHS[variant]
    thr = host.disk_threshold(r, shape[1:])
    F = int(np.floor(np.sqrt(thr)))
    case = M.Case(F, "production", shape[1:], True)
    assert case.NF == 20
    x, spec = M.inputs(case, thr=thr)
    y, mm, kinds = run_chain(torch.from_numpy(x).to(cuda_device), descs_for(spec), path)
    assert kinds == expected(case, path)
    check(case, y, reference(case, x, spec), mm)
