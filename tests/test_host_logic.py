"""Host-side logic (no GPU): integer mask thresholds are bit-exact against the reference's masks,
the ellipsoid shell list, Philox known answers, RNG draw order of the drop-in classes, error
behaviour, and the C-ABI library's exported symbols."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden_names, load_golden
from mvtb import _lib as B, host
from oracle import philox_ref, ref_port as P


def _centred_q(shape):
    grids = np.ogrid[tuple(slice(0, n) for n in shape)]
    return sum((2 * g - (n - 1)) ** 2 for g, n in zip(grids, shape))


def _disk_s(shape):
    grids = np.ogrid[tuple(slice(0, n) for n in shape)]
    return sum((g - n // 2) ** 2 for g, n in zip(grids, shape))


@pytest.mark.parametrize("name", golden_names("disk_"))
def test_disk_threshold_bit_exact(name):
    m, z = load_golden(name)
    r = float("inf") if m["r"] == "inf" else m["r"]
    shape = z["x"].shape[-3:]
    keep = _disk_s(shape) <= host.disk_threshold(r, shape)
    if m["inside_off"]:
        keep = ~keep
    assert np.array_equal(keep.astype(np.uint8), z["mask"])


@pytest.mark.parametrize("r", [0.0, 1.0, 9, 12.5, np.sqrt(200.0000001), np.sqrt(199.9999999), 35, 95, 1e9, float("inf"), float("nan")])
@pytest.mark.parametrize("shape", [(128, 128, 64), (240, 240, 155), (7, 9, 4)])
def test_disk_threshold_vs_torch_expression(r, shape):
    want = P.disk_binary_mask(shape, r, 3, False)
    got = torch.from_numpy((_disk_s(shape) <= host.disk_threshold(r, shape)).astype(np.float32))
    assert torch.equal(got, want)


@pytest.mark.parametrize("name", golden_names("gibbs_"))
def test_gibbs_threshold_bit_exact(name):
    m, z = load_golden(name)
    shape = z["x"].shape[1:]
    keep = _centred_q(shape) <= host.gibbs_threshold(m["alpha"], shape)
    assert np.array_equal(keep.astype(np.uint8), z["mask"])


@pytest.mark.parametrize("alpha", [0.0, 0.3, 0.5, 0.7, 0.95, 1.0])
@pytest.mark.parametrize("shape", [(128, 128, 64), (240, 240, 155)])
def test_gibbs_threshold_full_size(alpha, shape):
    keep = _centred_q(shape) <= host.gibbs_threshold(alpha, shape)
    assert np.array_equal(keep, P.gibbs_mask(shape, alpha))


@pytest.mark.parametrize("name", golden_names("layer_"))
def test_layer_threshold_bit_exact(name):
    m, z = load_golden(name)
    shape = z["x"].shape[1:]
    a = np.float32(min(max(m["alpha"], 0.), 1.))
    keep = _centred_q(shape) <= host.layer_threshold(a, shape)
    assert np.array_equal(keep.astype(np.uint8), z["mask"])


@pytest.mark.parametrize("alpha", [0.2167, 0.4, 0.5, 0.7, 0.71, 0.9, 1.0, 0.0])
@pytest.mark.parametrize("shape", [(1, 128, 128, 64), (1, 240, 240, 155), (4, 240, 240, 155), (128, 128, 64)])
def test_layer_threshold_full_size(alpha, shape):
    with torch.no_grad():
        want = P.gibbs_layer_mask(shape, torch.tensor([alpha], dtype=torch.float32)).numpy()
    keep = _centred_q(shape) <= host.layer_threshold(np.float32(alpha), shape)
    assert np.array_equal(keep.astype(np.float32), want)


@pytest.mark.parametrize("name", golden_names("planes_"))
def test_ellipsoid_shell_list(name):
    m, z = load_golden(name)
    got = host.ellipsoid_shell(tuple(z["x"].shape[1:]), m["a"], m["b"], m["c"])
    assert np.array_equal(got.astype(np.int32), z["shell"])
    R = np.random.RandomState(m["ell_seed"])
    assert list(got[R.randint(0, len(got))]) == m["idx"]


def test_ellipsoid_shell_brats_shapes():
    """(55,55,30) shell: 57 142 voxels for both 128x128x64 and 240x240x155 (SURVEY section 0)."""
    for shape in [(128, 128, 64), (240, 240, 155)]:
        got = host.ellipsoid_shell(shape, 55., 55., 30.)
        want = P.ellipsoid_shell_coords(shape, 55., 55., 30.).numpy()
        assert np.array_equal(got, want)


def test_philox_known_answers():
    for ctr, key, out in philox_ref.KAT:
        got = philox_ref.philox4x32_10(np.array([ctr], dtype=np.uint32), np.array([key], dtype=np.uint32))[0]
        assert tuple(int(v) for v in got) == out
    u = philox_ref.uniform_f32(1001, 42, 7)
    assert u.dtype == np.float32 and u.min() >= 0 and u.max() < 1 and abs(u.mean() - 0.5) < 0.05


def test_make_desc_dedup_and_limits():
    d = host.make_desc(spikes=[((1, 2, 3), 5.0), ((4, 5, 6), 6.0), ((1, 2, 3), 7.0)])
    assert d.n_spikes == 2 and d.spikes[0].amplitude == 7.0 and list(d.spikes[0].idx)[:3] == [1, 2, 3]
    with pytest.raises(ValueError):
        host.make_desc(spikes=[((i, 0, 0), 1.0) for i in range(9)])
    assert host.make_desc().wrap_naxes == 0


def test_exp_f32_matches_torch():
    for v in (5.0, 9.5, 15.0, 17.0):
        assert host.exp_f32(v) == float(torch.tensor([v]).exp()[0])


# ------------------------------------------------------------------ C ABI

def test_cabi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mvtb.h")).read()
    declared = sorted(set(re.findall(r"\b(mvtb_[a-z0-9_]+)\s*\(", header)))
    assert declared == B.exported_symbols()
    if not os.path.exists(B.LIB_PATH):
        from mvtb import build
        build.build_library()
    lib = B.bind(C.CDLL(B.LIB_PATH))          # raises AttributeError on a missing export
    assert lib.mvtb_version() == 200
    assert C.sizeof(B.ChainDesc) == 32 + 8 * 24 + 16 and C.sizeof(B.Spike) == 24       # + mask_u, mask_p, reserved


def test_no_cpu_fallback_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import filters_and_operators as F
    x = torch.zeros(1, 4, 4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        F.GibbsNoise(0.5)(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        F.SaltAndPepper(0.1).salt_and_pepper(x)
    lib = B.lib()
    h = C.c_void_p()
    rc = lib.mvtb_plan_create(C.byref(h), 3, (C.c_int * 3)(4, 4, 4), 1, 0)
    assert rc == B.MVTB_ENODEVICE and "no CPU path" in B.last_error(lib)


# ------------------------------------------------------------------ RNG draw order (SURVEY A.7), kernels stubbed out

@pytest.fixture
def stub_kernels(monkeypatch):
    import filters_and_operators as F
    calls = []

    def fake_chain(img, ndim_fft, descs, **kw):
        calls.append((ndim_fft, descs))
        return img

    monkeypatch.setattr(F, "_run_chain", fake_chain)
    monkeypatch.setattr(F.Fn, "to_device", lambda x, device=None: (x, x.device))
    monkeypatch.setattr(F.Fn, "kspace_chain", lambda x, n, descs, **kw: (calls.append((n, descs)), x)[1])
    monkeypatch.setattr(F.Fn, "back", lambda y, src: y)
    return calls


def test_rng_order_rand_gibbs(stub_kernels):
    import filters_and_operators as F
    m, z = load_golden("rng_randgibbs")
    t = F.RandGibbsNoise(prob=m["prob"], alpha=tuple(m["alpha"]))
    t.set_random_state(seed=m["seed"])
    x = torch.from_numpy(z["x"])
    for _ in range(3):
        t(x)
    assert t.sampled_alpha == m["sampled_alpha"]


def test_rng_order_rand_disk_list_radius_is_drawn_once(stub_kernels):
    import filters_and_operators as F
    m, z = load_golden("rng_randdisk")
    t = F.RandFourierDiskMaskd("image", r=list(m["r"]), prob=m["prob"])
    t.set_random_state(seed=m["seed"])
    for _ in range(4):
        t({"image": torch.from_numpy(z["x"])})
    assert float(t.r) == m["r_after"]


@pytest.mark.parametrize("cw", [0, 1])
def test_rng_order_rand_kspike(stub_kernels, cw):
    import filters_and_operators as F
    m, z = load_golden(f"rng_randkspike_cw{cw}")
    t = F.RandKSpaceSpikeNoise(prob=m["prob"], intensity_range=tuple(m["range"]), channel_wise=m["channel_wise"])
    t.set_random_state(seed=m["seed"])
    for _ in range(3):
        t(torch.from_numpy(z["x"]))
    assert [list(map(int, l)) for l in t.sampled_locs] == m["locs"]
    assert [float(v) for v in t.sampled_k_intensity] == m["ints"]


def test_rng_order_rand_planes(stub_kernels):
    import filters_and_operators as F
    m, z = load_golden("rng_randplanes")
    t = F.RandPlaneWaves_ellipsoid("image", 5., 4., 3., intensity_value=4.0, prob=0.6)
    t.set_random_state(seed=m["seed"])
    t.ellipsoid.set_random_state(seed=m["ell_seed"])
    got = []
    for _ in range(4):
        t({"image": torch.from_numpy(z["x"])})
        got.append(None if t.idx is None else [int(v) for v in t.idx])
    assert got == m["idxs"]


def test_reference_error_behaviour():
    import filters_and_operators as F
    with pytest.raises(AssertionError):
        F.RandFourierDiskMaskd("image", prob=1.5)
    with pytest.raises(AssertionError):
        F.GibbsNoise(1.5)
    with pytest.raises(AssertionError):
        F.RandGibbsNoise(alpha=(0.5, 0.2))
    with pytest.raises(AssertionError):
        F.KSpaceSpikeNoise((1, 2, 3), (5.0, 6.0))
    with pytest.raises(AssertionError):
        F.KSpaceSpikeNoise(((0, 1, 2, 3), (1, 1, 1)), 5.0)
    with pytest.raises(AssertionError):
        F.RandKSpaceSpikeNoise(intensity_range=((1, 2), (3, 4)), channel_wise=False)
    with pytest.raises(AssertionError):
        F.KSpaceSpikeNoise((0, 99, 0, 0), 5.0)(torch.zeros(1, 4, 4, 4))
    with pytest.warns(UserWarning):
        assert F.SaltAndPepper(1.5).p == 1.0
    with pytest.raises(KeyError):
        F.WrapArtifactd("missing")({"image": torch.zeros(1, 2, 2, 2)})
    assert F.WrapArtifactd("missing", allow_missing_keys=True)({"image": 1}) == {"image": 1}
    assert F.SaltAndPepper(0.3, "image", 0.0)({"image": 5}) == {"image": 5}      # positional order p, keys, prob


def test_disk_mask_class_bit_exact():
    import filters_and_operators as F
    for name in golden_names("diskmask2d_"):
        m, z = load_golden(name)
        dm = F.disk_mask(torch.zeros(m["shape"]), r=m["r"], dim=2, inside_off=m["inside_off"])
        assert torch.equal(dm.binary_mask.to(torch.uint8), torch.from_numpy(z["mask"]))
    k = torch.randn(2, 6, 5, 4, dtype=torch.complex64)
    dm = F.disk_mask(k, r=2.0, dim=3, inside_off=False)
    assert torch.equal(dm.binary_mask, P.disk_binary_mask(k.shape, 2.0, 3, False))
    assert torch.equal(dm.apply(k), k * dm.binary_mask)


def test_label_helpers():
    import filters_and_operators as F
    lab = np.array([[0, 1], [2, 3]])
    out = F.ConvertToMultiChannelBasedOnBratsClassesd("label")({"label": lab})["label"]
    assert out.shape == (3, 2, 2) and out.dtype == np.float32
    assert np.array_equal(out[0], [[0, 0], [1, 1]]) and np.array_equal(out[1], [[0, 1], [1, 1]]) and np.array_equal(out[2], [[0, 0], [1, 0]])
    x = torch.arange(24.).reshape(4, 3, 2)
    assert torch.equal(F.SelectChanneld("image", 2)({"image": x})["image"], x[2][None])
    d = F.SelectChanneld(["image", "label"], (3, 0))({"image": x, "label": x})
    assert torch.equal(d["image"], x[3][None]) and torch.equal(d["label"], x[0][None])
    assert np.array_equal(F.WholeTumorTCGA("label")({"label": np.array([0, 2, 4])})["label"], [[0., 1., 1.]])


def test_hostmem_cpulist_and_no_gpu_is_graceful():
    """NUMA placement helper for the host-buffer path: parses sysfs cpulists; without a visible device it reports, never raises."""
    from mvtb import hostmem
    assert hostmem._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert hostmem._parse_cpulist("") == set()
    if not torch.cuda.is_available():
        assert hostmem.gpu_numa_node(0) is None
        assert hostmem.bind_to_gpu_numa_node(0)["bound"] is False


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with the contract keys."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "volumes/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("volumes/sec") and line["value"] > 0 and line["n_gpus"] == 1
    assert line["config"]["workload"].startswith("cfg2")
    assert line["e2e"] == {"value": line["value"], "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value_1_thread"] > 0 and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]


def test_bench_output_sample_is_whole_or_a_fixed_sample():
    """`bench.py --dump-outputs`: an output that fits is written whole; a larger one is sampled at the same positions
    on every run, in float32 (float64 stays float64)."""
    import bench
    y = torch.arange(1000, dtype=torch.float32).reshape(10, 100)
    assert np.array_equal(bench.output_sample(y, budget=4000), y.numpy())
    a = bench.output_sample(y, budget=400)
    assert a.dtype == np.float32 and 50 < a.size <= 100 and np.all(np.diff(a) > 0)       # sorted distinct positions
    assert np.array_equal(a, bench.output_sample(y.clone(), budget=400))
    d = bench.output_sample(y.double(), budget=800)                                          # same element count
    assert d.dtype == np.float64 and np.array_equal(d, a)
    assert bench.output_sample(y.to(torch.float16), budget=4000).dtype == np.float32


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 2 and "error:" in out.stderr and not out.stdout


def test_gibbs_layer_reads_alpha_once_per_update():
    """GibbsNoiseLayer keeps alpha's host value until the attribute is reassigned or written in place (S:71 reads it
    on the host every forward; on a CUDA tensor that is a synchronising copy)."""
    import torch
    import stylization_layers as S
    layer = S.GibbsNoiseLayer(0.7)
    layer.alpha = torch.tensor([0.7])
    assert layer._alpha_on_host() == pytest.approx(0.7)
    first = layer._alpha_cache
    assert layer._alpha_on_host() == pytest.approx(0.7) and layer._alpha_cache is first      # no second read
    old = layer.alpha.clone()
    layer.alpha = old + 0.1                                                                   # the scripts' update (GD.py:261)
    assert layer._alpha_on_host() == pytest.approx(0.8) and layer._alpha_cache is not first
    with torch.no_grad():
        layer.alpha -= 0.3                                                                    # in place: version counter
    assert layer._alpha_on_host() == pytest.approx(0.5)
    layer.alpha = 0.25                                                                        # a plain float is accepted too
    assert layer._alpha_on_host() == 0.25
