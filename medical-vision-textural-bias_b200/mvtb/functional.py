"""Tensor-level entry points over the C ABI (include/mvtb.h): torch supplies device memory and
streams, libmvtb.so does the arithmetic.  No function here has a CPU implementation; on a
machine without CUDA they raise.

Layout contract (same as the reference): contiguous float32, FFT over the last `ndim_fft` axes,
every leading axis is a batch of independent volumes.
"""
import atexit
import math
import ctypes as C
import threading
from collections import OrderedDict
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, host

import os

# plan workspace: ~2 half-spectra of 240x240x155 for the general path (L2-resident between its kernels);
# the band-limited path fits ~16 volumes of intermediates in the same bytes.  MVTB_WS_MB overrides.
_WS_TARGET_BYTES = int(os.environ.get("MVTB_WS_MB", "80")) << 20
# A plan owns one workspace and one ring of staging slots, so it serves one stream at a time (include/mvtb.h).
# Plans are therefore cached per (thread, device, stream, shape, chunk): two streams, or two Python threads (ctypes
# releases the GIL during a call), never share one.  Each thread keeps at most _MAX_PLANS of them, least recently
# used first out (a pipeline fed with random crop sizes would otherwise grow device memory without bound);
# MVTB_MAX_PLANS overrides.
_MAX_PLANS = max(1, int(os.environ.get("MVTB_MAX_PLANS", "12")))
_tls = threading.local()
_registry_lock = threading.Lock()
_registry = []                      # every thread's cache, for the exit hook


def _cache() -> "OrderedDict":
    c = getattr(_tls, "plans", None)
    if c is None:
        c = _tls.plans = OrderedDict()
        with _registry_lock:
            _registry.append(c)
    return c


_cuda_ok = False


def require_cuda() -> None:
    global _cuda_ok
    if _cuda_ok:                                        # a device does not go away; the query costs ~5 us per call
        return
    if not torch.cuda.is_available():
        raise RuntimeError("mvtb: no CUDA device is available and there is no CPU fallback "
                           "(the transforms run only through libmvtb.so on a GPU)")
    _cuda_ok = True


def _stream(dev: torch.device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


class Origin(NamedTuple):
    """Where a transform's input came from: results go back to that device, in that precision."""
    device: torch.device
    dtype: torch.dtype


def to_device(x, device: Optional[torch.device] = None) -> Tuple[torch.Tensor, Origin]:
    """float32 contiguous CUDA view/copy of x, plus its origin for `back()`.

    The kernels compute in float32, the precision of every reference pipeline.  A float64 input (a tensor made from
    a default numpy array, say), for which the reference would run a complex128 FFT and return float64, is computed
    in float32 here and handed back as float64; integer inputs come back as float32, as from the reference's FFT."""
    require_cuda()
    if isinstance(x, np.ndarray):
        x = torch.as_tensor(x)
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor or numpy array, got {type(x).__name__}")
    if x.is_complex():
        raise TypeError(f"mvtb transforms take real images (got {x.dtype})")
    org = Origin(x.device, x.dtype if x.dtype == torch.float64 else torch.float32)
    if x.dtype != torch.float32:
        x = x.to(torch.float32)
    if x.is_cuda:
        return x.contiguous(), org
    dev = device or torch.device("cuda", torch.cuda.current_device())
    return x.contiguous().to(dev, non_blocking=False), org


def back(y: torch.Tensor, org) -> torch.Tensor:
    if isinstance(org, Origin):
        y = y if org.device == y.device else y.to(org.device)
        return y if org.dtype == y.dtype else y.to(org.dtype)
    return y if org == y.device else y.to(org)


def get_plan(fft_shape: Sequence[int], n_volumes: int, dev: torch.device):
    """The calling thread's plan for this shape on the current stream of `dev` (created on first use)."""
    fft_shape = tuple(int(s) for s in fft_shape)
    nh = fft_shape[-1] // 2 + 1
    half_bytes = 8 * nh * math.prod(fft_shape[:-1])
    chunk = int(max(1, min(n_volumes, _WS_TARGET_BYTES // max(half_bytes, 1))))
    if chunk > 8:
        chunk = 1 << (chunk.bit_length() - 1)        # few distinct plans per shape
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream, fft_shape, chunk)
    cache = _cache()
    h = cache.get(key)
    if h is not None:
        cache.move_to_end(key)
        return h
    L = _lib.lib()
    while len(cache) >= _MAX_PLANS:                   # evict this thread's least recently used plan
        _, old = cache.popitem(last=False)
        L.mvtb_plan_destroy(old)                      # waits for the device, then frees tables and workspace
    h = C.c_void_p()
    shp = (C.c_int * len(fft_shape))(*fft_shape)
    _lib.check(L, L.mvtb_plan_create(C.byref(h), len(fft_shape), shp, chunk, dev.index))
    if os.environ.get("MVTB_PATH"):                  # measurements: 1 = general FFT path only, 2 = pair kernels
        _lib.check(L, L.mvtb_plan_set_path(h, int(os.environ["MVTB_PATH"])))
    cache[key] = h
    return h


def plan_cache_size() -> int:
    """Plans currently held for the calling thread."""
    return len(_cache())


@atexit.register
def _destroy_plans():
    if _lib._lib is None:
        return
    with _registry_lock:
        caches = list(_registry)
    for c in caches:
        for h in list(c.values()):
            try:
                _lib._lib.mvtb_plan_destroy(h)
            except Exception:  # noqa: BLE001
                pass
        c.clear()


def kspace_chain(x: torch.Tensor, ndim_fft: int, descs: Sequence[_lib.ChainDesc], *, want_minmax: bool = False,
                 vols_per_sample: int = 1, out: Optional[torch.Tensor] = None):
    """out = Re ifftn(W (M fftn(x) + spikes)) over the last ndim_fft axes of a CUDA float32 tensor.

    descs: one shared descriptor or one per volume (volumes = product of the leading axes).
    Returns y, or (y, minmax[n_samples, 2]) when want_minmax."""
    L = _lib.lib()
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("kspace_chain expects a contiguous float32 CUDA tensor (use functional.to_device)")
    if x.dim() < ndim_fft:
        raise ValueError(f"input of rank {x.dim()} has fewer than ndim_fft={ndim_fft} axes")
    fft_shape = tuple(x.shape[-ndim_fft:])
    nvol = math.prod(x.shape[:-ndim_fft]) if x.dim() > ndim_fft else 1
    if len(descs) not in (1, nvol):
        raise ValueError(f"need 1 or {nvol} descriptors, got {len(descs)}")
    y = torch.empty_like(x) if out is None else out
    if x.numel() == 0:
        return (y, torch.empty((0, 2), device=x.device)) if want_minmax else y
    plan = get_plan(fft_shape, nvol, x.device)
    mm = None
    if want_minmax:
        mm = torch.empty(((nvol + vols_per_sample - 1) // vols_per_sample, 2), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        rc = L.mvtb_kspace_chain_f32(plan, _ptr(x), _ptr(y), nvol, host.desc_array(descs), len(descs), _ptr(mm),
                                     int(vols_per_sample), _stream(x.device))
    _lib.check(L, rc)
    return (y, mm) if want_minmax else y


def kspace_chain_sp(x: torch.Tensor, ndim_fft: int, descs: Sequence[_lib.ChainDesc], p: float, *, seed: int = 0,
                    offset: int = 0, vols_per_sample: int = 1, out: Optional[torch.Tensor] = None):
    """kspace_chain followed by the sparse salt-and-pepper sampler, as ONE library call (mvtb_kspace_chain_sp_f32):
    the same result as kspace_chain(..., want_minmax=True) + salt_pepper(..., sparse=True), bit for bit.  On the
    band-limited path the select pass runs inside the inverse kernel while the output is still in L2.
    `offset` counts 256-voxel blocks (advance it by n_samples * ceil(voxels per sample / 256) per call).
    Returns (y, minmax[n_samples, 2]); minmax is that of the chain's output before the select."""
    L = _lib.lib()
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("kspace_chain_sp expects a contiguous float32 CUDA tensor (use functional.to_device)")
    if x.dim() < ndim_fft:
        raise ValueError(f"input of rank {x.dim()} has fewer than ndim_fft={ndim_fft} axes")
    fft_shape = tuple(x.shape[-ndim_fft:])
    nvol = math.prod(x.shape[:-ndim_fft]) if x.dim() > ndim_fft else 1
    if len(descs) not in (1, nvol):
        raise ValueError(f"need 1 or {nvol} descriptors, got {len(descs)}")
    if nvol % vols_per_sample:
        raise ValueError(f"{nvol} volumes are not a whole number of samples of {vols_per_sample}")
    y = torch.empty_like(x) if out is None else out
    mm = torch.empty((nvol // vols_per_sample, 2), dtype=torch.float32, device=x.device)
    if x.numel() == 0:
        return y, mm
    plan = get_plan(fft_shape, nvol, x.device)
    with torch.cuda.device(x.device):
        rc = L.mvtb_kspace_chain_sp_f32(plan, _ptr(x), _ptr(y), nvol, host.desc_array(descs), len(descs), _ptr(mm),
                                        int(vols_per_sample), C.c_float(p), C.c_uint64(seed & (2 ** 64 - 1)),
                                        C.c_uint64(offset & (2 ** 64 - 1)), _stream(x.device))
    _lib.check(L, rc)
    return y, mm


def kspace_chain_ex(x: torch.Tensor, ndim_fft: int, descs: Sequence[_lib.ChainDesc], *, pre_abt: Optional[torch.Tensor] = None,
                    sp: Optional[Tuple[float, int, int]] = None, want_minmax: bool = False, vols_per_sample: int = 1,
                    out: Optional[torch.Tensor] = None):
    """mvtb_kspace_chain_ex_f32: [intensity prologue map on the way in] -> chain -> [sparse salt-and-pepper on the way
    out].  pre_abt: float32 CUDA tensor (n_volumes, 3) from intensity_coeffs(); sp: (p, seed, offset[, sample_stride]), the
    stride being the distance between samples' Philox span counters (mvtb_kspace_chain_ex_strided_f32; 0 = spans per sample).
    Returns y, or (y, minmax) when want_minmax or sp is given."""
    L = _lib.lib()
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("kspace_chain_ex expects a contiguous float32 CUDA tensor (use functional.to_device)")
    fft_shape = tuple(x.shape[-ndim_fft:])
    nvol = math.prod(x.shape[:-ndim_fft]) if x.dim() > ndim_fft else 1
    if len(descs) not in (1, nvol):
        raise ValueError(f"need 1 or {nvol} descriptors, got {len(descs)}")
    if pre_abt is not None and (pre_abt.shape != (nvol, 3) or pre_abt.dtype != torch.float32 or pre_abt.device != x.device or not pre_abt.is_contiguous()):
        raise ValueError("pre_abt must be a contiguous float32 (n_volumes, 3) tensor on x's device")
    y = torch.empty_like(x) if out is None else out
    need_mm = want_minmax or sp is not None
    mm = torch.empty(((nvol + vols_per_sample - 1) // vols_per_sample, 2), dtype=torch.float32, device=x.device) if need_mm else None
    if x.numel() == 0:
        return (y, mm) if need_mm else y
    plan = get_plan(fft_shape, nvol, x.device)
    spp = None
    if sp is not None:
        spp = _lib.SpParams(float(sp[0]), int(sp[1]) & (2 ** 64 - 1), int(sp[2]) & (2 ** 64 - 1))
    stride = int(sp[3]) if sp is not None and len(sp) > 3 else 0
    with torch.cuda.device(x.device):
        rc = L.mvtb_kspace_chain_ex_strided_f32(plan, _ptr(x), _ptr(y), nvol, host.desc_array(descs), len(descs), _ptr(pre_abt), _ptr(mm),
                                                int(vols_per_sample), C.byref(spp) if spp is not None else None, C.c_uint64(stride),
                                                _stream(x.device))
    _lib.check(L, rc)
    return (y, mm) if need_mm else y


# ----------------------------------------------------------------------------- intensity prologue (csrc/intensity.cu)
def intensity_coeffs(x: torch.Tensor, n_channels: int, *, scale=None, shift=None, want_stats: bool = False):
    """One read of x (n_channels contiguous channels): per channel the map (a, b, t) of
    NormalizeIntensity(nonzero, channel_wise) -> * scale -> + shift, i.e. y = x != 0 ? a x + b : t.
    scale / shift: None, a number, or one value per channel.  Returns abt (n_channels, 3) float32 on x.device
    [, stats (n_channels, 3) float64: count, mean, std]."""
    L = _lib.lib()
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("intensity_coeffs expects a contiguous float32 CUDA tensor")
    dev = x.device

    def vec(v, default):
        if v is None:
            return None
        t = torch.as_tensor(v, dtype=torch.float32).reshape(-1)
        if t.numel() == 1:
            t = t.expand(n_channels)
        if t.numel() != n_channels:
            raise ValueError(f"need 1 or {n_channels} values")
        return t.contiguous().to(dev, non_blocking=True)

    sc, sh = vec(scale, 1.0), vec(shift, 0.0)
    abt = torch.empty((n_channels, 3), dtype=torch.float32, device=dev)
    stats = torch.empty((n_channels, 3), dtype=torch.float64, device=dev) if want_stats else None
    scratch = torch.empty(max(int(L.mvtb_intensity_scratch_bytes(n_channels)), 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = L.mvtb_intensity_prologue_coeffs_f32(_ptr(x), x.numel() // max(n_channels, 1), n_channels, _ptr(sc), _ptr(sh),
                                                  _ptr(stats), _ptr(abt), _ptr(scratch), _stream(dev))
    _lib.check(L, rc)
    return (abt, stats) if want_stats else abt


def intensity_affine(x: torch.Tensor, abt: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = x != 0 ? a x + b : t with one (a, b, t) per leading block of x (abt: (n, 3))."""
    L = _lib.lib()
    n = int(abt.shape[0])
    y = torch.empty_like(x) if out is None else out
    if x.numel() == 0:
        return y
    with torch.cuda.device(x.device):
        rc = L.mvtb_intensity_affine_f32(_ptr(x), _ptr(y), x.numel() // n, n, _ptr(abt), _stream(x.device))
    _lib.check(L, rc)
    return y


def intensity_prologue(img, *, nonzero: bool = True, channel_wise: bool = True, scale: float = 1.0, shift: float = 0.0):
    """NormalizeIntensity(nonzero, channel_wise) -> * scale -> + shift on a (C, ...) image (tensor or numpy array, any
    device); the result comes back where the input lived, float32."""
    if not nonzero:
        raise NotImplementedError("only nonzero=True (the reference's setting) is built")
    x, org = to_device(img)
    n_ch = int(x.shape[0]) if channel_wise else 1
    abt = intensity_coeffs(x, n_ch, scale=scale, shift=shift)
    y = back(intensity_affine(x, abt), Origin(org.device, torch.float32))
    return y.numpy() if isinstance(img, np.ndarray) else y


def intensity_scale_shift(img, *, scale: float = 1.0, shift: float = 0.0):
    """ScaleIntensity(factor) / ShiftIntensity(offset) on their own: y = x * scale + shift for every voxel."""
    x, org = to_device(img)
    y = back(torch.addcmul(torch.full((), float(shift), device=x.device), x, torch.full((), float(scale), device=x.device)), Origin(org.device, torch.float32))
    return y.numpy() if isinstance(img, np.ndarray) else y


def logabs_mean25(x: torch.Tensor, ndim_fft: int) -> torch.Tensor:
    """2.5 * mean(log(|fftn(x)| + 1e-10)) per volume, float32 on x.device (F:932-933, F:1127-1129)."""
    L = _lib.lib()
    fft_shape = tuple(x.shape[-ndim_fft:])
    nvol = math.prod(x.shape[:-ndim_fft]) if x.dim() > ndim_fft else 1
    plan = get_plan(fft_shape, nvol, x.device)
    sums = torch.empty(nvol, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        rc = L.mvtb_kspace_logabs_sum_f32(plan, _ptr(x), nvol, _ptr(sums), _stream(x.device))
    _lib.check(L, rc)
    return (sums * (2.5 / float(np.prod(fft_shape)))).to(torch.float32).reshape(x.shape[:-ndim_fft])


def minmax(x: torch.Tensor, n_samples: int = 1) -> torch.Tensor:
    """(min, max) per sample -> float32 [n_samples, 2] on x.device."""
    L = _lib.lib()
    mm = torch.empty((n_samples, 2), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        rc = L.mvtb_minmax_f32(_ptr(x), x.numel() // max(n_samples, 1), n_samples, _ptr(mm), _stream(x.device))
    _lib.check(L, rc)
    return mm


def salt_pepper(x: torch.Tensor, p: float, *, u: Optional[torch.Tensor] = None, seed: int = 0, offset: int = 0,
                n_samples: int = 1, mm: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                sparse: bool = False) -> torch.Tensor:
    """Salt-and-pepper select (F:465-482) per sample; u injected (bit-exact parity) or Philox(seed, offset).

    sparse=True (Philox only): the geometric-gap Bernoulli sampler of mvtb_salt_pepper_sparse_f32, cost ~ p;
    `offset` then counts blocks of 256 voxels (advance it by n_samples * ceil(n_per_sample / 256) per call)."""
    L = _lib.lib()
    if mm is None:
        mm = minmax(x, n_samples)
    if sparse:
        if u is not None:
            raise ValueError("sparse=True draws its own random field; it cannot take injected uniforms")
        y = x if out is None or out.data_ptr() == x.data_ptr() else out.copy_(x)
        if out is None:
            y = x.clone()
        table = torch.empty(_lib.SP_BLOCK, dtype=torch.int32, device=x.device)
        with torch.cuda.device(x.device):
            rc = L.mvtb_salt_pepper_sparse_f32(_ptr(y), y.numel() // max(n_samples, 1), n_samples,
                                               C.c_uint64(seed & (2 ** 64 - 1)), C.c_uint64(offset & (2 ** 64 - 1)),
                                               C.c_float(p), _ptr(mm), _ptr(table), _stream(x.device))
        _lib.check(L, rc)
        return y
    if u is not None and (u.shape != x.shape or u.dtype != torch.float32 or u.device != x.device or not u.is_contiguous()):
        raise ValueError("u must be a contiguous float32 tensor of x's shape on x's device")
    y = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        rc = L.mvtb_salt_pepper_f32(_ptr(x), _ptr(y), x.numel() // max(n_samples, 1), n_samples, _ptr(u),
                                    C.c_uint64(seed & (2 ** 64 - 1)), C.c_uint64(offset & (2 ** 64 - 1)),
                                    C.c_float(p), _ptr(mm), _stream(x.device))
    _lib.check(L, rc)
    return y


def philox_uniform(n: int, seed: int, offset: int, device: torch.device) -> torch.Tensor:
    L = _lib.lib()
    out = torch.empty(n, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        rc = L.mvtb_philox_uniform_f32(_ptr(out), n, C.c_uint64(seed), C.c_uint64(offset), _stream(device))
    _lib.check(L, rc)
    return out


def wrap_fold(x: torch.Tensor, alpha: float) -> torch.Tensor:
    """Even-axis wraparound fold on (..., H, W, D); raises MvtbError(EUNSUPPORTED) for an odd axis."""
    L = _lib.lib()
    H, W, D = (int(s) for s in x.shape[-3:])
    nvol = x.numel() // (H * W * D) if x.numel() else 0
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = L.mvtb_wrap_fold_f32(_ptr(x), _ptr(y), nvol, H, W, D, C.c_float(alpha), _stream(x.device))
    _lib.check(L, rc)
    return y


def wrap_odd_last(x: torch.Tensor, alpha: float) -> torch.Tensor:
    """Wraparound on (..., H, W, D) with even H, W and any D: image-domain folds along H and W, a one-kernel
    FFT filter along D (mvtb_wrap_odd_last_f32); raises MvtbError(EUNSUPPORTED) for odd H or W."""
    L = _lib.lib()
    shp = tuple(int(s) for s in x.shape[-3:])
    nvol = x.numel() // (shp[0] * shp[1] * shp[2]) if x.numel() else 0
    y = torch.empty_like(x)
    if nvol == 0:
        return y
    plan = get_plan(shp, nvol, x.device)
    with torch.cuda.device(x.device):
        rc = L.mvtb_wrap_odd_last_f32(plan, _ptr(x), _ptr(y), nvol, C.c_float(alpha), _stream(x.device))
    _lib.check(L, rc)
    return y


# ----------------------------------------------------------------------------- batched chain-127 convenience
_chain127_descs: dict = {}


def chain127(x: torch.Tensor, *, r: float, spike_idx: Optional[Sequence[Sequence[int]]], intensity: float,
             alpha: Optional[float], p: Optional[float], u: Optional[torch.Tensor] = None, seed: int = 0,
             offset: int = 0, sparse: bool = False) -> torch.Tensor:
    """disk -> plane-wave spike -> wrap -> S&P on a batch (B, C, H, W, D), each (C,H,W,D) sample treated
    exactly as one pass through the 127-series Compose (one spike location per sample, shared by its
    channels; S&P min/max over the whole sample).  spike_idx: per-sample fftshift-ed (h,w,d), or None."""
    B_, C_ = x.shape[0], x.shape[1]
    # the descriptors depend only on the arguments, not on the data: a loader that draws the same spike locations again
    # (or none) gets the list back instead of B make_desc calls (~3 us each: a third of a 32-volume call's host time)
    key = (tuple(x.shape[-3:]), B_, C_, float(r), float(intensity), alpha,
           None if spike_idx is None else tuple(tuple(int(v) for v in i) for i in spike_idx))
    descs = _chain127_descs.get(key)
    if descs is None:
        thr = host.disk_threshold(r, x.shape[-3:])
        amp = host.exp_f32(intensity)
        descs = []
        for b in range(B_):
            sp = [(spike_idx[b], amp)] if spike_idx is not None else []
            d = host.make_desc(mask_kind=_lib.MASK_DISK, mask_ndim=3, mask_thresh=thr, spikes=sp, wrap_alpha=alpha)
            descs.extend([d] * C_)
        descs = host.desc_array(descs)                   # the ctypes array itself is kept: no per-call copy either
        if len(_chain127_descs) >= 32:
            _chain127_descs.clear()
        _chain127_descs[key] = descs
    if p is None:
        return kspace_chain(x, 3, descs)
    if sparse and u is None:                          # one call: the select pass rides on the inverse kernel
        return kspace_chain_sp(x, 3, descs, p, seed=seed, offset=offset, vols_per_sample=C_)[0]
    y, mm = kspace_chain(x, 3, descs, want_minmax=True, vols_per_sample=C_)
    return salt_pepper(y, p, u=u, seed=seed, offset=offset, n_samples=B_, mm=mm, out=y, sparse=sparse)
