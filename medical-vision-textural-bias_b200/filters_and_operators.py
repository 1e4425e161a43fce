"""Drop-in for the reference's source_code/filters_and_operators.py (F below).

Same class names, constructor signatures, public attributes, dict/array calling conventions,
random-draw order and error behaviour; the voxel and k-space arithmetic runs in the hand-written
CUDA kernels of libmvtb.so (mvtb/csrc) through the C ABI in include/mvtb.h.  There is no CPU
fallback: without a CUDA device the transforms raise.

Use it the way the reference scripts use theirs:
    sys.path.append(<repo>/medical-vision-textural-bias_b200); from filters_and_operators import ...
Tensors may live on the CPU (they are staged through the GPU and returned on the CPU, like the
reference's results) or already on a CUDA device (no copies).
"""
import warnings
from collections.abc import Sequence as _SeqABC
from math import floor
from typing import Any, Dict, Hashable, List, Mapping, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from mvtb import _lib, functional as Fn, host
from mvtb._monai_compat import (KeysCollection, MapTransform, Randomizable, RandomizableTransform, Transform,
                                ensure_tuple)

__all__ = [
    "SelectChanneld", "ConvertToMultiChannelBasedOnBratsClassesd", "WholeTumorTCGA", "disk_mask",
    "RandFourierDiskMaskd", "ellipsoid", "RandPlaneWaves_ellipsoid", "SaltAndPepper", "WrapArtifact",
    "WrapArtifactd", "SegmentationSlicesd", "Fourier", "GibbsNoise", "RandGibbsNoise", "RandGibbsNoised",
    "KSpaceSpikeNoise", "RandKSpaceSpikeNoise", "RandKSpaceSpikeNoised",
]


# ============================================================================ label / channel helpers
# (F:25-101, F:563-589: plain slicing and comparisons on labels - host-side, not part of the hot path)

class SelectChanneld(MapTransform):
    """Keep one channel of (C,H,W,D) data, preserving the channel axis (F:25-58)."""

    def __init__(self, keys, chan_num: Union[int, Sequence[int]], allow_missing_keys=False):
        self.chan_num = chan_num
        super().__init__(keys, allow_missing_keys)

    def __call__(self, data):
        d = dict(data)
        per_key = isinstance(self.chan_num, _SeqABC) and len(self.chan_num) > 1
        if per_key:
            for c, key in zip(self.chan_num, self.key_iterator(d)):
                if c > d[key].shape[0] - 1:
                    raise AssertionError(f'Provided channel index {c} larger than max channel index for key = {key}')
                d[key] = d[key][c][None, :]
        else:
            c = self.chan_num[0] if isinstance(self.chan_num, _SeqABC) else self.chan_num
            for key in self.key_iterator(d):
                d[key] = d[key][c][None, :]
        return d


class ConvertToMultiChannelBasedOnBratsClassesd(MapTransform):
    """BraTS labels -> (TC, WT, ET) float32 channels (F:61-87).  A CUDA tensor (mvtb.nifti.LoadImaged's output) stays on
    its device and comes back as CUDA float32."""

    def __call__(self, data):
        d = dict(data)
        for key in self.keys:
            lab = d[key]
            if isinstance(lab, torch.Tensor) and lab.is_cuda:
                tc = (lab == 2) | (lab == 3)
                d[key] = torch.stack([tc, tc | (lab == 1), lab == 2], dim=0).to(torch.float32)
                continue
            tc = np.logical_or(lab == 2, lab == 3)
            wt = np.logical_or(tc, lab == 1)
            et = lab == 2
            d[key] = np.stack([tc, wt, et], axis=0).astype(np.float32)
        return d


class WholeTumorTCGA(MapTransform):
    """TCGA segmentation -> whole-tumour mask with a channel axis (F:90-101)."""

    def __init__(self, keys, allow_missing_keys=False):
        MapTransform.__init__(self, keys, allow_missing_keys)

    def __call__(self, data):
        d = dict(data)
        for key in self.key_iterator(d):
            d[key] = (d[key] != 0)[None, :].astype(np.float32)
        return d


class SegmentationSlicesd(MapTransform, Randomizable):
    """Three consecutive slices around a non-trivial segmentation (F:563-589)."""

    def __init__(self, keys, seed: int = None, allow_missing_keys: bool = False):
        Randomizable.set_random_state(self, seed=seed)
        MapTransform.__init__(self, keys, allow_missing_keys)

    def __call__(self, data):
        d = dict(data)
        while True:
            c = self.R.randint(3, 60)
            if d["label"][0, :, :, c - 3].max() == d["label"][0, :, :, c + 3].max() == 1:
                break
        for key in self.key_iterator(d):
            d[key] = d[key].squeeze(0)[:, :, c:c + 3].transpose(0, 2)
        return d


# ============================================================================ helpers shared by the transforms

def _as_f32_tensor(img) -> torch.Tensor:
    if isinstance(img, np.ndarray):
        return torch.Tensor(img)               # the reference does exactly this (F:666-667, F:923-924)
    return img


def _run_chain(img: torch.Tensor, ndim_fft: int, descs, **kw):
    x, src = Fn.to_device(img)
    res = Fn.kspace_chain(x, ndim_fft, descs, **kw)
    if isinstance(res, tuple):
        return Fn.back(res[0], src), res[1]
    return Fn.back(res, src)


# ============================================================================ disk masks (F:105-279)

class disk_mask():
    """Binary ball (dim=3) / disk (dim=2) mask over the last `dim` axes of a k-space tensor (F:105-206).

    `binary_mask` is float32, same shape as `k_tensor`, bit-identical to the reference's: the float32
    comparison `sum (i - floor(N/2))^2 < r**2` is reduced to an integer threshold on the host."""

    def __init__(self, k_tensor: torch.Tensor, r: float = 2, dim: int = 2, inside_off=True):
        self.r = r
        self.dim = dim
        self.inside_off = inside_off
        self.last_dims = k_tensor.size(-1)
        if self.dim in (2, 3):
            self.binary_mask = self._build(k_tensor)
        else:
            print('Only 2- and 3-dimensional images.')

    def _build(self, k_tensor) -> torch.Tensor:
        tail = tuple(k_tensor.shape[-self.dim:])
        thr = host.disk_threshold(self.r, tail)
        dist2 = torch.zeros(tail, dtype=torch.int64)
        for ax, n in enumerate(tail):
            view = [1] * self.dim
            view[ax] = n
            dist2 = dist2 + ((torch.arange(n) - floor(n / 2)) ** 2).reshape(view)
        keep = dist2 <= thr
        if self.inside_off:
            keep = ~keep
        return keep.to(torch.float32).expand(tuple(k_tensor.shape)).contiguous()

    def binary_mask_2d(self, k_tensor) -> torch.Tensor:
        self.dim = 2
        return self._build(k_tensor)

    def binary_mask_3d(self, k_tensor) -> torch.Tensor:
        self.dim = 3
        return self._build(k_tensor)

    def apply(self, k_tensor: torch.Tensor) -> torch.Tensor:
        assert k_tensor.size(-1) == self.last_dims, f'Last dimension of input must be = {self.last_dims}'
        return k_tensor * self.binary_mask.to(k_tensor.device)


class RandFourierDiskMaskd(RandomizableTransform, MapTransform):
    """Gibbs ringing by truncating k-space to a ball of radius r over the last three axes (F:210-279).

    One fused forward+inverse FFT pass with the mask evaluated from integer frequencies: no fftshift
    copies, no materialised mask, no complex temporaries."""

    def __init__(self, keys: Union[str, List['str']], r: Union[float, List[float]] = float('Inf'),
                 inside_off: bool = False, prob: float = 0.5, allow_missing_keys: bool = False) -> None:
        assert prob <= 1 and prob >= 0, 'prob must take values in [0,1]'
        self.r = r
        self.inside_off = inside_off
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, prob=prob)

    def randomize(self) -> None:
        # gate first, then (first call only: the list is overwritten by the drawn float) the radius (F:254-261)
        super().randomize(None)
        if type(self.r) == list:
            self.r = self.R.uniform(self.r[0], self.r[1])

    def __call__(self, data):
        d = dict(data)
        self.randomize()
        if not self._do_transform:
            return d
        for key in self.key_iterator(d):
            x = d[key]
            if x.dim() < 3:
                raise RuntimeError("RandFourierDiskMaskd transforms the last three axes; got a tensor of rank "
                                   f"{x.dim()}")
            desc = host.make_desc(mask_kind=_lib.MASK_DISK, mask_ndim=3, inside_off=self.inside_off,
                                  mask_thresh=host.disk_threshold(self.r, x.shape[-3:]))
            d[key] = _run_chain(x, 3, [desc])
        return d


# ============================================================================ plane waves on an ellipsoid (F:284-414)

class ellipsoid(Randomizable):
    """(x-x0)^2/a^2 + (y-y0)^2/b^2 + (z-z0)^2/c^2 = 1 shell in fftshift-ed k-space (F:284-352)."""

    def __init__(self, a: float, b: float, c: float):
        self.a = a
        self.b = b
        self.c = c

    def _coords(self, k_tensor) -> np.ndarray:
        return host.ellipsoid_shell(tuple(int(s) for s in k_tensor.shape[-3:]), self.a, self.b, self.c)

    def binary_mask_3d(self, k_tensor) -> torch.Tensor:
        shape3 = tuple(k_tensor.shape[-3:])
        m = torch.zeros(shape3)
        c = self._coords(k_tensor)
        m[c[:, 0], c[:, 1], c[:, 2]] = 1
        return m.expand(tuple(k_tensor.shape)).contiguous()

    def sample_ellipsoid(self, k_tensor):
        """One R.randint(0, n) over the cached row-major shell list (F:342-352)."""
        coords = self._coords(k_tensor)
        i = self.R.randint(0, len(coords))
        return tuple(coords[i])


class RandPlaneWaves_ellipsoid(RandomizableTransform, MapTransform):
    """One k-space spike per call on the ellipsoid shell, same voxel in every channel (F:355-414).

    The reference rewrites log|k| at one voxel and rebuilds all of k from exp/angle; only the spiked
    bin (and its conjugate partner, since the real part is returned) actually changes, which is what
    the kernel applies."""

    def __init__(self, keys: Union[str, List['str']] = 'image', a: float = 10, b: float = 10, c: float = 10,
                 intensity_value: float = 1, prob: float = 0.2, allow_missing_keys: bool = False):
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, prob=prob)
        self.ellipsoid = ellipsoid(a, b, c)
        self.intensity_value = intensity_value
        self.idx = None

    def __call__(self, data):
        d = dict(data)
        self.randomize(None)
        if not self._do_transform:
            return d
        for key in self.key_iterator(d):
            x = d[key]
            self.idx = self.ellipsoid.sample_ellipsoid(x[0])
            desc = host.make_desc(spikes=[(self.idx, host.exp_f32(self.intensity_value))])
            d[key] = _run_chain(x, 3, [desc])
        return d


# ============================================================================ salt and pepper (F:419-482)

class SaltAndPepper(MapTransform, RandomizableTransform):
    """Salt-and-pepper voxel corruption (F:419-482): u<=p/2 -> min/2, p/2<u<=p -> max/2.

    rng="torch" (default) draws u with torch.rand on the CPU generator exactly where the reference does
    (F:472), so seeded runs reproduce it bit for bit; rng="philox" draws u inside the kernel from
    Philox4x32-10 keyed by `seed` (counter advances every call) and never touches host memory;
    rng="philox-sparse" walks from hit to hit with Philox-drawn geometric gaps (same Bernoulli(p) field
    statistics, cost proportional to p)."""

    def __init__(self, p: float = 0, keys: Union[str, List['str']] = 'image', prob: float = 1.,
                 allow_missing_keys: bool = False, *, rng: str = "torch", seed: int = 0):
        self.p = min(max(0, p), 1.)
        if p < 0 or p > 1:
            warnings.warn(f'Setting p to {self.p}.')
        if rng not in ("torch", "philox", "philox-sparse"):
            raise ValueError("rng must be 'torch', 'philox' or 'philox-sparse'")
        self.rng = rng
        self.seed = int(seed)
        self.offset = 0
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, prob=prob)

    def __call__(self, data):
        d = dict(data)
        self.randomize(None)
        if not self._do_transform:
            return d
        for key in self.key_iterator(d):
            d[key] = self.salt_and_pepper(d[key])
        return d

    def salt_and_pepper(self, x: torch.Tensor, u: Optional[torch.Tensor] = None):
        """x: any shape; min/max are taken over the whole tensor (F:476).  u: optional injected uniforms."""
        if u is None and self.rng == "torch":
            u = torch.rand(x.size())
        xd, src = Fn.to_device(x)
        ud = None
        if u is not None:
            ud = u.to(device=xd.device, dtype=torch.float32).contiguous()
        sparse = ud is None and self.rng == "philox-sparse"
        y = Fn.salt_pepper(xd, float(self.p), u=ud, seed=self.seed, offset=self.offset, n_samples=1, sparse=sparse)
        if ud is None:
            self.offset += (xd.numel() + 255) // 256 if sparse else (xd.numel() + 3) // 4
        return Fn.back(y, src)


# ============================================================================ wraparound (F:488-560)

class WrapArtifact(Transform):
    """Wraparound artifact: odd fftshift-ed k-space samples along H, W and D scaled by alpha (F:488-537).

    Even H, W, D: exact image-domain fold (8 taps, one read + one write per voxel).  Even H, W and odd D
    (240 x 240 x 155): folds along H and W plus a one-kernel FFT filter along D.  Otherwise the k-space chain with
    the parity weights."""

    def __init__(self, alpha: float = 0.5):
        self.alpha = alpha

    def __call__(self, img: torch.Tensor):
        if img.dim() != 4:
            raise IndexError(f"too many indices for tensor of dimension {img.dim()}" if img.dim() < 4 else
                             "WrapArtifact expects (C,H,W,D) input")
        x, src = Fn.to_device(img)
        if all(int(s) % 2 == 0 for s in x.shape[1:]):
            y = Fn.wrap_fold(x, float(self.alpha))
        elif int(x.shape[1]) % 2 == 0 and int(x.shape[2]) % 2 == 0:
            y = Fn.wrap_odd_last(x, float(self.alpha))
        else:
            y = Fn.kspace_chain(x, 3, [host.make_desc(wrap_alpha=float(self.alpha), wrap_naxes=3)])
        return Fn.back(y, src)


class WrapArtifactd(MapTransform):
    """Dictionary version of WrapArtifact (F:540-560)."""

    def __init__(self, keys: KeysCollection, alpha: float = 0.5, allow_missing_keys: bool = False):
        MapTransform.__init__(self, keys, allow_missing_keys)
        self.transform = WrapArtifact(alpha)

    def __call__(self, data: Mapping[Hashable, torch.Tensor]):
        d = dict(data)
        for key in self.key_iterator(d):
            d[key] = self.transform(d[key])
        return d


# ============================================================================ Gibbs noise (F:594-843)

class Fourier:
    """Centred k-space helpers kept for API compatibility (F:594-632).  The transforms below never call
    them (the kernels need no fftshift); they are thin torch.fft wrappers for user code that does."""

    @staticmethod
    def shift_fourier(x: torch.Tensor, n_dims: int) -> torch.Tensor:
        axes = tuple(range(-n_dims, 0))
        return torch.fft.fftshift(torch.fft.fftn(x, dim=axes), dim=axes)

    @staticmethod
    def inv_shift_fourier(k: torch.Tensor, n_dims: int) -> torch.Tensor:
        axes = tuple(range(-n_dims, 0))
        return torch.fft.ifftn(torch.fft.ifftshift(k, dim=axes), dim=axes).real


class GibbsNoise(Transform, Fourier):
    """Gibbs noise: keep k-space within radius (1-alpha)*max(shape)*sqrt(2)/2 of the (N-1)/2 centre (F:635-705)."""

    def __init__(self, alpha: float = 0.5, as_tensor_output: bool = True) -> None:
        if alpha > 1 or alpha < 0:
            raise AssertionError("alpha must take values in the interval [0,1].")
        self.alpha = alpha
        self.as_tensor_output = as_tensor_output

    def __call__(self, img: Union[np.ndarray, torch.Tensor]) -> Union[torch.Tensor, np.ndarray]:
        n_dims = len(img.shape[1:])
        img = _as_f32_tensor(img)
        if n_dims < 2 or n_dims > 4:
            raise ValueError(f"GibbsNoise supports 2 to 4 transformed axes, got {n_dims}")
        desc = host.make_desc(mask_kind=_lib.MASK_CENTRED, mask_ndim=n_dims,
                              mask_thresh=host.gibbs_threshold(self.alpha, img.shape[1:]))
        out = _run_chain(img, n_dims, [desc])
        return out if self.as_tensor_output else out.cpu().detach().numpy()


def _passthrough(img, as_tensor_output: bool):
    if isinstance(img, np.ndarray) and as_tensor_output:
        return torch.Tensor(img)
    if isinstance(img, torch.Tensor) and not as_tensor_output:
        return img.detach().cpu().numpy()
    return img


class RandGibbsNoise(RandomizableTransform):
    """Random Gibbs noise: gate, then alpha ~ U(a,b) is always drawn (F:708-768)."""

    def __init__(self, prob: float = 0.1, alpha: Sequence[float] = (0.0, 1.0), as_tensor_output: bool = True) -> None:
        if len(alpha) != 2:
            raise AssertionError("alpha length must be 2.")
        if alpha[1] > 1 or alpha[0] < 0:
            raise AssertionError("alpha must take values in the interval [0,1]")
        if alpha[0] > alpha[1]:
            raise AssertionError("When alpha = [a,b] we need a < b.")
        self.alpha = alpha
        self.sampled_alpha = -1.0
        self.as_tensor_output = as_tensor_output
        RandomizableTransform.__init__(self, prob=prob)

    def _randomize(self, _: Any) -> None:
        super().randomize(None)
        self.sampled_alpha = self.R.uniform(self.alpha[0], self.alpha[1])

    def __call__(self, img: Union[np.ndarray, torch.Tensor]) -> Union[torch.Tensor, np.ndarray]:
        self._randomize(None)
        if self._do_transform:
            return GibbsNoise(self.sampled_alpha, self.as_tensor_output)(img)
        return _passthrough(img, self.as_tensor_output)


class RandGibbsNoised(RandomizableTransform, MapTransform):
    """Dictionary version of RandGibbsNoise; one alpha shared by all keys (F:771-843)."""

    def __init__(self, keys: KeysCollection, prob: float = 0.1, alpha: Sequence[float] = (0.0, 1.0),
                 as_tensor_output: bool = True, allow_missing_keys: bool = False) -> None:
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, prob=prob)
        self.alpha = alpha
        self.sampled_alpha = -1.0
        self.as_tensor_output = as_tensor_output

    def _randomize(self, _: Any) -> None:
        super().randomize(None)
        self.sampled_alpha = self.R.uniform(self.alpha[0], self.alpha[1])

    def __call__(self, data: Mapping[Hashable, Union[torch.Tensor, np.ndarray]]) -> Dict[Hashable, Union[torch.Tensor, np.ndarray]]:
        d = dict(data)
        self._randomize(None)
        transform = GibbsNoise(self.sampled_alpha, self.as_tensor_output) if self._do_transform else None
        for key in self.key_iterator(d):
            d[key] = transform(d[key]) if transform is not None else _passthrough(d[key], self.as_tensor_output)
        return d

    def _to_numpy(self, d: Union[torch.Tensor, np.ndarray]) -> np.ndarray:
        if isinstance(d, torch.Tensor):
            return d.cpu().detach().numpy()
        return d


# ============================================================================ k-space spikes (F:846-1254)

class KSpaceSpikeNoise(Transform, Fourier):
    """Set log|k| at given fftshift-ed locations, keep the phase, return the real part (F:846-983).

    loc: (C,X,Y[,Z]) hits one channel, (X,Y[,Z]) all channels; or a sequence of such tuples with a
    matching sequence of k_intensity.  k_intensity None -> 2.5 * mean log(|k|+1e-10) per channel."""

    def __init__(self, loc: Union[Tuple, Sequence[Tuple]], k_intensity: Optional[Union[Sequence[float], float]] = None,
                 as_tensor_output: bool = True):
        self.loc = ensure_tuple(loc)
        self.as_tensor_output = as_tensor_output
        self.k_intensity = k_intensity
        if isinstance(k_intensity, _SeqABC):
            if not isinstance(loc[0], _SeqABC):
                raise AssertionError(
                    "If a sequence is passed to k_intensity, then a sequence of locations must be passed to loc")
            if len(k_intensity) != len(loc):
                raise AssertionError("There must be one intensity_factor value for each tuple of indices in loc.")
        if isinstance(self.loc[0], _SeqABC) and k_intensity is not None:
            if not isinstance(self.k_intensity, _SeqABC):
                raise AssertionError("There must be one intensity_factor value for each tuple of indices in loc.")

    def _check_indices(self, img) -> None:
        """AssertionError if any index is out of bounds (F:948-964)."""
        loc = list(self.loc)
        if not isinstance(loc[0], _SeqABC):
            loc = [loc]
        loc = [([0] + list(l)) if len(l) < len(img.shape) else list(l) for l in loc]
        for i in range(len(img.shape)):
            if img.shape[i] <= max(l[i] for l in loc):
                raise AssertionError(
                    f"The index value at position {i} of one of the tuples in loc = {self.loc} is out of bounds for current image.")

    def __call__(self, img: Union[np.ndarray, torch.Tensor]) -> Union[torch.Tensor, np.ndarray]:
        self._check_indices(img)
        rank = len(img.shape)
        if rank < 3:
            raise AssertionError("Image needs a channel direction.")
        multi = isinstance(self.loc[0], _SeqABC)
        if not multi and isinstance(self.loc[0], int) and rank == 4 and len(self.loc) == 2:
            raise AssertionError("Input images of dimension 4 need location tuple to be length 3 or 4")
        if multi and rank == 4 and min(len(l) for l in self.loc) == 2:
            raise AssertionError("Input images of dimension 4 need location tuple to be length 3 or 4")
        n_dims = rank - 1
        img = _as_f32_tensor(img)
        x, src = Fn.to_device(img)
        n_chan = x.shape[0]

        intensity = self.k_intensity
        default = None
        if intensity is None:
            # one extra forward transform + log reduction, read back to the host (F:932-933)
            default = [float(v) for v in Fn.logabs_mean25(x, n_dims).cpu()]

        # (location, log-intensity) pairs in the reference's order (F:936-940)
        if multi:
            vals = default if intensity is None else list(ensure_tuple(intensity))
            pairs = list(zip(self.loc, vals))
        else:
            pairs = [(self.loc, default if intensity is None else intensity)]

        pairs = [(self._wrap_negative(tuple(int(i) for i in idx), x.shape), val) for idx, val in pairs]
        if all(len(idx) == rank - 1 for idx, _ in pairs) and rank in (3, 4):
            # every spike hits all channels (F:980-983): one descriptor for the whole stack, however many channels
            shared = []
            for idx, val in pairs:
                if isinstance(val, _SeqABC):
                    raise TypeError("can't assign a tuple to a torch.FloatTensor")   # what F:981/983 raises
                shared.append((idx, host.exp_f32(val)))
            descs = [host.make_desc(spikes=shared)]
        else:
            per_chan: List[List[Tuple[Tuple[int, ...], float]]] = [[] for _ in range(n_chan)]
            for idx, val in pairs:
                if len(idx) == rank:                      # F:975-979: one channel
                    v = val[idx[0]] if isinstance(val, _SeqABC) else val
                    per_chan[idx[0]].append((idx[1:], host.exp_f32(v)))
                elif len(idx) == rank - 1 and rank in (3, 4):   # F:980-983: all channels
                    if isinstance(val, _SeqABC):
                        raise TypeError("can't assign a tuple to a torch.FloatTensor")   # what F:981/983 raises
                    for c in range(n_chan):
                        per_chan[c].append((idx, host.exp_f32(val)))
            made = {}
            descs = []
            for sp in per_chan:                           # channels with the same spikes share one descriptor object
                key = tuple(sp)
                if key not in made:
                    made[key] = host.make_desc(spikes=sp)
                descs.append(made[key])
        out = Fn.back(Fn.kspace_chain(x, n_dims, descs), src)
        return out if self.as_tensor_output else out.cpu().detach().numpy()


    @staticmethod
    def _wrap_negative(idx: Tuple[int, ...], shape) -> Tuple[int, ...]:
        """Negative indices count from the end, as in the reference's `k[idx] = val` (F:975-983; its bounds check
        F:958-962 only looks at the largest index); beyond -N torch raises IndexError, and so does this."""
        dims = tuple(shape)[len(shape) - len(idx):]
        out = []
        for d, (i, n) in enumerate(zip(idx, dims)):
            if i < -int(n):
                raise IndexError(f"index {i} is out of bounds for dimension {d + len(shape) - len(idx)} with size {int(n)}")
            out.append(i + int(n) if i < 0 else i)
        return tuple(out)


class RandKSpaceSpikeNoise(RandomizableTransform, Fourier):
    """Random k-space spikes (F:986-1131); draw order: gate, then per-axis randint, then uniform."""

    def __init__(self, prob: float = 0.1, intensity_range: Optional[Sequence[Union[Sequence[float], float]]] = None,
                 channel_wise=True, as_tensor_output: bool = True):
        self.intensity_range = intensity_range
        self.channel_wise = channel_wise
        self.as_tensor_output = as_tensor_output
        self.sampled_k_intensity: List = []
        self.sampled_locs: List[Tuple] = []
        if intensity_range is not None:
            if isinstance(intensity_range[0], _SeqABC) and not channel_wise:
                raise AssertionError(
                    "When channel_wise = False, intensity_range should be a 2-tuple (low, high) or None.")
        super().__init__(prob)

    def __call__(self, img: Union[np.ndarray, torch.Tensor]) -> Union[torch.Tensor, np.ndarray]:
        if self.intensity_range is not None:
            if isinstance(self.intensity_range[0], _SeqABC) and len(self.intensity_range) != img.shape[0]:
                raise AssertionError(
                    "If intensity_range is a sequence of sequences, then there must be one (low, high) tuple for each channel.")
        self.sampled_k_intensity = []
        self.sampled_locs = []
        if not isinstance(img, torch.Tensor):
            img = torch.Tensor(img)
        ranges = self._make_sequence(img)
        self._randomize(img, ranges)
        if self.sampled_locs:
            return KSpaceSpikeNoise(self.sampled_locs, self.sampled_k_intensity, self.as_tensor_output)(img)
        return img if self.as_tensor_output else img.detach().numpy()

    def _randomize(self, img: torch.Tensor, intensity_range: Sequence[Sequence[float]]) -> None:
        if self.channel_wise:
            for i in range(img.shape[0]):
                super().randomize(None)
                if self._do_transform:
                    self.sampled_locs.append((i,) + tuple(self.R.randint(0, k) for k in img.shape[1:]))
                    self.sampled_k_intensity.append(self.R.uniform(intensity_range[i][0], intensity_range[i][1]))
        else:
            super().randomize(None)
            if self._do_transform:
                spatial = tuple(self.R.randint(0, k) for k in img.shape[1:])
                self.sampled_locs = [(i,) + spatial for i in range(img.shape[0])]
                if isinstance(intensity_range[0], _SeqABC):
                    self.sampled_k_intensity = [self.R.uniform(p[0], p[1]) for p in intensity_range]
                else:
                    self.sampled_k_intensity = [self.R.uniform(intensity_range[0], intensity_range[1])] * len(img)

    def _make_sequence(self, x: torch.Tensor) -> Sequence[Sequence[float]]:
        if self.intensity_range is None:
            return self._set_default_range(x)
        if not isinstance(self.intensity_range[0], _SeqABC):
            return (ensure_tuple(self.intensity_range),) * x.shape[0]
        return ensure_tuple(self.intensity_range)

    def _set_default_range(self, img: torch.Tensor) -> Sequence[Sequence[float]]:
        """(0.95 m, 1.1 m) per channel, m = 2.5 mean log(|k|+1e-10): a full forward transform (F:1118-1131)."""
        x, _ = Fn.to_device(img)
        means = Fn.logabs_mean25(x, len(img.shape[1:])).cpu()
        return tuple((m * 0.95, m * 1.1) for m in means)


class RandKSpaceSpikeNoised(RandomizableTransform, MapTransform):
    """Dictionary version: one RandKSpaceSpikeNoise per key behind a global gate (F:1134-1254)."""

    def __init__(self, keys: KeysCollection, global_prob: float = 1.0, prob: float = 0.1,
                 intensity_ranges: Optional[Mapping[Hashable, Sequence[Union[Sequence[float], float]]]] = None,
                 channel_wise: bool = True, common_sampling: bool = False, common_seed: int = 42,
                 as_tensor_output: bool = True, allow_missing_keys: bool = False):
        MapTransform.__init__(self, keys, allow_missing_keys)
        RandomizableTransform.__init__(self, global_prob)
        self.common_sampling = common_sampling
        self.common_seed = common_seed
        self.as_tensor_output = as_tensor_output
        self.transforms = {}
        for k in self.keys:
            rng = intensity_ranges[k] if isinstance(intensity_ranges, Mapping) else None
            self.transforms[k] = RandKSpaceSpikeNoise(prob, rng, channel_wise, self.as_tensor_output)

    def __call__(self, data: Mapping[Hashable, Union[torch.Tensor, np.ndarray]]) -> Dict[Hashable, Union[torch.Tensor, np.ndarray]]:
        d = dict(data)
        super().randomize(None)
        if self.common_sampling:
            for k in self.keys:
                self.transforms[k].set_random_state(self.common_seed)
        for key, t in self.key_iterator(d, self.transforms):
            if self._do_transform:
                d[key] = self.transforms[t](d[key])
            else:
                d[key] = _passthrough(d[key], self.as_tensor_output)
        return d

    def set_rand_state(self, seed: Optional[int] = None, state: Optional[np.random.RandomState] = None) -> None:
        self.set_random_state(seed, state)
        for key in self.keys:
            self.transforms[key].set_random_state(seed, state)

    def _to_numpy(self, d: Union[torch.Tensor, np.ndarray]) -> np.ndarray:
        if isinstance(d, torch.Tensor):
            return d.cpu().detach().numpy()
        return d
