"""CPU restatement ("port") of the reference hot path.  TEST INFRASTRUCTURE ONLY.

This module is the checker for the CUDA path. Only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs may import it; the product
package (medical-vision-textural-bias_b200/) never does and fails loudly without
its CUDA extension.

Every function restates one routine of
/root/reference/source_code/filters_and_operators.py (F:line) or
stylization_layers.py (S:line) as a plain function over CPU torch tensors, using the
same torch op sequence (fftn -> fftshift -> pointwise -> ifftshift -> ifftn -> .real)
so that (a) results are bit-comparable with the unmodified reference and (b) its wall
time is a fair "reference CPU path" figure.

Pinned: oracle/make_golden.py runs the UNMODIFIED reference classes (imported from
/root/reference through oracle/monai_shim) on seeded inputs, asserts this port is
bit-identical to them (torch.equal), and stores the reference outputs under
tests/golden/.  tests/test_oracle_golden.py re-checks the port against those files.
The reference itself has no tests or golden vectors (SURVEY.md section 4), so the pin
is "reference run here", the strongest one available.
"""
from math import floor
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
from torch.fft import fftn, fftshift, ifftn, ifftshift

# --------------------------------------------------------------------------- FFT helpers


def kspace(x: torch.Tensor, n_dims: int) -> torch.Tensor:
    """Centered k-space of the last n_dims axes (F:611-614, F:270-271, S:33-34)."""
    axes = tuple(range(-n_dims, 0))
    return fftshift(fftn(x, dim=axes), dim=axes)


def image_real(k: torch.Tensor, n_dims: int) -> torch.Tensor:
    """Real part of the inverse of `kspace` (F:629-632, F:278-279 + F:251, S:49-51)."""
    axes = tuple(range(-n_dims, 0))
    return ifftn(ifftshift(k, dim=axes), dim=axes, norm="backward").real


# --------------------------------------------------------------------------- masks


def disk_binary_mask(shape: Sequence[int], r: float, dim: int, inside_off: bool) -> torch.Tensor:
    """fp32 ball/disk mask over the last `dim` axes, centre floor(N/2) (F:136-197).

    The int64 squared distance is compared with the Python float r**2; torch promotes
    that comparison to float32 (SURVEY A.1).
    """
    shape = tuple(int(s) for s in shape)
    m = torch.zeros(shape).reshape((-1,) + shape[-dim:])
    dist2 = None
    for ax in range(dim):
        n = shape[len(shape) - dim + ax]
        coord = torch.arange(0, n) - floor(n / 2)
        view = [1] * dim
        view[ax] = n
        term = (coord ** 2).reshape(view)
        dist2 = term if dist2 is None else dist2 + term
    keep = dist2 < r ** 2
    keep = keep.unsqueeze(0).repeat_interleave(m.size(0), 0)
    m[keep] = 1
    if inside_off:
        m = 1 - m
    return m.reshape(shape)


def fourier_disk_mask(x: torch.Tensor, r: float, inside_off: bool = False) -> torch.Tensor:
    """RandFourierDiskMaskd body for one key when the gate fires (F:244-251)."""
    k = kspace(x, 3)
    k = k * disk_binary_mask(k.shape, r, 3, inside_off)
    return image_real(k, 3)


def gibbs_mask(spatial_shape: Sequence[int], alpha: float) -> np.ndarray:
    """GibbsNoise boolean mask in numpy float64 (F:686-698)."""
    shape = tuple(int(s) for s in spatial_shape)
    r = (1 - alpha) * np.max(shape) * np.sqrt(2) / 2.0
    centre = (np.array(shape) - 1) / 2
    grid = np.ogrid[tuple(slice(0, n) for n in shape)]
    d2 = sum((g - c) ** 2 for g, c in zip(grid, centre))
    return np.sqrt(d2) <= r


def gibbs_noise(x: torch.Tensor, alpha: float) -> torch.Tensor:
    """GibbsNoise.__call__ (F:663-675, F:678-705)."""
    n_dims = x.dim() - 1
    k = kspace(x, n_dims)
    m = gibbs_mask(k.shape[1:], alpha)
    m = np.repeat(m[None], k.shape[0], axis=0)
    k = k * torch.tensor(m, device=k.device)
    return image_real(k, n_dims)


def gibbs_layer_mask(shape: Sequence[int], alpha: torch.Tensor) -> torch.Tensor:
    """GibbsNoiseLayer fp32 mask over k.shape[1:] (S:99-109)."""
    shape = tuple(int(s) for s in shape)
    centre = (torch.tensor(shape, dtype=torch.float) - 1) / 2
    grids = torch.meshgrid([torch.linspace(0, n - 1, n) for n in shape], indexing="ij")
    dist = torch.sqrt(sum((g - c) ** 2 for g, c in zip(grids, centre)))
    a_norm = alpha * dist.max()
    nd = dist / a_norm
    m = nd.where(nd < 1, torch.zeros_like(a_norm))
    m = m.where(nd > 1, torch.ones_like(a_norm))
    return m


def gibbs_layer(x: torch.Tensor, alpha: float) -> torch.Tensor:
    """GibbsNoiseLayer.forward (S:79-116). n_dims = x.dim()-1, so a 5-D batch is a 4-D FFT."""
    n_dims = x.dim() - 1
    a = torch.tensor([alpha], dtype=torch.float32)
    k = kspace(x, n_dims)
    m = gibbs_layer_mask(k.shape[1:], a)
    m = torch.repeat_interleave(m[None], k.size(0), 0)
    return image_real(k * m, n_dims)


# --------------------------------------------------------------------------- spikes


def ellipsoid_shell_coords(shape3: Sequence[int], a: float, b: float, c: float) -> torch.Tensor:
    """Row-major (n,3) index list of the shell .95 < sum((i-c)^2/a^2) < 1.05 (F:294-325, F:347-348)."""
    h, w, d = (int(s) for s in shape3)
    ch, cw, cd = floor(h / 2), floor(w / 2), floor(d / 2)
    ih, iw, id_ = torch.arange(0, h), torch.arange(0, w), torch.arange(0, d)
    t = (((ih[:, None, None] - ch) ** 2) / a ** 2
         + ((iw[None, :, None] - cw) ** 2) / b ** 2
         + ((id_[None, None, :] - cd) ** 2) / c ** 2)
    sel = torch.logical_and(t > .95, t < 1.05)
    m = torch.zeros((h, w, d))
    m[sel] = 1
    return m.nonzero()


def sample_ellipsoid(shape3, a, b, c, R: np.random.RandomState) -> Tuple[int, int, int]:
    """ellipsoid.sample_ellipsoid (F:342-352): one R.randint(0, n) draw."""
    coords = ellipsoid_shell_coords(shape3, a, b, c)
    i = R.randint(0, len(coords))
    return tuple(int(v) for v in coords[i].numpy())


def plane_wave_spike(x: torch.Tensor, idx: Tuple[int, int, int], intensity: float) -> torch.Tensor:
    """RandPlaneWaves_ellipsoid body for one key given the sampled shifted index (F:381-392)."""
    k = kspace(x, 3)
    la = k.abs().log()
    ph = k.angle()
    la[:, idx[0], idx[1], idx[2]] = intensity
    k2 = la.exp() * torch.exp(1j * ph)
    return image_real(k2, 3)


def kspace_spike(x: torch.Tensor, locs, intensities) -> torch.Tensor:
    """KSpaceSpikeNoise.__call__ (F:906-945) for a list of locs.

    locs: list of tuples, each either full-rank (C,X,Y[,Z]) or spatial (X,Y[,Z]);
    intensities: None (-> 2.5*mean log|k| per channel, F:932-933), or list of floats.
    """
    n_dims = x.dim() - 1
    k = kspace(x, n_dims)
    la = torch.log(torch.absolute(k) + 1e-10)
    ph = torch.angle(k)
    if intensities is None:
        intensities = tuple(torch.mean(la, dim=tuple(range(-n_dims, 0))) * 2.5)
        default = True
    else:
        default = False
    single = not isinstance(locs[0], (tuple, list))
    if single:
        locs = [tuple(locs)]
        vals = [intensities]
    else:
        vals = list(intensities) if isinstance(intensities, (tuple, list)) else [intensities]
    for idx, val in zip(locs, vals):
        idx = tuple(idx)
        if len(idx) == la.dim():
            if isinstance(val, (tuple, list)):      # F:976-977 (default-intensity tuple)
                la[idx] = val[idx[0]]
            else:
                la[idx] = val
        else:                                       # F:980-983: all channels
            if default and single:
                # F:940 hands the whole per-channel tuple of tensors to F:981; torch refuses it
                raise TypeError("can't assign a tuple to a torch.FloatTensor")
            la[(slice(None),) + idx] = val
    k2 = torch.exp(la) * torch.exp(1j * ph)
    return image_real(k2, n_dims)


def logabs_mean(x: torch.Tensor) -> torch.Tensor:
    """Per-channel 2.5*mean(log(|k|+1e-10)) (F:1127-1129, F:932-933)."""
    n_dims = x.dim() - 1
    la = torch.log(torch.absolute(kspace(x, n_dims)) + 1e-10)
    return torch.mean(la, dim=tuple(range(-n_dims, 0))) * 2.5


# --------------------------------------------------------------------------- wrap / S&P


def wrap_artifact(x: torch.Tensor, alpha: float) -> torch.Tensor:
    """WrapArtifact.__call__ on (C,H,W,D) (F:503-515)."""
    n_dims = x.dim() - 1
    k = kspace(x, n_dims)
    k[:, 1:k.size(1):2, :, :] = k[:, 1:k.size(1):2, :, :] * alpha
    k[:, :, 1:k.size(2):2, :] = k[:, :, 1:k.size(2):2, :] * alpha
    k[:, :, :, 1:k.size(3):2] = k[:, :, :, 1:k.size(3):2] * alpha
    return image_real(k, n_dims)


def salt_and_pepper(x: torch.Tensor, p: float, u: torch.Tensor) -> torch.Tensor:
    """SaltAndPepper.salt_and_pepper with the uniform field u injected (F:465-482).

    The reference draws u = torch.rand(x.size()) itself (F:472); everything after that
    line is restated here. F:480 is a self-assignment and is kept for timing fidelity.
    """
    p = min(max(0, p), 1.)
    y = x.clone()
    hi, lo = y.max() / 2, y.min() / 2
    y[u <= p / 2] = lo
    y[torch.logical_and(u > p / 2, u <= p)] = hi
    keep = torch.logical_and(u > p, u != 1.)
    y[keep] = y[keep]
    return y


# --------------------------------------------------------------------------- chains


def chain_127(x: torch.Tensor, r: float, idx, intensity: float, alpha: float, p: float,
              u: Optional[torch.Tensor]) -> torch.Tensor:
    """disk -> plane-wave spike -> wrap -> S&P, the 127-series pipeline
    (10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:138-141)."""
    y = fourier_disk_mask(x, r, False)
    y = plane_wave_spike(y, idx, intensity)
    y = wrap_artifact(y, alpha)
    if u is not None:
        y = salt_and_pepper(y, p, u)
    return y


def chain_127_exact_phase(x: torch.Tensor, r: float, idx, intensity: float, alpha: float) -> torch.Tensor:
    """disk -> plane-wave spike -> wrap (F:244-251, F:381-392, F:503-515) in float64 with the ONE place where the
    reference's result is rounding noise made exact.

    In the 125/126/127 chains the spike lands on a bin the disk stage set to zero.  The reference then reads
    `angle(k)` of the round-trip residue at that bin (F:385): its own fp32 and fp64 runs differ by rel-L2 ~ 1
    (SURVEY section 0).  In exact arithmetic the bin is 0 and `angle(0) = 0`, which is what the CUDA kernels compute.
    This restatement runs the three stages in float64 and, when the spike's bin is outside the disk, sets that bin
    of the disk stage's spectrum to exactly 0 before the spike stage -- nothing else differs from `chain_127`.
    tests/test_oracle_golden.py ties it to the unmodified reference: equal modulo the +-f_s plane wave, with the
    injected amplitude equal."""
    xd = x.to(torch.float64)
    k = kspace(xd, 3)
    m = disk_binary_mask(k.shape, r, 3, False).to(torch.float64)
    # +0 in the masked bins: 0 * k is -0 where Re k < 0, and angle(-0 + 0j) = pi would flip the spike's sign
    k = torch.where(m > 0, k * m, torch.zeros_like(k))
    # the reference goes back to the image and forward again between stages; in exact arithmetic that is the identity
    la = k.abs().log()
    ph = k.angle()                                       # angle(0) = 0 for the exactly-zero masked bins
    la[:, idx[0], idx[1], idx[2]] = intensity
    k2 = la.exp() * torch.exp(1j * ph)
    y = image_real(k2, 3)
    return wrap_artifact(y, alpha)


# --------------------------------------------------------------------------- synthetic data


def synthetic_volume(sample_index: int, shape: Sequence[int]) -> torch.Tensor:
    """SURVEY.md 8(d) synthetic input: seeded N(0,1) inside an ellipsoidal support, 0 outside."""
    g = torch.Generator().manual_seed(1234 + int(sample_index))
    x = torch.randn(*shape, generator=g, dtype=torch.float32)
    sp = shape[-3:] if len(shape) >= 4 else shape[-2:]
    grids = torch.meshgrid([torch.linspace(-1, 1, n) for n in sp], indexing="ij")
    rr = sum((gg / 0.9) ** 2 for gg in grids)
    return x * (rr < 1).to(torch.float32)


def synthetic_uniform(sample_index: int, shape: Sequence[int]) -> torch.Tensor:
    """SURVEY.md 8(d): S&P uniforms for parity runs."""
    g = torch.Generator().manual_seed(777 + int(sample_index))
    return torch.rand(*shape, generator=g, dtype=torch.float32)
