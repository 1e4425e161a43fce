"""Float64 reference and case table of the band-limited k-space chain.  TEST INFRASTRUCTURE ONLY.

`chain_ref` restates, on numpy.fft in float64, what mvtb_kspace_chain_f32 computes on the band-limited path
(csrc/bandlimited.cu, csrc/pointwise.cuh):

    y = Re ifftn(ifftshift(W * S(M_eff * fftshift(fftn(P(x))))))

- P: the optional intensity prologue map of mvtb_kspace_chain_ex_f32, y = x != 0 ? a x + b : t per volume;
- M_eff = (M(i) + M(i')) / 2, M the integer mask (`host.disk_threshold` / `host.gibbs_threshold` form) and
  i' the index of the negated frequency, i'_d = (2 floor(N_d / 2) - i_d) mod N_d;
- S: each spike replaces its bin by amp * k / |k|, and by amp where the mask zeroed the bin (angle(0) = 0);
- W: the wrap weight, alpha for every odd fftshift-ed index on each of the three axes.

Taking the real part at the end symmetrises a spike between its bin and the conjugate bin, which is what the
kernels' pointwise stage does explicitly.  tests/test_emu_bl_matrix.py pins this function against
oracle.ref_port.chain_127_exact_phase and ref_port.gibbs_noise.

The case table covers every NF bucket of `bl_chain` (F + 1 rounded up to one of BUCKETS) at both ends of its F
range, and for each F a small set of shapes that select the kernel variants of `bl_run`; two shapes per F must fall
back to the general FFT path (`bl_eligible`).
"""
from typing import NamedTuple, Optional, Sequence, Tuple

import numpy as np

BUCKETS = (4, 8, 13, 16, 20, 26, 32)
MASK_DISK, MASK_CENTRED = 1, 2          # mvtb.h MVTB_MASK_DISK / MVTB_MASK_CENTRED
AXES = (-3, -2, -1)

BL_KINDS_MID = {"k_bl_mid"}
BL_KINDS_SPLIT = {"k_bl_fwd_w", "k_bl_mid", "k_bl_inv_w"}
GENERAL_KINDS = {"k_rows_fwd", "k_axis<FWD>", "k_axis<MID>", "k_axis<INV>", "k_rows_inv"}


def nf_bucket(F: int) -> int:
    return next(nf for nf in BUCKETS if F + 1 <= nf)


def bucket_ends() -> Tuple[int, ...]:
    """F = 0 and both ends of every bucket: the previous bucket's top + 1 and NF - 1."""
    fs = {0}
    prev = 0
    for nf in BUCKETS:
        fs.update((prev, nf - 1))
        prev = nf
    return tuple(sorted(fs))


def _up(v: int, m: int, rem: int = 0) -> int:
    while v % m != rem:
        v += 1
    return v


class Case(NamedTuple):
    F: int
    kind: str            # shape kind, see SHAPE_KINDS
    shape: Tuple[int, int, int]
    bl: bool             # the band-limited path must take it

    @property
    def NF(self) -> int:
        return nf_bucket(self.F)

    @property
    def id(self) -> str:
        H, W, D = self.shape
        return f"F{self.F}-nf{self.NF}-{self.kind}-{H}x{W}x{D}"


# kind -> what it selects (H, W, D; K = 2F + 1; every band-limited shape has H >= 2 NF - 1)
SHAPE_KINDS = {
    "tc": "H % 16 == 0, W*D % 4 == 0: the tensor-core forward (and inverse) layout",
    "quad": "H % 4 == 0, H % 16 != 0, W*D % 4 == 0: the cp.async quad forward and the vector quad inverse",
    "quadodd": "H % 4 == 0, W*D odd, W = 2F+1: the quad kernels without vector or async access",
    "h2": "H % 4 == 2, W*D odd, D = 2F+1: the pair kernels",
    "odd": "H = 2 NF - 1 (odd, the smallest H the bucket takes), W*D % 4 == 0: the pair kernels",
    "fb_h": "H = 2 NF - 2: one row short, must fall back to the general path",
    "fb_w": "W = 2F: one column short of the kept box, must fall back to the general path",
}


def shape_for(F: int, kind: str) -> Optional[Tuple[int, int, int]]:
    nf = nf_bucket(F)
    hmin, K = 2 * nf - 1, 2 * F + 1
    if kind == "tc":
        return (_up(hmin, 16), K + 1, K + 3)
    if kind == "quad":
        H = _up(hmin, 4)
        return (H + 4 if H % 16 == 0 else H, K + 1, K + 1)
    if kind == "quadodd":
        return (_up(hmin, 4), K, K + 2)
    if kind == "h2":
        return (_up(hmin, 4, 2), K + 2, K)
    if kind == "odd":
        return (hmin, K + 1, K + 1)
    if kind == "fb_h":
        return (2 * nf - 2, K + 1, K + 1)
    if kind == "fb_w":
        return (_up(hmin, 16), 2 * F, K + 1) if F > 0 else None
    raise ValueError(kind)


def cases(kinds: Sequence[str] = tuple(SHAPE_KINDS)) -> Tuple[Case, ...]:
    out = []
    for F in bucket_ends():
        for k in kinds:
            s = shape_for(F, k)
            if s is not None:
                out.append(Case(F, k, s, not k.startswith("fb_")))
    return tuple(out)


def disk_radius(F: int) -> float:
    """A radius whose disk threshold is F^2 + F: the largest kept |f| on an axis is exactly F."""
    return F + 0.5


def centred_threshold(F: int) -> int:
    """A centred-mask threshold whose kept box is exactly |f| <= F on a shape with an even axis (bandlimited.cu:603)."""
    return (2 * F) ** 2


def spikes_for(shape: Sequence[int], F: int, rs: np.random.RandomState, n_in: int, n_out: int, amp: float):
    """n_in spikes inside the kept box (the first one inside the ball), n_out outside it on one axis at least;
    distinct bins, none the conjugate of another."""
    H, W, D = shape
    c = np.array([H // 2, W // 2, D // 2])
    n = np.array(shape)
    got, seen = [], set()

    def neg(i):
        return tuple(int((2 * (m // 2) - v) % m) for v, m in zip(i, n))

    def add(i, a):
        i = tuple(int(v) for v in i)
        if i in seen or neg(i) in seen:
            return False
        seen.update((i, neg(i)))
        got.append((i, a))
        return True

    add(c + np.array([min(F, 1), 0, -min(F, 1)]), amp)
    while len(got) < n_in:
        add(np.minimum(c + rs.randint(-F, F + 1, size=3), n - 1), amp * (0.5 + rs.rand()))
    tries = 0
    while len(got) < n_in + n_out and tries < 1000:
        tries += 1
        i = rs.randint(0, n)
        if np.all(np.abs(i - c) <= F):
            continue
        add(i, amp * (0.5 + rs.rand()))
    assert len(got) == n_in + n_out, (shape, F)
    return got


def inputs(case: Case, n_vol: int = 2, thr: Optional[int] = None):
    """Seeded white noise (every bin carries energy) and the chain's parameters (kind, thr, spikes, wrap alphas) for
    a disk mask with kept box |f| <= F: volume 0 with a spike in the ball, a second in-box spike (none at F = 0) and
    the two out-of-box spikes the inverse pass adds as plane waves, wrap 0.5; volume 1 with one in-box and one
    out-of-box spike, no wrap; any further volume plain."""
    import torch
    g = torch.Generator().manual_seed(1000 + 37 * case.F + sum(case.shape))
    x = torch.randn((n_vol,) + tuple(case.shape), generator=g, dtype=torch.float32).numpy()
    rs = np.random.RandomState(case.F * 101 + len(case.kind))
    amp = 4.0 * float(np.sqrt(np.prod(case.shape)))
    sp = [spikes_for(case.shape, case.F, rs, 2 if case.F else 1, 2, amp), spikes_for(case.shape, case.F, rs, 1, 1, amp)]
    sp = (sp + [[] for _ in range(n_vol)])[:n_vol]
    alphas = ([0.5] + [None] * n_vol)[:n_vol]
    return x, (MASK_DISK, case.F * (case.F + 1) if thr is None else thr, sp, alphas)


def _mask_terms(kind: int, n: int) -> Tuple[np.ndarray, np.ndarray]:
    i = np.arange(n)
    ineg = (2 * (n // 2) - i) % n
    if kind == MASK_DISK:
        t = lambda v: (v - n // 2) ** 2           # noqa: E731
    else:
        t = lambda v: (2 * v - (n - 1)) ** 2      # noqa: E731
    return t(i).astype(np.int64), t(ineg).astype(np.int64)


def meff(shape: Sequence[int], kind: int, thr: int) -> np.ndarray:
    """M_eff over the fftshift-ed grid, float64 in {0, 1/2, 1}."""
    tp, tn = zip(*(_mask_terms(kind, n) for n in shape))
    qp = tp[0][:, None, None] + tp[1][None, :, None] + tp[2][None, None, :]
    qn = tn[0][:, None, None] + tn[1][None, :, None] + tn[2][None, None, :]
    return 0.5 * ((qp <= thr).astype(np.float64) + (qn <= thr).astype(np.float64))


def wrap_weight(shape: Sequence[int], alpha: Optional[float]) -> np.ndarray:
    w = np.ones(tuple(shape))
    if alpha is not None:
        for ax, n in enumerate(shape):
            sl = [slice(None)] * 3
            sl[ax] = slice(1, n, 2)
            w[tuple(sl)] *= alpha
    return w


def chain_ref(x, kind: int, thr: int, spikes=None, wrap_alpha=None, abt=None) -> np.ndarray:
    """x: (V, H, W, D) array-like.  spikes: None, or one list of (fftshift-ed (h, w, d), amplitude) per volume;
    wrap_alpha: None or one value (or one per volume); abt: None or (V, 3) prologue coefficients (a, b, t).
    Returns y as float64."""
    x = np.asarray(x, dtype=np.float64)
    V = x.shape[0]
    shape = x.shape[-3:]
    if abt is not None:
        abt = np.asarray(abt, dtype=np.float64).reshape(V, 3, 1, 1, 1)
        x = np.where(x != 0, abt[:, 0] * x + abt[:, 1], abt[:, 2])
    k = np.fft.fftshift(np.fft.fftn(x, axes=AXES), axes=AXES)
    m = meff(shape, kind, thr)
    k = np.where(m > 0, k * m, 0.0)                # +0, so that angle() of a masked bin is 0
    alphas = wrap_alpha if isinstance(wrap_alpha, (list, tuple)) else [wrap_alpha] * V
    for v in range(V):
        for idx, amp in (spikes[v] if spikes is not None else ()):
            ko = k[(v,) + tuple(idx)]
            k[(v,) + tuple(idx)] = amp * ko / abs(ko) if ko != 0 else amp
        k[v] *= wrap_weight(shape, alphas[v])
    return np.fft.ifftn(np.fft.ifftshift(k, axes=AXES), axes=AXES).real


def errors(y, ref) -> Tuple[float, float]:
    """(image-domain rel-L2, max over ALL bins of |FFT(y) - FFT(ref)| / RMS of ref's nonzero bins), each the worst
    volume's."""
    y = np.asarray(y, dtype=np.float64).reshape((-1,) + tuple(np.shape(ref)[-3:]))
    ref = np.asarray(ref, dtype=np.float64).reshape(y.shape)
    worst_l2 = worst_bin = 0.0
    for v in range(y.shape[0]):
        den = np.linalg.norm(ref[v])
        worst_l2 = max(worst_l2, float(np.linalg.norm(y[v] - ref[v]) / den))
        ky, kr = np.fft.fftn(y[v]), np.fft.fftn(ref[v])
        mag = np.abs(kr)
        kept = mag > 1e-9 * mag.max()
        rms = np.sqrt(np.mean(mag[kept] ** 2))
        worst_bin = max(worst_bin, float(np.abs(ky - kr).max() / rms))
    return worst_l2, worst_bin
