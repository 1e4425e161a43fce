"""LoadImaged on the GPU: NIfTI-1/2 files read into pinned memory and decoded to channel-first float32 on the device, no
nibabel (127_...FLAIR.py:117-119, utils.py:186-188: LoadImaged -> AsChannelFirstd -> ConvertToMultiChannelBasedOnBratsClassesd).

The host does only what it must: read the file (and inflate a `.nii.gz` with zlib).  The payload goes straight into a
per-thread ring of pinned chunks, each chunk is copied to the device while the next is read, and one kernel
(`mvtb_nifti_decode_f32`, csrc/nifti.cuh) converts the type, swaps the bytes, scales, and turns file order into
(C, X, Y, Z).  The format rules below are restated from nibabel and MONAI 0.5 and **not pinned against nibabel**:

* header: NIfTI-1 (348 bytes, magic "n+1") or NIfTI-2 (540 bytes, "n+2\\0\\r\\n\\032\\n"); the byte order is the one in
  which sizeof_hdr reads 348 / 540; extensions up to vox_offset are skipped.  `.hdr`/`.img` pairs, dim[0] other than 3 or
  4, and datatypes other than uint8, int8, int16, uint16, int32, uint32, float32, float64 raise NotImplementedError; a
  malformed or truncated file raises ValueError.
* affine (nibabel's get_best_affine): sform_code > 0: the srow_* rows as float64; else qform_code > 0: quaternion
  (b, c, d) with a = sqrt(1 - b^2 - c^2 - d^2) (0 when |1 - b^2 - c^2 - d^2| < 3 float32 eps), rotation times
  diag(pixdim[1], pixdim[2], qfac pixdim[3]), qoffset translation; else shape_zoom_affine(shape, pixdim, x_flip=True).
  As nibabel's load-time check repairs them: qfac = pixdim[0] is -1 or else 1, and pixdim[1:4] are taken as |pixdim|.
* values (NibabelReader.get_fdata(dtype=float32)): scl_slope 0 or not finite: no scaling; a non-finite scl_inter reads
  as 0; (slope, inter) == (1, 0): no arithmetic; otherwise raw * slope + inter in np.result_type(raw, float32) (float32 for
  8/16-bit integers and float32, float64 for 32-bit integers and float64), multiply and add rounded separately, then
  rounded to float32.  Unscaled 32-bit integers and float64 round to nearest even."""
import ctypes as C
import math
import struct
import threading
import zlib
from typing import NamedTuple, Tuple

import numpy as np
import torch

from . import _lib, functional as Fn
from ._monai_compat import KeysCollection, MapTransform

# NIfTI datatype code -> numpy element type
DTYPES = {2: np.uint8, 4: np.int16, 8: np.int32, 16: np.float32, 64: np.float64, 256: np.int8, 512: np.uint16, 768: np.uint32}
_CHUNK_BYTES = 4 << 20          # pinned chunk: 4 MB ...
_RING = 4                       # ... four per thread and device
_GZ_BLOCK = 1 << 20             # compressed bytes read at a time


class Header(NamedTuple):
    path: str
    version: int                # 1 or 2
    byteorder: str              # "<" or ">"
    shape: Tuple[int, ...]      # dim[1 : dim[0] + 1]
    datatype: int
    vox_offset: int
    scl_slope: float
    scl_inter: float
    pixdim: Tuple[float, ...]   # after nibabel's repairs (qfac +-1, |pixdim[1:4]|)
    qform_code: int
    sform_code: int
    affine: np.ndarray          # 4x4 float64

    @property
    def channels(self) -> int:
        return self.shape[3] if len(self.shape) == 4 else 1

    @property
    def payload_bytes(self) -> int:
        return math.prod(self.shape) * np.dtype(DTYPES[self.datatype]).itemsize


# ----------------------------------------------------------------------------- reading

class _GzipReader:
    """readinto() over the inflated bytes of a (multi-member) gzip file, as the gzip module reads it: members follow one
    another, zero bytes between them are padding, and a member cut short is an error."""

    def __init__(self, f, path):
        self.f, self.path = f, path
        self.d = None            # the current member's decompressor; None between members
        self.tail = b""          # compressed bytes not yet given to self.d

    def _more(self) -> bytes:
        return self.f.read(_GZ_BLOCK)

    def readinto(self, mv) -> int:
        n, want = 0, len(mv)
        while n < want:
            if self.d is None:
                self.tail = self.tail.lstrip(b"\0")
                while not self.tail:
                    self.tail = self._more()
                    if not self.tail:
                        return n
                    self.tail = self.tail.lstrip(b"\0")
                self.d = zlib.decompressobj(16 + zlib.MAX_WBITS)
            try:
                out = self.d.decompress(self.tail, want - n)
                if not out and not self.d.eof:
                    self.tail = self._more()           # zlib has nothing pending: it needs input
                    if not self.tail:
                        raise ValueError(f"{self.path}: gzip stream ends inside a member")
                    out = self.d.decompress(self.tail, want - n)
            except zlib.error as e:
                raise ValueError(f"{self.path}: gzip error: {e}") from None
            self.tail = self.d.unused_data if self.d.eof else self.d.unconsumed_tail
            if self.d.eof:
                self.d = None
            mv[n:n + len(out)] = out
            n += len(out)
        return n


class _Source:
    """the file's (inflated) bytes through readinto(); gzip is recognised by its magic bytes"""

    def __init__(self, path):
        self.path = str(path)
        self.f = open(self.path, "rb")
        self.r = _GzipReader(self.f, self.path) if self.f.peek(2)[:2] == b"\x1f\x8b" else self.f

    def readinto(self, mv) -> int:
        """fills mv unless the file ends first; returns the bytes read"""
        n = 0
        while n < len(mv):
            k = self.r.readinto(mv[n:])
            if not k:
                break
            n += k
        return n

    def close(self):
        self.f.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _read_exact(src: _Source, n: int, chunk_bytes: int, what: str) -> bytearray:
    """n bytes in reads of at most chunk_bytes; ValueError if the file ends first"""
    buf = bytearray(n)
    mv, got = memoryview(buf), 0
    while got < n:
        step = min(chunk_bytes, n - got)
        k = src.readinto(mv[got:got + step])
        got += k
        if k < step:
            raise ValueError(f"{src.path}: file ends {got} bytes into the {what} ({n} bytes)")
    return buf


# ----------------------------------------------------------------------------- header and affine

_N1_MAGIC, _N2_MAGIC = b"n+1\0", b"n+2\0\r\n\x1a\n"


def _quat_affine(bcd, pixdim, qfac, offset, path):
    b, c, d = (float(v) for v in bcd)
    w2 = 1.0 - (b * b + c * c + d * d)
    if abs(w2) < 3 * float(np.finfo(np.float32).eps):
        a = 0.0
    elif w2 < 0:
        raise ValueError(f"{path}: qform quaternion (b, c, d) = {(b, c, d)} has norm over 1")
    else:
        a = math.sqrt(w2)
    n = a * a + b * b + c * c + d * d                      # nibabel's quat2mat
    if n < np.finfo(np.float64).eps:
        R = np.eye(3)
    else:
        s = 2.0 / n
        X, Y, Z = b * s, c * s, d * s
        wX, wY, wZ, xX, xY, xZ, yY, yZ, zZ = a * X, a * Y, a * Z, b * X, b * Y, b * Z, c * Y, c * Z, d * Z
        R = np.array([[1.0 - (yY + zZ), xY - wZ, xZ + wY], [xY + wZ, 1.0 - (xX + zZ), yZ - wX], [xZ - wY, yZ + wX, 1.0 - (xX + yY)]])
    vox = np.array(pixdim[1:4], dtype=np.float64)
    vox[2] *= qfac
    out = np.eye(4)
    out[:3, :3] = R @ np.diag(vox)
    out[:3, 3] = offset
    return out


def _fallback_affine(shape, pixdim):
    """nibabel's shape_zoom_affine(shape, zooms, x_flip=True)"""
    sh = np.array((list(shape[:3]) + [1, 1])[:3], dtype=np.float64)
    z = np.array((list(pixdim[1:len(shape[:3]) + 1]) + [1.0, 1.0])[:3], dtype=np.float64)
    z[0] *= -1
    aff = np.eye(4)
    aff[:3, :3] = np.diag(z)
    aff[:3, 3] = -(sh - 1) / 2.0 * z
    return aff


def _parse(raw: bytes, path: str) -> Header:
    """raw: the first 348 (NIfTI-1) or 540 (NIfTI-2) bytes"""
    n1 = len(raw) == 348
    o = "<" if struct.unpack_from("<i", raw, 0)[0] == len(raw) else ">"
    u = lambda fmt, off: struct.unpack_from(o + fmt, raw, off)   # noqa: E731
    if n1:
        magic = bytes(raw[344:348])
        if magic == b"ni1\0":
            raise NotImplementedError(f"{path}: a .hdr/.img pair (magic 'ni1') is not supported; only single-file NIfTI")
        if magic != _N1_MAGIC:
            raise ValueError(f"{path}: bad NIfTI-1 magic {magic!r}")
        dim = u("8h", 40)
        datatype = u("h", 70)[0]
        pixdim = list(u("8f", 76))
        vox_offset, slope, inter = u("3f", 108)
        qcode, scode = u("hh", 252)
        quat = u("6f", 256)
        srow = u("12f", 280)
    else:
        magic = bytes(raw[4:12])
        if magic[:4] == b"ni2\0":
            raise NotImplementedError(f"{path}: a .hdr/.img pair (magic 'ni2') is not supported; only single-file NIfTI")
        if magic != _N2_MAGIC:
            raise ValueError(f"{path}: bad NIfTI-2 magic {magic!r}")
        datatype = u("h", 12)[0]
        dim = u("8q", 16)
        pixdim = list(u("8d", 104))
        vox_offset = u("q", 168)[0]
        slope, inter = u("2d", 176)
        qcode, scode = u("ii", 344)
        quat = u("6d", 352)
        srow = u("12d", 400)
    nd = dim[0]
    if not 1 <= nd <= 7:
        raise ValueError(f"{path}: dim[0] = {nd}")
    if nd not in (3, 4):
        raise NotImplementedError(f"{path}: {nd}-D image: only 3-D (X, Y, Z) and 4-D (X, Y, Z, C) files are supported")
    shape = tuple(int(v) for v in dim[1:nd + 1])
    if min(shape) < 1:
        raise ValueError(f"{path}: dim {shape} has an axis below 1")
    if datatype not in DTYPES:
        raise NotImplementedError(f"{path}: NIfTI datatype {datatype} is not supported "
                                  "(uint8, int8, int16, uint16, int32, uint32, float32, float64 are)")
    if not math.isfinite(vox_offset) or vox_offset < len(raw):
        raise ValueError(f"{path}: vox_offset {vox_offset} lies inside the {len(raw)}-byte header")
    pixdim[0] = -1.0 if pixdim[0] == -1 else 1.0
    pixdim[1:4] = [abs(v) for v in pixdim[1:4]]
    if scode > 0:
        affine = np.eye(4)
        affine[:3] = np.array(srow, dtype=np.float64).reshape(3, 4)
    elif qcode > 0:
        affine = _quat_affine(quat[:3], pixdim, pixdim[0], np.array(quat[3:], dtype=np.float64), path)
    else:
        affine = _fallback_affine(shape, pixdim)
    return Header(path, 1 if n1 else 2, o, shape, int(datatype), int(vox_offset), float(slope), float(inter), tuple(pixdim),
                  int(qcode), int(scode), affine)


def _header(src: _Source, chunk_bytes: int) -> Header:
    """reads the header and skips to vox_offset (extensions), in reads of at most chunk_bytes"""
    first = _read_exact(src, 4, chunk_bytes, "header")
    sizes = {struct.unpack("<i", first)[0], struct.unpack(">i", first)[0]}
    if 348 in sizes:
        n = 348
    elif 540 in sizes:
        n = 540
    else:
        raise ValueError(f"{src.path}: sizeof_hdr {struct.unpack('<i', first)[0]} reads neither 348 nor 540 in either byte order")
    hdr = _parse(bytes(first) + bytes(_read_exact(src, n - 4, chunk_bytes, "header")), src.path)
    skip = hdr.vox_offset - n
    while skip > 0:
        k = min(skip, chunk_bytes)
        _read_exact(src, k, chunk_bytes, f"extensions before vox_offset {hdr.vox_offset}")
        skip -= k
    return hdr


def read_header(path, _chunk_bytes: int = _CHUNK_BYTES) -> Header:
    """the header of a .nii / .nii.gz file, with nibabel's best affine (see the module docstring)"""
    with _Source(path) as src:
        return _header(src, _chunk_bytes)


def value_rule(hdr: Header):
    """(scaled, slope, inter) of the value rule"""
    s, i = hdr.scl_slope, hdr.scl_inter
    if s == 0 or not math.isfinite(s):
        return False, 1.0, 0.0
    i = i if math.isfinite(i) else 0.0
    return not (s == 1 and i == 0), s, i


def decode_args(hdr: Header):
    """the arguments of mvtb_nifti_decode_f32 after (raw, out): datatype, swap_bytes (the device is little-endian), dims,
    slope, inter, scaled"""
    scaled, s, i = value_rule(hdr)
    X, Y, Z = hdr.shape[:3]
    return hdr.datatype, int(hdr.byteorder == ">"), (C.c_int64 * 4)(X, Y, Z, hdr.channels), s, i, int(scaled)


# ----------------------------------------------------------------------------- load

_tls = threading.local()


def _ring(dev: torch.device, chunk_bytes: int):
    """the calling thread's pinned chunks for `dev`: [(host uint8 tensor, its memoryview, event or None)]"""
    rings = getattr(_tls, "rings", None)
    if rings is None:
        rings = _tls.rings = {}
    key = (dev.index, chunk_bytes)
    r = rings.get(key)
    if r is None:
        r = []
        for _ in range(_RING):
            t = torch.empty(chunk_bytes, dtype=torch.uint8, pin_memory=True)
            r.append([t, memoryview(t.numpy()), None])
        rings[key] = r
    return r


def _read_payload(src: _Source, hdr: Header, views, before, after) -> None:
    """reads the payload into the chunk views in turn: before(slot) ahead of refilling one, after(slot, offset, n) once
    it holds payload bytes [offset, offset + n)"""
    nbytes, off, slot = hdr.payload_bytes, 0, 0
    while off < nbytes:
        before(slot)
        m = min(len(views[slot]), nbytes - off)
        got = src.readinto(views[slot][:m])
        if got < m:
            raise ValueError(f"{hdr.path}: {off + got} payload bytes after vox_offset {hdr.vox_offset}, "
                             f"{nbytes} needed for {hdr.shape} of datatype {hdr.datatype}")
        after(slot, off, m)
        off += m
        slot = (slot + 1) % len(views)


def load(path, _chunk_bytes: int = _CHUNK_BYTES) -> Tuple[torch.Tensor, Header]:
    """(C, X, Y, Z) C-contiguous float32 CUDA tensor of the file's voxels (out[c, i, j, k] = voxel (i, j, k, c)), on the
    current device and stream, and the header."""
    Fn.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    stream = torch.cuda.current_stream(dev)
    with _Source(path) as src:
        hdr = _header(src, _chunk_bytes)
        raw = torch.empty(max(hdr.payload_bytes, 1), dtype=torch.uint8, device=dev)
        ring = _ring(dev, _chunk_bytes)

        def before(slot):
            if ring[slot][2] is not None:
                ring[slot][2].synchronize()                    # the copy that last read this chunk is done

        def after(slot, off, n):
            raw[off:off + n].copy_(ring[slot][0][:n], non_blocking=True)
            if ring[slot][2] is None:
                ring[slot][2] = torch.cuda.Event()
            ring[slot][2].record(stream)

        _read_payload(src, hdr, [r[1] for r in ring], before, after)          # copies run on the current stream
        out = torch.empty((hdr.channels,) + hdr.shape[:3], dtype=torch.float32, device=dev)
        L = _lib.lib()
        rc = L.mvtb_nifti_decode_f32(Fn._ptr(raw), Fn._ptr(out), *decode_args(hdr), C.c_void_p(stream.cuda_stream))
        _lib.check(L, rc)
    return out, hdr


# ----------------------------------------------------------------------------- the transforms

class LoadImaged(MapTransform):
    """MONAI 0.5 LoadImaged with its NibabelReader, on the GPU: d[key] is a path; it becomes MONAI's layout as a CUDA
    float32 view of the decoded buffer ((X, Y, Z, C) for a 4-D file, (X, Y, Z) for a 3-D one), and d[f"{key}_{postfix}"]
    gets affine, original_affine, spatial_shape and filename_or_obj."""

    def __init__(self, keys: KeysCollection, reader=None, dtype=np.float32, meta_key_postfix: str = "meta_dict",
                 overwriting: bool = False, image_only: bool = False, allow_missing_keys: bool = False) -> None:
        super().__init__(keys, allow_missing_keys)
        if reader not in (None, "NibabelReader"):
            raise NotImplementedError(f"reader {reader!r}: only the NIfTI reader (None / 'NibabelReader') is implemented")
        if np.dtype(dtype) != np.float32:
            raise NotImplementedError(f"dtype {dtype}: the decode produces float32 only")
        self.meta_key_postfix, self.overwriting, self.image_only = meta_key_postfix, overwriting, image_only

    def __call__(self, data):
        d = dict(data)
        for key in self.key_iterator(d):
            path = d[key]
            buf, hdr = load(path)
            d[key] = buf.permute(1, 2, 3, 0) if len(hdr.shape) == 4 else buf[0]
            if self.image_only:
                continue
            meta_key = f"{key}_{self.meta_key_postfix}"
            if meta_key in d and not self.overwriting:
                raise KeyError(f"Meta data with key {meta_key} already exists and overwriting=False.")
            d[meta_key] = {"affine": hdr.affine.copy(), "original_affine": hdr.affine.copy(),
                           "spatial_shape": np.asarray(hdr.shape[:3]), "filename_or_obj": path}
        return d


class AsChannelFirstd(MapTransform):
    """MONAI 0.5 AsChannelFirstd: the channel axis to the front.  A tensor gets movedim (after LoadImaged, the decoded
    contiguous buffer again), a numpy array np.moveaxis, as in MONAI."""

    def __init__(self, keys: KeysCollection, channel_dim: int = -1, allow_missing_keys: bool = False) -> None:
        super().__init__(keys, allow_missing_keys)
        if not isinstance(channel_dim, int) or channel_dim < -1:
            raise AssertionError("invalid channel dimension.")
        self.channel_dim = channel_dim

    def __call__(self, data):
        d = dict(data)
        for key in self.key_iterator(d):
            x = d[key]
            d[key] = x.movedim(self.channel_dim, 0) if isinstance(x, torch.Tensor) else np.moveaxis(x, self.channel_dim, 0)
        return d
