"""NIfTI-1/2 files for the tests and tools/bench_load.py, and a numpy restatement of what mvtb.nifti.load returns.

Test infrastructure only (struct, gzip, numpy; no nibabel).  `write` covers both header versions in either byte order,
`.nii` and single- or multi-member `.nii.gz`, the eight datatypes mvtb.nifti supports (and any other code, for the error
tests), sform / qform / fallback geometry, extensions and scaling.  `decode_reference` parses the header with a numpy
structured dtype, independently of mvtb.nifti's parser, and applies the value rule in numpy:
    slope == 0 or not finite: no scaling; non-finite inter reads as 0; (slope, inter) == (1, 0): no arithmetic;
    otherwise raw * slope + inter in np.result_type(raw dtype, float32), then astype(float32).
It returns (C, X, Y, Z) float32 with out[c, i, j, k] = file element ((c Z + k) Y + j) X + i."""
import gzip
import struct

import numpy as np

DTYPES = {2: "u1", 4: "i2", 8: "i4", 16: "f4", 64: "f8", 256: "i1", 512: "u2", 768: "u4"}
CODES = {np.dtype(v).str[1:]: k for k, v in DTYPES.items()}


def write(path, data, *, version=1, byteorder="<", datatype=None, pixdim=(1.0, 1.0, 1.0), qfac=1.0, sform=None, qform=None,
          slope=0.0, inter=0.0, extensions=(), gzip_members=0, level=6, magic=None, vox_offset=None, payload=None):
    """Write `data` ((X, Y, Z) or (X, Y, Z, C)) to `path`.
    sform: a 3x4 / 4x4 matrix (sform_code 1); qform: (b, c, d, qx, qy, qz) (qform_code 1); neither: both codes 0.
    extensions: a sequence of (ecode, bytes).  gzip_members: 0 = plain file, n = the file gzip-compressed as n members.
    magic, vox_offset, datatype, payload (raw bytes): overrides for malformed files."""
    data = np.asarray(data)
    dt = CODES[data.dtype.str[1:]] if datatype is None else datatype
    dim = [data.ndim] + list(data.shape) + [1] * (7 - data.ndim)
    pd = [qfac] + list(pixdim) + [1.0] * (7 - len(pixdim))
    ext = b""
    for code, blob in extensions:
        size = 8 + len(blob) + (-(8 + len(blob)) % 16)
        ext += struct.pack(byteorder + "ii", size, code) + blob + b"\0" * (size - 8 - len(blob))
    hsize = 348 if version == 1 else 540
    off = hsize + 4 + len(ext) if vox_offset is None else vox_offset
    sf = np.zeros((3, 4)) if sform is None else np.asarray(sform, dtype=np.float64)[:3]
    qf = (0.0,) * 6 if qform is None else tuple(qform)
    scode, qcode = int(sform is not None), int(qform is not None)
    o = byteorder
    if version == 1:
        h = bytearray(348)
        struct.pack_into(o + "i", h, 0, 348)
        struct.pack_into(o + "8h", h, 40, *dim)
        struct.pack_into(o + "hh", h, 70, dt, 8 * np.dtype(DTYPES.get(dt, "u1")).itemsize)
        struct.pack_into(o + "8f", h, 76, *pd)
        struct.pack_into(o + "3f", h, 108, off, slope, inter)
        struct.pack_into(o + "hh", h, 252, qcode, scode)
        struct.pack_into(o + "6f", h, 256, *qf)
        struct.pack_into(o + "12f", h, 280, *sf.ravel())
        h[344:348] = b"n+1\0" if magic is None else magic
    else:
        h = bytearray(540)
        struct.pack_into(o + "i", h, 0, 540)
        h[4:12] = b"n+2\0\r\n\x1a\n" if magic is None else magic
        struct.pack_into(o + "hh", h, 12, dt, 8 * np.dtype(DTYPES.get(dt, "u1")).itemsize)
        struct.pack_into(o + "8q", h, 16, *dim)
        struct.pack_into(o + "8d", h, 104, *pd)
        struct.pack_into(o + "q", h, 168, off)
        struct.pack_into(o + "2d", h, 176, slope, inter)
        struct.pack_into(o + "ii", h, 344, qcode, scode)
        struct.pack_into(o + "6d", h, 352, *qf)
        struct.pack_into(o + "12d", h, 400, *sf.ravel())
    body = bytes(h) + (b"\1\0\0\0" if ext else b"\0\0\0\0") + ext
    body = body[:max(off, len(h))] + b"\0" * max(0, off - len(body))          # a vox_offset inside the header keeps it whole
    if payload is None and dt not in DTYPES:
        payload = data.tobytes(order="F")
    elif payload is None:
        payload = data.astype(np.dtype(DTYPES[dt]).newbyteorder(o)).tobytes(order="F")
    blob = body + payload
    if gzip_members:
        cuts = np.linspace(0, len(blob), gzip_members + 1).astype(int)
        blob = b"".join(gzip.compress(blob[a:b], compresslevel=level) for a, b in zip(cuts[:-1], cuts[1:]))
    with open(path, "wb") as f:
        f.write(blob)
    return path


def _header_dtype(version, o):
    if version == 1:
        return np.dtype({"names": ["dim", "datatype", "vox_offset", "scl_slope", "scl_inter"],
                         "formats": [o + "8i2", o + "i2", o + "f4", o + "f4", o + "f4"],
                         "offsets": [40, 70, 108, 112, 116], "itemsize": 348})
    return np.dtype({"names": ["dim", "datatype", "vox_offset", "scl_slope", "scl_inter"],
                     "formats": [o + "8i8", o + "i2", o + "i8", o + "f8", o + "f8"],
                     "offsets": [16, 12, 168, 176, 184], "itemsize": 540})


def decode_reference(path):
    """(C, X, Y, Z) float32 numpy array: the file's voxels by the value rule in the module docstring"""
    with open(path, "rb") as f:
        blob = f.read()
    if blob[:2] == b"\x1f\x8b":
        blob = gzip.decompress(blob)
    for o in "<>":
        (n,) = struct.unpack_from(o + "i", blob, 0)
        if n in (348, 540):
            break
    h = np.frombuffer(blob, _header_dtype(1 if n == 348 else 2, o), count=1)[0]
    nd = int(h["dim"][0])
    X, Y, Z = (int(v) for v in h["dim"][1:4])
    C = int(h["dim"][4]) if nd == 4 else 1
    raw = np.frombuffer(blob, np.dtype(DTYPES[int(h["datatype"])]).newbyteorder(o), count=X * Y * Z * C,
                        offset=int(h["vox_offset"]))
    raw = raw.reshape(C, Z, Y, X).transpose(0, 3, 2, 1)
    slope, inter = h["scl_slope"], h["scl_inter"]
    if slope == 0 or not np.isfinite(slope):
        return raw.astype(np.float32)
    inter = inter if np.isfinite(inter) else 0.0
    if slope == 1 and inter == 0:
        return raw.astype(np.float32)
    rt = np.result_type(raw.dtype, np.float32)
    return (raw.astype(rt) * rt.type(slope) + rt.type(inter)).astype(np.float32)
