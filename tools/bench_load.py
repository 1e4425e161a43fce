"""LoadImaged on the GPU (mvtb.nifti) at the scripts' size: a 4 x 240 x 240 x 155 float32 image with an LPS sform plus a
uint8 {0, 1, 2, 3} label, written as .nii and .nii.gz to a temporary directory (deleted at exit; the files are read from
the page cache).  Prints one JSON line with the card and its power limit (read in this run):

* decode kernel: device time of mvtb_nifti_decode_f32 (CUDA events, payload already on the device, 143 MB in > L2), its
  GB/s counted as bitpix / 8 + 4 bytes per voxel against the measured 6 545.6 GB/s, and torch's own composition on the
  same payload (view(dtype) -> float() -> permute().contiguous()) in the same run;
* files -> training grid: samples/s of LoadImaged -> AsChannelFirstd -> ConvertToMultiChannelBasedOnBratsClassesd ->
  SpacingOrientationd((1.5, 1.5, 2.0), "RAS"), for .nii and .nii.gz at 1 and N threads, against the host restatement
  (numpy decode, moveaxis, to_device, the same GPU resample) on the same files and thread counts;
* the share of a 1-thread load spent reading / inflating on the host (the same reads with no copy and no kernel).
The synthetic image is noise inside an ellipsoid, zeros outside: it does not compress like MRI, so the gzip level is
recorded.  Measurement tool, not product code.  Usage: python tools/bench_load.py [--threads 8] [--samples 16]"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import filters_and_operators as F  # noqa: E402
from mvtb import _lib, functional as Fn, nifti as N, spatial as S  # noqa: E402
from oracle import nifti_writer as W, ref_port as P  # noqa: E402

PEAK_GBS = 6545.6                   # measured HBM read + write bandwidth of the B200 this project is tuned on
SHAPE, PIXDIM, LEVEL, N_FILES = (240, 240, 155), (1.5, 1.5, 2.0), 1, 8
LPS = np.array([[-1.0, 0, 0, 120.0], [0, -1.0, 0, 120.0], [0, 0, 1.0, -77.0]])
KEYS = ["image", "label"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], float(q[1])
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def event_time(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / iters


def decode_rates(dev, iters):
    """per datatype: our kernel and torch's composition on the same device-resident payload"""
    res = {}
    img = np.moveaxis(P.synthetic_volume(1, (4,) + SHAPE).numpy(), 0, -1)
    for name, code, x in (("float32_image", 16, img), ("int16_image", 4, (img * 300).astype(np.int16)),
                          ("uint8_label", 2, (np.abs(img[..., 0]) * 2).astype(np.uint8))):
        dims = x.shape + (1,) * (4 - x.ndim)
        tdt = {np.float32: torch.float32, np.int16: torch.int16, np.uint8: torch.uint8}[x.dtype.type]
        raw = torch.from_numpy(np.frombuffer(x.tobytes(order="F"), np.uint8).copy()).to(dev)
        out = torch.empty((dims[3],) + dims[:3], dtype=torch.float32, device=dev)
        L = _lib.lib()
        args = (code, 0, (C.c_int64 * 4)(*dims), 1.0, 0.0, 0)

        def ours():
            _lib.check(L, L.mvtb_nifti_decode_f32(Fn._ptr(raw), Fn._ptr(out), *args, Fn._stream(dev)))

        def composed():
            return raw.view(tdt).float().view(dims[3], dims[2], dims[1], dims[0]) \
                .permute(0, 3, 2, 1).contiguous()

        t_ours, t_torch = event_time(ours, iters), event_time(composed, iters)
        assert torch.equal(out, composed())
        nbytes = int(np.prod(dims)) * (x.dtype.itemsize + 4)
        res[name] = {"us": 1e6 * t_ours, "gb_per_s": nbytes / t_ours / 1e9, "share_of_measured_peak": nbytes / t_ours / 1e9 / PEAK_GBS,
                     "torch_composition_us": 1e6 * t_torch, "torch_composition_gb_per_s": nbytes / t_torch / 1e9,
                     "speedup_over_torch": t_torch / t_ours, "bytes_per_voxel": x.dtype.itemsize + 4}
    return res


def write_files(tmp):
    img = np.moveaxis(P.synthetic_volume(2, (4,) + SHAPE).numpy(), 0, -1)
    lab = np.zeros(SHAPE, np.uint8)
    lab[60:180, 50:190, 30:120] = np.random.RandomState(3).randint(0, 4, size=(120, 140, 90))
    files = {}
    for ext, members in ((".nii", 0), (".nii.gz", 1)):
        t0 = time.perf_counter()
        ip = W.write(os.path.join(tmp, "img0" + ext), img, sform=LPS, gzip_members=members, level=LEVEL)
        lp = W.write(os.path.join(tmp, "seg0" + ext), lab, sform=LPS, gzip_members=members, level=LEVEL)
        pairs = [(ip, lp)]
        for n in range(1, N_FILES):
            pairs.append((shutil.copyfile(ip, os.path.join(tmp, f"img{n}{ext}")), shutil.copyfile(lp, os.path.join(tmp, f"seg{n}{ext}"))))
        files[ext] = {"pairs": pairs, "image_mb": os.path.getsize(ip) / 1e6, "label_mb": os.path.getsize(lp) / 1e6,
                      "write_s": time.perf_counter() - t0}
    return files


resample = S.SpacingOrientationd(KEYS, PIXDIM, axcodes="RAS", mode=("bilinear", "nearest"))
load_d = N.LoadImaged(KEYS)
first_d = N.AsChannelFirstd("image")
multi_d = F.ConvertToMultiChannelBasedOnBratsClassesd("label")


def gpu_sample(pair):
    d = resample(multi_d(first_d(load_d({"image": pair[0], "label": pair[1]}))))
    torch.cuda.current_stream().synchronize()
    return d


def host_sample(pair):
    img, lab = W.decode_reference(pair[0]), W.decode_reference(pair[1])[0]
    h = N.read_header(pair[0])
    d = {"image": np.moveaxis(np.moveaxis(img, 0, -1), -1, 0), "label": lab,
         "image_meta_dict": {"affine": h.affine.copy()}, "label_meta_dict": {"affine": h.affine.copy()}}
    d = multi_d(d)
    d = dict(d, image=Fn.to_device(d["image"])[0], label=Fn.to_device(d["label"])[0])
    d = resample(d)
    torch.cuda.current_stream().synchronize()
    return d


def rate(fn, pairs, threads, samples):
    work = [pairs[i % len(pairs)] for i in range(samples)]
    fn(work[0])
    t0 = time.perf_counter()
    if threads == 1:
        for p in work:
            fn(p)
    else:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(fn, work))
    return samples / (time.perf_counter() - t0)


def host_read_share(pairs, reps):
    """1 thread: seconds per sample of load() alone (synchronised) and of the same reads / inflation with no copy"""
    buf = bytearray(4 << 20)

    def read_only(p):
        with N._Source(p) as src:
            while src.readinto(memoryview(buf)) == len(buf):
                pass

    def load_only(p):
        N.load(p)
        torch.cuda.current_stream().synchronize()

    out = {}
    for name, fn in (("read_s", read_only), ("load_s", load_only)):
        for p in pairs[0]:
            fn(p)
        t0 = time.perf_counter()
        for i in range(reps):
            for p in pairs[i % len(pairs)]:
                fn(p)
        out[name] = (time.perf_counter() - t0) / reps
    out["host_read_share"] = out["read_s"] / out["load_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--samples", type=int, default=16, help="samples per timed run at N threads (half that at 1 thread)")
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_load needs a CUDA device")
    dev = torch.device("cuda:0")
    name, plim = card()
    result = {"tool": "bench_load", "gpu": name, "power_limit_w": plim, "host_threads": os.cpu_count(),
              "geometry": {"image": [*SHAPE, 4], "label": list(SHAPE), "pixdim": PIXDIM, "axcodes": "RAS"},
              "gzip_level": LEVEL, "peak_gb_per_s": PEAK_GBS, "decode": decode_rates(dev, args.iters)}
    tmp = tempfile.mkdtemp(prefix="bench_load_")
    try:
        files = write_files(tmp)
        pairs = files[".nii"]["pairs"]
        g, h = gpu_sample(pairs[0]), host_sample(pairs[0])
        parity = all(torch.equal(g[k].cpu(), h[k].cpu()) for k in KEYS)
        e2e = {}
        for ext, f in files.items():
            row = {"image_mb": f["image_mb"], "label_mb": f["label_mb"]}
            for threads, samples in ((1, max(2, args.samples // 2)), (args.threads, args.samples)):
                row[f"gpu_load_samples_per_s_{threads}t"] = rate(gpu_sample, f["pairs"], threads, samples)
                row[f"host_path_samples_per_s_{threads}t"] = rate(host_sample, f["pairs"], threads, samples)
            row.update(host_read_share(f["pairs"], 4))
            e2e[ext] = row
        result["files_to_grid"] = e2e
        result["parity_gpu_equals_host_path"] = parity
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
