"""Spacingd -> Orientationd on the GPU (mvtb.spatial.resample) at the scripts' geometry: a 4 x 240 x 240 x 155 image at 1 mm
to 4 x 160 x 160 x 78 (pixdim 1.5, 1.5, 2.0, bilinear) plus its 3-channel label (nearest), reoriented to RAS from an LPS
affine.  Prints one JSON line: the card and its power limit (read in this run), samples/s of the gather, its bytes/s
counted as 4 (in + out) voxels against the measured 6 545.6 GB/s peak, and on the same input torch's GPU grid_sample
(fp32, and fp64 as MONAI runs it) and the CPU oracle (MONAI's arithmetic on the host threads); plus a parity spot check.
Measurement tool, not product code.  Usage: python tools/bench_resample.py [--batch 8] [--iters 20]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from mvtb import geometry as G, spatial as S  # noqa: E402
from oracle import monai_resample as O, ref_port as P  # noqa: E402

PEAK_GBS = 6545.6                   # measured HBM read + write bandwidth of the B200 this project is tuned on
SHAPE, PIXDIM = (240, 240, 155), (1.5, 1.5, 2.0)
LPS = np.diag([-1.0, -1.0, 1.0, 1.0]) @ np.array([[1, 0, 0, -120.0], [0, 1, 0, -120.0], [0, 0, 1, -77.0], [0, 0, 0, 1]])


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], float(q[1])
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def timed(fn, iters, warmup=3):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8, help="samples per call (8: 1.1 GB of image, well over the 126 MB L2)")
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resample needs a CUDA device")
    dev = torch.device("cuda:0")
    name, plim = card()
    B = args.batch
    img1 = P.synthetic_volume(1, (4,) + SHAPE).numpy()
    lab1 = (P.synthetic_volume(2, (3,) + SHAPE).numpy() > 0.5).astype(np.float32)
    img = torch.from_numpy(img1).to(dev).repeat(B, 1, 1, 1)           # B samples of one geometry stacked on the channels
    lab = torch.from_numpy(lab1).to(dev).repeat(B, 1, 1, 1)
    p = G.plan(LPS, SHAPE, PIXDIM, axcodes="RAS")

    def ours():
        S.resample(img, p, "bilinear")
        S.resample(lab, p, "nearest")

    t_ours = timed(ours, args.iters)
    vox = 7 * B * (np.prod(SHAPE) + np.prod(p.shape))
    gbs = 4 * vox / t_ours / 1e9

    # torch's GPU grid_sample on the same input: MONAI's call (affine_grid over the full grid), then the flips
    sp = p.spacing
    theta = G.affine_theta(sp.transform, SHAPE, sp.shape)[:, :3]

    def torch_gs(dtype):
        th = theta.to(dev, dtype)
        gi = F.affine_grid(th.expand(B, 3, 4), [B, 4] + list(sp.shape), align_corners=False)
        gl = F.affine_grid(th.expand(B, 3, 4), [B, 3] + list(sp.shape), align_corners=False)
        xi, xl = img.view(B, 4, *SHAPE).to(dtype), lab.view(B, 3, *SHAPE).to(dtype)

        def run():
            a = F.grid_sample(xi, gi, mode="bilinear", padding_mode="border", align_corners=False).flip(2, 3).float()
            b = F.grid_sample(xl, gl, mode="nearest", padding_mode="border", align_corners=False).flip(2, 3).float()
            return a, b
        return run

    t_t32 = timed(torch_gs(torch.float32), max(3, args.iters // 4))
    t_t64 = timed(torch_gs(torch.float64), max(3, args.iters // 4), warmup=1)

    # the oracle on the host threads: one sample
    t0 = time.perf_counter()
    ref_img, ref_aff = O.spacing_orientation(img1, LPS, PIXDIM, "RAS", mode="bilinear")
    ref_lab, _ = O.spacing_orientation(lab1, LPS, PIXDIM, "RAS", mode="nearest")
    t_cpu = time.perf_counter() - t0

    # parity spot check on sample 0 (and the last sample of the batch)
    gi, gl = S.resample(img[:4], p, "bilinear").cpu().numpy(), S.resample(lab[-3:], p, "nearest").cpu().numpy()
    err = float(np.abs(gi - ref_img).max() / np.abs(ref_img).max())
    print(json.dumps({
        "tool": "bench_resample", "gpu": name, "power_limit_w": plim, "batch": B,
        "geometry": {"in": [4, *SHAPE], "out": [4, *p.shape], "label_channels": 3, "pixdim": PIXDIM, "axcodes": "RAS",
                     "path": "separable" if S.tap_tables(p, False) is not None else "general"},
        "samples_per_s": B / t_ours, "ms_per_sample": 1e3 * t_ours / B,
        "gb_per_s": gbs, "share_of_measured_peak": gbs / PEAK_GBS, "peak_gb_per_s": PEAK_GBS,
        "torch_gpu_fp32_samples_per_s": B / t_t32, "torch_gpu_fp64_samples_per_s": B / t_t64,
        "oracle_cpu_samples_per_s": 1.0 / t_cpu, "oracle_cpu_threads": torch.get_num_threads(),
        "parity": {"image_max_rel_err": err, "label_equal": bool(np.array_equal(gl, ref_lab)),
                   "affine_equal": bool(np.array_equal(p.affine, ref_aff))},
    }))


if __name__ == "__main__":
    main()
