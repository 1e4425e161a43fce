"""The training loader's batch stage (mvtb.train_stage) at the 127 scripts' shapes: a DeviceCache of 64 synthetic samples on
the training grid (4 x 160 x 160 x 78 image + 3-channel label), the tail RandSpatialCropd(128, 128, 64) -> RandFlipd ->
SelectChanneld(image, 0) -> NormalizeIntensityd -> RandScaleIntensityd -> RandShiftIntensityd -> disk 12.5 -> plane wave
-> wrap 0.5 -> SaltAndPepper(0.05, philox-sparse).  Prints one JSON line: the card and its power limit (read in this run),
and for (a) TrainStage.apply(draw(...)) at batch 2 and 64 and (b) the same transform objects called per sample through the
drop-ins at batch 2: samples/s, library launches per batch (mvtb_launch_count), and the nominal bytes per output image voxel
computed from shapes with the share of the measured 6 545.6 GB/s.  CUDA events around each batch with a synchronise; a
256 MB buffer is overwritten between batches so the L2 holds nothing of the cache.  Each figure is the median over
--repeats windows of --steps batches (batch 64 and the per-sample path: a quarter of the steps), with the smallest and largest window beside it.
Measurement tool, not product code.  Usage: python tools/bench_train_stage.py [--out FILE]"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

PEAK_GBS = 6545.6                   # measured HBM read + write bandwidth of the B200 this project is tuned on
GRID, ROI, N_ITEMS = (160, 160, 78), (128, 128, 64), 64


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], float(q[1])
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def tail(seed):
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(["image", "label"], roi_size=list(ROI), random_size=False),
         S.RandFlipd(["image", "label"], prob=0.5, spatial_axis=0), F.SelectChanneld("image", 0),
         I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), I.RandScaleIntensityd("image", factors=0.1, prob=0.5),
         I.RandShiftIntensityd("image", offsets=0.1, prob=0.5), F.RandFourierDiskMaskd("image", r=12.5, inside_off=False, prob=1.0),
         F.RandPlaneWaves_ellipsoid("image", 55, 55, 30, intensity_value=15, prob=1.0), F.WrapArtifactd("image", alpha=0.5),
         F.SaltAndPepper(0.05, "image", prob=1.0, rng="philox-sparse", seed=2024)]
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
    return t


def timed(fn, steps, repeats, warmup, flush):
    """(seconds per batch: median, min, max over the windows; library launches per batch)"""
    from mvtb import _lib
    L = _lib.lib()
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    n0, windows = L.mvtb_launch_count(), []
    for _ in range(repeats):
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        windows.append(tot / 1e3 / steps)
    return (float(np.median(windows)), min(windows), max(windows)), (L.mvtb_launch_count() - n0) / (steps * repeats)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=400, help="batches per timed window")
    ap.add_argument("--repeats", type=int, default=5, help="timed windows")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_stage needs a CUDA device")
    from mvtb.train_stage import DeviceCache, TrainStage
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plim = card()
    g = torch.Generator(device=dev).manual_seed(5)
    items = []
    for i in range(N_ITEMS):
        img = torch.randn((4,) + GRID, device=dev, generator=g).abs_()
        img *= img > 0.3                                            # zero background
        lab = (torch.rand((3,) + GRID, device=dev, generator=g) < 0.2).to(torch.float32)
        items.append({"image": img, "label": lab})
    cache = DeviceCache(items, [], num_workers=1)
    del items
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    rng = np.random.RandomState(1)
    res = {"metric": "train stage samples/s (127 tail, 128x128x64 crops of 4x160x160x78 + 3-channel label)", "card": name,
           "power_limit_w": plim, "cache_items": N_ITEMS, "cache_bytes": sum(b.numel() * 4 for b in cache.buffers.values())}
    vox = math.prod(ROI)
    # nominal traffic per sample from shapes: image gather 8 B/voxel (1 selected channel), statistics 4, chain with the map on
    # load and the select behind it 8; label gather 3 channels x 8
    bytes_per_sample = vox * (8 + 4 + 8) + 3 * vox * 8
    res["bytes_per_output_image_voxel"] = bytes_per_sample / vox
    with torch.no_grad():
        for bs in (2, 64):
            stage = TrainStage(cache, tail(0))
            (sec, lo, hi), launches = timed(lambda: stage.apply(stage.draw(rng.randint(0, N_ITEMS, bs))),
                                            max(args.steps // (1 if bs == 2 else 4), 5), args.repeats, 3, flush)
            res[f"batched_b{bs}"] = {"samples_per_s": bs / sec, "samples_per_s_range": [bs / hi, bs / lo], "ms_per_batch": sec * 1e3,
                                     "launches_per_batch": launches, "gbs": bs * bytes_per_sample / sec / 1e9,
                                     "share_of_peak": bs * bytes_per_sample / sec / 1e9 / PEAK_GBS}
        ref = tail(0)

        def per_sample():
            for i in rng.randint(0, N_ITEMS, 2):
                d = cache.item(int(i))
                for t in ref:
                    d = t(d)
        (sec, lo, hi), launches = timed(per_sample, max(args.steps // 4, 5), args.repeats, 3, flush)
        res["per_sample_b2"] = {"samples_per_s": 2 / sec, "samples_per_s_range": [2 / hi, 2 / lo], "ms_per_batch": sec * 1e3,
                                "launches_per_batch": launches}
    res["steps_per_window"], res["windows"] = args.steps, args.repeats
    res["speedup_b2"] = res["batched_b2"]["samples_per_s"] / res["per_sample_b2"]["samples_per_s"]
    res["peak_gbs"] = PEAK_GBS
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
