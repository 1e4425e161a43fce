"""Validation on the GPU (mvtb.train_stage) at the 127 scripts' shapes.  Prints one JSON line with the card and its power limit
(read in this run):

* validation pass: a DeviceCache of 32 synthetic BraTS-geometry samples (4 x 240 x 240 x 155 image + 3-channel label, LPS
  affine, on the device) filled through SpacingOrientationd((1.5, 1.5, 2.0), "RAS") -> CenterSpatialCropd(128, 128, 64),
  and the 127 validation tail SelectChanneld(image, 0) -> NormalizeIntensityd -> disk 12.5 -> plane wave -> wrap 0.5 ->
  SaltAndPepper(0.05, philox-sparse) over the whole cache: TrainStage.loader(2, shuffle=False) against the same transform
  objects called per sample through the drop-ins (and the pairs stacked into batches).  CUDA events around each pass with
  a synchronise; the cache (0.94 GB) is far over the L2, so a pass reads it from HBM.  Samples/s and library launches
  per sample (mvtb_launch_count);
* cache fill from .nii files: LoadImaged -> AsChannelFirstd -> ConvertToMultiChannelBasedOnBratsClassesd ->
  SpacingOrientationd -> CenterSpatialCropd, with the crop fused into the resampling gather (what DeviceCache does)
  against the same prefix run transform by transform (fill_steps replaced by list), at 1 and 8 threads.  Wall clock of
  DeviceCache(...) (which ends in a synchronise) over 16 items of 8 files in the page cache; the two variants alternate.

Each figure is the median over --repeats windows, with the smallest and largest window beside it.  The files go to a
temporary directory, deleted at exit.  Measurement tool, not product code.
Usage: python tools/bench_val_stage.py [--out FILE]"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPE, PIXDIM, ROI, N_ITEMS, N_FILES, N_FILL = (240, 240, 155), (1.5, 1.5, 2.0), (128, 128, 64), 32, 8, 16
LPS = np.array([[-1.0, 0, 0, 120.0], [0, -1.0, 0, 120.0], [0, 0, 1.0, -77.0], [0, 0, 0, 1]])
KEYS = ["image", "label"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], float(q[1])
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def resample():
    from mvtb import spatial as S
    return S.SpacingOrientationd(KEYS, PIXDIM, axcodes="RAS", mode=("bilinear", "nearest"))


def crop():
    from mvtb import spatial as S
    return S.CenterSpatialCropd(KEYS, list(ROI))


def tail(seed):
    import filters_and_operators as F
    from mvtb import intensity as I
    t = [F.SelectChanneld("image", 0), I.NormalizeIntensityd("image", nonzero=True, channel_wise=True),
         F.RandFourierDiskMaskd("image", r=12.5, inside_off=False, prob=1.0),
         F.RandPlaneWaves_ellipsoid("image", 55, 55, 30, intensity_value=15, prob=1.0), F.WrapArtifactd("image", alpha=0.5),
         F.SaltAndPepper(0.05, "image", prob=1.0, rng="philox-sparse", seed=2024)]
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
    return t


def windows(fn, steps, repeats, warmup, timer):
    """per-call seconds: (median, min, max) over the windows, and library launches per call"""
    from mvtb import _lib
    L = _lib.lib()
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    n0, w = L.mvtb_launch_count(), []
    for _ in range(repeats):
        w.append(timer(fn, steps) / steps)
    return (float(np.median(w)), min(w), max(w)), (L.mvtb_launch_count() - n0) / (steps * repeats)


def events(fn, steps):
    tot = 0.0
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b) / 1e3
    return tot


def validation_pass(dev, steps, repeats):
    from mvtb.train_stage import DeviceCache, TrainStage
    g = torch.Generator(device=dev).manual_seed(5)
    items = []
    for _ in range(N_ITEMS):
        img = torch.randn((4,) + SHAPE, device=dev, generator=g).abs_()
        img *= img > 0.3                                            # zero background
        lab = (torch.rand((3,) + SHAPE, device=dev, generator=g) < 0.2).to(torch.float32)
        items.append({"image": img, "label": lab, "image_meta_dict": {"affine": LPS.copy()}, "label_meta_dict": {"affine": LPS.copy()}})
    cache = DeviceCache(items, [resample(), crop()], num_workers=1)
    del items
    assert [tuple(s) for s in cache.shapes["image"]] == [ROI] * N_ITEMS
    res = {"cache_items": N_ITEMS, "cache_bytes": sum(b.numel() * 4 for b in cache.buffers.values())}
    stage = TrainStage(cache, tail(0))

    def batched():
        for _ in stage.loader(2, shuffle=False):
            pass
    ref = tail(0)

    def per_sample():
        for j in range(0, N_ITEMS, 2):
            outs = []
            for i in (j, j + 1):
                d = cache.item(i)
                for t in ref:
                    d = t(d)
                outs.append(d)
            _ = torch.stack([o["image"] for o in outs]), torch.stack([o["label"] for o in outs])
    for name, fn, n in (("batched_b2", batched, steps), ("per_sample_b2", per_sample, max(steps // 4, 3))):
        (sec, lo, hi), launches = windows(fn, n, repeats, 2, events)
        res[name] = {"samples_per_s": N_ITEMS / sec, "samples_per_s_range": [N_ITEMS / hi, N_ITEMS / lo], "ms_per_pass": sec * 1e3,
                     "launches_per_sample": launches / N_ITEMS}
    res["speedup"] = res["batched_b2"]["samples_per_s"] / res["per_sample_b2"]["samples_per_s"]
    del stage, cache
    torch.cuda.empty_cache()
    return res


def write_files(tmp):
    from oracle import nifti_writer as W, ref_port as P
    img = np.moveaxis(P.synthetic_volume(2, (4,) + SHAPE).numpy(), 0, -1)
    lab = np.zeros(SHAPE, np.uint8)
    lab[60:180, 50:190, 30:120] = np.random.RandomState(3).randint(0, 4, size=(120, 140, 90))
    ip = W.write(os.path.join(tmp, "img0.nii"), img, sform=LPS[:3])
    lp = W.write(os.path.join(tmp, "seg0.nii"), lab, sform=LPS[:3])
    pairs = [(ip, lp)] + [(shutil.copyfile(ip, os.path.join(tmp, f"img{n}.nii")), shutil.copyfile(lp, os.path.join(tmp, f"seg{n}.nii")))
                          for n in range(1, N_FILES)]
    return [{"image": pairs[i % N_FILES][0], "label": pairs[i % N_FILES][1]} for i in range(N_FILL)]


def cache_fill(repeats):
    import filters_and_operators as F
    from mvtb import nifti as N, train_stage as TS
    fused_steps = TS.fill_steps

    def prefix():
        return [N.LoadImaged(KEYS), N.AsChannelFirstd("image"), F.ConvertToMultiChannelBasedOnBratsClassesd("label"), resample(), crop()]

    tmp = tempfile.mkdtemp(prefix="bench_val_stage_")
    try:
        data = write_files(tmp)
        res = {"items": N_FILL, "files": N_FILES, "image_mb": os.path.getsize(data[0]["image"]) / 1e6}
        for threads in (1, 8):
            times = {"fused": [], "unfused": []}
            for r in range(repeats + 1):                            # the first round warms up
                warm = {}
                for name, steps in (("fused", fused_steps), ("unfused", list)):
                    TS.fill_steps = steps
                    t0 = time.perf_counter()
                    cache = TS.DeviceCache(data, prefix(), num_workers=threads)
                    dt = time.perf_counter() - t0
                    if r:
                        times[name].append(dt)
                    else:
                        warm[name] = cache
                    del cache
                if warm and threads == 1:                           # the two fills hold the same bits
                    res["fused_equals_unfused"] = all(torch.equal(warm["fused"].buffers[k], warm["unfused"].buffers[k]) for k in KEYS)
                del warm
            for name, w in times.items():
                med = float(np.median(w))
                res[f"{name}_{threads}t"] = {"samples_per_s": N_FILL / med, "samples_per_s_range": [N_FILL / max(w), N_FILL / min(w)],
                                             "s_per_fill": med}
            res[f"speedup_{threads}t"] = res[f"fused_{threads}t"]["samples_per_s"] / res[f"unfused_{threads}t"]["samples_per_s"]
    finally:
        TS.fill_steps = fused_steps
        shutil.rmtree(tmp, ignore_errors=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40, help="validation passes per timed window (per-sample path: a quarter)")
    ap.add_argument("--repeats", type=int, default=5, help="timed windows")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_val_stage needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plim = card()
    res = {"metric": "validation samples/s (127 validation tail on 128x128x64 centre crops of BraTS-geometry samples) and "
                     "cache fill samples/s with the fused centre crop", "card": name, "power_limit_w": plim,
           "host_threads": os.cpu_count(), "geometry": {"image": [4, *SHAPE], "label": [3, *SHAPE], "pixdim": PIXDIM, "roi": ROI}}
    with torch.no_grad():
        res["validation_pass"] = validation_pass(dev, args.steps, args.repeats)
        res["cache_fill"] = cache_fill(args.repeats)
    res["steps_per_window"], res["windows"] = args.steps, args.repeats
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
