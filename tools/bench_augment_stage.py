"""The k-space augmentation scripts' training tails through TrainStage(kspace_augment=True) at the scripts' 128 x 128 x 64 crop.
Prints one JSON line with the card and its power limit (read in this run).

A DeviceCache of 32 synthetic BraTS-geometry samples (4 x 240 x 240 x 155 image + 3-channel label, LPS affine, on the
device) resampled by SpacingOrientationd((1.5, 1.5, 2.0), "RAS") to 160 x 160 x 78, then per tail one shuffled epoch of
loader(batch_size=2) against the same transform objects called per sample through the drop-ins (and the pairs stacked
into batches).  Every tail is RandSpatialCropd(128, 128, 64) -> RandFlipd -> NormalizeIntensityd -> RandScaleIntensityd
-> RandShiftIntensityd -> the augmentation:

* gibbs_p0.1:  SelectChanneld(image, 0), RandGibbsNoised(prob=0.1, alpha=(0, 0.3))        (30_augmentation, ALPHA = .3)
* gibbs_p1_4ch: RandGibbsNoised(prob=1.0) on the 4-channel image                            (20_Gibbs_filters)
* spikes:      SelectChanneld(image, 0), RandKSpaceSpikeNoised(0.1, 1.0, {image: (10, 11)}) (30_augmentation spikes)

CUDA events around each epoch with a synchronise.  Samples/s are the median over --repeats windows with the smallest and
largest window beside it; launches are the library's (mvtb_launch_count) per sample: torch's own copies (the stage's
index_select / index_copy_ of the gated samples, the per-sample path's stacking) are not in that count.
Measurement tool, not product code.  Usage: python tools/bench_augment_stage.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPE, PIXDIM, ROI, N_ITEMS = (240, 240, 155), (1.5, 1.5, 2.0), (128, 128, 64), 32
LPS = np.array([[-1.0, 0, 0, 120.0], [0, -1.0, 0, 120.0], [0, 0, 1.0, -77.0], [0, 0, 0, 1]])
KEYS = ["image", "label"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], float(q[1])
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def tail(name, seed):
    import filters_and_operators as F
    from mvtb import intensity as I, spatial as S
    t = [S.RandSpatialCropd(KEYS, roi_size=list(ROI), random_size=False), S.RandFlipd(KEYS, prob=0.5, spatial_axis=0)]
    if name != "gibbs_p1_4ch":
        t.append(F.SelectChanneld("image", 0))
    t += [I.NormalizeIntensityd("image", nonzero=True, channel_wise=True), I.RandScaleIntensityd("image", factors=0.1, prob=0.5),
          I.RandShiftIntensityd("image", offsets=0.1, prob=0.5)]
    if name == "gibbs_p0.1":
        t.append(F.RandGibbsNoised("image", 0.1, alpha=(0.0, 0.3)))
    elif name == "gibbs_p1_4ch":
        t.append(F.RandGibbsNoised("image", 1.0))
    else:
        t.append(F.RandKSpaceSpikeNoised("image", 0.1, 1.0, intensity_ranges={"image": (10, 11)}))
    for k, x in enumerate(t):
        if hasattr(x, "set_random_state"):
            x.set_random_state(seed=seed * 1000 + k)
        for inner in getattr(x, "transforms", {}).values():
            inner.set_random_state(seed=seed * 1000 + k + 500)
    return t


def windows(fn, repeats, warmup):
    """per-epoch seconds over the windows (CUDA events, one epoch each) and library launches per epoch"""
    from mvtb import _lib
    L = _lib.lib()
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    n0, w = L.mvtb_launch_count(), []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        w.append(a.elapsed_time(b) / 1e3)
    return w, (L.mvtb_launch_count() - n0) / repeats


def main():
    from mvtb import spatial as S
    from mvtb.train_stage import DeviceCache, TrainStage
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5, help="timed epochs per arm")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_augment_stage needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plim = card()
    res = {"metric": "training samples/s of the k-space augmentation tails, TrainStage.loader(2) against per-sample drop-ins",
           "card": name, "power_limit_w": plim, "geometry": {"image": [4, *SHAPE], "label": [3, *SHAPE], "pixdim": PIXDIM,
                                                              "roi": ROI}, "cache_items": N_ITEMS, "windows": args.repeats}
    with torch.no_grad():
        g = torch.Generator(device=dev).manual_seed(5)
        items = []
        for _ in range(N_ITEMS):
            img = torch.randn((4,) + SHAPE, device=dev, generator=g).abs_()
            img *= img > 0.3                                            # zero background
            lab = (torch.rand((3,) + SHAPE, device=dev, generator=g) < 0.2).to(torch.float32)
            items.append({"image": img, "label": lab, "image_meta_dict": {"affine": LPS.copy()},
                          "label_meta_dict": {"affine": LPS.copy()}})
        cache = DeviceCache(items, [S.SpacingOrientationd(KEYS, PIXDIM, axcodes="RAS", mode=("bilinear", "nearest"))], num_workers=1)
        del items
        torch.cuda.empty_cache()
        res["cached_shape"] = [int(s) for s in cache.shapes["image"][0]]
        for tname in ("gibbs_p0.1", "gibbs_p1_4ch", "spikes"):
            stage = TrainStage(cache, tail(tname, 0), kspace_augment=True)
            ref = tail(tname, 0)
            gen = torch.Generator().manual_seed(0)
            gated = []

            def batched():
                for _ in stage.loader(2, generator=gen):
                    pass

            def per_sample():
                order = torch.randperm(N_ITEMS, generator=gen).tolist()
                for j in range(0, N_ITEMS, 2):
                    outs = []
                    for i in order[j:j + 2]:
                        d = cache.item(i)
                        for t in ref:
                            d = t(d)
                        outs.append(d)
                    _ = torch.stack([o["image"] for o in outs]), torch.stack([o["label"] for o in outs])
            rec = stage.draw(range(N_ITEMS))                        # the share of gated samples these settings give
            for b in range(N_ITEMS):
                gated.append(stage._sample_descs(rec, b, ROI, 4 if tname == "gibbs_p1_4ch" else 1)[1])
            row = {"gated_fraction_of_32_draws": float(np.mean(gated))}
            for arm, fn in (("batched_b2", batched), ("per_sample_b2", per_sample)):
                w, launches = windows(fn, args.repeats, 2)
                sec = float(np.median(w))
                row[arm] = {"samples_per_s": N_ITEMS / sec, "samples_per_s_range": [N_ITEMS / max(w), N_ITEMS / min(w)],
                            "ms_per_epoch": sec * 1e3, "launches_per_sample": launches / N_ITEMS}
            row["speedup"] = row["batched_b2"]["samples_per_s"] / row["per_sample_b2"]["samples_per_s"]
            res[tname] = row
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
