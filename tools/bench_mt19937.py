"""torch's CPU generator on the device (csrc/mt19937.cuh) against torch.rand on the host.  Prints one JSON line with the
card and its power limit (read in this run) and:
  device_*          mvtb_mt19937_uniform_f32 alone (states already on the device): uniforms/s and microseconds per call,
                    at the geometry mvtb.functional picks and at each chunk length of a sweep;
  host_rand_*       torch.rand(shape) per segment on the host plus the copy of u to the device (the parent path);
  torch_uniform_*   mvtb.functional.torch_uniform end to end: host jump per segment, state upload, device generator;
  host_jump_us      mt19937_advance for one sample's draws (jump polynomial cached, as a stage uses it);
  train_stage_*     TrainStage.apply(draw(...)) at batch 2 and 64 with SaltAndPepper(rng="torch", torch_generator=True)
                    beside rng="philox-sparse", and the same tail per sample through the drop-ins with host torch.rand
                    uniforms injected (what a seeded rng="torch" run cost before).
CUDA events around each timed call with a synchronise; medians over --repeats windows.  Measurement tool, not product code.
Usage: python tools/bench_mt19937.py [--out FILE]"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "medical-vision-textural-bias_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench_train_stage as BT  # noqa: E402

SIZES = {"2x1x128x128x64": (2, (1, 128, 128, 64)), "1x240x240x155": (1, (1, 240, 240, 155)),
         "1x4x240x240x155": (1, (4, 240, 240, 155))}


def events(fn, steps, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    win = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        win.append(a.elapsed_time(b) / 1e3 / steps)
    return float(np.median(win)), min(win), max(win)


def wall(fn, steps, repeats, warmup=2):
    """host clock around calls that end in a device synchronise"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    win = []
    for _ in range(repeats):
        t = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        win.append((time.perf_counter() - t) / steps)
    return float(np.median(win)), min(win), max(win)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mt19937 needs a CUDA device")
    from mvtb import _lib, functional as Fn
    L = _lib.lib()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plim = BT.card()
    res = {"metric": "torch.rand stream (MT19937) on the device vs the host", "card": name, "power_limit_w": plim}
    torch.manual_seed(0)
    for key, (S, shape) in SIZES.items():
        n = math.prod(shape)
        states = torch.from_numpy(Fn.mt19937_take(n, S)).to(dev)
        u = torch.empty((S, n), device=dev)
        chunk, nch = Fn._mt_geometry(n, S)
        ws = torch.empty(int(L.mvtb_mt19937_workspace_bytes(S)), dtype=torch.uint8, device=dev)
        stream = Fn._stream(dev)

        def run(chunk=chunk, nch=nch):
            table = Fn._mt_table(dev, chunk, nch)
            _lib.check(L, L.mvtb_mt19937_uniform_f32(Fn._ptr(u), n, S, Fn._ptr(states), Fn._ptr(table), C.c_uint64(chunk), nch,
                                                     Fn._ptr(ws), stream))
        sec, lo, hi = events(run, args.steps, args.repeats)
        res[f"device_{key}"] = {"uniforms": S * n, "chunk_len": chunk, "us_per_call": sec * 1e6, "us_range": [lo * 1e6, hi * 1e6],
                                "uniforms_per_s": S * n / sec, "us_per_segment": sec * 1e6 / S}
        sweep = {}
        for c in (4096, 8192, 16384, 32768, 65536, 131072, 262144, 524288, 1 << 20):
            if S * -(-n // c) > 4 * 148 or c > 4 * n:
                continue
            sweep[c] = events(lambda c=c: run(c, 128), max(args.steps // 5, 3), 3)[0] * 1e6
        res[f"device_{key}"]["us_by_chunk_len"] = sweep
        sec, lo, hi = wall(lambda: [torch.rand(shape).to(dev) for _ in range(S)], max(args.steps // 10, 2), 3)
        res[f"host_rand_{key}"] = {"us_per_call": sec * 1e6, "us_range": [lo * 1e6, hi * 1e6], "uniforms_per_s": S * n / sec}
        sec, lo, hi = wall(lambda: Fn.torch_uniform(shape, S, dev), max(args.steps // 5, 3), 3)
        res[f"torch_uniform_{key}"] = {"us_per_call": sec * 1e6, "us_range": [lo * 1e6, hi * 1e6], "uniforms_per_s": S * n / sec}
        words, nx, lf = Fn.mt19937_unpack(torch.get_rng_state())
        Fn.mt19937_advance(words, nx, lf, n)
        t = time.perf_counter()
        for _ in range(20):
            words, nx, lf = Fn.mt19937_advance(words, nx, lf, n)
        res[f"host_jump_us_{key}"] = (time.perf_counter() - t) / 20 * 1e6

    # the training stage: a smaller cache than bench_train_stage's (the host path is slow), same tail
    from mvtb.train_stage import DeviceCache, TrainStage
    import filters_and_operators as F
    g = torch.Generator(device=dev).manual_seed(5)
    items = []
    for _ in range(16):
        img = torch.randn((4,) + BT.GRID, device=dev, generator=g).abs_()
        img *= img > 0.3
        items.append({"image": img, "label": (torch.rand((3,) + BT.GRID, device=dev, generator=g) < 0.2).to(torch.float32)})
    cache = DeviceCache(items, [], num_workers=1)
    del items
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    rng = np.random.RandomState(1)

    def tail(kind):
        t = BT.tail(0)
        t[-1] = F.SaltAndPepper(0.05, "image", prob=1.0, rng=kind, seed=2024)
        return t
    with torch.no_grad():
        for kind in ("torch", "philox-sparse"):
            for bs in (2, 64):
                stage = TrainStage(cache, tail(kind), torch_generator=kind == "torch")
                (sec, lo, hi), launches = BT.timed(lambda: stage.apply(stage.draw(rng.randint(0, 16, bs))),
                                                   max(args.steps // (1 if bs == 2 else 5), 3), args.repeats, 2, flush)
                res[f"train_stage_{kind}_b{bs}"] = {"samples_per_s": bs / sec, "samples_per_s_range": [bs / hi, bs / lo],
                                                    "ms_per_batch": sec * 1e3, "launches_per_batch": launches}

        class HostRand(F.SaltAndPepper):
            def salt_and_pepper(self, x, u=None):
                return super().salt_and_pepper(x, u=torch.rand(x.size()))
        ref = BT.tail(0)
        ref[-1] = HostRand(0.05, "image", prob=1.0, rng="torch")

        def per_sample():
            for i in rng.randint(0, 16, 2):
                d = cache.item(int(i))
                for t in ref:
                    d = t(d)
        (sec, lo, hi), launches = BT.timed(per_sample, max(args.steps // 5, 3), args.repeats, 2, flush)
        res["per_sample_host_rand_b2"] = {"samples_per_s": 2 / sec, "samples_per_s_range": [2 / hi, 2 / lo], "ms_per_batch": sec * 1e3}
    res["speedup_torch_b2_vs_per_sample_host_rand"] = res["train_stage_torch_b2"]["samples_per_s"] / res["per_sample_host_rand_b2"]["samples_per_s"]
    res["steps"], res["repeats"] = args.steps, args.repeats
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
