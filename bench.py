#!/usr/bin/env python
"""bench.py — throughput of the MRI artifact chain on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg3|cfg1]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic volumes (SURVEY.md 8(d)):
  cfg2 (default, the configuration BASELINE.json's metric is quoted on): the 127-series chain
       Gibbs disk r=12.5 -> plane-wave spike I=15 on the (55,55,30) shell -> wraparound 0.5 ->
       salt-and-pepper 0.05 on 64 x (1x240x240x155) fp32 volumes per GPU;
  cfg3: Gibbs disk r=12.5 -> salt-and-pepper 0.15 on (4x240x240x155) samples;
  cfg1: Gibbs disk r=12.5 on 1x240x240x155 volumes (the reference's own CPU-runnable case).
Prints ONE JSON line (rank 0).  `value` = volumes/s with inputs resident in HBM; `e2e` = the same
metric through the public API with HOST buffers (pinned H2D of the inputs and D2H of the outputs
inside the timed region); `roofline` = dominant kernel against the measured HBM peak;
`cpu_baseline` = the oracle port of the reference timed on this box's host cores.
With --impl reference only the CPU reference arm runs (rank 0), on the same config and metric.
--dump-outputs DIR writes what the last timed step returned on rank 0 as DIR/out.npy (see output_sample), so that
two builds can be compared output for output: the inputs, spike locations and S&P seeds are fixed, so the same
arguments give the same inputs on every run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "medical-vision-textural-bias_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPE = (240, 240, 155)
# in-kernel S&P sampler: the geometric-gap sampler (default; voxels hit are i.i.d. Bernoulli(p) with a fair
# salt/pepper coin, exactly the reference's distribution, at a cost ~ p: 6.7 us/vol) or one Philox uniform per
# voxel (MVTB_SPARSE_SP=0; bound by Philox's 32x32->64 multiplies: 7.9 us/vol)
SPARSE_SP = os.environ.get("MVTB_SPARSE_SP", "1") == "1"
# chain and select pass as ONE library call: on the band-limited path the select runs inside the persistent inverse
# kernel, on output lines still in L2 (MVTB_TWO_CALLS=1: the round-1 sequence of two calls, same result bit for bit)
FUSED_SP = os.environ.get("MVTB_TWO_CALLS", "0") != "1"
BYTES_PER_VOXEL = 8            # algorithmic: read fp32 once + write fp32 once (SURVEY 8(d))
FALLBACK_HBM_GBS = 6650.0      # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent

WORKLOADS = {
    "cfg2": dict(name="chain-127: Gibbs disk r=12.5 + k-space spike I=15 on (55,55,30) shell + wraparound 0.5 + salt-and-pepper 0.05",
                 channels=1, batch=64, r=12.5, spike=True, alpha=0.5, p=0.05),
    "cfg3": dict(name="Gibbs disk r=12.5 + salt-and-pepper 0.15 on 4-channel samples",
                 channels=4, batch=16, r=12.5, spike=False, alpha=None, p=0.15),
    "cfg1": dict(name="Gibbs disk r=12.5 (RandFourierDiskMaskd)", channels=1, batch=64, r=12.5, spike=False, alpha=None, p=None),
    # BASELINE.json configs[2] as written: 256 samples in total, sharded 256/128/64/32 per GPU at 1/2/4/8 GPUs (strong scaling)
    "cfg3s": dict(name="Gibbs disk r=12.5 + salt-and-pepper 0.15 on 4-channel samples, 256 samples in total (strong scaling)",
                  channels=4, batch=256, strong_total=256, r=12.5, spike=False, alpha=None, p=0.15),
}
# configs[3] and configs[4] of BASELINE.json have other units of work (2-D slices; 128x128x64 crops): bench.py --workload cfg4|cfg5
AUX_WORKLOADS = ("cfg4", "cfg5", "train127")
DUMP_BYTES = 32 << 20          # --dump-outputs: largest array written whole; larger outputs are sampled down to it


def output_sample(y, budget=DUMP_BYTES):
    """y as a float32 (float64 if it is one) host array: whole if it fits in `budget` bytes, else at most the k elements
    that fit, taken from y.reshape(-1) at increasing positions whose gaps numpy.random.default_rng(0) draws uniformly
    from [1, 2 n / k) (n elements): the same positions for the same output shape on every run."""
    y = torch.as_tensor(y).detach()
    if y.dtype != torch.float64:
        y = y.to(torch.float32)
    n, k = y.numel(), budget // y.element_size()
    if n <= k:
        return y.cpu().numpy()
    idx = np.cumsum(np.random.default_rng(0).integers(1, 2 * (n // k), size=k)) - 1
    idx = idx[idx < n]
    return y.reshape(-1)[torch.from_numpy(idx).to(y.device)].cpu().numpy()


def write_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def shard_range(total, rank, world):
    """Contiguous slice of `total` units owned by `rank` (SURVEY 8(e))."""
    base, extra = divmod(total, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def aggregate(stats, world):
    """(max over ranks, sum over ranks) of a per-rank statistics vector: the only collective on the path.
    NCCL on the GPUs (a few dozen bytes over NVLink), gloo in the CPU tests."""
    if world <= 1:
        return stats.clone(), stats.clone()
    import torch.distributed as dist
    mx, sm = stats.clone(), stats.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    return mx, sm


def spike_indices(first_sample, n):
    """Per-sample spike location: RandomState(sample_index).randint over the cached (55,55,30) shell."""
    from mvtb import host
    shell = host.ellipsoid_shell(SHAPE, 55., 55., 30.)
    return [tuple(int(v) for v in shell[np.random.RandomState(first_sample + i).randint(0, len(shell))]) for i in range(n)]


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Median SM clock and active throttle reasons over the samples taken in [t0, t1] (the timed region)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 is None or (t0 - 0.05 <= t <= t1 + 0.05)]
        if not rows:
            rows = [r for (_, r) in self.rows]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU reference arm
def reference_modules():
    """The UNMODIFIED reference (oracle/_ref, placed by oracle/build_ref.py, imported through oracle/monai_shim), or None."""
    try:
        from oracle import build_ref
        return build_ref.import_reference()
    except Exception:  # noqa: BLE001
        return None


def cpu_reference_step(cfg, sample_index, n_volumes, mods=None):
    """The reference's CPU path on n_volumes samples; yields the transform time of each.  With `mods` the reference's
    own classes run (kind "reference"); without, oracle/ref_port.py (kind "port": the same torch op sequence)."""
    from oracle import ref_port as P
    C = cfg["channels"]
    idxs = spike_indices(sample_index, n_volumes) if cfg["spike"] else [None] * n_volumes
    chain = None
    if mods is not None:
        RF = mods[0]
        chain = [RF.RandFourierDiskMaskd(keys='image', r=cfg["r"], inside_off=False, prob=1.)]
        if cfg["spike"]:
            chain.append(RF.RandPlaneWaves_ellipsoid('image', 55., 55., 30., intensity_value=15., prob=1.))
        if cfg["alpha"] is not None:
            chain.append(RF.WrapArtifactd("image", cfg["alpha"]))
        if cfg["p"] is not None:
            chain.append(RF.SaltAndPepper(cfg["p"]))
    for i in range(n_volumes):
        x = P.synthetic_volume(sample_index + i, (C,) + SHAPE)
        t0 = time.perf_counter()
        if chain is not None:
            d = {"image": x}
            for tr in chain:
                d = tr(d)
        else:
            y = P.fourier_disk_mask(x, cfg["r"], False)
            if cfg["spike"]:
                y = P.plane_wave_spike(y, idxs[i], 15.0)
            if cfg["alpha"] is not None:
                y = P.wrap_artifact(y, cfg["alpha"])
            if cfg["p"] is not None:
                y = P.salt_and_pepper(y, cfg["p"], torch.rand(y.size()))      # the reference draws u itself (F:472)
        yield time.perf_counter() - t0


def time_cpu_reference(cfg, n_volumes, warm=1):
    """(volumes/s on all host threads, threads, per-volume times, volumes/s on ONE thread, kind)."""
    mods = reference_modules()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    list(cpu_reference_step(cfg, 10_000, warm, mods))
    ts = list(cpu_reference_step(cfg, 0, n_volumes, mods))
    torch.set_num_threads(1)
    t1 = list(cpu_reference_step(cfg, 0, 1, mods))
    torch.set_num_threads(cores)
    return n_volumes / sum(ts), cores, ts, 1.0 / sum(t1), ("reference" if mods is not None else "port")


def run_reference_arm(args, cfg, rank):
    if rank != 0:
        return
    mods = reference_modules()
    kind = "reference" if mods is not None else "port"
    n_per_step = 1 if cfg["channels"] > 1 else 2
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    list(cpu_reference_step(cfg, 10_000, 1, mods))
    for _ in range(args.warmup):
        list(cpu_reference_step(cfg, 20_000, n_per_step, mods))
    dt = 0.0                               # transform time only; generating the synthetic input is not timed
    for s in range(args.steps):
        dt += sum(cpu_reference_step(cfg, s * n_per_step, n_per_step, mods))
    value = args.steps * n_per_step / dt
    torch.set_num_threads(1)
    one = 1.0 / sum(cpu_reference_step(cfg, 0, 1, mods))
    torch.set_num_threads(cores)
    sample = f"{n_per_step} sample(s) of {cfg['channels']}x240x240x155 per step, {args.steps} steps, torch {torch.__version__} CPU, {cores} threads"
    what = ("the UNMODIFIED reference classes (oracle/_ref = source_code/filters_and_operators.py, through oracle/monai_shim)" if mods is not None else
            "oracle/ref_port.py, the bit-identical restatement of filters_and_operators.py (oracle/_ref is absent on this box)")
    line = {
        "impl": "reference", "metric": "volumes/sec (240x240x155 fp32)", "value": value, "unit": "volumes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {cfg['name']}", "volume": "%dx240x240x155" % cfg["channels"],
                   "volumes_per_step": n_per_step, "note": "reference CPU path = " + what},
        "cpu_baseline": {"value": value, "unit": "volumes/s", "cores": cores, "kind": kind, "sample": sample,
                         "value_1_thread": one, "torch_config": torch.__config__.parallel_info().split("\n")[0:3]},
        "e2e": {"value": value, "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def make_inputs(cfg, first_sample, dev):
    """Synthetic BraTS-shaped batch generated on the device from per-sample seeds (SURVEY 8(d))."""
    B, C = cfg["batch"], cfg["channels"]
    grids = torch.meshgrid([torch.linspace(-1, 1, n, device=dev) for n in SHAPE], indexing="ij")
    support = (sum((g / 0.9) ** 2 for g in grids) < 1).to(torch.float32)
    x = torch.empty((B, C) + SHAPE, dtype=torch.float32, device=dev)
    for b in range(B):
        g = torch.Generator(device=dev).manual_seed(1234 + first_sample + b)
        x[b] = torch.randn((C,) + SHAPE, generator=g, dtype=torch.float32, device=dev) * support
    return x


_DESC_CACHE = {}


def gpu_step(cfg, x, idxs, out, step, group_offset=None):
    """One pass of the workload over the batch x (B, C, H, W, D) on the current stream.  The S&P uniforms of
    voxel group g of the whole batch come from Philox counter step * (groups per batch) + g; a slice of the
    batch passes its own group_offset so that slicing does not change the result."""
    from mvtb import functional as Fn, host, _lib
    B, C = x.shape[0], x.shape[1]
    # the per-sample descriptors depend only on the configuration and the spike locations: built once, reused every step
    # (64 make_desc calls cost the host ~0.5 ms, a third of the step's GPU time)
    key = (cfg["r"], cfg["spike"], cfg["alpha"], B, C, None if idxs is None else tuple(idxs))
    descs = _DESC_CACHE.get(key)
    if descs is None:
        thr = host.disk_threshold(cfg["r"], SHAPE)
        amp = host.exp_f32(15.0)
        descs = []
        for b in range(B):
            sp = [(idxs[b], amp)] if cfg["spike"] else []
            d = host.make_desc(mask_kind=_lib.MASK_DISK, mask_ndim=3, mask_thresh=thr, spikes=sp, wrap_alpha=cfg["alpha"])
            descs.extend([d] * C)
        if len(_DESC_CACHE) > 64:
            _DESC_CACHE.clear()
        _DESC_CACHE[key] = descs
    if cfg["p"] is None:
        return Fn.kspace_chain(x, 3, descs, out=out)
    if SPARSE_SP:                                   # geometric-gap Bernoulli sampler: counters count 256-voxel blocks
        nb = B * ((x.numel() // B + 255) // 256)
        off = step * nb if group_offset is None else group_offset // 64
        if FUSED_SP:                                # chain + select as one library call (mvtb_kspace_chain_sp_f32)
            return Fn.kspace_chain_sp(x, 3, descs, cfg["p"], seed=2024, offset=off, vols_per_sample=C, out=out)[0]
        y, mm = Fn.kspace_chain(x, 3, descs, want_minmax=True, vols_per_sample=C, out=out)
        return Fn.salt_pepper(y, cfg["p"], seed=2024, offset=off, n_samples=B, mm=mm, out=y, sparse=True)
    y, mm = Fn.kspace_chain(x, 3, descs, want_minmax=True, vols_per_sample=C, out=out)
    n4 = (x.numel() + 3) // 4
    off = step * n4 if group_offset is None else group_offset
    return Fn.salt_pepper(y, cfg["p"], seed=2024, offset=off, n_samples=B, mm=mm, out=y)


def run_aux_workload(args):
    """BASELINE.json configs[3] (2-D k-space spike on a stack of 8192 slices of 240 x 240) and configs[4] (chain-127 +
    GibbsNoiseLayer on (B,1,128,128,64) crops) through the drop-in classes; every rank runs its own copy (weak scaling)."""
    import torch.distributed as dist
    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the mvtb hot path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import filters_and_operators as F
    import stylization_layers as S
    from mvtb import _lib, functional as Fn
    L = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(4321 + rank)
    if args.workload == "cfg4":
        x = torch.randn(8192, 240, 240, device=dev, generator=g)
        t4 = F.KSpaceSpikeNoise((120 + 31, 120 - 17), 15.0)
        step = lambda: t4(x)                                              # noqa: E731
        units, unit, voxels, metric = 8192, "slices/s", x.numel(), "slices/sec (240x240 fp32)"
        name = "cfg4: KSpaceSpikeNoise 2-D, one location for (8192,240,240) (F:982-983)"
    elif args.workload == "train127":
        # The 127 scripts' per-sample training transform from the resampled volume on (127_...FLAIR.py:130-141), at the
        # scripts' own shapes: (1, 160, 160, 78) after Spacingd(1.5, 1.5, 2.0) -> RandSpatialCropd(128,128,64) -> RandFlipd ->
        # NormalizeIntensityd / RandScale / RandShift (one statistics pass; the map rides on the chain's forward kernel)
        # -> disk 12.5 -> plane-wave spike -> wrap 0.5 -> S&P 0.05, for a batch of 64 samples
        import ctypes as C
        from mvtb import host
        B = 64
        src = torch.randn(B, 1, 160, 160, 78, device=dev, generator=g).abs_()
        src *= (src > 0.3)                                                # zero background
        R = np.random.RandomState(99 + rank)
        starts = [(int(R.randint(0, 33)), int(R.randint(0, 33)), int(R.randint(0, 15))) for _ in range(B)]
        flips = [int(R.rand() < 0.5) for _ in range(B)]
        scales = torch.tensor([1.0 + R.uniform(-0.1, 0.1) for _ in range(B)], dtype=torch.float32)
        shifts = torch.tensor([R.uniform(-0.1, 0.1) for _ in range(B)], dtype=torch.float32)
        shell = host.ellipsoid_shell((128, 128, 64), 55., 55., 30.)
        idxs = [tuple(int(v) for v in shell[R.randint(0, len(shell))]) for _ in range(B)]
        thr = host.disk_threshold(12.5, (128, 128, 64))
        descs = host.desc_array([host.make_desc(mask_kind=_lib.MASK_DISK, mask_ndim=3, mask_thresh=thr, spikes=[(i, host.exp_f32(15.0))], wrap_alpha=0.5)
                                 for i in idxs])
        xc = torch.empty(B, 1, 128, 128, 64, device=dev)
        yo = torch.empty_like(xc)
        i3 = C.c_int32 * 3
        stream = Fn._stream(dev)

        st_dev = torch.tensor(starts, dtype=torch.int32, device=dev)
        fl_dev = torch.tensor(flips, dtype=torch.int32, device=dev)

        def step():
            # crop + flip: one gather for the batch (the windows and flips were drawn on the host, as the loader does)
            _lib.check(L, L.mvtb_crop_flip_batch_f32(Fn._ptr(src), Fn._ptr(xc), B, 1, i3(160, 160, 78), i3(128, 128, 64), Fn._ptr(st_dev),
                                                     Fn._ptr(fl_dev), stream))
            abt = Fn.intensity_coeffs(xc, B, scale=scales, shift=shifts)  # one read of the crops
            return Fn.kspace_chain_ex(xc, 3, descs, pre_abt=abt, sp=(0.05, 7, 0), out=yo)[0]

        units, unit, voxels, metric = B, "volumes/s", xc.numel() * 20 / 8, "volumes/sec (train transform, 128x128x64 fp32)"
        name = ("train127: crop + flip (8 B/voxel) -> intensity statistics (4) -> chain-127 with the intensity map applied on load and the "
                "select pass (8) on (64,1,128,128,64) crops of (64,1,160,160,78) volumes = 20 B/voxel")
    else:
        B = 32
        x = torch.randn(B, 1, 128, 128, 64, device=dev, generator=g)
        idxs = [(64 + (b % 5), 64 - (b % 7), 32 + (b % 3)) for b in range(B)]
        layer = S.GibbsNoiseLayer(0.7)
        step = lambda: layer(Fn.chain127(x, r=12.5, spike_idx=idxs, intensity=15.0, alpha=0.5, p=0.05, seed=7, sparse=True))   # noqa: E731
        units, unit, voxels, metric = B, "volumes/s", 2 * x.numel(), "volumes/sec (128x128x64 fp32)"
        name = "cfg5: chain-127 then GibbsNoiseLayer(0.7) on (32,1,128,128,64); two transforms = 16 B/voxel"
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)              # > L2, written between steps
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step()
        torch.cuda.synchronize(dev)
        n0 = L.mvtb_launch_count()
        tot = 0.0
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            y = step()
            b.record()
            torch.cuda.synchronize(dev)
            tot += a.elapsed_time(b)
        launches = int(L.mvtb_launch_count() - n0)
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"out": output_sample(y)})
    stats = torch.tensor([tot, float(units)], dtype=torch.float64, device=dev)
    mx, sm = aggregate(stats, world)
    if rank == 0:
        ms = float(mx[0]) / args.steps
        peak, peak_src = peak_hbm()
        gbs = BYTES_PER_VOXEL * voxels / 2 ** 0 / (ms * 1e-3) / 1e9 if args.workload == "cfg4" else 8.0 * voxels / (ms * 1e-3) / 1e9
        print(json.dumps({"metric": metric, "value": float(sm[1]) / (ms * 1e-3), "unit": unit, "n_gpus": world, "steps": args.steps,
                          "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32", "data": "synthetic", "config": {"workload": name, "l2": "flushed between steps (256 MB written)"},
                          "roofline_whole_step": {"achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": peak_src,
                                                  "note": "20 B per output voxel (see config.workload)" if args.workload == "train127" else "8 B/voxel per transform"},
                          "gpu_launches": launches}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + list(AUX_WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: the workload's)")
    ap.add_argument("--cpu-volumes", type=int, default=6, help="bounded CPU-baseline sample (volumes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (kernel sweeps)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle spot check printed in the JSON line")
    ap.add_argument("--disk-r", type=float, default=None, help="override the disk radius (sweeps; the headline uses the workload's 12.5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (rank 0) to DIR/out.npy, sampled down to %d MB if larger"
                         % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.workload in AUX_WORKLOADS:
        return run_aux_workload(args)
    cfg = dict(WORKLOADS[args.workload])
    if args.batch:
        cfg["batch"] = args.batch
    if args.disk_r is not None:
        cfg["r"] = args.disk_r
        cfg["name"] += " [disk radius overridden: r=%g]" % args.disk_r
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    import torch.distributed as dist
    from mvtb import _lib, functional as Fn

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the mvtb hot path has no CPU fallback (use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    strong = "strong_total" in cfg and not args.batch
    if strong:                                         # strong scaling: the fixed total is split over the ranks
        lo_s, hi_s = shard_range(cfg["strong_total"], rank, world)
        cfg["batch"] = hi_s - lo_s
    B, C = cfg["batch"], cfg["channels"]
    first = lo_s if strong else rank * B               # weak scaling: every rank owns its own B samples; seeds from the global index
    x = make_inputs(cfg, first, dev)
    out = torch.empty_like(x)
    idxs = spike_indices(first, B) if cfg["spike"] else None
    vols_per_step = B * C
    voxels = vols_per_step * SHAPE[0] * SHAPE[1] * SHAPE[2]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing
    sampler = ClockSampler(local_rank)
    sampler.start()
    for s in range(max(args.warmup, 3)):
        gpu_step(cfg, x, idxs, out, s)
    barrier()
    launches0 = L.mvtb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    th0 = time.perf_counter()
    e0.record()
    for s in range(args.steps):
        y = gpu_step(cfg, x, idxs, out, 100 + s)
    e1.record()
    barrier()
    th1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    launches = int(L.mvtb_launch_count() - launches0)
    clocks = sampler.stop(th0, th1)
    checksum = float(out.double().sum())
    # taken before the profiling and parity passes below reuse `out`
    dumped = {"out": output_sample(y)} if args.dump_outputs and rank == 0 else None

    # ---- per-kernel device time (cudaEvents around every launch, on the launching stream)
    plan = Fn.get_plan(SHAPE, vols_per_step, dev)
    _lib.check(L, L.mvtb_plan_profile(plan, 1))
    prof_steps = min(args.steps, 3)
    sp_ms = []
    for s in range(prof_steps):
        gpu_step(cfg, x, idxs, out, 200 + s)
    torch.cuda.synchronize(dev)
    import ctypes as Ct
    ms_sum = (Ct.c_double * _lib.K_KINDS)()
    cnts = (Ct.c_int * _lib.K_KINDS)()
    _lib.check(L, L.mvtb_plan_profile_read(plan, ms_sum, cnts))
    _lib.check(L, L.mvtb_plan_profile(plan, 0))
    kernels = {}
    for k in range(_lib.K_KINDS):
        if cnts[k]:
            kernels[L.mvtb_kernel_name(k).decode()] = {"launches_per_step": cnts[k] / prof_steps, "ms_per_step": ms_sum[k] / prof_steps,
                                                       "avg_launch_ms": ms_sum[k] / cnts[k]}
    if cfg["p"] is not None and not (FUSED_SP and SPARSE_SP):   # a separate select pass is launched from Python: time it the same way
        from mvtb import functional as Fn2
        mm = Fn2.minmax(out, B)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for s in range(3):
            Fn2.salt_pepper(out, cfg["p"], seed=1, offset=0, n_samples=B, mm=mm, out=out, sparse=SPARSE_SP)
        b.record()
        torch.cuda.synchronize(dev)
        kernels["k_salt_pepper<philox>"] = {"launches_per_step": 1, "ms_per_step": a.elapsed_time(b) / 3, "avg_launch_ms": a.elapsed_time(b) / 3}
    # roofline kernel = the most expensive kernel of the step.  Bytes it must move per voxel (DESIGN.md 3): the chain's
    # 8 B/voxel (SURVEY 8(d)) are split between the kernel that reads the volume once and the one that writes it once; the
    # intermediates they exchange are NF/H of a volume.  The whole-step figure below uses the full 8 B/voxel.
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"]) if kernels else None
    peak, peak_src = peak_hbm()
    roofline = None
    if dom:
        kd = kernels[dom]
        vox = SHAPE[0] * SHAPE[1] * SHAPE[2]
        units_per_launch = vols_per_step / kd["launches_per_step"]
        nf = 13
        half = 4 + 8.0 * nf / SHAPE[0]
        own = {"k_bl_fwd_h": half, "k_bl_fwd_tc": half, "k_bl_inv_h": half, "k_bl_inv_sp": half,
               "k_salt_pepper<philox>": 4.0 * (cfg["p"] or 0.0)}.get(dom, 8.0)
        # DRAM bytes per volume of that kernel from the committed ncu capture of this command (profiles/r02_ncu_traffic.json,
        # keyed by workload and kernel); null when no capture matches this configuration
        ncu_traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                tr = json.load(f)
            key = args.workload if args.disk_r is None and (FUSED_SP and SPARSE_SP) else None
            ncu_traffic = tr.get(key, {}).get(dom) if key else None
        except Exception:  # noqa: BLE001
            ncu_traffic = None
        alg_bytes = own * vox * units_per_launch
        achieved = alg_bytes / (kd["avg_launch_ms"] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": None if ncu_traffic is None else ncu_traffic * units_per_launch,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                    "algorithmic_bytes_per_voxel_this_kernel": own,
                    "share_of_step": kd["ms_per_step"] / sum(v["ms_per_step"] for v in kernels.values()),
                    "chain_bytes_per_voxel": BYTES_PER_VOXEL}

    # ---- end to end through the public API with host buffers: every step copies the batch from pinned host
    # memory, runs the chain, and copies the result back.  The batch moves in slices so that the H2D copy of
    # slice i+1, the kernels of slice i and the D2H copy of slice i-1 overlap (three streams, PCIe is duplex).
    e2e_steps = max(1, min(args.steps, 20))
    if args.no_e2e:
        e2e_steps = 0
    from mvtb import hostmem
    affinity0 = os.sched_getaffinity(0)
    numa = hostmem.bind_to_gpu_numa_node(local_rank)           # pinned pages are first-touched on the GPU's node
    Be = B if B * C <= 64 else max(1, 64 // C)                 # the host-buffer leg moves at most 64 volumes (2.3 GB each way) per step
    hx = torch.empty((Be,) + tuple(x.shape[1:]), dtype=torch.float32, pin_memory=True)
    hx.copy_(x[:Be])
    hy = torch.empty(hx.shape, dtype=torch.float32, pin_memory=True)
    xd = torch.empty((Be,) + tuple(x.shape[1:]), dtype=torch.float32, device=dev)     # device staging, transformed in place
    n_slices = 8 if Be % 8 == 0 else (4 if Be % 4 == 0 else 1)
    sl = Be // n_slices
    main = torch.cuda.current_stream(dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ev_in = [torch.cuda.Event() for _ in range(n_slices)]
    ev_done = [torch.cuda.Event() for _ in range(n_slices)]
    ev_out = [torch.cuda.Event() for _ in range(n_slices)]
    groups_per_slice = sl * C * SHAPE[0] * SHAPE[1] * SHAPE[2] // 4

    def e2e_step(s, compute=True):
        for i in range(n_slices):
            lo_, hi_ = i * sl, (i + 1) * sl
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_out[i])                     # the previous step's result has left this slice
                xd[lo_:hi_].copy_(hx[lo_:hi_], non_blocking=True)
                ev_in[i].record(s_in)
            main.wait_event(ev_in[i])
            if compute:
                gpu_step(cfg, xd[lo_:hi_], None if idxs is None else idxs[lo_:hi_], xd[lo_:hi_], 300 + s,
                         group_offset=(300 + s) * n_slices * groups_per_slice + i * groups_per_slice)
            ev_done[i].record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_done[i])
                hy[lo_:hi_].copy_(xd[lo_:hi_], non_blocking=True)
                ev_out[i].record(s_out)
        main.wait_stream(s_out)

    e2e_ms, e2e_checksum = float("nan"), None
    if e2e_steps:
        e2e_step(0)
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        barrier()
        t0.record()
        for s in range(e2e_steps):
            e2e_step(s + 1)
        t1.record()
        barrier()
        e2e_ms = t0.elapsed_time(t1)
        e2e_checksum = float(hy.double().sum())
    os.sched_setaffinity(0, affinity0)

    # ---- raw ceiling of the host link for this step's traffic: the same pinned buffers, H2D and D2H at once on two
    # streams, no kernels (what e2e could reach if the chain were free)
    ceiling_ms = float("nan")
    if e2e_steps:
        e2e_step(0, compute=False)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        for s_ in range(5):
            e2e_step(s_ + 1, compute=False)
        c1.record()
        barrier()
        ceiling_ms = c0.elapsed_time(c1) / 5

    # ---- parity spot check, outside every timed region: sample 0 of this rank's batch through the same calls against
    # the oracle (float64 exact-phase chain for the k-space part; SaltAndPepper on the coordinates the kernel hit)
    parity = None
    if rank == 0 and args.workload == "cfg2" and not args.no_parity:
        from oracle import ref_port as P
        x0 = x[0:1]
        y3 = gpu_step(dict(cfg, p=None), x0, idxs[0:1], torch.empty_like(x0), 0)
        y4 = gpu_step(cfg, x0, idxs[0:1], torch.empty_like(x0), 0)
        torch.cuda.synchronize(dev)
        a3, a4 = y3[0].cpu(), y4[0].cpu()
        ref3 = P.chain_127_exact_phase(x0[0].cpu(), cfg["r"], idxs[0], 15.0, cfg["alpha"]).to(torch.float32)
        hit = a4 != a3
        u = torch.ones_like(a3)
        u[hit] = torch.where(a4[hit] == a3.min() / 2, torch.tensor(cfg["p"] / 4), torch.tensor(3 * cfg["p"] / 4))
        parity = {"kspace_rel_l2_vs_fp64_oracle": float((a3 - ref3).norm() / ref3.norm()), "tolerance": 1e-5,
                  "select_equals_oracle_on_its_coordinates": bool(torch.equal(P.salt_and_pepper(a3, cfg["p"], u), a4)),
                  "select_rate": float(hit.float().mean()), "sample": "sample 0 of rank 0, same library calls as the timed step"}

    # ---- max over ranks, whole-job aggregate; NCCL only gathers statistics
    stats = torch.tensor([ms, e2e_ms, float(B), checksum, ceiling_ms, float(Be)], dtype=torch.float64, device=dev)
    mx, sm = aggregate(stats, world)
    ms, e2e_ms, ceiling_ms = float(mx[0]), float(mx[1]), float(mx[4])
    total_vols_per_step, checksum, total_e2e_per_step = float(sm[2]), float(sm[3]), float(sm[5])

    if dumped:
        write_outputs(args.dump_outputs, dumped)
    if rank == 0:
        value = total_vols_per_step * args.steps / (ms * 1e-3)
        e2e_value = total_e2e_per_step * e2e_steps / (e2e_ms * 1e-3) if e2e_steps else None
        step_bytes = BYTES_PER_VOXEL * voxels
        line = {
            "metric": "volumes/sec (240x240x155 fp32)", "value": value, "unit": "volumes/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {cfg['name']}", "volume": "%dx240x240x155" % C, "samples_per_gpu": B,
                       "volumes_per_step_per_gpu": vols_per_step, "parallelism": f"batch-sharded x{world}, no data-path collective",
                       "l2": "inputs larger than L2 (%.2f GB in + out per step per GPU)" % (2 * voxels * 4 / 1e9),
                       "rng": "in-kernel Philox4x32-10, " + ("geometric-gap sampler: i.i.d. Bernoulli(p) hits + fair salt/pepper coin, cost ~ p" if SPARSE_SP else "one uniform per voxel")},
            "channel_volumes_per_s": value * C,
            "roofline": roofline,
            "roofline_whole_step": {"achieved": step_bytes / (ms / args.steps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": (step_bytes / (ms / args.steps * 1e-3) / 1e9) / peak,
                                    "note": "8 B/voxel x voxels per step / step time: the figure the 60% target refers to"},
            "kernels": kernels,
            "e2e": {"value": e2e_value, "unit": "volumes/s", "h2d_bytes_per_step": int(hx.numel() * 4), "d2h_bytes_per_step": int(hx.numel() * 4),
                    "samples_per_step_per_gpu": Be,
                    "steps": e2e_steps, "slices_per_step": n_slices, "checksum": e2e_checksum, "numa_rank0": numa,
                    "host_link_ceiling": None if not e2e_steps else {
                        "value": total_e2e_per_step / (ceiling_ms * 1e-3), "unit": "volumes/s",
                        "GBps_each_way_per_gpu": hx.numel() * 4 / (ceiling_ms * 1e-3) / 1e9,
                        "how": "the e2e step with the library calls left out: the same slices copied H2D and D2H on the same streams and events, max over ranks",
                        "e2e_frac_of_ceiling": (e2e_value or 0.0) / (total_e2e_per_step / (ceiling_ms * 1e-3))}},
            "parity_spot_check": parity,
            "gpu_launches": launches,
            "clocks": clocks,
            "checksum": checksum,
        }
        if not args.no_cpu_baseline and world >= 1:
            nv = max(1, args.cpu_volumes // (C * C))
            v, cores, ts, v1, kind = time_cpu_reference(cfg, nv)
            src = ("the unmodified reference classes (oracle/_ref through oracle/monai_shim)" if kind == "reference"
                   else "oracle/ref_port.py (same torch op sequence as the reference)")
            line["cpu_baseline"] = {"value": v, "unit": "volumes/s", "cores": cores, "kind": kind, "value_1_thread": v1,
                                    "sample": f"{nv} sample(s) of {C}x240x240x155 through {src}, {cores} threads, {sum(ts):.1f} s; "
                                              f"1 more on one thread"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
