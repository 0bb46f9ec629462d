#!/usr/bin/env python
"""Benchmark of the B200 video_unscreen hot path (contract: see the task brief).

Default workload = BASELINE.json configs[1]: bg_step temporal-median
background estimation over 300 synthetic 1080p frames.  A "step" is one pass
of the exact temporal median over the whole clip (1.87 GB, far larger than the
126 MB L2, so every step streams from HBM).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` = frames/s with the clip resident in
HBM; `e2e` = the same through the public numpy-style API with the clip in pinned
host memory (H2D of the clip and D2H of the background inside the timed
region); `roofline` = algorithmic bytes of the dominant kernel / its CUDA-event
duration against the measured HBM copy bandwidth; `cpu_baseline` = the oracle
port on this box's host cores over a bounded sample.

The same line carries `configs`: one block per BASELINE.json config (frames/s,
roofline, cpu_baseline, e2e, bit-exact check; tools/bench_configs.py), sharded
the way north_star names when run under torchrun (frame ranges for the
per-frame configs, row tiles of ONE 4K clip for bg_step: "scaling": "strong"),
`roofline_worst_case` (the median on uniform-random bytes) and `per_frame` (the
reference's per-frame numpy API).  `--configs none` skips them.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (frames, H, W, description)
    "median_1080p": (300, 1080, 1920, "bg_step temporal-median background over 300 synthetic 1080p frames (BASELINE configs[1])"),
    "median_4k": (300, 2160, 3840, "bg_step temporal-median background over 300 synthetic 4K frames"),
    "median_4k_tile2000": (2000, 270, 3840, "one GPU's row tile (270 rows) of the 4K 2000-frame clip of BASELINE configs[4]: temporal median"),
}
METRIC = "frames/sec at 1080p & 4K (1/2/4/8 B200) + % HBM roofline vs host-CPU ref"
KERNELS = {
    "median_1080p": "vu::msad::median_sad_tma_kernel<2,38,30,8,8,1> (TMA tiles, VABSDIFF4 estimate + windowed Fibonacci search)",
    "median_4k": "vu::msad::median_sad_tma_kernel<2,38,30,8,8,1> (TMA tiles, VABSDIFF4 estimate + windowed Fibonacci search)",
    "median_4k_tile2000": "vu::msad::median_sad_tma_kernel (every 7th frame) + vu::msad::median_refine_kernel (streaming S at 8 probes) + "
                          "median_kernel fix-up; algorithmic bytes / time of the three launches",
}
FALLBACK_HBM_GBS = 6650.0
DUMP_BYTES = 64 * 10**6   # cap of what --dump-outputs writes


def dump_outputs(path, background):
    """--dump-outputs: the background the timed path returned in its last step, as float32 `background.npy` under
    `path`, with the image rows it holds in `background_rows.npy`: every row, or a fixed seeded sample of them when
    the whole image would exceed DUMP_BYTES."""
    h = background.shape[0]
    row_bytes = background[0].size * 4 + 8
    rows = np.arange(h)
    if h * row_bytes > DUMP_BYTES - 1024:   # 1024: room for the two .npy headers
        rows = np.sort(np.random.default_rng(0).choice(h, (DUMP_BYTES - 1024) // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "background.npy"), background[rows].astype(np.float32))
    np.save(os.path.join(path, "background_rows.npy"), rows.astype(np.float64))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def measured_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            v = json.load(open(p)).get(workload)
            return int(v) if v is not None else None
        except Exception:
            pass
    return None


# --------------------------------------------------------------------------
# CPU arm: the oracle port of the temporal median on all host threads
# --------------------------------------------------------------------------

def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def config_dict(args, wl):
    """identical in both arms (the driver compares them)"""
    n, h, w, desc = wl
    return {"workload": args.workload, "description": desc, "frames": n, "height": h, "width": w}


def pin_to_gpu_cpus(index):
    """bind this rank to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is allocated, so the
    staging memory of the e2e path sits on the GPU's NUMA node.  Returns what was done (for the bench line)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        want = cpus & allowed
        if want and want != allowed:
            os.sched_setaffinity(0, want)
            return {"pinned": True, "cpus": len(want), "of_allowed": len(allowed)}
        return {"pinned": False, "cpus": len(allowed), "why": "the GPU's CPU set already equals the allowed set" if want else "no overlap"}
    except Exception as ex:
        return {"pinned": False, "why": str(ex)[:80]}


def cpu_median_sample(frames_host, rows, threads):
    """oracle median (oracle.refport.temporal_median == np.median(...).astype(u8))
    over `rows` rows of every frame, split over `threads` host threads."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import refport as R
    n = frames_host.shape[0]
    chunks = [c for c in np.array_split(np.arange(rows), threads) if len(c)]

    def work(c):
        return R.temporal_median(frames_host[:, c[0]:c[-1] + 1])
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        out = list(ex.map(work, chunks))
    dt = time.perf_counter() - t0
    return dt, np.concatenate(out, 0), n


def synth_clip_host(n, h, w, rows=None, seed=0):
    """numpy version of the synthetic bg_step clip (used when no GPU is around)."""
    from video_unscreen_b200 import synth
    rows = rows or h
    frames, _, _ = synth.bgstep_clip(n, rows, w, seed=seed)
    return frames


def run_reference_arm(args, wl):
    n, h, w, desc = wl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    rows = min(h, max(threads, int(args.sample_rows)))
    frames = synth_clip_host(n, h, w, rows=rows)
    times = []
    for i in range(args.warmup_ref + args.steps_ref):
        dt, _, _ = cpu_median_sample(frames, rows, threads)
        if i >= args.warmup_ref:
            times.append(dt)
    dt = float(np.mean(times))
    fps = n * (rows / h) / dt
    sample = f"{rows} of {h} rows of all {n} frames per step ({rows * w * 3 * n / 1e6:.0f} MB), {len(times)} timed steps; frames/s scaled by rows/{h}"
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup_ref, "ms_per_step": dt * 1e3 * (h / rows), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": config_dict(args, wl),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": sample + "; oracle.refport.temporal_median (np.partition, the survey's np.median spec; the reference has no median)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "a per-pixel-independent op: the rows/h scaling of the sampled rows is exact up to cache effects",
    }
    if args.configs != "none":
        line["configs"] = reference_configs(threads)
    print(json.dumps(line), flush=True)
    return 0


def reference_configs(threads):
    """the oracle port of the per-frame BASELINE configs on the host cores (one frame per thread), for the reference arm"""
    from oracle import refport as R
    BC = _bench_configs()
    from video_unscreen_b200 import synth
    c = np.load(os.path.join(ROOT, "tests", "golden", "colorfilter.npz"))
    tabs = {}
    for tag in ("x2", "x4"):
        lb = np.stack([R.gmm_lut(c[f"{tag}_bg{i}_means"], c[f"{tag}_bg{i}_covs"], c[f"{tag}_bg{i}_weights"]) for i in range(3)])
        lf = np.stack([R.gmm_lut(c[f"{tag}_fg{i}_means"], c[f"{tag}_fg{i}_covs"], c[f"{tag}_fg{i}_weights"]) for i in range(3)])
        tabs[tag] = (lb, lf, R.bg_color_hsv([np.atleast_1d(c[f"{tag}_bg{i}_means"])[0] for i in range(3)]))
    col = np.array(synth.GREEN_BG, np.uint8)
    out = {}
    fr, sg = zip(*[synth.green_frame(1080, 1920, t=t, n=6, seed=0) for t in range(2)])

    def cfg1(i):
        a, _, _ = R.cf_forward_predict(fr[i % 2], sg[i % 2], *tabs["x2"], 960)
        return R.generate_trimap_withbg(a, fr[i % 2], col, 960)
    dt, _ = BC.parallel_cpu(cfg1, list(range(threads)), threads)
    out["cf_trimap_1080p"] = {"value": threads / dt, "unit": "frames/s", "cores": threads, "kind": "port", "sample": f"{threads} frames in {dt:.1f} s"}
    f4, s4 = synth.green_frame(2160, 3840, t=1, n=3, seed=0)

    def cfg3(i):
        a, _, _ = R.cf_forward_predict(f4, s4, *tabs["x4"], 960)
        R.generate_trimap_withbg(a, f4, col, 960)
        b = R.patch_bg(np.broadcast_to(col, f4.shape), f4, a, "lt128")
        return R.get_fg(f4, a, b)
    th4 = min(threads, 8)
    dt, _ = BC.parallel_cpu(cfg3, list(range(th4)), th4)
    out["green_4k"] = {"value": th4 / dt, "unit": "frames/s", "cores": th4, "kind": "port", "sample": f"{th4} 4K frames in {dt:.1f} s"}
    rng = np.random.default_rng(3)
    fg, al, bg = rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8), rng.integers(0, 256, (1080, 1920), dtype=np.uint8), \
        rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    dt, _ = BC.parallel_cpu(lambda i: R.replace_blend(fg, al, bg), list(range(2 * threads)), threads)
    out["replace_1080p"] = {"value": 2 * threads / dt, "unit": "frames/s", "cores": threads, "kind": "port", "sample": f"{2 * threads} frames in {dt:.1f} s"}
    return out


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    def __init__(self, index, period=0.001):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": int(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _bench_configs():
    import importlib
    if os.path.join(ROOT, "tools") not in sys.path:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
    return importlib.import_module("bench_configs")


def make_masks_device(n, h, w, device):
    return _bench_configs().make_masks_device(n, h, w, device)


def make_clip_device(n, h, w, seed, device):
    return _bench_configs().make_clip_device(n, h, w, seed, device)


def run_gpu_arm(args, wl):
    import torch
    import torch.distributed as dist

    from video_unscreen_b200 import _lib, ops
    from video_unscreen_b200.unscreen.utils import temporal_median

    n, h, w, desc = wl
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_to_gpu_cpus(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    # ---- data: one clip per rank (weak scaling: spatial tiles / clips are independent) ----
    frames = make_clip_device(n, h, w, seed=rank, device=dev)
    out = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
    m = h * w * 3
    algo_bytes = (n + 1) * m

    def step():
        ops.temporal_median(frames, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = L.vu_launch_count()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    evs[0].record()
    for i in range(args.steps):
        step()
        evs[i + 1].record()
    evs[-1].synchronize()
    barrier()
    launches = int(L.vu_launch_count() - launches0)
    clocks = sampler.stop()
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    kernel_ms = float(np.mean(per_launch_ms))
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())

    # ---- parity spot-check of what was just timed (cheap, outside the timed region) ----
    strip = frames[:, h // 2:h // 2 + 4].to(torch.int16)
    s, _ = strip.sort(0)
    want = ((s[(n - 1) // 2] + s[n // 2]) >> 1).to(torch.uint8)
    if not torch.equal(out[h // 2:h // 2 + 4], want):
        raise SystemExit("bench: temporal median output failed its spot check")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out.cpu().numpy())   # before the worst-case block below overwrites `out`

    # ---- e2e: public API, clip in pinned host memory, result read back to the host ----
    e2e = None
    host = None
    try:
        host = torch.empty((n, h, w, 3), dtype=torch.uint8, pin_memory=True)
        host.copy_(frames)
        torch.cuda.synchronize()
        e2e_steps = max(3, min(args.steps, args.e2e_steps))
        res = None
        for _ in range(2):
            res = temporal_median(host).cpu()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            res = temporal_median(host).cpu()   # H2D of the clip, kernel, D2H of the background
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        assert torch.equal(res, out.cpu())
        # the ceiling of this path: the same bytes through a plain cudaMemcpyAsync from the same pinned buffer, all ranks at once
        stage = torch.empty_like(frames)
        stage.copy_(host, non_blocking=True)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(3):
            stage.copy_(host, non_blocking=True)
        c1.record()
        c1.synchronize()
        barrier()
        copy_ms = c0.elapsed_time(c1) / 3
        del stage
        if world > 1:
            t = torch.tensor([copy_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            copy_ms = float(t.item())
        ceiling_fps = world * n / (copy_ms * 1e-3)
        e2e = {"value": world * n * e2e_steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": int(host.numel()),
               "d2h_bytes_per_step": int(res.numel()), "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
               "api": "video_unscreen_b200.unscreen.utils.temporal_median(pinned host clip) -> host background",
               "h2d_ceiling": {"gbs_per_gpu": host.numel() / copy_ms / 1e6, "ms": copy_ms, "frames_per_s": ceiling_fps,
                               "what": f"plain cudaMemcpyAsync of the same pinned clip on all {world} ranks at once (max over ranks)"},
               "frac_of_h2d_ceiling": (world * n * e2e_steps / e2e_s) / ceiling_fps, "cpu_affinity": affinity}
    except RuntimeError as ex:  # e.g. not enough pinnable host memory
        e2e = {"value": None, "unit": "frames/s", "error": str(ex)[:200]}

    # ---- CPU baseline (rank 0, N == 1 only): oracle port on a bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = host_threads()
        rows = min(h, max(threads, int(args.sample_rows)))
        src = host if host is not None else frames.cpu()
        sample_np = src[:, :rows].numpy()
        dt, ref, _ = cpu_median_sample(sample_np, rows, threads)
        if not np.array_equal(ref, out[:rows].cpu().numpy()):
            raise SystemExit("bench: GPU median differs from the CPU oracle on the sampled rows")
        cpu = {"value": n * (rows / h) / dt, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"{rows} of {h} rows of all {n} frames ({rows * w * 3 * n / 1e6:.0f} MB) in {dt:.1f} s, scaled by rows/{h}; "
                         "oracle.refport.temporal_median (np.partition == the np.median spec; the reference has no median); "
                         "output compared bit-exactly with the GPU result"}

    # ---- the median's worst case: uniform-random bytes (no concentration around the estimate: every warp falls back) ----
    peak, peak_src = measured_peak()
    worst = None
    if args.configs != "none":
        g = torch.Generator(device=dev).manual_seed(7)
        frames.random_(0, 256, generator=g)
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for _ in range(10):
            step()
        w1.record()
        w1.synchronize()
        wms = w0.elapsed_time(w1) / 10
        s16, _ = frames[:, :8].to(torch.int16).sort(0)
        if not torch.equal(out[:8], ((s16[(n - 1) // 2] + s16[n // 2]) >> 1).to(torch.uint8)):
            raise SystemExit("bench: temporal median of the uniform-random clip failed its spot check")
        worst = {"data": "uniform-random bytes", "launch_ms": wms, "achieved": algo_bytes / (wms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                 "frac": algo_bytes / (wms * 1e-3) / 1e9 / peak, "frames_per_s": n / (wms * 1e-3)}
    del frames, host
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, sharded the way north_star names ----
    configs, per_frame = None, None
    if args.configs != "none":
        BC = _bench_configs()
        D = BC.Dist()
        configs = {}
        names = list(BC.RUNNERS) if args.configs == "all" else [c for c in args.configs.split(",") if c in BC.RUNNERS]
        for name in names:
            configs[name] = BC.RUNNERS[name](D, args.config_steps, 3, peak, cpu=(world == 1 and not args.no_cpu))
            torch.cuda.empty_cache()
        if world == 8 and "bgstep_4k" in names:
            configs["bgstep_4k_2000"] = BC.run_bgstep_4k(D, args.config_steps, 3, peak, cpu=False, frames=2000)
            torch.cuda.empty_cache()
        if world == 1 and rank == 0:
            per_frame = BC.per_frame_latency(D)

    if rank == 0:
        achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = measured_traffic(args.workload)
        line = {
            "metric": METRIC, "value": world * n * args.steps / (total_ms * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_dict(args, wl),
            "notes": {"clip_bytes": n * m, "l2": "inputs (1.87 GB at 1080p) larger than the 126 MB L2; no flush needed",
                      "sharding": "one clip (spatial tile set) per GPU, no collective"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": KERNELS.get(args.workload, KERNELS["median_1080p"]), "algorithmic_bytes_per_launch": algo_bytes,
                         "launch_ms": kernel_ms, "peak_source": peak_src},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "roofline_worst_case": worst, "configs": configs, "per_frame": per_frame,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 3 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="median_1080p", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--sample-rows", type=int, default=540, help="rows of every frame the CPU arm processes per step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--configs", default="all", help="'all', 'none' or a comma list of tools/bench_configs.py workloads for the `configs` block")
    ap.add_argument("--config-steps", type=int, default=10, help="timed steps per workload of the `configs` block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the background of the last timed step to DIR/background.npy "
                    "(float32; rank 0's clip under torchrun)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm times a separate, reduced-height clip (synth_clip_host): nothing comparable to dump
        ap.error("--dump-outputs applies to the GPU arm only")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        # each step is a bounded sample of the workload (--sample-rows rows of every frame); by default 3 of them,
        # which keeps the whole run to a few minutes
        args.steps_ref = 3 if args.steps is None else args.steps
        args.warmup_ref = 1 if args.warmup > 0 else 0
        return run_reference_arm(args, wl)
    if args.steps is None:
        args.steps = 200
    return run_gpu_arm(args, wl)


if __name__ == "__main__":
    sys.exit(main())
