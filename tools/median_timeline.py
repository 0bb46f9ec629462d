"""Timeline and timing of the temporal median's TMA tile kernels on 1080p clips: the bench clip (bench.make_clip_device)
and uniform random bytes.

For every tile-kernel variant of tools/median_timeline.cu at the frame counts it serves, this
  1. checks that the variant's output equals ops.temporal_median's on the bytes its tiles cover;
  2. times it with CUDA events (--launches per sample, --rounds samples, the variants of one n alternated round by round);
  3. launches its TRACE build once and reports, per tile and warp, the mbarrier wait, the ldmatrix drain and the search
     (mean and p90, microseconds), the share of the warps' time in each, the share of time in which no warp of an SM
     (of one of its four schedulers) is searching, how many warps each scheduler holds, and when the SMs finish.

    python tools/median_timeline.py [--lib SO] [--out JSON]

Without --lib the variants are compiled with nvcc into a temporary directory."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from video_unscreen_b200 import ops  # noqa: E402

TRACE_WORDS = 6   # msad::TRACE_WORDS
# (clip, frame count) -> variants <C,G,SS,warps per pipeline,CTAs per SM,pipelines per CTA> to compare (names as in
# tools/median_timeline.cu); the first of each list is the old dispatch.  "bench": bench.make_clip_device; "random": uniform random bytes (every warp takes the full-range search).
CASES = {
    ("bench", 300): ["4,38,19,8,1,1", "4,38,19,4,2,1", "4,38,19,4,1,2", "2,19,9,8,2,1"],
    ("random", 300): ["4,38,19,8,1,1", "4,38,19,4,2,1", "4,38,19,4,1,2"],
    ("bench", 232): ["4,29,12,8,1,1", "4,29,12,4,2,1", "4,29,12,4,3,1", "4,29,12,4,1,3"],
    ("random", 232): ["4,29,12,8,1,1", "4,29,12,4,3,1", "4,29,12,4,1,3"],
    ("bench", 152): ["4,19,6,8,2,1", "4,19,6,4,2,1", "4,19,6,4,3,1", "4,19,6,4,4,1", "4,19,6,4,1,4"],
    ("random", 152): ["4,19,6,8,2,1", "4,19,6,4,4,1", "4,19,6,4,1,4"],
    ("bench", 600): ["2,38,19,8,1,1"],
}


def build(tmp):
    so = os.path.join(tmp, "median_timeline.so")
    subprocess.run(["nvcc", "-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-shared", "-o", so, os.path.join(ROOT, "tools", "median_timeline.cu"),
                    os.path.join(ROOT, "video_unscreen_b200", "csrc", "vu_api.cu")], check=True)
    return so


def segments(iv):
    """total length of the union of intervals iv[:, 0] .. iv[:, 1]"""
    iv = iv[np.argsort(iv[:, 0])]
    tot, cs, ce = 0, iv[0, 0], iv[0, 1]
    for s, e in iv[1:]:
        if s > ce:
            tot += ce - cs
            cs, ce = s, e
        else:
            ce = max(ce, e)
    return tot + ce - cs


def analyse(tr):
    """tr: [records, TRACE_WORDS] of one traced launch (zero rows: slots of tiles a warp did not get)"""
    tr = tr[tr[:, 0] != 0].astype(np.int64)
    wait, drain, search = tr[:, 1] - tr[:, 0], tr[:, 2] - tr[:, 1], tr[:, 3] - tr[:, 2]
    st = lambda x: {"mean_us": round(float(x.mean()) / 1e3, 3), "p90_us": round(float(np.percentile(x, 90)) / 1e3, 3)}
    busy = wait + drain + search
    stamps = np.sort(np.unique(tr[:, :4]))
    res = {"tiles_x_warps": int(len(tr)), "wait": st(wait), "drain": st(drain), "search": st(search),
           "share_of_warp_time": {k: round(float(v.sum() / busy.sum()), 3) for k, v in (("wait", wait), ("drain", drain), ("search", search))},
           "globaltimer_step_ns": int(np.diff(stamps)[np.diff(stamps) > 0].min())}
    sm, smsp = tr[:, 5] >> 40, (tr[:, 5] >> 32) & 3   # SM, and the scheduler (sub-partition) of the warp's slot
    t0 = tr[:, 0].min()
    idle, idle_sp, ends, per_sp = [], [], [], []
    for s in np.unique(sm):
        r, sp = tr[sm == s], smsp[sm == s]
        span = r[:, 3].max() - r[:, 0].min()
        idle.append(1 - segments(r[:, [2, 3]]) / span)
        ends.append(r[:, 3].max() - t0)
        for p in range(4):
            rp = r[sp == p]
            per_sp.append(len(np.unique(rp[:, 5] >> 32)))
            idle_sp.append(1 - segments(rp[:, [2, 3]]) / span if len(rp) else 1.0)
    res["sm_share_no_warp_searching"] = round(float(np.mean(idle)), 3)
    res["smsp_share_no_warp_searching"] = round(float(np.mean(idle_sp)), 3)
    res["warps_per_smsp"] = {str(k): int(v) for k, v in zip(*np.unique(per_sp, return_counts=True))}
    res["sm_end_us"] = {"min": round(float(min(ends)) / 1e3, 2), "mean": round(float(np.mean(ends)) / 1e3, 2), "max": round(float(max(ends)) / 1e3, 2)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="prebuilt tools/median_timeline.cu (.so linked with vu_api.cu)")
    ap.add_argument("--out", help="write the results as JSON here")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--cases", help="comma list of cases to run, e.g. bench300,random300 (default: all)")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="median_timeline_")
    lib = ctypes.CDLL(args.lib or build(tmp))
    lib.mt_name.restype = ctypes.c_char_p
    lib.mt_run.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
                           ctypes.POINTER(ctypes.c_longlong), ctypes.c_void_p]
    names = {lib.mt_name(i).decode(): i for i in range(lib.mt_count())}
    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    result = {"device": props.name, "nvidia_smi": smi, "clips": "bench: bench.make_clip_device(n, 1080, 1920, seed 0); random: torch.randint, generator seed n", "launches": args.launches,
              "rounds": args.rounds, "cases": {}}
    print(json.dumps({"device": props.name, "nvidia_smi": smi}), flush=True)
    h, w = 1080, 1920
    stream = torch.cuda.current_stream().cuda_stream
    only = set(args.cases.split(",")) if args.cases else None
    for (clip, n), variants in CASES.items():
        if only and f"{clip}{n}" not in only:
            continue
        if clip == "bench":
            frames = bench.make_clip_device(n, h, w, 0, dev)
        else:
            g = torch.Generator(device=dev).manual_seed(n)
            frames = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
        m = frames[0].numel()
        ref = ops.temporal_median(frames).reshape(-1)
        outs = {v: torch.zeros(m, dtype=torch.uint8, device=dev) for v in variants}
        done = ctypes.c_longlong()

        def run(v, trace=None):
            e = lib.mt_run(names[v], frames.data_ptr(), n, m, outs[v].data_ptr(), trace.data_ptr() if trace is not None else None,
                           ctypes.byref(done), stream)
            if e != 0:
                raise SystemExit(f"variant {v} at n={n}: status {e}")
            return done.value * lib.mt_seg(names[v])

        case = {}
        for v in variants:
            covered = run(v)
            torch.cuda.synchronize()
            if not torch.equal(outs[v][:covered], ref[:covered]):
                raise SystemExit(f"variant {v} at n={n}: output differs from ops.temporal_median")
            case[v] = {"bytes_covered": covered, "ms": []}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.rounds):
            for v in variants:
                for _ in range(3):
                    run(v)
                ev[0].record()
                for _ in range(args.launches):
                    run(v)
                ev[1].record()
                ev[1].synchronize()
                case[v]["ms"].append(round(ev[0].elapsed_time(ev[1]) / args.launches, 4))
        for v in variants:
            i = names[v]
            warps, ctas, pipes = (int(x) for x in v.split(",")[3:6])
            ms = case[v]["ms"]
            case[v]["ms_median"] = float(np.median(ms))
            case[v]["ms_spread"] = [min(ms), max(ms)]
            ntiles = case[v]["bytes_covered"] // (warps * lib.mt_seg(i))
            grid = min(-(-ntiles // pipes), props.multi_processor_count * ctas)
            per = -(-ntiles // (grid * pipes))
            trace = torch.zeros(grid * pipes * warps * per * TRACE_WORDS, dtype=torch.int64, device=dev)
            run(v, trace)
            ev[0].record()
            run(v, trace)
            ev[1].record()
            ev[1].synchronize()
            if not torch.equal(outs[v][:case[v]["bytes_covered"]], ref[:case[v]["bytes_covered"]]):
                raise SystemExit(f"traced variant {v} at n={n}: output differs")
            case[v]["traced_ms"] = round(ev[0].elapsed_time(ev[1]), 4)
            case[v]["timeline"] = analyse(trace.cpu().numpy().reshape(-1, TRACE_WORDS))
            print(json.dumps({"clip": clip, "n": n, "variant": v, **case[v]}), flush=True)
        result["cases"][f"{clip}{n}"] = case
        del frames, outs, ref
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
