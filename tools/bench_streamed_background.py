"""Rates of the streamed temporal backgrounds (ops.TemporalMedianAccumulator / ops.MaskedMeanAccumulator and the
clip.streamed_* helpers).  One JSON line per case on stdout (and appended to --out):

  hbm / h2d     the measured device-copy and pinned host->device bandwidths every fraction below refers to;
  add / finish  median accumulator on device-resident chunks, 1080p and 4K, k = 16 / 64 / 256: frames/s, the bytes
                of the traffic model (add: k*m frames + 1024*m state; finish: 512*m + m) and their share of `hbm`;
  mean_add      the same for the masked-mean accumulator (fused dilation, 4*k*npix + 32*npix bytes);
  streamed      clip.streamed_temporal_median / streamed_masked_temporal_mean against the resident
                unscreen.utils.temporal_median / masked_temporal_mean, both from one pinned host clip, alternated:
                seconds, share of the H2D ceiling (clip bytes / h2d), torch.cuda.max_memory_allocated, equality;
  long_clip     a 4K clip of --long-frames frames (8000: 199 GB, more than one B200 holds) produced chunk by chunk on
                the device from a seed (a stand-in for a decoder), accumulated, checked on a seeded sample of rows
                against ops.temporal_median of those rows' regenerated time series.

The card's name and power limit are read in the same run and written into every line.  Needs a CUDA device.
Usage: python tools/bench_streamed_background.py [--out FILE] [--long-frames 8000] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from video_unscreen_b200 import _lib, clip, ops  # noqa: E402
from video_unscreen_b200.unscreen.utils import masked_temporal_mean, temporal_median  # noqa: E402

SIZES = {"1080p": (1080, 1920), "4k": (2160, 3840)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:   # the numbers still carry the torch device name
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


class Clip:
    """a bg_step-like synthetic clip generated on the device frame range by frame range: a static random background,
    per-frame noise in [-6, 6] and a block (the 'person', masked 255) that sweeps the frame, covering any pixel in far
    fewer than half of the frames.  Frame t depends only on (seed, t)."""

    def __init__(self, h, w, seed=0, device="cuda"):
        self.h, self.w, self.seed, self.dev = h, w, seed, torch.device(device)
        g = torch.Generator(device=self.dev)
        g.manual_seed(seed)
        self.bg = torch.randint(0, 256, (h, w, 3), generator=g, device=self.dev, dtype=torch.int16)

    def fill(self, f0, frames, masks=None, sub=16):
        k = frames.shape[0]
        bw = max(1, self.w // 8)
        for s in range(0, k, sub):
            e = min(k, s + sub)
            g = torch.Generator(device=self.dev)
            g.manual_seed(self.seed * 1000003 + f0 + s)
            noise = torch.randint(-6, 7, (e - s, self.h, self.w, 3), generator=g, device=self.dev, dtype=torch.int16)
            frames[s:e] = (noise + self.bg).clamp_(0, 255).to(torch.uint8)
            if masks is not None:
                masks[s:e] = 0
            for i in range(s, e):
                x0 = ((f0 + i) * 37) % (self.w - bw)
                frames[i, self.h // 8:self.h - self.h // 8, x0:x0 + bw] = 40 + (f0 + i) % 160
                if masks is not None:
                    masks[i, self.h // 8:self.h - self.h // 8, x0:x0 + bw] = 255
        return frames, masks


def timed(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def host_timed(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, torch.cuda.max_memory_allocated() - base, r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    ap.add_argument("--long-frames", type=int, default=8000)
    ap.add_argument("--reps", type=int, default=3, help="alternated repetitions of the streamed / resident cases")
    ap.add_argument("--quick", action="store_true", help="small sizes (a dry run of the script itself)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_streamed_background.py needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    info = card()
    sizes = {"small": (72, 128)} if args.quick else SIZES
    n_stream = 40 if args.quick else 300

    def emit(rec):
        rec = {**rec, **info}
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")

    # ---- ceilings ------------------------------------------------------------------------------------------------
    nb = (1 << 26) if args.quick else (8 << 30)
    src = torch.empty(nb, dtype=torch.uint8, device=dev).fill_(1)
    dst = torch.empty_like(src)
    t = timed(lambda: dst.copy_(src), 10)
    hbm = 2 * nb / t
    emit({"case": "hbm", "what": "device-to-device copy, read + write bytes / time", "bytes": 2 * nb, "seconds": t, "bytes_per_s": hbm})
    del src, dst
    hb = torch.empty(nb // 2, dtype=torch.uint8).pin_memory()
    db = torch.empty(nb // 2, dtype=torch.uint8, device=dev)
    t = timed(lambda: db.copy_(hb, non_blocking=True), 5, warmup=1)
    h2d = (nb // 2) / t
    emit({"case": "h2d", "what": "pinned host-to-device copy", "bytes": nb // 2, "seconds": t, "bytes_per_s": h2d})
    del hb, db
    torch.cuda.empty_cache()

    L = _lib.lib()
    stream = lambda: ops._stream()  # noqa: E731

    # ---- add / finish on device-resident chunks ---------------------------------------------------------------------
    for label, (h, w) in sizes.items():
        m = h * w * 3
        gen = Clip(h, w, seed=1)
        chunk = torch.empty((256, h, w, 3), dtype=torch.uint8, device=dev)
        masks = torch.empty((256, h, w), dtype=torch.uint8, device=dev)
        gen.fill(0, chunk, masks)
        acc = ops.TemporalMedianAccumulator((h, w, 3))
        macc = ops.MaskedMeanAccumulator(h, w)
        for k in (16, 64, 256):
            fr = chunk[:k]
            # n_before = 1: every timed add reads and writes the whole state (the counts themselves are not used)
            fn = lambda: _lib.check(L.vu_median_accum_add_u8(ops._p(acc.state), m, ops._p(fr), k, 1, stream()))  # noqa: E731
            t = timed(fn, 10 if label != "small" else 3)
            model = k * m + 1024 * m
            emit({"case": "add", "size": label, "k": k, "m": m, "seconds": t, "frames_per_s": k / t, "model_bytes": model,
                  "bytes_per_s": model / t, "hbm_fraction": model / t / hbm})
            mfr, mms = chunk[:k], masks[:k]
            fn = lambda: _lib.check(L.vu_masked_mean_accum_add_dilate32(ops._p(macc.state), ops._p(mfr), ops._p(mms), k, h, w, stream()))  # noqa: E731
            t = timed(fn, 10)
            model = 4 * k * h * w + 32 * h * w
            emit({"case": "mean_add", "size": label, "k": k, "npix": h * w, "seconds": t, "frames_per_s": k / t, "model_bytes": model,
                  "bytes_per_s": model / t, "hbm_fraction": model / t / hbm})
        out = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
        t = timed(lambda: _lib.check(L.vu_median_accum_finish_u8(ops._p(acc.state), m, 300, ops._p(out), stream())), 10)
        model = 512 * m + m
        emit({"case": "finish", "size": label, "m": m, "seconds": t, "model_bytes": model, "bytes_per_s": model / t, "hbm_fraction": model / t / hbm})
        del chunk, masks, acc, macc, out
        torch.cuda.empty_cache()

    # ---- streamed against resident, from one pinned host clip ------------------------------------------------------------
    for label, (h, w) in sizes.items():
        gen = Clip(h, w, seed=2)
        hf = torch.empty((n_stream, h, w, 3), dtype=torch.uint8).pin_memory()
        hm = torch.empty((n_stream, h, w), dtype=torch.uint8).pin_memory()
        df = torch.empty((64, h, w, 3), dtype=torch.uint8, device=dev)
        dm = torch.empty((64, h, w), dtype=torch.uint8, device=dev)
        for s in range(0, n_stream, 64):
            e = min(n_stream, s + 64)
            gen.fill(s, df[:e - s], dm[:e - s])
            hf[s:e].copy_(df[:e - s])
            hm[s:e].copy_(dm[:e - s])
        del df, dm
        torch.cuda.empty_cache()
        fbytes, mbytes = hf.numel(), hm.numel()
        variants = [
            ("median", "resident", None, lambda: temporal_median(hf), fbytes),
            ("median", "streamed", 32, lambda: clip.streamed_temporal_median(hf, chunk=32), fbytes),
            ("median", "streamed", 128, lambda: clip.streamed_temporal_median(hf, chunk=128), fbytes),
            ("masked_mean", "resident", None, lambda: masked_temporal_mean(hf, hm), fbytes + mbytes),
            ("masked_mean", "streamed", 32, lambda: clip.streamed_masked_temporal_mean(hf, hm, chunk=32), fbytes + mbytes),
            ("masked_mean", "streamed", 128, lambda: clip.streamed_masked_temporal_mean(hf, hm, chunk=128), fbytes + mbytes),
        ]
        ref = {}
        for est, kind, ch, fn, nbytes in variants:      # warm-up: module loads, allocator, pinned staging
            r = fn()
            if kind == "resident":
                ref[est] = r
            del r
        times = {v[:3]: [] for v in variants}
        peaks = {v[:3]: 0 for v in variants}
        equal = {}
        for _ in range(args.reps):
            for est, kind, ch, fn, nbytes in variants:
                torch.cuda.empty_cache()
                t, peak, r = host_timed(fn)
                times[(est, kind, ch)].append(t)
                peaks[(est, kind, ch)] = max(peaks[(est, kind, ch)], peak)
                want = ref[est]
                same = torch.equal(r, want) if est == "median" else all(torch.equal(a, b) for a, b in zip(r, want))
                equal[(est, kind, ch)] = equal.get((est, kind, ch), True) and same
                del r
        for est, kind, ch, fn, nbytes in variants:
            ts = sorted(times[(est, kind, ch)])
            tmed = ts[len(ts) // 2]
            emit({"case": "streamed", "estimator": est, "path": kind, "chunk": ch, "size": label, "frames": n_stream, "host_bytes": nbytes,
                  "seconds_median": tmed, "seconds_all": ts, "h2d_ceiling_fraction": nbytes / h2d / tmed,
                  "max_memory_allocated": peaks[(est, kind, ch)], "equals_resident": equal[(est, kind, ch)]})
        del hf, hm, ref, variants
        torch.cuda.empty_cache()

    # ---- a clip longer than HBM ------------------------------------------------------------------------------------------------
    h, w = sizes["small"] if args.quick else SIZES["4k"]
    n, k = args.long_frames, 256
    gen = Clip(h, w, seed=3)
    buf = torch.empty((k, h, w, 3), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    acc = ops.TemporalMedianAccumulator((h, w, 3))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    gen_s = add_s = 0.0
    t0 = time.perf_counter()
    for s in range(0, n, k):
        e = min(n, s + k)
        ev[0].record()
        gen.fill(s, buf[:e - s])
        ev[1].record()
        acc.add(buf[:e - s])
        ev[2].record()
        torch.cuda.synchronize()
        gen_s += ev[0].elapsed_time(ev[1]) / 1e3
        add_s += ev[1].elapsed_time(ev[2]) / 1e3
    ev[0].record()
    res = acc.result()
    ev[1].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated()
    dev_s = add_s + ev[0].elapsed_time(ev[1]) / 1e3       # accumulate + finish (generation excluded)
    # check: a seeded sample of rows, their whole time series regenerated and reduced by the resident kernel
    rows = sorted(int(r) for r in torch.randperm(h, generator=torch.Generator().manual_seed(12345))[:8])
    ts = torch.empty((n, len(rows), w, 3), dtype=torch.uint8, device=dev)
    for s in range(0, n, k):
        e = min(n, s + k)
        gen.fill(s, buf[:e - s])
        ts[s:e] = buf[:e - s, rows]
    want = ops.temporal_median(ts)
    same = bool(torch.equal(res[rows], want))
    emit({"case": "long_clip", "size": f"{h}x{w}", "frames": n, "chunk": k, "clip_bytes": n * h * w * 3, "rows_checked": rows,
          "rows_equal": same, "accumulate_and_finish_seconds": dev_s, "frames_per_s": n / dev_s, "wall_seconds_with_generation": wall,
          "generation_seconds": gen_s, "max_memory_allocated": peak, "state_bytes": acc.state.numel()})
    if not same:
        raise SystemExit("long clip: the sampled rows differ from ops.temporal_median")


if __name__ == "__main__":
    main()
