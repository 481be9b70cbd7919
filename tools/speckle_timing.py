#!/usr/bin/env python
"""Cost of the speckle filter (stereo_ctx_set_speckle_filter): each workload timed with the filters off, the speckle
filter alone and the left-right check plus the speckle filter, alternating call by call in one process, on inputs rotated
past the 126 MB L2.

    python tools/speckle_timing.py [--reps N] [--profile DIR]      -> one JSON line

Workloads (max_size 100, max_diff 1; the left-right check with max_diff 1):
  4k_x4_i16     stereo_disparity_pair_batch_u8_device, 2160 x 3840, 256 disparities, 11 x 11, 4 pairs, int16 maps
  720p_x16_i8   stereo_disparity_pair_batch_u8_device, 720 x 1280, 64 disparities, 9 x 9, 16 pairs, int8 maps
  4k_x4_f32host stereo_disparity_pair_batch_f32_host, the first workload from CV_32FC1 host images (upload, compute,
                download; timed with the host clock around the synchronous call)
Device workloads are timed with CUDA events on the call's stream.  Every line holds the median ms of each mode, the
differences to "off", the share of pixels the filter removed, and the GPU's name and power limit read in the same run.
The filter's kernels alone (stereo_filter_speckles_device) are timed on one 4K map of the first workload and on a 4K
serpentine map (one 1-pixel-wide path through the whole map, the deepest union-find trees).
--profile DIR: instead of the timing, one torch.profiler trace of the filter alone on the 4K x 4 maps, per kernel, written
to DIR/speckle_kernels.json (a separate run: tracing slows the host)."""
import argparse
import ctypes as C
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from lr_check_timing import gpu_info      # noqa: E402

MAX_SIZE, MAX_DIFF, LR_DIFF = 100, 1, 1
L2_BYTES = 126 << 20
MODES = ("off", "speckle", "lr_speckle")


def set_mode(ctx, mode):
    ctx.set_lr_check(LR_DIFF if mode == "lr_speckle" else None)
    ctx.set_speckle_filter(MAX_SIZE if mode != "off" else None, MAX_DIFF)


def summarize(times):
    med = {m: statistics.median(t) for m, t in times.items()}
    rec = {f"median_ms_{m}": round(v, 4) for m, v in med.items()}
    for m in MODES[1:]:
        rec[f"diff_ms_{m}"] = round(med[m] - med["off"], 4)
        rec[f"diff_pct_{m}"] = round(100.0 * (med[m] - med["off"]) / med["off"], 2)
    rec.update({f"spread_ms_{m}": [round(min(t), 4), round(max(t), 4)] for m, t in times.items()})
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30, help="timed calls per mode and workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", default=None, help="write a per-kernel torch.profiler table of the filter alone here")
    args = ap.parse_args()

    import torch
    import introtocomputervision_b200 as sb
    from introtocomputervision_b200 import _capi, synth
    lib = _capi.lib()
    dev = torch.device("cuda", 0)
    ctx = sb.Context(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = C.c_void_p(stream.cuda_stream)

    def check(rc):
        if rc != 0:
            raise RuntimeError(_capi.last_error())

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    def filter_alone(maps, rng, rows, cols, elem):
        for m in maps:
            check(lib.stereo_filter_speckles_device(ctx.handle, m.data_ptr(), cols * elem, elem, rows, cols, -(rng + 1), MAX_SIZE,
                                                    MAX_DIFF, sp))

    result = {"tool": "speckle_timing", "max_size": MAX_SIZE, "max_diff": MAX_DIFF, "lr_max_diff": LR_DIFF, "reps": args.reps,
              "workloads": {}}

    def device_workload(tag, rows, cols, nd, R, B, elem, timing=True):
        tdt = {1: torch.int8, 2: torch.int16}[elem]
        rng = nd - 1
        sets = max(2, -(-L2_BYTES // (B * 2 * rows * cols)) + 1)       # input sets rotated so that each call's inputs miss the L2
        imgs = []
        for s in range(sets):
            L, Rt, _ = synth.make_pair(rows, cols, nd, 100 + s)
            imgs.append((torch.from_numpy(np.stack([L] * B)).to(dev), torch.from_numpy(np.stack([Rt] * B)).to(dev)))
        out = torch.empty((2, B, rows, cols), dtype=tdt, device=dev)

        def call(s):
            dl, dr = imgs[s % sets]
            check(lib.stereo_disparity_pair_batch_u8_device(ctx.handle, sb.COST_SSD, B, dl.data_ptr(), dr.data_ptr(), cols, rows * cols,
                                                            rows, cols, R, rng, out[0].data_ptr(), out[1].data_ptr(), cols * elem,
                                                            rows * cols * elem, elem, sp))

        if not timing:
            set_mode(ctx, "off")
            call(0)
            torch.cuda.synchronize()
            return out, rng
        times = {m: [] for m in MODES}
        for i in range(args.warmup + args.reps):
            order = MODES if i % 2 == 0 else MODES[::-1]
            for mode in order:
                set_mode(ctx, mode)
                t = timed(lambda: call(i))
                if i >= args.warmup:
                    times[mode].append(t)
        launches = {}
        for mode in MODES:
            set_mode(ctx, mode)
            call(0)
            launches[mode] = ctx.last_launches
        removed = float((out == -(rng + 1)).float().mean().item())       # (lr_speckle, the last mode)
        set_mode(ctx, "speckle")
        call(0)
        removed_speckle = float((out == -(rng + 1)).float().mean().item())
        set_mode(ctx, "off")
        rec = summarize(times)
        rec.update(shape=f"{rows}x{cols}", disparities=nd, window=2 * R + 1, pairs=B, elem_bytes=elem, input_sets=sets,
                   timing="cuda events", launches=launches, sentinel_share_speckle=round(removed_speckle, 4),
                   sentinel_share_lr_speckle=round(removed, 4))
        result["workloads"][tag] = rec
        return out, rng

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        out4k, rng4k = device_workload("4k_x4_i16", 2160, 3840, 256, 5, 4, 2, timing=False)
        maps = [out4k[s, k].clone() for s in range(2) for k in range(out4k.shape[1])]
        filter_alone(maps, rng4k, 2160, 3840, 2)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                fresh = [m.clone() for m in maps]
                filter_alone(fresh, rng4k, 2160, 3840, 2)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if "speckle" in e.key:
                per[e.key] = {"calls": e.count, "mean_us": round(e.device_time_total / max(e.count, 1), 2)}
        name, limit = gpu_info()
        rec = {"tool": "speckle_timing --profile", "maps": len(maps), "shape": "2160x3840", "elem_bytes": 2, "kernels": per,
               "gpu": name or torch.cuda.get_device_name(0), "power_limit": limit}
        Path(args.profile).mkdir(parents=True, exist_ok=True)
        (Path(args.profile) / "speckle_kernels.json").write_text(json.dumps(rec) + "\n")
        print(json.dumps(rec))
        ctx.close()
        return

    out4k, rng4k = device_workload("4k_x4_i16", 2160, 3840, 256, 5, 4, 2)
    # the filter's kernels alone on one 4K map of the workload (unfiltered: a copy is restored before each call) and on the
    # serpentine map
    rows, cols = 2160, 3840
    set_mode(ctx, "off")
    out4k, _ = device_workload("4k_x4_i16", rows, cols, 256, 5, 4, 2, timing=False)
    src = out4k[0, 0].clone()
    d = np.zeros((rows, cols), np.int16)
    d[1::2] = 9
    for k, y in enumerate(range(1, rows, 2)):
        d[y, cols - 1 if k % 2 == 0 else 0] = 0
    serp = torch.from_numpy(d).to(dev)
    alone = {}
    for tag, base in (("4k_map", src), ("4k_serpentine", serp)):
        work = base.clone()
        ts = []
        for i in range(args.warmup + args.reps):
            work.copy_(base)
            t = timed(lambda: filter_alone([work], rng4k, rows, cols, 2))
            if i >= args.warmup:
                ts.append(t)
        alone[tag] = {"median_ms": round(statistics.median(ts), 4), "spread_ms": [round(min(ts), 4), round(max(ts), 4)],
                      "removed_share": round(float((work != base).float().mean().item()), 4)}
    result["filter_kernels_alone"] = alone

    device_workload("720p_x16_i8", 720, 1280, 64, 4, 16, 1)

    # CV_32FC1 host images, 4K x 4 pairs
    rows, cols, nd, R, B = 2160, 3840, 256, 5, 4
    rng = nd - 1
    sets = 2
    host = []
    for s in range(sets):
        L, Rt, _ = synth.make_pair(rows, cols, nd, 200 + s)
        host.append((np.stack([L.astype(np.float32)] * B), np.stack([Rt.astype(np.float32)] * B)))
    times = {m: [] for m in MODES}
    share = {}
    for i in range(args.warmup + args.reps):
        for mode in (MODES if i % 2 == 0 else MODES[::-1]):
            set_mode(ctx, mode)
            Ls, Rs = host[i % sets]
            t0 = time.perf_counter()
            dl, dr = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, R, rng, dtype=np.int16)
            t1 = time.perf_counter()
            if i >= args.warmup:
                times[mode].append((t1 - t0) * 1e3)
            share[mode] = float(np.mean(np.concatenate([dl.ravel(), dr.ravel()]) == -(rng + 1)))
    set_mode(ctx, "off")
    rec = summarize(times)
    rec.update(shape=f"{rows}x{cols}", disparities=nd, window=2 * R + 1, pairs=B, elem_bytes=2, input_sets=sets,
               timing="host clock around the synchronous call", sentinel_share_speckle=round(share["speckle"], 4),
               sentinel_share_lr_speckle=round(share["lr_speckle"], 4))
    result["workloads"]["4k_x4_f32host"] = rec

    name, limit = gpu_info()
    result["gpu"] = name or torch.cuda.get_device_name(0)
    result["power_limit"] = limit
    print(json.dumps(result))
    ctx.close()


if __name__ == "__main__":
    main()
