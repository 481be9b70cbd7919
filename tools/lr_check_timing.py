#!/usr/bin/env python
"""Cost of the left-right consistency check (stereo_ctx_set_lr_check): each workload timed with the check off and on,
alternating call by call in one process, on inputs rotated past the 126 MB L2.

    python tools/lr_check_timing.py [--reps N]      -> one JSON line

Workloads:
  4k_x4_i16    stereo_disparity_pair_batch_u8_device, 2160 x 3840, 256 disparities, 11 x 11, 4 pairs, int16 maps
  720p_x16_i8  stereo_disparity_pair_batch_u8_device, 720 x 1280, 64 disparities, 9 x 9, 16 pairs, int8 maps
  4k_x4_f32host stereo_disparity_pair_batch_f32_host, the first workload from CV_32FC1 host images (upload, compute,
               download; timed with the host clock around the synchronous call)
Device workloads are timed with CUDA events on the call's stream.  Every line holds the median ms of each mode, their
difference, the share of pixels the check invalidated, and the GPU's name and power limit read in the same run.  The
check's kernel alone (stereo_lr_check_device over the 4K maps) is timed as well."""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

MAX_DIFF = 1
L2_BYTES = 126 << 20


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:                      # (reported, not hidden: the numbers need the card they came from)
        return None, f"unavailable: {type(e).__name__}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30, help="timed calls per mode and workload")
    ap.add_argument("--warmup", type=int, default=3)
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

    result = {"tool": "lr_check_timing", "max_diff": MAX_DIFF, "reps": args.reps, "workloads": {}}

    def device_workload(tag, rows, cols, nd, R, B, elem):
        tdt = {1: torch.int8, 2: torch.int16}[elem]
        rng = nd - 1
        pair_bytes = 2 * rows * cols
        sets = max(2, -(-L2_BYTES // (B * pair_bytes)) + 1)       # input sets rotated so that each call's inputs miss the L2
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

        times = {"off": [], "on": []}
        for i in range(args.warmup + args.reps):
            for mode in (("off", "on") if i % 2 == 0 else ("on", "off")):
                ctx.set_lr_check(MAX_DIFF if mode == "on" else None)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                call(i)
                e1.record(stream)
                e1.synchronize()
                if i >= args.warmup:
                    times[mode].append(e0.elapsed_time(e1))
        ctx.set_lr_check(MAX_DIFF)
        call(0)
        launches_on = ctx.last_launches
        invalid = float((out == -(rng + 1)).float().mean().item())
        ctx.set_lr_check(None)
        rec = summarize(times)
        rec.update(shape=f"{rows}x{cols}", disparities=nd, window=2 * R + 1, pairs=B, elem_bytes=elem, input_sets=sets,
                   timing="cuda events", launches_on=launches_on, invalidated_share=round(invalid, 4))
        result["workloads"][tag] = rec
        return out, rng

    out4k, rng4k = device_workload("4k_x4_i16", 2160, 3840, 256, 5, 4, 2)

    # the check's kernel alone over the 4K maps just computed (in place: a second pass finds the same pixels inconsistent)
    rows, cols, B = out4k.shape[2], out4k.shape[3], out4k.shape[1]
    alone = []
    for i in range(args.warmup + args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(B):
            check(lib.stereo_lr_check_device(ctx.handle, out4k[0, k].data_ptr(), out4k[1, k].data_ptr(), cols * 2, 2, rows, cols, rng4k,
                                             MAX_DIFF, sp))
        e1.record(stream)
        e1.synchronize()
        if i >= args.warmup:
            alone.append(e0.elapsed_time(e1))
    map_bytes = 2 * B * rows * cols * 2
    med = statistics.median(alone)
    result["workloads"]["4k_x4_i16"]["check_kernel_alone_ms"] = round(med, 4)
    result["workloads"]["4k_x4_i16"]["check_kernel_alone_note"] = (
        f"{B} stereo_lr_check_device calls; maps {map_bytes / 1e6:.1f} MB, read twice: {2 * map_bytes / med / 1e6:.0f} GB/s of reads")

    device_workload("720p_x16_i8", 720, 1280, 64, 4, 16, 1)

    # CV_32FC1 host images, 4K x 4 pairs
    rows, cols, nd, R, B = 2160, 3840, 256, 5, 4
    rng = nd - 1
    sets = 2
    host = []
    for s in range(sets):
        L, Rt, _ = synth.make_pair(rows, cols, nd, 200 + s)
        host.append((np.stack([L.astype(np.float32)] * B), np.stack([Rt.astype(np.float32)] * B)))
    times = {"off": [], "on": []}
    outs = None
    for i in range(args.warmup + args.reps):
        for mode in (("off", "on") if i % 2 == 0 else ("on", "off")):
            ctx.set_lr_check(MAX_DIFF if mode == "on" else None)
            Ls, Rs = host[i % sets]
            t0 = time.perf_counter()
            dl, dr = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, R, rng, dtype=np.int16)
            t1 = time.perf_counter()
            if i >= args.warmup:
                times[mode].append((t1 - t0) * 1e3)
            if mode == "on":
                outs = (dl, dr)
    ctx.set_lr_check(None)
    rec = summarize(times)
    rec.update(shape=f"{rows}x{cols}", disparities=nd, window=2 * R + 1, pairs=B, elem_bytes=2, input_sets=sets,
               timing="host clock around the synchronous call",
               invalidated_share=round(float(np.mean(np.concatenate([outs[0].ravel(), outs[1].ravel()]) == -(rng + 1))), 4))
    result["workloads"]["4k_x4_f32host"] = rec

    name, limit = gpu_info()
    result["gpu"] = name or torch.cuda.get_device_name(0)
    result["power_limit"] = limit
    print(json.dumps(result))
    ctx.close()


def summarize(times):
    off, on = statistics.median(times["off"]), statistics.median(times["on"])
    return {"median_ms_off": round(off, 4), "median_ms_on": round(on, 4), "diff_ms": round(on - off, 4),
            "diff_pct": round(100.0 * (on - off) / off, 2),
            "spread_ms_off": [round(min(times["off"]), 4), round(max(times["off"]), 4)],
            "spread_ms_on": [round(min(times["on"]), 4), round(max(times["on"]), 4)]}


if __name__ == "__main__":
    main()
