#!/usr/bin/env python
"""Cost of the sub-pixel disparity (stereo_ctx_set_subpixel): each workload timed with the block matcher without and with
it, and with SGM over 8 paths (P1 = 10, P2 = 120) without and with it, the four modes alternating call by call in one
process on inputs rotated past the 126 MB L2 (median of --reps calls); then, in a second pass under torch.profiler, the
device time of every kernel of the block-matcher and SGM calls with it on (the sub-pixel pass's pad and refine kernels,
or its apply kernel after the offset-storing last path) and of the SGM call without it.

    python tools/subpixel_timing.py [--reps N] [--out FILE]          -> one JSON line (also written to FILE)

Workloads (stereo_disparity_pair_batch_u8_device, int16 maps, the sizes the project's users run):
  720p_x16       720 x 1280, 64 disparities, 9 x 9, 16 pairs
  1080p_x4       1080 x 1920, 128 disparities, 9 x 9, 4 pairs
  4k_x1          2160 x 3840, 256 disparities, 11 x 11, 1 pair
  4k_x4          2160 x 3840, 256 disparities, 11 x 11, 4 pairs
Call times are CUDA events on the call's stream; the GPU's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import statistics
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from lr_check_timing import gpu_info      # noqa: E402

P1, P2 = 10, 120
L2_BYTES = 126 << 20
MODES = ("bm_off", "bm_on", "sgm8_off", "sgm8_on")
WORKLOADS = [("720p_x16", 720, 1280, 64, 4, 16, 2), ("1080p_x4", 1080, 1920, 128, 4, 4, 2),
             ("4k_x1", 2160, 3840, 256, 5, 1, 2), ("4k_x4", 2160, 3840, 256, 5, 4, 2)]
PASS_KERNELS = ("subpix_pad_kernel", "subpix_bm_kernel", "subpix_apply_kernel")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="timed calls per mode and workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
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

    def set_mode(mode):
        ctx.set_sgm(8 if mode.startswith("sgm8") else None, P1, P2)
        ctx.set_subpixel(mode.endswith("_on"))

    result = {"tool": "subpixel_timing", "p1": P1, "p2": P2, "reps": args.reps, "workloads": {}}
    for tag, rows, cols, nd, R, B, elem in WORKLOADS:
        tdt = {1: torch.int8, 2: torch.int16}[elem]
        rng = nd - 1
        sets = max(2, -(-L2_BYTES // (B * 2 * rows * cols)) + 1)
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

        times = {m: [] for m in MODES}
        for i in range(args.warmup + args.reps):
            for mode in (MODES if i % 2 == 0 else MODES[::-1]):
                set_mode(mode)
                t = timed(lambda: call(i))
                if i >= args.warmup:
                    times[mode].append(t)
        med = {m: statistics.median(t) for m, t in times.items()}
        rec = {f"median_ms_{m}": round(v, 4) for m, v in med.items()}
        rec.update({f"spread_ms_{m}": [round(min(t), 4), round(max(t), 4)] for m, t in times.items()})
        rec["ratio_bm_on_over_off"] = round(med["bm_on"] / med["bm_off"], 4)
        rec["ratio_sgm8_on_over_off"] = round(med["sgm8_on"] / med["sgm8_off"], 4)
        rec.update(shape=f"{rows}x{cols}", disparities=nd, range=rng, window=2 * R + 1, pairs=B, elem_bytes=elem, input_sets=sets,
                   timing="cuda events")
        # per-kernel device time per call, a separate pass under the profiler
        kernels = {}
        for mode in ("bm_off", "bm_on", "sgm8_off", "sgm8_on"):
            set_mode(mode)
            call(0)
            torch.cuda.synchronize()
            n = max(3, args.reps // 3)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(n):
                    call(i)
                torch.cuda.synchronize()
            k = {}
            for e in prof.key_averages():
                if e.device_time_total <= 0 or "Memset" in e.key or "Memcpy" in e.key:
                    continue
                name = e.key.split("(")[0].split("<")[0].replace("void ", "").replace("sb::", "")
                d = k.setdefault(name, {"launches_per_call": 0.0, "ms_per_call": 0.0})
                d["launches_per_call"] += e.count / n
                d["ms_per_call"] += e.device_time_total / 1e3 / n
            kernels[mode] = {name: {a: round(v, 4) for a, v in d.items()} for name, d in sorted(k.items(), key=lambda kv: -kv[1]["ms_per_call"])}
        rec["kernels"] = kernels
        for mode in ("bm_on", "sgm8_on"):
            rec[f"subpixel_kernels_ms_per_call_{mode}"] = round(
                sum(d["ms_per_call"] for name, d in kernels[mode].items() if name in PASS_KERNELS), 4)
        set_mode("bm_off")
        result["workloads"][tag] = rec
        del imgs, out
        torch.cuda.empty_cache()

    name, limit = gpu_info()
    result["gpu"] = name or torch.cuda.get_device_name(0)
    result["power_limit"] = limit
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
