#!/usr/bin/env python
"""Cost of StereoBM's X-Sobel prefilter and texture threshold (stereo_ctx_set_prefilter): each workload timed with both off,
with the prefilter alone (cap 31) and with the prefilter and the texture threshold (T = 500), the three modes alternating
call by call in one process on inputs rotated past the 126 MB L2 (median of --reps calls); then, in a second pass under
torch.profiler, the device time of every kernel of the call with both on, and the achieved bytes/s of the two new kernels
against 7.7 TB/s.

    python tools/prefilter_timing.py [--reps N] [--out FILE]          -> one JSON line (also written to FILE)

Workloads (stereo_disparity_pair_batch_u8_device unless noted):
  720p_x16_i8     720 x 1280, 64 disparities, 9 x 9, 16 pairs, int8 maps
  1080p_x4_i8     1080 x 1920, 128 disparities, 9 x 9, 4 pairs, int8 maps
  4k_x1_i16       2160 x 3840, 256 disparities, 11 x 11, 1 pair, int16 maps
  4k_x4_i16       the same, 4 pairs
  4k_x4_f32_dev   the same 4 pairs as noisy CV_32FC1 images, 4 stereo_disparity_pair_f32_device calls
Bytes of the new kernels: prefilter_kernel reads each image once (1 or 4 bytes a pixel; its three-row stencil re-reads from
L1 / L2) and writes 1 byte a pixel; texture_kernel reads each map's prefiltered reference once (1 byte a pixel) and writes
only the rejected pixels (not counted).  Call times are CUDA events on the call's stream; the GPU's name and power limit are
read in the same run."""
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

CAP, TEXTURE = 31, 500
HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126 << 20
MODES = ("off", "prefilter", "prefilter_texture")
WORKLOADS = [("720p_x16_i8", 720, 1280, 64, 4, 16, 1, False), ("1080p_x4_i8", 1080, 1920, 128, 4, 4, 1, False),
             ("4k_x1_i16", 2160, 3840, 256, 5, 1, 2, False), ("4k_x4_i16", 2160, 3840, 256, 5, 4, 2, False),
             ("4k_x4_f32_dev", 2160, 3840, 256, 5, 4, 2, True)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30, help="timed calls per mode and workload")
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
        ctx.set_prefilter(CAP if mode != "off" else None, TEXTURE if mode == "prefilter_texture" else 0)

    result = {"tool": "prefilter_timing", "cap": CAP, "texture_threshold": TEXTURE, "reps": args.reps, "workloads": {}}
    for tag, rows, cols, nd, R, B, elem, f32 in WORKLOADS:
        tdt = {1: torch.int8, 2: torch.int16}[elem]
        rng = nd - 1
        px = 4 if f32 else 1
        sets = max(2, -(-L2_BYTES // (B * 2 * rows * cols * px)) + 1)
        imgs = []
        for s in range(sets):
            L, Rt, _ = synth.make_pair(rows, cols, nd, 100 + s)
            if f32:
                Ls = np.stack([synth.noisy_variant(L, 10 * s + k) for k in range(B)])
                Rs = np.stack([synth.noisy_variant(Rt, 10 * s + k + 5) for k in range(B)])
            else:
                Ls, Rs = np.stack([L] * B), np.stack([Rt] * B)
            imgs.append((torch.from_numpy(Ls).to(dev), torch.from_numpy(Rs).to(dev)))
        out = torch.empty((2, B, rows, cols), dtype=tdt, device=dev)

        def call(s):
            dl, dr = imgs[s % sets]
            if f32:
                for k in range(B):
                    check(lib.stereo_disparity_pair_f32_device(ctx.handle, sb.COST_SSD, dl[k].data_ptr(), cols * 4, dr[k].data_ptr(),
                                                               cols * 4, rows, cols, R, rng, out[0, k].data_ptr(), out[1, k].data_ptr(),
                                                               cols * elem, elem, sp))
                return
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
        rec["added_pct_prefilter"] = round(100 * (med["prefilter"] / med["off"] - 1), 2)
        rec["added_pct_prefilter_texture"] = round(100 * (med["prefilter_texture"] / med["off"] - 1), 2)
        rec.update(shape=f"{rows}x{cols}", disparities=nd, range=rng, window=2 * R + 1, pairs=B, elem_bytes=elem,
                   images="noisy CV_32FC1, pair_f32_device" if f32 else "u8, pair_batch_u8_device", input_sets=sets, timing="cuda events")
        # per-kernel device time per call, a separate pass under the profiler
        set_mode("prefilter_texture")
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
        rec["kernels"] = {name: {a: round(v, 4) for a, v in d.items()} for name, d in sorted(k.items(), key=lambda kv: -kv[1]["ms_per_call"])}
        pix = rows * cols * B
        for kname, nbytes in (("prefilter_kernel", 2 * pix * (px + 1)), ("texture_kernel", 2 * pix)):
            ms = k.get(kname, {}).get("ms_per_call", 0.0)
            if ms > 0:
                rec[f"{kname}_gbps"] = round(nbytes / (ms * 1e-3) / 1e9, 1)
                rec[f"{kname}_hbm_fraction"] = round(nbytes / (ms * 1e-3) / HBM_BYTES_PER_S, 3)
        set_mode("off")
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
