#!/usr/bin/env python
"""Cost of semi-global matching (stereo_ctx_set_sgm): each workload timed with SGM off, over 4 paths and over 8 paths,
alternating call by call in one process, on inputs rotated past the 126 MB L2; then, in a second pass under
torch.profiler, the device time of every SGM kernel and its achieved bytes/s over the bytes the algorithm moves.

    python tools/sgm_timing.py [--cost {ssd,ncc}] [--ncc-scale Q] [--reps N] [--out FILE]
                                                            -> one JSON line (also written to FILE)

Workloads (stereo_disparity_pair_batch_u8_device, P1 = 10, P2 = 120):
  720p_x16_i8    720 x 1280, 64 disparities, 9 x 9, 16 pairs, int8 maps
  1080p_x4_i8    1080 x 1920, 128 disparities, 9 x 9, 4 pairs, int8 maps
  4k_x1_i16      2160 x 3840, 256 disparities, 11 x 11, 1 pair, int16 maps
--cost ncc (SGM of NCC pair calls, stereo_ctx_set_sgm_ncc_scale Q, default 2^15, with P1 = Q / 100 and P2 = Q / 10) times
the same workloads - 8-bit images, sliding cost kernel - and, through stereo_disparity_pair_f32_device, one float workload
whose images are not 8-bit-valued (per-cell cost kernel):
  720p_noisy_f32_i8  720 x 1280, 64 disparities, 9 x 9, 1 pair, noise sigma 10 (synth.noisy_variant), int8 maps
"off" is then the NCC block matcher; each workload also reports the SSD cost kernel's time on the same images (a third
profiled pass), against which the 8-bit NCC cost kernel is compared.
Algorithmic bytes per direction, with cells = rows x cols x Dp (Dp: candidates padded to a multiple of 32):
  sgm_cost_kernel, sgm_ncc_cell_kernel  4 cells written;  sgm_ncc_norm_kernel  16 bytes per pixel written;
  sgm_path_kernel  4 cells of C read plus 4 (first path) or 8 (the others) of S;
  the winner-take-all is folded into the last path (its map writes are not counted).
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
HBM_BYTES_PER_S = 7.7e12
MODES = ("off", "sgm4", "sgm8")
WORKLOADS = [("720p_x16_i8", 720, 1280, 64, 4, 16, 1), ("1080p_x4_i8", 1080, 1920, 128, 4, 4, 1),
             ("4k_x1_i16", 2160, 3840, 256, 5, 1, 2)]
NCC_FLOAT_WORKLOADS = [("720p_noisy_f32_i8", 720, 1280, 64, 4, 1, 1)]
KERNELS = ("sgm_cost_kernel", "sgm_ncc_cell_kernel", "sgm_ncc_norm_kernel", "sgm_path_kernel")


def padded_candidates(cols, R, rng, ncc=False):
    lim = cols - 1 if ncc else cols - 1 + R
    return 32 * ((min(rng, lim) + 1 + 31) // 32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cost", choices=("ssd", "ncc"), default="ssd")
    ap.add_argument("--ncc-scale", type=int, default=1 << 15, help="q of stereo_ctx_set_sgm_ncc_scale (--cost ncc)")
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

    ncc = args.cost == "ncc"
    cost = sb.COST_NCORR if ncc else sb.COST_SSD
    q = args.ncc_scale
    p1, p2 = (q // 100, q // 10) if ncc else (P1, P2)

    def set_mode(mode):
        ctx.set_sgm({"off": None, "sgm4": 4, "sgm8": 8}[mode], p1, p2)

    if ncc:
        ctx.set_sgm_ncc_scale(q)
    result = {"tool": "sgm_timing", "p1": p1, "p2": p2, "reps": args.reps, "hbm_bytes_per_s": HBM_BYTES_PER_S, "workloads": {}}
    if ncc:
        result = {"tool": "sgm_timing", "cost": "ncc", "ncc_scale": q, **{k: v for k, v in result.items() if k != "tool"}}
    for tag, rows, cols, nd, R, B, elem in WORKLOADS + (NCC_FLOAT_WORKLOADS if ncc else []):
        tdt = {1: torch.int8, 2: torch.int16}[elem]
        rng = nd - 1
        f32 = tag in [w[0] for w in NCC_FLOAT_WORKLOADS]
        px = 4 if f32 else 1
        sets = max(2, -(-L2_BYTES // (B * 2 * rows * cols * px)) + 1)
        imgs = []
        for s in range(sets):
            L, Rt, _ = synth.make_pair(rows, cols, nd, 100 + s)
            if f32:
                L, Rt = synth.noisy_variant(L, 200 + s), synth.noisy_variant(Rt, 300 + s)
            imgs.append((torch.from_numpy(np.stack([L] * B)).to(dev), torch.from_numpy(np.stack([Rt] * B)).to(dev)))
        out = torch.empty((2, B, rows, cols), dtype=tdt, device=dev)

        def call(s, c=None):
            c = cost if c is None else c
            dl, dr = imgs[s % sets]
            if f32:
                check(lib.stereo_disparity_pair_f32_device(ctx.handle, c, dl.data_ptr(), cols * 4, dr.data_ptr(), cols * 4, rows, cols, R,
                                                           rng, out[0].data_ptr(), out[1].data_ptr(), cols * elem, elem, sp))
                return
            check(lib.stereo_disparity_pair_batch_u8_device(ctx.handle, c, B, dl.data_ptr(), dr.data_ptr(), cols, rows * cols,
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
        rec.update({f"ratio_{m}_over_off": round(med[m] / med["off"], 2) for m in MODES[1:]})
        dp = padded_candidates(cols, R, rng, ncc)
        cells = rows * cols * dp
        dirs = 2 * B
        rec.update(shape=f"{rows}x{cols}", disparities=nd, range=rng, window=2 * R + 1, pairs=B, elem_bytes=elem, input_sets=sets,
                   padded_candidates=dp, timing="cuda events")
        # per-kernel device time, a separate pass under the profiler
        kernels = {}
        passes = [("sgm4", 4, cost), ("sgm8", 8, cost)] + ([("ssd_sgm8", 8, sb.COST_SSD)] if ncc and not f32 else [])
        for mode, paths, c in passes:
            set_mode(mode[-4:])
            call(0, c)
            torch.cuda.synchronize()
            n = max(3, args.reps // 3)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(n):
                    call(i, c)
                torch.cuda.synchronize()
            tot = {name: [0.0, 0] for name in KERNELS}
            for e in prof.key_averages():
                for name in KERNELS:
                    if name in e.key:
                        tot[name][0] += e.device_time_total
                        tot[name][1] += e.count
            algorithmic = {"sgm_cost_kernel": 4.0 * cells, "sgm_ncc_cell_kernel": 4.0 * cells, "sgm_ncc_norm_kernel": 16.0 * rows * cols,
                           "sgm_path_kernel": (8.0 + 12.0 * (paths - 1)) * cells}
            k = {}
            for name in KERNELS:
                us, cnt = tot[name]
                if cnt == 0:
                    continue
                b = algorithmic[name] * dirs * n
                s = us * 1e-6
                k[name] = {"launches": cnt, "mean_us": round(us / max(cnt, 1), 2), "total_ms_per_call": round(us / 1e3 / n, 4),
                           "algorithmic_gb_per_call": round(b / n / 1e9, 3),
                           "achieved_tb_per_s": round(b / s / 1e12, 3) if s > 0 else None,
                           "share_of_hbm": round(b / s / HBM_BYTES_PER_S, 3) if s > 0 else None}
            kernels[mode] = k
        rec["kernels"] = kernels
        if ncc and not f32:
            ssd_cost = kernels["ssd_sgm8"]["sgm_cost_kernel"]["total_ms_per_call"]
            rec["ncc_over_ssd_cost_kernel"] = round(kernels["sgm8"]["sgm_cost_kernel"]["total_ms_per_call"] / ssd_cost, 2)
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
