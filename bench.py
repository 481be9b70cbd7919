#!/usr/bin/env python
"""bench.py — disparity Mpix x disparities / s of the ps2 stereo block matcher on B200.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU implementation, host cores
    python bench.py --dump-outputs DIR ...    # also the last timed step's disparity maps as DIR/*.npy, to compare two builds

A step = one pass of the hot path over one batch of synthetic stereo pairs (both directions per
pair, like the reference's disparitySSDPair, main.cpp:21-48).  Workload at every N: per GPU a batch
of B = 4 synthetic 3840x2160 pairs, 256 disparities, 11x11 window, SSD (BASELINE config 4's shape and
the config the north-star target is quoted on), pairs sharded by rank (weak scaling); for N > 1 every
rank's disparity maps are gathered on every rank inside the timed region (BASELINE config 5's "sharded
by pair ... with ... gather"): by default with copy-engine pushes over NVLink into peer-mapped buffers
(--gather p2p; they overlap the next step's kernels, which an SM-resident collective cannot because the
hot kernel is persistent and fills every SM), or with an NCCL all_gather (--gather nccl).

`value`   : whole-job Mpix x disp / s with inputs resident in HBM, one CUDA event pair on the launching stream
            around all timed steps (joined with the copy-engine streams), inputs rotating over more sets
            than the L2 holds, max over ranks.
`e2e`     : the same metric through the reference-facing C-ABI call with HOST float32 (CV_32FC1)
            buffers — H2D and D2H copies inside the timed region, wall clock, max over ranks.  One
            stereo_disparity_pair_batch_f32_host call per step; `per_pair_calls_value` is the same work as
            separate synchronous stereo_disparity_pair_f32_host calls, `u8_host_api_value` the uint8 entry.
`roofline`: the hot kernel (fast_ssd_kernel) against the FP32/INT32 issue roofline of SURVEY.md §8d
            (8 algorithmic lane-ops per pixel x disparity; peak = SMs x 128 lanes x max SM clock), plus
            the HBM view (algorithmic bytes / kernel time vs the measured copy bandwidth).
`cpu_baseline`: the reference's own serial::disparitySSD / serial::disparityNCorr (compiled in place into
            oracle/_ref) on a bounded sample of the same workload on this box's host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "disparity Mpix x disparities/s"
UNIT = "Mpix*disp/s"
OPS_PER_UNIT = {"ssd": 8, "ncc": 9}          # SURVEY.md §8d algorithmic lane-ops per pixel x disparity
# Fused pair launches (SURVEY.md §8 f2) compute ONE cost volume for both maps of a pair: of the 8 SSD ops per pixel x
# disparity, the 6 that build the window sum (sub, mul, 2 vertical adds, 2 horizontal adds) are shared by the two
# directions' units and only the 2 winner-take-all ops are per unit: (6 + 2 * 2) / 2 = 5 lane-ops per unit.
# NCC: the 5 window-sum ops (mul, 2 vertical adds, 2 horizontal adds) are shared, the 2 normalising multiplies and the 2
# winner-take-all ops are per unit: (5 + 2 * 4) / 2 = 6.5.
OPS_PER_UNIT_FUSED = {"ssd": 5, "ncc": 6.5}

WORKLOADS = {
    # name: rows, cols, n_disp, window_rad, seed
    "4k_d256_w11": dict(rows=2160, cols=3840, ndisp=256, R=5, seed=1002),
    "1080p_d128_w9": dict(rows=1080, cols=1920, ndisp=128, R=4, seed=1001),
    "720p_d64_w9": dict(rows=720, cols=1280, ndisp=64, R=4, seed=2000),
    # the reference's own problems (config/ps2.yaml:19-41) at the logged image sizes (output/ps2_cpu.log:6,12,49);
    # synthetic stand-ins of the same shape (the bundled pixels are Git-LFS stubs)
    "ps2_pair0_128_d4_w13": dict(rows=128, cols=128, ndisp=4, R=6, seed=10),
    "ps2_pair1_511x640_d96_w15": dict(rows=511, cols=640, ndisp=96, R=7, seed=11),
    "ps2_pair2_529x640_d81_w15": dict(rows=529, cols=640, ndisp=81, R=7, seed=12),
}


def ncu_traffic(workload: str, cost: str, jobs_per_launch: float):
    """DRAM bytes (read + write) of ONE hot-kernel launch from the committed `ncu --set full` capture
    (profiles/roofline_traffic.json, written from the .ncu-rep by tools/ncu_summary.py); None when no
    capture of this workload / cost / directions-per-launch exists."""
    p = ROOT / "profiles" / "roofline_traffic.json"
    if not p.exists():
        return None
    for e in json.loads(p.read_text()).get("captures", []):
        if e["workload"] == workload and e["cost"] == cost and abs(e["directions_per_launch"] - jobs_per_launch) < 1e-9:
            return int(e["dram_bytes_read"] + e["dram_bytes_write"])
    return None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=float(d["hbm_gbs"]), sm_max_mhz=float(d.get("sm_max_mhz", 1965.0)), source="measured")
    return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, source="fallback")


# ---------------------------------------------------------------------------------------------------
# clocks during the timed region (NVML)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.005)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_cpus(index: int):
    """Multi-rank runs: keep this rank's threads (and, by first touch, its pinned host buffers) on the CPUs NVML
    reports as local to its GPU.  Returns the number of CPUs bound to, or None when nothing was changed."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 1) + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        avail = os.sched_getaffinity(0)
        cpus &= avail
        if cpus and cpus != avail:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
        # every GPU reports the same CPUs (one NUMA node, a VM): give each rank its own slice so that the ranks' host
        # threads do not migrate over each other
        world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        local = int(os.environ.get("LOCAL_RANK", "0"))
        order = sorted(avail)
        per = len(order) // max(world, 1)
        if world > 1 and per >= 2:
            mine = set(order[local * per:(local + 1) * per])
            os.sched_setaffinity(0, mine)
            return len(mine)
    except Exception:
        pass
    return None


# ---------------------------------------------------------------------------------------------------
# the reference's CPU implementation on host cores (bounded sample)
# ---------------------------------------------------------------------------------------------------
def cpu_reference_sample(wl, rows_per_thread: int, threads: int, cost: str = "ssd"):
    """Times the reference's serial::disparitySSD / serial::disparityNCorr (oracle/_ref; falls back to the C port
    when the compiled reference is absent) on `threads` disjoint full-width row bands of the workload's
    left->right problem.  Returns (Mpix*disp/s, seconds, description dict)."""
    import oracle
    from introtocomputervision_b200 import synth

    R, nd = wl["R"], wl["ndisp"]
    band = max(1, rows_per_thread)
    L, Rt, _ = synth.make_pair(band * threads, wl["cols"], nd, wl["seed"])
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    have = oracle.have_ref() if cost == "ssd" else oracle.have_ref_ncc()
    kind = "reference" if have else "port"
    oracle.set_num_threads(1)
    fn = {("ssd", "reference"): oracle.ref_ssd, ("ssd", "port"): oracle.ssd,
          ("ncc", "reference"): oracle.ref_ncorr, ("ncc", "port"): oracle.ncorr}[(cost, kind)]

    def work(i):
        a = np.ascontiguousarray(Lf[i * band:(i + 1) * band])
        b = np.ascontiguousarray(Rf[i * band:(i + 1) * band])
        fn(a, b, R, -(nd - 1), 0)          # disparitySSDPair / disparityNCorrPair (main.cpp:21-78): left-referenced map ...
        fn(b, a, R, 0, nd - 1)             # ... then the images swapped over [0, +range]

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(work, range(threads)))
    dt = time.perf_counter() - t0
    units = 2 * threads * band * wl["cols"] * nd      # every row of every band is computed, both directions
    what = {("ssd", "reference"): "reference serial::disparitySSD compiled -O2 from /root/reference (oracle/_ref)",
            ("ssd", "port"): "C port of serial::disparitySSD (oracle/stereo_oracle.c)",
            ("ncc", "reference"): "reference serial::disparityNCorr compiled -O2 from /root/reference (oracle/_ref) over the "
                                  "shim's direct-sum cv::matchTemplate (OpenCV itself is not installed in C++)",
            ("ncc", "port"): "C port of serial::disparityNCorr (oracle/stereo_oracle.c)"}[(cost, kind)]
    desc = {"kind": kind, "cores": threads,
            "sample": f"{threads} threads x {band}-row full-width bands ({wl['cols']} cols, {nd} disparities, "
                      f"{2 * R + 1}x{2 * R + 1} window), both directions of the pair, {cost.upper()}, " + what}
    return units / dt / 1e6, dt, desc


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    for _ in range(args.warmup):
        cpu_reference_sample(wl, 1, threads, args.cost)
    vals, times = [], []
    for _ in range(args.steps):
        v, dt, desc = cpu_reference_sample(wl, args.ref_rows, threads, args.cost)
        vals.append(v), times.append(dt)
    total_units = sum(v * t for v, t in zip(vals, times))
    value = total_units / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * sum(times) / len(times), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32->int32" if args.cost == "ssd" else "f32 (f64 window energies)", "data": "synthetic",
        "config": {"workload": args.workload + f"_{args.cost}_pair", **{k: wl[k] for k in ("rows", "cols", "ndisp")},
                   "window": 2 * wl["R"] + 1, "directions": 2, "sample_rows_per_thread": args.ref_rows},
        "cpu_baseline": {**desc, "value": round(value, 3), "unit": UNIT},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def oracle_band_check(L, Rt, R, nd, cost, got_l, got_r, r0, n):
    """Outside the timed region: rows [r0, r0 + n) of both maps of one pair against the oracle (oracle/ is the checker here,
    never the thing measured).  The oracle runs on the slab of image rows the band depends on - window halo R plus the row
    the SSD flat-index wrap reads (SURVEY.md A.1) - and its interior rows are compared.  got_l / got_r: numpy maps of the
    whole image.  Returns a small report dict."""
    import oracle
    rows = L.shape[0]
    lo, hi = max(0, r0 - R - 1), min(rows, r0 + n + R + 1)
    Ls, Rs = np.ascontiguousarray(L[lo:hi]).astype(np.float32), np.ascontiguousarray(Rt[lo:hi]).astype(np.float32)
    # slab borders that are not image borders see different padding: compare only rows whose halo lies inside the slab
    a = r0 - lo if lo > 0 else 0
    b = a + n
    rep = {"rows": [r0, r0 + n], "oracle": "oracle.ssd_fast" if cost == "ssd" else "oracle.ncorr_fast"}
    if cost == "ssd":
        ref_l = oracle.ssd_fast(Ls, Rs, R, -(nd - 1), 0)[a:b]
        ref_r = oracle.ssd_fast(Rs, Ls, R, 0, nd - 1)[a:b]
        bad = int(np.count_nonzero(ref_l.astype(np.int64) != got_l[r0:r0 + n].astype(np.int64))
                  + np.count_nonzero(ref_r.astype(np.int64) != got_r[r0:r0 + n].astype(np.int64)))
        rep.update(pixels=int(2 * ref_l.size), mismatches=bad, ok=bad == 0, rule="bit-exact")
    else:
        ref_l = oracle.ncorr_fast(Ls, Rs, R, -(nd - 1), 0)[a:b]
        ref_r = oracle.ncorr_fast(Rs, Ls, R, 0, nd - 1)[a:b]
        agree = float((np.count_nonzero(ref_l == got_l[r0:r0 + n]) + np.count_nonzero(ref_r == got_r[r0:r0 + n])) / (2 * ref_l.size))
        rep.update(pixels=int(2 * ref_l.size), agreement=round(agree, 6), ok=agree >= 0.999, rule=">= 99.9 % equal disparities")
    return rep


DUMP_BYTES = 64_000_000      # --dump-outputs: all files of all ranks together


def dump_maps(out_dir, maps, budget, suffix=""):
    """--dump-outputs: every tensor of `maps` ({name: disparity maps [..., rows, cols]}, one image shape) as float32
    `out_dir/<name><suffix>.npy`.  Maps larger than `budget` bytes together keep one fixed, seeded sample of pixel positions
    (the same for every map, increasing); its flat indices (row * cols + col) go to `sample_index<suffix>.npy` as float64.
    Returns a description for the JSON line."""
    import torch
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rows, cols = next(iter(maps.values())).shape[-2:]
    pix = rows * cols
    n_maps = sum(t.numel() // pix for t in maps.values())
    idx = None
    files = []
    if n_maps * pix * 4 > budget:
        k = (budget - 1024) // (n_maps * 4 + 8)          # 1024: the .npy headers; 8: the float64 index of a sampled pixel
        idx = np.sort(np.random.default_rng(0).choice(pix, k, replace=False))
        np.save(out_dir / f"sample_index{suffix}.npy", idx.astype(np.float64))
        files.append(f"sample_index{suffix}.npy")
    for name, t in maps.items():
        if idx is None:
            a = t.to(torch.float32).cpu().numpy()
        else:
            a = t.reshape(-1, pix)[:, torch.from_numpy(idx).to(t.device)].to(torch.float32).cpu().numpy().reshape(*t.shape[:-2], -1)
        np.save(out_dir / f"{name}{suffix}.npy", a)
        files.append(f"{name}{suffix}.npy")
    rep = {"dir": str(out_dir), "files": files, "pixels_per_map": pix if idx is None else int(idx.size), "of_pixels": pix}
    if idx is not None:
        rep["sample_index"] = "flat pixel index row * cols + col, stored as float64 (exact below 2^53)"
    return rep


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    import introtocomputervision_b200 as sb
    from introtocomputervision_b200 import _capi, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bound_cpus = bind_to_gpu_cpus(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _capi.lib()
    ctx = sb.Context(local)
    if args.pipe_bands:
        ctx.set_pipe_bands(args.pipe_bands)
    cost = sb.COST_SSD if args.cost == "ssd" else sb.COST_NCORR
    rows, cols, nd, R = wl["rows"], wl["cols"], wl["ndisp"], wl["R"]
    if args.mode == "bands":
        return run_bands(args, wl, lib, ctx, cost, dev, rank, world, local)
    B = args.pairs
    elem_dtype, elem = (torch.int8, 1) if nd <= 128 else (torch.int16, 2)
    from introtocomputervision_b200 import sharding

    # synthetic pairs of this rank (pair-sharded batch: rank r owns pairs r*B .. r*B+B-1).  The inputs rotate
    # over S sets whose total size exceeds the L2, so no step finds its images cached from the step before
    # (set 0 is generated, the others are its rows rolled: throughput is data-independent, only residency matters).
    Ls, Rs = [], []
    for i in range(B):
        L, Rt, _ = synth.make_pair(rows, cols, nd, wl["seed"] + rank * B + i)
        Ls.append(L), Rs.append(Rt)
    h_left = torch.from_numpy(np.stack(Ls))
    h_right = torch.from_numpy(np.stack(Rs))
    props = torch.cuda.get_device_properties(dev)
    l2_bytes = int(getattr(props, "L2_cache_size", 126 << 20))
    set_bytes = 2 * B * rows * cols
    S = max(2, -(-int(1.25 * l2_bytes) // set_bytes) + 1)
    d_left = torch.stack([torch.roll(h_left, 17 * s_, dims=1) for s_ in range(S)]).to(dev)     # S x B x rows x cols
    d_right = torch.stack([torch.roll(h_right, 17 * s_, dims=1) for s_ in range(S)]).to(dev)
    d_out = torch.empty((2, 2, B, rows, cols), dtype=elem_dtype, device=dev)                    # [parity][direction][pair]
    map_bytes = 2 * B * rows * cols * elem                                                      # one rank's maps of one step
    stream = torch.cuda.Stream(device=dev)              # a real (non-default) stream: the library enqueues on it
    torch.cuda.set_stream(stream)
    sp = C.c_void_p(stream.cuda_stream)
    units_rank = B * 2 * rows * cols * nd
    nwarm = max(3, args.warmup)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class Gather:
        """The exchange step of a pair-sharded batch.  root: every rank's maps pushed into rank 0's buffer (the consumer) by the
        copy engines over NVLink; all: into every rank's buffer; nccl: all_gather_into_tensor inside the step; none: N = 1."""

        def __init__(self, kind):
            self.kind, self.note, self.pg, self.gathered, self.tickets = kind, "", None, None, {}
            if kind in ("root", "all"):
                # the buffer: [parity][rank][direction][pair][rows][cols]; filled by copy-engine pushes
                try:
                    self.pg = sharding.PeerGather(ctx, 2 * world * map_bytes)
                except sharding.PeerGatherUnavailable as e:       # raised on every rank together
                    self.kind, self.note = "nccl", f" (peer buffers unavailable: {e})"
            if self.kind == "nccl":
                self.gathered = torch.empty((world, 2, B, rows, cols), dtype=elem_dtype, device=dev)
            self.to = [0] if self.kind == "root" else None
            # bytes every rank sends / the busiest rank receives per step over NVLink
            self.tx = {"root": map_bytes if rank != 0 else 0, "all": (world - 1) * map_bytes, "nccl": (world - 1) * map_bytes}.get(self.kind, 0)
            self.rx_max = {"root": (world - 1) * map_bytes, "all": (world - 1) * map_bytes, "nccl": (world - 1) * map_bytes}.get(self.kind, 0)

        def before(self, k):
            if self.pg is not None and k - 2 in self.tickets:
                self.pg.wait(self.tickets.pop(k - 2), stream.cuda_stream)       # the pushes that read d_out[par] two steps ago

        def after(self, k, par):
            if self.pg is not None:
                self.pg.push((par * world + rank) * map_bytes, d_out[par].data_ptr(), map_bytes, stream.cuda_stream, to=self.to)
                self.tickets[k] = self.pg.mark()
            elif self.gathered is not None:
                dist.all_gather_into_tensor(self.gathered.view(torch.uint8).view(-1), d_out[par].view(torch.uint8).view(-1))   # bytes: NCCL has no int16

        def join(self):
            if self.pg is not None:
                for k in sorted(self.tickets):
                    self.pg.wait(self.tickets.pop(k), stream.cuda_stream)

        def holds_all(self):
            return self.pg is not None and (self.kind == "all" or rank == 0)

        def close(self):
            if self.pg is not None:
                self.join()
                torch.cuda.synchronize()
                self.pg.close()
                self.pg = None

    def step_device(G, k):
        par, s_ = k & 1, k % S
        G.before(k)
        rc = lib.stereo_disparity_pair_batch_u8_device(
            ctx.handle, cost, B, d_left[s_].data_ptr(), d_right[s_].data_ptr(), cols, rows * cols, rows, cols, R, nd - 1,
            d_out[par, 0].data_ptr(), d_out[par, 1].data_ptr(), cols * elem, rows * cols * elem, elem, sp)
        if rc != 0:
            raise RuntimeError(_capi.last_error())
        G.after(k, par)

    def timed_pairs(G, steps):
        """nwarm untimed steps, then `steps` steps inside one event pair (joined with the copy-engine streams); ms = max over ranks."""
        for k in range(nwarm):
            step_device(G, k)
        G.join()
        barrier()
        if G.holds_all():      # the gather delivers: this rank's buffer holds the last warm-up step's maps of this rank
            par = (nwarm - 1) & 1
            got = G.pg.local_bytes(dev)[(par * world + rank) * map_bytes:(par * world + rank + 1) * map_bytes]
            assert torch.equal(got, d_out[par].view(torch.uint8).view(-1)), "peer gather: own slot differs from the computed maps"
        n_launch = 0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(steps):
            step_device(G, nwarm + k)
            n_launch += ctx.last_launches
        G.join()                                         # the timed region ends when every push has landed
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if G.pg is not None:      # cross-rank check after the barrier: every slot of the last step equals what that rank computed
            par = (nwarm + steps - 1) & 1
            mine_sum = d_out[par].view(torch.uint8).view(-1).to(torch.int64).sum().reshape(1)
            all_sums = torch.empty(world, dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(all_sums, mine_sum)
            if G.holds_all():
                sums = G.pg.local_bytes(dev)[par * world * map_bytes:(par + 1) * world * map_bytes].view(world, -1).to(torch.int64).sum(dim=1)
                assert torch.equal(sums, all_sums), f"peer gather ({G.kind}): slots {sums.tolist()} != ranks' maps {all_sums.tolist()} (parity {par})"
            barrier()             # nobody pushes the next step into a slot the consumer is still checking
        return float(t.item()), n_launch

    G = Gather(args.gather if world > 1 else "none")
    gather, gather_note, pg = G.kind, G.note, G.pg
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, launches = timed_pairs(G, args.steps)
    clocks = sampler.stop()
    dump = None
    if args.dump_outputs:     # before any later step reuses d_out
        last = nwarm + args.steps - 1
        dump = dump_maps(args.dump_outputs, {"disparity_left": d_out[last & 1, 0], "disparity_right": d_out[last & 1, 1]},
                         DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")
        dump.update(step=last, input_set=last % S, input_roll_rows=17 * (last % S))
    hot_ms, hot_n = 0.0, 0
    # hot-kernel time of the last step (events recorded by the library on the same stream)
    ms, nmeas = ctx.last_hot_kernel_ms()
    hot_jobs = ctx.last_hot_jobs
    fused = ctx.last_fused_pairs > 0
    if nmeas > 0:
        hot_ms, hot_n = ms, nmeas
    # the same batch with one cost volume per direction (untimed: one step, for the roofline of the unfused kernel)
    unfused = None
    if fused:
        ctx.set_fuse_pairs(False)
        G.join()
        step_device(G, nwarm + args.steps + (nwarm + args.steps) % 2)
        G.join()
        torch.cuda.synchronize()
        ms_u, n_u = ctx.last_hot_kernel_ms()
        if n_u > 0:
            unfused = (ms_u, n_u, ctx.last_hot_jobs)
        ctx.set_fuse_pairs(True)
    value = world * units_rank * args.steps / (dev_ms * 1e-3) / 1e6

    def join_pushes():
        G.join()

    # the other exchange variants, a few steps each (multi-GPU runs only): sub-lines of the same JSON line
    gather_sub = {}
    if world > 1 and not args.no_suite:
        G.join()
        barrier()
        for kind in ("root", "all", "nccl"):
            if kind == G.kind:
                continue
            G2 = Gather(kind)
            ms2, _ = timed_pairs(G2, max(3, min(args.steps, 5)))
            gather_sub[kind if G2.kind == kind else f"{kind}->nccl"] = {
                "value": round(world * units_rank * max(3, min(args.steps, 5)) / (ms2 * 1e-3) / 1e6, 1), "unit": UNIT,
                "ms_per_step": round(ms2 / max(3, min(args.steps, 5)), 4),
                "nvlink_tx_bytes_per_rank_per_step": map_bytes if G2.kind == "root" else (world - 1) * map_bytes,
                "nvlink_rx_bytes_busiest_rank_per_step": G2.rx_max}
            G2.close()
            barrier()

    # ---- e2e: reference-facing host call, float32 (CV_32FC1) host buffers, copies inside the timed region
    hf_left = h_left.to(torch.float32).pin_memory()
    hf_right = h_right.to(torch.float32).pin_memory()
    h_dl = torch.empty((B, rows, cols), dtype=elem_dtype).pin_memory()
    h_dr = torch.empty((B, rows, cols), dtype=elem_dtype).pin_memory()

    def step_host():
        # ONE call of the public host API per step: the step's batch of pairs as CV_32FC1 host images in, both
        # disparity maps of every pair out (a batch of the reference's disparitySSDPair calls, main.cpp:21-48)
        rc = lib.stereo_disparity_pair_batch_f32_host(
            ctx.handle, cost, B, hf_left.data_ptr(), hf_right.data_ptr(), cols * 4, rows * cols * 4, rows, cols, R, nd - 1,
            h_dl.data_ptr(), h_dr.data_ptr(), cols * elem, rows * cols * elem, elem)
        if rc != 0:
            raise RuntimeError(_capi.last_error())

    def step_host_per_pair():
        # the same work as B separate synchronous pair calls (the reference's calling pattern, one pair at a time)
        for i in range(B):
            rc = lib.stereo_disparity_pair_f32_host(
                ctx.handle, cost, hf_left[i].data_ptr(), cols * 4, hf_right[i].data_ptr(), cols * 4, rows, cols, R, nd - 1,
                h_dl[i].data_ptr(), h_dr[i].data_ptr(), cols * elem, elem)
            if rc != 0:
                raise RuntimeError(_capi.last_error())

    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = world * units_rank * e2e_steps / e2e_s / 1e6
    e2e_launches = ctx.last_launches * e2e_steps

    def timed_host(fn):
        fn(), fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fn()
        barrier()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return world * units_rank * e2e_steps / float(tt.item()) / 1e6

    e2e_pp_value = timed_host(step_host_per_pair)
    # the same batch call with host-side packing switched the other way (the default packs from 8 host threads up)
    host_threads = ctx.host_threads
    packing = host_threads >= 8
    alt_threads = -1 if packing else max(2, host_threads)      # forced on with the threads this rank would get
    ctx.set_host_threads(alt_threads)
    e2e_alt_value = timed_host(step_host)
    ctx.set_host_threads(0)

    # u8 host entry (same computation for callers that hold 8-bit images)
    hu_l, hu_r = h_left.pin_memory(), h_right.pin_memory()

    def step_host_u8():
        rc = lib.stereo_disparity_pair_batch_u8_host(
            ctx.handle, cost, B, hu_l.data_ptr(), hu_r.data_ptr(), cols, rows * cols, rows, cols, R, nd - 1,
            h_dl.data_ptr(), h_dr.data_ptr(), cols * elem, rows * cols * elem, elem)
        if rc != 0:
            raise RuntimeError(_capi.last_error())

    e2e8_value = timed_host(step_host_u8)

    # self-check outside every timed region: the host API's maps equal the device path's on the same pairs (set 0)
    step_host()
    if pg is not None:
        join_pushes()
    step_device(G, 2 * S)               # even step number: parity 0, input set 0 (the un-rolled images)
    if pg is not None:
        join_pushes()
    barrier()                            # every rank's pushes of that step have landed in the consumer's buffer
    assert torch.equal(d_out[0, 0].cpu(), h_dl) and torch.equal(d_out[0, 1].cpu(), h_dr), "host and device entry points disagree"

    # parity check outside every timed region (rank 0): a 64-row band of the step's maps - and, in multi-GPU runs, of a
    # PEER rank's maps as they arrived in this rank's gather buffer - against the oracle
    parity = None
    if rank == 0 and not args.no_parity:
        r0 = max(0, min(rows - 64, (rows // 2) // 8 * 8 + 3))
        nrow = min(64, rows)
        mine_l, mine_r = d_out[0, 0, 0].cpu().numpy(), d_out[0, 1, 0].cpu().numpy()
        parity = {"own_pair0": oracle_band_check(Ls[0], Rs[0], R, nd, args.cost, mine_l, mine_r, r0, nrow)}
        if pg is not None and world > 1:
            peer = 1
            slot = pg.local_bytes(dev)[(0 * world + peer) * map_bytes:(0 * world + peer + 1) * map_bytes]      # parity 0, rank `peer`
            maps = slot.view(elem_dtype).view(2, B, rows, cols)
            pl, pr_ = maps[0, B - 1].cpu().numpy(), maps[1, B - 1].cpu().numpy()
            PL, PR, _ = synth.make_pair(rows, cols, nd, wl["seed"] + peer * B + (B - 1))
            parity[f"rank{peer}_pair{B - 1}_from_gather_buffer"] = oracle_band_check(PL, PR, R, nd, args.cost, pl, pr_, r0, nrow)
        parity["ok"] = all(v["ok"] for v in parity.values())

    # BASELINE config 4 next to the pair-sharded line (multi-GPU runs): the same 4K pair cut into row bands, strong scaling
    bands_sub = None
    if world > 1 and not args.no_suite:
        G.join()
        barrier()
        torch.cuda.set_stream(torch.cuda.default_stream(dev))
        bands_sub = bands_line(args, wl, lib, ctx, cost, dev, rank, world, local, max(5, min(args.steps, 20)), "root", use_graph=not args.no_graph)
        torch.cuda.set_stream(stream)
        barrier()

    if rank == 0:
        peaks = measured_peaks()
        props = torch.cuda.get_device_properties(dev)
        sms = props.multi_processor_count
        peak_lane_ops = sms * 128 * peaks["sm_max_mhz"] * 1e6               # lane-ops / s
        roof = None
        if hot_n > 0:
            jobs_per_launch = hot_jobs / hot_n                              # directions one hot launch covers
            units_hot = hot_jobs * rows * cols * nd
            t_hot = hot_ms * 1e-3
            opu = OPS_PER_UNIT_FUSED[args.cost] if fused else OPS_PER_UNIT[args.cost]
            achieved = opu * units_hot / t_hot
            b_in, b_out = 1, elem
            alg_bytes = int(jobs_per_launch * rows * cols * (2 * b_in + b_out))   # per launch (SURVEY.md §8d)
            roof = {
                "bound": "alu", "kernel": (f"fast_cost_kernel<R={R},K={16 if (nd <= 64 or R >= 6 or args.cost == 'ncc') else 20},NW=8,{args.cost.upper()},fused pair>" if fused
                                           else f"fast_cost_kernel<R={R},K={20 if R >= 6 else 24},NW=8,{args.cost.upper()}>"),
                "achieved": round(achieved / 1e12, 3), "peak": round(peak_lane_ops / 1e12, 3), "unit": "Tlane-op/s",
                "frac": round(achieved / peak_lane_ops, 4),
                "ops_per_unit": opu, "units_per_launch": int(jobs_per_launch * rows * cols * nd),
                "directions_per_launch": jobs_per_launch,
                "launch_ms": round(hot_ms / hot_n, 4), "launches_timed": hot_n,
                "peak_def": f"{sms} SMs x 128 lanes x {peaks['sm_max_mhz']:.0f} MHz ({peaks['source']} sm_max_mhz)",
                "traffic": ncu_traffic(args.workload, args.cost, jobs_per_launch),
                "hbm": {"achieved": round(alg_bytes / (hot_ms / hot_n * 1e-3) / 1e9, 2), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": round(alg_bytes / (hot_ms / hot_n * 1e-3) / 1e9 / peaks["hbm_gbs"], 5),
                        "algorithmic_bytes_per_launch": alg_bytes, "of": peaks["source"]},
            }
            if fused:
                ceiling = peak_lane_ops / OPS_PER_UNIT[args.cost]                  # SURVEY.md 8d: pixel x disparity / s at 8 (9) ops per unit
                roof["note"] = ("fused pair launch: one cost volume serves both maps of a pair, so a unit costs "
                                f"{OPS_PER_UNIT_FUSED[args.cost]} algorithmic lane-ops instead of SURVEY.md 8d's {OPS_PER_UNIT[args.cost]} "
                                "(the window-sum ops are shared by the two maps, the per-map ops are not); frac is quoted on the smaller figure")
                roof["vs_survey_8d_ceiling"] = {
                    "ceiling": round(ceiling / 1e6, 1), "unit": UNIT,
                    "def": "peak lane-ops / 8 ops per unit, the ceiling the north-star '>= 70 % of roofline' is stated against",
                    "hot_kernel": round(units_hot / t_hot / ceiling, 4),
                    "whole_step": round(value * 1e6 / world / ceiling, 4)}
                if args.cost == "ssd":
                    # measured ceiling of the kernel's own instruction mix (tools/microbench/mix.cu, profiles/r2w_microbench_mix.txt):
                    # with every operand in registers and no memory, barriers or row code, the mix issues 0.716 inst/clk/SMSP at the
                    # kernel's occupancy - the register file delivers ~1.65 operand reads per clock per SMSP to three-operand
                    # integer instructions - i.e. 40.2 clocks per warp pixel step (256 units)
                    mix_units_per_s = 256 / 40.2 * sms * 4 * peaks["sm_max_mhz"] * 1e6
                    roof["instruction_mix_ceiling"] = {
                        "inst_per_clk_per_smsp": 0.716, "clk_per_warp_pixel_step": 40.2, "value": round(mix_units_per_s / 1e6, 1), "unit": UNIT,
                        "hot_kernel_frac": round(units_hot / t_hot / mix_units_per_s, 4),
                        "def": "core mix of one pixel step (6 IDP.2A, 4 IADD3, 8 IMAD, 4 minima, REDUX, SHFL, 1.5 LDS.128 = 28.75 SASS instructions) "
                               "issued from registers at 2 warps per scheduler on this GPU model; the kernel executes 37.5 instructions per step at 0.69 inst/clk",
                        "source": "profiles/r2w_microbench_mix.txt"}
                if unfused is not None:
                    ms_u, n_u, jobs_u = unfused
                    ach_u = OPS_PER_UNIT[args.cost] * jobs_u * rows * cols * nd / (ms_u * 1e-3)
                    roof["unfused_kernel"] = {"kernel": f"fast_cost_kernel<R={R},K=24,NW=8,{args.cost.upper()}>", "ops_per_unit": OPS_PER_UNIT[args.cost],
                                              "launch_ms": round(ms_u / n_u, 4), "directions_per_launch": jobs_u / n_u,
                                              "achieved": round(ach_u / 1e12, 3), "frac": round(ach_u / peak_lane_ops, 4),
                                              "how": "same batch, one untimed step with stereo_ctx_set_fuse_pairs(0)"}
        cpu = None
        if world == 1 and not args.no_cpu:
            v, dt, desc = cpu_reference_sample(wl, args.ref_rows, os.cpu_count() or 1, args.cost)
            cpu = {**desc, "value": round(v, 3), "unit": UNIT, "seconds": round(dt, 2)}
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": round(dev_ms / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 (int32 accumulate)", "data": "synthetic",
            "config": {"workload": args.workload + f"_{args.cost}_pair", "rows": rows, "cols": cols, "ndisp": nd,
                       "window": 2 * R + 1, "pairs_per_gpu_per_step": B, "directions": 2,
                       "pair_fusion": "both maps of a pair from one cost volume" if fused else "one cost volume per direction",
                       "sharding": "by pair" + {
                           "root": ", every rank's maps pushed into rank 0's gather buffer (the consumer) by the copy engines over NVLink "
                                   "(stereo_peer_push), overlapping the next step's kernels; all pushes joined inside the timed region",
                           "all": ", every rank's maps pushed into EVERY rank's gather buffer by the copy engines over NVLink "
                                  "(stereo_peer_push), overlapping the next step's kernels; all pushes joined inside the timed region",
                           "nccl": ", NCCL all_gather of maps inside the step" + gather_note, "none": ""}[gather],
                       "gather_bytes_per_step": {"nvlink_tx_per_rank": (map_bytes if gather == "root" else (world - 1) * map_bytes) if world > 1 else 0,
                                                 "nvlink_rx_busiest_rank": (world - 1) * map_bytes if world > 1 else 0},
                       "l2": f"inputs rotate over {S} sets = {S * set_bytes >> 20} MiB > L2 ({l2_bytes >> 20} MiB); "
                             f"one event pair around all timed steps",
                       "out_dtype": str(elem_dtype).replace("torch.", "")},
            "roofline": roof, "cpu_baseline": cpu,
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": B * 2 * rows * cols * 4,
                    "d2h_bytes_per_step": B * 2 * rows * cols * elem, "steps": e2e_steps,
                    "api": "stereo_disparity_pair_batch_f32_host: one call per step, the step's pairs as pinned CV_32FC1 host "
                           "images in, int8/int16 host maps out",
                    "per_pair_calls_value": round(e2e_pp_value, 1), "u8_host_api_value": round(e2e8_value, 1),
                    "host_pack": {"threads": host_threads, "on": packing,
                                  "what": "CV_32FC1 host images converted to u8 by host threads into pinned staging, 1 byte per pixel "
                                          "over the link" if packing else "float rows uploaded, converted on the device",
                                  ("value_with_float_upload" if packing else f"value_with_host_pack_forced_{alt_threads}_threads"): round(e2e_alt_value, 1)},
                    "host_cpus_bound_per_rank": bound_cpus},
            "gpu_launches": launches, "e2e_gpu_launches": e2e_launches, "clocks": clocks,
            "parity_check": parity,
        }
        if dump is not None:
            line["dump_outputs"] = dump
        if gather_sub:
            line["gather_variants"] = gather_sub
        if bands_sub is not None:
            line["bands"] = bands_sub
        if world == 1 and not args.no_suite:
            # the other configurations, each a short device-resident run (same clocks sampler idea: one sample set around all)
            s2 = ClockSampler(local)
            s2.start()
            lines = []
            for wname, cname, b, st_ in (("4k_d256_w11", "ncc", 2, 5), ("1080p_d128_w9", "ssd", 4, 10), ("1080p_d128_w9", "ncc", 4, 10),
                                         ("720p_d64_w9", "ssd", 16, 5), ("720p_d64_w9", "ncc", 16, 5)):
                if wname == args.workload and cname == args.cost:
                    continue
                lines.append(suite_batch_line(torch, lib, ctx, dev, stream, wname, cname, b, st_, peak_lane_ops))
            ps2 = suite_ps2_lines(torch, lib, ctx, dev, stream, 10, peak_lane_ops)
            line["suite"] = {"batches": lines, "ps2": ps2, "clocks": s2.stop()}
        print(json.dumps(line), flush=True)
    G.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# suite: the other configurations next to the headline line (device-resident inputs, CUDA events)
# ---------------------------------------------------------------------------------------------------
# Published GTX 1080 kernel figures for the reference's own problems (BASELINE.md, output/ps2_gpu.log): Mpix*disp/s per map
PS2_PUBLISHED = {
    "p1_ssd_128x128_d4_w13": (226 + 256) / 2, "p2_ssd_511x640_d96_w15": (1628 + 1709) / 2,
    "p3_ssd_noisy_511x640_d96_w15": (1651 + 1568) / 2, "p3_ssd_contrast_511x640_d96_w15": (1628 + 1542) / 2,
    "p4_ncc_511x640_d96_w15": (1127 + 1081) / 2, "p4_ncc_noisy_511x640_d96_w15": (1199 + 1187) / 2,
    "p4_ncc_contrast_511x640_d96_w15": (1198 + 1187) / 2, "p5_ncc_529x640_d81_w15": (1219 + 1295) / 2,
}


def _events_ms(torch, stream, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def suite_batch_line(torch, lib, ctx, dev, stream, wl_name, cost_name, B, steps, peak_lane_ops):
    """One device-resident line like the headline's: B pairs per step of a WORKLOADS shape, inputs rotating over more sets
    than the L2 holds."""
    import introtocomputervision_b200 as sb
    from introtocomputervision_b200 import _capi, synth
    wl = WORKLOADS[wl_name]
    rows, cols, nd, R = wl["rows"], wl["cols"], wl["ndisp"], wl["R"]
    cost = sb.COST_SSD if cost_name == "ssd" else sb.COST_NCORR
    elem_dtype, elem = (torch.int8, 1) if nd <= 128 else (torch.int16, 2)
    Ls, Rs = zip(*[synth.make_pair(rows, cols, nd, wl["seed"] + i)[:2] for i in range(min(B, 4))])
    h_l = torch.from_numpy(np.stack([Ls[i % len(Ls)] for i in range(B)]))
    h_r = torch.from_numpy(np.stack([Rs[i % len(Rs)] for i in range(B)]))
    l2 = int(getattr(torch.cuda.get_device_properties(dev), "L2_cache_size", 126 << 20))
    set_bytes = 2 * B * rows * cols
    S = max(2, -(-int(1.25 * l2) // set_bytes) + 1)
    S = min(S, 64)
    d_l = torch.stack([torch.roll(h_l, 17 * s_, dims=1) for s_ in range(S)]).to(dev)
    d_r = torch.stack([torch.roll(h_r, 17 * s_, dims=1) for s_ in range(S)]).to(dev)
    d_out = torch.empty((2, B, rows, cols), dtype=elem_dtype, device=dev)
    sp = C.c_void_p(stream.cuda_stream)
    k = [0]

    def step():
        s_ = k[0] % S
        k[0] += 1
        rc = lib.stereo_disparity_pair_batch_u8_device(
            ctx.handle, cost, B, d_l[s_].data_ptr(), d_r[s_].data_ptr(), cols, rows * cols, rows, cols, R, nd - 1,
            d_out[0].data_ptr(), d_out[1].data_ptr(), cols * elem, rows * cols * elem, elem, sp)
        if rc != 0:
            raise RuntimeError(_capi.last_error())

    ms = _events_ms(torch, stream, step, steps, 3)
    hot_ms, hot_n = ctx.last_hot_kernel_ms()
    units = B * 2 * rows * cols * nd
    fused = ctx.last_fused_pairs > 0
    opu = (OPS_PER_UNIT_FUSED if fused and cost_name in OPS_PER_UNIT_FUSED else OPS_PER_UNIT)[cost_name]
    # last_hot_kernel_ms covers at most 16 launches of the last call; scale to the directions they covered
    hot_units = ctx.last_hot_jobs * rows * cols * nd
    line = {"workload": f"{wl_name}_{cost_name}_pair", "pairs_per_step": B, "ms_per_step": round(ms, 4),
            "value": round(units / (ms * 1e-3) / 1e6, 1), "unit": UNIT,
            "pair_fusion": bool(fused), "gpu_launches_per_step": ctx.last_launches,
            "l2": f"inputs rotate over {S} sets = {S * set_bytes >> 20} MiB"}
    if hot_n > 0:
        line["hot_kernel_ms_per_step"] = round(hot_ms * (units / hot_units), 4)
        line["hot_share_of_step"] = round(hot_ms * (units / hot_units) / ms, 3)
        line["roofline_frac"] = round(opu * hot_units / (hot_ms * 1e-3) / peak_lane_ops, 4)
        line["ops_per_unit"] = opu
    del d_l, d_r, d_out
    return line


def suite_ps2_lines(torch, lib, ctx, dev, stream, steps, peak_lane_ops):
    """The reference executable's own problems (config/ps2.yaml:19-41, main.cpp:80-330) as device-resident CV_32FC1 pair
    calls (what the reference wrapper holds after its uploads): ms per pair call = two maps, Mpix*disp/s per map next to
    the published GTX 1080 kernel figure (BASELINE.md)."""
    import introtocomputervision_b200 as sb
    from introtocomputervision_b200 import _capi, synth
    problems = []
    L0, R0, _ = synth.make_pair(128, 128, 4, 10)
    L1, R1, _ = synth.make_pair(511, 640, 96, 11)
    L2, R2, _ = synth.make_pair(529, 640, 81, 12)
    f = lambda a: a.astype(np.float32)
    noisy = (synth.noisy_variant(L1, 12), synth.noisy_variant(R1, 13))
    contrast = (synth.contrast_variant(L1), f(R1))
    problems.append(("p1_ssd_128x128_d4_w13", sb.COST_SSD, f(L0), f(R0), 6, 3))
    problems.append(("p2_ssd_511x640_d96_w15", sb.COST_SSD, f(L1), f(R1), 7, 95))
    problems.append(("p3_ssd_noisy_511x640_d96_w15", sb.COST_SSD, *noisy, 7, 95))
    problems.append(("p3_ssd_contrast_511x640_d96_w15", sb.COST_SSD, *contrast, 7, 95))
    problems.append(("p4_ncc_511x640_d96_w15", sb.COST_NCORR, f(L1), f(R1), 7, 95))
    problems.append(("p4_ncc_noisy_511x640_d96_w15", sb.COST_NCORR, *noisy, 7, 95))
    problems.append(("p4_ncc_contrast_511x640_d96_w15", sb.COST_NCORR, *contrast, 7, 95))
    problems.append(("p5_ncc_529x640_d81_w15", sb.COST_NCORR, f(L2), f(R2), 7, 80))
    sp = C.c_void_p(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out, total_ms, total_kernel_ms = [], 0.0, 0.0
    paths = {sb.PATH_EXACT_F32: "exact_f32 (brute force)", sb.PATH_FAST_U8: "fast_u8", sb.PATH_FAST_F32: "fast_f32"}
    for name, cost, Lf, Rf, R, rng in problems:
        rows, cols = Lf.shape
        d_l, d_r = torch.from_numpy(Lf).to(dev), torch.from_numpy(Rf).to(dev)
        d_dl = torch.empty((rows, cols), dtype=torch.int8, device=dev)
        d_dr = torch.empty_like(d_dl)

        def call():
            rc = lib.stereo_disparity_pair_f32_device(ctx.handle, cost, d_l.data_ptr(), cols * 4, d_r.data_ptr(), cols * 4, rows, cols,
                                                      R, rng, d_dl.data_ptr(), d_dr.data_ptr(), cols, 1, sp)
            if rc != 0:
                raise RuntimeError(_capi.last_error())

        for _ in range(3):
            call()
        torch.cuda.synchronize()
        ms_call, ms_kern, ms_hot = [], [], []
        for _ in range(steps):
            flush.zero_()                                    # L2 flushed between the timed calls
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            torch.cuda.synchronize()
            ms_call.append(e0.elapsed_time(e1))
            ms_kern.append(ctx.last_kernel_ms)
            h, n = ctx.last_hot_kernel_ms()
            ms_hot.append(h if n > 0 else float("nan"))
        ms = statistics.median(ms_call)
        units_map = rows * cols * (rng + 1)
        per_map = 2 * units_map / (ms * 1e-3) / 1e6 / 2            # Mpix*disp/s of one map at half the pair call's time
        pub = PS2_PUBLISHED.get(name)
        out.append({"problem": name, "cost": "ssd" if cost == sb.COST_SSD else "ncc", "rows": rows, "cols": cols,
                    "ndisp": rng + 1, "window": 2 * R + 1, "path": paths.get(ctx.last_path, str(ctx.last_path)),
                    "pair_fusion": bool(ctx.last_fused_pairs), "ms_per_pair_call": round(ms, 4), "ms_per_map": round(ms / 2, 4),
                    "kernel_ms": round(statistics.median(ms_kern), 4),
                    "hot_kernel_ms": round(statistics.median(ms_hot), 4), "launches": ctx.last_launches,
                    "value_per_map": round(per_map, 1), "unit": UNIT,
                    "published_gtx1080_kernel": pub, "vs_baseline": round(per_map / pub, 1) if pub else None})
        total_ms += ms
        total_kernel_ms += statistics.median(ms_kern)
    return {"problems": out, "all_problems_ms": round(total_ms, 4), "all_problems_kernel_ms": round(total_kernel_ms, 4),
            "kernel_ms_def": "stereo_ctx_last_kernel_ms: first to last kernel of the call on the device, without the host round trip of the "
                             "classification verdict (the quantity the reference logs per kernel, 360 ms for the same 16 maps)",
            "timing": "device-resident CV_32FC1 images, CUDA events around one stereo_disparity_pair_f32_device call (classification, "
                      "its 16-byte read-back, prep, hot and merge kernels), L2 flushed before every timed call, median of "
                      f"{steps}; the reference's published figure is its kernel alone (GpuTimer, DisparitySSD.cu:192-203)"}


def bands_line(args, wl, lib, ctx, cost, dev, rank, world, local, steps, gather_kind, use_graph=True, dump_dir=None):
    """BASELINE config 4: ONE synthetic pair, output rows sharded over the ranks (R+1 halo rows from the rank's own slab, no
    neighbour exchange), both maps of the band from one launch sequence, the bands gathered inside the timed step: pushed by
    the copy engines into rank 0's buffer (root), into every rank's (all), or all_gather'ed (nccl).  Strong scaling: a step is
    a fraction of a millisecond per rank, so the step (library call + pushes + join) is captured once into a CUDA graph and
    replayed - one graph launch per step instead of a dozen API calls.  Returns the JSON line (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from introtocomputervision_b200 import _capi, sharding, synth

    rows, cols, nd, R = wl["rows"], wl["cols"], wl["ndisp"], wl["R"]
    elem_dtype, elem = (torch.int8, 1) if nd <= 128 else (torch.int16, 2)
    L, Rt, _ = synth.make_pair(rows, cols, nd, wl["seed"])
    r0, r1 = sharding.band_shard(rows, world, rank)
    h0, h1 = sharding.band_halo(rows, r0, r1, R)
    band = -(-rows // world)
    d_l, d_r = torch.from_numpy(L[h0:h1].copy()).to(dev), torch.from_numpy(Rt[h0:h1].copy()).to(dev)   # this rank's slab only
    mine = torch.zeros((2, band, cols), dtype=elem_dtype, device=dev)              # [direction]
    band_bytes = 2 * band * cols * elem
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(device=dev)
    prev_stream = torch.cuda.current_stream(dev)
    torch.cuda.set_stream(stream)
    sp = C.c_void_p(stream.cuda_stream)
    gather = gather_kind if world > 1 else "none"
    pg, gathered, gather_note = None, None, ""
    if gather in ("root", "all"):          # the buffer: [rank][direction][band rows][cols], filled by copy-engine pushes
        try:
            pg = sharding.PeerGather(ctx, world * band_bytes)
        except sharding.PeerGatherUnavailable as e:
            gather, gather_note = "nccl", f" (peer buffers unavailable: {e})"
    if gather == "nccl":
        gathered = torch.empty((world, 2, band, cols), dtype=elem_dtype, device=dev)
    to = [0] if gather == "root" else None

    def step():
        # ONE image pair per step: the gather is part of the step (strong scaling has nothing to overlap it with), so a
        # step ends when this rank's pushes have landed / the collective has finished
        rc = lib.stereo_disparity_pair_band_halo_u8_device(ctx.handle, cost, d_l.data_ptr(), cols, d_r.data_ptr(), cols, rows, cols,
                                                           r0, r1, h0, h1, R, nd - 1, mine[0].data_ptr(), mine[1].data_ptr(),
                                                           cols * elem, elem, sp)
        if rc != 0:
            raise RuntimeError(_capi.last_error())
        if pg is not None:
            pg.push(rank * band_bytes, mine.data_ptr(), band_bytes, stream.cuda_stream, to=to)
            pg.wait(pg.mark(), stream.cuda_stream)
        elif gathered is not None:
            dist.all_gather_into_tensor(gathered.view(torch.uint8).view(-1), mine.view(torch.uint8).view(-1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    launches_per_step = ctx.last_launches
    fused = bool(ctx.last_fused_pairs)
    graph, graph_note = None, "off"
    if use_graph and gather != "nccl":
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream, capture_error_mode="thread_local"):
                step()
            graph_note = "step captured once into a CUDA graph, replayed per step"
        except Exception as e:                       # capture refused (driver / a call that is illegal during capture): plain launches
            graph, graph_note = None, f"capture failed ({type(e).__name__}), plain launches"
            torch.cuda.synchronize()
        ok = torch.tensor([1 if graph is not None else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)        # all ranks replay or none does
        if int(ok.item()) == 0:
            graph = None
    run = (lambda: graph.replay()) if graph is not None else step
    for _ in range(2):
        run()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    evs = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    clocks = sampler.stop()
    dump = None
    if dump_dir:              # this rank's band of both maps, as the last timed step left it
        dump = dump_maps(dump_dir, {"disparity_left": mine[0, :r1 - r0], "disparity_right": mine[1, :r1 - r0]},
                         DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")
        dump.update(rows=[r0, r1])
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    # parity of the gathered image (rank 0's buffer, or this rank's own band for N = 1 / nccl) against the oracle: 64 rows
    # straddling the seam between the first two bands
    parity = None
    if rank == 0 and not args.no_parity:
        if pg is not None:
            buf = pg.local_bytes(dev).view(elem_dtype).view(world, 2, band, cols)
        elif gathered is not None:
            buf = gathered
        else:
            buf = mine.unsqueeze(0)
        full_l = buf[:, 0].reshape(world * band, cols)[:rows].cpu().numpy()
        full_r = buf[:, 1].reshape(world * band, cols)[:rows].cpu().numpy()
        seam = max(0, min(rows - 64, band - 32)) if world > 1 else max(0, rows // 2 - 32)
        parity = oracle_band_check(L, Rt, R, nd, args.cost, full_l, full_r, seam, min(64, rows))
    line = None
    if rank == 0:
        units = 2 * rows * cols * nd * steps                       # the WHOLE image pair, all ranks together
        line = {"metric": METRIC, "value": round(units / (dev_ms * 1e-3) / 1e6, 1), "unit": UNIT, "n_gpus": world,
                "steps": steps, "warmup": max(3, args.warmup), "ms_per_step": round(dev_ms / steps, 4),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8 (int32 accumulate)",
                "data": "synthetic",
                "config": {"workload": args.workload + f"_{args.cost}_pair_bands", "rows": rows, "cols": cols, "ndisp": nd,
                           "window": 2 * R + 1, "band_rows": band, "halo_rows": R + 1, "directions": 2,
                           "pair_fusion": "both maps of a band from one cost volume" if fused else "one cost volume per direction",
                           "sharding": "by row band, slab with halo resident per rank"
                                       + {"root": ", every rank's band pushed into rank 0's buffer by the copy engines over NVLink "
                                                  "(stereo_peer_push), joined inside the step",
                                          "all": ", every rank's band pushed into every rank's buffer by the copy engines over "
                                                 "NVLink (stereo_peer_push), joined inside the step",
                                          "nccl": ", NCCL all_gather of the bands inside the step" + gather_note, "none": ""}[gather],
                           "gather_bytes_per_step": {"nvlink_tx_per_rank": (band_bytes if gather == "root" else (world - 1) * band_bytes) if world > 1 else 0,
                                                     "nvlink_rx_busiest_rank": (world - 1) * band_bytes if world > 1 else 0},
                           "launch": graph_note, "l2": "flushed between steps"},
                "gpu_launches": launches_per_step * steps, "clocks": clocks, "parity_check": parity}
        if dump is not None:
            line["dump_outputs"] = dump
    if pg is not None:
        # cross-rank check: every slot the consumer holds equals what that rank computed
        dist.barrier()
        torch.cuda.synchronize()
        mine_sum = mine.view(torch.uint8).view(-1).to(torch.int64).sum().reshape(1)
        all_sums = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(all_sums, mine_sum)
        if gather == "all" or rank == 0:
            sums = pg.local_bytes(dev).view(world, -1).to(torch.int64).sum(dim=1)
            assert torch.equal(sums, all_sums), "peer gather: a rank's slot does not match that rank's band"
        del graph
        pg.close()
    torch.cuda.set_stream(prev_stream)
    return line


def run_bands(args, wl, lib, ctx, cost, dev, rank, world, local):
    import torch.distributed as dist
    line = bands_line(args, wl, lib, ctx, cost, dev, rank, world, local, args.steps, args.gather, use_graph=not args.no_graph,
                      dump_dir=args.dump_outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="4k_d256_w11", choices=sorted(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=4, help="stereo pairs per GPU per step (a launch sequence carries up to 16 pairs = 32 directions)")
    ap.add_argument("--ref-rows", type=int, default=4, help="CPU sample: image rows per host thread")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-suite", action="store_true", help="skip the suite of other configurations (N = 1 only)")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed oracle check of a band of the step's maps")
    ap.add_argument("--pipe-bands", type=int, default=0, help="row bands per pair in the pipelined host entry points (0 = automatic)")
    ap.add_argument("--cost", default="ssd", choices=["ssd", "ncc"], help="window cost (the headline line is ssd)")
    ap.add_argument("--gather", default="root", choices=["root", "all", "nccl"],
                    help="N > 1: where the ranks' maps go - root: copy-engine pushes over NVLink into rank 0's buffer (the consumer); "
                         "all: into every rank's buffer; nccl: an NCCL all_gather inside the step")
    ap.add_argument("--no-graph", action="store_true", help="bands mode: plain launches instead of replaying a captured CUDA graph")
    ap.add_argument("--mode", default="pairs", choices=["pairs", "bands"],
                    help="pairs: batch sharded by pair, weak scaling (default, the driver's line); "
                         "bands: ONE image sharded by row band with halo, strong scaling (BASELINE config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write both disparity maps of the last timed step as float32 DIR/<name>.npy "
                         f"(at most {DUMP_BYTES // 10**6} MB in all: a fixed, seeded sample of pixels when the maps are larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the maps of --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
