"""bench.py --dump-outputs: the files it writes (whole maps, or one fixed sample of pixels within the byte budget), and on the
GPU box that they hold the maps of the last timed step, against the oracle."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import bench
import oracle
from introtocomputervision_b200 import synth

ROOT = Path(__file__).resolve().parents[1]


def test_dump_maps_whole_and_sampled(tmp_path):
    import torch
    g = torch.Generator().manual_seed(1)
    maps = {"left": torch.randint(-128, 128, (3, 50, 60), dtype=torch.int8, generator=g),
            "right": torch.randint(-300, 300, (3, 50, 60), dtype=torch.int16, generator=g)}
    whole = bench.dump_maps(tmp_path / "whole", maps, 10**6)
    assert whole["pixels_per_map"] == whole["of_pixels"] == 3000 and sorted(whole["files"]) == ["left.npy", "right.npy"]
    for name, t in maps.items():
        a = np.load(tmp_path / "whole" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy())
    budget = 20_000
    reps = {d: bench.dump_maps(tmp_path / d, maps, budget) for d in ("s1", "s2")}
    for d in reps:
        assert sum(p.stat().st_size for p in (tmp_path / d).iterdir()) <= budget
    idx = np.load(tmp_path / "s1" / "sample_index.npy")
    assert np.array_equal(np.load(tmp_path / "s2" / "sample_index.npy"), idx)          # the same sample every run
    assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0) and reps["s1"]["pixels_per_map"] == idx.size > 0
    assert "float64" in reps["s1"]["sample_index"]
    for name, t in maps.items():
        a = np.load(tmp_path / "s1" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy().reshape(3, -1)[:, idx.astype(np.int64)])


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    name, pairs, steps = "ps2_pair1_511x640_d96_w15", 2, 2
    wl = bench.WORKLOADS[name]
    rows, cols, nd, R = wl["rows"], wl["cols"], wl["ndisp"], wl["R"]
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", name, "--pairs", str(pairs), "--steps", str(steps),
                          "--warmup", "3", "--no-cpu", "--no-suite", "--no-parity", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    line = json.loads([s for s in res.stdout.splitlines() if s.startswith("{")][-1])
    d = line["dump_outputs"]
    assert line["steps"] == steps and d["step"] == 3 + steps - 1 and d["pixels_per_map"] == rows * cols
    got_l, got_r = np.load(out / "disparity_left.npy"), np.load(out / "disparity_right.npy")
    assert got_l.shape == got_r.shape == (pairs, rows, cols) and got_l.dtype == np.float32
    for i in range(pairs):
        L, Rt, _ = synth.make_pair(rows, cols, nd, wl["seed"] + i)
        L, Rt = (np.roll(a, d["input_roll_rows"], axis=0).astype(np.float32) for a in (L, Rt))
        assert np.array_equal(got_l[i], oracle.ssd_fast(L, Rt, R, -(nd - 1), 0)), i
        assert np.array_equal(got_r[i], oracle.ssd_fast(Rt, L, R, 0, nd - 1)), i
