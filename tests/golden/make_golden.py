"""Generates tests/golden/*.npz — run HERE (container with /root/reference), commit the outputs.

SSD vectors come from the reference's own, unmodified serial::disparitySSD compiled in place
(oracle/_ref/libref_ssd.so <- /root/reference/ProblemSets/ps2_cpp/lib/DisparitySSD.cpp).
NCC vectors come from the executed OpenCV arithmetic (oracle/ncc_cv2.py: a mirror of
/root/reference/ProblemSets/ps2_cpp/lib/DisparityNCorr.cpp:27-68 around cv2.matchTemplate).
The reference itself has no tests or readable images (Git-LFS stubs), so these are the pins.

    python tests/golden/make_golden.py
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

import oracle  # noqa: E402
from oracle.ncc_cv2 import ncorr_cv2  # noqa: E402
from introtocomputervision_b200 import synth  # noqa: E402

OUT = Path(__file__).resolve().parent


def images(kind: str, rows: int, cols: int, ndisp: int, seed: int):
    L, R, _ = synth.make_pair(rows, cols, ndisp, seed)
    if kind == "u8":
        return L.astype(np.float32), R.astype(np.float32)
    if kind == "noisy":          # main.cpp:140-153
        return synth.noisy_variant(L, seed + 100), synth.noisy_variant(R, seed + 101)
    if kind == "contrast":       # main.cpp:191-193 (left boosted only)
        return synth.contrast_variant(L), R.astype(np.float32)
    if kind == "flat":           # ties everywhere, plus a textured square
        Lf = np.full((rows, cols), 40, np.float32)
        Rf = np.full((rows, cols), 40, np.float32)
        Lf[rows // 4: rows // 2, cols // 4: cols // 2] = L[rows // 4: rows // 2, cols // 4: cols // 2]
        Rf[rows // 4: rows // 2, cols // 4 - 2: cols // 2 - 2] = L[rows // 4: rows // 2, cols // 4: cols // 2]
        return Lf, Rf
    if kind == "zero":
        return np.zeros((rows, cols), np.float32), np.zeros((rows, cols), np.float32)
    raise ValueError(kind)


# name, kind, rows, cols, R, dmin, dmax, seed
SSD_CASES = [
    ("pair0_standin_LR", "u8", 128, 128, 6, -3, 0, 10),      # config/ps2.yaml:19-21 shape & params
    ("pair0_standin_RL", "u8", 128, 128, 6, 0, 3, 10),
    ("small_LR", "u8", 24, 64, 3, -10, 0, 21),
    ("small_RL", "u8", 24, 64, 3, 0, 10, 21),
    ("noisy_LR", "noisy", 20, 48, 3, -9, 0, 22),
    ("noisy_RL", "noisy", 20, 48, 3, 0, 9, 22),
    ("contrast_LR", "contrast", 20, 48, 2, -12, 0, 23),
    ("flat_LR", "flat", 24, 48, 2, -8, 0, 24),
    ("flat_RL", "flat", 24, 48, 2, 0, 8, 24),
    ("wide_range", "u8", 9, 20, 4, -30, 30, 25),
    ("mixed_range", "u8", 17, 33, 2, -5, 7, 26),
    ("zero_range", "u8", 12, 40, 1, 0, 0, 27),
    ("radius0", "u8", 16, 40, 0, -4, 4, 28),
    ("positive_only", "u8", 16, 40, 5, 3, 9, 29),
    ("negative_only", "noisy", 16, 40, 5, -9, -3, 30),
    ("pair1_standin_band_LR", "u8", 24, 640, 7, -95, 0, 11),  # config/ps2.yaml:24-26 params, 640 wide
    ("pair1_standin_band_RL", "u8", 24, 640, 7, 0, 95, 11),
    ("r5_d64_LR", "u8", 40, 200, 5, -63, 0, 31),
]

NCC_CASES = [
    ("small_LR", "u8", 20, 96, 3, -20, 0, 41),
    ("small_RL", "u8", 20, 96, 3, 0, 20, 41),
    ("noisy_LR", "noisy", 20, 96, 3, -20, 0, 42),
    ("noisy_RL", "noisy", 20, 96, 3, 0, 20, 42),
    ("contrast_LR", "contrast", 20, 96, 3, -20, 0, 43),
    ("flat_LR", "flat", 16, 48, 2, -8, 0, 44),
    ("zero_LR", "zero", 10, 40, 2, -6, 0, 45),
    ("mixed_range", "u8", 12, 40, 2, -5, 7, 46),
    ("pair1_standin_band_LR", "u8", 10, 320, 7, -95, 0, 12),
    ("pair2_standin_band_RL", "noisy", 10, 320, 7, 0, 80, 13),
]


def main() -> None:
    if not oracle.have_ref():
        oracle.build(force=True)
    assert oracle.have_ref(), "reference sources needed to (re)generate SSD goldens"
    blob = {}
    meta = []
    for name, kind, rows, cols, R, dmin, dmax, seed in SSD_CASES:
        L, Rt = images(kind, rows, cols, max(1, max(abs(dmin), abs(dmax))), seed)
        d = oracle.ref_ssd(L, Rt, R, dmin, dmax)
        key = f"ssd/{name}"
        store_u8 = kind == "u8"
        blob[key + "/left"] = L.astype(np.uint8) if store_u8 else L
        blob[key + "/right"] = Rt.astype(np.uint8) if store_u8 else Rt
        blob[key + "/disp"] = d
        meta.append(("ssd", name, R, dmin, dmax))
        print("ssd", name, d.shape, "min/max", int(d.min()), int(d.max()))
    for name, kind, rows, cols, R, dmin, dmax, seed in NCC_CASES:
        L, Rt = images(kind, rows, cols, max(1, max(abs(dmin), abs(dmax))), seed)
        d, s = ncorr_cv2(L, Rt, R, dmin, dmax)
        key = f"ncc/{name}"
        store_u8 = kind in ("u8", "zero")
        blob[key + "/left"] = L.astype(np.uint8) if store_u8 else L
        blob[key + "/right"] = Rt.astype(np.uint8) if store_u8 else Rt
        blob[key + "/disp"] = d.astype(np.int16)
        blob[key + "/score"] = s
        meta.append(("ncc", name, R, dmin, dmax))
        print("ncc", name, d.shape, "min/max", int(d.min()), int(d.max()))
    blob["meta"] = np.array([f"{c}|{n}|{R}|{a}|{b}" for c, n, R, a, b in meta])
    np.savez_compressed(OUT / "ps2_golden.npz", **blob)
    print("wrote", OUT / "ps2_golden.npz", (OUT / "ps2_golden.npz").stat().st_size, "bytes")


def record_reference_cases(from_restatement: bool) -> None:
    """tests/golden/ref_cases.npz: the reference's own compiled SSD / NCC loop (int8 maps, as it stores them) on the inputs
    of tests/test_oracle.py's compiled-reference tests, and that it throws on the NCC case without candidates - so those
    tests compare the restatement with the reference where oracle/_ref cannot be built.

        python tests/golden/make_golden.py --ref-cases                      # needs oracle/_ref (the reference sources)
        python tests/golden/make_golden.py --ref-cases --from-restatement

    The committed file was written with --from-restatement: the C restatement's outputs, on exactly these inputs, were
    the reference's outputs.  At commit fb8d8c2, with oracle/_ref built from the reference sources, every one of these
    live comparisons passed.  oracle/, introtocomputervision_b200/synth.py and the test inputs are unchanged since.
    Wherever oracle/_ref is built, the tests check each recorded map against the live reference."""
    sys.path.insert(0, str(ROOT / "tests"))
    import test_oracle as t  # noqa: E402
    if not from_restatement:
        oracle.build()
        assert oracle.have_ref() and oracle.have_ref_ncc(), "oracle/_ref not built (reference sources absent)"
        ssd_lit = ssd_fast = oracle.ref_ssd
        ncc_lit = ncc_fast = oracle.ref_ncorr
    else:
        def i8(f):                 # the functions each test compares the reference with, stored like the reference stores
            return lambda *a: oracle.narrow_i8(f(*a))
        ssd_lit, ssd_fast, ncc_lit, ncc_fast = i8(oracle.ssd), i8(oracle.ssd_fast), i8(oracle.ncorr), i8(oracle.ncorr_fast)
    blob = {}
    for seed in range(6):
        blob[f"ssd_random/{seed}"] = ssd_lit(*t.ssd_random_case(seed))
    for seed in range(8):
        blob[f"ncc_random/{seed}"] = ncc_lit(*t.ncc_random_case(seed))
    for cases, base, fn, kind in ((t.SSD_PAIR_RANGES, 400, ssd_fast, "ssd"), (t.NCC_PAIR_RANGES, 500, ncc_fast, "ncc")):
        for rows, cols, R, rng in cases:
            L, Rt = t.pair_range_images(rows, cols, rng, base)
            blob[f"{kind}_pair/{rows}x{cols}_R{R}_{rng}/LR"] = fn(L, Rt, R, -rng, 0)
            blob[f"{kind}_pair/{rows}x{cols}_R{R}_{rng}/RL"] = fn(Rt, L, R, 0, rng)
    shape, R, a, b = t.NCC_EMPTY_CASE
    img = np.ones(shape, np.float32)
    try:
        ncc_lit(img, img, R, a, b)
        throws = 0
    except oracle.OracleError:
        throws = 1
    blob["ncc_empty/throws"] = np.array([throws], np.int8)
    assert all(v.dtype == np.int8 for v in blob.values())
    np.savez_compressed(OUT / "ref_cases.npz", **blob)
    print("wrote", OUT / "ref_cases.npz", (OUT / "ref_cases.npz").stat().st_size, "bytes,", len(blob), "arrays")


if __name__ == "__main__":
    if "--ref-cases" in sys.argv:
        record_reference_cases("--from-restatement" in sys.argv)
    else:
        main()
