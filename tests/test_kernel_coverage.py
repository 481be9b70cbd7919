"""Every hot-kernel instantiation and every launch schedule the dispatcher can pick, run against the oracle.

The hot path picks one of 100 compiled kernel variants per launch (fast_ctx_init in csrc/fast.cuh lists them) and one of three
ways to cut the (tile, row) space over the CTAs (fast_geometry_nw).  The matrix below states both axes once:

* an instantiation cell is (family, R, strips per warp, gen); gen (fused 8-bit SSD only) is 0 for the kernel compiled for
  launches whose blocks are all MODE 1 - fast_fused_all_mode1: R <= 5 and a candidate count that is a multiple of the
  128 / strips disparities of a group - and 1 for the general one;
* a schedule cell is (family, schedule, border kernel): schedule 0 linear split, 1 equal row segments, 2 row-band-major
  items (counted only with two or more bands, so that band seams are inside the launch); the border kernel (8-bit fused
  SSD only) takes the candidates centred in the right padding.

A cell is credited only to a launch an entry point really makes, derived with stereo_launch_plan (pure host arithmetic):
pair calls put both directions of up to 16 pairs of 8-bit images in one launch sequence, float images that are not
8-bit-valued go one pair per launch, and a single-direction call is one launch whose schedule the plan does not model (it
credits its instantiation only).  The fixed shape tables of test_gpu_parity.py are credited with the launches their tests
make; seeded random shapes are not.  CASES adds the launches the tables miss, and the CPU tests below hold the union to
the whole matrix: a dispatcher change that moves a case off its cell, or a case removed, fails them by name.
"""
import ctypes as C

import numpy as np
import pytest

import ncc_check as nc
import oracle
import test_gpu_parity as parity
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth

SSD, NCC = sb.COST_SSD, sb.COST_NCORR
B200_SMS = 148
FMAXR = 7                   # fast_kernel.cuh
FFREE_MASK_R = 5            # fast_kernel.cuh: largest radius whose invalid candidates lose through the key alone
FGROUP = 128                # fast_kernel.cuh: disparities per warp group with one strip per warp (64 with two)
MAX_SIDE = 32768             # the entry points refuse larger images (stereo_b200.cu validate)
FAMILIES = ("u8_ssd", "u8_ncc", "u8_fused_ssd", "u8_fused_ncc", "f32_ssd", "f32_fused_ssd", "f32_ncc")


def instantiation_matrix():
    """The kernels fast_ctx_init requires from the build, as (family, R, strips per warp, gen)."""
    cells = set()
    for R in range(FMAXR + 1):
        for hs in (1, 2):
            cells |= {("u8_ssd", R, hs, None), ("u8_ncc", R, hs, None), ("u8_fused_ncc", R, hs, None)}
            cells |= {("u8_fused_ssd", R, hs, gen) for gen in ((0, 1) if R <= FFREE_MASK_R else (1,))}
        cells |= {(fam, R, 1, None) for fam in ("f32_ssd", "f32_fused_ssd", "f32_ncc")}     # float operands: one strip
    return cells


def schedule_matrix():
    """(family, schedule, border kernel) of every launch cut a pair launch can get (test_schedule_sweep_stays_in_the_matrix
    shows each reachable and nothing outside)."""
    return {(fam, s, 0) for fam in FAMILIES for s in (0, 1, 2)} | {("u8_fused_ssd", s, 1) for s in (0, 1, 2)}


# Cells no launch can get, and why (fast_geometry_nw): the border kernel exists for 8-bit fused SSD only.
UNREACHABLE = {(fam, s, 1): "fused_border_kernel serves 8-bit fused SSD launches only"
               for fam in FAMILIES if fam != "u8_fused_ssd" for s in (0, 1, 2)}


def plan(cost, f32, n_pairs, rows, cols, R, rng, fuse, sms=B200_SMS):
    p = _capi.LaunchPlan()
    rc = _capi.lib().stereo_launch_plan(cost, int(f32), n_pairs, rows, cols, R, rng, int(fuse), sms, C.byref(p))
    assert rc == 0, _capi.last_error()
    return p


def family(cost, f32, fused):
    return ("f32_" if f32 else "u8_") + ("fused_" if fused else "") + ("ssd" if cost == SSD else "ncc")


def pair_launch_cells(cost, f32, n_pairs, rows, cols, R, rng, fuse, sms=B200_SMS):
    """(plan, instantiation cell, schedule cell or None) of the hot launch over n_pairs whole image pairs."""
    assert rows <= MAX_SIDE and cols <= MAX_SIDE, "no entry point takes such images"
    p = plan(cost, f32, n_pairs, rows, cols, R, rng, fuse, sms)
    fam = family(cost, f32, p.fused)
    gen = None
    if fam == "u8_fused_ssd":      # fast_fused_all_mode1 (csrc/fast.cuh)
        gen = 0 if R <= FFREE_MASK_R and (rng + 1) % (FGROUP // p.strips_per_warp) == 0 else 1
    sched = (fam, p.schedule, p.border_kernel) if p.schedule != 2 or p.bands >= 2 else None
    return p, (fam, R, p.strips_per_warp, gen), sched


def direction_cell(cost, f32, rows, cols, R, dmin, dmax):
    """Instantiation cell of a single-direction launch: strips per warp depend on the candidate count only, so the unfused
    plan of a pair with as many candidates names the kernel."""
    _, inst, _ = pair_launch_cells(cost, f32, 1, rows, cols, R, dmax - dmin, 0)
    return inst


def _params(test_fn):
    (mark,) = [m for m in getattr(test_fn, "pytestmark", []) if m.name == "parametrize"]
    return list(mark.args[1])


def fixed_table_cells():
    """Cells the fixed tables of test_gpu_parity.py reach, with the launches their tests make."""
    cells = set()
    for table, cost, f32 in ((parity.FAST_SHAPES, SSD, 0), (parity.NCC_FAST_SHAPES, NCC, 0), (parity.F32_SHAPES, SSD, 1),
                             (_params(parity.test_ncc_float_kernels_vs_oracle), NCC, 1)):
        cells |= {direction_cell(cost, f32, rows, cols, R, dmin, dmax) for rows, cols, R, dmin, dmax in table}
    # pair calls of one small pair: one pipeline item, the whole pair in one launch, with pair fusion on and off
    for table, cost, f32 in ((parity.FUSED_SHAPES, SSD, 0), (parity.GENERAL_FUSED_SHAPES, SSD, 0), (parity.NCC_PAIR_SHAPES, NCC, 0),
                             (_params(parity.test_ssd_float_fused_pairs_vs_oracle), SSD, 1)):
        for rows, cols, R, rng in table:
            for fuse in (1, 0):
                _, inst, sched = pair_launch_cells(cost, f32, 1, rows, cols, R, rng, fuse)
                cells |= {inst} | ({sched} if sched else set())
    return cells


class Case:
    """One launch of an entry point.  entry: "pair_batch_u8_device" (n pairs of u8 images), "pair_f32_device" (one pair of
    float images), "u8_device" / "f32_device" (one direction over [dmin, dmax], returning the costs / scores).  operands:
    "u8", "f32_8bit" (float images holding 8-bit values) or "f32_noisy".  low: the right half of every image is quantised to
    multiples of 64 (_images), so that exact ties cross band seams.  comb: the sign comb _images describes (NCC, R = 0)."""

    def __init__(self, name, entry, cost, operands, pairs, rows, cols, R, rng=None, dmin=None, dmax=None, fuse=1, low=False,
                 comb=False, inst=None, sched=None):
        self.name, self.entry, self.cost, self.operands = name, entry, cost, operands
        self.pairs, self.rows, self.cols, self.R, self.fuse, self.low, self.comb = pairs, rows, cols, R, fuse, low, comb
        self.single = entry in ("u8_device", "f32_device")
        self.dmin, self.dmax = (dmin, dmax) if self.single else (-rng, 0)
        self.rng = rng
        self.inst, self.sched = inst, sched          # the cells this case claims
        self.f32 = operands == "f32_noisy"           # (8-bit-valued float images take the packed kernels)

    def cells(self, sms=B200_SMS):
        """(plan or None, instantiation cell, schedule cell or None) of the launch this case makes."""
        if self.single:
            return None, direction_cell(self.cost, self.f32, self.rows, self.cols, self.R, self.dmin, self.dmax), None
        return pair_launch_cells(self.cost, self.f32, self.pairs, self.rows, self.cols, self.R, self.rng, self.fuse, sms)

    def __repr__(self):
        return self.name


def _case(name, entry, cost, operands, pairs, rows, cols, R, rng=None, inst=None, sched=None, **kw):
    return pytest.param(Case(name, entry, cost, operands, pairs, rows, cols, R, rng=rng, inst=inst, sched=sched, **kw), id=name)


B, F, U1, U2 = "pair_batch_u8_device", "pair_f32_device", "u8_device", "f32_device"

CASES = [
    # the benchmark's own launch (bench.py, 4k_d256_w11): 4 pairs of 3840x2160, 256 disparities, 11x11, fused SSD, 3 bands
    _case("bench_4k_x4_fused_ssd", B, SSD, "u8", 4, 2160, 3840, 5, 255, low=True,
          inst=("u8_fused_ssd", 5, 1, 0), sched=("u8_fused_ssd", 2, 0)),
    # row-band-major items (two or more bands) of every family, and the fused SSD border kernel under each cut
    _case("bands_u8_ssd", B, SSD, "u8", 4, 48, 10000, 1, 31, fuse=0, low=True, inst=("u8_ssd", 1, 2, None), sched=("u8_ssd", 2, 0)),
    _case("bands_u8_ncc", B, NCC, "u8", 4, 48, 10000, 1, 31, fuse=0, low=True, inst=("u8_ncc", 1, 2, None), sched=("u8_ncc", 2, 0)),
    _case("bands_u8_fused_ncc", B, NCC, "u8", 16, 96, 8000, 1, 15, low=True,
          inst=("u8_fused_ncc", 1, 2, None), sched=("u8_fused_ncc", 2, 0)),
    _case("bands_border_u8_fused_ssd", B, SSD, "u8", 4, 96, 640, 1, 4000, low=True,
          inst=("u8_fused_ssd", 1, 1, 1), sched=("u8_fused_ssd", 2, 1)),
    _case("segments_border_u8_fused_ssd", B, SSD, "u8", 1, 256, 1280, 1, 63,
          inst=("u8_fused_ssd", 1, 2, 0), sched=("u8_fused_ssd", 1, 1)),
    _case("bands_f32_ssd", F, SSD, "f32_noisy", 1, 160, 30000, 0, 7, fuse=0, low=True,
          inst=("f32_ssd", 0, 1, None), sched=("f32_ssd", 2, 0)),
    _case("segments_f32_ssd", F, SSD, "f32_noisy", 1, 12, 5000, 3, 15, fuse=0, inst=("f32_ssd", 3, 1, None), sched=("f32_ssd", 1, 0)),
    _case("bands_f32_fused_ssd", F, SSD, "f32_noisy", 1, 192, 32768, 0, 7, low=True,
          inst=("f32_fused_ssd", 0, 1, None), sched=("f32_fused_ssd", 2, 0)),
    _case("segments_f32_fused_ssd", F, SSD, "f32_noisy", 1, 256, 800, 1, 15,
          inst=("f32_fused_ssd", 1, 1, None), sched=("f32_fused_ssd", 1, 0)),
    _case("bands_f32_ncc", F, NCC, "f32_noisy", 1, 192, 32768, 1, 7, low=True, inst=("f32_ncc", 1, 1, None), sched=("f32_ncc", 2, 0)),
    _case("segments_f32_ncc", F, NCC, "f32_noisy", 1, 384, 200, 2, 15, inst=("f32_ncc", 2, 1, None), sched=("f32_ncc", 1, 0)),
    _case("linear_f32_ncc", F, NCC, "f32_noisy", 1, 24, 100, 2, 20, sched=("f32_ncc", 0, 0), inst=("f32_ncc", 2, 1, None)),
    _case("ncc_f32_r0", U2, NCC, "f32_noisy", 1, 24, 100, 0, dmin=-20, dmax=0, comb=True, inst=("f32_ncc", 0, 1, None)),
    # fused SSD pairs: the MODE-1-only (gen 0) and general (gen 1) kernels the tables miss
    _case("fused_ssd_r0_1strip_gen1", B, SSD, "u8", 2, 20, 300, 0, 99, inst=("u8_fused_ssd", 0, 1, 1), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r0_2strips_gen0", F, SSD, "f32_8bit", 1, 24, 200, 0, 63, inst=("u8_fused_ssd", 0, 2, 0), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r1_2strips_gen1", B, SSD, "u8", 3, 18, 260, 1, 40, inst=("u8_fused_ssd", 1, 2, 1), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r2_1strip_gen1", B, SSD, "u8", 1, 16, 400, 2, 150, inst=("u8_fused_ssd", 2, 1, 1), sched=("u8_fused_ssd", 0, 1)),
    _case("fused_ssd_r3_2strips_gen0", B, SSD, "u8", 2, 22, 333, 3, 63, inst=("u8_fused_ssd", 3, 2, 0), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r3_2strips_gen1", F, SSD, "f32_8bit", 1, 20, 150, 3, 50, inst=("u8_fused_ssd", 3, 2, 1), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r4_2strips_gen1", B, SSD, "u8", 5, 14, 200, 4, 33, inst=("u8_fused_ssd", 4, 2, 1), sched=("u8_fused_ssd", 0, 0)),
    _case("fused_ssd_r5_2strips_gen1", B, SSD, "u8", 2, 26, 310, 5, 60, inst=("u8_fused_ssd", 5, 2, 1), sched=("u8_fused_ssd", 0, 0)),
    # fused NCC pairs: one strip (more than 64 candidates) and two strips (up to 64) at the radii the tables miss
    _case("fused_ncc_r0_1strip", B, NCC, "u8", 2, 20, 300, 0, 100, inst=("u8_fused_ncc", 0, 1, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r2_1strip", F, NCC, "f32_8bit", 1, 24, 280, 2, 127, inst=("u8_fused_ncc", 2, 1, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r4_1strip", B, NCC, "u8", 3, 16, 250, 4, 90, inst=("u8_fused_ncc", 4, 1, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r3_2strips", B, NCC, "u8", 2, 20, 200, 3, 63, inst=("u8_fused_ncc", 3, 2, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r5_2strips", B, NCC, "u8", 1, 30, 220, 5, 40, inst=("u8_fused_ncc", 5, 2, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r6_2strips", B, NCC, "u8", 2, 22, 180, 6, 50, inst=("u8_fused_ncc", 6, 2, None), sched=("u8_fused_ncc", 0, 0)),
    _case("fused_ncc_r7_2strips", B, NCC, "u8", 2, 28, 240, 7, 63, inst=("u8_fused_ncc", 7, 2, None), sched=("u8_fused_ncc", 1, 0)),
    # packed NCC, one direction (the scores come back too)
    _case("ncc_r0_1strip", U1, NCC, "u8", 1, 20, 300, 0, dmin=-100, dmax=0, inst=("u8_ncc", 0, 1, None)),
    _case("ncc_r2_1strip", U1, NCC, "u8", 1, 24, 260, 2, dmin=0, dmax=90, inst=("u8_ncc", 2, 1, None)),
    _case("ncc_r3_2strips", U1, NCC, "u8", 1, 30, 200, 3, dmin=-20, dmax=20, inst=("u8_ncc", 3, 2, None)),
    _case("ncc_r7_2strips", U1, NCC, "u8", 1, 26, 240, 7, dmin=-63, dmax=0, inst=("u8_ncc", 7, 2, None)),
]

CASE_LIST = [p.values[0] for p in CASES]
BENCH_CASE = "bench_4k_x4_fused_ssd"


# ---- CPU: the cases reach what they claim, and with the fixed tables the whole matrix ----------------------------------------

def test_cases_claim_their_planned_cells():
    wrong = []
    for c in CASE_LIST:
        p, inst, sched = c.cells()
        if (inst, sched) != (c.inst, c.sched):
            wrong.append(f"{c.name}: plans {inst} / {sched}, claims {c.inst} / {c.sched}")
        if p is not None and p.schedule == 2:
            assert p.bands >= 2, f"{c.name}: one band only"
    assert not wrong, "cases whose planned cell changed:\n" + "\n".join(wrong)


def test_cases_and_fixed_tables_cover_the_matrix():
    covered = fixed_table_cells()
    for c in CASE_LIST:
        _, inst, sched = c.cells()
        covered |= {inst} | ({sched} if sched else set())
    matrix = instantiation_matrix() | schedule_matrix()
    missing = sorted(matrix - covered, key=str)
    assert not missing, f"{len(missing)} cells no case reaches:\n" + "\n".join(map(str, missing))
    assert covered <= matrix, f"cells outside the matrix: {sorted(covered - matrix, key=str)}"


def test_every_case_adds_a_cell():
    """Each case reaches a cell that neither the fixed tables nor the other cases reach (the benchmark's launch is kept
    whatever the rest covers)."""
    fixed = fixed_table_cells()
    mine = {c.name: {x for x in c.cells()[1:] if x} for c in CASE_LIST}
    idle = []
    for c in CASE_LIST:
        others = set(fixed)
        for n, s in mine.items():
            if n != c.name:
                others |= s
        if c.name != BENCH_CASE and not (mine[c.name] - others):
            idle.append(c.name)
    assert not idle, f"cases that add no cell: {idle}"


def test_bench_case_is_the_benchmark_launch():
    import bench
    wl = bench.WORKLOADS["4k_d256_w11"]
    (c,) = [c for c in CASE_LIST if c.name == BENCH_CASE]
    assert (c.entry, c.cost, c.operands, c.fuse) == (B, SSD, "u8", 1)
    assert (c.pairs, c.rows, c.cols, c.R, c.rng) == (4, wl["rows"], wl["cols"], wl["R"], wl["ndisp"] - 1)


def test_schedule_sweep_stays_in_the_matrix():
    """A sweep of pair launches (8-bit batches of 1 .. 16 pairs, float images one pair per launch) over shapes, windows and
    ranges: every schedule cell it meets is in the matrix, and it meets every one of them."""
    seen = set()
    for cost in (SSD, NCC):
        for f32 in (0, 1):
            for fuse in (0, 1):
                for n in ((1,) if f32 else (1, 4, 16)):
                    for R in (0, 1, 7):
                        for rows in (16, 96, 512):
                            for cols in (256, 640, 8000, MAX_SIDE):
                                for rng in (1, 63, 255, 4095):
                                    _, inst, sched = pair_launch_cells(cost, f32, n, rows, cols, R, rng, fuse)
                                    assert inst in instantiation_matrix(), inst
                                    if sched:
                                        seen.add(sched)
    assert seen <= schedule_matrix(), sorted(seen - schedule_matrix(), key=str)
    assert not seen & set(UNREACHABLE)
    assert seen == schedule_matrix(), sorted(schedule_matrix() - seen, key=str)


# ---- GPU: every case runs its planned launch and matches the oracle ------------------------------------------------------------

def _images(c):
    """The pairs of a case as float32 arrays of what the entry point gets (and the arrays it is handed).  Low-texture cases
    quantise the right half of every image to multiples of 64 (+ 0.25 for noisy float images, which keeps them off the
    8-bit path): flat runs whose candidates tie exactly, across every band seam."""
    pairs = []
    for i in range(c.pairs):
        L, Rt, _ = synth.make_pair(c.rows, c.cols, max(2, min(c.rng if c.rng else c.dmax - c.dmin, c.cols // 2, 64)),
                                   60000 + 97 * i + c.rows + c.cols + c.R)
        if c.operands == "f32_noisy":
            Lf, Rf = synth.noisy_variant(L, 7 + i), synth.noisy_variant(Rt, 8 + i)
        else:
            Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        if c.comb:
            # A 1x1 NCC window scores only the sign of l * r: on float images every same-sign candidate of a pixel scores 1
            # up to one float32 rounding, and which one the oracle ranks first is rounding noise below any key resolution.
            # So the reference is positive and the target negative except in one column of every dmax - dmin + 1: every
            # pixel has exactly one candidate that scores +1.
            Lf = np.abs(Lf) + np.float32(1)
            Rf = -(np.abs(Rf) + np.float32(1))
            Rf[:, ::c.dmax - c.dmin + 1] *= -1
        if c.low:
            h = c.cols // 2
            off = np.float32(0.25 if c.operands == "f32_noisy" else 0.0)
            for img, src in ((Lf, L), (Rf, Rt)):
                img[:, h:] = (src[:, h:] // 64 * 64).astype(np.float32) + off
        pairs.append((Lf, Rf))
    return pairs


def _run(ctx, c, pairs):
    """Calls the case's entry point; returns the maps (and the costs / scores of single-direction calls)."""
    import torch
    lib = _capi.lib()
    rows, cols = c.rows, c.cols
    dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).cuda()
    if c.entry == B:
        Ls = dev(np.stack([p[0] for p in pairs]), np.uint8)
        Rs = dev(np.stack([p[1] for p in pairs]), np.uint8)
        ol = torch.zeros((c.pairs, rows, cols), dtype=torch.int16, device="cuda")
        orr = torch.zeros_like(ol)
        rc = lib.stereo_disparity_pair_batch_u8_device(ctx.handle, c.cost, c.pairs, Ls.data_ptr(), Rs.data_ptr(), cols, rows * cols,
                                                       rows, cols, c.R, c.rng, ol.data_ptr(), orr.data_ptr(), cols * 2, rows * cols * 2,
                                                       2, None)
    elif c.entry == F:
        Ls, Rs = dev(pairs[0][0], np.float32), dev(pairs[0][1], np.float32)
        ol = torch.zeros((1, rows, cols), dtype=torch.int16, device="cuda")
        orr = torch.zeros_like(ol)
        rc = lib.stereo_disparity_pair_f32_device(ctx.handle, c.cost, Ls.data_ptr(), cols * 4, Rs.data_ptr(), cols * 4, rows, cols,
                                                  c.R, c.rng, ol.data_ptr(), orr.data_ptr(), cols * 2, 2, None)
    else:
        kind = np.uint8 if c.entry == U1 else np.float32
        a, b = dev(pairs[0][0], kind), dev(pairs[0][1], kind)
        d = torch.zeros((rows, cols), dtype=torch.int32, device="cuda")
        best = torch.zeros((rows, cols), dtype=torch.int32 if c.cost == SSD else torch.float32, device="cuda")
        fn = lib.stereo_disparity_u8_device if c.entry == U1 else lib.stereo_disparity_f32_device
        rc = fn(ctx.handle, c.cost, a.data_ptr(), a.stride(0) * a.element_size(), b.data_ptr(), b.stride(0) * b.element_size(),
                rows, cols, c.R, c.dmin, c.dmax, d.data_ptr(), cols * 4, 4, best.data_ptr(), cols * 4, None)
    assert rc == 0, _capi.last_error()
    ctx.synchronize()
    if c.single:
        return d.cpu().numpy(), best.cpu().numpy()
    return ol.cpu().numpy(), orr.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_case_runs_its_launch_and_matches_the_oracle(ctx, case):
    import torch
    c = case
    p, inst, sched = c.cells(torch.cuda.get_device_properties(0).multi_processor_count)
    assert (inst, sched) == (c.inst, c.sched), f"on this device's SM count the case plans {inst} / {sched}"
    pairs = _images(c)
    ctx.set_fuse_pairs(bool(c.fuse))
    try:
        out = _run(ctx, c, pairs)
    finally:
        ctx.set_fuse_pairs(True)
    # the launch the plan describes: the kernel family, fused or not, every direction in ONE hot launch
    assert ctx.last_path == (sb.PATH_FAST_F32 if c.f32 else sb.PATH_FAST_U8)
    fused = bool(p is not None and p.fused)
    assert ctx.last_fused_pairs == (c.pairs if fused else 0)
    assert ctx.last_hot_jobs == (1 if c.single else 2 * c.pairs)
    assert ctx.last_hot_kernel_ms()[1] == 1, "the directions did not share one hot launch"
    fam = "f32" if c.f32 else ("u8_fused" if fused else "u8")
    if c.single:
        d, best = out
        a, b = pairs[0]
        if c.cost == SSD:
            d_ref, c_ref = oracle.ssd_fast(a, b, c.R, c.dmin, c.dmax, return_cost=True)
            bad = np.argwhere(d != d_ref)
            assert bad.size == 0, f"{c.name}: differs at {bad[:5].tolist()} (of {len(bad)})"
            assert np.array_equal(best, c_ref), c.name
        else:
            d_ref = oracle.ncorr_fast(a, b, c.R, c.dmin, c.dmax)
            nc.check_ncc_map(d, a, b, c.R, c.dmin, c.dmax, fam, oracle_disp=d_ref, what=c.name)
            nc.check_best(best, d, a, b, c.R, c.dmin, c.dmax, what=c.name)
        return
    dl, dr = out
    for i, (a, b) in enumerate(pairs):
        for got, ref, tgt, lo, hi, what in ((dl[i], a, b, -c.rng, 0, "L->R"), (dr[i], b, a, 0, c.rng, "R->L")):
            tag = f"{c.name} pair {i} {what}"
            if c.cost == SSD:
                want = oracle.ssd_fast(ref, tgt, c.R, lo, hi)
                bad = np.argwhere(got != want)
                assert bad.size == 0, f"{tag}: differs at {bad[:5].tolist()} (of {len(bad)})"
            else:
                nc.check_ncc_map(got, ref, tgt, c.R, lo, hi, fam, oracle_disp=oracle.ncorr_fast(ref, tgt, c.R, lo, hi), what=tag)
