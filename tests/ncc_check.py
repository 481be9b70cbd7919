"""Per-pixel check of NCC disparity maps against the oracle (TEST INFRASTRUCTURE, no GPU needed).

The north-star fraction ("≥ 99.9 % of pixels equal the oracle") says nothing about the pixels that differ.  The kernels rank
candidates by fixed-point keys (fast_kernel.cuh, "NCC keys"), so every disagreement they may legitimately produce is a near-tie:
two candidates whose oracle scores differ by more than the key's resolution must come out in the oracle's order.
:func:`check_ncc_map` checks exactly that for every pixel, with a tolerance τ derived per kernel family below.

Score of a named candidate (:func:`score_at`).  The oracle's rules (oracle/stereo_oracle.c, serial::disparityNCorr +
TM_CCORR_NORMED): with padded centre xp = x + R,

    first = max(xp + dmin, R),  last = min(xp + dmax, cols - 1 + R)
    centre = d + first + (last - first if dmin <= 0 and dmax <= 0 else 0)        (DisparityNCorr.cpp:67)

and the candidate is legal iff first <= centre <= last.  Its score is computed in the literal oracle's arithmetic: products in
double summed in (wy, k) order and rounded to float32, energies in double in the same order, the 10·FLT_EPSILON zero-energy rule
and the 1.125·t rule, stored as float32.

Tolerances (gap = score(oracle's d) - score(got), both by :func:`score_at`; a pixel fails when gap > τ, or when τ = 0 and the
maps differ).  EL(x) is the energy of the reference window at x, ER(c) that of the target window at candidate c.

* ``exact`` (EXACT_F32): the kernel IS the literal oracle (exact.cuh: the same sums in the same order).  τ = 0.
* ``u8_fused`` (FAST_U8, NCC pairs from one cost volume): a key holds round((C·rs + 2^e) · 2^23 / 2^e) with ONE 2^e per pixel,
  the power of two just above its Cauchy-Schwarz bound sqrt(EL)·(1 + 2^-20), so 2^e <= 2·sqrt(EL)·(1 + 2^-20) and one key step
  is 2^(e-23) / sqrt(EL) <= 2^-22 in score units.  Two candidates can trade places when their true scores differ by at most one
  step (each key rounds by half a step) plus the float32 roundings of rs and of the oracle's own stored scores (~2^-24 each).
  τ = 2^-20, four steps.
* ``u8`` (FAST_U8, unfused kernels): the same key with one 2^e per STRIP row (fast.cuh prep_scale_kernel /
  prep_scale_pair_kernel: the power of two above sqrt(max EL over the strip's K <= 24 pixels)).  A dark window next to a bright
  one shares the bright one's scale: τ(x) = 2^-20 · sqrt(max EL over the strip) / sqrt(EL(x)), the strip over-bounded by
  columns x-23 .. x+23 of the row.
* ``f32`` (FAST_F32, general float images, unfused): the key is C·rs + 3·2^e in the binade [2·2^e, 4·2^e) with
  2^e <= 2·sqrt(max EL over the strip)·(1 + 2^-10) (fast.cuh prep_scale_f_kernel / prep_scale_pair_kernel), a step of
  2^(e-22): twice the u8 step, so the key term is 2^-19 · sqrt(max EL over the strip) / sqrt(EL(x)).  On top of it C itself
  carries the rounding of the float32 running sums (fast_kernel.cuh fast_row, OPF): per row each column sum takes two FFMA
  (+ l_new·r_new, - l_old·r_old), every result of magnitude <= (2R+2)·P with P = max|ref|·max|tgt|, so each rounds by at most
  2^-24·(2R+2)·P.  Column sums restart at zero at the start of every row segment a CTA walks (fast_kernel.cuh: col = 0 before
  the segment's warm-up rows) and a segment never leaves its tile's rows, so over a segment of N rows plus the 2R+1 warm-up
  rows a column sum is off by at most 2·(N + 2R+1)·2^-24·(2R+2)·P; C adds 2R+1 of them, and the horizontal sums (2R
  initial adds, two per step over K <= 24 steps) round 2R + 48 more times at magnitude <= (2R+2)(2R+1)·P:
      ΔC <= 2^-24 · (2R+2)·(2R+1)·P · (2·(N + 2R+1) + 2R + 48).
  In score units a candidate c moves by ΔC / sqrt(EL(x)·ER(c)), so τ = key term + ΔC·(1/sqrt(EL·ER(a)) + 1/sqrt(EL·ER(b))).
  N defaults to the image's rows (the bound the code gives for any launch); callers that know the launch's longest segment
  (stereo_launch_plan) pass it.  The bound is a worst case (every rounding in one direction); :func:`check_ncc_map` also
  reports the largest gap over the key term alone, which is how the drift actually behaves.

Where EL(x) = 0 every score of the pixel is 0 and the map must hold the oracle's first candidate (τ = 0).

The returned score (best_out of single-direction calls) is recomputed by the merge kernel (fast.cuh merge_ncc_block) in the
literal oracle's arithmetic and order, for 8-bit-valued AND float images (float x float products are exact in double, so a
contracted FMA changes nothing): it equals :func:`score_at` of the returned disparity bit for bit (:func:`check_best`).
"""
from __future__ import annotations

import numpy as np

import oracle

NCC_DISP_AGREE = 0.999          # BASELINE.json north star: >= 99.9 % equal disparities
FLT_EPSILON = float(np.finfo(np.float32).eps)
FAMILIES = ("exact", "u8_fused", "u8", "f32")
KEY_STEPS_U8 = 2.0 ** -20       # four key steps of 2^-22 (derivation above)
KEY_STEPS_F32 = 2.0 ** -19      # four key steps of 2^-21
STRIP_REACH = 23                # K <= 24: the strip of x lies inside columns x-23 .. x+23
STRIP_K = 24


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def candidate_range(cols, R, dmin, dmax, xs):
    """(first, last) padded candidate centres of unpadded columns xs (stereo_oracle.c:272-274, :415-416)."""
    xp = np.asarray(xs, np.int64) + R
    first = np.maximum(xp + dmin, R)
    last = np.minimum(xp + dmax, cols - 1 + R)
    return first, last


def decode(cols, R, dmin, dmax, xs, disp):
    """(padded centre, legal) of the candidate each disparity names (DisparityNCorr.cpp:67 read backwards)."""
    first, last = candidate_range(cols, R, dmin, dmax, xs)
    right = dmin <= 0 and dmax <= 0
    centre = np.asarray(disp, np.int64) + first + ((last - first) if right else 0)
    return centre, (first <= centre) & (centre <= last)


def unwrap_i8(d8, cols, R, dmin, dmax):
    """The unique legal disparity congruent (mod 256) to each value of an int8 map (the reference's char store wraps ranges
    wider than 127).  Values with no legal representative stay as they are (and fail the legality check)."""
    rows = d8.shape[0]
    xs = np.broadcast_to(np.arange(cols), (rows, cols))
    first, last = candidate_range(cols, R, dmin, dmax, xs)
    n = last - first
    if n.max() >= 256:
        raise ValueError("an int8 map cannot name one of more than 256 candidates")
    lo = -n if (dmin <= 0 and dmax <= 0) else np.zeros_like(n)
    v = d8.astype(np.int64)
    cand = v + 256 * -((v - lo) // 256)             # smallest value >= lo congruent to v
    return np.where(cand <= lo + n, cand, v)


def score_at(ref, tgt, R, dmin, dmax, ys, xs, disp, energies=False):
    """TM_CCORR_NORMED score (float32) of the candidate `disp` names at pixels (ys, xs), in the literal oracle's arithmetic
    (stereo_oracle.c ncorr_row).  Illegal candidates raise.  energies=True also returns (EL, ER) in double."""
    ref, tgt = _f32(ref), _f32(tgt)
    rows, cols = ref.shape
    ys = np.asarray(ys, np.int64).ravel()
    xs = np.asarray(xs, np.int64).ravel()
    centre, legal = decode(cols, R, dmin, dmax, xs, np.asarray(disp).ravel())
    if not legal.all():
        raise ValueError(f"{int((~legal).sum())} disparities name no legal candidate")
    Lp = np.pad(ref, R, mode="edge").astype(np.float64)
    Rp = np.pad(tgt, R, mode="edge").astype(np.float64)
    acc = np.zeros(len(xs))
    el = np.zeros(len(xs))
    er = np.zeros(len(xs))
    for wy in range(-R, R + 1):                        # (wy, k) order, one double rounding per term like the oracle
        yy = ys + R + wy
        for k in range(-R, R + 1):
            a = Lp[yy, xs + R + k]
            b = Rp[yy, centre + k]
            acc += a * b
            el += a * a
            er += b * b
    num = acc.astype(np.float32).astype(np.float64)
    diff2 = np.where(er > 0, er, 0.0)
    lim = np.minimum(0.5, 10 * FLT_EPSILON * er)
    t = np.where(diff2 <= lim, 0.0, np.sqrt(diff2) * np.sqrt(el))
    with np.errstate(divide="ignore", invalid="ignore"):
        sc = np.where(np.abs(num) < t, num / t, np.where(np.abs(num) < t * 1.125, np.sign(num), 0.0))
    sc = sc.astype(np.float32)
    return (sc, el, er) if energies else sc


def _el_map(ref, R):
    """Window energies of the reference image (double box sums; only used to bound a strip's largest energy)."""
    P = np.pad(_f32(ref).astype(np.float64) ** 2, R, mode="edge")
    w = 2 * R + 1
    c = np.zeros((P.shape[0] + 1, P.shape[1] + 1))
    c[1:, 1:] = P.cumsum(0).cumsum(1)
    return c[w:, w:] - c[:-w, w:] - c[w:, :-w] + c[:-w, :-w]


def _strip_max_el(ref, R, ys, xs):
    from scipy.ndimage import maximum_filter1d
    el = _el_map(ref, R)
    rows_needed = np.unique(ys)
    mx = np.zeros_like(el)
    mx[rows_needed] = maximum_filter1d(el[rows_needed], size=2 * STRIP_REACH + 1, axis=1, mode="nearest")
    return mx[ys, xs]


def drift_bound(ref, tgt, R, seg_rows):
    """ΔC of the float32 running sums over a segment of seg_rows rows (module docstring, ``f32``)."""
    P = float(np.max(np.abs(_f32(ref)))) * float(np.max(np.abs(_f32(tgt))))
    w = 2 * R + 1
    return 2.0 ** -24 * (w + 1) * w * P * (2 * (seg_rows + w) + 2 * R + 2 * STRIP_K)


def tolerance(family, ref, tgt, R, ys, xs, el, er_a, er_b, seg_rows):
    """(τ, key term of τ) for pixels (ys, xs) whose reference window has energy el, between candidates of target energies
    er_a and er_b (module docstring)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        if family == "exact":
            key = np.zeros(len(ys))
        elif family == "u8_fused":
            key = np.full(len(ys), KEY_STEPS_U8)
        else:
            ratio = np.sqrt(_strip_max_el(ref, R, ys, xs) / el)
            key = (KEY_STEPS_U8 if family == "u8" else KEY_STEPS_F32) * ratio
        tau = key.copy()
        if family == "f32":
            tau += drift_bound(ref, tgt, R, seg_rows) * (1 / np.sqrt(el * er_a) + 1 / np.sqrt(el * er_b))
    # EL = 0: every score is 0, the first candidate must win
    return np.where(el > 0, tau, 0.0), np.where(el > 0, key, 0.0)


def check_ncc_map(got, ref, tgt, R, dmin, dmax, family, oracle_disp=None, seg_rows=None, min_agree=NCC_DISP_AGREE, what=""):
    """Assert that every pixel of the NCC map `got` names a legal candidate and, where it differs from the oracle's
    disparity, one whose oracle score is within τ (module docstring) of the oracle's winner; then the north-star fraction.
    oracle_disp: the oracle's int32 map (computed with oracle.ncorr_fast when omitted).  Returns a dict of statistics:
    differing pixels, largest gap / τ, largest gap and (f32) largest gap over the key term alone."""
    assert family in FAMILIES, family
    ref, tgt = _f32(ref), _f32(tgt)
    rows, cols = ref.shape
    got = np.asarray(got)
    assert got.shape == (rows, cols), (got.shape, ref.shape)
    g = unwrap_i8(got, cols, R, dmin, dmax) if got.dtype == np.int8 else got.astype(np.int64)
    if oracle_disp is None:
        oracle_disp = oracle.ncorr_fast(ref, tgt, R, dmin, dmax)
    o = np.asarray(oracle_disp)
    o = unwrap_i8(o, cols, R, dmin, dmax) if o.dtype == np.int8 else o.astype(np.int64)
    tag = f"{what} ({family}, {rows}x{cols}, R={R}, [{dmin}, {dmax}])"
    xs_all = np.broadcast_to(np.arange(cols), (rows, cols))
    _, legal = decode(cols, R, dmin, dmax, xs_all, g)
    if not legal.all():
        bad = np.argwhere(~legal)
        raise AssertionError(f"{tag}: {len(bad)} disparities name no legal candidate, first (y, x, d) "
                             f"{[(int(y), int(x), int(g[y, x])) for y, x in bad[:5]]}")
    ys, xs = np.nonzero(g != o)
    stats = {"pixels": rows * cols, "differ": int(len(ys)), "max_ratio": 0.0, "max_gap": 0.0, "max_gap_over_key": 0.0}
    if len(ys):
        s_o, el, er_o = score_at(ref, tgt, R, dmin, dmax, ys, xs, o[ys, xs], energies=True)
        s_g, _, er_g = score_at(ref, tgt, R, dmin, dmax, ys, xs, g[ys, xs], energies=True)
        gap = s_o.astype(np.float64) - s_g.astype(np.float64)
        tau, key = tolerance(family, ref, tgt, R, ys, xs, el, er_o, er_g, rows if seg_rows is None else seg_rows)
        with np.errstate(divide="ignore", invalid="ignore"):
            fail = (gap > tau) | ((tau == 0) & (g[ys, xs] != o[ys, xs]))
            ratio_tau = np.where(tau > 0, gap / tau, np.where(gap > 0, np.inf, 0.0))
        stats["max_ratio"] = float(np.max(ratio_tau))
        stats["max_gap"] = float(np.max(gap))
        if family == "f32":
            stats["max_gap_over_key"] = float(np.max(np.where(key > 0, gap / key, 0.0)))
        if fail.any():
            idx = np.argsort(-np.where(fail, ratio_tau, -np.inf))[:5]
            worst = [(int(ys[i]), int(xs[i]), int(g[ys[i], xs[i]]), int(o[ys[i], xs[i]]), float(gap[i]), float(tau[i])) for i in idx]
            raise AssertionError(f"{tag}: {int(fail.sum())} of {len(ys)} differing pixels beyond tau, largest gap/tau "
                                 f"{stats['max_ratio']:.3g}; worst (y, x, got, oracle, gap, tau): {worst}")
    agree = 1.0 - stats["differ"] / stats["pixels"]
    assert agree >= min_agree, f"{tag}: disparity agreement {agree:.5f} < {min_agree}"
    return stats


def check_best(best, got, ref, tgt, R, dmin, dmax, mask=None, what=""):
    """The returned score map equals the literal oracle's score of the returned disparity, bit for bit, at every pixel (or
    at the pixels of `mask`)."""
    rows, cols = np.asarray(ref).shape
    got = np.asarray(got)
    g = unwrap_i8(got, cols, R, dmin, dmax) if got.dtype == np.int8 else got.astype(np.int64)
    ys, xs = np.nonzero(np.ones((rows, cols), bool) if mask is None else mask)
    want = score_at(ref, tgt, R, dmin, dmax, ys, xs, g[ys, xs])
    have = np.asarray(best, np.float32)[ys, xs]
    bad = np.nonzero(have.view(np.uint32) != want.view(np.uint32))[0]
    assert bad.size == 0, (f"{what}: returned score differs from the oracle's score of the returned disparity at {len(bad)} "
                           f"pixels, first (y, x, got, want) {[(int(ys[i]), int(xs[i]), float(have[i]), float(want[i])) for i in bad[:5]]}")


def family_of(ctx):
    """The kernel family of the context's last call, as check_ncc_map names it."""
    import introtocomputervision_b200 as sb
    path = ctx.last_path
    if path == sb.PATH_EXACT_F32:
        return "exact"
    if path == sb.PATH_FAST_F32:
        return "f32"
    assert path == sb.PATH_FAST_U8, path
    return "u8_fused" if ctx.last_fused_pairs > 0 else "u8"
