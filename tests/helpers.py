"""Shared helpers for the parity tests: golden-fixture loading and comparison rules.

Comparison rules (SURVEY.md 8d "Parity criteria"):
  * ``err`` maps must be equal (a documented handful of FP32 near-ties may be allowed by the caller);
  * on pixels where the reference succeeded (err == 1): integer walk (Ncalls) equal,
    dx/dy within tol * max(1, |ref|), T/df/f within tol relative;
  * on err == 0 pixels only ``err`` is compared -- the reference's other outputs
    are partly uninitialised there (Model.cpp:566, 927; SURVEY.md 3.3).
"""
import glob
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz"))
                  if not p.endswith("hooks.npz") and not os.path.basename(p).startswith("post_"))


def load_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    c = {k: z[k] for k in z.files}
    Na = int(c["Na"])
    c["sam"] = [c.pop(f"sam{k}") for k in range(Na)]
    c["ref"] = [c.pop(f"ref{k}") for k in range(Na)]
    c["mask"] = [c.pop(f"mask{k}") for k in range(Na)] if "mask0" in c else None
    c["pos"] = [tuple(int(v) for v in p) for p in c["pos"]] if "pos" in c else None
    c["kind"] = str(c["kind"])
    for k in ("Nw", "max_shift", "padding"):
        c[k] = int(c[k])
    c["assign"] = str(c["assign"]) if "assign" in c else None
    c["subpx"] = int(c["subpx"]) if "subpx" in c else None
    c["step"] = int(c["step"]) if "step" in c else None
    c["ROI"] = tuple(tuple(int(v) for v in r) for r in c["ROI"]) if "ROI" in c else None
    c["dxdy"] = tuple(float(v) for v in c["dxdy"]) if "dxdy" in c else None
    c["abc"] = c.get("abc")
    c["expected"] = {k[4:]: c[k] for k in list(c) if k.startswith("out_")}
    return c


def roi_of(case):
    """The ((start,stop,step),(start,stop,step)) the reference ended up using."""
    r = case["ROI_after"]
    return tuple(tuple(int(v) for v in x) for x in r)


def reference_matcher(kind, sam, ref, **model_kw):
    """What a full-size parity test compares the product with: the UNMODIFIED reference (oracle/_ref) where its
    compiled extension is present, otherwise the C restatement (oracle/port.py), which the golden vectors pin to the
    reference.  The reference's sources are not part of this repository, so a plain checkout takes the restatement.
    Returns (match(ROI, **kw) -> maps with the debug arrays fp32_parity_stats reads, name of the one used)."""
    from oracle import port, ref as oref
    R = oref.load()
    threads = os.cpu_count()
    if R is not None:
        cls = {"NoDF": R.UMPAModelNoDF, "DF": R.UMPAModelDF, "DFKernel": R.UMPAModelDFKernel}[kind]
        m = cls(list(sam), list(ref), **model_kw)
        return (lambda ROI, **kw: m.match(ROI=ROI, num_threads=threads, quiet=True, **kw)), "reference"
    om = port.OracleModel(kind, list(sam), list(ref), **model_kw)
    return (lambda ROI, **kw: om.match(ROI=ROI, num_threads=threads, **kw)), "C restatement"


def compare(got, exp, tol=1e-9, walk_exact=True, max_err_mismatch=0, max_outliers=0, outlier_tol=None,
            label=""):
    """Returns a dict of statistics; raises AssertionError with a readable message."""
    stats = {}
    err_g, err_e = np.asarray(got["err"]), np.asarray(exp["err"])
    assert err_g.shape == err_e.shape, f"{label}: shape {err_g.shape} vs {err_e.shape}"
    mism = int((err_g != err_e).sum())
    stats["err_mismatch"] = mism
    assert mism <= max_err_mismatch, f"{label}: err map differs in {mism} pixels"
    ok = (err_e == 1) & (err_g == 1)
    if walk_exact and "debug_Ncalls" in got and "debug_Ncalls" in exp:
        nm = int((np.asarray(got["debug_Ncalls"])[ok] != np.asarray(exp["debug_Ncalls"])[ok]).sum())
        stats["ncalls_mismatch"] = nm
        assert nm <= max_outliers, f"{label}: Ncalls differs in {nm} ok-pixels"
    for k in ("dx", "dy", "T", "df", "f"):
        if k not in exp or k not in got:
            continue
        g, e = np.asarray(got[k], dtype=np.float64)[ok], np.asarray(exp[k], dtype=np.float64)[ok]
        if g.size == 0:
            continue
        scale = np.maximum(1., np.abs(e)) if k in ("dx", "dy") else np.maximum(np.abs(e), 1e-300)
        rel = np.abs(g - e) / scale
        rel = np.where(np.isfinite(rel), rel, np.inf)
        bad = rel > tol
        stats[k + "_max"] = float(rel.max())
        stats[k + "_outliers"] = int(bad.sum())
        assert bad.sum() <= max_outliers, (
            f"{label}: {k} exceeds {tol:g} in {int(bad.sum())} of {g.size} ok-pixels (max {rel.max():.3g})")
        if outlier_tol is not None and bad.any():
            assert rel.max() <= outlier_tol, f"{label}: {k} outlier {rel.max():.3g} > {outlier_tol:g}"
    return stats


# ---------------------------------------------------------------------------------------------
# FP32 table path: which deviations are "documented exceptions"?
#
# The table path feeds the reference's own spline/Newton refinement with costs that carry FP32
# rounding (relative ~1e-6 of the block's cost scale, see tests/test_table_algebra.py).  In a
# well-conditioned pixel that moves dx/dy by ~1e-6.  In an ill-conditioned one (flat or saddle-
# like 4x4 block: Newton wanders far outside the block, or stops one iteration earlier/later on
# its absolute 1e-8 criterion) the REFERENCE'S OWN answer moves by more than the tolerance when
# its own inputs are perturbed at that level -- e.g. its -ffast-math and strict builds already
# disagree there.  sensitivity() measures exactly that, with the oracle's spline on the
# reference's debug_a block; a deviation is excused only where the reference is that sensitive.

def block_corner(d, a):
    """(ip, jp) such that a == d[ip:ip+4, jp:jp+4] (Optim.cpp:344-384)."""
    d5 = np.asarray(d).reshape(5, 5)
    a4 = np.asarray(a).reshape(4, 4)
    for ip in (0, 1):
        for jp in (0, 1):
            if np.array_equal(d5[ip:ip + 4, jp:jp + 4], a4):
                return ip, jp
    return None


def sensitivity(d, a, eps, trials=12, seed=0):
    """Largest move of the reference's sub-pixel position / value when its 4x4 block is perturbed
    by eps * max|a| (Gaussian); inf when the block cannot be located."""
    from oracle import port
    c = block_corner(d, a)
    if c is None:
        return np.inf, np.inf
    ip, jp = c
    a = np.asarray(a, dtype=np.float64).reshape(16)
    p0, v0 = port.spmin(a, (1. - ip, 1. - jp))
    rng = np.random.default_rng(seed)
    dp, dv = 0., 0.
    for _ in range(trials):
        p1, v1 = port.spmin(a + eps * np.abs(a).max() * rng.standard_normal(16), (1. - ip, 1. - jp))
        if not (np.all(np.isfinite(p1)) and np.isfinite(v1)):
            return np.inf, np.inf
        dp = max(dp, float(np.abs(p1 - p0).max()))
        dv = max(dv, abs(v1 - v0))
    return dp, dv


def fp32_parity_stats(got, exp, tol=1e-4, eps=3e-6, noise_floor=3e-6, max_probe=400):
    """Everything the parity criteria of SURVEY.md 8(d) ask for, as numbers (no assertion): how `got` (the FP32 table
    path) differs from `exp` (the reference, with its debug arrays).  JSON-serialisable.
      err_mismatch      pixels whose err flag differs
      ncalls_mismatch   ok-pixels whose number of cost evaluations differs (the integer walk took another route) ...
      walk_ties         ... of which the reference's own cache shows a neighbour within 1e-5 of the cost scale of the
                        centre (its `> d +- 1e-8` test is a coin flip there); walk_unexplained = the rest
      T_ties / df_ties  ok-pixels (walk equal) whose T / df differs by more than tol: same tie criterion; *_unexplained
      exceptions        ok-pixels (walk equal) with dx, dy beyond tol*max(1,|ref|) or f beyond tol*|ref| + floor
      excused           ... of which the reference's own sub-pixel answer moves by more than tol/2 when its 4x4 block is
                        perturbed at the eps level (ill-conditioned refinement); unexcused = the rest
      <k>_max, <k>_p999 largest / 99.9th-percentile deviation of k in {dx, dy, T, df, f} over the compared pixels"""
    err_g, err_e = np.asarray(got["err"]), np.asarray(exp["err"])
    st = {"n_px": int(err_e.size), "n_ok": int((err_e == 1).sum()), "err_mismatch": int((err_g != err_e).sum()),
          "tol": tol}
    ok = (err_e == 1) & (err_g == 1)
    dpos = exp["debug_d"][err_e == 1]
    cost_scale = float(np.median(dpos[dpos > 0])) if (dpos > 0).any() else 1.
    st["cost_scale"] = cost_scale

    def near_tie(i, j):
        # every comparison the walk makes is between two entries of its cache: the centre against a neighbour
        # (Optim.cpp:294, 325), the two neighbours of an axis against each other (337, 344-345), a 4x4 entry against
        # the centre (364) -- at the final centre AND at the centres it passed on the way, whose entries are still in
        # the cache.  A "tie": two evaluated entries of the reference's own (final) cache agree to FP32 noise.  (With
        # 25 entries spread over ~0.5 cost scales a random pixel has such a pair with probability ~0.2 %; all three
        # pixels of config 2's 4.1 M whose walk differs from the FP64 evaluation have one, at 1e-7 ... 1.4e-6 of the
        # cost scale, and end at the same minimum: tools/diag_walk_mismatch.py.)
        d5 = exp["debug_d"][i, j]
        known = np.sort(d5[d5 > -.5])
        return known.size > 1 and float(np.diff(known).min()) <= 1e-5 * cost_scale

    nc = ok & (np.asarray(got["debug_Ncalls"]) != exp["debug_Ncalls"])
    st["ncalls_mismatch"] = int(nc.sum())
    ties = sum(1 for i, j in np.argwhere(nc) if near_tie(i, j))
    st["walk_ties"], st["walk_unexplained"] = ties, int(nc.sum()) - ties
    ok = ok & ~nc
    for k in ("T", "df"):
        if k not in exp or k not in got:
            continue
        rel = np.abs(np.asarray(got[k]) - exp[k]) / np.maximum(np.abs(exp[k]), .25)
        bad = ok & ~(rel <= tol)
        t = sum(1 for i, j in np.argwhere(bad) if near_tie(i, j))
        st[k + "_ties"], st[k + "_unexplained"] = t, int(bad.sum()) - t
        st[k + "_max"] = float(rel[ok].max()) if ok.any() else 0.
        st[k + "_p999"] = float(np.percentile(rel[ok], 99.9)) if ok.any() else 0.
    bad = np.zeros(err_e.shape, dtype=bool)
    for k in ("dx", "dy"):
        rel = np.abs(np.asarray(got[k]) - exp[k]) / np.maximum(1., np.abs(exp[k]))
        bad |= ok & ~(rel <= tol)
        st[k + "_max"] = float(rel[ok].max()) if ok.any() else 0.
        st[k + "_p999"] = float(np.percentile(rel[ok], 99.9)) if ok.any() else 0.
    df_ = np.abs(np.asarray(got["f"]) - exp["f"])
    relf = df_ / np.maximum(np.abs(exp["f"]), 1e-300)
    st["f_max"] = float(relf[ok].max()) if ok.any() else 0.
    st["f_p999"] = float(np.percentile(relf[ok], 99.9)) if ok.any() else 0.
    bad_f = ok & ~(df_ <= tol * np.abs(exp["f"]) + noise_floor * cost_scale)
    idx = np.argwhere(bad | bad_f)
    st["exceptions"] = int(len(idx))
    excused = probed = 0
    for i, j in idx[:max_probe]:
        probed += 1
        dp, dv = sensitivity(exp["debug_d"][i, j], exp["debug_a"][i, j], eps)
        if bad[i, j]:
            excused += dp > tol / 2
        else:
            excused += dv > (tol * abs(exp["f"][i, j]) + noise_floor * cost_scale) / 2
    st["excused"], st["unexcused"], st["probed"] = int(excused), int(probed - excused), int(probed)
    return st


# ---------------------------------------------------------------------------------------------
# Table costs entry by entry.  With sub_pixel_mode = 0 the walk leaves uv at its integer centre (walk_refine,
# walk.cuh; Optim.cpp:399), so dy = c0 and dx = c1 exactly, and cell t of the 5x5 cache debug_d (-1: not evaluated)
# holds the cost of the shift (si, sj) = (c0 + t // 5 - 2, c1 + t % 5 - 2).  A pixel that stopped with a bound error
# (err == 0) has no reliable centre: locate_centre() finds it from the cached values.

# |cost - cost64| <= COST_BOUND * (median FP64 cost of the case): the FP32 restatement of the table algebra meets it
# (test_table_algebra.py), so a kernel that does not has another arithmetic, not other rounding
COST_BOUND = 3e-5


def cached_cells(res):
    """(i, j, si, sj, cost) arrays of every cached cost of the err == 1 pixels of a sub_pixel_mode = 0 match."""
    d, ok = np.asarray(res["debug_d"]), np.asarray(res["err"]) == 1
    c0, c1 = np.asarray(res["dy"]), np.asarray(res["dx"])
    assert np.array_equal(c0[ok], np.rint(c0[ok])) and np.array_equal(c1[ok], np.rint(c1[ok])), "non-integer centre"
    i, j, t = np.nonzero(ok[:, :, None] & (d != -1))
    return i, j, c0[i, j].astype(int) + t // 5 - 2, c1[i, j].astype(int) + t % 5 - 2, d[i, j, t]


def locate_centre(d5, table, margin=100.):
    """Centre (c0, c1) of a 5x5 walk cache whose centre is unknown: the offset at which its evaluated cells match the
    pixel's (S, S) FP64 cost table best.  None when no cell was evaluated, or when another offset matches within a
    factor `margin` as well (the match would be a guess)."""
    d5 = np.asarray(d5)
    t = np.nonzero(d5 != -1)[0]
    h = (table.shape[0] - 1) // 2
    if t.size == 0:
        return None
    devs = []
    for c0 in range(-h - 2, h + 3):
        for c1 in range(-h - 2, h + 3):
            si, sj = c0 + t // 5 - 2, c1 + t % 5 - 2
            if np.all(np.abs(si) <= h) and np.all(np.abs(sj) <= h):
                devs.append((float(np.abs(d5[t] - table[si + h, sj + h]).max()), c0, c1))
    devs.sort()
    if not devs or (len(devs) > 1 and devs[1][0] <= margin * devs[0][0]):
        return None
    return devs[0][1], devs[0][2]


def check_costs(got, exp, scale, label="", rows=None, bound=COST_BOUND):
    """|got - exp| <= bound * scale for every cell; returns (max, 99.9th percentile) of |got - exp| / scale.
    rows: the output row of every cell, named in the failure message."""
    got, exp = np.asarray(got, np.float64), np.asarray(exp, np.float64)
    assert got.size > 0, f"{label}: no cells compared"
    r = np.abs(got - exp) / scale
    r = np.where(np.isfinite(r), r, np.inf)
    bad = r > bound
    if bad.any():
        where = "" if rows is None else ", rows %s" % sorted(set(int(v) for v in np.asarray(rows)[bad]))[:40]
        raise AssertionError(f"{label}: {int(bad.sum())} of {r.size} costs off by more than {bound:g} of the cost "
                             f"scale (max {r.max():.3g}{where})")
    return float(r.max()), float(np.percentile(r, 99.9))


def compare_fp32(got, exp, tol=1e-4, eps=3e-6, max_exception_frac=0.03, noise_floor=3e-6, label=""):
    """Parity check of the FP32 table path (tolerances of BASELINE.json north_star):
    err map and Ncalls (the integer walk) must be EQUAL; T, df within tol relative; dx, dy within
    tol*max(1,|ref|) and f within tol*|ref| + noise_floor*cost_scale, except in pixels where the
    reference's own refinement is that sensitive to eps-level input noise (see above)."""
    err_g, err_e = np.asarray(got["err"]), np.asarray(exp["err"])
    assert np.array_equal(err_g, err_e), f"{label}: err map differs in {(err_g != err_e).sum()} pixels"
    ok = err_e == 1
    stats = {"n_ok": int(ok.sum())}
    dpos = exp["debug_d"][ok]
    cost_scale = float(np.median(dpos[dpos > 0])) if (dpos > 0).any() else 1.
    # the integer walk (Ncalls) must be equal, except at a documented tie (see below): there the walk
    # may settle on the neighbouring shift, and the sub-pixel fit then starts from another 4x4 block
    walk_ties = 0
    for i, j in np.argwhere(ok & (np.asarray(got["debug_Ncalls"]) != exp["debug_Ncalls"])):
        d5 = exp["debug_d"][i, j]
        near = min(abs(d5[n] - d5[12]) for n in (7, 11, 13, 17) if d5[n] > -.5)
        assert near <= 1e-5 * cost_scale, (
            f"{label}: Ncalls {got['debug_Ncalls'][i, j]} vs {exp['debug_Ncalls'][i, j]} at ({i},{j}) without a tie "
            f"(nearest neighbour cost differs by {near:.3g})")
        walk_ties += 1
        ok = ok.copy()
        ok[i, j] = False
    stats["walk_ties"] = walk_ties
    assert walk_ties <= max(2, int(2e-3 * ok.sum())), f"{label}: {walk_ties} walk ties"
    # T and df belong to the INTEGER shift the walk settled on (reference's args_copy).  They may
    # differ only at a documented tie: two neighbouring integer shifts whose costs agree to FP32
    # noise (|d_n - d_centre| <= 1e-5 * cost scale in the reference's own 5x5 cache), where the
    # reference's `> d + tol` comparisons (tol = 1e-8 absolute, Optim.cpp:294,325) are a coin flip.
    ties = 0
    for k in ("T", "df"):
        if k in exp:
            # relative for |value| >= 0.25 (T ~ 0.8, df ~ 0.5-1 on real data), absolute tol/4 below:
            # on the noisy fixtures df = K/T passes through zero, where "relative" is meaningless
            rel = np.abs(got[k] - exp[k]) / np.maximum(np.abs(exp[k]), .25)
            for i, j in np.argwhere(ok & ~(rel <= tol)):
                d5 = exp["debug_d"][i, j]
                near = min(abs(d5[n] - d5[12]) for n in (7, 11, 13, 17) if d5[n] > -.5)
                assert near <= 1e-5 * cost_scale, (
                    f"{label}: {k} off by {rel[i, j]:.3g} at ({i},{j}) without a tie (nearest neighbour cost "
                    f"differs by {near:.3g})")
                ties += 1
            stats[k] = float(np.max(rel[ok])) if ok.any() else 0.
    stats["ties"] = ties
    assert ties <= max(2, int(2e-3 * ok.sum())), f"{label}: {ties} integer-shift ties"
    bad = np.zeros(err_e.shape, dtype=bool)
    for k in ("dx", "dy"):
        rel = np.abs(got[k] - exp[k]) / np.maximum(1., np.abs(exp[k]))
        bad |= ok & ~(rel <= tol)
        stats[k + "_p99"] = float(np.percentile(rel[ok], 99)) if ok.any() else 0.
    df_ = np.abs(got["f"] - exp["f"])
    bad_f = ok & ~(df_ <= tol * np.abs(exp["f"]) + noise_floor * cost_scale)
    idx = np.argwhere(bad | bad_f)
    stats["exceptions"] = len(idx)
    assert len(idx) <= max(2, int(max_exception_frac * ok.sum())), (
        f"{label}: {len(idx)} of {int(ok.sum())} ok-pixels deviate by more than {tol:g}")
    for i, j in idx:
        dp, dv = sensitivity(exp["debug_d"][i, j], exp["debug_a"][i, j], eps)
        if bad[i, j]:
            assert dp > tol / 2, (f"{label}: pixel ({i},{j}) dx/dy off by "
                                  f"{abs(got['dx'][i, j] - exp['dx'][i, j]):.3g}/{abs(got['dy'][i, j] - exp['dy'][i, j]):.3g} "
                                  f"but the reference moves only {dp:.3g} under eps={eps:g}")
        else:
            assert dv > (tol * abs(exp["f"][i, j]) + noise_floor * cost_scale) / 2, (
                f"{label}: pixel ({i},{j}) f off by {df_[i, j]:.3g} but the reference moves only {dv:.3g}")
    return stats
