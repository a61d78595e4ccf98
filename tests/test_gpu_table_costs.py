"""GPU: the FP32 table path's costs, entry by entry, against FP64 -- for every instantiation of the table kernels and
every tile plan the planner can be made to choose.

Reading the costs.  With sub_pixel_mode = 0 the walk leaves uv at its integer centre, so (dy, dx) is the centre and
debug_d (the walk's 5x5 cache) holds the costs the walk read from the tables at known shifts (helpers.cached_cells;
test_table_algebra.py pins the convention on the reference's C restatement).  Pixels that stopped with a bound error
(err == 0: every pixel of max_shift 2, whose 3x3 shift range holds no 4x4 block) have no reliable centre: it is found
by matching the cached values against the pixel's FP64 costs (helpers.locate_centre), and a pixel whose match is not
unique by two orders of magnitude is left out.

References: the vectorised FP64 cost tables (tests/table_algebra.py, pinned to the reference by test_table_algebra.py)
for NoDF / DF with assign_coordinates 'sam'; the C restatement's direct cost for 'ref' and for DFKernel, on a pixel
sample that holds whole rows at the top and bottom of the output and the columns on both sides of every strip
boundary.  Bound: |cost - cost64| <= 3e-5 x the median FP64 cost of the case, which the FP32 restatement of the same
algebra meets on the same cells (asserted where it models the arithmetic: NoDF / DF, 'sam').

DF with a one-pixel window (Nw 0) is left out: its dark-field fit is singular (den = t2 t3 - t6^2 = 0) and the
reference's costs are NaN there.

The environment knobs UMPA_TAB_EH / _STREAM / _FB / _G / _NST / _NSEG / _CTAS select tile plans the cost model does not
prefer.  The planner reads them on every call, and so does umpa_table_plan, from which the tests read the plan a match
will use (same arguments as table_path.cu: rows, cols + dxX, the device's SM count)."""
import math

import numpy as np
import pytest

from helpers import cached_cells, check_costs, locate_centre
from table_algebra import cost_tables

pytestmark = pytest.mark.gpu

KNOBS = ("UMPA_TAB_EH", "UMPA_TAB_STREAM", "UMPA_TAB_FB", "UMPA_TAB_G", "UMPA_TAB_NST", "UMPA_TAB_NSEG", "UMPA_TAB_CTAS")
NA = 11                  # no FB the planner picks divides it: the last TMA box of every pass is partial
TAB_SIZES = [(N0, N1) for N0 in (45, 53, 61, 75, 83, 99) for N1 in (70, 75)]


@pytest.fixture(autouse=True)
def _plain_env(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("UMPA_NO_STREAMING", "1")        # one table launch over the whole ROI, not row bands


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def plan_of(Na, Nw, ms, rows, cols):
    """umpa_table_plan as a dict; None where the planner has no plan."""
    import ctypes
    from umpa_b200 import _capi
    out = (ctypes.c_int * 10)()
    if _capi.lib().umpa_table_plan(Na, Nw, ms, rows, cols, sm_count(), out):
        return None
    p = dict(zip(("EH", "order", "G", "npass", "FB", "nstage", "TW", "nseg", "nstrips", "nt"), list(out)))
    # what plan_tiles derives from them (table_path.cu)
    H2 = 2 * Nw
    p["seg_rows"] = p["EH"] - H2 if p["order"] == 0 else -(-rows // p["nseg"])
    p["nchunk_full"] = -(-(p["seg_rows"] + H2) // p["EH"])
    p["nchunk_last"] = -(-(rows - (p["nseg"] - 1) * p["seg_rows"] + H2) // p["EH"])
    p["items"] = p["nstrips"] * p["nseg"]
    return p


def table_plan(kind, Nw, ms, Na, N0, N1, coff=0):
    """The cross table's plan of a match over output rows 0..N0-1, columns coff..coff+N1-1."""
    dxX = (ms + Nw + coff - Nw) & 3
    return plan_of(Na, Nw, ms, N0, N1 + dxX), dxX


def stack(kind, Nw, ms, N0, N1, seed):
    from umpa_b200 import synth
    pad = ms + Nw + (8 if kind == "DFKernel" else 0)
    Na = 26 if Nw == 0 else NA           # the table path needs K^2 Na >= 25 samples per cost
    return synth.speckle_stack(Na, N0 + 2 * pad, N1 + 2 * pad, seed=seed, max_shift=ms, dark_field=kind != "NoDF")


def model(kind, d, Nw, ms, assign="sam"):
    import umpa_b200
    cls = {"NoDF": umpa_b200.UMPAModelNoDF, "DF": umpa_b200.UMPAModelDF, "DFKernel": umpa_b200.UMPAModelDFKernel}[kind]
    m = cls(list(d["sam"]), list(d["ref"]), window_size=Nw, max_shift=ms)
    m.assign_coordinates = assign
    m.sub_pixel_mode = 0
    return m


def match(m, path, ROI=None, step=None, abc=None):
    m.cuda_path = path
    kw = {"abc": abc} if abc is not None else {}
    res = m.match(ROI=ROI, step=step, debug=True, quiet=True, **kw)
    assert m.last_match_info["path"] == path, m.last_match_info
    return res


def compared_cells(res, table_at, cells_at, pixels=None):
    """The cached FP32 costs of a match and the FP64 costs of the same shifts: (i, j, si, sj, got, exp, n_located,
    n_unlocated).  table_at(i, j) -> the pixel's (S, S) FP64 costs; cells_at(i, j, si, sj) -> FP64 costs of those
    cells (arrays).  pixels: boolean mask of the pixels to compare (default all)."""
    err = np.asarray(res["err"])
    sel = np.ones(err.shape, bool) if pixels is None else pixels
    i, j, si, sj, v = cached_cells({k: res[k] for k in ("debug_d", "dy", "dx")} | {"err": np.where(sel, err, 0)})
    cells, exp = [(i, j, si, sj, v)], [cells_at(i, j, si, sj)]
    located = unlocated = 0
    d = np.asarray(res["debug_d"])
    for a, b in np.argwhere(sel & (err != 1) & (d != -1).any(axis=2)):
        tab = table_at(a, b)
        c = locate_centre(d[a, b], tab)
        if c is None:
            unlocated += 1
            continue
        located += 1
        h = (tab.shape[0] - 1) // 2
        t = np.nonzero(d[a, b] != -1)[0]
        cs, ct = c[0] + t // 5 - 2, c[1] + t % 5 - 2
        cells.append((np.full(t.size, a), np.full(t.size, b), cs, ct, d[a, b, t]))
        exp.append(tab[cs + h, ct + h])
    return tuple(np.concatenate(c) for c in zip(*cells)) + (np.concatenate(exp), located, unlocated)


def df_tolerance(tables64, tables32):
    """Relative tolerance of df at the integer shift: 1e-5, or ten times the largest deviation the FP32 model of the
    table algebra itself has at the FP64 cost minima of the case, where that is larger.  The dark-field fit solves a
    2x2 system whose determinant t2 t3 - t6^2 is small for small windows, so df amplifies the FP32 noise of the sums
    (Nw 1: the model alone deviates by up to ~6e-5; the kernels sum in another order, so the factor 10)."""
    c64, _, D64 = tables64
    D32 = tables32[2]
    k = c64.reshape(-1, *c64.shape[2:]).argmin(axis=0)
    S = c64.shape[0]
    I, J = np.indices(k.shape)
    e = np.abs(D32[k // S, k % S, I, J] - D64[k // S, k % S, I, J]) / np.abs(D64[k // S, k % S, I, J])
    return max(1e-5, 10 * float(e.max()))


def check_lazy(res, lazy, kind, label, df_tol=1e-5):
    """T and df at the integer shift against the FP64 lazy path, on the pixels whose walks agree: T within 1e-5
    relative, df within df_tol."""
    same = (res["err"] == 1) & (lazy["err"] == 1) & (res["debug_Ncalls"] == lazy["debug_Ncalls"]) \
        & (res["dx"] == lazy["dx"]) & (res["dy"] == lazy["dy"])
    assert same.sum() >= .9 * (lazy["err"] == 1).sum(), f"{label}: walks differ in {(~same & (lazy['err'] == 1)).sum()} px"
    for k, tol in (("T", 1e-5), ("df", df_tol)) if kind == "DF" else (("T", 1e-5),):
        rel = np.abs(res[k] - lazy[k])[same] / np.abs(lazy[k])[same]
        assert not (rel > tol).any(), f"{label}: {k} off by {rel.max():.3g} relative to the lazy path (tolerance {tol:.3g})"


def run_cost_tables_case(kind, Nw, ms, N0, N1, coff=0, seed=0, label=""):
    """NoDF / DF, assign 'sam': every cached cost of the table path against cost_tables(float64), the FP32 model on
    the same cells, T / df against the lazy path.  Returns (max, p999) of the cost ratio."""
    d = stack(kind, Nw, ms, N0, N1 + coff, seed)
    m = model(kind, d, Nw, ms)
    ROI = ((0, N0, 1), (coff, coff + N1, 1))
    res = match(m, "table", ROI)
    t64 = cost_tables(d["sam"], d["ref"], Nw, ms, kind == "DF", np.float64)
    t32 = cost_tables(d["sam"], d["ref"], Nw, ms, kind == "DF", np.float32)
    c64, c32 = t64[0], t32[0]
    h = ms - 1
    scale = float(np.median(c64))
    i, j, si, sj, got, exp, located, unlocated = compared_cells(
        res, lambda a, b: c64[:, :, a, b + coff], lambda i, j, si, sj: c64[si + h, sj + h, i, j + coff])
    ok = (res["err"] == 1).mean()
    if ms >= 3:
        assert ok >= .9, f"{label}: only {ok:.3f} of the pixels finished"
        assert got.size >= 10 * N0 * N1, f"{label}: {got.size} cells"
    else:
        assert got.size >= N0 * N1 and unlocated <= .1 * located, f"{label}: {got.size} cells, {unlocated} unlocated"
    st = check_costs(got, exp, scale, label, rows=i)
    # the FP32 model of the same algebra meets the bound on the same cells
    check_costs(c32[si + h, sj + h, i, j + coff], c64[si + h, sj + h, i, j + coff], scale, label + " (FP32 model)")
    check_lazy(res, match(m, "lazy", ROI), kind, label, df_tolerance(t64, t32) if kind == "DF" else None)
    print(f"{label}: {got.size} cells ({located} px located, {unlocated} not), max {st[0]:.3g}, p99.9 {st[1]:.3g}")
    return st


def choose_size(Nw, ms, Na):
    """The first (N0, N1) whose default plan has several strips, a ragged last strip, several segments and a ragged
    last segment."""
    for N0, N1 in TAB_SIZES:
        p, dxX = table_plan("DF", Nw, ms, Na, N0, N1)
        if p["nstrips"] > 1 and (N1 + dxX) % p["TW"] and p["nseg"] > 1 and N0 % p["seg_rows"]:
            return N0, N1, p
    raise AssertionError(f"no size in {TAB_SIZES} gives Nw {Nw} max_shift {ms} ragged strips and segments")


# ---------------------------------------------------------------------------------------------------------------------
# 1 (a): every filtered shift-table instantiation (S = 3 ... 19 x Nw = 0 ... 6), NoDF and DF, default plans

SWEEP = [(kind, Nw, ms) for kind in ("NoDF", "DF") for Nw in range(7) for ms in range(2, 11) if not (kind == "DF" and Nw == 0)]


@pytest.mark.parametrize("kind,Nw,ms", SWEEP)
def test_table_costs_equal_fp64(kind, Nw, ms):
    Na = 26 if Nw == 0 else NA
    N0, N1, p = choose_size(Nw, ms, Na)
    assert Na % p["FB"], p                        # the last box of a pass is partial
    run_cost_tables_case(kind, Nw, ms, N0, N1, seed=10 * Nw + ms, label=f"{kind} Nw {Nw} max_shift {ms} plan {p}")


def test_default_plans_can_have_more_items_than_ctas():
    """One default plan with more items (strips x segments) than CTAs: a CTA works through several items, and the
    frame ring runs on across them."""
    kind, Nw, ms, N0, N1 = "NoDF", 0, 3, 250, 330
    p, _ = table_plan(kind, Nw, ms, 26, N0, N1)
    assert p["order"] == 0 and p["items"] > sm_count(), p
    run_cost_tables_case(kind, Nw, ms, N0, N1, seed=7, label=f"{kind} Nw {Nw} max_shift {ms} plan {p}")


# 1 (d): unaligned ROI origins -- the table origin moves left by dxX = (ox - Nw) & 3 (cross table) and dxM = ox & 3
# (mean table); column offsets 0 ... 3 give both every residue

@pytest.mark.parametrize("ms", [5, 7, 10])
@pytest.mark.parametrize("coff", [0, 1, 2, 3])
def test_table_costs_equal_fp64_unaligned_roi(ms, coff):
    Nw = 2
    N0, N1, _ = choose_size(Nw, ms, NA)
    run_cost_tables_case("DF", Nw, ms, N0, N1, coff=coff, seed=3, label=f"DF Nw {Nw} max_shift {ms} column offset {coff}")


# ---------------------------------------------------------------------------------------------------------------------
# 1 (b), (c): assign_coordinates 'ref' and DFKernel, against the direct FP64 cost on a pixel sample

def direct_case(kind, Nw, ms, assign, N0, N1, step=1, seed=0, boundary_cols=(), boundary_rows=(), n_extra=24):
    from oracle import port
    from umpa_b200 import synth
    d = stack(kind, Nw, ms, (N0 - 1) * step + 1, (N1 - 1) * step + 1, seed)
    m = model(kind, d, Nw, ms, assign)
    abc = synth.blur_abc(N0, N1) if kind == "DFKernel" else None
    res = match(m, "table", step=step if step > 1 else None, abc=abc)
    assert res["err"].shape == (N0, N1)
    o = port.OracleModel(kind, list(d["sam"]), list(d["ref"]), window_size=Nw, max_shift=ms)
    o.set_options(sub_pixel_mode=0, reference_shift=int(assign == "ref"))
    h, pad = ms - 1, o.padding
    args = lambda a, b: () if abc is None else abc[a, b]
    cost = lambda a, b, s, t: o.cost(pad + step * a, pad + step * b, s, t, args(a, b))[0][0]
    table_at = lambda a, b: np.array([[cost(a, b, s, t) for t in range(-h, h + 1)] for s in range(-h, h + 1)])
    cells_at = lambda i, j, si, sj: np.array([cost(*c) for c in zip(i, j, si, sj)])
    sel = np.zeros((N0, N1), bool)
    sel[[0, 1, N0 - 2, N0 - 1], :] = True
    sel[:, [0, N1 - 1]] = True
    for c in boundary_cols:
        sel[:, [c for c in (c - 1, c) if 0 <= c < N1]] = True
    for r in boundary_rows:
        sel[[r for r in (r - 1, r) if 0 <= r < N0], :] = True
    rng = np.random.default_rng(seed)
    sel[rng.integers(0, N0, n_extra), rng.integers(0, N1, n_extra)] = True
    i, _, _, _, got, exp, located, unlocated = compared_cells(res, table_at, cells_at, pixels=sel)
    # cost scale: the median FP64 cost over all shifts of a few pixels
    scale = float(np.median([table_at(a, b) for a, b in zip(rng.integers(0, N0, 6), rng.integers(0, N1, 6))]))
    label = f"{kind} Nw {Nw} max_shift {ms} assign {assign} step {step}"
    if ms >= 3:
        assert (res["err"] == 1).mean() >= .9, f"{label}: {(res['err'] == 1).mean():.3f} finished"
        assert got.size >= 10 * sel.sum(), f"{label}: {got.size} cells"
    else:
        assert got.size >= sel.sum() and unlocated <= .1 * located, f"{label}: {got.size} cells, {unlocated} unlocated"
    st = check_costs(got, exp, scale, label, rows=i)
    df_tol = None
    if kind == "DF":          # (the FP32 model of assign_coordinates 'sam' on the same stack: the same sums)
        df_tol = df_tolerance(*(cost_tables(d["sam"], d["ref"], Nw, ms, True, t) for t in (np.float64, np.float32)))
    check_lazy(res, match(m, "lazy", step=step if step > 1 else None, abc=abc), kind, label, df_tol)
    print(f"{label}: {got.size} cells of {int(sel.sum())} px, max {st[0]:.3g}, p99.9 {st[1]:.3g}")
    return st


REF_CASES = [(kind, Nw, ms) for kind in ("NoDF", "DF") for ms in (5, 7, 10) for Nw in (1, 4, 6)]


@pytest.mark.parametrize("kind,Nw,ms", REF_CASES)
def test_table_costs_equal_fp64_assign_ref(kind, Nw, ms):
    N0, N1, p = choose_size(Nw, ms, NA)
    dxX = (ms + Nw - Nw) & 3
    direct_case(kind, Nw, ms, "ref", N0, N1, seed=ms + Nw,
                boundary_cols=[k * p["TW"] - dxX for k in range(1, p["nstrips"])],
                boundary_rows=[k * p["seg_rows"] for k in range(1, p["nseg"])])


# the blur-table kernels of UMPAModelDFKernel (kernel_path.cu: ktable_pick)
KTABLE = [(1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (2, 2), (2, 3), (2, 4), (2, 5), (2, 6), (3, 2), (3, 3), (3, 4), (3, 5)]


@pytest.mark.parametrize("assign", ["sam", "ref"])
@pytest.mark.parametrize("Nw,ms", KTABLE)
def test_blur_table_costs_equal_fp64(Nw, ms, assign):
    """Every blur-table instantiation, step 1 and step 2 (where the kernel's shared memory allows a step > 1: the
    table path reports 'outside the instantiated blur-table kernels' otherwise)."""
    from umpa_b200 import _capi
    direct_case("DFKernel", Nw, ms, assign, 23, 29, seed=Nw + 3 * ms)
    try:
        direct_case("DFKernel", Nw, ms, assign, 17, 19, step=2, seed=Nw + 3 * ms + 1, n_extra=8)
    except _capi.UmpaError as e:
        assert "blur-table" in str(e), e
        print(f"DFKernel Nw {Nw} max_shift {ms} assign {assign}: no blur-table kernel for step 2")


# ---------------------------------------------------------------------------------------------------------------------
# 2: every tile plan returns the same bits.  Nothing in the arithmetic of a table entry depends on the plan: frame
# order, tap order and FFMA2 pairing are fixed by S and Nw, strips are TW wide whatever the plan, carry values are
# copies of the row-filtered values, and the zero-filled rows above a segment feed only rows that are never stored.

FORCED = [(7, 0), (9, 2), (5, 6), (15, 3), (19, 6)]      # (S, Nw): no halo, config 2's kernel, 8-row chunks < 2 Nw,
#                                                           pass-major on a BIG kernel, SH = 1
FORCED_SIZE = (53, 75)                                   # NSEG 4: segments of 14 rows, the last one of 11
MAPS = ("f", "T", "dx", "dy", "df", "err", "debug_Ncalls", "debug_d")


def forced_settings(Nw):
    out = [{"UMPA_TAB_EH": eh, "UMPA_TAB_STREAM": o} for eh in (8, 16, 24, 32, 48) for o in ((0, 1, 2) if Nw else (0,))]
    out += [{"UMPA_TAB_G": 1}, {"UMPA_TAB_FB": 1}, {"UMPA_TAB_FB": 2}, {"UMPA_TAB_NST": 2},
            {"UMPA_TAB_NSEG": 1}, {"UMPA_TAB_NSEG": 4}, {"UMPA_TAB_NSEG": 1000}, {"UMPA_TAB_CTAS": 2}]
    return out


def forced_plan_matches(p, env, Na, rows):
    """An accepted plan is the forced one."""
    want = {"EH": env.get("UMPA_TAB_EH"), "order": env.get("UMPA_TAB_STREAM"), "G": env.get("UMPA_TAB_G"),
            "nstage": env.get("UMPA_TAB_NST")}
    if "UMPA_TAB_FB" in env:
        want["FB"] = min(env["UMPA_TAB_FB"], Na)
    if "UMPA_TAB_CTAS" in env:
        want["EH"] = 8
    if "UMPA_TAB_NSEG" in env and p["order"]:
        want["nseg"] = math.ceil(rows / math.ceil(rows / env["UMPA_TAB_NSEG"]))
    for k, v in want.items():
        assert v is None or p[k] == v, (env, k, p)


def test_every_tile_plan_returns_the_same_bits(monkeypatch):
    from umpa_b200 import _capi
    ledger = []
    N0, N1 = FORCED_SIZE
    for S, Nw in FORCED:
        ms = (S + 1) // 2
        kind = "DF" if Nw else "NoDF"
        Na = 26 if Nw == 0 else NA
        d = stack(kind, Nw, ms, N0, N1, seed=S)
        m = model(kind, d, Nw, ms)
        base = match(m, "table")
        fp64 = None
        if (S, Nw) == (5, 6):
            c64, _, _ = cost_tables(d["sam"], d["ref"], Nw, ms, True, np.float64)
            h = ms - 1
            fp64 = (lambda a, b: c64[:, :, a, b], lambda i, j, si, sj: c64[si + h, sj + h, i, j], float(np.median(c64)))
        rejected = 0
        for env in forced_settings(Nw):
            for k, v in env.items():
                monkeypatch.setenv(k, str(v))
            p, _ = table_plan(kind, Nw, ms, Na, N0, N1)
            label = f"S {S} Nw {Nw} {env}"
            if p is None:
                rejected += 1
                if rejected == 1:                     # a match under a rejected plan fails cleanly
                    with pytest.raises(_capi.UmpaError, match="table path: "):
                        match(m, "table")
            else:
                forced_plan_matches(p, env, Na, N0)
                got = match(m, "table")
                if fp64 is not None:
                    i, _, _, _, g, e, _, _ = compared_cells(got, fp64[0], fp64[1])
                    check_costs(g, e, fp64[2], label, rows=i)
                for k in MAPS:
                    if k in base:
                        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(base[k]).view(np.uint8)), \
                            f"{label}: {k} differs from the default plan's in {int((got[k] != base[k]).sum())} entries"
                ledger.append((S, Nw, tuple(sorted(env.items())), p))
            for k in env:
                monkeypatch.delenv(k)
    for S, Nw, env, p in ledger:
        print(f"S {S:2d} Nw {Nw} {dict(env)}: EH {p['EH']} order {p['order']} G {p['G']} npass {p['npass']} FB {p['FB']} "
              f"nstage {p['nstage']} strips {p['nstrips']} nseg {p['nseg']} chunks {p['nchunk_full']}/{p['nchunk_last']} "
              f"items {p['items']}")
    plans = [p for *_, p in ledger]
    assert {p["order"] for p in plans} == {0, 1, 2}
    assert {p["EH"] for p in plans} == {8, 16, 24, 32, 48}
    assert any((26 if Nw == 0 else NA) % p["FB"] for _, Nw, _, p in ledger)
    assert any(p["nseg"] > 1 and p["nchunk_last"] < p["nchunk_full"] for p in plans)
    grid = sm_count()
    assert any(p["items"] > grid * (2 if ("UMPA_TAB_CTAS", 2) in env else 1) for _, _, env, p in ledger)
