"""CPU: the algebraic regrouping behind the table path is exact.

tests/table_algebra.py evaluates every shift's cost the way the CUDA kernels do (centred frames,
frame-summed unwindowed correlation + ONE separable window filter per shift, per-frame filtered
images for the mean term, FP64 solve).  In float64 it must reproduce the oracle's direct
evaluation to rounding; in float32 it bounds the error the kernels can have."""
import numpy as np
import pytest

from helpers import cached_cells, check_costs, load_case, locate_centre
from oracle import port
from table_algebra import cost_tables


@pytest.mark.parametrize("name", ["nodf_clean", "df_clean", "df_lowcontrast", "df_nw3_ms6"])
def test_regrouped_cost_equals_direct(name):
    c = load_case(name)
    sam, ref = np.array(c["sam"]), np.array(c["ref"])
    df = c["kind"] == "DF"
    o = port.OracleModel(c["kind"], c["sam"], c["ref"], window_size=c["Nw"], max_shift=c["max_shift"])
    h, p = c["max_shift"] - 1, c["padding"]
    N0, N1 = o.extent
    cost64, T64, D64 = cost_tables(sam, ref, c["Nw"], c["max_shift"], df, np.float64)
    cost32, T32, D32 = cost_tables(sam, ref, c["Nw"], c["max_shift"], df, np.float32)
    rng = np.random.default_rng(0)
    scale = np.median(cost64)
    for _ in range(60):
        i, j = int(rng.integers(0, N0)), int(rng.integers(0, N1))
        si, sj = int(rng.integers(-h, h + 1)), int(rng.integers(-h, h + 1))
        (f, t, v), st = o.cost(p + i, p + j, si, sj)
        assert st == 1
        assert abs(cost64[si + h, sj + h, i, j] - f) <= 1e-12 * max(scale, abs(f))
        assert abs(T64[si + h, sj + h, i, j] - t) <= 1e-11 * abs(t)
        if df:
            assert abs(D64[si + h, sj + h, i, j] - v) <= 1e-10 * max(1., abs(v))
        # FP32 accumulation: error stays at the 1e-5 level of the cost scale
        assert abs(cost32[si + h, sj + h, i, j] - f) <= 3e-5 * scale


@pytest.mark.parametrize("refshift", [0, 1])
def test_dfkernel_blur_table_identities(refshift):
    """The blur-table form of DFKernel's cost (kernel_path.cu): blurred CENTRED reference patch once per
    pixel, t3 / t5 rebuilt from the centred sums and the frame constants -- for assign_coordinates='sam'
    (the blurred window moves over the patch) and 'ref' (the blurred window stays, the sample window moves
    by -s; Model.cpp:1045-1051).  FP64 numpy against the oracle's direct evaluation."""
    c = load_case("dfk_assign_ref" if refshift else "dfk_roi_step")
    sam, ref = np.array(c["sam"]), np.array(c["ref"])
    Nw, ms, pad = c["Nw"], c["max_shift"], c["padding"]
    K, h = 2 * Nw + 1, ms - 1
    o = port.OracleModel("DFKernel", c["sam"], c["ref"], window_size=Nw, max_shift=ms)
    o.set_options(reference_shift=refshift)
    w = port.make_window(Nw)
    sw = w.sum()
    ck, dk = ref.mean(axis=(1, 2)), sam.mean(axis=(1, 2))         # any constants do
    Rc, Sc = ref - ck[:, None, None], sam - dk[:, None, None]
    cd, cc, dd = (ck * dk).sum(), (ck * ck).sum(), (dk * dk).sum()
    rng = np.random.default_rng(3)
    for _ in range(12):
        i, j = (int(rng.integers(pad, sam.shape[1] - pad)), int(rng.integers(pad, sam.shape[2] - pad)))
        abc = tuple(rng.uniform(.2, .8, 2)) + (float(rng.uniform(.2, .8)),)
        abc = (abc[0], float(rng.uniform(-.1, .1)), abc[2])
        kern = port.blur_kernel(*abc).reshape(17, 17)
        sig = kern.sum()
        win = lambda img, y, x: img[:, y - Nw:y + Nw + 1, x - Nw:x + Nw + 1]   # (Na, K, K) window at (y, x)
        # blurred centred reference on the patch the shifts can reach
        P = K + 2 * h
        Bp = np.zeros((len(ref), P, P))
        for y in range(P):
            for x in range(P):
                qy, qx = i - Nw - h + y, j - Nw - h + x
                Bp[:, y, x] = (Rc[:, qy - 8:qy + 9, qx - 8:qx + 9] * kern).sum(axis=(1, 2))
        for si in (-h, -1, 0, 2):
            for sj in (-2, 0, 1, h):
                (f, t, _), st = o.cost(i, j, si, sj, abc)
                assert st == 1
                if refshift:        # reference window at the pixel, sample window at p - s
                    Bw = Bp[:, h:h + K, h:h + K]
                    Sw, Sr = win(Sc, i - si, j - sj), win(sam, i - si, j - sj)
                else:               # blurred window at p + s, sample window at the pixel
                    Bw = Bp[:, h + si:h + si + K, h + sj:h + sj + K]
                    Sw, Sr = win(Sc, i, j), win(sam, i, j)
                t5c = (w * Bw * Sr).sum()
                t3c = (w * (Bw * Bw + 2. * sig * ck[:, None, None] * Bw)).sum()
                V = (ck[:, None, None] * w * Sw).sum()
                T1, P1 = (w * Sw * Sw).sum(), (dk[:, None, None] * w * Sw).sum()
                t1 = T1 + 2. * P1 + sw * dd
                t5 = t5c + sig * (V + sw * cd)
                t3 = t3c + sig * sig * sw * cc
                T = t5 / t3
                cost = (t1 - t5 * T) / len(ref)
                assert abs(T - t) <= 1e-11 * abs(t)
                assert abs(cost - f) <= 1e-11 * max(abs(f), t1 / len(ref) * 1e-3)


@pytest.mark.parametrize("kind", ["NoDF", "DF"])
def test_binary_shared_mask_is_the_unmasked_sums_minus_the_dead_window_positions(kind):
    """What table_path.cu's masked_walk_kernel computes for a 0 / 1 mask shared by all frames: the UNMASKED sums of a
    cost evaluation (Model.cpp:415-458 / 709-773; the tables hold them) minus the window positions at which either
    window sees a dead pixel, with t2 and wt scaled by the live window weight -- against the oracle's masked branch
    (Model.cpp:461-499, 775-847).  The frame's reference mean m_k stays unmasked, as in the reference."""
    rng = np.random.default_rng(5)
    Na, H, W, Nw, ms = 6, 40, 44, 2, 4
    S = 1. + .3 * rng.standard_normal((Na, H, W))
    R = 1. + .3 * rng.standard_normal((Na, H, W))
    M = (rng.random((H, W)) > .05).astype(np.float64)
    win = port.make_window(Nw)
    sw = win.sum()
    om = port.OracleModel(kind, list(S), list(R), mask_list=[M] * Na, window_size=Nw, max_shift=ms)
    for _ in range(200):
        i = int(rng.integers(om.padding, H - om.padding)); j = int(rng.integers(om.padding, W - om.padding))
        si, sj = (int(v) for v in rng.integers(-ms + 1, ms, 2))
        qi, qj = i + si, j + sj
        ws = S[:, i - Nw:i + Nw + 1, j - Nw:j + Nw + 1]
        wr = R[:, qi - Nw:qi + Nw + 1, qj - Nw:qj + Nw + 1]
        mk = (win * wr).sum((1, 2)) / sw
        t1, t3, t5 = (win * ws * ws).sum(), (win * wr * wr).sum(), (win * wr * ws).sum()
        t2, t4, t6 = (mk ** 2).sum(), (mk * (win * ws).sum((1, 2))).sum(), (mk * (win * wr).sum((1, 2))).sum()
        dead = (M[qi - Nw:qi + Nw + 1, qj - Nw:qj + Nw + 1] == 0) | (M[i - Nw:i + Nw + 1, j - Nw:j + Nw + 1] == 0)
        cw = 0.
        for a, b in np.argwhere(dead):
            w, s, r = win[a, b], ws[:, a, b], wr[:, a, b]
            cw += w
            t1 -= w * (s * s).sum(); t3 -= w * (r * r).sum(); t5 -= w * (r * s).sum()
            t4 -= w * (mk * s).sum(); t6 -= w * (mk * r).sum()
        t2 *= sw - cw
        wt = Na * (sw - cw)
        if kind == "NoDF":
            t = t5 / t3
            f, v = (t1 - t5 * t) / wt, 0.
        else:
            den = t2 * t3 - t6 * t6
            Kc, beta = (t2 * t5 - t4 * t6) / den, (t3 * t4 - t5 * t6) / den
            t, v = beta + Kc, Kc / (beta + Kc)
            f = (t1 - beta * t4 - Kc * t5) / wt
        (fo, to, vo), st = om.cost(i, j, si, sj)
        assert st == 1
        assert abs(f - fo) <= 1e-11 * abs(fo) and abs(t - to) <= 1e-11 * abs(to) and abs(v - vo) <= 1e-10 * max(1., abs(vo))


MAPPING_CASES = [("DF", 2, 4, "sam"), ("NoDF", 1, 3, "sam"), ("NoDF", 0, 5, "sam"), ("NoDF", 0, 3, "ref"), ("DF", 1, 2, "sam"),
                 ("DF", 2, 4, "ref"), ("NoDF", 1, 3, "ref"), ("DFKernel", 1, 3, "sam"), ("DFKernel", 2, 2, "ref")]


def _oracle_match(kind, Nw, ms, assign, Na=6, H=40, W=44, seed=3):
    from umpa_b200 import synth
    Na = 26 if Nw == 0 else Na
    pad = 8 if kind == "DFKernel" else 0
    d = synth.speckle_stack(Na, H + 2 * pad, W + 2 * pad, seed=seed, max_shift=ms, dark_field=kind != "NoDF")
    o = port.OracleModel(kind, list(d["sam"]), list(d["ref"]), window_size=Nw, max_shift=ms)
    o.set_options(sub_pixel_mode=0, reference_shift=int(assign == "ref"))
    N0, N1 = o.extent
    abc = synth.blur_abc(N0, N1) if kind == "DFKernel" else None
    return d, o, abc, o.match(abc=abc)


@pytest.mark.parametrize("kind,Nw,ms,assign", MAPPING_CASES)
def test_walk_cache_maps_to_shifts(kind, Nw, ms, assign):
    """What tests/test_gpu_table_costs.py relies on to read the costs a match used: with sub_pixel_mode = 0 the
    reference's walk returns its integer centre (dy, dx) = (c0, c1), and cell t of its 5x5 cache holds the cost of the
    shift (c0 + t // 5 - 2, c1 + t % 5 - 2) -- the FP64 cost tables (assign_coordinates 'sam') or the direct cost
    (any model).  max_shift 2: no pixel can complete its 4x4 block (err == 0), and locate_centre() finds the centre
    from the cached values."""
    d, o, abc, r = _oracle_match(kind, Nw, ms, assign)
    h, p = ms - 1, o.padding
    ok = r["err"] == 1
    if ms == 2:
        assert not ok.any()
    else:
        assert ok.mean() > .9
    direct = kind == "DFKernel" or assign == "ref"
    cost = lambda a, b, s, t: o.cost(p + a, p + b, s, t, () if abc is None else abc[a, b])[0][0]
    if not direct:
        c64, _, _ = cost_tables(d["sam"], d["ref"], Nw, ms, kind == "DF", np.float64)
    if ms == 2:                                     # centres from the cached values
        cells = []
        for a, b in np.argwhere(~ok)[::8 if direct else 1]:
            tab = c64[:, :, a, b] if not direct else np.array([[cost(a, b, s, t) for t in range(-h, h + 1)]
                                                                for s in range(-h, h + 1)])
            c = locate_centre(r["debug_d"][a, b], tab)
            assert c is not None, (a, b)
            cells += [(r["debug_d"][a, b, n], tab[c[0] + n // 5 - 2 + h, c[1] + n % 5 - 2 + h])
                      for n in np.nonzero(r["debug_d"][a, b] != -1)[0]]
        v, e = np.array(cells).T
    else:
        i, j, si, sj, v = cached_cells(r)
        if not direct:
            e = c64[si + h, sj + h, i, j]
        else:
            sel = np.arange(0, v.size, max(1, v.size // 400))    # the direct evaluation is slow for DFKernel
            v = v[sel]
            e = np.array([cost(*c) for c in zip(i[sel], j[sel], si[sel], sj[sel])])
    scale = np.median(e)
    assert v.size >= 100
    np.testing.assert_array_less(np.abs(v - e), 1e-10 * scale)


def test_cost_comparator_has_teeth(monkeypatch):
    """check_costs (the FP64 comparison of tests/test_gpu_table_costs.py) on the cells a walk reads: it passes the FP32
    restatement of the table algebra, and fails a table that lost one frame and one whose column filter reads one tap
    a row too low."""
    import table_algebra
    kind, Nw, ms = "DF", 2, 4
    d, o, _, r = _oracle_match(kind, Nw, ms, "sam", Na=11)
    i, j, si, sj, v = cached_cells(r)
    h = ms - 1
    c64, _, _ = cost_tables(d["sam"], d["ref"], Nw, ms, True, np.float64)
    scale = np.median(c64)
    at = lambda c: c[si + h, sj + h, i, j]
    c32, _, _ = cost_tables(d["sam"], d["ref"], Nw, ms, True, np.float32)
    mx, _ = check_costs(at(c32), at(c64), scale, "float32 model")
    assert mx > 0
    dropped, _, _ = cost_tables(d["sam"][:-1], d["ref"][:-1], Nw, ms, True, np.float64)
    with pytest.raises(AssertionError, match="costs off by"):
        check_costs(at(dropped), at(c64), scale, "frame dropped")

    def moved_tap(img, g, dtype):                   # table_algebra._filt, but column tap 0 reads row 1 instead of row 0
        K = len(g)
        H, W = img.shape[-2:]
        tmp = np.zeros(img.shape[:-1] + (W - K + 1,), dtype=dtype)
        for u in range(K):
            tmp = (tmp + g[u] * img[..., :, u:u + W - K + 1]).astype(dtype)
        out = np.zeros(img.shape[:-2] + (H - K + 1, W - K + 1), dtype=dtype)
        for u in range(K):
            r = u + (u == 0)
            out = (out + g[u] * tmp[..., r:r + H - K + 1, :]).astype(dtype)
        return out
    monkeypatch.setattr(table_algebra, "_filt", moved_tap)
    moved, _, _ = table_algebra.cost_tables(d["sam"], d["ref"], Nw, ms, True, np.float64)
    with pytest.raises(AssertionError, match="costs off by"):
        check_costs(at(moved), at(c64), scale, "tap moved")
