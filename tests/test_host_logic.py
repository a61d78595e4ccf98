"""CPU: host-side logic (geometry / ROI / step, window, sharding arithmetic) and the C-ABI surface."""
import ctypes
import os
import re

import numpy as np
import pytest

from helpers import golden_names, load_case
from umpa_b200.geometry import Geometry
from umpa_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAFE_CROP = {"NoDF": 0, "DF": 0, "DFKernel": 8}


def _geo(c):
    shapes = [s.shape for s in c["sam"]]
    pos = c["pos"] if c["pos"] is not None else [(0, 0)] * len(shapes)
    return Geometry(shapes, pos, c["max_shift"] + c["Nw"] + SAFE_CROP[c["kind"]])


@pytest.mark.parametrize("name", golden_names())
def test_geometry_matches_reference(name):
    """extent, the ROI the reference ended up with after match(step=/ROI=), and its output shape."""
    c = load_case(name)
    g = _geo(c)
    assert g.padding == c["padding"]
    assert g.extent() == tuple(int(v) for v in c["extent"])
    s0, s1 = g.match_roi(ROI=c["ROI"], step=c["step"])
    assert (s0, s1) == tuple(tuple(int(v) for v in r) for r in c["ROI_after"])
    assert g.ROI == (s0, s1)                      # sticky (model.pyx:406)
    assert g.sh == tuple(int(v) for v in c["sh_after"]) == c["expected"]["err"].shape


def test_roi_semantics():
    g = Geometry([(40, 44)] * 3, [(0, 0)] * 3, 6)
    assert g.ROI == ((0, 28, 1), (0, 32, 1))
    assert g.convert(ROI=(slice(2, 20, 2), slice(None, None, 3))) == ((2, 20, 2), (0, 32, 3))
    with pytest.raises(RuntimeError):
        g.convert(ROI=((0, 4, 1), (0, 4, 1)), step=2)        # model.pyx:566-568
    assert g.match_roi(ROI=((1, 9, 2), (0, 8, 1)), step=5) == ((1, 9, 2), (0, 8, 1))   # step ignored, 372-375
    assert g.set_step(3) == ((1, 9, 3), (0, 8, 3))           # re-slices the STORED ROI (576-580)
    assert g.sh == (3, 3)
    r, c = g.coords()
    assert list(r) == [7, 10, 13] and list(c) == [6, 9, 12]
    assert Geometry.shape_of((5, 5, 1), (0, 3, 1)) == (0, 3)


def test_window_is_the_reference_window():
    from oracle import port
    c = load_case("df_nw3_ms6")
    np.testing.assert_allclose(port.make_window(3), c["window"], rtol=0, atol=1e-16)


def test_row_bands():
    for n, w in ((2034, 8), (10, 4), (3, 8), (28, 1)):
        b = sharding.row_bands(n, w)
        assert len(b) == w and b[0][0] == 0 and b[-1][1] == n
        assert all(b[k][1] == b[k + 1][0] for k in range(w - 1))
        sizes = [y - x for x, y in b]
        assert max(sizes) - min(sizes) <= 1
    assert sharding.band_input_rows((10, 20), 7) == (10, 34)


def test_capi_exports_every_declared_symbol():
    """The C-ABI library loads without a GPU and exports what include/umpa_b200.h declares."""
    from umpa_b200 import _capi, build
    build.build()
    lib = ctypes.CDLL(_capi.LIB_PATH)
    hdr = open(os.path.join(ROOT, "include", "umpa_b200.h")).read()
    declared = set(re.findall(r"UMPA_API[^;(]*?\b(umpa_[a-z0-9_]+)\s*\(", hdr))
    assert declared and declared == set(_capi.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    L = _capi.lib()
    assert b"sm_100a" in L.umpa_version()


def test_product_does_not_import_oracle():
    """The product path may not route through the oracle (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "umpa_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
    for fn in os.listdir(os.path.join(pkg, "csrc")):
        if fn.endswith((".cu", ".cuh")):
            assert "oracle" not in open(os.path.join(pkg, "csrc", fn)).read(), fn


def test_host_staging_helpers():
    """hoststage.cu without a GPU: the conversion is (float)(x - c) exactly (AVX2 and scalar tails, padded
    pitch, unaligned destinations), the sampled mean is the mean of rows 0, step, 2 step, ..."""
    import ctypes as C
    from umpa_b200 import _capi
    L = _capi.lib()
    rng = np.random.default_rng(0)
    for rows, W, pitch, off in ((7, 64, 64, 0), (5, 37, 40, 0), (3, 129, 132, 3), (1, 5, 8, 1)):
        src = rng.normal(3., 2., (rows, W))
        buf = np.full(rows * pitch + 8, np.float32(-7.), dtype=np.float32)
        dst = buf[off:off + rows * pitch]
        c = 2.9375 + 1e-9
        L.umpa_host_center_rows(dst.ctypes.data_as(C.POINTER(C.c_float)), src.ctypes.data_as(C.POINTER(C.c_double)),
                                rows, W, pitch, c)
        out = dst.reshape(rows, pitch)
        np.testing.assert_array_equal(out[:, :W], (src - c).astype(np.float32))
        assert np.all(out[:, W:] == 0) and np.all(buf[:off] == -7) and np.all(buf[off + rows * pitch:] == -7)
        # float32 source rows (pageable float32 frames): widened, centred, rounded once
        src32 = src.astype(np.float32)
        buf[:] = -7.
        L.umpa_host_center_rows_f32(dst.ctypes.data_as(C.POINTER(C.c_float)), src32.ctypes.data_as(C.POINTER(C.c_float)),
                                    rows, W, pitch, c)
        np.testing.assert_array_equal(out[:, :W], (src32.astype(np.float64) - c).astype(np.float32))
        assert np.all(out[:, W:] == 0) and np.all(buf[:off] == -7) and np.all(buf[off + rows * pitch:] == -7)
    # a NaN / Inf pixel on a sampled row counts as 0: the constant stays finite (any constant is valid)
    bad = rng.normal(1., .5, (64, 50))
    good = bad.copy()
    bad[32, 7], bad[0, 49] = np.nan, np.inf
    good[32, 7] = good[0, 49] = 0.
    assert (L.umpa_host_sampled_mean(bad.ctypes.data_as(C.POINTER(C.c_double)), 64, 50, 2) ==
            L.umpa_host_sampled_mean(good.ctypes.data_as(C.POINTER(C.c_double)), 64, 50, 2))
    fr = rng.normal(1., .5, (100, 77))
    for step in (1, 3, 32, 1000):
        got = L.umpa_host_sampled_mean(fr.ctypes.data_as(C.POINTER(C.c_double)), 100, 77, step)
        assert abs(got - fr[::step].mean()) < 1e-13
        # float32 frames (umpa_set_frames_f32): the mean of the widened frame, bit for bit
        f32 = fr.astype(np.float32)
        wide = np.ascontiguousarray(f32, dtype=np.float64)
        assert (L.umpa_host_sampled_mean_f32(f32.ctypes.data_as(C.POINTER(C.c_float)), 100, 77, step) ==
                L.umpa_host_sampled_mean(wide.ctypes.data_as(C.POINTER(C.c_double)), 100, 77, step))


def test_bench_algorithmic_flops_match_survey():
    """SURVEY.md 8(d): F_alg per output pixel of the five BASELINE configurations, and the tile model
    bench.py uses for the executed-flop figure agrees with plan_tiles (table_path.cu) on the tile height."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    want = {"cfg1": 24500, "cfg2": 101250, "cfg3": 3648150, "cfg4": 882000, "cfg5": 66248}
    for name, f in want.items():
        assert bench.algorithmic_flops_per_px(bench.CONFIGS[name]) == f, name
    # executed FMAs per output pixel of the cross-table kernel: configs 1, 2, 5 stream 16-row chunks (every chunk row
    # is an output row, 28 / 20 of 32 columns are outputs), config 4 streams 24-row chunks pass by pass (the carry of
    # all 225 shift planes does not fit, that of one pass does)
    assert bench.table_plan(bench.CONFIGS["cfg2"]) == (True, 16) and bench.table_plan(bench.CONFIGS["cfg1"]) == (True, 16)
    assert bench.table_plan(bench.CONFIGS["cfg5"]) == (True, 16) and bench.table_plan(bench.CONFIGS["cfg4"]) == (True, 24)
    S, K, Na = 9, 5, 25
    assert abs(bench.executed_fma_per_px_cross(bench.CONFIGS["cfg2"]) - S * S * ((Na + K) * 32 / 28. + K)) < 1e-9
    e5 = bench.executed_fma_per_px_cross(bench.CONFIGS["cfg5"])
    assert abs(e5 - 49 * ((4 + 13) * 32 / 20. + 13)) < 1e-9
    e4 = bench.executed_fma_per_px_cross(bench.CONFIGS["cfg4"])
    assert abs(e4 - 225 * ((40 + 7) * 32 / 24. + 7)) < 1e-9      # (Nw = 3: 24 of 32 columns are outputs)


def test_table_plan_covers_every_supported_model(monkeypatch):
    """umpa_table_plan (plan_tiles, table_path.cu; host arithmetic): for every window / shift range / stack depth the
    table path accepts, the plan is one the kernel can run -- chunk height from the instantiated set, at least two ring
    stages, the passes cover all S shift rows, the strips cover all columns, pass-major streaming (order 2) only
    where it is compiled (S >= 11) and needed (more than one pass), and a streaming chunk at least as high as its carry
    (2 Nw rows: the next chunk's column pass reads all of them).  The same with 8-row chunks (two CTAs per SM,
    UMPA_TAB_CTAS=2, or UMPA_TAB_EH=8): there Nw 5 and 6 have no plan (a halo tile of 8 rows holds no output row, a
    streaming chunk of 8 rows is shorter than its carry), nor do some of the larger Nw 4 tables (shared memory), and
    the planner says so instead of returning a plan."""
    import ctypes
    from umpa_b200 import _capi
    L = _capi.lib()
    out = (ctypes.c_int * 10)()
    seen = set()
    for ctas, eh in ((None, None), ("2", None), (None, "8"), ("2", "8")):
        for name, v in (("UMPA_TAB_CTAS", ctas), ("UMPA_TAB_EH", eh)):
            if v is None:
                monkeypatch.delenv(name, raising=False)
            else:
                monkeypatch.setenv(name, v)
        short = ctas is not None or eh is not None
        env = (ctas, eh)
        for Nw in range(0, 7):
            for ms in range(1, 11):
                for Na in (1, 4, 25, 40, 120):
                    for rows, cols in ((1, 1), (37, 500), (254, 2034), (4074, 4074)):
                        rc = L.umpa_table_plan(Na, Nw, ms, rows, cols, 148, out)
                        if short and Nw >= 4 and rc != 0:
                            assert rc == -4 and L.umpa_last_error().startswith(b"table path:"), (env, Nw, ms, rc)
                            continue
                        assert rc == 0, (env, Nw, ms, Na, rows, cols, L.umpa_last_error())
                        assert not (short and Nw >= 5), (env, Nw, ms, list(out))
                        EH, order, G, npass, FB, nstage, TW, nseg, nstrips, nt = list(out)
                        S = 2 * ms - 1
                        SH = 3 if S <= 9 else (2 if S <= 17 else 1)
                        assert EH in ((8,) if short else (8, 16, 24, 32, 48)) and order in (0, 1, 2)
                        assert G >= 1 and npass >= 1 and npass * G * SH >= S and (npass - 1) * G * SH < S
                        assert 1 <= FB <= Na and nstage >= 2
                        assert TW == (32 - 2 * Nw) & ~3 and nstrips * TW >= cols > (nstrips - 1) * TW
                        assert nseg >= 1 and nt == G * EH * 8 and nt <= (192 if ctas else 384)
                        if order == 2:
                            assert S >= 11 and npass > 1
                        if order == 0 and Nw > 0:
                            assert EH - 2 * Nw >= 2
                        if order in (1, 2):
                            assert EH >= 2 * Nw, (env, Nw, ms, list(out))
                        seen.add((short, order))
    assert seen == {(s, o) for s in (False, True) for o in (0, 1, 2)}
    assert L.umpa_table_plan(25, 7, 5, 100, 100, 148, out) != 0          # Nw > 6 is not a table model
