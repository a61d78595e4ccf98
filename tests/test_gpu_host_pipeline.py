"""GPU: every route of the pipelined host-to-host match (umpa_match_host, DESIGN §2.4) that a caller can force.

One pipeline serves float64 and float32 host frames: each band's rows go up either directly, in the frames' own
element type, or staged as centred FP32 by host threads.  Which of the two, and where the frames are split, depends on
the element type, on whether the frames are pinned and on UMPA_HOST_THREADS / UMPA_HOST_FRAC.  Every route must
report the split it took, return maps bit-identical to the unpipelined float64 match of the same (widened) frames, and
leave the FP64 stacks ready for the cost() hook (they are completed on demand when some rows crossed as FP32)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MAX_SHIFT = 4
THREADS = 4

# (element type, pinned frames, environment, host threads, staged rows per frame for H rows)
ROUTES = {
    "f64_pinned_split": (np.float64, True, {"UMPA_HOST_THREADS": THREADS, "UMPA_HOST_FRAC": 0.5}, THREADS, lambda H: int(.5 * H)),
    "f64_pinned_frac0": (np.float64, True, {"UMPA_HOST_THREADS": THREADS, "UMPA_HOST_FRAC": 0}, 0, lambda H: 0),
    "f64_pinned_no_threads": (np.float64, True, {"UMPA_HOST_THREADS": 0}, 0, lambda H: 0),
    "f64_pageable": (np.float64, False, {"UMPA_HOST_THREADS": THREADS}, THREADS, lambda H: H),
    "f64_pageable_no_threads": (np.float64, False, {"UMPA_HOST_THREADS": 0}, 0, lambda H: 0),
    "f32_pinned": (np.float32, True, {"UMPA_HOST_THREADS": THREADS}, 0, lambda H: 0),
    "f32_pageable": (np.float32, False, {"UMPA_HOST_THREADS": THREADS}, THREADS, lambda H: H),
    "f32_pageable_no_threads": (np.float32, False, {"UMPA_HOST_THREADS": 0}, 0, lambda H: 0),
}

# 531 x 515: the FP32 rows are padded to a pitch of 516 floats, so float32 rows go up with one 2-D copy per frame
SHAPES = [(700, 640), (531, 515)]


def _frames(seed, H, W, dtype, pinned, Na=8):
    """float32-representable stacks in `dtype`: pinned as one torch allocation per stack, else one array per frame"""
    import torch
    from umpa_b200 import synth
    d = synth.speckle_stack(Na, H, W, seed=seed, max_shift=MAX_SHIFT, dark_field=True)
    out = []
    for x in (d["sam"], d["ref"]):
        x = np.asarray(x, dtype=np.float32).astype(dtype)
        if pinned:
            t = torch.empty(x.shape, dtype=torch.from_numpy(x).dtype, pin_memory=True)
            t.copy_(torch.from_numpy(x))
            out.append(list(t.numpy()))
        else:
            out.append([f.copy() for f in x])
    return out


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("kind", ["DF", "NoDF"])
@pytest.mark.parametrize("route", list(ROUTES))
def test_pipelined_route_equals_unpipelined_float64(route, kind, H, W, monkeypatch):
    import umpa_b200
    dtype, pinned, env, threads, staged = ROUTES[route]
    cls = {"DF": umpa_b200.UMPAModelDF, "NoDF": umpa_b200.UMPAModelNoDF}[kind]
    # frames differ from test to test: a model's FP64 stacks may come from the block cache, still holding the
    # frames of an earlier model, and must not pass the cost() probe below by that accident
    seed = 1000 + 10 * list(ROUTES).index(route) + 2 * SHAPES.index((H, W)) + (kind == "DF")
    sam, ref = _frames(seed, H, W, dtype, pinned)
    wide = [[np.asarray(f, dtype=np.float64) for f in s] for s in (sam, ref)]

    monkeypatch.setenv("UMPA_NO_STREAMING", "1")
    m64 = cls(*wide, max_shift=MAX_SHIFT)                # kept alive: its stacks stay out of the block cache
    want = m64.match(quiet=True)
    monkeypatch.delenv("UMPA_NO_STREAMING")

    monkeypatch.setenv("UMPA_STAGE_SYNC", "1")
    monkeypatch.delenv("UMPA_HOST_FRAC", raising=False)
    monkeypatch.delenv("UMPA_BANDS", raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    m = cls(sam, ref, max_shift=MAX_SHIFT)
    assert m._f32 == (dtype == np.float32)
    got = m.match(quiet=True)
    info = m.last_stream_info
    assert m.last_match_info["path"] == "table"
    assert info["bands"] > 1, info
    assert info["host_threads"] == threads and info["host_rows_per_frame"] == staged(H), info

    keys = ("f", "T", "dx", "dy", "err", "debug_Ncalls", "debug_d") + (("df",) if kind == "DF" else ())
    for k in keys:
        assert np.array_equal(got[k], want[k], equal_nan=True), k

    # the cost() hook reads the FP64 stacks: rows that crossed as FP32 must be brought up first
    pad = m.padding
    for i, j in ((pad + 11, pad + 17), (H - pad - 5, W - pad - 7)):
        c, c64 = m.cost(i, j, 1, -2), m64.cost(i, j, 1, -2)
        assert np.all(np.isfinite(c64)) and c == c64, (i, j, c, c64)
