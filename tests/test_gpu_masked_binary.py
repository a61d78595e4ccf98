"""GPU: dead-pixel maps (mask values 0 / 1, the same in every frame) on the table path.

The reference's masked branch (Model.cpp:461-499 NoDF, 775-847 DF) weights every window position with
combine_weights(mask(p+s+u), mask(p+u)) (Utils.cpp:125-130) -- for 0 / 1 masks a constant where both pixels are
live, 0 otherwise.  The product keeps such models on the table kernels: the sums of a pixel with a dead pixel
within reach are the unmasked table sums minus the window positions the mask removes (table_path.cu:
masked_walk_kernel; the algebra itself is checked on CPU in tests/test_table_algebra.py).  Oracle: the C
restatement of the reference (oracle/port.py) on the same stacks and masks.  Criteria: those of the unmasked table
path (helpers.compare_fp32: err map and integer walk equal, values to 1e-4)."""
import os

import numpy as np
import pytest

from helpers import compare_fp32
from oracle import port

pytestmark = pytest.mark.gpu


def _stacks(Na, H, W, seed, ms, dark_field):
    from umpa_b200 import synth
    d = synth.speckle_stack(Na, H, W, seed=seed, max_shift=ms, dark_field=dark_field)
    return [np.array(s) for s in d["sam"]], [np.array(r) for r in d["ref"]]


def _dead_map(H, W, frac, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((H, W)) >= frac).astype(np.float64)


def _product(kind, sam, ref, masks, Nw, ms):
    import umpa_b200
    cls = {"NoDF": umpa_b200.UMPAModelNoDF, "DF": umpa_b200.UMPAModelDF}[kind]
    return cls(sam, ref, mask_list=masks, window_size=Nw, max_shift=ms)


@pytest.mark.parametrize("kind,Nw,ms,frac", [("DF", 2, 4, .03), ("NoDF", 2, 4, .03), ("DF", 1, 3, .08), ("NoDF", 3, 5, .02),
                                             ("DF", 3, 5, .01), ("DF", 2, 4, .3)])
def test_dead_pixel_map_on_the_table_path(kind, Nw, ms, frac):
    """Random dead pixels (1 % ... 30 %: up to most of a window gone), odd frame width (the bit image's last word)."""
    H, W, Na = 96, 109, 6
    sam, ref = _stacks(Na, H, W, seed=11 + Nw, ms=ms, dark_field=kind == "DF")
    M = _dead_map(H, W, frac, seed=5)
    rng = np.random.default_rng(9)
    for k in range(Na):                       # what a dead pixel reads is arbitrary (within the live range)
        sam[k][M == 0] = rng.random(int((M == 0).sum())) * 2.
        ref[k][M == 0] = rng.random(int((M == 0).sum())) * 2.
    masks = [M.copy() for _ in range(Na)]
    m = _product(kind, sam, ref, masks, Nw, ms)
    got = m.match(quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    exp = port.OracleModel(kind, sam, ref, mask_list=masks, window_size=Nw, max_shift=ms).match()
    st = compare_fp32(got, exp, tol=1e-4, label="%s Nw=%d dead %.2f" % (kind, Nw, frac))
    print(st)
    # and the FP64 lazy evaluation (the path such a model took before) agrees with both
    m.cuda_path = "lazy"
    lazy = m.match(quiet=True)
    ok = (exp["err"] == 1) & (got["debug_Ncalls"] == exp["debug_Ncalls"])
    assert ok.mean() > .5
    assert np.abs(lazy["T"][ok] - got["T"][ok]).max() < 1e-4


def test_roi_with_a_step():
    H, W, Na, Nw, ms = 90, 100, 5, 2, 4
    sam, ref = _stacks(Na, H, W, seed=3, ms=ms, dark_field=True)
    masks = [_dead_map(H, W, .04, seed=6)] * Na
    m = _product("DF", sam, ref, masks, Nw, ms)
    N0, N1 = m.sh
    got = m.match(ROI=((4, N0 - 5, 3), (2, N1 - 7, 3)), quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    om = port.OracleModel("DF", sam, ref, mask_list=masks, window_size=Nw, max_shift=ms)
    exp = om.match(ROI=((4, N0 - 5, 3), (2, N1 - 7, 3)))
    compare_fp32(got, exp, tol=1e-4, label="roi/step")


def test_what_does_not_qualify_stays_on_the_lazy_evaluation():
    """Masks that differ between frames, fractional weights, a hot dead pixel far outside the live range, and
    UMPA_MASK_TABLES=0: the mixed path with the FP64 lazy evaluation, as before -- same results as the oracle."""
    H, W, Na, Nw, ms = 80, 84, 5, 2, 4
    sam, ref = _stacks(Na, H, W, seed=4, ms=ms, dark_field=True)
    M = _dead_map(H, W, .03, seed=8)
    per_frame = [M.copy() for _ in range(Na)]
    per_frame[2][40, 41] = 0. if M[40, 41] else 1.
    frac = [np.where(M == 0, .5, 1.) for _ in range(Na)]
    for masks in (per_frame, frac):
        m = _product("DF", sam, ref, masks, Nw, ms)
        got = m.match(quiet=True)
        assert m.last_match_info["path"] == "mixed", m.last_match_info
        exp = port.OracleModel("DF", sam, ref, mask_list=masks, window_size=Nw, max_shift=ms).match()
        compare_fp32(got, exp, tol=1e-4, label="general masks")
    hot = [s.copy() for s in sam]
    yy, xx = next((y, x) for y, x in np.argwhere(M == 0) if y % 2 == 1 and 20 < y < 60)   # (not on a row the centring samples)
    hot[1][yy, xx] = 1e3
    m = _product("DF", hot, ref, [M] * Na, Nw, ms)
    got = m.match(quiet=True)
    assert m.last_match_info["path"] == "mixed", m.last_match_info
    exp = port.OracleModel("DF", hot, ref, mask_list=[M] * Na, window_size=Nw, max_shift=ms).match()
    compare_fp32(got, exp, tol=1e-4, label="hot dead pixel")


def test_options_changed_after_the_first_match():
    """The classification of the mask stack is cached per set of frames; window size and assign_coordinates may
    change afterwards: a new window size rebuilds the window words, assign_coordinates='ref' takes the role-swapped
    corrected walk."""
    H, W, Na, ms = 84, 90, 5, 4
    sam, ref = _stacks(Na, H, W, seed=6, ms=ms, dark_field=True)
    masks = [_dead_map(H, W, .03, seed=4)] * Na
    m = _product("DF", sam, ref, masks, 3, ms)
    m.match(quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    m.Nw = 2                                   # (the padding stays that of window_size 3, model.pyx:702-704)
    got = m.match(quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    om = port.OracleModel("DF", sam, ref, mask_list=masks, window_size=3, max_shift=ms)
    om.set_Nw(2)
    compare_fp32(got, om.match(), tol=1e-4, label="Nw 3 -> 2")
    m.assign_coordinates = "ref"               # (the sample window moves: Model.cpp:686-692)
    got = m.match(quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    om.set_options(reference_shift=1)
    compare_fp32(got, om.match(), tol=1e-4, label="assign_coordinates = ref")


@pytest.mark.parametrize("kind,Nw", [("NoDF", 4), ("DF", 2)])
def test_assign_coordinates_ref(kind, Nw):
    """assign_coordinates='ref' with a dead-pixel map, also with the window-row words of Nw > 3."""
    H, W, Na, ms = 88, 93, 5, 4
    sam, ref = _stacks(Na, H, W, seed=8, ms=ms, dark_field=kind == "DF")
    masks = [_dead_map(H, W, .02, seed=7)] * Na
    m = _product(kind, sam, ref, masks, Nw, ms)
    m.assign_coordinates = "ref"
    got = m.match(quiet=True)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    om = port.OracleModel(kind, sam, ref, mask_list=masks, window_size=Nw, max_shift=ms)
    om.set_options(reference_shift=1)
    compare_fp32(got, om.match(), tol=1e-4, label="%s ref Nw=%d" % (kind, Nw))


def test_dfkernel_keeps_the_lazy_evaluation():
    import umpa_b200
    from umpa_b200 import synth
    H, W, Na, ms = 80, 86, 5, 4
    sam, ref = _stacks(Na, H, W, seed=7, ms=ms, dark_field=True)
    masks = [_dead_map(H, W, .02, seed=3)] * Na
    m = umpa_b200.UMPAModelDFKernel(sam, ref, mask_list=masks, window_size=2, max_shift=ms)
    abc = synth.blur_abc(*m.sh)
    got = m.match(abc=abc, quiet=True)
    assert m.last_match_info["path"] == "mixed", m.last_match_info
    exp = port.OracleModel("DFKernel", sam, ref, mask_list=masks, window_size=2, max_shift=ms).match(abc=abc)
    compare_fp32(got, exp, tol=1e-4, label="DFKernel with a dead-pixel map")


def test_env_switch_off(monkeypatch):
    H, W, Na, Nw, ms = 70, 72, 4, 2, 3
    sam, ref = _stacks(Na, H, W, seed=5, ms=ms, dark_field=False)
    M = _dead_map(H, W, .03, seed=2)
    monkeypatch.setenv("UMPA_MASK_TABLES", "0")
    m = _product("NoDF", sam, ref, [M] * Na, Nw, ms)
    m.match(quiet=True)
    assert m.last_match_info["path"] == "mixed", m.last_match_info


@pytest.mark.timeout(600)
def test_full_size_block_against_the_reference():
    """Config 2 shapes with a 3 % dead-pixel map (every pixel has a dead pixel within reach): a block of rows against
    the UNMODIFIED reference (oracle/_ref, else its C restatement: helpers.reference_matcher), the whole frame timed;
    the times and the parity record are printed."""
    import json
    import time
    import torch
    import umpa_b200
    from umpa_b200 import synth
    from helpers import fp32_parity_stats, reference_matcher
    Na, N, Nw, ms = 25, 2048, 2, 5
    d = synth.speckle_stack(Na, N, N, seed=2, max_shift=ms, dark_field=True, device="cuda", as_numpy=False)
    sam, ref = d["sam"].cpu().numpy(), d["ref"].cpu().numpy()
    M = _dead_map(N, N, .03, seed=1)
    masks = [M] * Na
    m = umpa_b200.UMPAModelDF(list(sam), list(ref), mask_list=masks, window_size=Nw, max_shift=ms)
    m.match(quiet=True, debug=False)
    assert m.last_match_info["path"] == "masked_table", m.last_match_info
    t0 = time.perf_counter()
    m.match(quiet=True, debug=False)
    t_masked = time.perf_counter() - t0
    roi = ((1000, 1032, 1), (0, 2034, 1))
    got = m.match(ROI=roi, quiet=True, debug=False)
    rec = {"workload": "UMPAModelDF 25x2048^2 Nw=2 max_shift=5, 3 % dead pixels (0/1 mask shared by all frames)",
           "match_ms_host_to_host": 1e3 * t_masked}
    match_ref, against = reference_matcher("DF", sam, ref, mask_list=masks, window_size=Nw, max_shift=ms)
    st = fp32_parity_stats(got, match_ref(roi))
    rec["parity_vs_reference"] = dict(st, against=against)
    assert st["err_mismatch"] == 0 and st["walk_unexplained"] == 0, st
    assert st["exceptions"] - st["excused"] == 0, st
    os.environ["UMPA_MASK_TABLES"] = "0"
    try:
        ml = umpa_b200.UMPAModelDF(list(sam), list(ref), mask_list=masks, window_size=Nw, max_shift=ms)
        ml.match(quiet=True, debug=False)             # (full frame: a ROI would stick, model.pyx:406)
        assert ml.last_match_info["path"] == "mixed", ml.last_match_info
        t0 = time.perf_counter()
        ml.match(quiet=True, debug=False)
        rec["match_ms_lazy_evaluation"] = 1e3 * (time.perf_counter() - t0)
    finally:
        del os.environ["UMPA_MASK_TABLES"]
    print(json.dumps(rec))
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "masked_cfg2.json"), "w") as f:
            json.dump(rec, f, indent=1, sort_keys=True)
    torch.cuda.empty_cache()
