"""GPU: the BASELINE.json configurations at FULL size against the UNMODIFIED reference (oracle/_ref, the
reference's own C++/OpenMP model: UMPA/model.pyx:476-492 -> Model.cpp / Optim.cpp), directly where its compiled
extension is present, otherwise against the C restatement of it (oracle/port.py, pinned to the reference by the
golden vectors): helpers.reference_matcher.

The product matches the whole frame on the GPU (table path); the reference matches a block of rows of the SAME
float64 stacks on the host cores (pixels are independent, so a block is exactly what the full run would
give there).  The blocks are placed across what the small golden fixtures cannot see: the edge of two row
segments / chunks of the streaming table kernel, the edge of two column strips, the 2048- / 4096-wide pitch, S = 15.

Every comparison goes through helpers.fp32_parity_stats and is written to gpurun_out/parity_<config>.json
(copied to profiles/parity_r02.json).  On this clean synthetic speckle the budget is: err maps equal, no walk or
T/df deviation that is not a documented tie, NO dx/dy/f exception."""
import json
import os

import numpy as np
import pytest

from helpers import fp32_parity_stats, reference_matcher

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _record(name, stats):
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parity_%s.json" % name), "w") as f:
            json.dump(stats, f, indent=1, sort_keys=True)
    print(name, json.dumps(stats, sort_keys=True))


def _check(name, stats, min_ok=.999):
    _record(name, stats)
    assert stats["err_mismatch"] == 0, stats
    assert stats["n_ok"] >= min_ok * stats["n_px"], stats
    assert stats["walk_unexplained"] == 0 and stats["walk_ties"] <= max(2, 2e-3 * stats["n_ok"]), stats
    for k in ("T", "df"):
        assert stats.get(k + "_unexplained", 0) == 0, stats
    assert stats["exceptions"] == 0, stats                  # clean synthetic data: nothing to excuse
    for k in ("dx", "dy"):
        assert stats[k + "_max"] <= 1e-4, stats


def _run(kind, Na, N, Nw, ms, blocks, seed=2, abc_fn=None):
    """blocks: list of ROIs ((r0, r1, 1), (c0, c1, 1)) in output coordinates.  Returns the merged stats."""
    import torch
    import umpa_b200
    from umpa_b200 import synth
    d = synth.speckle_stack(Na, N, N, seed=seed, max_shift=ms, dark_field=kind != "NoDF", device="cuda", as_numpy=False)
    cls = {"NoDF": umpa_b200.UMPAModelNoDF, "DF": umpa_b200.UMPAModelDF, "DFKernel": umpa_b200.UMPAModelDFKernel}[kind]
    m = cls(list(d["sam"]), list(d["ref"]), window_size=Nw, max_shift=ms)
    kw = {}
    abc = None
    if kind == "DFKernel":
        abc = synth.blur_abc(*m.sh)
    sam_np, ref_np = d["sam"].cpu().numpy(), d["ref"].cpu().numpy()
    match_ref, against = reference_matcher(kind, sam_np, ref_np, window_size=Nw, max_shift=ms)
    merged = None
    for roi in blocks:
        (r0, r1, _), (c0, c1, _) = roi
        if abc is not None:
            kw["abc"] = np.ascontiguousarray(abc[r0:r1, c0:c1])
        got = m.match(ROI=roi, quiet=True, debug=False, **kw)
        assert m.last_match_info["path"] == "table", m.last_match_info
        exp = match_ref(roi, **kw)
        st = fp32_parity_stats(got, exp)
        if merged is None:
            merged = st
        else:
            for k, v in st.items():
                if k.endswith("_max") or k.endswith("_p999"):
                    merged[k] = max(merged[k], v)
                elif k not in ("tol", "cost_scale"):
                    merged[k] += v
    merged["blocks"] = [list(map(list, b)) for b in blocks]
    merged["workload"] = "%s %dx%d^2 Nw=%d max_shift=%d" % (kind, Na, N, Nw, ms)
    merged["against"] = against
    del m, match_ref, d
    torch.cuda.empty_cache()
    return merged


def test_cfg2_block_vs_reference():
    """Config 2 (the metric): 96 full-width rows across the middle of the frame (where the streaming table kernel
    joins two row segments) and a 160-column block down the left edge over 600 rows (segment starts, chunk edges)."""
    st = _run("DF", 25, 2048, 2, 5, [((969, 1065, 1), (0, 2034, 1)), ((0, 600, 1), (0, 160, 1))])
    _check("cfg2", st)


def test_cfg4_block_vs_reference():
    """Config 4 (DF 40 x 4096^2, Nw=3, max_shift=8, S=15): 64 rows through a tile edge, full width."""
    st = _run("DF", 40, 4096, 3, 8, [((2010, 2074, 1), (0, 4074, 1))])
    _check("cfg4", st)


def test_cfg5_block_vs_reference():
    """Config 5 (NoDF 4 x 2048^2, Nw=6): 128 rows across the middle, full width."""
    st = _run("NoDF", 4, 2048, 6, 4, [((950, 1078, 1), (0, 2028, 1))])
    _check("cfg5", st, min_ok=.99)


def test_cfg3_roi_vs_reference():
    """Config 3 (DFKernel 25 x 2048^2, Nw=3): a 48 x 48 ROI (the reference needs ~1 s per 2000 pixels here)."""
    st = _run("DFKernel", 25, 2048, 3, 5, [((1000, 1048, 1), (700, 748, 1))])
    _check("cfg3", st)


def test_cfg1_full_vs_reference():
    """Config 1 (NoDF 10 x 256^2): the whole frame."""
    st = _run("NoDF", 10, 256, 2, 4, [((0, 244, 1), (0, 244, 1))])
    _check("cfg1", st, min_ok=.99)
