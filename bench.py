#!/usr/bin/env python
"""bench.py -- output pixels/s of UMPAModelDF.match() (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2] [--dump-outputs DIR]

One "step" = one match() over one synthetic speckle stack of the named configuration; each GPU measurement below
(value, e2e, stage times, gather) times K steps.  The stacks are generated from a fixed seed, so the same arguments
give the same inputs on every run.
N > 1 is launched with torchrun (one rank per GPU); the output rows of the SAME stack are
split into N row bands (+ halo), no collective on the data path (strong scaling).

Printed JSON (one line, rank 0):
  value        device-resident throughput: centred FP32 stacks already in HBM, result maps left
               in HBM; CUDA events around K steps, max over ranks.
  e2e          same metric through the public drop-in API with HOST buffers: per step the float64
               stacks go host(pinned)->device, are converted, matched, and the result maps come
               back to pinned host memory.
  roofline     the kernel with the largest share of the step: its BINDING resource (the largest of executed FP32
               FMAs / measured FFMA peak, DRAM bytes / measured copy bandwidth, shared-memory wavefronts / cycle,
               issued instructions / issue slots) as achieved / peak = frac <= ~1; per kernel the live CUDA-event
               time x the per-launch counters of the committed ncu capture (profiles/r02_kernels.json).  The
               direct-form figure of SURVEY.md 8d (2*S^2*Na*K^2 flop/px) is reported beside it as
               `algorithmic_speedup` / `frac_alg_step`: the kernels execute ~13x fewer FMAs than that form.
  parity       the maps of this run against the UNMODIFIED reference on the block of rows the cpu_baseline leg
               computes anyway (tests/helpers.py::fp32_parity_stats).
  cpu_baseline the reference's own OpenMP CPU path (oracle/_ref, built from /root/reference) or
               the C port, timed on this box's host cores on a bounded ROI of the same workload.

--dump-outputs DIR writes the maps the last timed step returned (see dump_outputs) so that two builds can be
compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    "cfg1": dict(kind="NoDF", Na=10, H=256, W=256, Nw=2, ms=4, desc="UMPAModelNoDF 10x256^2 Nw=2 max_shift=4"),
    "cfg2": dict(kind="DF", Na=25, H=2048, W=2048, Nw=2, ms=5, desc="UMPAModelDF 25x2048^2 Nw=2 max_shift=5"),
    "cfg3": dict(kind="DFKernel", Na=25, H=2048, W=2048, Nw=3, ms=5, desc="UMPAModelDFKernel 25x2048^2 Nw=3 max_shift=5"),
    "cfg4": dict(kind="DF", Na=40, H=4096, W=4096, Nw=3, ms=8, desc="UMPAModelDF 40x4096^2 Nw=3 max_shift=8"),
    "cfg5": dict(kind="NoDF", Na=4, H=2048, W=2048, Nw=6, ms=4, desc="UMPAModelNoDF 4x2048^2 Nw=6 max_shift=4"),
}
SAFE_CROP = {"NoDF": 0, "DF": 0, "DFKernel": 8}
# Per-launch counters of the kernels of one config-2 step (N = 1), from `ncu --set full` of `python tools/prof_step.py cfg2`
# (tools/ncu_kernels.py writes the file; everything in `roofline` that is not a live time comes from it).
NCU_KERNELS = os.path.join(ROOT, "profiles", "r02_kernels.json")


def algorithmic_flops_per_px(cfg):
    """SURVEY.md 8(d): F_alg = 2*S^2*Na*K^2 (+ blur for DFKernel)."""
    S, K, Na = 2 * cfg["ms"] - 1, 2 * cfg["Nw"] + 1, cfg["Na"]
    f = 2. * S * S * Na * K * K
    if cfg["kind"] == "DFKernel":
        f = 2. * Na * ((K + S - 1) ** 2 * 17 ** 2 + 2 * S * S * K * K)
    return f


def table_plan(cfg):
    """(streaming, chunk rows) of the cross-table kernel for a configuration: the plan the library itself makes
    (umpa_table_plan -> plan_tiles, table_path.cu; host arithmetic, no device needed)."""
    import ctypes
    from umpa_b200 import _capi
    out = (ctypes.c_int * 10)()
    rows, cols = (cfg[k] - 2 * (cfg["Nw"] + cfg["ms"]) for k in ("H", "W"))
    _capi.check(_capi.lib().umpa_table_plan(cfg["Na"], cfg["Nw"], cfg["ms"], rows, cols, 148, out))
    return out[1] > 0, out[0]


def executed_fma_per_px_cross(cfg):
    """FMAs the cross-table kernel executes per output pixel (shift_table.cuh): Na per (chunk pixel, shift) -- a chunk
    is 32 columns wide for 32 - 2 Nw output columns -- plus the separable filter (row pass on the chunk rows, column
    pass on the outputs).  Streaming segments pay the window halo in y once per segment (not at all, to first order);
    halo tiles compute EH rows for EH - 2 Nw output rows."""
    S, K, Na, Nw = 2 * cfg["ms"] - 1, 2 * cfg["Nw"] + 1, cfg["Na"], cfg["Nw"]
    stream, eh = table_plan(cfg)
    tw = (32 - 2 * Nw) & ~3
    th = eh if stream else eh - 2 * Nw
    return S * S * ((Na + K) * eh * 32. + K * th * tw) / (th * tw)


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_stacks(cfg, device, seed=2):
    from umpa_b200 import synth
    d = synth.speckle_stack(cfg["Na"], cfg["H"], cfg["W"], seed=seed, max_shift=cfg["ms"],
                            dark_field=cfg["kind"] != "NoDF", device=device, as_numpy=False)
    return d["sam"], d["ref"]


# ------------------------------------------------------------------------------ reference arm

def cpu_model(cfg, sam_np, ref_np):
    """(model factory result, kind): the compiled reference when available, else the C port."""
    from oracle import ref as oref
    R = oref.load(build_if_missing=os.path.exists("/root/reference"))
    sam_l, ref_l = [s for s in sam_np], [r for r in ref_np]
    if R is not None:
        cls = {"NoDF": R.UMPAModelNoDF, "DF": R.UMPAModelDF, "DFKernel": R.UMPAModelDFKernel}[cfg["kind"]]
        return cls(sam_l, ref_l, window_size=cfg["Nw"], max_shift=cfg["ms"]), "reference"
    from oracle import port
    return port.OracleModel(cfg["kind"], sam_l, ref_l, window_size=cfg["Nw"], max_shift=cfg["ms"]), "port"


def cpu_match(model, kind, roi, cores, cfg):
    kw = {}
    if cfg["kind"] == "DFKernel":
        from umpa_b200 import synth
        n0 = 1 + (roi[0][1] - roi[0][0] - 1) // roi[0][2]
        n1 = 1 + (roi[1][1] - roi[1][0] - 1) // roi[1][2]
        kw["abc"] = synth.blur_abc(n0, n1)
    t = time.perf_counter()
    if kind == "reference":
        res = model.match(ROI=roi, num_threads=cores, quiet=True, **kw)
    else:
        res = model.match(ROI=roi, num_threads=cores, debug=False, **kw)
    dt = time.perf_counter() - t
    return res["err"].size, dt, res


def centred_roi(cfg, n_px_target):
    pad = cfg["ms"] + cfg["Nw"] + SAFE_CROP[cfg["kind"]]
    N0, N1 = cfg["H"] - 2 * pad, cfg["W"] - 2 * pad
    rows = int(max(8, min(N0, round(n_px_target / float(N1)))))
    r0 = (N0 - rows) // 2
    return ((r0, r0 + rows, 1), (0, N1, 1)), rows * N1


def run_cpu_sample(cfg, sam_np, ref_np, target_s, steps=1, warmup=0, keep_result=False):
    """Times the CPU path on a centred full-width row block sized for ~target_s per step.
    keep_result: also return (roi, result dict of the last step) for the parity record."""
    cores = os.cpu_count() or 1
    model, kind = cpu_model(cfg, sam_np, ref_np)
    roi, npx = centred_roi(cfg, 20000)
    _, dt, _ = cpu_match(model, kind, roi, cores, cfg)              # calibration (also warms caches)
    rate = npx / max(dt, 1e-6)
    roi, npx = centred_roi(cfg, rate * target_s)
    for _ in range(warmup):
        cpu_match(model, kind, roi, cores, cfg)
    times, res = [], None
    for _ in range(steps):
        n, dt, res = cpu_match(model, kind, roi, cores, cfg)
        times.append(dt)
    t = float(np.mean(times))
    sample = "centred full-width block of %d rows (%d px) of %s, %d threads" % (
        roi[0][1] - roi[0][0], npx, cfg["desc"], cores)
    base = dict(value=npx / t, unit="output pixels/s", cores=cores, kind=kind, sample=sample)
    if keep_result:
        return base, t, npx, roi, res
    return base, t, npx


def reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    sam, ref = make_stacks(cfg, dev)
    sam_np, ref_np = sam.cpu().numpy(), ref.cpu().numpy()
    del sam, ref
    # each step ~ (120 s budget) / (steps + warmup + calibration)
    per_step = max(1.0, min(15.0, 120.0 / (args.steps + args.warmup + 1)))
    base, t, npx = run_cpu_sample(cfg, sam_np, ref_np, per_step, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": "output pixels/s", "value": base["value"], "unit": "output pixels/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": cfg["desc"], "sample": base["sample"]},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "output pixels/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ our arm

DUMP_SAMPLE_PX = 1 << 20


def dump_outputs(out, directory, seed=0):
    """Writes each map of one match_device() result as DIR/<name>.npy: float64 maps as float64, the integer maps (err,
    debug_Ncalls) as float32, which holds them exactly.  A map of more than DUMP_SAMPLE_PX pixels is written as the
    1-D sample np.sort(np.random.default_rng(seed).choice(pixels, DUMP_SAMPLE_PX, replace=False)) of its row-major
    pixels, the same sample for every map: at most 2^20 x (5 x 8 + 2 x 4) bytes = 48 MiB in all."""
    os.makedirs(directory, exist_ok=True)
    maps = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}     # (not the "_keepalive" entry)
    n_px = next(iter(maps.values())).size
    idx = None
    if n_px > DUMP_SAMPLE_PX:
        idx = np.sort(np.random.default_rng(seed).choice(n_px, DUMP_SAMPLE_PX, replace=False))
    for k, v in maps.items():
        v = v.astype(np.float64 if v.dtype == np.float64 else np.float32)
        np.save(os.path.join(directory, k + ".npy"), v if idx is None else v.reshape(-1)[idx])

STAGES = ("moments", "cross_table", "mean_table", "walk")


def kernel_roofline(cfg_name, world, stage_ms, fma_peak, hbm_gbs, sm_mhz, sms):
    """Per kernel of the step: live CUDA-event time x the per-launch counters of the committed ncu capture ->
    fraction of each resource; the kernel's `frac` is its binding (largest) one.  Returns (per-kernel dict, source)."""
    try:
        ncu = json.load(open(NCU_KERNELS))
    except Exception:
        return None, None
    if cfg_name != ncu.get("config", "cfg2") or world != 1:
        return None, None
    pick = {}
    for name, k in ncu["kernels"].items():
        if name.startswith("moments"):
            pick["moments"] = (name, k)
        elif name.startswith("shift_table_kernel") and name.rstrip(">").endswith("-1"):
            pick["mean_table"] = (name, k)
        elif name.startswith("shift_table_kernel") or name.startswith("ktable"):
            pick["cross_table"] = (name, k)
        elif name.startswith("table_walk"):
            pick["walk"] = (name, k)
    out = {}
    for st, ms in zip(STAGES, stage_ms):
        if st not in pick or ms <= 0.:
            continue
        name, k = pick[st]
        scale = k["ncu_duration_ns"] * 1e-6 / ms                 # same work, profiled duration vs live duration
        if k.get("captured_before"):                             # the kernel issues less work than when it was profiled:
            scale = 1.                                           # its pipe utilisations are reported as profiled
        dram = k["dram_read_bytes"] + k["dram_write_bytes"]
        fr = {"fma_pipe": k["fma_pipe_pct"] / 100. * scale,
              "hbm": dram / (ms * 1e-3) / 1e9 / hbm_gbs,
              "shared_memory": k["smem_wavefronts"] / (sms * k["sm_cycles"]) * scale,
              "issue_slots": k["issue_active_pct"] / 100. * scale}
        bound = max(fr, key=fr.get)
        out[st] = {"kernel": name, "ms": ms, "ncu_ms": k["ncu_duration_ns"] * 1e-6, "dram_bytes": dram,
                   "warp_inst": k["warp_inst"], "smem_wavefronts": k["smem_wavefronts"],
                   "fractions": fr, "bound": bound, "frac": fr[bound]}
        if k.get("captured_before"):
            out[st]["note"] = k["captured_before"]
    return out, "profiles/%s (%s; ncu --set full of `%s`)" % (os.path.basename(NCU_KERNELS), ncu.get("source"), ncu.get("command"))


def ours(args, cfg):
    import torch
    import torch.distributed as dist
    import umpa_b200
    from umpa_b200 import _capi
    from umpa_b200.sharding import ShardedMatcher
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    cls = {"NoDF": umpa_b200.UMPAModelNoDF, "DF": umpa_b200.UMPAModelDF,
           "DFKernel": umpa_b200.UMPAModelDFKernel}[cfg["kind"]]
    sam, ref = make_stacks(cfg, dev)
    pad = cfg["ms"] + cfg["Nw"] + SAFE_CROP[cfg["kind"]]
    N0, N1 = cfg["H"] - 2 * pad, cfg["W"] - 2 * pad
    total_px = N0 * N1
    kw = {}
    if cfg["kind"] == "DFKernel":
        from umpa_b200 import synth
        kw["abc"] = synth.blur_abc(N0, N1, as_numpy=False).to(dev)
    keys = ("f", "T", "dx", "dy") + (("df",) if cfg["kind"] == "DF" else ()) + ("err", "debug_Ncalls")

    # ---- device-resident metric -------------------------------------------------
    # one step = one match of this rank's row band.  For N > 1 the maps are then gathered on rank 0 -- the only
    # inter-GPU traffic of the path (north_star) -- which SURVEY.md 5 / 8(d) keep outside the kernel-timed region
    # and report separately: `gather` below (and `value_incl_gather`)
    sm = ShardedMatcher(cls, list(sam), list(ref), rank, world, window_size=cfg["Nw"], max_shift=cfg["ms"])
    band_rows = sm.band[1] - sm.band[0]
    lo, hi = sm.band[0], sm.band[1] + 2 * pad

    def step():
        return sm.match_device(**kw)
    launches = 0
    for _ in range(args.warmup):
        out = step()
    info = sm.model.last_match_info if sm.model is not None else {"path": "none", "kernel_launches": 0}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(args.steps):
            out = step()
            launches += info["kernel_launches"]
        e1.record()
        torch.cuda.synchronize()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    value = total_px / (ms * 1e-3)
    launches = int(sum_over_ranks(launches))
    gather = None
    if world > 1:                                 # the final gather of the maps on rank 0, timed on its own
        full = sm.gather(out, keys=keys, dst=0)   # (warm-up: NCCL sets up its channels on first use)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        g0.record()
        for _ in range(args.steps):
            full = sm.gather(out, keys=keys, dst=0)
        g1.record()
        torch.cuda.synchronize()
        barrier()
        g_ms = max_over_ranks(g0.elapsed_time(g1) / args.steps)
        nbytes = sum_over_ranks(0. if rank == 0 else float(sum(out[k].numel() * out[k].element_size() for k in keys if k in out)))
        gather = {"gather_ms": g_ms, "bytes_to_rank0": int(nbytes), "gbs_into_rank0": nbytes / (g_ms * 1e-3) / 1e9,
                  "value_incl_gather": total_px / ((ms + g_ms) * 1e-3),
                  "how": "point to point (sharding.gather_bands: one torch.distributed.batch_isend_irecv group over NCCL / "
                         "NVLink; four ranks and more: every rank sends each map straight into its row slice of the full "
                         "map; fewer: two packed messages per rank) after the timed steps; rank 0 ends with the full "
                         "(N0, N1) maps in its HBM"}
        if rank == 0:
            out = full
    err_ok = None
    if rank == 0:
        err_ok = float((out["err"] == 1).sum().item()) / total_px          # rank 0 holds the whole map (gathered for N > 1)
        if args.dump_outputs:
            dump_outputs(out, args.dump_outputs)

    # ---- stage times of the kernels (events inside the library, same stream) -------
    stage_ms = None
    if sm.model is not None and info["path"] == "table":
        _capi.check(_capi.lib().umpa_set_profiling(sm.model._h, 1))
        acc = []
        for _ in range(args.steps):
            sm.match_device(**kw)
            buf = (C.c_float * 4)()
            if _capi.lib().umpa_last_stage_ms(sm.model._h, buf, 4) == 4:
                acc.append(list(buf[:4]))
        _capi.check(_capi.lib().umpa_set_profiling(sm.model._h, 0))
        stage_ms = np.median(np.array(acc), axis=0).tolist() if acc else None      # (median: robust against a stray slow launch)
    peak = C.c_double(0.)
    sms = C.c_int(0)
    _capi.check(_capi.lib().umpa_fma_peak(C.byref(peak), C.byref(sms)))
    out_host = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out_host = {k: v.cpu().numpy() for k, v in out.items() if k in keys}

    # ---- end to end through the drop-in API with host buffers --------------------------------
    e2e = None
    if not args.no_e2e:
        hs = torch.empty((cfg["Na"], hi - lo, cfg["W"]), dtype=torch.float64, pin_memory=True)
        hr = torch.empty_like(hs, pin_memory=True)
        hs.copy_(sam[:, lo:hi]); hr.copy_(ref[:, lo:hi])
        torch.cuda.synchronize()
        sam_np, ref_np = hs.numpy(), hr.numpy()
        kw_h = {}
        if "abc" in kw:
            kw_h["abc"] = kw["abc"][sm.band[0]:sm.band[1]].cpu().numpy()
        del sm, out
        steps_e = args.steps
        d2h = 0

        stream_info = {}

        def one():
            m = cls(list(sam_np), list(ref_np), window_size=cfg["Nw"], max_shift=cfg["ms"])
            r = m.match(quiet=True, debug=False, **kw_h)
            stream_info.update(m.last_stream_info)
            return sum(v.nbytes for v in r.values())
        barrier()
        t0 = time.perf_counter()
        d2h = one()                              # the first host-to-host call of the process (pins staging / result buffers)
        first_ms = max_over_ranks(1e3 * (time.perf_counter() - t0))
        # the pinned staging buffer of the host conversion is built in the background (the first calls go by plain
        # DMA): warm up until the pipeline has reached its steady state, then three more calls (they measure the host rates)
        t_w = time.perf_counter()
        while stream_info.get("host_threads", 0) == 0 and time.perf_counter() - t_w < 5.:
            d2h = one()
        for _ in range(max(3, args.warmup)):
            d2h = one()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps_e):
            d2h = one()
        torch.cuda.synchronize()
        t_e = (time.perf_counter() - t0) / steps_e
        barrier()
        t_own = t_e
        t_e = max_over_ranks(t_e)
        e2e = {"value": total_px / t_e, "unit": "output pixels/s", "ms_per_step": 1e3 * t_e, "first_call_ms": first_ms,
               "h2d_bytes_per_step": int(sum_over_ranks(float(sam_np.nbytes + ref_np.nbytes))),
               "d2h_bytes_per_step": int(sum_over_ranks(float(d2h))), "steps": steps_e,
               "api": "%s(sam, ref, window_size, max_shift).match(debug=False) on pinned host float64 arrays"
                      % cls.__name__,
               "pipeline": dict(stream_info, note="upload / kernels / download overlapped in row bands; host_threads "
                                "convert the lower host_rows_per_frame rows of every frame to centred FP32 in pinned "
                                "staging while the DMA engine uploads the upper rows as FP64 (UMPA_HOST_THREADS=0 "
                                "disables the host part)")}
        if world > 1:
            # what every rank's pipeline did (all ranks of a box share one host memory system): its own time per call,
            # host threads, rows per frame converted on the host, and the PCIe rate of its own link
            mine = {"rank": rank, "ms_per_step": 1e3 * t_own, "host_threads": stream_info.get("host_threads", 0),
                    "host_rows_per_frame": stream_info.get("host_rows_per_frame", 0), "rows": hi - lo}
            hrows = mine["host_rows_per_frame"]
            up = 2 * cfg["Na"] * cfg["W"] * (4 * hrows + 8 * (hi - lo - hrows))
            mine["pcie_up_gbs"] = up / t_own / 1e9
            mine["host_conversion_gbs"] = 2 * cfg["Na"] * cfg["W"] * 8 * hrows / t_own / 1e9
            t = torch.tensor([mine[k] for k in ("rank", "ms_per_step", "host_threads", "host_rows_per_frame", "rows",
                                                "pcie_up_gbs", "host_conversion_gbs")], dtype=torch.float64, device=dev)
            allr = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(allr, t)
            e2e["per_rank"] = [dict(zip(("rank", "ms_per_step", "host_threads", "host_rows_per_frame", "rows", "pcie_up_gbs",
                                         "host_conversion_gbs"), (round(v, 3) for v in a.tolist()))) for a in allr]
        # the same call on float32 host frames (detector data; umpa_set_frames_f32): half the upload, no host
        # conversion.  Reported beside the headline, not instead of it: the reference's API is float64.
        hs32 = torch.empty(hs.shape, dtype=torch.float32, pin_memory=True)
        hr32 = torch.empty(hs.shape, dtype=torch.float32, pin_memory=True)
        hs32.copy_(hs); hr32.copy_(hr)
        s32, r32 = hs32.numpy(), hr32.numpy()

        def one32():
            m = cls(list(s32), list(r32), window_size=cfg["Nw"], max_shift=cfg["ms"])
            m.match(quiet=True, debug=False, **kw_h)
        for _ in range(max(3, args.warmup)):
            one32()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps_e):
            one32()
        torch.cuda.synchronize()
        t_32 = (time.perf_counter() - t0) / steps_e
        barrier()
        t_32 = max_over_ranks(t_32)
        e2e["float32_frames"] = {"value": total_px / t_32, "ms_per_step": 1e3 * t_32,
                                 "h2d_bytes_per_step": int(sum_over_ranks(float(s32.nbytes + r32.nbytes))),
                                 "note": "same call, frames given as float32 numpy arrays (widened and centred on the GPU)"}

    # ---- CPU baseline + parity against it (rank 0, N=1 only) ------------------------------------
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu, _, _, roi, res = run_cpu_sample(cfg, sam.cpu().numpy(), ref.cpu().numpy(), args.cpu_seconds, keep_result=True)
        except Exception as e:      # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": "output pixels/s", "cores": os.cpu_count(), "kind": "unavailable",
                   "sample": "failed: %r" % (e,)}
            res = None
        if res is not None and "debug_d" in res:
            # the block the reference just computed against the same rows of the device-resident maps of the timed steps
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from helpers import fp32_parity_stats
            (r0, r1, _), (c0, c1, _) = roi
            got = {k: v[r0:r1, c0:c1] for k, v in out_host.items()}
            parity = fp32_parity_stats(got, res)
            parity["against"] = "%s on rows [%d, %d) x cols [%d, %d) of the output" % (cpu["kind"], r0, r1, c0, c1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.)
    clocks = clk.summary()
    alg_bytes = 2. * cfg["Na"] * cfg["H"] * cfg["W"] * 4 + 6 * 4. * total_px
    roof = None
    if stage_ms is not None:
        dfk = cfg["kind"] == "DFKernel"
        names = ["moments", "blur_table" if dfk else "cross_table", "mean_table", "walk"]
        px_rank = band_rows * N1                         # rank 0's launches process its band
        f_alg = algorithmic_flops_per_px(cfg)
        kern, src = kernel_roofline(args.config, world, stage_ms, peak.value, hbm_peak, clocks.get("sm_mhz") or 1965., sms.value)
        top = int(np.argmax(stage_ms))
        roof = {"stage_ms": dict(zip(names, stage_ms)), "kernels": kern, "source": src,
                "peaks": {"fp32_fma_tflops": peak.value, "fp32_fma_source": "FFMA probe measured in this run on this GPU (umpa_fma_peak)",
                          "hbm_gbs": hbm_peak, "hbm_source": "MEASURED_PEAKS.json" if peaks else "fallback of B200_PROFILING.md",
                          "shared_memory": "128 B (one wavefront) per SM and cycle", "issue_slots": "4 per SM and cycle"},
                # the direct form of SURVEY.md 8d, for the record: the kernels do the same sums with far fewer FMAs
                "algorithmic_flop_per_px": f_alg,
                "frac_alg_step": f_alg * px_rank / (sum(stage_ms) * 1e-3) / 1e12 / peak.value,
                "note_alg": "frac_alg_step = direct-form flops (2*S^2*Na*K^2 per px, SURVEY 8d) / step time / FFMA peak; "
                            "above 1 because the frames are summed before the window filter (exact algebra)"}
        if kern:
            st = STAGES[top]
            k = kern[st]
            unit = {"fma_pipe": "TFLOP/s", "hbm": "GB/s", "shared_memory": "wavefronts/cycle/SM", "issue_slots": "inst/cycle/SM"}[k["bound"]]
            pk = {"fma_pipe": peak.value, "hbm": hbm_peak, "shared_memory": 1., "issue_slots": 4.}[k["bound"]]
            roof.update({"kernel": k["kernel"], "bound": k["bound"], "achieved": k["frac"] * pk, "peak": pk, "unit": unit,
                         "frac": k["frac"], "traffic": k["dram_bytes"], "kernel_ms": k["ms"]})
            tot = sum(v["dram_bytes"] for v in kern.values())
            roof["step"] = {"dram_bytes": tot, "algorithmic_bytes": alg_bytes, "traffic_over_algorithmic": tot / alg_bytes,
                            "hbm_floor_ms_of_traffic": tot / hbm_peak / 1e6, "hbm_floor_ms_algorithmic": alg_bytes / hbm_peak / 1e6,
                            "step_ms": sum(stage_ms)}
            if not dfk:
                f_exe = 2. * executed_fma_per_px_cross(cfg) + (2. * (2 * cfg["ms"] - 1) ** 2 * cfg["Na"] if cfg["kind"] == "DF" else 0.)
                roof["algorithmic_speedup"] = f_alg / f_exe
        else:
            roof.update({"kernel": names[top], "bound": None, "achieved": None, "peak": None, "unit": None, "frac": None,
                         "traffic": None, "kernel_ms": stage_ms[top],
                         "note": "no ncu capture committed for this configuration / GPU count: stage times only"})
    line = {"metric": "output pixels/s", "value": value, "unit": "output pixels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["desc"], "output_px": total_px, "sharding": "row bands x%d + %d-row halo" % (world, pad),
                       "path": info["path"], "l2": "inputs (%.0f MB FP32 stacks) larger than the 126 MB L2, no flush" % (alg_bytes / 1e6),
                       "inputs_resident": "mean-centred FP32 stacks in HBM; result maps (f,T,dx,dy,df f64; err,Ncalls i32) left in HBM"
                                          + (" of each rank (then gathered on rank 0: see `gather`)" if world > 1 else ""),
                       "err_ok_fraction": err_ok},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "gather": gather, "parity": parity,
            "roofline_hbm_step": {"bound": "hbm", "achieved": alg_bytes / (ms * 1e-3) / 1e9 / world, "peak": hbm_peak,
                                  "unit": "GB/s", "frac": alg_bytes / (ms * 1e-3) / 1e9 / world / hbm_peak,
                                  "note": "algorithmic bytes of the whole step (stacks once + 6 maps) per GPU-second"},
            "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the maps of the last timed step to DIR/<name>.npy (float32 / float64, a fixed seeded "
                         "sample of 2^20 pixels of larger maps)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the maps of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        reference_arm(args, cfg)
    else:
        ours(args, cfg)


if __name__ == "__main__":
    main()
